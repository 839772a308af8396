"""fit.p of every window of a fit-window scan, jointly, on the device: ``scan.D`` and the joint covariance ``scan.p``
against plans of each window alone (``Plan.propagate`` for D and the window's own covariance, numpy D_w C D_v^T between
windows), the parent's own propagation for a full-range window, the bootstrap spread of the windows' copies, a
correlated average of windows, the C ABI's refusals, and that asking for ``p`` changes no other result."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _need_gpu():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (no CPU fallback)")


def _data(K, ny=64, seed=3, corr=True, exact=False):
    from lsqfit_b200 import configs
    cfg = configs.correlator(K, ny=ny)
    rng = np.random.default_rng(seed)
    L = np.linalg.cholesky(cfg["ycov"])
    y = cfg["f"] if exact else cfg["f"] + L @ rng.standard_normal(ny)
    ycov = cfg["ycov"] if corr else np.sqrt(np.diag(cfg["ycov"]))
    return cfg, y, ycov


def _fit(K, svdcut=False, corr=True, yp=False, exact=False):
    import lsqfit_b200 as lb
    cfg, y, ycov = _data(K, corr=corr, exact=exact)
    prior = (cfg["prior_mean"], cfg["prior_sdev"])
    kw = {}
    if yp:                      # data-prior correlation: every data row with the first prior entry
        ny, npar = cfg["ny"], cfg["np"]
        C = np.zeros((ny + npar, ny + npar))
        C[:ny, :ny] = ycov
        C[ny:, ny:] = np.diag(cfg["prior_sdev"] ** 2)
        s = np.sqrt(np.diag(C))
        C[:ny, ny] = C[ny, :ny] = 0.1 * s[:ny] * s[ny]
        kw["yp_cov"] = C
    return lb.nonlinear_fit(data=(cfg["x"], y, ycov), fcn="multiexp", prior=prior, svdcut=svdcut, **kw), cfg


def _ranges(ny, npar):
    r = [(0, ny), (0, npar), (ny - npar, ny), (1, 40), (3, 48), (5, 56), (8, ny), (10, 30), (0, 20), (16, ny),
         (30, ny), (2, ny - 1)]
    m = np.zeros((len(r), ny), dtype=bool)
    for w, (lo, hi) in enumerate(r):
        m[w, lo:hi] = True
    return m


def _input_cov(fit):
    pdf = fit.yp_pdf
    return pdf.cov_in if pdf.cov_in is not None else np.diag(pdf.sdev_in ** 2)


def _reference(fit, scan):
    """D_w from a plan of window w alone (embedded in the full y (+) prior), the window's own fit.p covariance, and
    the joint covariance: D_w C D_v^T off the diagonal, the window's own covariance on it."""
    from lsqfit_b200.engine import Plan
    from lsqfit_b200.whiten import PDF
    from lsqfit_b200.windows import window_cov
    spec, pdf = fit._spec, fit.yp_pdf
    cov = pdf.cov_in if pdf.cov_in is not None else pdf.sdev_in
    C = _input_cov(fit)
    nw, npar, N = scan.nwin, spec.np, C.shape[0]
    D = np.zeros((nw, npar, N))
    own = []
    for w, m in enumerate(scan.masks):
        sel, c = window_cov(cov, spec.ny, m)
        alone = PDF(pdf.mean[sel], c, svdcut=pdf.svdcut, eps=pdf.eps)
        plan = Plan(spec.functor, spec.np, int(m.sum()), spec.functor.xrows(spec.x, spec.ny)[m], alone.i_invwgts,
                    noprior=spec.noprior)
        Dw, cw = plan.propagate(scan.pmean[w:w + 1], scan.cov[w:w + 1], alone.cov)
        D[w][:, sel] = Dw[0].cpu().numpy()
        own.append(cw[0].cpu().numpy())
        plan.close()
    S = np.einsum("wai,ij,vbj->wavb", D, C, D)
    for w in range(nw):
        S[w, :, w, :] = own[w]
    return D, S


def _normalised(err, S):
    n = S.shape[0] * S.shape[1]
    s = np.sqrt(np.diagonal(S.reshape(n, n)))
    return np.abs(err.reshape(n, n)) / np.outer(s, s)


def _check(fit, scan):
    Dref, Sref = _reference(fit, scan)
    pmean, S = scan.p
    nw, npar = scan.nwin, scan.np
    assert pmean is scan.pmean and S.shape == (nw, npar, nw, npar)
    D = scan.D
    assert D.shape == Dref.shape
    for w, sel in enumerate(scan.sels):
        scale = np.maximum(np.max(np.abs(Dref[w][:, sel]), axis=0), 1e-300)
        err = np.max(np.abs(D[w][:, sel] - Dref[w][:, sel]), axis=0) / scale
        assert err.max() <= 1e-12, (w, err.max())
        out = np.ones(D.shape[2], dtype=bool)
        out[sel] = False
        assert not D[w][:, out].any(), w
    n = nw * npar
    err = _normalised(S - Sref, Sref)
    assert err.max() <= 1e-10, np.unravel_index(np.argmax(err), err.shape)
    asym = _normalised(S - S.reshape(n, n).T.reshape(S.shape), Sref)
    assert asym.max() <= 1e-14, asym.max()
    assert np.array_equal(scan.p_sdev, np.sqrt(np.diagonal(S.reshape(n, n))).reshape(nw, npar))
    return S


@pytest.mark.parametrize("K", [4, 8])
def test_joint_covariance_against_windows_alone(K):
    _need_gpu()
    fit, cfg = _fit(K)
    scan = fit.window_fits(_ranges(cfg["ny"], cfg["np"]))
    assert np.all(scan.stopping_criterion > 0)
    S = _check(fit, scan)
    # overlapping windows are far from independent: ground-state energy of t = 1..64 and t = 17..64
    n0 = scan.np // 2
    r = S[0, n0, 9, n0] / np.sqrt(S[0, n0, 0, n0] * S[9, n0, 9, n0])
    assert r > 0.5, r


@pytest.mark.parametrize("case", ["svdcut", "drop", "uncorrelated", "yp_cov"])
def test_other_shapes(case):
    _need_gpu()
    fit, cfg = _fit(4, svdcut={"svdcut": 0.05, "drop": -0.01}.get(case, False), corr=case != "uncorrelated",
                    yp=case == "yp_cov")
    scan = fit.window_fits(_ranges(cfg["ny"], cfg["np"]))
    if case == "svdcut":
        assert scan.svdn.max() > 0                      # the svd corrections of the diagonal blocks run
    if case == "drop":
        assert len(set(scan.nchiv)) > 3 and scan.svdn.max() > 0
    if case == "uncorrelated":
        assert all(len(p.i_invwgts) == 1 for p in scan.pdfs)
    if case == "yp_cov":
        assert any(np.any(b >= cfg["ny"]) for b, _ in scan.pdfs[0].i_invwgts[1:])
    _check(fit, scan)


def test_full_range_window_is_the_fit():
    _need_gpu()
    fit, cfg = _fit(4)
    scan = fit.window_fits(np.ones((1, cfg["ny"]), dtype=bool))
    D, covp = fit._spec.plan().propagate(scan.pmean[0], scan.cov[0], fit.yp_pdf.cov)
    D, covp = D[0].cpu().numpy(), covp[0].cpu().numpy()
    S = scan.p[1][0, :, 0, :]
    assert _normalised(S - covp, covp[None, :, None, :]).max() <= 1e-10
    assert np.max(np.abs(scan.D[0] - D)) <= 1e-12 * np.max(np.abs(D))


def test_against_bootstrap():
    """The windows' bootstrap copies: their cross-window correlations and spreads of a_0, E_0 are those of p.

    p is lsqfit's fit.p: the first-order propagation with the Gauss-Newton D = cov J^T W, which leaves out the
    residuals' curvature.  A bootstrap measures the whole response, so the two agree only where both are linear and
    the residuals vanish at the solution.  On the CPU oracle, one window fitted alone, copy by copy: with noisy central
    data its copies spread a_0 and E_0 by 0.94 to 1.19 times its own fit.p sdev at any size of the fluctuations
    (0.1 or 0.01 of the bootstrap's), and at their full size by 1.2 to 10 times (heavy tails from the prior-dominated
    excited states).  So the central data are the exact model values (zero residuals) and the copies are drawn at a
    tenth of the fluctuation; they are compared with a tenth of p's sdevs."""
    _need_gpu()
    fit, cfg = _fit(4, svdcut=1e-12, exact=True)
    scan = fit.window_fits(_ranges(cfg["ny"], cfg["np"]))
    S = scan.p[1]
    n, K, nw, scale = 10000, cfg["K"], scan.nwin, 0.1
    means = fit.bootstrap_means(n, 123)
    center = torch.as_tensor(fit._spec.mean).to(means.device)
    a = scan.bootstrapped_fits(means=center[None, :] + scale * (means - center[None, :])).arrays()
    ok = (a["status"] > 0).reshape(nw, n).all(axis=0)
    assert ok.mean() > 0.99
    idx = [0, K]                                        # a_0, E_0
    x = a["x"].reshape(nw, n, -1)[:, ok][:, :, idx]     # [nw, copies, 2]
    X = x.transpose(1, 0, 2).reshape(ok.sum(), -1)
    emp = np.cov(X, rowvar=False) / scale ** 2
    sub = S[:, idx][:, :, :, idx].reshape(2 * nw, 2 * nw)
    sd_e, sd_p = np.sqrt(np.diag(emp)), np.sqrt(np.diag(sub))
    assert np.max(np.abs(sd_e / sd_p - 1)) <= 0.05, sd_e / sd_p
    corr_e = emp / np.outer(sd_e, sd_e)
    corr_p = sub / np.outer(sd_p, sd_p)
    assert np.max(np.abs(corr_e - corr_p)) <= 0.05, np.max(np.abs(corr_e - corr_p))
    # the windows are strongly correlated, and the copies see it
    assert np.max(np.abs(corr_p - np.eye(2 * nw))) > 0.5


def test_correlated_average_of_windows():
    """lb.wavg of the ground state (a_0, E_0) of three windows with their joint block of p, against the numpy GLS
    average.  (All np parameters of several windows are not averaged: the prior-dominated excited states make that
    block of p singular, condition ~1e16 on the CPU oracle; the ground-state block's is ~1e6.)"""
    _need_gpu()
    import lsqfit_b200 as lb
    fit, cfg = _fit(4)
    scan = fit.window_fits(_ranges(cfg["ny"], cfg["np"]))
    ws, idx = [4, 6, 9], [0, cfg["K"]]
    m = len(idx)
    S = scan.p[1][ws][:, idx][:, :, ws][:, :, :, idx].reshape(len(ws) * m, len(ws) * m)
    y = scan.pmean[ws][:, idx]
    avg = lb.wavg(y, S, svdcut=None)
    X = np.tile(np.eye(m), (len(ws), 1))
    Si = np.linalg.inv(S)
    cov = np.linalg.inv(X.T @ Si @ X)
    mean = cov @ X.T @ Si @ y.reshape(-1)
    sd = np.sqrt(np.diag(cov))
    assert np.max(np.abs(avg.mean - mean) / sd) <= 1e-8
    assert np.max(np.abs(avg.cov - cov) / np.outer(sd, sd)) <= 1e-8


def test_abi_and_nothing_else_changes():
    _need_gpu()
    from lsqfit_b200 import _cabi
    fit, cfg = _fit(8)
    parent = fit.bootstrapped_fits(500, seed=4).arrays()
    scan = fit.window_fits(_ranges(cfg["ny"], cfg["np"]))
    keys = ("pmean", "psdev", "cov", "chi2", "dof", "Q", "logGBF", "svdn", "nit", "stopping_criterion")
    before = dict((k, np.array(getattr(scan, k), copy=True)) for k in keys)
    before_out = scan.out.numpy()
    bs0 = scan.bootstrapped_fits(300, seed=8).arrays()
    S = scan.p[1]
    assert scan.p[1] is S                               # computed once
    for k in keys:
        assert np.asarray(getattr(scan, k)).tobytes() == before[k].tobytes(), k
    for k, v in scan.out.numpy().items():
        assert v.tobytes() == before_out[k].tobytes(), k
    bs1 = scan.bootstrapped_fits(300, seed=8).arrays()
    for k in bs0:
        assert bs0[k].tobytes() == bs1[k].tobytes(), k
    after = fit.bootstrapped_fits(500, seed=4).arrays()
    for k in parent:
        assert parent[k].tobytes() == after[k].tobytes(), k
    # the C ABI
    lib, plan = _cabi.lib, scan.plan
    h = plan._h
    nw, npar, N = scan.nwin, scan.np, plan.N
    kw = dict(device=plan.tdev, dtype=torch.float64)
    cov = torch.as_tensor(scan.cov).to(plan.tdev)
    J = torch.zeros((nw, plan.nchiv, npar), **kw)
    C = torch.as_tensor(_input_cov(fit)).to(plan.tdev)
    D = torch.empty((nw, npar, N), **kw)
    covp = torch.empty((nw * npar, nw * npar), **kw)
    st = plan._stream()
    wp = lib.b200lm_window_propagate
    assert wp(None, cov.data_ptr(), J.data_ptr(), C.data_ptr(), None, D.data_ptr(), None, st) == _cabi.EINVAL
    assert "NULL handle" in _cabi.last_error()
    for args in ((None, J.data_ptr(), C.data_ptr(), None, D.data_ptr(), None),
                 (cov.data_ptr(), None, C.data_ptr(), None, D.data_ptr(), None),
                 (cov.data_ptr(), J.data_ptr(), C.data_ptr(), None, None, None)):
        assert wp(h, *args, st) == _cabi.EINVAL and "NULL required" in _cabi.last_error(h)
    assert wp(h, cov.data_ptr(), J.data_ptr(), None, None, D.data_ptr(), covp.data_ptr(), st) == _cabi.EINVAL
    assert "d_C" in _cabi.last_error(h)
    assert wp(h, cov.data_ptr(), J.data_ptr(), None, None, D.data_ptr(), None, st) == _cabi.OK
    torch.cuda.synchronize()
    # a plan without windows
    ph = fit._spec.plan()._h
    assert wp(ph, cov.data_ptr(), J.data_ptr(), C.data_ptr(), None, D.data_ptr(), None, st) == _cabi.EINVAL
    assert "no windows" in _cabi.last_error(ph)
    with pytest.raises(ValueError, match="windows"):
        fit._spec.plan().window_propagate(scan.cov, J, None)
    with pytest.raises(ValueError, match="dC must hold"):
        plan.window_propagate(scan.cov, J, None, np.zeros(plan._win_dC + 1))
    # the single-fit entries keep refusing windows
    p0 = torch.as_tensor(scan.pmean).to(plan.tdev).contiguous()
    mean = torch.as_tensor(fit._spec.mean).to(plan.tdev)
    f = torch.empty((1, plan.nchiv), **kw)
    assert lib.b200lm_residual_jacobian(h, 1, p0.data_ptr(), npar, mean.data_ptr(), 0, f.data_ptr(), None, None,
                                        st) == _cabi.EINVAL
    cv = torch.eye(npar, **kw)
    assert lib.b200lm_propagate(h, 1, p0.data_ptr(), cv.data_ptr(), None, D.data_ptr(), None, st) == _cabi.EINVAL
