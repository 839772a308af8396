"""Fit-window scans on the device: every window of a scan, and every bootstrap copy of it, gives the bits of a plan made
for that window alone (one warp per fit); the full-range window reproduces the parent's batch; the scan's fit attributes
agree with the oracle's fit of the window data."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

KEYS = ("x", "chi2", "cov", "logdet", "nit", "status")
NCOPY = 2000


def _need_gpu():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (no CPU fallback)")


def _data(K, ny=64, seed=3, corr=True):
    from lsqfit_b200 import configs
    cfg = configs.correlator(K, ny=ny)
    rng = np.random.default_rng(seed)
    L = np.linalg.cholesky(cfg["ycov"])
    y = cfg["f"] + L @ rng.standard_normal(ny)
    ycov = cfg["ycov"] if corr else np.sqrt(np.diag(cfg["ycov"]))
    return cfg, y, ycov


def _fit(K, svdcut=False, corr=True, fcn="multiexp", prior=None, **kw):
    import lsqfit_b200 as lb
    cfg, y, ycov = _data(K, corr=corr)
    prior = (cfg["prior_mean"], cfg["prior_sdev"]) if prior is None else prior
    return lb.nonlinear_fit(data=(cfg["x"], y, ycov), fcn=fcn, prior=prior, svdcut=svdcut, **kw), cfg


def _ranges(ny, npar, extra=()):
    r = [(0, ny), (0, npar), (ny - npar, ny), (1, 40), (3, 48), (5, 56), (8, ny), (10, 30), (0, 20), (16, ny),
         (30, ny), (2, ny - 1)] + list(extra)
    m = np.zeros((len(r), ny), dtype=bool)
    for w, (lo, hi) in enumerate(r):
        m[w, lo:hi] = True
    return m


def _same_bits(a, b, what, keys=KEYS):
    for k in keys:
        x, y = np.asarray(a[k]), np.asarray(b[k])
        assert x.dtype == y.dtype and x.shape == y.shape, (what, k, x.shape, y.shape)
        assert x.tobytes() == y.tobytes(), (what, k, np.max(np.abs(x.astype(float) - y.astype(float))))


def _standalone_check(fit, scan, ncopy, seed=11):
    """Every window of ``scan`` against a one-warp plan of the window alone: the whitening, the central fit and
    ``ncopy`` bootstrap copies give the same bits (f and J included; rows beyond the window's nchiv are zero)."""
    from lsqfit_b200.engine import Plan
    from lsqfit_b200.whiten import PDF
    from lsqfit_b200.windows import window_cov
    spec = fit._spec
    pdf = fit.yp_pdf
    cov = pdf.cov_in if pdf.cov_in is not None else pdf.sdev_in
    means = fit.bootstrap_means(ncopy, seed)
    tol = dict(tol=fit.tol, maxit=fit.maxit)
    nw = scan.nwin
    cen = scan.plan.fit_batch(spec.mean, scan.p0, B=nw, want_fJ=True, **tol).numpy()
    _same_bits(cen, dict(x=scan.pmean, chi2=scan.chi2, cov=scan.cov, logdet=scan.out.logdet.cpu().numpy(),
                         nit=scan.nit, status=scan.out.status.cpu().numpy()), "central twice")
    bs = scan.plan.fit_batch(means, scan.pmean, B=nw * ncopy, want_fJ=True, **tol).numpy()
    assert scan.plan.last_team() == 1
    nchiv = scan.plan.window_nchiv()
    assert list(nchiv) == list(scan.nchiv) and scan.plan.nchiv == max(nchiv)
    for w, m in enumerate(scan.masks):
        sel, c = window_cov(cov, spec.ny, m)
        alone = PDF(pdf.mean[sel], c, svdcut=pdf.svdcut, eps=pdf.eps)
        mine = scan.pdfs[w]
        assert alone.nmod == mine.nmod and alone.logdet == mine.logdet and alone.nchiv == nchiv[w] == mine.nchiv
        for (i0, w0), (i1, w1) in zip(alone.i_invwgts, mine.i_invwgts):
            assert np.array_equal(i0, i1) and np.asarray(w0).tobytes() == np.asarray(w1).tobytes(), w
        x = spec.functor.xrows(spec.x, spec.ny)[m]
        plan = Plan(spec.functor, spec.np, int(m.sum()), x, alone.i_invwgts, noprior=spec.noprior, team=1)
        n = nchiv[w]
        one = plan.fit_batch(pdf.mean[sel], scan.p0[w], want_fJ=True, **tol).numpy()
        ref = plan.fit_batch(means[:, torch.as_tensor(sel, device=means.device)], scan.pmean[w], want_fJ=True,
                             **tol).numpy()
        assert plan.last_team() == 1
        for got, exp, what, rows in ((cen, one, "central", slice(w, w + 1)),
                                     (bs, ref, "copies", slice(w * ncopy, (w + 1) * ncopy))):
            part = dict((k, got[k][rows]) for k in KEYS)
            part["f"], part["J"] = got["f"][rows][:, :n], got["J"][rows][:, :n]
            _same_bits(part, exp, (what, w), KEYS + ("f", "J"))
            assert not got["f"][rows][:, n:].any() and not got["J"][rows][:, n:].any(), (what, w)
        plan.close()
    return bs


@pytest.mark.parametrize("K", [4, 8])
def test_bits_against_standalone_plans(K):
    _need_gpu()
    fit, cfg = _fit(K)
    scan = fit.window_fits(_ranges(cfg["ny"], cfg["np"]))
    assert scan.nwin >= 12
    assert np.all(scan.stopping_criterion > 0), scan.stopping_criterion
    _standalone_check(fit, scan, NCOPY)


def test_full_range_equals_parent():
    """One window of all rows is the parent's own problem: its copies are the parent's batch.  They start from the
    window's central pmean (a refit from fit.pmean), so the parent's batch is run from that same start."""
    _need_gpu()
    for K in (4, 8):
        fit, cfg = _fit(K)
        scan = fit.window_fits(np.ones((1, cfg["ny"]), dtype=bool))
        # the refit may take the parent's point on by what its ftol test left (|d chi2| < 1e-10 chi2: ~1e-4 sdev)
        assert np.max(np.abs(scan.pmean[0] - fit.pmean) / fit.psdev) < 1e-3, (scan.pmean[0], fit.pmean, fit.psdev)
        assert abs(scan.chi2[0] - fit.chi2) <= 1e-8 * fit.chi2, (scan.chi2[0], fit.chi2)
        assert scan.dof[0] == fit.dof and scan.svdn[0] == fit.svdn and scan.pdfs[0].logdet == fit.yp_pdf.logdet
        bs = scan.bootstrapped_fits(500, seed=5)
        ref = fit._batch(fit.bootstrap_means(500, 5), scan.pmean[0], kernel=1)
        _same_bits(bs.window(0).arrays(), ref.arrays(), ("full range", K))
        # and with the parent's own start
        same = fit.window_fits(np.ones((1, cfg["ny"]), dtype=bool))
        out = same.plan.fit_batch(fit.bootstrap_means(500, 5), fit.pmean, tol=fit.tol, maxit=fit.maxit, B=500).numpy()
        _same_bits(out, fit.bootstrapped_fits(500, seed=5, kernel=1).arrays(), ("parent start", K))


def test_attributes_against_oracle():
    _need_gpu()
    from oracle.fit import nonlinear_fit as ofit
    fit, cfg = _fit(4)
    masks = _ranges(cfg["ny"], cfg["np"])[[0, 1, 3, 5, 9, 11]]
    scan = fit.window_fits(masks)
    _, y, ycov = _data(4)
    for w, m in enumerate(masks):
        fo = ofit("multiexp", cfg["x"][m], y[m], ycov[np.ix_(m, m)], prior_mean=cfg["prior_mean"],
                  prior_cov=np.diag(cfg["prior_sdev"] ** 2), p0=fit.pmean, svdcut=fit.svdcut, tol=fit.tol)
        v = scan[w]
        assert v.dof == fo.dof == scan.dof[w] and v.svdn == fo.svdn == scan.svdn[w], w
        assert abs(v.chi2 - fo.chi2) <= 1e-9 * fo.chi2, (w, v.chi2, fo.chi2)
        assert abs(v.Q - fo.Q) <= 1e-6 * max(fo.Q, 1e-3), (w, v.Q, fo.Q)
        assert abs(v.logGBF - fo.logGBF) <= 1e-8 * max(1.0, abs(fo.logGBF)), (w, v.logGBF, fo.logGBF)
        assert scan.logGBF[w] == v.logGBF and scan.Q[w] == v.Q
        # both solvers stop where their ftol test lets them (|d chi2| < 1e-10 chi2: ~1e-4 sdev from the minimum)
        assert np.max(np.abs(scan.pmean[w] - fo.pmean) / fo.psdev) < 1e-3, (w, scan.pmean[w], fo.pmean)


def test_other_shapes():
    _need_gpu()
    # uncorrelated data: 1x1 rows only
    fit, cfg = _fit(4, corr=False)
    scan = fit.window_fits(_ranges(cfg["ny"], cfg["np"])[:6])
    assert all(len(p.i_invwgts) == 1 for p in scan.pdfs)
    _standalone_check(fit, scan, 300)
    # svdcut < 0: modes dropped, nchiv differs by window, f / J padded with zeros
    fit, cfg = _fit(4, svdcut=-0.01)
    scan = fit.window_fits(_ranges(cfg["ny"], cfg["np"]))
    assert len(set(scan.nchiv)) > 3 and scan.svdn.max() > 0
    _standalone_check(fit, scan, 300)


def test_cuda_functor_plugin():
    _need_gpu()
    import lsqfit_b200 as lb
    uf = lb.cuda_functor("ut_window_exp", "return b[0] * exp(-b[1] * x[0]);", 2,
                         host=lambda x, p: p[0] * np.exp(-p[1] * np.asarray(x)[:, 0]))
    cfg, _, ycov = _data(1)
    fit = lb.nonlinear_fit(data=(cfg["x"], cfg["f"], ycov), fcn=uf, prior=(cfg["prior_mean"], cfg["prior_sdev"]))
    scan = fit.window_fits(_ranges(cfg["ny"], 2)[[0, 3, 7, 10]])
    _standalone_check(fit, scan, 300)


def test_refusals_and_kernel_choice():
    _need_gpu()
    import lsqfit_b200 as lb
    from lsqfit_b200 import _cabi
    fit, cfg = _fit(4)
    ny, npar = cfg["ny"], cfg["np"]
    masks = _ranges(ny, npar)[:4]
    for kw in (dict(bounds=(np.full(npar, -10.0), np.full(npar, 10.0))), dict(loss="huber"), dict(policy="gsl")):
        with pytest.raises(ValueError, match="not built for window scans"):
            fit.window_fits(masks, **kw)
    noisy, _ = _fit(4, noise=True, noise_seed=3)
    with pytest.raises(ValueError, match="not built for window scans"):
        noisy.window_fits(masks)
    for bad in (masks[:, :-1], masks.astype(int), np.zeros((2, ny), dtype=bool)):
        with pytest.raises(ValueError, match="not built for window scans"):
            fit.window_fits(bad)
    base = fit.window_fits(masks)
    bb = base.bootstrapped_fits(200, seed=9).arrays()
    for kernel in (4, "wave", 2):
        sc = fit.window_fits(masks, kernel=kernel)
        _same_bits(dict(x=sc.pmean, chi2=sc.chi2, cov=sc.cov, logdet=sc.out.logdet.cpu().numpy(), nit=sc.nit,
                        status=sc.out.status.cpu().numpy()),
                   dict(x=base.pmean, chi2=base.chi2, cov=base.cov, logdet=base.out.logdet.cpu().numpy(),
                        nit=base.nit, status=base.out.status.cpu().numpy()), ("kernel", kernel))
        _same_bits(sc.bootstrapped_fits(200, seed=9).arrays(), bb, ("kernel copies", kernel))
        assert sc.plan.last_team() == 1
    # the C ABI
    plan, lib = base.plan, _cabi.lib
    h = plan._h
    nw = base.nwin
    kw = dict(device=plan.tdev, dtype=torch.float64)
    B = 3 * nw + 1
    mean = torch.as_tensor(fit._spec.mean).to(plan.tdev)
    p0 = torch.as_tensor(base.pmean).to(plan.tdev).contiguous()
    x, chi2, ld = torch.empty((B, npar), **kw), torch.empty(B, **kw), torch.empty(B, **kw)
    it = torch.empty(2 * B, device=plan.tdev, dtype=torch.int32)

    def fb(B):
        return lib.b200lm_fit_batch(h, B, mean.data_ptr(), 0, p0.data_ptr(), npar, 1e-8, 1e-10, 1e-10, 1000, 1, 0,
                                    x.data_ptr(), chi2.data_ptr(), None, ld.data_ptr(), it.data_ptr(),
                                    it[B:].data_ptr(), None, None, plan._stream())
    assert fb(B) == _cabi.EINVAL and "multiple" in _cabi.last_error(h)
    assert fb(3 * nw) == _cabi.OK
    torch.cuda.synchronize()
    _cabi.check(lib.b200lm_set_policy(h, 1), h)
    assert fb(nw) == _cabi.EINVAL
    _cabi.check(lib.b200lm_set_policy(h, 0), h)
    lb_, ub_ = np.full(npar, -10.0), np.full(npar, 10.0)
    _cabi.check(lib.b200lm_set_bounds(h, lb_.ctypes.data, ub_.ctypes.data), h)
    assert fb(nw) == _cabi.EINVAL
    _cabi.check(lib.b200lm_set_bounds(h, None, None), h)
    f = torch.empty((1, plan.nchiv), **kw)
    assert lib.b200lm_residual_jacobian(h, 1, p0.data_ptr(), npar, mean.data_ptr(), 0, f.data_ptr(), None, None,
                                        plan._stream()) == _cabi.EINVAL
    D = torch.empty((1, npar, plan.N), **kw)
    cv = torch.eye(npar, **kw)
    assert lib.b200lm_propagate(h, 1, p0.data_ptr(), cv.data_ptr(), None, D.data_ptr(), None,
                                plan._stream()) == _cabi.EINVAL
    # malformed descriptions: the error names the window
    from lsqfit_b200.windows import window_weights
    good = window_weights(base.sels, [p.i_invwgts for p in base.pdfs])

    def bad_desc(edit):
        d = dict((k, np.array(v, copy=True)) for k, v in good.items())
        edit(d)
        with pytest.raises(_cabi.B200LMError) as e:
            plan.set_windows(d)
        assert e.value.code == _cabi.EINVAL
        return str(e.value)
    nd0 = good["ndiag"][0]
    assert "window 0" in bad_desc(lambda d: d["blk_idx"].__setitem__(0, ny + npar))          # out of range
    assert "window 0" in bad_desc(lambda d: d["blk_idx"].__setitem__(1, d["blk_idx"][0]))   # repeated
    assert "window 1" in bad_desc(lambda d: d["blk_idx"].__setitem__(
        d["blk_nin"][0] + 1, d["diag_idx"][0] if nd0 else d["blk_idx"][0]))             # a row of window 0 elsewhere
    assert "window" in bad_desc(lambda d: d["diag_idx"].__setitem__(nd0 - 1, ny - 1) if nd0 else
                                d["blk_idx"].__setitem__(0, -1))

    def two_blocks(d):          # window 0's first block split in two, its last row also listed in the second part
        n0 = int(d["blk_nin"][0])
        idx = d["blk_idx"]
        d["nblk"][0] += 1
        d["blk_nin"] = np.insert(d["blk_nin"], 1, 1)
        d["blk_nout"] = np.insert(d["blk_nout"], 1, 1)
        d["blk_idx"] = np.insert(idx, n0, idx[n0 - 1])
        d["blk_w"] = np.insert(d["blk_w"], int(d["blk_nin"][0] * d["blk_nout"][0]), 1.0)
    assert "window 0" in bad_desc(two_blocks)
    # set_weights switches back: the plan's original bits
    means = fit.bootstrap_means(300, 21)
    plan.set_weights(fit._spec.i_invwgts)
    assert plan.nwin == 0 and plan.nchiv == fit._spec.plan().nchiv
    plan.set_team(1)
    fit._spec.plan().set_team(1)
    try:
        a = plan.fit_batch(means, fit.pmean, tol=fit.tol).numpy()
        b = fit._spec.plan().fit_batch(means, fit.pmean, tol=fit.tol).numpy()
    finally:
        fit._spec.plan().set_team(0)
    _same_bits(a, b, "set_weights after set_windows")


def test_host_entry_with_windows():
    """fit_batch_host with windows set fits nwin x copies (means [copies, N], p0 [nwin, np]), with the bits of
    fit_batch, whether or not the number of copies equals the number of windows."""
    _need_gpu()
    fit, cfg = _fit(4)
    scan = fit.window_fits(_ranges(cfg["ny"], cfg["np"])[:6])
    for ncopy in (50, scan.nwin):
        means = fit.bootstrap_means(ncopy, 17)
        dev = scan.plan.fit_batch(means, scan.pmean, tol=fit.tol, maxit=fit.maxit).numpy()
        host = scan.plan.fit_batch_host(means.cpu().numpy(), scan.pmean, tol=fit.tol, maxit=fit.maxit)
        assert host["x"].shape == (scan.nwin * ncopy, cfg["np"])
        _same_bits(host, dev, ("host entry", ncopy))


def test_parent_plan_untouched():
    _need_gpu()
    fit, cfg = _fit(8)
    a = fit.bootstrapped_fits(1000, seed=4).arrays()
    scan = fit.window_fits(_ranges(cfg["ny"], cfg["np"]))
    scan.bootstrapped_fits(100, seed=4)
    b = fit.bootstrapped_fits(1000, seed=4).arrays()
    _same_bits(a, b, "parent before / after a scan")
    bs = scan.bootstrapped_fits(100, seed=4)
    w = bs.window(3)
    assert len(w) == 100 and len(bs) == 100 * scan.nwin
    views = list(w)
    assert views[0].dof == scan.dof[3] and views[0].svdn == scan.svdn[3]
    m, c = w.pmean_stats()
    assert m.shape == (cfg["np"],) and c.shape == (cfg["np"], cfg["np"])
