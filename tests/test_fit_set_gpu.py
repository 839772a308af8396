"""Fit sets on the device: every problem of a set, and every bootstrap copy of it, gives the bits of a plan made for
that problem alone (one warp per fit); the set's fit attributes agree with the oracle's fit of each problem; the C ABI
refuses what a set plan is not built for."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

KEYS = ("x", "chi2", "cov", "logdet", "nit", "status")
NCOPY = 2000


def _need_gpu():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (no CPU fallback)")


def _problems(nexp, nprob, corr_prior=False, seed=3, sdev_every=0):
    """nprob problems of an nexp-exponential model: ny 24 ... 64 and an x grid of its own each, correlated data (a
    vector of standard deviations for every sdev_every-th problem), priors scaled per problem (correlated ones with
    corr_prior)."""
    from lsqfit_b200 import configs
    rng = np.random.default_rng(seed)
    data, priors = [], []
    for k in range(nprob):
        ny = int(rng.integers(24, 65))
        cfg = configs.correlator(nexp, ny=ny, dt=0.1 + 0.005 * k)
        y = cfg["f"] + np.linalg.cholesky(cfg["ycov"]) @ rng.standard_normal(ny)
        ycov = np.sqrt(np.diag(cfg["ycov"])) if sdev_every and k % sdev_every == 0 else cfg["ycov"]
        psd = cfg["prior_sdev"] * (1 + 0.05 * k)
        if corr_prior:
            n = psd.size
            pc = 0.4 ** np.abs(np.subtract.outer(np.arange(n), np.arange(n)))
            prior = (cfg["prior_mean"], psd[:, None] * psd[None, :] * pc)
        else:
            prior = (cfg["prior_mean"], psd)
        data.append((cfg["x"], y, ycov))
        priors.append(prior)
    return data, priors


def _same_bits(a, b, what, keys=KEYS):
    for k in keys:
        x, y = np.asarray(a[k]), np.asarray(b[k])
        assert x.dtype == y.dtype and x.shape == y.shape, (what, k, x.shape, y.shape)
        assert x.tobytes() == y.tobytes(), (what, k, np.max(np.abs(x.astype(float) - y.astype(float))))


def _alone_check(fs, ncopy, seed=11):
    """Every problem of ``fs`` against a one-warp plan of the problem alone: the whitening, the central fit and
    ``ncopy`` bootstrap copies (each problem's own stream) give the same bits, f and J included."""
    from lsqfit_b200.bootstrap import bootstrap_means
    from lsqfit_b200.engine import Plan
    from lsqfit_b200.whiten import PDF
    d = fs.description
    tol = dict(tol=fs.tol, maxit=fs.maxit)
    K = fs.K
    cen = fs.plan.fit_batch(fs._mean, fs.p0, B=K, want_fJ=True, **tol).numpy()
    _same_bits(cen, dict(x=fs.pmean, chi2=fs.chi2, cov=fs.cov, logdet=fs.out.logdet.cpu().numpy(), nit=fs.nit,
                         status=fs.out.status.cpu().numpy()), "central twice")
    means = fs.bootstrap_means(ncopy, seed)
    assert len(fs.seeds) == K
    assert fs.seeds == [int(s) for s in np.random.SeedSequence(seed).generate_state(K, np.uint64)]
    bs = fs.plan.fit_batch(means, fs.pmean, B=K * ncopy, want_fJ=True, **tol).numpy()
    assert fs.plan.last_team() == 1
    nchiv = fs.plan.window_nchiv()
    assert list(nchiv) == list(fs.nchiv) and fs.plan.nchiv == max(nchiv)
    bsf = fs.bootstrapped_fits(ncopy, seed=seed)
    for k in range(K):
        alone = PDF(d["means"][k], d["covs"][k], svdcut=fs.svdcut, eps=fs.eps)
        mine = fs.pdfs[k]
        assert alone.nmod == mine.nmod and alone.logdet == mine.logdet and alone.nchiv == nchiv[k] == mine.nchiv
        for (i0, w0), (i1, w1) in zip(alone.i_invwgts, mine.i_invwgts):
            assert np.array_equal(i0, i1) and np.asarray(w0).tobytes() == np.asarray(w1).tobytes(), k
        # the problem's columns of the stacked copies are its own bootstrap stream, bit for bit
        own = bootstrap_means(alone.mean, alone.sqrt_cov(), ncopy, fs.seeds[k])
        sel = torch.as_tensor(fs.sels[k], device=means.device)
        assert torch.equal(means[:, sel], own), k
        nyk = int(d["nys"][k])
        o = int(d["row_off"][k])
        plan = Plan(fs.fcn, fs.np, nyk, d["x"][o:o + nyk], alone.i_invwgts, noprior=fs.noprior, team=1)
        n = nchiv[k]
        one = plan.fit_batch(alone.mean, fs.p0[k], want_fJ=True, **tol).numpy()
        ref = plan.fit_batch(own, fs.pmean[k], want_fJ=True, **tol).numpy()
        assert plan.last_team() == 1
        for got, exp, what, rows in ((cen, one, "central", slice(k, k + 1)),
                                     (bs, ref, "copies", slice(k * ncopy, (k + 1) * ncopy))):
            part = dict((key, got[key][rows]) for key in KEYS)
            part["f"], part["J"] = got["f"][rows][:, :n], got["J"][rows][:, :n]
            _same_bits(part, exp, (what, k), KEYS + ("f", "J"))
            assert not got["f"][rows][:, n:].any() and not got["J"][rows][:, n:].any(), (what, k)
        _same_bits(bsf.problem(k).arrays(), ref, ("bootstrapped_fits", k))
        plan.close()
    assert len(bsf) == K * ncopy


@pytest.mark.parametrize("svdcut", [1e-8, 0.05, -0.01])
@pytest.mark.parametrize("corr_prior", [False, True])
@pytest.mark.parametrize("nexp", [4, 8])
def test_bits_against_problems_alone(nexp, corr_prior, svdcut):
    _need_gpu()
    import lsqfit_b200 as lb
    data, priors = _problems(nexp, 6, corr_prior, sdev_every=4)
    fs = lb.fit_set(data, priors, fcn="multiexp", svdcut=svdcut)
    assert fs.K == 6 and len(set(fs.description["nys"])) > 2
    assert np.all(fs.stopping_criterion > 0), fs.stopping_criterion
    if svdcut == 0.05:
        assert fs.svdn.max() > 0
    _alone_check(fs, NCOPY)


def test_attributes_against_oracle():
    _need_gpu()
    import lsqfit_b200 as lb
    from oracle.fit import nonlinear_fit as ofit
    data, priors = _problems(4, 4, corr_prior=True)
    fs = lb.fit_set(data, priors, fcn="multiexp", svdcut=0.05)
    assert len(fs) == 4
    for k, ((x, y, ycov), (pm, pc)) in enumerate(zip(data, priors)):
        fo = ofit("multiexp", x, y, ycov, prior_mean=pm, prior_cov=pc, p0=fs.p0[k], svdcut=fs.svdcut, tol=fs.tol)
        v = fs[k]
        assert v.dof == fo.dof == fs.dof[k] and v.svdn == fo.svdn == fs.svdn[k], k
        assert abs(v.chi2 - fo.chi2) <= 1e-9 * fo.chi2, (k, v.chi2, fo.chi2)
        assert abs(v.Q - fo.Q) <= 1e-6 * max(fo.Q, 1e-3), (k, v.Q, fo.Q)
        assert abs(v.logGBF - fo.logGBF) <= 1e-8 * max(1.0, abs(fo.logGBF)), (k, v.logGBF, fo.logGBF)
        assert fs.logGBF[k] == v.logGBF and fs.Q[k] == v.Q
        assert np.max(np.abs(fs.pmean[k] - fo.pmean) / fo.psdev) < 1e-3, (k, fs.pmean[k], fo.pmean)
    # and against nonlinear_fit of each problem (the same whitening and the same start)
    for k in (0, 3):
        f = lb.nonlinear_fit(data=data[k], prior=priors[k], fcn="multiexp", svdcut=0.05)
        assert np.array_equal(f.p0, fs.p0[k]) and f.dof == fs.dof[k] and f.svdn == fs.svdn[k]
        assert f.yp_pdf.logdet == fs.pdfs[k].logdet
        assert abs(f.chi2 - fs.chi2[k]) <= 1e-9 * f.chi2


def test_no_prior_shared_prior_and_plugin():
    _need_gpu()
    import lsqfit_b200 as lb
    from lsqfit_b200 import configs
    # no prior: p0 required, N = ny
    data, _ = _problems(2, 5, sdev_every=2)
    fs = lb.fit_set([(x, y, c) for x, y, c in data], None, fcn="multiexp", p0=configs.correlator(2)["ptrue"])
    assert fs.noprior and fs.plan.N == fs.ny and fs.logGBF is None and fs[0].logGBF is None
    _alone_check(fs, 300)
    # one prior shared by every problem
    data, priors = _problems(4, 5)
    fs = lb.fit_set(data, priors[0], fcn="multiexp")
    assert all(np.array_equal(m, priors[0][0]) for m, _ in fs.prior)
    _alone_check(fs, 300)
    # a cuda_functor plug-in
    uf = lb.cuda_functor("ut_set_exp", "return b[0] * exp(-b[1] * x[0]);", 2,
                         host=lambda x, p: p[0] * np.exp(-p[1] * np.asarray(x)[:, 0]))
    data = []
    for k in range(4):
        cfg = configs.correlator(1, ny=30 + 8 * k, dt=0.1 + 0.01 * k)
        data.append((cfg["x"], cfg["f"] * (1 + 0.001 * k), cfg["ycov"]))
    fs = lb.fit_set(data, (cfg["prior_mean"], cfg["prior_sdev"]), fcn=uf, kernel=4)
    _alone_check(fs, 300)


def test_host_entry_on_set_plan():
    _need_gpu()
    import lsqfit_b200 as lb
    data, priors = _problems(4, 5)
    fs = lb.fit_set(data, priors, fcn="multiexp")
    for ncopy in (40, fs.K):
        means = fs.bootstrap_means(ncopy, 17)
        dev = fs.plan.fit_batch(means, fs.pmean, tol=fs.tol, maxit=fs.maxit).numpy()
        host = fs.plan.fit_batch_host(means.cpu().numpy(), fs.pmean, tol=fs.tol, maxit=fs.maxit)
        assert host["x"].shape == (fs.K * ncopy, fs.np)
        _same_bits(host, dev, ("host entry", ncopy))


def test_refusals():
    _need_gpu()
    import ctypes as C
    import lsqfit_b200 as lb
    from lsqfit_b200 import _cabi
    from lsqfit_b200.engine import Plan
    from lsqfit_b200.windows import window_weights
    data, priors = _problems(4, 3)
    npar = 8
    for kw in (dict(bounds=(np.full(npar, -10.0), np.full(npar, 10.0))), dict(loss="huber"), dict(policy="gsl"),
               dict(noise=True), dict(yp_cov=np.eye(3))):
        with pytest.raises(ValueError, match="not built for fit sets"):
            lb.fit_set(data, priors, fcn="multiexp", **kw)
    with pytest.raises(ValueError, match="not built for fit sets"):
        lb.fit_set(data, [priors[0], None, priors[2]], fcn="multiexp")
    with pytest.raises(ValueError, match="not built for fit sets"):
        lb.fit_set([], priors, fcn="multiexp")
    with pytest.raises(ValueError, match="not built for fit sets"):
        lb.fit_set(data, [priors[0], priors[1], (np.ones(6), np.ones(6))], fcn="multiexp")
    with pytest.raises(ValueError, match="not built for fit sets"):
        lb.fit_set([(np.arange(5.0), np.ones(5), np.ones(5))], (np.ones(9), np.ones(9)), fcn="xerr_logistic")
    fs = lb.fit_set(data, priors, fcn="multiexp")
    lib, plan = _cabi.lib, fs.plan
    h = plan._h
    fam = plan.functor.family
    # b200lm_create_set argument errors
    out = _cabi.handle_t()
    for args in ((fam, 10, npar, 1, 0, 0), (fam, 0, npar, 1, 2, 0), (fam, 10, 0, 1, 2, 0), (fam, 10, npar, 2, 2, 0),
                 (fam, 10, npar, 1, 2 ** 30, 0)):
        assert lib.b200lm_create_set(*args[:4], args[4], args[5], 0, C.byref(out)) == _cabi.EINVAL, args
    assert lib.b200lm_create_set(fam, 10, 7, 1, 2, 0, 0, C.byref(out)) == _cabi.ENOFUNCTOR
    # set_weights on a set plan; fit_batch before set_windows
    with pytest.raises(_cabi.B200LMError) as e:
        plan.set_weights(fs.pdfs[0].i_invwgts)
    assert e.value.code == _cabi.EINVAL and "fit sets" in str(e.value)
    fresh = Plan(fs.fcn, npar, fs.ny, fs.description["x"], None, nslot=fs.K)
    with pytest.raises(_cabi.B200LMError) as e:
        fresh.fit_batch(fs._mean, fs.p0[0], B=1)
    assert e.value.code == _cabi.EINVAL and "b200lm_set_windows" in str(e.value)
    fresh.close()
    # windows over two slots, part of a slot, or another problem's slot entry: the error names the window
    good = window_weights(fs.sels, [p.i_invwgts for p in fs.pdfs])
    ny = fs.ny

    def bad_desc(edit):
        d = dict((k, np.array(v, copy=True)) for k, v in good.items())
        edit(d)
        with pytest.raises(_cabi.B200LMError) as e:
            plan.set_windows(d)
        assert e.value.code == _cabi.EINVAL
        return str(e.value)
    # window 0's prior entries are 1x1 rows (diagonal prior): the last diag entries
    nd0 = int(good["ndiag"][0])
    assert good["diag_idx"][nd0 - 1] == ny + npar - 1
    # one entry of slot 0 replaced by an entry of slot 2: two slots
    msg = bad_desc(lambda d: d["diag_idx"].__setitem__(nd0 - 1, ny + 2 * npar + npar - 1))
    assert "window 0" in msg and "two prior slots" in msg, msg
    # part of a slot: window 0 drops its last prior row

    def drop_last(d):
        d["ndiag"][0] -= 1
        d["diag_idx"] = np.delete(d["diag_idx"], nd0 - 1)
        d["diag_w"] = np.delete(d["diag_w"], nd0 - 1)
    msg = bad_desc(drop_last)
    assert "window 0" in msg and "part of a prior slot" in msg, msg
    # window 1 lists window 0's slot entry instead of its own
    nd1 = int(good["ndiag"][1])
    msg = bad_desc(lambda d: d["diag_idx"].__setitem__(nd0 + nd1 - 1, ny + npar - 1))
    assert "window 1" in msg, msg
    # propagate, residual_jacobian and window_propagate
    kw = dict(device=plan.tdev, dtype=torch.float64)
    p0 = torch.as_tensor(fs.pmean).to(plan.tdev).contiguous()
    mean = torch.as_tensor(fs._mean).to(plan.tdev)
    f = torch.empty((1, plan.nchiv), **kw)
    assert lib.b200lm_residual_jacobian(h, 1, p0.data_ptr(), npar, mean.data_ptr(), 0, f.data_ptr(), None, None,
                                        plan._stream()) == _cabi.EINVAL
    D = torch.empty((fs.K, npar, plan.N), **kw)
    cv = torch.eye(npar, **kw).repeat(fs.K, 1, 1).contiguous()
    assert lib.b200lm_propagate(h, 1, p0.data_ptr(), cv.data_ptr(), None, D.data_ptr(), None,
                                plan._stream()) == _cabi.EINVAL
    J = torch.zeros((fs.K, plan.nchiv, npar), **kw)
    assert lib.b200lm_window_propagate(h, cv.data_ptr(), J.data_ptr(), None, None, D.data_ptr(), None,
                                       plan._stream()) == _cabi.EINVAL
    assert "fit sets" in _cabi.last_error(h)
    # the set still fits after the refusals
    again = plan.fit_batch(fs._mean, fs.p0, B=fs.K, tol=fs.tol, maxit=fs.maxit).numpy()
    _same_bits(again, dict(x=fs.pmean, chi2=fs.chi2, cov=fs.cov, logdet=fs.out.logdet.cpu().numpy(), nit=fs.nit,
                           status=fs.out.status.cpu().numpy()), "after refusals")
