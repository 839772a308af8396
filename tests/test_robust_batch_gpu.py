"""Batched robust fits (scipy's ``loss`` / ``f_scale``, ``lsqfit.scipy_least_squares(loss=...)``, reference
src/lsqfit/_scipy.py:77): the one-warp kernel's robust driver (csrc/lm_kernel.cuh: fit_one<F, 6>; numpy model
tests/lm_model_robust.py, checked on the CPU by test_robust_model_cpu.py), the C ABI's b200lm_set_loss,
Plan.fit_batch's ``loss`` / ``f_scale`` and the batch drivers of nonlinear_fit / MultiFitter, against scipy's robust
trf through the oracle (a process pool on the host cores).  Needs a GPU (pytest -m gpu).
"""
import ctypes as C

import numpy as np
import pytest

import lm_model_robust as M
from parity_util import _W, correlator_problem, rel_cov

pytestmark = pytest.mark.gpu

TOL = (1e-10, 1e-10, 1e-10)
LOSSES = ("huber", "soft_l1", "cauchy", "arctan")
KEYS = ("x", "chi2", "cov", "logdet", "nit", "status")


def _need_gpu():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (no CPU fallback)")


# ---- oracle workers (spawned pool: module-level functions) ------------------------------------------------------
def _corr_init(K):
    import os
    import warnings
    os.environ["OPENBLAS_NUM_THREADS"] = "1"
    warnings.simplefilter("ignore")
    _W["cfg"], _W["pdf"] = correlator_problem(K)


def _result(fo):
    res = getattr(fo.fitter_results, "results", fo.fitter_results)
    return dict(x=fo.pmean, sd=fo.psdev, cov=fo.cov, chi2=fo.chi2, cost=float(res.cost), ok=fo.stopping_criterion > 0,
                logGBF=fo.logGBF, c=-fo.yp_pdf.logdet - fo.dof * np.log(2.0 * np.pi))


def _corr_job(arg):
    from oracle.fit import nonlinear_fit
    mean, p0, loss, fs = arg
    cfg, pdf = _W["cfg"], _W["pdf"]
    ny = cfg["ny"]
    fo = nonlinear_fit("multiexp", cfg["x"], mean[:ny], prior_mean=mean[ny:], _yp_pdf=pdf, p0=p0, tol=TOL,
                       maxit=1000, x_scale="jac", loss=loss, f_scale=fs)
    return _result(fo)


def _nist_init():
    import json
    import os
    import warnings
    os.environ["OPENBLAS_NUM_THREADS"] = "1"
    warnings.simplefilter("ignore")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with open(os.path.join(root, "tests", "golden", "nist.json")) as f:
        _W["nist"] = json.load(f)["problems"]


def _nist_job(arg):
    from oracle.fit import nonlinear_fit
    k, y, loss, fs = arg
    pr = _W["nist"][k]
    x = np.array(pr["x"])
    fo = nonlinear_fit(pr["form"], x, y, pr["ysdev"], prior_mean=pr["prior_mean"], prior_cov=pr["prior_sdev"],
                       p0=pr["p0"], tol=TOL, maxit=1000, x_scale="jac", loss=loss, f_scale=fs)
    return _result(fo)


def _pool(init, initargs, job, jobs):
    import multiprocessing as mp
    import os
    nproc = min(os.cpu_count() or 1, 32)
    with mp.get_context("spawn").Pool(nproc, initializer=init, initargs=initargs) as pool:
        return pool.map(job, jobs, chunksize=max(1, len(jobs) // (nproc * 8)))


# ---- problems ---------------------------------------------------------------------------------------------------
def _corr(K, B, seed, outliers):
    """Plan and B bootstrap copies of the K-exponential correlator (one 64 x 64 data block + 1x1 prior rows); with
    ``outliers``, 3 % of the copies get one data point moved by 30 sigma (the copies' means)."""
    import lsqfit_b200 as lb
    from lsqfit_b200 import configs
    cfg, opdf = correlator_problem(K)
    ny = cfg["ny"]
    means = configs.bootstrap_means(cfg, B, seed, cov=opdf.cov[:ny, :ny], vary_prior=False)
    if outliers:
        rng = np.random.default_rng(seed)
        rows = rng.choice(B, size=max(1, B * 3 // 100), replace=False)
        pts = rng.integers(0, ny, size=rows.size)
        means[rows, pts] += 30.0 * np.sqrt(np.diag(cfg["ycov"]))[pts] * rng.choice([-1.0, 1.0], size=rows.size)
    plan = lb.Plan("multiexp", cfg["np"], ny, cfg["x"], opdf.i_invwgts)
    return cfg, opdf, plan, means


def _robust_cost(f, loss, fs):
    return 0.5 * np.sum(M.robust_row(loss, fs, f)[0], axis=-1)


# cauchy and arctan are not convex in the residual: from the same start, two solvers whose sub-problem solutions differ
# in rounding (the kernel's Cholesky secular equation, scipy's SVD) can take different steps where the cost surface
# folds, and end in different local minima.  tests/lm_model_robust.py, the kernel's decisions in numpy, ends in the
# same minimum as the kernel on the copies checked (C4 copy 119 with arctan, f_scale 1: both 5.8 % above scipy's robust
# cost, 3.2 sdev away; misra1a copies with cauchy, f_scale 1: the largest splits, 16.2 and 14.8 sdev, to the last digit
# printed; on some split copies the kernel's minimum is the lower one, on others scipy's).  Such copies are counted, not
# compared; huber and soft_l1 (convex in the residual) may have none.  Measured on a B200 (200 copies each), f_scale 1:
# arctan 3 (C3-like), 1 (C4), 19 (misra1a), cauchy 0, 0, 7; f_scale 3: arctan 0, 0, 1, cauchy none.
SPLIT_SHARE = dict(huber=0.0, soft_l1=0.0, cauchy=0.05, arctan=0.12)


def _check(dev, orc, loss, fs, xbar, covbar, tag):
    """the bars of test_robust_loss, copy by copy, on the copies that end in scipy's minimum; returns the worst
    deviations and the number of copies in another minimum"""
    ok_d = dev["status"] > 0
    ok_o = np.array([o["ok"] for o in orc])
    assert np.mean(ok_d == ok_o) >= 0.999, tag
    worst = dict(cost=0.0, x=0.0, chi2=0.0, cov=0.0, lgbf=0.0)
    split = 0
    for b, o in enumerate(orc):
        if not (ok_d[b] and o["ok"]):
            continue
        cost = _robust_cost(dev["f"][b], loss, fs)
        if abs(cost - o["cost"]) > 1e-6 * o["cost"] or np.max(np.abs(dev["x"][b] - o["x"]) / o["sd"]) > 0.05:
            split += 1
            continue
        lgbf = 0.5 * (o["c"] - dev["logdet"][b] - dev["chi2"][b])
        w = dict(cost=abs(cost - o["cost"]) / o["cost"], x=np.max(np.abs(dev["x"][b] - o["x"]) / o["sd"]),
                 chi2=abs(dev["chi2"][b] - o["chi2"]) / o["chi2"], cov=rel_cov(dev["cov"][b], o["cov"]),
                 lgbf=abs(lgbf - o["logGBF"]) / max(1.0, abs(o["logGBF"])))
        for k in worst:
            worst[k] = max(worst[k], w[k])
    print("robust parity", tag, "copies in another minimum:", split, "worst:", worst)
    # arctan at f_scale 1 leaves most rows beyond the knee (clipped): the robust cost is so flat that both solvers stop,
    # each on its own tolerance, where the chi2 of the TRUE residuals (first order in the distance, unlike the cost)
    # still differs by up to 9.4e-5 (logGBF 1.4e-4, C4 shape); every other case stays below 2.6e-6
    flat = 3e-4 if (loss == "arctan" and fs < 2.0) else 1e-5
    assert worst["cost"] < 1e-9 and worst["x"] < xbar and worst["chi2"] < flat, (tag, worst)
    assert worst["cov"] < covbar and worst["lgbf"] < flat, (tag, worst)
    assert split <= SPLIT_SHARE[loss] * len(orc), (tag, split)
    return worst, split


def _vs_scipy(dev_fit, init, initargs, job, args, xbar, covbar):
    """every loss, f_scale 1 and 3: the device batch against the oracle copy by copy (one pool for all of them)"""
    cases = [(loss, fs) for loss in LOSSES for fs in (1.0, 3.0)]
    orc = _pool(init, initargs, job, [a + c for c in cases for a in args])
    n = len(args)
    for i, (loss, fs) in enumerate(cases):
        _check(dev_fit(loss, fs), orc[i * n:(i + 1) * n], loss, fs, xbar, covbar, (initargs, loss, fs))


@pytest.mark.parametrize("K,outliers,xbar,covbar", [(8, True, 1e-3, 1e-3), (3, False, 1e-4, 1e-4)])
def test_correlator_copies_vs_scipy(K, outliers, xbar, covbar):
    """200 bootstrap copies of the C3-like correlator (8 exponentials, one 64 x 64 data block, outliers in 3 % of the
    copies) and of the C4 shape (3 exponentials), every loss, f_scale 1 and 3, against scipy's robust trf copy by
    copy.  Measured on a B200, copies in scipy's minimum: robust cost within 1.1e-10 relative, x within 8.0e-4 sdev
    (C3-like, huber at f_scale 3) and 1.7e-5 (C4), chi2 within 2.6e-6 (arctan at f_scale 1: 9.4e-5, see _check), cov
    within 7.9e-4 and 9.0e-5, logGBF within 1.4e-4 (arctan at f_scale 1) and 1.3e-6 otherwise."""
    _need_gpu()
    cfg, opdf, plan, means = _corr(K, 200, 97 + K, outliers)
    p0 = cfg["prior_mean"] if K == 8 else cfg["ptrue"]
    _vs_scipy(lambda loss, fs: plan.fit_batch(means, p0, tol=TOL, loss=loss, f_scale=fs, want_fJ=True).numpy(),
              _corr_init, (K,), _corr_job, [(m, p0) for m in means], xbar, covbar)


def test_nist_copies_vs_scipy(nist_problems):
    """A NIST problem with 1x1 data rows (misra1a, three planted outliers) in 200 copies of its data, every loss, two
    f_scale values, against scipy's robust trf copy by copy.  Measured on a B200, copies in scipy's minimum: robust
    cost within 5e-14, x within 3.4e-5 sdev, chi2 within 3.5e-6, cov within 2.5e-5, logGBF within 3.5e-6."""
    _need_gpu()
    import lsqfit_b200 as lb
    k = next(i for i, q in enumerate(nist_problems) if q["name"] == "misra1a")
    pr = nist_problems[k]
    y0, sd = np.array(pr["y"], dtype=float), np.array(pr["ysdev"], dtype=float) * np.ones(len(pr["y"]))
    for j, i in enumerate((1, len(y0) // 2, len(y0) - 2)):
        y0[i] += (12.0 + 5.0 * j) * sd[i] * (-1) ** j
    ys = y0 + 0.5 * sd * np.random.default_rng(5).standard_normal((200, y0.size))
    # (a functor named by string: device parameter order is the fit's own)
    fit = lb.nonlinear_fit(data=(np.array(pr["x"]), y0, pr["ysdev"]), fcn=pr["form"],
                           prior=(pr["prior_mean"], pr["prior_sdev"]), p0=pr["p0"], tol=TOL)
    plan = fit._spec.plan(fit.device)
    means = np.concatenate([ys, np.broadcast_to(pr["prior_mean"], (200, len(pr["p0"])))], axis=1)
    p0 = np.array(pr["p0"], dtype=float)
    _vs_scipy(lambda loss, fs: plan.fit_batch(means, p0, tol=TOL, loss=loss, f_scale=fs, want_fJ=True).numpy(),
              _nist_init, (), _nist_job, [(k, y) for y in ys], 1e-4, 1e-4)


def _c3_fit(**kw):
    """the C3-like correlator with one outlier in its data, fitted with soft_l1 on the single-fit path"""
    import lsqfit_b200 as lb
    cfg, _ = correlator_problem(8)
    ymean = cfg["f"] * (1.0 + 1e-4 * np.sin(np.arange(cfg["ny"])))
    ymean[7] += 25.0 * np.sqrt(cfg["ycov"][7, 7])
    fit = lb.nonlinear_fit(data=(cfg["x"], ymean, cfg["ycov"]), fcn="multiexp",
                           prior=(cfg["prior_mean"], cfg["prior_sdev"]), p0=cfg["prior_mean"] * 1.05, tol=TOL, **kw)
    return cfg, fit


def test_central_copy_reproduces_single_fit():
    """The copy whose means are the fit's own data reproduces the central nonlinear_fit(..., loss=...) (which stays on
    the single-fit path)."""
    _need_gpu()
    cfg, fit = _c3_fit(loss="soft_l1", f_scale=2.0)
    assert fit._dense is not None
    same = fit.bootstrapped_fits(means=fit.yp_pdf.mean[None, :]).arrays()
    assert same["status"][0] > 0
    assert abs(same["chi2"][0] - fit.chi2) <= 1e-6 * fit.chi2, (same["chi2"][0], fit.chi2)
    assert np.max(np.abs(same["x"][0] - fit.pmean) / fit.psdev) <= 1e-3


def _same_bits(a, b, keys=KEYS):
    for k in keys:
        assert np.array_equal(a[k], b[k], equal_nan=True), k


def test_bits():
    """A fit alone (B = 1) equals its row in a batch of 2000, with the ordered queue on and off; loss='linear' is
    today's batch; kernel=2 / 4 / 'wave' with a loss equals kernel=None (one warp per fit, last_team 1); a plain batch
    after a robust one on the same cached plan equals one before it; fit_batch_host with pinned outputs equals
    fit_batch."""
    _need_gpu()
    import torch
    cfg, opdf, plan, means = _corr(3, 2000, 11, True)
    p0 = cfg["ptrue"]
    rob = dict(tol=TOL, loss="soft_l1", f_scale=2.0)
    plain0 = plan.fit_batch(means, p0, tol=TOL).numpy()
    try:
        for order in (0, 1):
            plan.set_order(order)
            whole = plan.fit_batch(means, p0, **rob).numpy()
            for b in (0, 17, 1999):
                one = plan.fit_batch(means[b:b + 1], p0, **rob).numpy()
                _same_bits(dict((k, one[k][0]) for k in KEYS), dict((k, whole[k][b]) for k in KEYS))
    finally:
        plan.set_order(None)
    _same_bits(plan.fit_batch(means, p0, tol=TOL, loss="linear", f_scale=5.0).numpy(), plain0)
    _same_bits(plan.fit_batch(means, p0, tol=TOL).numpy(), plain0)          # after the robust batches
    dev = plan.fit_batch(means[:300], p0, want_fJ=True, **rob).numpy()
    pin = lambda shp, dt: torch.empty(shp, dtype=dt, pin_memory=True).numpy()
    f8, i4 = torch.float64, torch.int32
    out = dict(x=pin((300, 6), f8), chi2=pin(300, f8), cov=pin((300, 6, 6), f8), logdet=pin(300, f8),
               nit=pin(300, i4), status=pin(300, i4), f=pin((300, plan.nchiv), f8), J=pin((300, plan.nchiv, 6), f8))
    host = plan.fit_batch_host(means[:300], p0, out=out, **rob)
    _same_bits(host, dev, keys=KEYS + ("f", "J"))
    cfg8, fit = _c3_fit(loss="cauchy", f_scale=2.0)
    ref = fit.bootstrapped_fits(500, seed=9).arrays()
    plan8 = fit._spec.plan(fit.device)
    for kernel in (2, 4, "wave"):
        got = fit.bootstrapped_fits(500, seed=9, kernel=kernel).arrays()
        assert plan8.last_team() == 1, kernel
        _same_bits(ref, got)


def test_the_loss_acts():
    """huber with an f_scale above every residual is the plain fit; soft_l1 moves the copies with outliers by more
    than half a standard deviation; f / J are the true rows at the returned x (Plan.residual_jacobian)."""
    _need_gpu()
    cfg, opdf, plan, means = _corr(3, 2000, 23, True)
    p0 = cfg["ptrue"]
    plain = plan.fit_batch(means, p0, tol=TOL).numpy()
    sd = np.sqrt(np.einsum("bii->bi", plain["cov"]))
    wide = plan.fit_batch(means, p0, tol=TOL, loss="huber", f_scale=1e6).numpy()
    ok = (plain["status"] > 0) & (wide["status"] > 0)
    assert ok.mean() > 0.99
    assert np.max(np.abs(wide["x"] - plain["x"])[ok] / sd[ok]) < 1e-10
    rob = plan.fit_batch(means, p0, tol=TOL, loss="soft_l1", f_scale=1.0, want_fJ=True).numpy()
    hit = np.flatnonzero(np.any(np.abs(means - _corr(3, 2000, 23, False)[3]) > 0, axis=1))
    assert hit.size > 10
    moved = np.max(np.abs(rob["x"][hit] - plain["x"][hit]) / sd[hit], axis=1)
    assert np.max(moved) > 0.5, np.max(moved)
    f, J, chi2 = plan.residual_jacobian(rob["x"], means)
    f, J, chi2 = (t.cpu().numpy() for t in (f, J, chi2))
    assert np.array_equal(f, rob["f"]) and np.array_equal(J, rob["J"])
    assert np.allclose(chi2, rob["chi2"], rtol=1e-12, atol=0)


def test_cuda_functor_plugin():
    """A cuda_functor plug-in gets the robust kernel with no registry change: copies against scipy least_squares."""
    _need_gpu()
    import lsqfit_b200 as lb
    from scipy.optimize import least_squares
    fun = lb.cuda_functor("ut_robust_line", "return b[0] + b[1] * x[0] + b[2] * exp(-x[0]);", 3)
    t = np.linspace(0.0, 4.0, 40)
    ptrue, pm, ps = np.array([1.0, 0.5, 2.0]), np.zeros(3), np.full(3, 10.0)
    sig = 0.05 * np.ones(t.size)
    rng = np.random.default_rng(3)
    ys = ptrue[0] + ptrue[1] * t + ptrue[2] * np.exp(-t) + sig * rng.standard_normal((64, t.size))
    ys[:, 5] += 20.0 * sig[5]
    means = np.concatenate([ys, np.broadcast_to(pm, (64, 3))], axis=1)
    plan = lb.Plan(fun, 3, t.size, t[:, None], [(np.arange(t.size + 3), 1.0 / np.concatenate([sig, ps]))])
    out = plan.fit_batch(means, pm, tol=TOL, loss="cauchy", f_scale=2.0).numpy()
    for b in range(0, 64, 8):
        def chiv(p, y=ys[b]):
            return np.concatenate([(p[0] + p[1] * t + p[2] * np.exp(-t) - y) / sig, (p - pm) / ps])
        r = least_squares(chiv, pm, method="trf", x_scale="jac", loss="cauchy", f_scale=2.0, xtol=1e-10, ftol=1e-10,
                          gtol=1e-10)
        sd = np.sqrt(np.diag(out["cov"][b]))
        assert out["status"][b] > 0 and np.max(np.abs(out["x"][b] - r.x) / sd) < 1e-4, b


def test_multifitter_bootstrap_with_loss():
    """MultiFitter.bootstrapped_fits with a loss: a few copies agree with robust single fits (single-fit path) of the
    same means and whitening."""
    _need_gpu()
    import lsqfit_b200 as lb
    from test_seam import _multi_problem
    models, data, prior = _multi_problem()
    mf = lb.MultiFitter(models, tol=1e-10, loss="huber", f_scale=1.0)
    fit = mf.lsqfit(data, prior)
    a = mf.bootstrapped_fits(64, seed=5).arrays()
    means = fit.bootstrap_means(64, seed=5).cpu().numpy()
    ny = fit.y.size
    for b in (0, 1, 2, 3):
        fd = lb.nonlinear_fit(data=(fit.x, means[b, :ny], None), prior=(means[b, ny:], fit.prior[1]), fcn=fit.fcn,
                              _yp_pdf=fit.yp_pdf, p0=fit.pmean, tol=1e-10, loss="huber", f_scale=1.0)
        assert abs(a["chi2"][b] - fd.chi2) <= 1e-6 * fd.chi2, b
        assert np.max(np.abs(a["x"][b] - fd.pmean) / fd.psdev) <= 1e-3, b


def test_refusals():
    """Python: a batch driver given a loss other than its fit's own, and the copies of a robust fit with bounds, with
    parameter distributions or with policy='gsl', are a ValueError; window scans keep refusing a loss.  C ABI: b200lm_set_loss refuses an unknown code, a bad f_scale, windows, fit sets,
    bounds, distributions and the GSL policy; while a loss is set, set_bounds (finite), set_param_dist (nonzero),
    set_policy(1) and set_windows are refused."""
    _need_gpu()
    import lsqfit_b200 as lb
    from lsqfit_b200 import _cabi
    cfg, opdf, plan, means = _corr(3, 16, 5, False)
    npar = cfg["np"]
    fit = lb.nonlinear_fit(data=(cfg["x"], cfg["f"], cfg["ycov"]), fcn="multiexp",
                           prior=(cfg["prior_mean"], cfg["prior_sdev"]), tol=TOL)
    fr = lb.nonlinear_fit(data=(cfg["x"], cfg["f"], cfg["ycov"]), fcn="multiexp",
                          prior=(cfg["prior_mean"], cfg["prior_sdev"]), tol=TOL, loss="huber", f_scale=1.5)
    for f, kw in ((fit, dict(loss="huber")), (fr, dict(loss="cauchy")), (fr, dict(f_scale=2.0)),
                  (fr, dict(loss="linear"))):
        with pytest.raises(ValueError, match="fit's own robust loss"):
            f.bootstrapped_fits(10, seed=1, **kw)
    assert np.all(fr.bootstrapped_fits(10, seed=1, loss="huber", f_scale=1.5).arrays()["status"] > 0)
    box = (np.full(npar, -10.0), np.full(npar, 10.0))
    with pytest.raises(ValueError, match="robust loss together with bounds"):
        fr.bootstrapped_fits(10, seed=1, bounds=box)
    with pytest.raises(ValueError, match="gsl"):
        fr.bootstrapped_fits(10, seed=1, policy="gsl")
    fp = lb.nonlinear_fit(data=(cfg["x"], cfg["f"], cfg["ycov"]), fcn="multiexp",
                          prior=(cfg["prior_mean"], cfg["prior_sdev"]), tol=TOL, pdist=["log"] + [None] * (npar - 1),
                          loss="huber")
    with pytest.raises(ValueError, match="pdist"):
        fp.bootstrapped_fits(10, seed=1)
    with pytest.raises(ValueError, match="loss"):
        plan.fit_batch(means, cfg["ptrue"], loss="nonsense")
    with pytest.raises(ValueError, match="f_scale"):
        plan.fit_batch(means, cfg["ptrue"], loss="huber", f_scale=0.0)
    masks = np.ones((2, cfg["ny"]), bool)
    masks[1, :8] = False
    with pytest.raises(ValueError, match="robust loss"):
        fit.window_fits(masks, loss="huber")
    # ---- the C ABI
    h = plan._h
    err = lambda rc, what: rc == _cabi.EINVAL and what in _cabi.last_error(h)
    set_loss = lambda code, fs=1.0: _cabi.lib.b200lm_set_loss(h, code, fs)
    assert err(set_loss(5), "unknown loss")
    assert err(set_loss(-1), "unknown loss")
    for bad in (0.0, -1.0, np.inf, np.nan):
        assert err(set_loss(1, bad), "f_scale")
    assert set_loss(0, np.nan) == _cabi.OK                       # code 0 clears, f_scale unread
    lo, hi = (np.ascontiguousarray(b) for b in box)
    codes = np.ascontiguousarray([1] + [0] * (npar - 1), dtype=np.int32)
    try:
        assert _cabi.lib.b200lm_set_bounds(h, lo.ctypes.data, hi.ctypes.data) == _cabi.OK
        assert err(set_loss(1), "bounds")
        assert _cabi.lib.b200lm_set_bounds(h, None, None) == _cabi.OK
        assert _cabi.lib.b200lm_set_param_dist(h, codes.ctypes.data, None, None) == _cabi.OK
        assert err(set_loss(1), "parameter distributions")
        assert _cabi.lib.b200lm_set_param_dist(h, None, None, None) == _cabi.OK
        assert _cabi.lib.b200lm_set_policy(h, 1) == _cabi.OK
        assert err(set_loss(1), "GSL")
        assert _cabi.lib.b200lm_set_policy(h, 0) == _cabi.OK
        assert set_loss(2, 1.5) == _cabi.OK
        assert err(_cabi.lib.b200lm_set_bounds(h, lo.ctypes.data, hi.ctypes.data), "robust loss")
        inf = np.full(npar, np.inf)
        assert _cabi.lib.b200lm_set_bounds(h, (-inf).ctypes.data, inf.ctypes.data) == _cabi.OK   # no box: fine
        assert err(_cabi.lib.b200lm_set_param_dist(h, codes.ctypes.data, None, None), "robust loss")
        zero = np.zeros(npar, np.int32)
        assert _cabi.lib.b200lm_set_param_dist(h, zero.ctypes.data, None, None) == _cabi.OK     # all plain: fine
        assert err(_cabi.lib.b200lm_set_policy(h, 1), "robust loss")
        one = np.ones(1, np.int32)
        assert err(_cabi.lib.b200lm_set_windows(h, 1, one.ctypes.data, None, None, one.ctypes.data, None, None, None,
                                                None), "robust loss")
    finally:
        set_loss(0)
        _cabi.lib.b200lm_set_bounds(h, None, None)
        _cabi.lib.b200lm_set_param_dist(h, None, None, None)
        _cabi.lib.b200lm_set_policy(h, 0)
    scan = fit.window_fits(masks)
    assert _cabi.lib.b200lm_set_loss(scan.plan._h, 1, 1.0) == _cabi.EINVAL
    assert "window scans or fit sets" in _cabi.last_error(scan.plan._h)
    hs = _cabi.handle_t()
    assert _cabi.lib.b200lm_create_set(plan.functor.family, cfg["ny"], npar, 1, 2, 0, 0, C.byref(hs)) == _cabi.OK
    try:
        assert _cabi.lib.b200lm_set_loss(hs, 1, 1.0) == _cabi.EINVAL
        assert "window scans or fit sets" in _cabi.last_error(hs)
    finally:
        _cabi.lib.b200lm_destroy(hs)

