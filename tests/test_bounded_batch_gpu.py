"""Batched bound-constrained fits (scipy's ``bounds``, ``lsqfit.scipy_least_squares(bounds=...)``, reference
src/lsqfit/_scipy.py:77): the one-warp kernel's bounded driver (csrc/lm_kernel.cuh: fit_one<F, 3>; numpy model
tests/lm_model_bounded.py, checked on the CPU by test_bounded_model_cpu.py), the C ABI's b200lm_set_bounds, Plan.fit_batch's
``bounds`` and the batch drivers of nonlinear_fit / MultiFitter, against scipy's bounded trf through the oracle (a
process pool on the host cores).  Needs a GPU (pytest -m gpu).
"""
import numpy as np
import pytest

from parity_util import _W, correlator_problem

pytestmark = pytest.mark.gpu

BENCH_TOL = (1e-8, 1e-10, 1e-10)
INF = np.inf


def _need_gpu():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (no CPU fallback)")


# ---- oracle workers with bounds (spawned pool: module-level functions) ------------------------------------------
def _corr_init(K):
    import os
    import warnings
    os.environ["OPENBLAS_NUM_THREADS"] = "1"
    warnings.simplefilter("ignore")
    _W["cfg"], _W["pdf"] = correlator_problem(K)


def _corr_job(arg):
    from oracle.fit import nonlinear_fit
    mean, p0, tol, lo, hi = arg
    cfg, pdf = _W["cfg"], _W["pdf"]
    ny = cfg["ny"]
    fo = nonlinear_fit("multiexp", cfg["x"], mean[:ny], prior_mean=mean[ny:], _yp_pdf=pdf, p0=p0, tol=tol,
                       maxit=1000, x_scale="jac", bounds=(lo, hi))
    return dict(x=fo.pmean, cov=fo.cov, chi2=fo.chi2, nit=fo.nit, crit=fo.stopping_criterion)


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
    k, p0, lo, hi = arg
    pr = _W["nist"][k]
    fo = nonlinear_fit(pr["form"], np.array(pr["x"]), pr["y"], pr["ysdev"], prior_mean=pr["prior_mean"],
                       prior_cov=pr["prior_sdev"], p0=p0, tol=1e-10, maxit=1000, x_scale="jac", bounds=(lo, hi))
    return dict(x=fo.pmean, chi2=fo.chi2, crit=fo.stopping_criterion, sd=fo.psdev)


def _pool(init, initargs, job, jobs):
    import multiprocessing as mp
    import os
    nproc = min(os.cpu_count() or 1, 32)
    with mp.get_context("spawn").Pool(nproc, initializer=init, initargs=initargs) as pool:
        return pool.map(job, jobs, chunksize=max(1, len(jobs) // (nproc * 8)))


# ---- C4: simulated copies ----------------------------------------------------------------------------------------
def _c4(B=2000):
    import lsqfit_b200 as lb
    from lsqfit_b200 import configs
    cfg, opdf = correlator_problem(3)
    ny, npar = cfg["ny"], cfg["np"]
    means = configs.bootstrap_means(cfg, B, 4245, cov=opdf.cov[:ny, :ny], vary_prior=False)
    plan = lb.Plan("multiexp", npar, ny, cfg["x"], opdf.i_invwgts)
    return cfg, plan, means, cfg["ptrue"].copy()


KEYS = ("x", "chi2", "cov", "logdet", "nit", "status")


def _same_bits(a, b, rows=slice(None)):
    for k in KEYS:
        assert np.array_equal(a[k][rows], b[k][rows], equal_nan=True), k


def test_noop_box_and_batch_independence():
    """(1) an all-infinite box is no box: scipy then runs its unbounded trf, and the batch gives the bits of an
    unbounded batch.  (2) a bounded fit alone (B = 1) and inside a batch of 2000 give the same bits."""
    _need_gpu()
    cfg, plan, means, p0 = _c4()
    npar = cfg["np"]
    free = plan.fit_batch(means, p0, tol=BENCH_TOL).numpy()
    noop = plan.fit_batch(means, p0, tol=BENCH_TOL, bounds=(np.full(npar, -INF), np.full(npar, INF))).numpy()
    _same_bits(free, noop)
    lo, hi = np.full(npar, -INF), np.full(npar, INF)
    lo[npar - 1] = p0[npar - 1] - 0.02
    whole = plan.fit_batch(means, p0, tol=BENCH_TOL, bounds=(lo, hi)).numpy()
    for b in (0, 17, 1999):
        one = plan.fit_batch(means[b:b + 1], p0, tol=BENCH_TOL, bounds=(lo, hi)).numpy()
        for k in KEYS:
            assert np.array_equal(one[k][0], whole[k][b], equal_nan=True), (b, k)


def _active(x, lo, hi):
    on_lo = np.isfinite(lo) & (np.abs(x - lo) <= 1e-7 * np.maximum(1.0, np.abs(lo)))
    on_hi = np.isfinite(hi) & (np.abs(x - hi) <= 1e-7 * np.maximum(1.0, np.abs(hi)))
    return np.where(on_lo, -1, np.where(on_hi, 1, 0))


def test_c4_2000_copies_vs_scipy_bounded_trf():
    """2000 simulated C4 copies (p0 = pexact) with a box on the two highest energies, each pexact -/+ one standard
    deviation of the unbounded copies: a good share of the copies ends with an active bound.  Against scipy's bounded
    trf on the same copies: every x in the box, the same copies converge, the same active set, chi2, and the free
    parameters.  Measured on a B200: 39.6 % of the copies end on a bound, the active set agrees on every copy, chi2
    within 6.5e-13 relative, free parameters within 3.6e-6 sdev (mean nfev 11.29 vs scipy's 11.30).  Bars: those
    worst cases with headroom -- chi2 1e-11, free parameters 1e-5 sdev, active set on >= 99.9 % of the copies."""
    _need_gpu()
    cfg, plan, means, p0 = _c4()
    npar = cfg["np"]
    free = plan.fit_batch(means, p0, tol=BENCH_TOL).numpy()
    sd = free["x"][free["status"] > 0].std(axis=0)
    lo, hi = np.full(npar, -INF), np.full(npar, INF)
    for j in (npar - 2, npar - 1):
        lo[j], hi[j] = p0[j] - sd[j], p0[j] + sd[j]
    out = plan.fit_batch(means, p0, tol=BENCH_TOL, bounds=(lo, hi)).numpy()
    assert np.all((out["x"] >= lo) & (out["x"] <= hi))
    ref = _pool(_corr_init, (3,), _corr_job, [(m, p0, BENCH_TOL, lo, hi) for m in means])
    conv_d = out["status"] > 0
    conv_o = np.array([r["crit"] != 0 for r in ref])
    assert np.array_equal(conv_d, conv_o)
    ok = conv_d & conv_o
    xo = np.array([r["x"] for r in ref])
    act_d = np.array([_active(x, lo, hi) for x in out["x"]])
    act_o = np.array([_active(x, lo, hi) for x in xo])
    frac_active = float(np.mean(np.any(act_o != 0, axis=1)[ok]))
    same_act = float(np.mean(np.all(act_d == act_o, axis=1)[ok]))
    chi2o = np.array([r["chi2"] for r in ref])
    dchi2 = (np.abs(out["chi2"] - chi2o) / chi2o)[ok]
    sdo = np.sqrt(np.array([np.diag(r["cov"]) for r in ref]))
    both = ok & np.all(act_d == act_o, axis=1)
    dp = np.array([np.max(np.where(act_o[b] == 0, np.abs(out["x"][b] - xo[b]) / sdo[b], 0.0)) for b in range(len(ref))])[both]
    print("C4 bounded, %d copies: active on %.1f %%, same active set %.2f %%, chi2 max %.2e, free p max %.2e q99 %.2e sd, "
          "mean nfev %.2f vs %.2f" % (len(ref), 100 * frac_active, 100 * same_act, dchi2.max(), dp.max(),
                                      np.quantile(dp, 0.99), out["nit"].mean(), np.mean([r["nit"] for r in ref])))
    assert 0.1 <= frac_active <= 0.9
    assert same_act >= 0.999
    assert dchi2.max() <= 1e-11
    assert dp.max() <= 1e-5


BOX_PROBLEMS = ("misra1a", "chwirut2", "gauss1", "rat42", "thurber")


def _nist_box(pr):
    cert, p0 = np.array(pr["certified"]), np.array(pr["p0"])
    lo = np.minimum(cert, p0) - 0.5 * np.abs(cert - p0) - 1e-3 * np.abs(cert)
    hi = np.maximum(cert, p0) + 0.5 * np.abs(cert - p0) + 1e-3 * np.abs(cert)
    mid = 0.5 * (cert[0] + p0[0])
    if p0[0] < cert[0]:
        hi[0] = mid
    else:
        lo[0] = mid
    return lo, hi, mid


def test_nist_box_perturbed_starts_vs_oracle(nist_problems):
    """The five NIST problems of the single-fit bounds test with its box, from 200 starts p0 (1 + 0.1 u) each,
    clipped into the box: the cut parameter ends on its bound and chi2 agrees with scipy's bounded trf to 1e-6
    (measured on a B200: every start converges on both sides and ends on the bound; chi2 within 1.4e-13)."""
    _need_gpu()
    import lsqfit_b200 as lb
    rng = np.random.default_rng(7)
    names = [pr["name"] for pr in nist_problems]
    for name in BOX_PROBLEMS:
        k = names.index(name)
        pr = nist_problems[k]
        lo, hi, mid = _nist_box(pr)
        p0 = np.array(pr["p0"])
        starts = np.clip(p0[None, :] * (1 + 0.1 * rng.uniform(-1, 1, (200, p0.size))), lo, hi)
        fit = lb.nonlinear_fit(data=(np.array(pr["x"]), pr["y"], pr["ysdev"]), fcn=pr["form"],
                               prior=(pr["prior_mean"], pr["prior_sdev"]), p0=pr["p0"], tol=1e-10)
        out = fit._spec.plan(0).fit_batch(fit._spec.mean, starts, tol=1e-10, maxit=1000, bounds=(lo, hi)).numpy()
        ref = _pool(_nist_init, (), _nist_job, [(k, s, lo, hi) for s in starts])
        assert np.all((out["x"] >= lo) & (out["x"] <= hi)), name
        chi2o = np.array([r["chi2"] for r in ref])
        ok = (out["status"] > 0) & np.array([r["crit"] != 0 for r in ref])
        on_bound = np.abs(out["x"][:, 0] - mid) <= 1e-6 * abs(mid)
        dchi2 = np.abs(out["chi2"] - chi2o) / chi2o
        print("%s: %d / 200 converge on both sides, cut parameter on its bound %d, chi2 max %.2e"
              % (name, ok.sum(), on_bound[ok].sum(), dchi2[ok].max()))
        assert ok.mean() >= 0.99, name
        assert np.all(on_bound[ok]), name
        assert dchi2[ok].max() <= 1e-6, name


def test_reference_bounds_test_as_bootstrap():
    """The reference's own bounds test (tests/test_lsqfit.py:1779-1808: fcn(p) = p, data 0.9(1), 2.2(2), no prior,
    bounds [0, 0.5] x [0, 1]) as 1000 bootstrap copies: every copy ends on the upper bounds (7 places)."""
    _need_gpu()
    import lsqfit_b200 as lb
    box = ([0.0, 0.0], [0.5, 1.0])
    fit = lb.nonlinear_fit(data=(np.array([0.0, 1.0]), [0.9, 2.2], [0.1, 0.2]), fcn="gather", p0=[0.25, 0.5], bounds=box)
    bs = fit.bootstrapped_fits(1000, seed=11).arrays()
    assert np.all(bs["status"] > 0)
    assert np.max(np.abs(bs["x"] - np.array([0.5, 1.0]))) < 1e-7


def _c4_fit(**kw):
    import lsqfit_b200 as lb
    from lsqfit_b200 import configs
    cfg = configs.correlator(3)
    rng = np.random.default_rng(3)
    y = cfg["f"] + np.linalg.cholesky(cfg["ycov"]) @ rng.standard_normal(cfg["ny"])
    return cfg, lb.nonlinear_fit(data=(cfg["x"], y, cfg["ycov"]), fcn="multiexp",
                                 prior=(cfg["prior_mean"], cfg["prior_sdev"]), **kw)


def test_drivers_respect_the_box():
    """nonlinear_fit(..., bounds=box).bootstrapped_fits / .simulated_fits (and their iterators) keep every copy inside
    the box (before the bounds reached the kernel, the copies were fitted without them); the copy whose mean is the
    parent's agrees with the bounded parent fit (single-fit path)."""
    _need_gpu()
    cfg, probe = _c4_fit()
    npar = cfg["np"]
    lo, hi = np.full(npar, -INF), np.full(npar, INF)
    lo[npar - 1] = probe.pmean[npar - 1] + 0.5 * probe.psdev[npar - 1]     # cuts off the unbounded minimum
    p0 = probe.pmean.copy()
    p0[npar - 1] = lo[npar - 1] + 0.1 * probe.psdev[npar - 1]              # (scipy refuses a start outside the box)
    cfg, fit = _c4_fit(bounds=(lo, hi), p0=p0)
    assert abs(fit.pmean[npar - 1] - lo[npar - 1]) < 1e-7 * abs(lo[npar - 1])
    for bs in (fit.bootstrapped_fits(2000, seed=1), fit.simulated_fits(2000, seed=2)):
        a = bs.arrays()
        assert np.all((a["x"] >= lo) & (a["x"] <= hi))
        assert np.mean(a["status"] > 0) > 0.99
    assert all(np.all(f.pmean >= lo) for f in fit.bootstrapped_fit_iter(50, seed=3))
    same = fit.bootstrapped_fits(means=fit.yp_pdf.mean[None, :]).arrays()
    assert abs(same["chi2"][0] - fit.chi2) <= 1e-6 * fit.chi2
    assert np.max(np.abs(same["x"][0] - fit.pmean) / fit.psdev) <= 1e-3


def test_multifitter_bootstrap_with_bounds():
    """MultiFitter.bootstrapped_fits on the shared-energy composite (multiexp_shared2, whose parameter order is its
    own: amplitudes, then energies) with a lower bound on the first energy: every copy inside the box, and a few copies
    agree with bounded single fits (b200_dense path) of the same means and whitening."""
    _need_gpu()
    import lsqfit_b200 as lb
    from test_seam import _multi_problem
    models, data, prior = _multi_problem()
    fit0 = lb.MultiFitter(models, tol=1e-10).lsqfit(data, prior)
    n = fit0.pmean.size
    nE = len(prior[0][models[0].E])
    j = n - nE                                          # the first energy in the composite's order
    lo, hi = np.full(n, -INF), np.full(n, INF)
    lo[j] = fit0.pmean[j] + 0.5 * fit0.psdev[j]
    p0 = fit0.pmean.copy()
    p0[j] = lo[j] + 0.1 * fit0.psdev[j]
    mf = lb.MultiFitter(models, tol=1e-10, bounds=(lo, hi))
    fit = mf.lsqfit(data, prior, p0=p0[fit0.pflat_order])             # (p0 in the prior dictionary's order)
    bs = mf.bootstrapped_fits(256, seed=5)
    a = bs.arrays()
    assert np.all((a["x"] >= lo) & (a["x"] <= hi))
    means = fit.bootstrap_means(256, seed=5).cpu().numpy()
    ny = fit.y.size
    for b in (0, 1, 2, 3):
        fd = lb.nonlinear_fit(data=(fit.x, means[b, :ny], None), prior=(means[b, ny:], fit.prior[1]), fcn=fit.fcn,
                              _yp_pdf=fit.yp_pdf, p0=fit.pmean, tol=1e-10, bounds=(lo, hi))
        assert abs(a["chi2"][b] - fd.chi2) <= 1e-6 * fd.chi2, b
        assert np.max(np.abs(a["x"][b] - fd.pmean) / fd.psdev) <= 1e-3, b


def test_kernel_choice_and_refusals():
    """Bounded batches run in the one-warp kernel whatever kernel is asked for (same bits); batched robust loss, GSL
    with bounds, an infeasible start and lb >= ub are refused -- by Python with ValueError and by the C ABI with
    B200LM_EINVAL."""
    _need_gpu()
    import lsqfit_b200 as lb
    from lsqfit_b200 import _cabi
    cfg, fit = _c4_fit()
    npar = cfg["np"]
    lo, hi = np.full(npar, -INF), np.full(npar, INF)
    lo[npar - 1] = fit.pmean[npar - 1] - 0.5 * fit.psdev[npar - 1]
    ref = fit.bootstrapped_fits(500, seed=9, bounds=(lo, hi), kernel=1).arrays()
    plan = fit._spec.plan(0)
    for kernel in (4, "wave"):
        got = fit.bootstrapped_fits(500, seed=9, bounds=(lo, hi), kernel=kernel).arrays()
        assert plan.last_team() == 1
        _same_bits(ref, got)
    with pytest.raises(ValueError, match="robust"):
        fit.bootstrapped_fits(10, seed=1, loss="huber")
    with pytest.raises(ValueError, match="gsl"):
        fit.bootstrapped_fits(10, seed=1, bounds=(lo, hi), policy="gsl")
    with pytest.raises(ValueError, match="infeasible"):
        fit.bootstrapped_fits(10, seed=1, bounds=(fit.pmean + 1.0, np.full(npar, INF)))
    with pytest.raises(ValueError, match="strictly less"):
        fit.bootstrapped_fits(10, seed=1, bounds=(hi, lo))
    with pytest.raises(ValueError, match="infeasible"):
        plan.fit_batch_host(fit._spec.mean, fit.pmean - 1.0, bounds=(fit.pmean, np.full(npar, INF)))
    # ---- the C ABI
    h = plan._h
    dbl = lambda a: np.ascontiguousarray(a, dtype=np.float64)
    lo_, hi_ = dbl(lo), dbl(hi)
    assert _cabi.lib.b200lm_set_bounds(h, hi_.ctypes.data, lo_.ctypes.data) == _cabi.EINVAL
    assert "strictly less" in _cabi.last_error(h)
    nan = dbl(np.where(np.isfinite(lo), np.nan, lo))
    assert _cabi.lib.b200lm_set_bounds(h, nan.ctypes.data, hi_.ctypes.data) == _cabi.EINVAL
    mean = dbl(fit._spec.mean)
    x0 = dbl(fit.pmean)
    outs = dict(x=np.empty(npar), chi2=np.empty(1), logdet=np.empty(1), nit=np.empty(1, np.int32),
                status=np.empty(1, np.int32))
    ptr = lambda k: outs[k].ctypes.data
    call = lambda p0: _cabi.lib.b200lm_fit_batch_host(h, 1, mean.ctypes.data, 0, p0.ctypes.data, 0, 1e-8, 1e-10, 1e-10,
                                                      1000, 1, 0, ptr("x"), ptr("chi2"), None, ptr("logdet"),
                                                      ptr("nit"), ptr("status"), None, None)
    try:
        assert _cabi.lib.b200lm_set_bounds(h, lo_.ctypes.data, hi_.ctypes.data) == _cabi.OK
        bad = dbl(fit.pmean - 10.0 * fit.psdev)
        assert call(bad) == _cabi.EINVAL and "infeasible" in _cabi.last_error(h)
        assert call(x0) == _cabi.OK and np.all(outs["x"] >= lo)
        assert _cabi.lib.b200lm_set_policy(h, 1) == _cabi.OK
        assert call(x0) == _cabi.EINVAL and "GSL" in _cabi.last_error(h)
    finally:
        _cabi.lib.b200lm_set_policy(h, 0)
        _cabi.lib.b200lm_set_bounds(h, None, None)
