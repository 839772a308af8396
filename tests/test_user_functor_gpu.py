"""User-defined device models on the GPU (lsqfit_b200.cuda_functor): a plug-in that instantiates the library's kernels
for a model gives the same bits as the built-in model with the same code, on every kernel; a model the registry does
not have agrees with its host callable and with scipy; the fitters, drivers and MultiFitter take it; and loading
further plug-ins leaves existing plans alone.  Needs a GPU (pytest -m gpu); the plug-ins are compiled with nvcc where
they are not in the cache."""
import collections
import os
import sys

import numpy as np
import pytest

from parity_util import TIGHT, correlator_problem

pytestmark = pytest.mark.gpu

BENCH_TOL = (1e-8, 1e-10, 1e-10)
KEYS = ("x", "chi2", "cov", "logdet", "nit", "status")
MULTIEXP = "template <int NP> using Model = MultiExp<NP / 2>;"
DAMPED = """
const double t = x[0];
return b[0] * exp(-(b[1] * t)) * cos(b[2] * t + b[3]) + b[4];
"""
# every function of csrc/dual_more.cuh, in a body whose derivatives are all non-trivial
MATHFNS = """
const double t = x[0];
const T u = b[0] * t, v = b[1] + 0.5 * t;
return tanh(u) + sinh(v) * 0.1 + cosh(b[2] * 0.5) + expm1(-u) + log1p(b[1] * b[1] * t) + erf(u - b[2])
       + atan2(v, b[2] + 2.0) + atan2(b[1], t) + atan2(t, b[2] + 3.0) + abs(u - 5.0) * 0.1 + abs(b[1]);
"""


def damped_host(x, p):
    """the model on the host, for numpy arrays and for the dual numbers of the CPU oracle (lsqfit's fcn protocol)"""
    from oracle import dual as D
    t = np.asarray(x)
    return p[0] * D.exp(-(p[1] * t)) * D.cos(p[2] * t + p[3]) + p[4]


def mathfns_host(x, p):
    from scipy.special import erf
    t = np.asarray(x)
    u, v = p[0] * t, p[1] + 0.5 * t
    return (np.tanh(u) + np.sinh(v) * 0.1 + np.cosh(p[2] * 0.5) + np.expm1(-u) + np.log1p(p[1] * p[1] * t)
            + erf(u - p[2]) + np.arctan2(v, p[2] + 2.0) + np.arctan2(p[1], t) + np.arctan2(t, p[2] + 3.0)
            + np.abs(u - 5.0) * 0.1 + np.abs(p[1]))


def _need_gpu():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (no CPU fallback)")


def _rat43_body():
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with open(os.path.join(root, "lsqfit_b200", "csrc", "functors.cuh")) as fh:
        return re.search(r"B200LM_BODY\(Rat43Body\) \{(.*?)\} \};", fh.read()).group(1).strip()


@pytest.fixture(scope="module")
def user():
    """the module's plug-ins, compiled in parallel where the cache does not have them, then loaded"""
    import concurrent.futures
    import lsqfit_b200 as lb
    from lsqfit_b200 import functors, user_functor as uf
    _need_gpu()
    specs = dict(
        rat43=("ut_rat43", _rat43_body(), 4, 1, functors._HOST["rat43"], "body"),
        multiexp=("ut_multiexp", MULTIEXP, (6, 16), 1, functors._HOST["multiexp"], "functor"),
        damped=("ut_damped", DAMPED, 5, 1, damped_host, "body"),
        mathfns=("ut_mathfns", MATHFNS, 3, 1, mathfns_host, "body"),
    )
    with concurrent.futures.ThreadPoolExecutor(len(specs)) as ex:
        list(ex.map(lambda s: uf.build_plugin(s[0], s[1], s[2], s[3], s[5]), specs.values()))
    return dict((k, lb.cuda_functor(n, src, npar, nx, host=h, form=form))
                for k, (n, src, npar, nx, h, form) in specs.items())


def _same_bits(a, b, what):
    for k in KEYS:
        x, y = np.asarray(a[k]), np.asarray(b[k])
        assert x.dtype == y.dtype and x.shape == y.shape, (what, k)
        assert x.tobytes() == y.tobytes(), (what, k, np.max(np.abs(x.astype(float) - y.astype(float))))


# ---- bit identity: one-warp kernel (scipy, GSL, bounded) and the single-fit path --------------------------------------
def test_rat43_copy_bits(user, nist_problems):
    import lsqfit_b200 as lb
    pr = [p for p in nist_problems if p["name"] == "rat43"][0]
    x = np.array(pr["x"])
    ny, npar = len(pr["y"]), len(pr["p0"])
    mean = np.concatenate([pr["y"], pr["prior_mean"]])
    sd = np.concatenate([pr["ysdev"], pr["prior_sdev"]])
    means = mean + sd * np.random.default_rng(43).standard_normal((1000, mean.size))     # 1000 bootstrap copies
    w = [(np.arange(ny + npar), 1.0 / sd)]
    ref, mine = lb.Plan("rat43", npar, ny, x, w), lb.Plan(user["rat43"], npar, ny, x, w)
    p0 = np.array(pr["p0"])
    box = (np.array([0.0, 0.0, 0.0, 0.5]), np.array([1e3, 10.0, 2.0, 5.0]))
    for kw in (dict(), dict(policy="gsl"), dict(bounds=box)):
        a = ref.fit_batch(means, p0, tol=1e-10, maxit=1000, **kw).numpy()
        b = mine.fit_batch(means, p0, tol=1e-10, maxit=1000, **kw).numpy()
        assert np.mean(a["status"] != 0) > 0.9, kw
        _same_bits(a, b, kw)
    data, prior = (x, pr["y"], pr["ysdev"]), (pr["prior_mean"], pr["prior_sdev"])
    fa = lb.nonlinear_fit(data=data, prior=prior, fcn="rat43", p0=p0, tol=1e-10, fitter="b200_dense")
    fb = lb.nonlinear_fit(data=data, prior=prior, fcn=user["rat43"], p0=p0, tol=1e-10, fitter="b200_dense")
    for k in ("pmean", "cov", "chi2"):
        assert np.asarray(getattr(fa, k)).tobytes() == np.asarray(getattr(fb, k)).tobytes(), k


# ---- bit identity: team and wave kernels ------------------------------------------------------------------------------
def _correlator(K, B, seed):
    from lsqfit_b200 import configs
    cfg, opdf = correlator_problem(K)
    ny = cfg["ny"]
    return cfg, opdf, configs.bootstrap_means(cfg, B, seed, cov=opdf.cov[:ny, :ny])


def test_multiexp_reexport_team_and_wave_bits(user):
    import lsqfit_b200 as lb
    for K, B, teams in ((8, 10000, (0, 4)), (3, 10000, (32,))):             # C3: team of two, team of four; C4: wave
        cfg, opdf, means = _correlator(K, B, 7 + K)
        ny, npar = cfg["ny"], cfg["np"]
        ref = lb.Plan("multiexp", npar, ny, cfg["x"], opdf.i_invwgts)
        mine = lb.Plan(user["multiexp"], npar, ny, cfg["x"], opdf.i_invwgts)
        for team in teams:
            ref.set_team(team)
            mine.set_team(team)
            a = ref.fit_batch(means, cfg["prior_mean"], tol=BENCH_TOL, maxit=1000).numpy()
            b = mine.fit_batch(means, cfg["prior_mean"], tol=BENCH_TOL, maxit=1000).numpy()
            assert ref.last_team() == mine.last_team() == (team or 2), (K, team, ref.last_team(), mine.last_team())
            assert np.mean(a["status"] > 0) > 0.99
            _same_bits(a, b, (K, team))


# ---- a model the registry does not have -------------------------------------------------------------------------------
def _osc_problem(ny=40):
    t = np.linspace(0.0, 6.0, ny)
    ptrue = np.array([1.5, 0.3, 2.1, 0.4, 0.2])
    sig = np.full(ny, 0.02)
    pm, ps = ptrue * np.array([1.05, 0.9, 1.02, 0.9, 1.1]), np.array([0.5, 0.2, 0.5, 0.5, 0.2])
    return t, ptrue, sig, pm, ps


@pytest.mark.parametrize("model", ["damped", "mathfns"])
def test_residual_jacobian_vs_host(user, model):
    import lsqfit_b200 as lb
    f = user[model]
    host = damped_host if model == "damped" else mathfns_host
    npar = 5 if model == "damped" else 3
    t = np.linspace(0.05, 4.0, 37)
    ny = t.size
    w = [(np.arange(ny + npar), np.ones(ny + npar))]
    plan = lb.Plan(f, npar, ny, t, w)
    rng = np.random.default_rng(5)
    P = (np.array([1.5, 0.3, 2.1, 0.4, 0.2]) if model == "damped" else np.array([0.7, 0.4, 0.3]))[None, :] \
        * (1 + 0.2 * rng.uniform(-1, 1, size=(16, npar)))
    mean = np.zeros(ny + npar)                     # y = 0, sigma = 1: the data rows of chiv are the model values
    fd, Jd, _ = (a.cpu().numpy() for a in plan.residual_jacobian(P, mean))
    for b in range(P.shape[0]):
        fh = host(t, P[b])
        assert np.max(np.abs(fd[b, :ny] - fh)) <= 1e-13 * np.max(np.abs(fh)), (model, b)
        Jfd = np.empty((ny, npar))
        for j in range(npar):
            h = 1e-5 * max(abs(P[b, j]), 1e-2)
            e = np.zeros(npar)
            e[j] = h
            Jfd[:, j] = (host(t, P[b] + e) - host(t, P[b] - e)) / (2 * h)
        assert np.max(np.abs(Jd[b, :ny] - Jfd)) <= 1e-7 * np.max(np.abs(Jfd)), (model, b)
        np.testing.assert_array_equal(Jd[b, ny:], np.eye(npar))        # prior rows: (p - prior mean) / sdev


def _scipy_init():
    os.environ["OPENBLAS_NUM_THREADS"] = "1"


def _scipy_job(arg):
    from scipy.optimize import least_squares
    mean, p0 = arg
    t, _, sig, pm, ps = _osc_problem()
    ny = t.size
    fun = lambda p: np.concatenate([(damped_host(t, p) - mean[:ny]) / sig, (p - mean[ny:]) / ps])
    r = least_squares(fun, p0, method="trf", x_scale="jac", jac="3-point", xtol=1e-14, ftol=1e-14, gtol=1e-14,
                      max_nfev=2000)
    J = r.jac
    return r.x, 2 * r.cost, np.linalg.inv(J.T @ J), r.status


def test_damped_oscillator_vs_scipy(user):
    """2000 simulated copies against scipy's trf on the host callable.  Both solvers stop where cost differences drop
    below eps * cost, ~sqrt(eps chi2) sdev short of the stationary point (tests/parity_util.py); p is compared at ten
    times that plus the 1e-8 sdev of the tight-tolerance parity tests, chi2 to 1e-9."""
    import multiprocessing as mp
    import lsqfit_b200 as lb
    t, ptrue, sig, pm, ps = _osc_problem()
    ny, npar, B = t.size, 5, 2000
    rng = np.random.default_rng(2024)
    means = np.concatenate([damped_host(t, ptrue) + sig * rng.standard_normal((B, ny)),
                            np.broadcast_to(pm, (B, npar))], axis=1)
    sd = np.concatenate([sig, ps])
    plan = lb.Plan(user["damped"], npar, ny, t, [(np.arange(ny + npar), 1.0 / sd)])
    o = plan.fit_batch(means, pm, tol=TIGHT, maxit=2000).numpy()
    nproc = min(os.cpu_count() or 1, 32)
    with mp.get_context("spawn").Pool(nproc, initializer=_scipy_init) as pool:
        ref = pool.map(_scipy_job, [(m, pm) for m in means], chunksize=max(1, B // (nproc * 8)))
    xo = np.array([r[0] for r in ref])
    chio = np.array([r[1] for r in ref])
    sdo = np.sqrt(np.array([np.diag(r[2]) for r in ref]))
    conv = (o["status"] > 0) & np.array([r[3] > 0 for r in ref])
    assert conv.mean() > 0.99
    dp = np.max(np.abs(o["x"] - xo) / sdo, axis=1)
    tol = 10 * np.sqrt(np.finfo(float).eps * np.maximum(chio, 1.0)) + 1e-8
    ok = conv & (dp <= tol) & (np.abs(o["chi2"] - chio) <= 1e-9 * chio)
    assert ok.sum() >= 0.99 * conv.sum(), (ok.sum(), conv.sum(), np.median(dp[conv]), np.max(dp[conv]))
    s = np.sqrt(np.einsum("bii->bi", o["cov"]))
    assert np.median(np.max(np.abs(s - sdo) / sdo, axis=1)[ok]) < 1e-6


# ---- end to end: the lsqfit protocol, its iterators, MultiFitter ------------------------------------------------------
def test_user_functor_through_lsqfit_protocol(user):
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    import lsqfit_double as L
    import lsqfit_b200 as lb
    lb.register(L)
    t, ptrue, sig, pm, ps = _osc_problem()
    y = damped_host(t, ptrue) + sig * np.random.default_rng(1).standard_normal(t.size)
    data, prior = (t, y, np.diag(sig ** 2)), (pm, ps)
    dev = L.nonlinear_fit(data=data, prior=prior, fcn=user["damped"], fitter="b200_lm", tol=TIGHT, polish=8)
    ref = L.nonlinear_fit(data=data, prior=prior, fcn=damped_host, fitter="scipy_least_squares", tol=TIGHT,
                          x_scale="jac")
    assert dev.error is None
    np.testing.assert_allclose(dev.pmean, ref.pmean, rtol=0, atol=1e-6 * np.max(ref.psdev))
    np.testing.assert_allclose(dev.chi2, ref.chi2, rtol=1e-9)
    n = 0
    for bd in dev.bootstrapped_fit_iter(n=20, seed=3):
        assert bd.error is None and np.all(np.isfinite(bd.pmean))
        n += 1
    assert n == 20
    byname = L.nonlinear_fit(data=data, prior=prior, fcn=lb.Functor("ut_damped"), fitter="b200_lm", tol=TIGHT, polish=8)
    assert byname.pmean.tobytes() == dev.pmean.tobytes()
    # MultiFitter: a FunctorModel on the user functor
    mf = lb.MultiFitter([lb.FunctorModel("osc", user["damped"], t, ("a", "g", "w", "phi", "c"))], tol=TIGHT)
    keys = ("a", "g", "w", "phi", "c")
    ch = mf.chained_lsqfit({"osc": (y, sig)}, (collections.OrderedDict(zip(keys, pm)), dict(zip(keys, ps))))
    np.testing.assert_allclose(ch.fits[0].pmean, ref.pmean, rtol=0, atol=1e-6 * np.max(ref.psdev))


# ---- registry stability -----------------------------------------------------------------------------------------------
def test_plans_survive_later_plugins(user):
    import lsqfit_b200 as lb
    t, ptrue, sig, pm, ps = _osc_problem()
    sd = np.concatenate([sig, ps])
    means = np.concatenate([damped_host(t, ptrue) + sig * np.random.default_rng(9).standard_normal((256, t.size)),
                            np.broadcast_to(pm, (256, 5))], axis=1)
    plan = lb.Plan(user["damped"], 5, t.size, t, [(np.arange(t.size + 5), 1.0 / sd)])
    a = plan.fit_batch(means, pm, tol=BENCH_TOL).numpy()
    n0 = len(lb.available())
    later = lb.cuda_functor("ut_later", "return b[0] + b[1] * x[0] + b[2] * exp(-x[0]);", (3, 4))
    assert len(lb.available()) == n0 + 2 and later.family > user["damped"].family
    b = plan.fit_batch(means, pm, tol=BENCH_TOL).numpy()
    _same_bits(a, b, "after a later plug-in")
