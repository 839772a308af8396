"""Parameter distributions on the device (fit_kernel<F, 5>, resjac_trans_kernel, the single-fit path): fits whose
model sees q = T(p) for lsqfit's log(k), sqrt(k) and uniform prior keys, against the oracle fitting f(x, T(p)) with the
chain-rule gradient, against a plug-in that takes exp of its own energies, in batches, and the refusals.
Needs a GPU (pytest -m gpu)."""
import os
import warnings

import numpy as np
import pytest

from parity_util import TIGHT, exact_minimum, rel_cov
from lsqfit_b200 import configs
from lsqfit_b200 import pdist as P
from oracle import dual as D
from oracle.models import multiexp

pytestmark = pytest.mark.gpu


def t_dual(code, lo, hi, p):
    if isinstance(p, D.Dual):
        q, dq = P.transform(code, lo, hi, p.v)
        return D.Dual(q, dq[:, None] * p.d)
    return P.transform(code, lo, hi, p)[0]


def problem(K, cov="dense", dist="mixed", seed=11):
    """Correlator data (configs.correlator) with a prior in fit space: log(E_k) = log(0.5 k)(0.3); with dist='mixed'
    also sqrt(a_0) = sqrt(0.5)(0.3) and a_1 uniform on (0, 2) (prior 0(1), gvar's idiom)."""
    cfg = configs.correlator(K)
    ny = cfg["ny"]
    rng = np.random.default_rng(seed)
    ycov = cfg["ycov"].copy()
    if cov == "block":
        h = ny // 2
        ycov[:h, h:] = 0.0
        ycov[h:, :h] = 0.0
    y = cfg["f"] + np.linalg.cholesky(ycov) @ rng.standard_normal(ny)
    yerr = np.sqrt(np.diag(ycov)) if cov == "diag" else ycov
    pm = cfg["prior_mean"].copy()
    ps = cfg["prior_sdev"].copy()
    pdist = [None] * K + ["log"] * K
    pm[K:], ps[K:] = np.log(cfg["ptrue"][K:]), 0.3
    if dist == "mixed":
        pdist[0] = "sqrt"
        pm[0], ps[0] = np.sqrt(0.5), 0.3
        pdist[1] = ("uniform", 0.0, 2.0)
        pm[1], ps[1] = 0.0, 1.0
    return dict(x=cfg["x"], y=y, yerr=yerr, ycov=ycov, pm=pm, ps=ps, pdist=pdist, K=K, ny=ny,
                codes=P.codes(pdist, 2 * K))


def model(pr):
    code, lo, hi = pr["codes"]
    return lambda x, p: multiexp(x, t_dual(code, lo, hi, p))


def device_fit(pr, svdcut=1e-8, **kw):
    import lsqfit_b200 as lb
    args = dict(tol=TIGHT, maxit=2000, polish=100)
    args.update(kw)
    return lb.nonlinear_fit(data=(pr["x"], pr["y"], pr["yerr"]), prior=(pr["pm"], pr["ps"]), fcn="multiexp",
                            pdist=pr["pdist"], svdcut=svdcut, **args)


def oracle_fit(pr, svdcut=1e-8, tol=TIGHT, **kw):
    from oracle.fit import nonlinear_fit as ofit
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return ofit(model(pr), pr["x"], pr["y"], pr["yerr"], prior_mean=pr["pm"], prior_cov=pr["ps"], svdcut=svdcut,
                    tol=tol, maxit=2000, x_scale="jac", **kw)


def logGBF_at(ofit, J, f):
    """logGBF (src/lsqfit/__init__.py:720-725) at the exact minimum"""
    ld = np.linalg.slogdet(J.T @ J)[1]
    return 0.5 * (-ld - ofit.yp_pdf.logdet - f @ f - ofit.dof * np.log(2 * np.pi))


CASES = [(K, cov, svdcut) for K in (4, 8) for cov in ("dense", "block", "diag") for svdcut in (1e-8, 0.05, -0.01)]


@pytest.mark.parametrize("K,cov,svdcut", CASES)
def test_central_fit_against_oracle(K, cov, svdcut):
    pr = problem(K, cov)
    fit = device_fit(pr, svdcut)
    fo = oracle_fit(pr, svdcut)
    xe, f, J, cov_e = exact_minimum(fo)
    sd = np.sqrt(np.diag(cov_e))
    assert fit.error is None
    assert np.max(np.abs(fit.pmean - xe) / sd) <= 1e-8
    assert abs(fit.chi2 - f @ f) <= 1e-9 * (f @ f)
    assert rel_cov(fit.cov, cov_e) <= 1e-8
    lg = logGBF_at(fo, J, f)
    assert abs(fit.logGBF - lg) <= 1e-8 * abs(lg)
    assert fit.dof == fo.dof and fit.svdn == fo.svdn


def test_log_only_against_oracle():
    pr = problem(4, "dense", dist="log")
    fit = device_fit(pr)
    xe, f, J, cov_e = exact_minimum(oracle_fit(pr))
    assert np.max(np.abs(fit.pmean - xe) / np.sqrt(np.diag(cov_e))) <= 1e-8
    assert rel_cov(fit.cov, cov_e) <= 1e-8


def test_nit_and_stopping_criterion_follow_the_oracle():
    """The trust-region decisions are scipy's: at the default tolerances the evaluation counts and stopping criteria of
    the central fits agree with the oracle's (rounding may move a stopping test by one evaluation on a few cases)."""
    same = n = 0
    for K, cov, svdcut in CASES:
        pr = problem(K, cov)
        fit = device_fit(pr, svdcut, tol=1e-10, polish=0)
        fo = oracle_fit(pr, svdcut, tol=1e-10)
        assert fit.stopping_criterion > 0 and fo.stopping_criterion > 0
        same += int(fit.nit == fo.nit and fit.stopping_criterion == fo.stopping_criterion)
        n += 1
    assert same >= (2 * n) // 3, (same, n)


@pytest.fixture(scope="module")
def plugin_cache(tmp_path_factory):
    old = os.environ.get("B200LM_FUNCTOR_CACHE")
    os.environ["B200LM_FUNCTOR_CACHE"] = str(tmp_path_factory.mktemp("functors"))
    yield
    if old is None:
        del os.environ["B200LM_FUNCTOR_CACHE"]
    else:
        os.environ["B200LM_FUNCTOR_CACHE"] = old


EXP_ENERGIES = """
const double t = x[0];
T s = b[0] * exp(-(exp(b[4]) * t));
s = s + b[1] * exp(-(exp(b[5]) * t));
s = s + b[2] * exp(-(exp(b[6]) * t));
s = s + b[3] * exp(-(exp(b[7]) * t));
return s;
"""


def test_log_codes_against_a_plugin_taking_exp(plugin_cache):
    """multiexp with log(E) codes = a body-form plug-in that takes exp of its own energy parameters, plain keys."""
    import lsqfit_b200 as lb
    pr = problem(4, "dense", dist="log")
    fcn = lb.cuda_functor("pdist_expE", EXP_ENERGIES, 8, host=lambda x, p: multiexp(x, np.concatenate(
        [p[:4], np.exp(p[4:])])))
    fit = device_fit(pr)
    ref = lb.nonlinear_fit(data=(pr["x"], pr["y"], pr["yerr"]), prior=(pr["pm"], pr["ps"]), fcn=fcn, svdcut=1e-8,
                           tol=TIGHT, maxit=2000, polish=100)
    sd = np.sqrt(np.diag(ref.cov))
    assert np.max(np.abs(fit.pmean - ref.pmean) / sd) <= 1e-9
    assert abs(fit.chi2 - ref.chi2) <= 1e-10 * ref.chi2
    assert rel_cov(fit.cov, ref.cov) <= 1e-10


def test_functor_plugin_with_codes_is_the_builtin(plugin_cache):
    """A functor-form plug-in of the built-in model has MODE 5 too: the same bits as the built-in model."""
    import lsqfit_b200 as lb
    pr = problem(4, "dense")
    fcn = lb.cuda_functor("pdist_multiexp", "template <int NP> using Model = MultiExp<NP / 2>;", 8, host=multiexp,
                          form="functor")
    fit = device_fit(pr)
    fp = lb.nonlinear_fit(data=(pr["x"], pr["y"], pr["yerr"]), prior=(pr["pm"], pr["ps"]), fcn=fcn, svdcut=1e-8,
                          pdist=pr["pdist"], tol=TIGHT, maxit=2000, polish=100)
    assert np.array_equal(fit.pmean, fp.pmean) and np.array_equal(fit.cov, fp.cov) and fit.chi2 == fp.chi2
    a = fit.bootstrapped_fits(300, seed=5).arrays()
    b = fp.bootstrapped_fits(300, seed=5).arrays()
    for k in ("x", "chi2", "cov", "nit", "status"):
        assert np.array_equal(a[k], b[k]), k


def test_bootstrap_and_simulated_batches():
    from oracle.fit import nonlinear_fit as ofit
    from oracle.whiten import PDF as OPDF
    pr = problem(4, "dense")
    fit = device_fit(pr)
    ny = pr["ny"]
    n = 2000
    bf = fit.bootstrapped_fits(n, seed=7, tol=TIGHT, polish=100)
    out = bf.arrays()
    assert len(bf) == n and np.all(out["status"] > 0)
    means = fit.bootstrap_means(n, seed=7).cpu().numpy()
    C = np.zeros((ny + 8, ny + 8))
    C[:ny, :ny] = pr["ycov"]
    C[ny:, ny:] = np.diag(pr["ps"] ** 2)
    opdf = OPDF(np.concatenate([pr["y"], pr["pm"]]), C, svdcut=1e-8)
    dev, ref = [], []
    for b in range(0, n, n // 100):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            fo = ofit(model(pr), pr["x"], means[b, :ny], prior_mean=means[b, ny:], _yp_pdf=opdf, p0=fit.pmean,
                      tol=TIGHT, maxit=2000, x_scale="jac")
        # The stationary point, found independently: Newton's method on the oracle's analytic gradient J^T f with a
        # central-difference Hessian (undamped Gauss-Newton, as in exact_minimum, diverges on some of these copies: the
        # residual curvature of the transformed model is too large for it)
        x = out["x"][b]
        xs, cov_s = newton_minimum(fo._chiv, fo.pmean, fo.psdev)
        fs = np.asarray(fo._chiv(xs))
        sd = np.sqrt(np.diag(cov_s))
        dev.append(float(np.max(np.abs(x - xs) / sd)))
        ref.append(float(np.max(np.abs(fo.pmean - xs) / sd)))
        assert abs(out["chi2"][b] - fs @ fs) <= 1e-9 * (fs @ fs)
        # the device's chi2 and covariance at its own answer: the oracle's chiv and (J^T J)^-1 there
        f = np.asarray(fo._chiv(x))
        J = D.deriv(fo._chiv(D.Dual.variables(x)), x.size)
        _, sv, VT = np.linalg.svd(J, full_matrices=False)
        assert abs(out["chi2"][b] - f @ f) <= 1e-12 * (f @ f)
        assert rel_cov(out["cov"][b], (VT.T / sv ** 2) @ VT) <= 1e-8
    # On the copies where undamped Gauss-Newton does not converge, the polish (Gauss-Newton steps accepted while the
    # Newton decrement falls) stops where the trust-region loop left the fit, a distance of order sqrt(eps chi2) from the
    # stationary point -- where the reference's own solver stops; as in the untransformed parity tests, the device's
    # worst case must not exceed 3x the reference's (DESIGN 8.4)
    dev, ref = np.array(dev), np.array(ref)
    print("distance to the stationary point, sdev: device worst %.2e, oracle worst %.2e, device copies above 1e-8: "
          "%d of %d" % (dev.max(), ref.max(), int(np.sum(dev > 1e-8)), dev.size))
    assert dev.max() <= max(1e-8, 3 * ref.max()), (dev.max(), ref.max())
    # simulated data: f(x, T(pexact)) plus the bootstrap noise
    pexact = fit.pmean + 0.1 * fit.psdev
    sm, pe = fit.simulated_means(50, pexact=pexact, seed=3)
    bm = fit.bootstrap_means(50, seed=3)
    noise = (bm - torch_tensor(fit.yp_pdf.mean, bm))[:, :ny]
    fx = multiexp(pr["x"], P.transform(*pr["codes"], pexact)[0])
    got = (sm[:, :ny] - noise).cpu().numpy()
    assert np.max(np.abs(got - fx[None, :]) / np.abs(fx)[None, :]) < 1e-12
    assert np.array_equal(sm[:, ny:].cpu().numpy(), np.broadcast_to(fit.yp_pdf.mean[ny:], (50, 8)))
    sf = fit.simulated_fits(500, pexact=pexact, seed=3)
    a = sf.arrays()
    assert np.all(a["status"] > 0)
    assert np.median(np.abs(a["x"] - pexact) / fit.psdev) < 2.0


def newton_minimum(chiv, x0, sd, iters=40):
    """(x, (J^T J)^-1 at x) at the stationary point of |chiv|^2 next to x0: Newton steps on the analytic gradient
    J^T f with the Hessian from central differences of that gradient (its error slows the convergence, it does not move
    the fixed point g = 0)"""
    def grad(x):
        r = chiv(D.Dual.variables(x))
        J = D.deriv(r, x.size)
        return J.T @ D.value(r), J
    x = np.array(x0, dtype=float)
    for _ in range(iters):
        g, J = grad(x)
        H = np.empty((x.size, x.size))
        for j in range(x.size):
            e = np.zeros(x.size)
            e[j] = 1e-5 * sd[j]
            H[:, j] = (grad(x + e)[0] - grad(x - e)[0]) / (2 * e[j])
        dx = -np.linalg.solve(0.5 * (H + H.T), g)
        x = x + dx
        if np.max(np.abs(dx) / sd) < 1e-14:
            break
    J = grad(x)[1]
    _, sv, VT = np.linalg.svd(J, full_matrices=False)
    return x, (VT.T / sv ** 2) @ VT


def torch_tensor(a, like):
    import torch
    return torch.as_tensor(np.asarray(a, dtype=float)).to(like.device)[None, :]


def test_derivatives_against_oracle():
    """fit.J / residual_jacobian = the oracle's chiv Jacobian of f(x, T(p)) with the same whitening; fit.D and fit.p =
    the oracle's D and D C D^T."""
    from oracle.chiv import Chiv, Chivw
    pr = problem(4, "dense")
    fit = device_fit(pr)
    fcn = lambda p: multiexp(pr["x"], t_dual(*pr["codes"], p))
    ch, chw = Chiv(fit.yp_pdf, fcn, False), Chivw(fit.yp_pdf, fcn, False)
    p = fit.pmean
    Jo = D.deriv(ch(D.Dual.variables(p)), p.size)
    fo = np.asarray(ch(p))
    for J in (fit.J, fit._chiv.jacobian(p)):
        assert np.max(np.abs(J - Jo)) <= 1e-12 * np.max(np.abs(Jo))
    assert np.max(np.abs(fit._chiv(p) - fo)) <= 1e-12 * np.max(np.abs(fo))
    Do = fit.cov @ D.deriv(chw(D.Dual.variables(p)), p.size).T
    assert np.max(np.abs(fit.D - Do)) <= 1e-10 * np.max(np.abs(Do))
    assert rel_cov(fit.p[1], Do @ fit.yp_pdf.cov @ Do.T) <= 1e-8


@pytest.mark.parametrize("cov", ["dense", "diag"])
def test_single_fit_path(cov):
    """fitter='b200_dense' with codes (diag: np = 8, the one-pass normal_diag kernel with J^T J, J^T r scaled by T')
    against the oracle."""
    pr = problem(4, cov)
    fit = device_fit(pr, fitter="b200_dense")
    xe, f, J, cov_e = exact_minimum(oracle_fit(pr))
    sd = np.sqrt(np.diag(cov_e))
    assert fit.error is None
    assert np.max(np.abs(fit.pmean - xe) / sd) <= 1e-7
    assert abs(fit.chi2 - f @ f) <= 1e-9 * (f @ f)
    assert rel_cov(fit.cov, cov_e) <= 1e-7
    # fit.D and fit.p from the single-fit path's propagation (its J carries T' through the scaled model rows)
    from oracle.chiv import Chivw
    fcn = lambda p: multiexp(pr["x"], t_dual(*pr["codes"], p))
    Do = fit.cov @ D.deriv(Chivw(fit.yp_pdf, fcn, False)(D.Dual.variables(fit.pmean)), fit.pmean.size).T
    assert np.max(np.abs(fit.D - Do)) <= 1e-8 * np.max(np.abs(Do))
    assert rel_cov(fit.p[1], Do @ fit.yp_pdf.cov @ Do.T) <= 1e-8


def test_single_fit_path_robust_loss():
    """codes with a robust loss (the single-fit path) against scipy least_squares on a chiv that applies T itself."""
    from scipy.optimize import least_squares
    pr = problem(4, "diag")
    fit = device_fit(pr, loss="huber", f_scale=1.5, tol=(1e-12, 1e-12, 1e-12), polish=0)
    x = pr["x"]

    def chiv(p):
        q = P.transform(*pr["codes"], p)[0]
        return np.concatenate([(multiexp(x, q) - pr["y"]) / pr["yerr"], (p - pr["pm"]) / pr["ps"]])

    def jac(p):
        q, dq = P.transform(*pr["codes"], p)
        G = D.deriv(multiexp(x, D.Dual.variables(q)), p.size) * dq[None, :]
        return np.concatenate([G / pr["yerr"][:, None], np.diag(1.0 / pr["ps"])])
    r = least_squares(chiv, pr["pm"], jac=jac, method="trf", x_scale="jac", loss="huber", f_scale=1.5,
                      xtol=1e-12, ftol=1e-12, gtol=1e-12, max_nfev=2000)
    assert np.max(np.abs(fit.pmean - r.x) / fit.psdev) <= 1e-6


def test_all_plain_codes_are_todays_fit():
    import lsqfit_b200 as lb
    pr = problem(8, "dense")
    args = dict(data=(pr["x"], pr["y"], pr["yerr"]), prior=(pr["pm"], pr["ps"]), fcn="multiexp", svdcut=1e-8)
    f0 = lb.nonlinear_fit(**args)
    f1 = lb.nonlinear_fit(pdist=[None] * 16, **args)
    assert f1.pdist is None
    assert np.array_equal(f0.pmean, f1.pmean) and np.array_equal(f0.cov, f1.cov)
    a = f0.bootstrapped_fits(500, seed=1).arrays()
    b = f1.bootstrapped_fits(500, seed=1).arrays()
    for k in ("x", "chi2", "cov", "nit", "status"):
        assert np.array_equal(a[k], b[k]), k
    # the C3 shape runs a team of two by default; with codes, one warp per fit
    f2 = device_fit(problem(8, "dense"))
    f2.bootstrapped_fits(64, seed=1)
    assert f2._spec.plan(0).last_team() == 1


def test_refusals():
    import lsqfit_b200 as lb
    from lsqfit_b200 import _cabi
    from lsqfit_b200.engine import Plan
    pr = problem(4, "dense")
    fit = device_fit(pr)
    for k in (2, 4, 32, "wave"):
        with pytest.raises(ValueError, match="parameter distributions"):
            fit.bootstrapped_fits(10, seed=1, kernel=k)
    with pytest.raises(ValueError, match="not built for window scans"):
        fit.window_fits(np.ones((2, pr["ny"]), dtype=bool))
    with pytest.raises(ValueError, match="parameter distributions"):
        device_fit(pr, bounds=(-np.inf, np.inf))
    with pytest.raises(ValueError, match="parameter distributions"):
        device_fit(pr, policy="gsl")
    with pytest.raises(ValueError, match="parameter distributions"):
        device_fit(pr, fitter="b200_dense", bounds=(-10.0, 10.0))
    with pytest.raises(ValueError, match="parameter distributions"):
        fit.bootstrapped_fits(10, seed=1, bounds=(-10.0, 10.0))
    # the C ABI
    ny = pr["ny"]
    plan = Plan("multiexp", 8, ny, pr["x"], fit.yp_pdf.i_invwgts)
    lo, hi = np.zeros(8), np.ones(8)

    def einval(call, match):
        with pytest.raises(_cabi.B200LMError, match=match) as e:
            call()
        assert e.value.code == _cabi.EINVAL
    for bad in (5, -1):
        einval(lambda: plan.set_param_dist(np.array([0] * 7 + [bad]), lo, hi), "unknown distribution code")
    for a, b in ((1.0, 1.0), (2.0, 1.0), (0.0, np.inf), (np.nan, 1.0)):
        l2, h2 = lo.copy(), hi.copy()
        l2[3], h2[3] = a, b
        einval(lambda: plan.set_param_dist(np.array([0, 0, 0, 3, 1, 1, 1, 1]), l2, h2), "uniform")
    code = pr["codes"][0]
    plan.set_param_dist(code, pr["codes"][1], pr["codes"][2])
    h = plan._h
    lb_, ub_ = np.full(8, -10.0), np.full(8, 10.0)
    einval(lambda: _cabi.check(_cabi.lib.b200lm_set_bounds(h, lb_.ctypes.data, ub_.ctypes.data), h), "bounds")
    einval(lambda: _cabi.check(_cabi.lib.b200lm_set_policy(h, 1), h), "GSL")
    from lsqfit_b200.windows import window_weights
    desc = window_weights([np.arange(ny + 8)], [fit.yp_pdf.i_invwgts])
    einval(lambda: plan.set_windows(desc), "window")
    mean = fit._spec.mean
    for team in (2, 4, 32):
        plan.set_team(team)
        einval(lambda: plan.fit_batch(mean, fit.pmean), "one warp per fit")
    plan.set_team(0)
    out = plan.fit_batch(mean, fit.pmean, tol=TIGHT, maxit=2000, polish=100).numpy()
    assert plan.last_team() == 1 and np.max(np.abs(out["x"][0] - fit.pmean) / fit.psdev) <= 1e-8
    plan.set_param_dist()                                   # cleared: bounds and the GSL policy are allowed again
    _cabi.check(_cabi.lib.b200lm_set_policy(h, 1), h)
    einval(lambda: plan.set_param_dist(code, pr["codes"][1], pr["codes"][2]), "GSL")
    _cabi.check(_cabi.lib.b200lm_set_policy(h, 0), h)
    _cabi.check(_cabi.lib.b200lm_set_bounds(h, lb_.ctypes.data, ub_.ctypes.data), h)
    einval(lambda: plan.set_param_dist(code, pr["codes"][1], pr["codes"][2]), "bounds")
    _cabi.check(_cabi.lib.b200lm_set_bounds(h, None, None), h)
    sp = Plan("multiexp", 8, ny, pr["x"], None, nslot=2)
    einval(lambda: sp.set_param_dist(code, pr["codes"][1], pr["codes"][2]), "fit sets")
    with pytest.raises(ValueError, match="not built for fit sets"):
        lb.fit_set([(pr["x"], pr["y"], pr["yerr"])] * 2, prior=(pr["pm"], pr["ps"]), fcn="multiexp", pdist=pr["pdist"])
