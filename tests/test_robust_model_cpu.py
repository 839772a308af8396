"""The robust-loss device loop, restated in numpy (tests/lm_model_robust.py), against scipy's robust trf --
``scipy.optimize.least_squares(method='trf', x_scale='jac', loss=..., f_scale=...)``, the solver behind
``lsqfit.scipy_least_squares(loss=...)`` (reference src/lsqfit/_scipy.py:77) -- through the oracle; and the kernel's
per-row arithmetic (csrc/lm_kernel.cuh: robust_row) against scipy's own loss and row-scaling functions.

Measured on the 27 NIST problems with three planted outliers, four losses and two f_scale values (216 fits, scipy's
sub-problem iteration): the same convergence flag on all 216 (both stop at maxit on the same two lanczos fits); the
same status on 207 (the other 9 stop one or a few evaluations apart on ftol vs xtol: the last step differs in
rounding between the Cholesky secular-equation solve and scipy's SVD); the same evaluation count on 199 (92 %); the
robust cost within 1.6e-9 relative on every converged fit with the same count (lanczos3, sigma_y = 1e-5 of the
data; 6e-12 on all others).
"""
import copy
import warnings

import numpy as np
import pytest

import lm_model_robust as M
from oracle import dual as D
from oracle.fit import nonlinear_fit as ofit

LOSSES = ("huber", "soft_l1", "cauchy", "arctan")


@pytest.mark.parametrize("loss", LOSSES)
@pytest.mark.parametrize("f_scale", [0.7, 2.0])
def test_robust_row_matches_scipy(loss, f_scale):
    """z in {0, just below 1, 1, just above 1, 1e6} and a spread between, both signs of the residual: C^2 rho, the row
    scale and the scaled residual as scipy's construct_loss_function / scale_for_robust_loss_function compute them,
    including the rows where scipy clips the scale to EPS (cauchy and arctan beyond z = 1)."""
    from scipy.optimize._lsq.common import scale_for_robust_loss_function
    from scipy.optimize._lsq.least_squares import construct_loss_function
    zs = np.array([0.0, 1.0 - 1e-12, 1.0, 1.0 + 1e-12, 1e6, 0.25, 3.0, 50.0])
    r = np.concatenate([np.sqrt(zs), -np.sqrt(zs)]) * f_scale
    lf = construct_loss_function(r.size, loss, f_scale)
    rho = lf(r.copy())
    J = np.ones((r.size, 1))
    Js, fs = scale_for_robust_loss_function(J.copy(), r.copy(), rho.copy())
    c2rho, s, rs = M.robust_row(loss, f_scale, r)
    np.testing.assert_allclose(c2rho, rho[0], rtol=1e-14, atol=0)
    # rho' + 2 z rho'' cancels for large z (soft_l1 at z = 1e6: t^-1/2 - z t^-3/2 = t^-3/2): both sides round it,
    # to ~z eps relative
    np.testing.assert_allclose(s, Js[:, 0], rtol=1e-9, atol=0)
    np.testing.assert_allclose(rs, fs, rtol=1e-9, atol=1e-300)
    cost = 0.5 * np.sum(c2rho)
    assert abs(cost - lf(r.copy(), cost_only=True)) <= 1e-14 * cost
    if loss in ("cauchy", "arctan"):
        clipped = (r / f_scale) ** 2 > 1.0 + 1e-9
        assert clipped.any() and np.all(s[clipped] == np.sqrt(np.finfo(float).eps))


def _outliers(pr):
    """three gross outliers in the data (the rows of test_robust_loss)"""
    pr = copy.deepcopy(pr)
    y, sd = np.array(pr["y"], dtype=float), np.array(pr["ysdev"], dtype=float) * np.ones(len(pr["y"]))
    for k, i in enumerate((1, len(y) // 2, len(y) - 2)):
        y[i] += (12.0 + 5.0 * k) * sd[i] * (-1) ** k
    pr["y"] = y
    return pr


def test_robust_model_matches_scipy_on_nist(nist_problems):
    """Every NIST problem with planted outliers, every loss, two f_scale values: the model's decisions against scipy's
    robust trf from the certified start."""
    same_status = same_nfev = total = 0
    worst = 0.0
    for pr0 in nist_problems:
        pr = _outliers(pr0)
        x = np.array(pr["x"])
        for loss in LOSSES:
            for fs in (1.0, 3.0):
                with warnings.catch_warnings():
                    warnings.simplefilter("ignore")
                    fo = ofit(pr["form"], x[:, None] if x.ndim == 1 else x, pr["y"], np.array(pr["ysdev"]),
                              prior_mean=pr["prior_mean"], prior_cov=np.array(pr["prior_sdev"]), p0=pr["p0"],
                              tol=1e-10, maxit=1000, x_scale="jac", loss=loss, f_scale=fs)
                    chiv = fo._chiv
                    r = M.lm_fit_robust(lambda p: np.asarray(chiv(p)),
                                        lambda p: D.deriv(chiv(D.Dual.variables(p)), p.size),
                                        np.array(pr["p0"], dtype=float), loss, fs, xtol=1e-10, gtol=1e-10, ftol=1e-10)
                res = getattr(fo.fitter_results, "results", fo.fitter_results)
                tag = (pr["name"], loss, fs)
                assert (r["status"] > 0) == (res.status > 0), (tag, r["status"], res.status)
                total += 1
                same_status += r["status"] == res.status
                same_nfev += r["nfev"] == fo.nit
                if r["nfev"] == fo.nit and res.status > 0:
                    assert abs(r["cost"] - res.cost) <= 1e-8 * res.cost, (tag, r["cost"], res.cost)
                    worst = max(worst, abs(r["cost"] - res.cost) / res.cost)
    assert same_status >= 0.95 * total and same_nfev >= 0.9 * total, (same_status, same_nfev, total)
    assert worst < 2e-9, worst
