"""The bounded device trust-region loop, restated in numpy (tests/lm_model_bounded.py: lm_fit_bounded), against
scipy's bounded trf -- ``scipy.optimize.least_squares(method='trf', x_scale='jac', bounds=...)``, the solver behind
``lsqfit.scipy_least_squares(bounds=...)`` (reference src/lsqfit/_scipy.py:77) -- through the oracle.

The kernel (csrc/lm_kernel.cuh: fit_one<F, 3>) solves the Coleman-Li sub-problem with the Cholesky secular-equation
solver of the unbounded loop (the Coleman-Li diagonal added next to the Levenberg shift) and restates scipy's
select_step on the warp.  This test shows on the CPU that this reformulation reaches scipy's constrained minimum.
"""
import warnings

import numpy as np
import pytest

import lm_model_bounded
from oracle import dual as D
from oracle.fit import nonlinear_fit as ofit

BOX_PROBLEMS = ("misra1a", "chwirut2", "gauss1", "rat42", "thurber")


def _box(pr):
    """A box around the start and the certified point whose first parameter cannot reach its certified value
    (the box of the single-fit bounds test in test_gpu_parity.py); returns (lb, ub, the cut value)."""
    cert, p0 = np.array(pr["certified"]), np.array(pr["p0"])
    lo = np.minimum(cert, p0) - 0.5 * np.abs(cert - p0) - 1e-3 * np.abs(cert)
    hi = np.maximum(cert, p0) + 0.5 * np.abs(cert - p0) + 1e-3 * np.abs(cert)
    mid = 0.5 * (cert[0] + p0[0])
    if p0[0] < cert[0]:
        hi[0] = mid
    else:
        lo[0] = mid
    return lo, hi, mid


def _cut_box(pr, k):
    """Unbounded but for parameter k, whose bound sits halfway between the start and the certified value."""
    cert, p0 = np.array(pr["certified"]), np.array(pr["p0"])
    lo, hi = np.full(cert.size, -np.inf), np.full(cert.size, np.inf)
    mid = 0.5 * (cert[k] + p0[k])
    if p0[k] < cert[k]:
        hi[k] = mid
    else:
        lo[k] = mid
    return lo, hi, mid


def _compare(pr, lo, hi, device_solver):
    x = np.array(pr["x"])
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        fo = ofit(pr["form"], x[:, None] if x.ndim == 1 else x, pr["y"], np.array(pr["ysdev"]),
                  prior_mean=pr["prior_mean"], prior_cov=np.array(pr["prior_sdev"]), p0=pr["p0"],
                  tol=1e-10, maxit=1000, x_scale="jac", bounds=(lo, hi))
        chiv = fo._chiv
        r = lm_model_bounded.lm_fit_bounded(
            lambda p: np.asarray(chiv(p)), lambda p: D.deriv(chiv(D.Dual.variables(p)), p.size),
            np.array(pr["p0"], dtype=float), lo, hi, xtol=1e-10, gtol=1e-10, ftol=1e-10, maxit=1000,
            device_solver=device_solver)
    assert r["status"] > 0, pr["name"]
    assert np.all(r["x"] >= lo) and np.all(r["x"] <= hi), pr["name"]
    # active set: the same parameters end on (within 1e-6 relative of) the same bound
    def active(x):
        on_lo = np.isfinite(lo) & (np.abs(x - lo) <= 1e-6 * np.maximum(1.0, np.abs(lo)))
        on_hi = np.isfinite(hi) & (np.abs(x - hi) <= 1e-6 * np.maximum(1.0, np.abs(hi)))
        return np.where(on_lo, -1, np.where(on_hi, 1, 0))
    act_m, act_o = active(r["x"]), active(fo.pmean)
    assert np.array_equal(act_m, act_o), (pr["name"], act_m, act_o)
    free = act_o == 0
    dp = np.max(np.abs(r["x"] - fo.pmean)[free] / fo.psdev[free]) if np.any(free) else 0.0
    return r["nfev"], fo.nit, dp, int(np.count_nonzero(act_o))


@pytest.mark.parametrize("device_solver", [False, True])
def test_bounded_model_matches_scipy_on_box_problems(nist_problems, device_solver):
    """The five NIST problems of the single-fit bounds test, with its box.  Measured: the same evaluation counts as
    scipy on all five with either sub-problem iteration, free parameters within 2.6e-15 sdev."""
    worst = 0.0
    for name in BOX_PROBLEMS:
        pr = next(q for q in nist_problems if q["name"] == name)
        lo, hi, mid = _box(pr)
        nfev, nit, dp, nact = _compare(pr, lo, hi, device_solver)
        assert nact >= 1, name
        assert abs(nfev - nit) <= max(4, nit // 10), (name, nfev, nit)
        worst = max(worst, dp)
    assert worst < 1e-5, worst


LANCZOS = ("lanczos1", "lanczos2", "lanczos3")


@pytest.mark.parametrize("device_solver", [False, True])
def test_bounded_model_matches_scipy_on_nist_cut(nist_problems, device_solver):
    """All 27 NIST problems, each with one bound halfway between the start and the certified value of its first
    parameter.  Measured with scipy's sub-problem iteration: identical evaluation counts on all 27, free parameters
    within 2.7e-7 sdev (lanczos1 aside, see test_lm_model_cpu).  With the kernel's (coarser secular tolerance) the
    counts stay within the slack of test_lm_model_cpu (mgh10: 71 vs 35) and the end points within 3.3e-4 sdev
    (mgh17, 379 evaluations along a flat valley; every problem but mgh17 and the lanczos family: 2.2e-7); the
    lanczos family (sigma_y down to 9e-14) ends 2e-4 ... 9e-3 sdev apart and is left out of that bar."""
    worst = 0.0
    for pr in nist_problems:
        lo, hi, mid = _cut_box(pr, 0)
        nfev, nit, dp, nact = _compare(pr, lo, hi, device_solver)
        if device_solver:
            assert nfev <= 3 * nit + 5, (pr["name"], nfev, nit)
            if pr["name"] not in LANCZOS:
                worst = max(worst, dp)
        else:
            assert abs(nfev - nit) <= max(4, nit // 10), (pr["name"], nfev, nit)
            if pr["name"] != "lanczos1":          # sigma_y = 9e-14: rounding of exp() is amplified 1e13-fold
                worst = max(worst, dp)
    assert worst < (1e-3 if device_solver else 1e-5), worst
