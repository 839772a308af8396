"""numpy model of the device trust-region loop with a robust loss (csrc/lm_kernel.cuh: fit_one<F, 6>, robust_row).

The kernel runs scipy's ``trf_no_bounds`` with a ``loss_function`` (scipy/optimize/_lsq/trf.py; least_squares.py:
construct_loss_function; common.py: scale_for_robust_loss_function): every chiv row is rescaled by the loss before it
enters J^T J and J^T f, the cost is 1/2 C^2 sum rho((f / C)^2), and the sub-problem is solved by the kernel's Cholesky
secular-equation solvers (tests/lm_model.py, unchanged).  ``robust_row`` restates the kernel's per-row arithmetic.
"""
import numpy as np

import lm_model

LOSS_CODES = {"linear": 0, "huber": 1, "soft_l1": 2, "cauchy": 3, "arctan": 4}
EPS = float(np.finfo(float).eps)


def robust_row(loss, C, r):
    """The kernel's robust_row on an array of residuals -> (C^2 rho(z), s, r rho' / s), z = (r / C)^2."""
    r = np.asarray(r, dtype=float)
    u = r / C
    z = u * u
    if loss == "huber":
        small = z <= 1.0
        sz = np.sqrt(np.where(small, 1.0, z))
        rho0 = np.where(small, z, 2.0 * sz - 1.0)
        rho1 = np.where(small, 1.0, 1.0 / sz)
        rho2 = np.where(small, 0.0, -0.5 * (1.0 / sz) / np.where(small, 1.0, z))
    elif loss == "soft_l1":
        t = 1.0 + z
        st = np.sqrt(t)
        rho0, rho1 = 2.0 * (st - 1.0), 1.0 / st
        rho2 = -0.5 * rho1 / t
    elif loss == "cauchy":
        rho0, rho1 = np.log1p(z), 1.0 / (1.0 + z)
        rho2 = -rho1 * rho1
    elif loss == "arctan":
        rho0, rho1 = np.arctan(z), 1.0 / (z * z + 1.0)
        rho2 = -2.0 * z * rho1 * rho1
    else:
        rho0, rho1, rho2 = z, np.ones_like(z), np.zeros_like(z)
    C2 = C * C
    js = np.maximum(rho1 + 2.0 * (rho2 / C2) * (r * r), EPS)
    s = np.sqrt(js)
    return C2 * rho0, s, r * (rho1 / s)


def lm_fit_robust(fun, jac, x0, loss, f_scale, xtol=1e-8, gtol=1e-10, ftol=1e-10, maxit=1000, device_solver=False):
    """The loop of lm_model.lm_fit (More' scaling) on the rescaled rows and the robust cost.  Returns dict(x, f (true
    residuals), J (rescaled), cost (robust), nfev, status)."""
    def rows(x):
        f = fun(x)
        J = jac(x)
        c2rho, s, fs = robust_row(loss, f_scale, f)
        return f, 0.5 * np.sum(c2rho), s[:, None] * J, fs

    x = np.array(x0, dtype=float)
    f, cost, J, fs = rows(x)
    nfev = 1
    n = J.shape[1]
    g = J.T @ fs
    scale_inv = np.sqrt(np.sum(J ** 2, axis=0))
    scale_inv[scale_inv == 0] = 1
    Delta = np.linalg.norm(x * scale_inv)
    if Delta == 0:
        Delta = 1.0
    alpha = 0.0
    status = None
    while True:
        if np.max(np.abs(g)) < gtol:
            status = 1
        if status is not None or nfev >= maxit:
            break
        d = 1.0 / scale_inv
        A = (J.T @ J) * d[:, None] * d[None, :]
        g_h = d * g
        actual_reduction = -1.0
        gn = {}
        while actual_reduction <= 0 and nfev < maxit:
            if device_solver:
                step_h, alpha, _ = lm_model.solve_tr_device(A, g_h, Delta, alpha, gn)
            else:
                step_h, alpha, _ = lm_model.solve_tr(A, g_h, Delta, alpha)
            predicted_reduction = -(0.5 * step_h @ A @ step_h + g_h @ step_h)
            step = d * step_h
            x_new = x + step
            nfev += 1
            step_h_norm = np.linalg.norm(step_h)
            f_new, cost_new, J_new, fs_new = rows(x_new)
            if not np.isfinite(cost_new):
                Delta = 0.25 * step_h_norm
                continue
            actual_reduction = cost - cost_new
            if predicted_reduction > 0:
                ratio = actual_reduction / predicted_reduction
            elif predicted_reduction == actual_reduction == 0:
                ratio = 1
            else:
                ratio = 0
            Delta_new = Delta
            if ratio < 0.25:
                Delta_new = 0.25 * step_h_norm
            elif ratio > 0.75 and step_h_norm > 0.95 * Delta:
                Delta_new = Delta * 2.0
            ft = actual_reduction < ftol * cost and ratio > 0.25
            xt = np.linalg.norm(step) < xtol * (xtol + np.linalg.norm(x))
            if ft and xt:
                status = 4
            elif ft:
                status = 2
            elif xt:
                status = 3
            if status is not None:
                break
            alpha *= Delta / Delta_new
            Delta = Delta_new
        if actual_reduction > 0:
            x, f, cost, J, fs = x_new, f_new, cost_new, J_new, fs_new
            g = J.T @ fs
            scale_inv = np.maximum(scale_inv, np.sqrt(np.sum(J ** 2, axis=0)))
    if status is None:
        status = 0
    return dict(x=x, f=f, J=J, cost=cost, nfev=nfev, status=status)
