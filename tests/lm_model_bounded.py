"""Host model (numpy) of the DEVICE trust-region loop WITH BOUND CONSTRAINTS -- test infrastructure.

The bounded driver of the one-warp kernel (csrc/lm_kernel.cuh: fit_one<F, 3>) restates scipy's trf_bounds
(scipy/optimize/_lsq/trf.py: trf_bounds, select_step; common.py: CL_scaling_vector, step_size_to_bound,
intersect_trust_region, minimize_quadratic_1d, make_strictly_feasible) around the unbounded device loop of
tests/lm_model.py: the same Cholesky secular-equation solvers, on the scaled normal matrix plus the Coleman-Li
diagonal.  This file restates that loop in numpy; it is never imported by lsqfit_b200.
"""
import numpy as np

from lm_model import solve_tr, solve_tr_device, solve_tr_dual


def make_strictly_feasible(x, lb, ub, rstep=1e-10):
    xn = np.array(x, dtype=float)
    if rstep == 0:
        lo, up = x <= lb, x >= ub
        xn[lo] = np.nextafter(lb[lo], ub[lo])
        xn[up] = np.nextafter(ub[up], lb[up])
    else:
        ld, ud = x - lb, ub - x
        lt, ut = rstep * np.maximum(1, np.abs(lb)), rstep * np.maximum(1, np.abs(ub))
        lo = np.isfinite(lb) & (ld <= np.minimum(ud, lt))
        up = np.isfinite(ub) & (ud <= np.minimum(ld, ut))
        xn[lo] = lb[lo] + rstep * np.maximum(1, np.abs(lb[lo]))
        xn[up] = ub[up] - rstep * np.maximum(1, np.abs(ub[up]))
    tight = (xn < lb) | (xn > ub)
    xn[tight] = 0.5 * (lb[tight] + ub[tight])
    return xn


def cl_scaling_vector(x, g, lb, ub):
    v, dv = np.ones_like(x), np.zeros_like(x)
    m = (g < 0) & np.isfinite(ub)
    v[m] = ub[m] - x[m]
    dv[m] = -1
    m = (g > 0) & np.isfinite(lb)
    v[m] = x[m] - lb[m]
    dv[m] = 1
    return v, dv


def step_size_to_bound(x, s, lb, ub):
    """(min over s_i != 0 of the step to the box, hits = sign(s) where that minimum is reached)"""
    steps = np.full_like(x, np.inf)
    nz = s != 0
    with np.errstate(over="ignore", invalid="ignore", divide="ignore"):
        steps[nz] = np.maximum((lb - x)[nz] / s[nz], (ub - x)[nz] / s[nz])
    m = np.min(steps)
    return m, np.equal(steps, m) * np.sign(s)


def intersect_trust_region(x, s, Delta):
    a, b, c = s @ s, x @ s, x @ x - Delta ** 2
    d = np.sqrt(max(b * b - a * c, 0.0))
    q = -(b + np.copysign(d, b))
    t1, t2 = q / a, c / q
    return (t1, t2) if t1 < t2 else (t2, t1)


def minimize_quadratic_1d(a, b, lb, ub, c=0.0):
    t = [lb, ub]
    if a != 0:
        e = -0.5 * b / a
        if lb < e < ub:
            t.append(e)
    t = np.asarray(t)
    y = t * (a * t + b) + c
    i = int(np.argmin(y))
    return t[i], y[i]


def select_step(x, Ah, gh, p_h, d, Delta, theta, lb, ub):
    """The trust-region step if it stays inside the box, else the best of: that step cut back to the box, its
    reflection off the box (1-d quadratic minimisation), the cut-back anti-gradient step -- compared on
    q(s) = 1/2 s^T Ah s + gh^T s, Ah = d J^T J d + diag(diag_h).  Returns (step, step_h, predicted reduction)."""
    q = lambda s: 0.5 * s @ Ah @ s + gh @ s
    p = d * p_h
    if np.all((x + p >= lb) & (x + p <= ub)):
        return p, p_h, -q(p_h)
    p_stride, hits = step_size_to_bound(x, p, lb, ub)
    r_h = np.where(hits != 0, -p_h, p_h)
    r = d * r_h
    p, p_h = p * p_stride, p_h * p_stride
    _, to_tr = intersect_trust_region(p_h, r_h, Delta)
    to_bound, _ = step_size_to_bound(x + p, r, lb, ub)
    r_stride = min(to_bound, to_tr)
    if r_stride > 0:
        r_lo = (1 - theta) * p_stride / r_stride
        r_up = theta * to_bound if r_stride == to_bound else to_tr
    else:
        r_lo, r_up = 0.0, -1.0
    if r_lo <= r_up:
        Ar = Ah @ r_h
        a, b, c = 0.5 * r_h @ Ar, gh @ r_h + p_h @ Ar, q(p_h)
        t, r_value = minimize_quadratic_1d(a, b, r_lo, r_up, c=c)
        r_h = r_h * t + p_h
        r = d * r_h
    else:
        r_value = np.inf
    p, p_h = p * theta, p_h * theta
    p_value = q(p_h)
    ag_h = -gh
    ag = d * ag_h
    to_tr = Delta / np.linalg.norm(ag_h)
    to_bound, _ = step_size_to_bound(x, ag, lb, ub)
    ag_stride = theta * to_bound if to_bound < to_tr else to_tr
    t, ag_value = minimize_quadratic_1d(0.5 * ag_h @ Ah @ ag_h, gh @ ag_h, 0, ag_stride)
    ag_h, ag = ag_h * t, ag * t
    if p_value < r_value and p_value < ag_value:
        return p, p_h, -p_value
    if r_value < p_value and r_value < ag_value:
        return r, r_h, -r_value
    return ag, ag_h, -ag_value


def lm_fit_bounded(fun, jac, x0, lb, ub, xtol=1e-8, gtol=1e-10, ftol=1e-10, maxit=1000, scaler="more",
                   device_solver=False, stats=None, dual=False):
    """The bounded device loop (fit_kernel<F, 3>): lm_model.lm_fit with scipy's trf_bounds changes -- the start made
    strictly feasible, the gtol test on |g v|_inf, the scaling d = sqrt(v) / scale_inv, the Coleman-Li diagonal in the
    sub-problem, select_step, strictly feasible trial points.  x0 must lie in the box [lb, ub].
    Returns dict(x, f, J, nfev, status, nfac)."""
    x = np.array(x0, dtype=float)
    lb = np.broadcast_to(np.asarray(lb, dtype=float), x.shape)
    ub = np.broadcast_to(np.asarray(ub, dtype=float), x.shape)
    x = make_strictly_feasible(x, lb, ub)
    f = fun(x)
    nfev = 1
    J = jac(x)
    m, n = J.shape
    cost = 0.5 * f @ f
    g = J.T @ f
    if scaler == "more":
        scale_inv = np.sqrt(np.sum(J ** 2, axis=0))
        scale_inv[scale_inv == 0] = 1
    else:
        scale_inv = np.ones(n)
    v, dv = cl_scaling_vector(x, g, lb, ub)
    v[dv != 0] *= scale_inv[dv != 0]
    Delta = np.linalg.norm(x * scale_inv / v ** 0.5)
    if Delta == 0:
        Delta = 1.0
    alpha = 0.0
    status = None
    nfac = 0
    lm_state = {}
    while True:
        v, dv = cl_scaling_vector(x, g, lb, ub)
        g_norm = np.max(np.abs(g * v))
        if g_norm < gtol:
            status = 1
        if status is not None or nfev >= maxit:
            break
        v[dv != 0] *= scale_inv[dv != 0]
        d = v ** 0.5 / scale_inv
        diag_h = g * dv / scale_inv                      # Coleman-Li diagonal of the sub-problem
        theta = max(0.995, 1 - g_norm)
        A = (J.T @ J) * d[:, None] * d[None, :] + np.diag(diag_h)
        g_h = d * g
        actual_reduction = -1.0
        gn = {}
        while actual_reduction <= 0 and nfev < maxit:
            if dual:
                step_h, alpha, k = solve_tr_dual(A, g_h, Delta, alpha, gn, lm_state, stats)
            elif device_solver:
                step_h, alpha, k = solve_tr_device(A, g_h, Delta, alpha, gn, stats)
            else:
                step_h, alpha, k = solve_tr(A, g_h, Delta, alpha)
            nfac += k
            step, step_h, predicted_reduction = select_step(x, A, g_h, step_h, d, Delta, theta, lb, ub)
            x_new = make_strictly_feasible(x + step, lb, ub, rstep=0)
            f_new = fun(x_new)
            nfev += 1
            step_h_norm = np.linalg.norm(step_h)
            if not np.all(np.isfinite(f_new)):
                Delta = 0.25 * step_h_norm
                continue
            cost_new = 0.5 * f_new @ f_new
            actual_reduction = cost - cost_new
            # update_tr_radius
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
            # check_termination
            step_norm = np.linalg.norm(step)
            ft = actual_reduction < ftol * cost and ratio > 0.25
            xt = step_norm < xtol * (xtol + np.linalg.norm(x))
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
            x, f, cost = x_new, f_new, cost_new
            J = jac(x)
            g = J.T @ f
            if scaler == "more":
                scale_inv = np.maximum(scale_inv, np.sqrt(np.sum(J ** 2, axis=0)))
    if status is None:
        status = 0
    return dict(x=x, f=f, J=J, nfev=nfev, status=status, nfac=nfac)
