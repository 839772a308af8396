"""One LARGE fit spread over the whole GPU (BASELINE config 5: 2000 params x 5000 correlated data).

The batched engine (engine.py / csrc/lm_kernel.cuh) gives one warp to each fit and keeps J^T J in
registers; that stops making sense when a single Jacobian is 5000 x 2000.  ``DenseFit`` runs the
same pipeline -- whiten (reference src/lsqfit/__init__.py:1895-1900) -> residual + Jacobian
(src/lsqfit/_utilities.pyx:65-94) -> trust-region Levenberg-Marquardt with the decisions of scipy's
unbounded TRF (the solver behind src/lsqfit/_scipy.py:156-161) -> covariance and fit.p propagation
(src/lsqfit/_scipy.py:171-175, src/lsqfit/__init__.py:897-922) -- with every O(n^3) / O(n^2) step
on our own kernels through the C ABI:

    whitening              b200lm_whiten      (block-Jacobi eigensolver, csrc/whiten_large.cu)
    model rows [G|delta]   b200lm_model_rows (any registered functor) / b200lm_multiexp_dense (any number of terms)
    uncorrelated data      b200lm_normal_diag (J^T J, J^T r, r^T r in one pass over millions of rows)
    W.G, J^T J, J^T f, ... b200lm_dgemm       (FP64 DMMA GEMM)
    chol(d J^T J d + aI)   b200lm_potrf       (blocked, DMMA trailing updates)
    secular-equation solves, (J^T J)^-1        b200lm_trsm

The trust-region control flow (a few dozen scalar decisions per iteration) runs on the host; torch
is used for buffers and for O(n) / O(n^2) element-wise glue only.  There is no CPU fallback.
"""
import ctypes as C
import time

import numpy as np
import torch

from . import _cabi
from .engine import STOPPING_CRITERION, normalize_tol
from .whiten import PDF


class _LA(object):
    """Thin torch-tensor wrappers over the dense C-ABI entry points."""

    def __init__(self, device):
        if not torch.cuda.is_available():
            raise RuntimeError("lsqfit_b200.dense: no CUDA device visible; there is no CPU fallback")
        self.device = int(device)
        self.tdev = torch.device("cuda", self.device)
        self.launches = 0

    def stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.tdev).cuda_stream)

    def empty(self, *shape):
        return torch.empty(shape, dtype=torch.float64, device=self.tdev)

    def gemm(self, transA, transB, M, N, K, alpha, A, lda, B, ldb, beta, Cm, ldc):
        _cabi.check(_cabi.lib.b200lm_dgemm(self.device, int(transA), int(transB), 1, M, N, K, float(alpha),
                                           A.data_ptr(), 0, lda, B.data_ptr(), 0, ldb, float(beta),
                                           Cm.data_ptr(), 0, ldc, self.stream()))
        self.launches += 1

    def mm(self, A, B, transA=False, transB=False, out=None, alpha=1.0, beta=0.0):
        """out = alpha * op(A) . op(B) + beta * out for contiguous 2-D (or 1-D = column) tensors."""
        A2 = A if A.dim() == 2 else A.unsqueeze(1)
        B2 = B if B.dim() == 2 else B.unsqueeze(1)
        M, K = (A2.shape[1], A2.shape[0]) if transA else A2.shape
        N = B2.shape[0] if transB else B2.shape[1]
        assert (B2.shape[1] if transB else B2.shape[0]) == K
        if out is None:
            out = self.empty(M, N) if (B.dim() == 2 or transB) else self.empty(M)
        if transA and not transB and M <= 128 and N <= 128 and K >= 65536:
            # A^T B with a small result and a very long contraction (J^T J of a fit with a handful of parameters and
            # millions of rows): one output tile would leave the whole sum to ONE CTA.  Split K over the batch
            # dimension of b200lm_dgemm -- chunk c of A and B starts c * Kc rows further down -- and add the
            # partial products in a fixed order (deterministic).
            Kc = 2048
            S = K // Kc
            part = self.empty(S, M, N)
            _cabi.check(_cabi.lib.b200lm_dgemm(self.device, 1, 0, S, M, N, Kc, 1.0, A2.data_ptr(), Kc * A2.stride(0),
                                               A2.stride(0), B2.data_ptr(), Kc * B2.stride(0), B2.stride(0), 0.0,
                                               part.data_ptr(), M * N, N, self.stream()))
            self.launches += 1
            res = part.sum(0)
            if K > S * Kc:
                tail = self.empty(M, N)
                self.gemm(True, False, M, N, K - S * Kc, 1.0, A2[S * Kc:], A2.stride(0), B2[S * Kc:], B2.stride(0), 0.0,
                          tail, N)
                res += tail
            res = res.reshape(out.shape)
            if beta == 0.0:
                out.copy_(res if alpha == 1.0 else alpha * res)
            else:
                out.mul_(beta).add_(res, alpha=alpha)
            return out
        self.gemm(transA, transB, M, N, K, alpha, A2, A2.stride(0), B2, B2.stride(0), beta, out,
                  out.stride(0) if out.dim() == 2 else 1)
        return out

    def potrf(self, A, shift, L, linv, info):
        n = A.shape[0]
        _cabi.check(_cabi.lib.b200lm_potrf(self.device, n, A.data_ptr(), A.stride(0), float(shift), L.data_ptr(),
                                           L.stride(0), linv.data_ptr(), info.data_ptr(), self.stream()))
        self.launches += 3 * ((n + 63) // 64)
        return int(info.item()) == 0

    def trsm(self, L, linv, trans, B, X):
        n = L.shape[0]
        nrhs = 1 if B.dim() == 1 else B.shape[1]
        _cabi.check(_cabi.lib.b200lm_trsm(self.device, n, nrhs, L.data_ptr(), L.stride(0), linv.data_ptr(), int(trans),
                                          B.data_ptr(), nrhs if B.dim() == 1 else B.stride(0),
                                          X.data_ptr(), nrhs if X.dim() == 1 else X.stride(0), self.stream()))
        self.launches += 2 * ((n + 63) // 64)
        return X


# ---- bound constraints: the reflective step selection of scipy's trf (the solver behind lsqfit.scipy_least_squares with
# ``bounds=``, reference src/lsqfit/_scipy.py:56-79, tests/test_lsqfit.py:1779-1808).  scipy is third party; its published
# algorithm (scipy/optimize/_lsq/trf.py: trf_bounds, select_step; common.py: CL_scaling_vector, step_size_to_bound,
# intersect_trust_region, minimize_quadratic_1d, make_strictly_feasible) is restated here on length-np host vectors --
# the O(np^2) products stay on the device.
def _in_bounds(x, lb, ub):
    return bool(np.all((x >= lb) & (x <= ub)))


def _make_strictly_feasible(x, lb, ub, rstep=1e-10):
    xn = x.copy()
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


def _cl_scaling_vector(x, g, lb, ub):
    v, dv = np.ones_like(x), np.zeros_like(x)
    m = (g < 0) & np.isfinite(ub)
    v[m] = ub[m] - x[m]; dv[m] = -1
    m = (g > 0) & np.isfinite(lb)
    v[m] = x[m] - lb[m]; dv[m] = 1
    return v, dv


def _step_size_to_bound(x, s, lb, ub):
    nz = np.nonzero(s)
    steps = np.full_like(x, np.inf)
    with np.errstate(over="ignore", invalid="ignore"):
        steps[nz] = np.maximum((lb - x)[nz] / s[nz], (ub - x)[nz] / s[nz])
    m = np.min(steps)
    return m, np.equal(steps, m) * np.sign(s).astype(int)


def _intersect_trust_region(x, s, Delta):
    a = s @ s
    b = x @ s
    c = x @ x - Delta ** 2
    d = np.sqrt(max(b * b - a * c, 0.0))
    q = -(b + np.copysign(d, b))
    t1, t2 = q / a, c / q
    return (t1, t2) if t1 < t2 else (t2, t1)


def _minimize_quadratic_1d(a, b, lb, ub, c=0.0):
    t = [lb, ub]
    if a != 0:
        e = -0.5 * b / a
        if lb < e < ub:
            t.append(e)
    t = np.asarray(t)
    y = t * (a * t + b) + c
    i = int(np.argmin(y))
    return t[i], y[i]


# ---- robust loss functions: scipy's ``loss`` / ``f_scale`` (lsqfit.scipy_least_squares passes them on, reference
# src/lsqfit/_scipy.py:56-79, 156-161).  scipy is third party; restated from scipy/optimize/_lsq/least_squares.py
# (IMPLEMENTED_LOSSES, construct_loss_function) and common.py (scale_for_robust_loss_function): the cost is
# 1/2 C^2 sum rho(f_i^2 / C^2), and the trust-region model uses rows of J and f scaled by functions of rho', rho''.
LOSSES = ("linear", "huber", "soft_l1", "cauchy", "arctan")
_EPS = float(np.finfo(float).eps)


def _rho(loss, z):
    """(rho, rho', rho'') at z = (f / f_scale)^2 as device vectors."""
    if loss == "huber":
        m = z <= 1.0
        zs = torch.where(m, torch.ones_like(z), z)              # (keeps the unused branch finite)
        return (torch.where(m, z, 2.0 * zs ** 0.5 - 1.0), torch.where(m, torch.ones_like(z), zs ** -0.5),
                torch.where(m, torch.zeros_like(z), -0.5 * zs ** -1.5))
    if loss == "soft_l1":
        t = 1.0 + z
        return 2.0 * (t ** 0.5 - 1.0), t ** -0.5, -0.5 * t ** -1.5
    if loss == "cauchy":
        t = 1.0 + z
        return torch.log1p(z), 1.0 / t, -1.0 / t ** 2
    if loss == "arctan":
        t = 1.0 + z ** 2
        return torch.atan(z), 1.0 / t, -2.0 * z / t ** 2
    raise ValueError("`loss` must be one of %s" % (LOSSES,))


def _dense_weights(pdf, n):
    """the whitening of a PDF (``i_invwgts``: 1x1 weights + block matrices) as ONE dense [nchiv, n] matrix"""
    W = np.zeros((pdf.nchiv, n))
    idx0, w0 = pdf.i_invwgts[0]
    W[np.arange(len(idx0)), idx0] = w0
    r = len(idx0)
    for idx, Wk in pdf.i_invwgts[1:]:
        W[r:r + Wk.shape[0], idx] = Wk
        r += Wk.shape[0]
    return W


class DenseFit(object):
    """Least-squares fit of ONE large problem: a model from the device registry (``fcn``: functor name, default
    ``'multiexp'`` with any number of terms), data with a dense covariance, a block structure or plain standard
    deviations, Gaussian priors that may be correlated with each other.

    ``data = (x, ymean, ycov)`` with ``ycov`` a matrix, a vector of standard deviations (uncorrelated data: millions of
    points are fine, nothing of size ny x ny is ever formed -- reference examples/uncorrelated.py:30-41) or None (see
    ``pdf``); ``prior = (pmean, psdev)`` or ``(pmean, pcov)`` with a covariance MATRIX (reference examples/p-corr.py:44-61).
    Attributes follow the reference's ``nonlinear_fit`` (src/lsqfit/__init__.py:665-725): ``pmean psdev cov chi2 dof Q
    logGBF nit stopping_criterion error svdcut svdn time``; ``p_cov`` / ``D`` are the propagated covariance and
    derivative matrix of ``fit.p`` (``_getp``, :897-922).
    """

    def __init__(self, data, prior, p0=None, svdcut=False, eps=False, tol=1e-8, maxit=1000, scaler="more",
                 polish=0, device=0, pdf=None, fcn="multiexp", spec=None, bounds=None, loss="linear", f_scale=1.0):
        from .fit import resolve_svdcut_eps
        if loss not in LOSSES:
            raise ValueError("`loss` must be one of %s" % (LOSSES,))
        self.loss, self.f_scale = loss, float(f_scale)
        if not self.f_scale > 0.0:
            raise ValueError("`f_scale` must be positive")
        self.robust = loss != "linear"
        self._prow = None                                       # row scale of the prior residuals (robust loss only)
        from .functors import Functor
        svdcut, eps = resolve_svdcut_eps(svdcut, eps)
        la = self.la = _LA(device)
        self.joint = False
        if spec is not None:
            # the plugin route (b200_dense below): everything comes from the ChivSpec of the fitter seam -- the joint
            # whitening of y (+) prior as ONE matrix [Wy | Wp] (data and prior may be correlated with each other)
            t, fcn, pdf = spec.x, spec.functor, spec.pdf
            ymean = np.asarray(pdf.mean, dtype=float)[:spec.ny]
            pm = np.zeros(spec.np) if spec.noprior else np.asarray(pdf.mean, dtype=float)[spec.ny:]
            ycov, pcov = None, np.ones(spec.np)
            self.joint = len(pdf.i_invwgts) > 1             # correlated blocks: one dense matrix; only 1x1 weights: vectors
            if self.joint and float(pdf.nchiv) * float(len(pdf.mean)) > 1.5e9:
                raise ValueError("b200_dense: the joint whitening matrix would need %.0f GB; give data and prior to "
                                 "lsqfit_b200.DenseFit separately" % (8e-9 * pdf.nchiv * len(pdf.mean)))
        else:
            t, ymean, ycov = data
            pm, pcov = prior
        ymean = np.asarray(ymean, dtype=float).reshape(-1)
        pm = np.asarray(pm, dtype=float).reshape(-1)
        pcov = np.asarray(pcov, dtype=float)
        self.ny, self.np = ymean.size, pm.size
        self.functor = fcn if isinstance(fcn, Functor) else Functor(fcn)
        self.tol = normalize_tol(tol)
        self.maxit = int(maxit)
        self.scaler = scaler
        self.times = {}
        dev = la.tdev
        # ---- the model evaluator: a compiled functor of this size, or the any-size multi-exponential kernel ----
        self._h = None
        self.xrows = self.functor.xrows(t, self.ny)
        compiled = any(f == self.functor.family and n == self.np for f, n, _, _ in _cabi.functor_table())
        if compiled:
            self._h = _cabi.handle_t()
            _cabi.check(_cabi.lib.b200lm_create(self.functor.family, self.ny, self.np, self.functor.nx, 0, la.device,
                                                C.byref(self._h)))
            _cabi.check(_cabi.lib.b200lm_set_const(self._h, self.xrows.ctypes.data, self.xrows.size), self._h)
        elif self.functor.name == "multiexp":
            if self.np % 2:
                raise ValueError("multiexp needs an even number of parameters [a..., E...]")
            self.K = self.np // 2
            self.t = self.xrows[:, 0].copy()
        else:
            raise ValueError("no device functor for %s with np=%d (lsqfit_b200.available() lists the compiled ones)"
                             % (self.functor.name, self.np))
        t0 = time.perf_counter()
        # ---- whitening of the data on the device (a-1): dense block / general block structure / 1x1 weights ----
        ycov = None if ycov is None else np.asarray(ycov, dtype=float)
        self.Wd = self.wdiag = self.Wpj = None
        if spec is not None and self.joint:
            N = self.ny if spec.noprior else self.ny + self.np
            Wfull = torch.as_tensor(_dense_weights(pdf, N)).to(dev)
            self.Wd = Wfull[:, :self.ny].contiguous()
            self.Wpj = None if spec.noprior else Wfull[:, self.ny:].contiguous()
            self._Cfull = torch.as_tensor(np.ascontiguousarray(pdf.cov)).to(dev)
            self._Cd = None
            self.svdcut, self.eps, self.svdn = pdf.svdcut, pdf.eps, pdf.nmod
            nd, data_logdet, data_mean = pdf.nchiv, pdf.logdet, ymean
        elif spec is not None:
            # only 1x1 weights (possibly millions of them): data and prior weights straight from the PDF
            idx0, w0 = pdf.i_invwgts[0]
            wall = np.empty(len(idx0)); wall[np.asarray(idx0)] = np.asarray(w0, dtype=float)
            sd = 1.0 / wall[:self.ny]
            self.wdiag = torch.as_tensor(wall[:self.ny].copy()).to(dev)
            self._Cd = torch.as_tensor(sd ** 2).to(dev)
            self.svdcut, self.eps, self.svdn = pdf.svdcut, pdf.eps, 0
            nd, data_logdet, data_mean = self.ny, 2.0 * float(np.sum(np.log(sd))), ymean
            if not spec.noprior:
                pcov = 1.0 / wall[self.ny:]
        elif pdf is None and ycov is not None and ycov.ndim <= 1:
            # uncorrelated data: 1x1 weights (src/lsqfit/_utilities.pyx:85-89), never a matrix
            sd = np.full(self.ny, float(ycov)) if ycov.ndim == 0 else ycov.reshape(-1)
            self.wdiag = torch.as_tensor(1.0 / sd).to(dev)
            self._Cd = torch.as_tensor(sd ** 2).to(dev)          # (diagonal of the data covariance)
            self.svdcut, self.eps, self.svdn = svdcut, eps, 0
            nd, data_logdet, data_mean = self.ny, 2.0 * float(np.sum(np.log(sd))), ymean
        elif pdf is None and ycov.ndim == 2 and np.count_nonzero(ycov) == ycov.size:
            # one fully correlated block: W and the corrected covariance never leave the device
            from .whiten import whiten_blocks
            if svdcut is not None:
                eps = None
            W, Cc, nout, nmod, logdet = whiten_blocks([self.ny], ycov.reshape(-1), svdcut, eps, device, as_torch=True)
            nd = int(nout[0])
            self.Wd = W[:nd * self.ny].view(nd, self.ny)
            self._Cd = Cc.view(self.ny, self.ny)
            self.svdcut, self.eps, self.svdn = svdcut, eps, int(nmod[0])
            data_logdet = float(logdet[0])
            data_mean = ymean
        else:
            if pdf is None:
                pdf = PDF(ymean, ycov, svdcut=svdcut, eps=eps, device=device)
            self.svdcut, self.eps, self.svdn = pdf.svdcut, pdf.eps, pdf.nmod
            nd = pdf.nchiv
            self.Wd = torch.as_tensor(_dense_weights(pdf, self.ny)).to(dev)
            self._Cd = torch.as_tensor(pdf.cov).to(dev)
            data_logdet = pdf.logdet
            data_mean = pdf.mean
        # ---- prior: independent (1x1 weights) or correlated (its own whitening, same svdcut / eps) ----
        self.Wp = self._Cp = None
        self.noprior_rows = spec is not None and (self.joint or spec.noprior)      # no separate prior residuals
        if self.noprior_rows:
            psd = np.ones(self.np)
            prior_logdet, npr = 0.0, 0
        elif pcov.ndim <= 1:
            psd = np.full(self.np, float(pcov)) if pcov.ndim == 0 else pcov.reshape(-1)
            prior_logdet = 2.0 * float(np.sum(np.log(psd)))
            npr = self.np
        else:
            ppdf = PDF(pm, pcov, svdcut=svdcut, eps=eps, device=device)
            psd = np.sqrt(np.diag(pcov))
            self.Wp = torch.as_tensor(_dense_weights(ppdf, self.np)).to(dev)
            self._Cp = torch.as_tensor(ppdf.cov).to(dev)
            self.PtP = la.mm(self.Wp, self.Wp, transA=True)
            self.svdn += ppdf.nmod
            prior_logdet = ppdf.logdet
            npr = ppdf.nchiv
        torch.cuda.synchronize(dev)
        self.times["whiten"] = time.perf_counter() - t0
        self.pdf = pdf
        self.nd = nd
        self.d_x = torch.as_tensor(self.xrows).to(dev)
        self.d_t = self.d_x[:, 0].contiguous()
        self.d_y = torch.as_tensor(np.ascontiguousarray(data_mean)).to(dev)
        self.d_pm = torch.as_tensor(pm).to(dev)
        self.d_wp = torch.as_tensor(np.zeros(self.np) if self.noprior_rows else 1.0 / psd).to(dev)
        # parameter distributions (lsqfit_b200/pdist.py): the model rows see q = T(p), their columns are scaled by T'(p)
        self._pd = None
        if spec is not None and spec.pdist is not None:
            if bounds is not None:
                raise ValueError("b200_dense: bounds are not built for fits with parameter distributions")
            self._pd = tuple(torch.as_tensor(a).to(dev) for a in spec.device_pdist)
        self.prior_mean, self.prior_sdev = pm, psd
        self.logdet_pdf = data_logdet + prior_logdet
        self.nchiv = nd + npr
        self.dof = self.nchiv - self.np
        # ---- workspaces ----
        n = self.np
        # b200lm_normal_diag in the loop (a robust loss rescales every row: materialised passes)
        self.fused = self.wdiag is not None and self._h is not None and n <= 8 and not self.robust
        self.G = la.empty(self.ny, n)
        self.delta = la.empty(self.ny)
        self.J = self.G if self.wdiag is not None else la.empty(nd, n)             # (uncorrelated: J = diag(w) G in place)
        self.A = la.empty(n, n)
        self.As = la.empty(n, n)
        self.L = la.empty(n, n)
        self.linv = la.empty((n + 63) // 64, 64, 64)
        self.info = torch.zeros(1, dtype=torch.int32, device=dev)
        self.nacc = la.empty(n * (n + 1) // 2 + n + 1)
        self._triu = torch.triu_indices(n, n, device=dev)
        self.polish = int(polish)
        x0 = pm.copy() if p0 is None else np.asarray(p0, dtype=float).reshape(-1)
        self.lb = self.ub = None
        if bounds is not None:
            lb, ub = (np.broadcast_to(np.asarray(b, dtype=float), (n,)).copy() for b in bounds)
            if not np.all(lb < ub):
                raise ValueError("Each lower bound must be strictly less than each upper bound.")     # scipy least_squares
            if not _in_bounds(x0, lb, ub):
                raise ValueError("`x0` is infeasible.")
            self.lb, self.ub = lb, ub
            x0 = _make_strictly_feasible(x0, lb, ub)
        t0 = time.perf_counter()
        self._fit(torch.as_tensor(x0).to(dev))
        torch.cuda.synchronize(dev)
        self.times["fit"] = time.perf_counter() - t0
        self._p_cov = self._D = None

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            _cabi.lib.b200lm_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- residuals and Jacobian (a-2) -------------------------------------------------------
    def _transform(self, p):
        """(q = T(p), T'(p)) on the device; (p, None) without parameter distributions"""
        if self._pd is None:
            return p, None
        code, lo, hi = self._pd
        e = torch.exp(torch.where(code == 1, p, torch.zeros_like(p)))
        u = lo + (hi - lo) * (0.5 * torch.special.erfc(-0.7071067811865476 * p))
        du = (hi - lo) * 0.3989422804014327 * torch.exp(-0.5 * p * p)
        q = torch.where(code == 1, e, torch.where(code == 2, p * p, torch.where(code == 3, u, p)))
        dq = torch.where(code == 1, e, torch.where(code == 2, 2.0 * p, torch.where(code == 3, du, torch.ones_like(p))))
        return q.contiguous(), dq

    def _model(self, p, with_G):
        p, dq = self._transform(p)
        self._keep_q = p                                        # (the launch reads it asynchronously)
        self._model_at(p, with_G)
        if with_G and dq is not None:
            self.G.mul_(dq[None, :])

    def _model_at(self, p, with_G):
        la = self.la
        if self._h is not None:
            _cabi.check(_cabi.lib.b200lm_model_rows(
                self._h, p.data_ptr(), self.d_y.data_ptr(), self.G.data_ptr() if with_G else None, self.G.stride(0),
                self.delta.data_ptr(), la.stream()), self._h)
        else:
            _cabi.check(_cabi.lib.b200lm_multiexp_dense(
                la.device, self.ny, self.K, self.d_t.data_ptr(), p.data_ptr(), self.d_y.data_ptr(),
                self.G.data_ptr() if with_G else None, self.G.stride(0), self.delta.data_ptr(), la.stream()))
        la.launches += 1

    def _prior_residual(self, p):
        dp = p - self.d_pm
        return dp * self.d_wp if self.Wp is None else self.la.mm(self.Wp, dp)

    def _data_residual(self, p):
        if self.wdiag is not None:
            return self.delta * self.wdiag
        fd = self.la.mm(self.Wd, self.delta)
        if self.Wpj is not None:                                 # joint whitening: the rows also see p - prior mean
            fd += self.la.mm(self.Wpj, p - self.d_pm)
        return fd

    def residual(self, p):
        """(f_data [nd], f_prior) = whitened residuals at p."""
        self._model(p, False)
        return self._data_residual(p), self._prior_residual(p)

    def _add_prior(self, fp, g):
        if self._prow is not None:                               # robust loss: prior rows scaled like every other row
            if self.Wp is None:
                w = self.d_wp * self._prow
                self.A.diagonal().add_(w ** 2)
                return g + w * fp
            Wps = self.Wp * self._prow[:, None]
            self.la.mm(Wps, Wps, transA=True, out=self.A, beta=1.0)
            return g + self.la.mm(Wps, fp, transA=True)
        if self.Wp is None:
            self.A.diagonal().add_(self.d_wp ** 2)
            return g + self.d_wp * fp
        self.A.add_(self.PtP)
        return g + self.la.mm(self.Wp, fp, transA=True)

    def _cost(self, fd, fp):
        """1/2 |f|^2, or scipy's robust cost 1/2 C^2 sum rho((f/C)^2) over data AND prior residuals."""
        if not self.robust:
            return 0.5 * float(fd @ fd + fp @ fp)
        c = self.f_scale                                         # z = (f / C)^2 exactly as scipy forms it (same side of huber's kink)
        return 0.5 * c * c * float(torch.sum(_rho(self.loss, (fd / c) ** 2)[0]) + torch.sum(_rho(self.loss, (fp / c) ** 2)[0]))

    def _robust_rows(self, f):
        """scale_for_robust_loss_function: (row scale of J, scaled residuals)."""
        z = (f / self.f_scale) ** 2
        _, r1, r2 = _rho(self.loss, z)
        js = torch.sqrt(torch.clamp(r1 + 2.0 * (r2 / self.f_scale ** 2) * f ** 2, min=_EPS))     # (scipy's order of operations)
        return js, f * r1 / js

    def jacobian(self, p, materialize=False, robust=None):
        """Normal matrix into self.A (and J_data = W.G into self.J unless the fused one-pass kernel is used);
        returns (fd, fp, g).  In fused mode fd is None and self.cost_data holds f_data . f_data.  With a robust loss
        (``robust``, default self.robust) J, f and the prior rows are the SCALED ones of scipy's trust-region model and
        self.cost_true holds the robust cost of the unscaled residuals."""
        la = self.la
        robust = self.robust if robust is None else robust
        self._prow = None
        fp = self._prior_residual(p)
        self.nfev_jac += 1
        if self.fused and not materialize:
            q, dq = self._transform(p)
            self._keep_q = q
            _cabi.check(_cabi.lib.b200lm_normal_diag(self._h, q.data_ptr(), self.d_y.data_ptr(), self.wdiag.data_ptr(),
                                                     self.nacc.data_ptr(), la.stream()), self._h)
            la.launches += 2
            n = self.np
            nt = n * (n + 1) // 2
            self.A.zero_()
            self.A[self._triu[0], self._triu[1]] = self.nacc[:nt]
            self.A.copy_(self.A + self.A.T - torch.diag(self.A.diagonal()))
            g = self.nacc[nt:nt + n].clone()
            if dq is not None:                                  # J = J_q diag(T'): J^T J and J^T r in fit space
                self.A.mul_(dq[:, None] * dq[None, :])
                g.mul_(dq)
            self.cost_data = self.nacc[nt + n].clone()
            return None, fp, self._add_prior(fp, g)
        self._model(p, True)
        if self.wdiag is not None:
            fd = self.delta * self.wdiag
            self.J.mul_(self.wdiag[:, None])                    # J = diag(w) G, in place (self.J is self.G)
        else:
            fd = self._data_residual(p)
            la.mm(self.Wd, self.G, out=self.J)
            if self.Wpj is not None:
                self.J.add_(self.Wpj)
        if robust:
            self.cost_true = self._cost(fd, fp)
            jd, fd = self._robust_rows(fd)
            self._prow, fp = self._robust_rows(fp)
            self.J.mul_(jd[:, None])
        la.mm(self.J, self.J, transA=True, out=self.A)
        g = la.mm(self.J, fd, transA=True)
        self.cost_data = fd @ fd
        return fd, fp, self._add_prior(fp, g)

    # ---- trust-region sub-problem -------------------------------------------------------------
    def _factor_solve(self, alpha, gs):
        """chol(As + alpha I); p = -(As + alpha I)^-1 gs; returns (ok, p, |p|, |L^-1 p|^2)."""
        la = self.la
        ok = la.potrf(self.As, alpha, self.L, self.linv, self.info)
        self.nfac += 1
        if not ok:
            return False, None, 0.0, 0.0
        b = -gs
        y = la.trsm(self.L, self.linv, 0, b, torch.empty_like(b))
        p = la.trsm(self.L, self.linv, 1, y, torch.empty_like(b))
        w = la.trsm(self.L, self.linv, 0, p.clone(), torch.empty_like(b))
        pn = float(torch.linalg.vector_norm(p))
        w2 = float(torch.dot(w, w))
        return True, p, pn, w2

    def _solve_tr(self, gs, Delta, alpha, cache):
        """Levenberg parameter by safeguarded Newton on the secular equation |p(alpha)| = Delta
        (decisions of scipy common.py: solve_lsq_trust_region; Cholesky instead of SVD)."""
        if "gn" not in cache:
            cache["gn"] = self._factor_solve(0.0, gs)
        ok0, p0, pn0, w20 = cache["gn"]
        if ok0 and pn0 <= Delta:
            return p0, 0.0
        alpha_upper = float(torch.linalg.vector_norm(gs)) / Delta
        alpha_lower = 0.0
        if ok0:
            alpha_lower = (pn0 - Delta) * pn0 / w20
        if alpha == 0.0 or alpha is None:
            alpha = max(0.001 * alpha_upper, (alpha_lower * alpha_upper) ** 0.5)
        p = None
        for _ in range(10):
            if alpha < alpha_lower or alpha > alpha_upper:
                alpha = max(0.001 * alpha_upper, (alpha_lower * alpha_upper) ** 0.5)
            ok, p_try, pn, w2 = self._factor_solve(alpha, gs)
            if not ok:
                alpha_lower = max(alpha_lower, alpha)
                alpha = max(2 * alpha, 0.001 * alpha_upper)
                continue
            p = p_try
            phi = pn - Delta
            if phi < 0:
                alpha_upper = alpha
            ratio = -phi * pn / w2
            alpha_lower = max(alpha_lower, alpha - ratio)
            alpha_used = alpha
            alpha -= (phi + Delta) * ratio / Delta
            if abs(phi) < 0.1 * Delta:
                self._alpha_used = alpha_used
                break
        if p is None:
            raise FloatingPointError("normal matrix is not positive definite at any damping")
        return p * (Delta / float(torch.linalg.vector_norm(p))), alpha

    def _select_step(self, x, g_h, p_h, d, Delta, theta):
        """scipy trf.py: select_step -- the trust-region step if it stays inside the bounds, else the best of: that step
        cut back to the bound, its reflection off the bound, and the (cut back) anti-gradient step, compared on the
        quadratic model  q(s) = 1/2 s^T As s + g_h^T s  (As = d J^T J d + C, on the device)."""
        lb, ub = self.lb, self.ub
        dev_t = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=float)).to(self.la.tdev)
        gh = g_h.cpu().numpy()
        p_h = p_h.cpu().numpy().copy()

        def As_dot(s):
            return self.la.mm(self.As, dev_t(s)).cpu().numpy()

        def quad(s):
            return 0.5 * float(s @ As_dot(s)) + float(gh @ s)

        def quad_1d(s, s0=None):
            As_s = As_dot(s)
            a = 0.5 * float(s @ As_s)
            b = float(gh @ s)
            if s0 is None:
                return a, b
            b += float(s0 @ As_s)
            return a, b, quad(s0)
        p = d * p_h
        if _in_bounds(x + p, lb, ub):
            return p, p_h, -quad(p_h)
        p_stride, hits = _step_size_to_bound(x, p, lb, ub)
        r_h = p_h.copy()
        r_h[hits.astype(bool)] *= -1
        r = d * r_h
        p = p * p_stride
        p_h = p_h * p_stride
        x_on_bound = x + p
        _, to_tr = _intersect_trust_region(p_h, r_h, Delta)
        to_bound, _ = _step_size_to_bound(x_on_bound, r, lb, ub)
        r_stride = min(to_bound, to_tr)
        if r_stride > 0:
            r_stride_l = (1 - theta) * p_stride / r_stride
            r_stride_u = theta * to_bound if r_stride == to_bound else to_tr
        else:
            r_stride_l, r_stride_u = 0, -1
        if r_stride_l <= r_stride_u:
            a, b, c = quad_1d(r_h, s0=p_h)
            r_stride, r_value = _minimize_quadratic_1d(a, b, r_stride_l, r_stride_u, c=c)
            r_h = r_h * r_stride + p_h
            r = r_h * d
        else:
            r_value = np.inf
        p = p * theta
        p_h = p_h * theta
        p_value = quad(p_h)
        ag_h = -gh
        ag = d * ag_h
        to_tr = Delta / np.linalg.norm(ag_h)
        to_bound, _ = _step_size_to_bound(x, ag, lb, ub)
        ag_stride = theta * to_bound if to_bound < to_tr else to_tr
        a, b = quad_1d(ag_h)
        ag_stride, ag_value = _minimize_quadratic_1d(a, b, 0, ag_stride)
        ag_h = ag_h * ag_stride
        ag = ag * ag_stride
        if p_value < r_value and p_value < ag_value:
            return p, p_h, -p_value
        if r_value < p_value and r_value < ag_value:
            return r, r_h, -r_value
        return ag, ag_h, -ag_value

    # ---- the fit (a-3) ---------------------------------------------------------------------
    def _fit(self, x):
        la = self.la
        xtol, gtol, ftol = self.tol
        self.nfev_jac = self.nfac = 0
        fd, fp, g = self.jacobian(x)
        nfev = 1
        cost = self.cost_true if self.robust else 0.5 * float(self.cost_data + fp @ fp)
        more = self.scaler == "more"

        def colnorm():
            return torch.sqrt(self.A.diagonal())                 # |J_j| over data and prior rows
        if more:
            scale_inv = colnorm()
            scale_inv[scale_inv == 0] = 1.0
        else:
            scale_inv = torch.ones_like(x)
        bounded = self.lb is not None
        dev_t = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=float)).to(la.tdev)
        if bounded:
            lbn, ubn = self.lb, self.ub
            v, dv = _cl_scaling_vector(x.cpu().numpy(), g.cpu().numpy(), lbn, ubn)
            si = scale_inv.cpu().numpy()
            v[dv != 0] *= si[dv != 0]
            Delta = float(np.linalg.norm(x.cpu().numpy() * si / v ** 0.5)) or 1.0
        else:
            Delta = float(torch.linalg.vector_norm(x * scale_inv)) or 1.0
        alpha = 0.0
        status = None
        error = None
        while True:
            if bounded:
                xh, gh_ = x.cpu().numpy(), g.cpu().numpy()
                v, dv = _cl_scaling_vector(xh, gh_, lbn, ubn)
                g_norm = float(np.max(np.abs(gh_ * v)))
            else:
                g_norm = float(torch.max(torch.abs(g)))
            if g_norm < gtol:
                status = 1
            if status is not None or nfev >= self.maxit:
                break
            if bounded:
                si = scale_inv.cpu().numpy()
                v[dv != 0] *= si[dv != 0]
                dh = v ** 0.5 / si                                   # "hat" space: x = d x_h
                diag_h = gh_ * dv / si                               # diagonal term of the Coleman-Li model
                theta = max(0.995, 1 - g_norm)
                d = dev_t(dh)
            else:
                d = 1.0 / scale_inv
            torch.mul(self.A, d[:, None] * d[None, :], out=self.As)
            if bounded:
                self.As.diagonal().add_(dev_t(diag_h))
            gs = d * g
            cache = {}
            actual = -1.0
            while actual <= 0 and nfev < self.maxit:
                step_h, alpha = self._solve_tr(gs, Delta, alpha, cache)
                if bounded:
                    step, step_h, predicted = self._select_step(xh, gs, step_h, dh, Delta, theta)
                    x_new = dev_t(_make_strictly_feasible(xh + step, lbn, ubn, rstep=0))
                    step, step_h = dev_t(step), dev_t(step_h)
                else:
                    As_step = la.mm(self.As, step_h)
                    predicted = -float(0.5 * (step_h @ As_step) + gs @ step_h)
                    step = d * step_h
                    x_new = x + step
                fd_new, fp_new = self.residual(x_new)
                nfev += 1
                shn = float(torch.linalg.vector_norm(step_h))
                cost_new = self._cost(fd_new, fp_new)
                if not np.isfinite(cost_new):
                    Delta = 0.25 * shn
                    continue
                actual = cost - cost_new
                if predicted > 0:
                    ratio = actual / predicted
                elif predicted == actual == 0:
                    ratio = 1.0
                else:
                    ratio = 0.0
                Delta_new = Delta
                if ratio < 0.25:
                    Delta_new = 0.25 * shn
                elif ratio > 0.75 and shn > 0.95 * Delta:
                    Delta_new = 2.0 * Delta
                step_norm = float(torch.linalg.vector_norm(step))
                ft = actual < ftol * cost and ratio > 0.25
                xt = step_norm < xtol * (xtol + float(torch.linalg.vector_norm(x)))
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
            if actual > 0:
                x, cost = x_new, cost_new
                fd, fp, g = self.jacobian(x)
                if more:
                    scale_inv = torch.maximum(scale_inv, colnorm())
        if status is None:
            status = 0
            error = "maxit=%d iterations exceeded" % self.maxit
        # ---- optional Gauss-Newton polish towards the exact stationary point ----
        # (same rule as the batched kernel: a full GN step is kept while the Newton decrement shrinks)
        d = 1.0 / scale_inv
        dd = d[:, None] * d[None, :]

        def gn(g):
            torch.mul(self.A, dd, out=self.As)
            ok, sh, _, _ = self._factor_solve(0.0, d * g)
            return ok, sh, (-float((d * g) @ sh) if ok else np.inf)
        if self.polish > 0 and not bounded and not self.robust:   # (undamped steps would leave the feasible region)
            ok, sh, dec = gn(g)
            for _ in range(self.polish):
                if not ok or not (dec > 1e-30 * max(1.0, 2 * cost)):
                    break
                x_old = x
                x = x + d * sh
                fd, fp, g = self.jacobian(x)
                nfev += 1
                ok2, sh2, dec2 = gn(g)
                if not ok2 or not (dec2 < dec):
                    x = x_old
                    fd, fp, g = self.jacobian(x)
                    break
                sh, dec = sh2, dec2
        # ---- results (a-5; src/lsqfit/__init__.py:665-682, 706-725) ----
        if fd is None:                                           # fused loop: one materialised pass for f, J, covariance
            fd, fp, g = self.jacobian(x, materialize=True)
        self.nit = nfev
        self.status = status
        self.stopping_criterion = STOPPING_CRITERION[status]
        self.error = error
        self.x = x
        self.pmean = x.cpu().numpy()
        prow = self._prow                                        # (scaled rows: the covariance below is that of scipy's fit.jac)
        if self.robust:
            fd, fp = self.residual(x)                            # the reference reports the TRUE residuals (fit.f = f(x))
            self.cost = self._cost(fd, fp)
        self.f = fd if self.noprior_rows else torch.cat([fd, fp])
        self.chi2 = float(fd @ fd + fp @ fp)
        from .fit import gammaQ, _logGBF
        self.Q = float(gammaQ(self.dof / 2.0, self.chi2 / 2.0))
        # covariance (J^T J)^-1 by CholeskyQR2: the Cholesky factor of the (scaled) normal matrix
        # alone loses cond(J)^2 eps; one re-orthogonalisation pass  Q1 = Js L^-T,  L2 L2^T = Q1^T Q1,
        # R = L2^T L^T  restores the cond(J) eps accuracy of the reference's SVD of J
        # (src/lsqfit/_scipy.py:171-175) using nothing but GEMMs and the blocked Cholesky.
        torch.mul(self.A, dd, out=self.As)
        if not la.potrf(self.As, 0.0, self.L, self.linv, self.info):
            self.error = "normal matrix not positive definite at the solution"
            self.cov = None
            return
        n = self.np
        eye = torch.eye(n, dtype=torch.float64, device=la.tdev)
        X = la.trsm(self.L, self.linv, 0, eye, la.empty(n, n))           # X = L^-1
        logdet = 2.0 * float(torch.sum(torch.log(torch.diagonal(self.L))))
        Js = self.J * d[None, :]
        Q1 = la.mm(Js, X, transB=True)                                   # data rows of Q1
        del Js
        A2 = la.mm(Q1, Q1, transA=True)
        del Q1
        if self.Wp is None:
            wp = self.d_wp if prow is None else self.d_wp * prow
            Xp = X * (wp * d)[None, :]                                   # prior rows: diag(wp d) X^T
            la.mm(Xp, Xp, transB=True, out=A2, beta=1.0)
        else:
            Wp = self.Wp if prow is None else self.Wp * prow[:, None]
            Q1p = la.mm(Wp * d[None, :], X, transB=True)                 # prior rows of Q1
            la.mm(Q1p, Q1p, transA=True, out=A2, beta=1.0)
        if la.potrf(A2, 0.0, self.L, self.linv, self.info):
            eye = torch.eye(n, dtype=torch.float64, device=la.tdev)
            X2 = la.trsm(self.L, self.linv, 0, eye, la.empty(n, n))
            logdet += 2.0 * float(torch.sum(torch.log(torch.diagonal(self.L))))
            X = la.mm(X2, X)
        cov_s = la.mm(X, X, transA=True)
        self.d_cov = cov_s * dd
        self.cov = self.d_cov.cpu().numpy()
        self.psdev = np.sqrt(np.diag(self.cov))
        self.logdet_JtJ = logdet - 2.0 * float(torch.sum(torch.log(d)))
        if self.robust:
            # fit.J of the reference's plugin is the TRUE Jacobian (Dfun(x), src/lsqfit/_scipy.py:166): restore it for
            # fit.p's propagation and take log det(J^T J) from it (src/lsqfit/__init__.py:712-725)
            self.jacobian(x, robust=False)
            torch.mul(self.A, dd, out=self.As)
            if la.potrf(self.As, 0.0, self.L, self.linv, self.info):
                self.logdet_JtJ = (2.0 * float(torch.sum(torch.log(torch.diagonal(self.L))))
                                   - 2.0 * float(torch.sum(torch.log(d))))
        self.logGBF = _logGBF(self.logdet_JtJ, self.logdet_pdf, self.chi2, self.dof)

    # ---- fit.p propagation (a-6; src/lsqfit/__init__.py:897-922) ------------------------------
    def propagate(self):
        """D = cov . J^T . W  (np x N) and cov(p) = D . C . D^T with the svd-corrected C."""
        la = self.la
        t0 = time.perf_counter()
        n, ny = self.np, self.ny
        M = la.mm(self.d_cov, self.J, transB=True)               # np x nd   = cov . J_data^T
        if self.joint:
            Wfull = self.Wd if self.Wpj is None else torch.cat([self.Wd, self.Wpj], dim=1)
            D = la.mm(M, Wfull.contiguous())                     # np x N
            covp = la.mm(la.mm(D, self._Cfull), D, transB=True)
            torch.cuda.synchronize(la.tdev)
            self.times["propagate"] = time.perf_counter() - t0
            self._D, self._p_cov = D, covp
            return D, covp
        if self.wdiag is not None:
            Dd = M * self.wdiag[None, :]                         # uncorrelated data: W and C are diagonal
            covp = la.mm(Dd * self._Cd[None, :], Dd, transB=True)
        else:
            Dd = la.mm(M, self.Wd)                               # np x ny
            T = la.mm(Dd, self._Cd)                              # svd-corrected data covariance
            covp = la.mm(T, Dd, transB=True)
        if self.Wp is None:
            Dp = self.d_cov * self.d_wp[None, :] ** 2            # cov . diag(wp) . diag(wp)
            Dps = Dp * torch.as_tensor(self.prior_sdev).to(la.tdev)[None, :]
            la.mm(Dps, Dps, transB=True, out=covp, beta=1.0)
        else:
            Dp = la.mm(self.d_cov, self.PtP)                     # cov . Wp^T Wp
            la.mm(la.mm(Dp, self._Cp), Dp, transB=True, out=covp, beta=1.0)
        torch.cuda.synchronize(la.tdev)
        self.times["propagate"] = time.perf_counter() - t0
        self._D = torch.cat([Dd, Dp], dim=1)
        self._p_cov = covp
        return self._D, covp

    @property
    def p_cov(self):
        if self._p_cov is None:
            self.propagate()
        return self._p_cov.cpu().numpy()

    @property
    def D(self):
        if self._D is None:
            self.propagate()
        return self._D.cpu().numpy()


class b200_dense(object):
    """The single-fit path with the reference's plugin signature (``FITTERS[name](p0, nf, chiv, tol=, maxit=, **fitterargs)``,
    src/lsqfit/__init__.py:662-664; result attributes as src/lsqfit/_scipy.py:115-181): one fit spread over the whole GPU
    -- for parameter counts the batched kernels are not compiled for (np > 25 for most models, any np for 'multiexp'), for
    millions of uncorrelated points, fits with BOUNDS, or on request (``fitter='b200_dense'``).  ``b200_lm`` routes here by
    itself when no batched kernel exists for the model's parameter count or when ``bounds`` are given.  Extra fitterargs:
    ``scaler`` ('more' | 'levenberg'), ``device``, ``polish``, ``bounds=(lower, upper)`` (scipy's argument of
    ``lsqfit.scipy_least_squares``, reference src/lsqfit/_scipy.py:77, tests/test_lsqfit.py:1779-1808: the reflective
    trust-region step selection of scipy's trf)."""

    def __init__(self, x0, n, f, tol=(1e-8, 1e-10, 1e-10), maxit=1000, scaler="more", device=0, polish=0, bounds=None,
                 loss="linear", f_scale=1.0, method=None, **extra_args):
        if extra_args:
            raise ValueError("b200_dense: unknown fitter arguments: " + ", ".join(sorted(extra_args)))
        if method not in (None, "trf"):
            raise ValueError("b200_dense implements scipy's method='trf' only (got %r)" % (method,))
        spec = getattr(f, "b200", None)
        if spec is None:
            raise ValueError("the b200_dense fitter needs a device functor: use lsqfit_b200.Functor(...) as fcn "
                             "and install the hook with lsqfit_b200.register() (no CPU fallback exists)")
        if spec.pdist_error is not None:
            raise ValueError("b200_dense: " + spec.pdist_error)
        self.tol, self.maxit, self.n = normalize_tol(tol), maxit, n
        self.x0 = np.array(x0, dtype=float)
        if spec.np < 0:
            spec.np = self.x0.size
        self.description = "dense    scaler = {}    device = cuda:{}".format(scaler, device)
        if bounds is not None:                                    # (lower, upper) in the caller's parameter order (scipy's argument)
            bounds = tuple(spec.to_device(np.broadcast_to(np.asarray(b, dtype=float), self.x0.shape)) for b in bounds)
            self.description += "    bounds"
        if loss != "linear":
            self.description += "    loss = {}".format(loss)
        fit = DenseFit(None, None, p0=spec.to_device(self.x0), tol=self.tol, maxit=maxit, scaler=scaler, polish=polish,
                       device=device, spec=spec, bounds=bounds, loss=loss, f_scale=f_scale)
        if n != fit.nchiv:
            raise ValueError("b200_dense: n=%d does not match the whitening (%d residuals)" % (n, fit.nchiv))
        self.dense = fit
        if fit.cov is None:
            self.cov = np.full((spec.np, spec.np), np.nan)
        x, cov, J = spec.from_device(fit.pmean, fit.cov if fit.cov is not None else self.cov, fit.J.cpu().numpy())
        self.x, self.cov = x, cov
        self.f = fit.f.cpu().numpy()
        # chiv rows: data (+ joint) rows, then the separate 1x1 prior rows
        if fit.noprior_rows:
            self.J = J
        else:
            Jp = np.diag(1.0 / fit.prior_sdev) if fit.Wp is None else fit.Wp.cpu().numpy()
            self.J = np.concatenate([J, spec.from_device(J=Jp)[2]], axis=0)
        self.nit = fit.nit
        self.logdet_JtJ = getattr(fit, "logdet_JtJ", float("nan"))
        self.results = dict(status=fit.status, nfev=fit.nit, chi2=fit.chi2, logdet_JtJ=self.logdet_JtJ, times=dict(fit.times))
        self.stopping_criterion = fit.stopping_criterion
        self.error = fit.error
