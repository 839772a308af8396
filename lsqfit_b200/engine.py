"""Plan objects and batched launches (thin layer over the C ABI).

``Plan`` owns one ``b200lm_handle``: a functor, the constant ``x`` array and the
whitening (the reference's ``yp_pdf.i_invwgts``).  ``fit_batch`` fits B independent
problems that differ only in their mean vectors / starting points -- exactly what the
reference's ``bootstrapped_fit_iter`` and ``simulated_fit_iter`` loop over one
``nonlinear_fit`` at a time (src/lsqfit/__init__.py:1391-1469, 1548-1642).

PyTorch is used only to own device buffers and streams.
"""
import ctypes as C

import numpy as np
import torch

from . import _cabi
from .functors import Functor

# solver status -> lsqfit stopping_criterion (reference src/lsqfit/_scipy.py:178-181)
# (11, 12, 14: the GSL policy's info 1 / 2 / 27, reference src/lsqfit/_gsl.pyx:689-701)
STOPPING_CRITERION = {0: 0, 1: 2, 2: 3, 3: 1, 4: 1, -1: 0, 11: 1, 12: 2, 14: 4}
SCALER = {"more": 1, "jac": 1, 1: 1, "none": 0, "levenberg": 0, None: 0, 0: 0, "marquardt": 2, 2: 2}
POLICY = {"trf": 0, "scipy": 0, "scipy_least_squares": 0, 0: 0, None: 0, "gsl": 1, "gsl_lm": 1, "gsl_multifit": 1, "lm": 1, 1: 1}


def normalize_tol(tol):
    """Exactly the reference's normalisation (src/lsqfit/_scipy.py:124-132)."""
    if np.shape(tol) == ():
        tol = (tol, 1e-10, 1e-10)
    elif np.shape(tol) == (1,):
        tol = (tol[0], 1e-10, 1e-10)
    elif np.shape(tol) == (2,):
        tol = (tol[0], tol[1], 1e-10)
    elif np.shape(tol) != (3,):
        raise ValueError("tol must be number or a 1-, 2-, or 3-tuple")
    return tuple(float(t) for t in tol)


class BatchResult(object):
    """Device-resident results of one batch (torch tensors on the plan's device)."""

    def __init__(self, x, chi2, cov, logdet, nit, status, f=None, J=None):
        self.x, self.chi2, self.cov, self.logdet = x, chi2, cov, logdet
        self.nit, self.status, self.f, self.J = nit, status, f, J

    def numpy(self):
        return dict((k, getattr(self, k).cpu().numpy()) for k in
                    ("x", "chi2", "cov", "logdet", "nit", "status", "f", "J") if getattr(self, k) is not None)


class Plan(object):
    def __init__(self, functor, np_, ny, x, i_invwgts, noprior=False, device=0, team=None, nslot=1, pdist=None):
        """nslot > 1: a fit set (b200lm_create_set) -- y (+) prior is ny data rows, then nslot prior slots of np
        entries; ``i_invwgts`` must be None, and the plan fits once ``set_windows`` has given one window per problem.
        pdist: None or (code, lo, hi) in device parameter order (lsqfit_b200/pdist.py, b200lm_set_param_dist): every
        fit and residual / Jacobian of the plan then sees the model at q = T(p)."""
        if isinstance(functor, str):
            functor = Functor(functor)
        self.functor = functor
        self.np, self.ny, self.noprior, self.nslot = int(np_), int(ny), bool(noprior), int(nslot)
        self.N = self.ny if self.noprior else self.ny + self.nslot * self.np
        self.device = int(device)
        self._h = _cabi.handle_t()
        if not torch.cuda.is_available():
            raise RuntimeError("lsqfit_b200: no CUDA device visible; this engine has no CPU fallback")
        if self.nslot > 1 and i_invwgts is not None:
            raise ValueError("a plan with nslot > 1 has no whitening of its own: pass i_invwgts=None, then set_windows")
        _cabi.check(_cabi.lib.b200lm_create_set(functor.family, self.ny, self.np, functor.nx, self.nslot,
                                                1 if noprior else 0, self.device, C.byref(self._h)))
        xr = functor.xrows(x, self.ny)
        _cabi.check(_cabi.lib.b200lm_set_const(self._h, xr.ctypes.data, xr.size), self._h)
        self.nchiv, self.nwin = 0, 0
        if i_invwgts is not None:
            self.set_weights(i_invwgts)
        self.tdev = torch.device("cuda", self.device)
        if team is not None:
            self.set_team(team)
        self.pdist = None
        if pdist is not None:
            self.set_param_dist(*pdist)

    def set_param_dist(self, code=None, lo=None, hi=None):
        """Parameter distributions (b200lm_set_param_dist): code [np] (0 plain, 1 log, 2 sqrt, 3 uniform), lo / hi [np]
        (read for code 3), device parameter order; no arguments clear them."""
        if code is None:
            _cabi.check(_cabi.lib.b200lm_set_param_dist(self._h, None, None, None), self._h)
            self.pdist = None
            return
        code = np.ascontiguousarray(code, dtype=np.int32)
        lo = np.ascontiguousarray(np.zeros(self.np) if lo is None else lo, dtype=np.float64)
        hi = np.ascontiguousarray(np.ones(self.np) if hi is None else hi, dtype=np.float64)
        if code.shape != (self.np,) or lo.shape != (self.np,) or hi.shape != (self.np,):
            raise ValueError("set_param_dist: code, lo and hi need np = %d entries" % self.np)
        _cabi.check(_cabi.lib.b200lm_set_param_dist(self._h, code.ctypes.data, lo.ctypes.data, hi.ctypes.data), self._h)
        self.pdist = (code, lo, hi) if code.any() else None

    # ---- whitening ---------------------------------------------------------------
    def set_weights(self, i_invwgts):
        idx0, w0 = i_invwgts[0]
        idx0 = np.ascontiguousarray(idx0, dtype=np.int32)
        w0 = np.ascontiguousarray(w0, dtype=np.float64)
        nin = np.array([len(i) for i, _ in i_invwgts[1:]], dtype=np.int32)
        nout = np.array([len(w) for _, w in i_invwgts[1:]], dtype=np.int32)
        bidx = (np.concatenate([np.asarray(i, dtype=np.int32) for i, _ in i_invwgts[1:]])
                if len(nin) else np.zeros(0, dtype=np.int32))
        bw = (np.concatenate([np.asarray(w, dtype=np.float64).reshape(-1) for _, w in i_invwgts[1:]])
              if len(nin) else np.zeros(0))
        bidx = np.ascontiguousarray(bidx)
        bw = np.ascontiguousarray(bw)
        _cabi.check(_cabi.lib.b200lm_set_weights(
            self._h, len(idx0), idx0.ctypes.data, w0.ctypes.data, len(nin),
            nin.ctypes.data, nout.ctypes.data, bidx.ctypes.data, bw.ctypes.data), self._h)
        self.nchiv = _cabi.lib.b200lm_nchiv(self._h)
        self.nwin = 0

    def set_windows(self, desc):
        """Fit windows instead of the weights (b200lm_set_windows): ``desc`` as made by
        ``lsqfit_b200.windows.window_weights``.  fit_batch then fits B = nwin x copies: means [copies, N] (or [N]),
        p0 [nwin, np] (or [np]); fit b is copy b % copies of window b // copies.  ``set_weights`` switches back."""
        d = dict((k, np.ascontiguousarray(desc[k], dtype=np.float64 if k in ("diag_w", "blk_w") else np.int32))
                 for k in ("ndiag", "diag_idx", "diag_w", "nblk", "blk_nin", "blk_nout", "blk_idx", "blk_w"))
        nwin = len(d["ndiag"])
        _cabi.check(_cabi.lib.b200lm_set_windows(
            self._h, nwin, *[d[k].ctypes.data for k in ("ndiag", "diag_idx", "diag_w", "nblk", "blk_nin", "blk_nout",
                                                       "blk_idx", "blk_w")]), self._h)
        self.nchiv = _cabi.lib.b200lm_nchiv(self._h)
        self.nwin = nwin
        self._win_dC = int(np.sum(d["blk_nin"].astype(np.int64) ** 2))      # doubles of window_propagate's dC

    def window_nchiv(self):
        out = np.zeros(self.nwin, dtype=np.int32)
        _cabi.check(_cabi.lib.b200lm_window_nchiv(self._h, out.ctypes.data), self._h)
        return out

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            _cabi.lib.b200lm_destroy(self._h)
            self._h = _cabi.handle_t()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- helpers -----------------------------------------------------------------
    def _dev(self, a, cols):
        """-> (tensor on device, stride): 1-d input = shared across the batch."""
        if isinstance(a, torch.Tensor):
            t = a.to(self.tdev, dtype=torch.float64).contiguous()
        else:
            t = torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64)).to(self.tdev)
        if t.dim() == 1:
            assert t.numel() == cols, (t.shape, cols)
            return t, 0
        assert t.dim() == 2 and t.shape[1] == cols, (t.shape, cols)
        return t, cols

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.tdev).cuda_stream)

    # ---- the batch fit -------------------------------------------------------------
    def _set_policy(self, policy, scaler):
        """policy: 'trf' (decisions of scipy's trf, the solver behind lsqfit.scipy_least_squares; nit = function
        evaluations) or 'gsl' (decisions of lsqfit.gsl_multifit with alg='lm'; nit = iterations, maxit limits
        iterations, scaler may also be 'marquardt')."""
        if policy not in POLICY:
            raise ValueError("unknown policy %r (use 'trf' or 'gsl')" % (policy,))
        if scaler not in SCALER:
            raise ValueError("unkown scaler " + str(scaler))
        _cabi.check(_cabi.lib.b200lm_set_policy(self._h, POLICY[policy]), self._h)
        return SCALER[scaler]

    def _bounds(self, bounds):
        """(lb, ub) -> two contiguous float64 host arrays of np entries (scalars broadcast)."""
        lb, ub = (np.array(np.broadcast_to(np.asarray(b, dtype=np.float64), (self.np,))) for b in bounds)
        if np.isnan(lb).any() or np.isnan(ub).any():
            raise ValueError("bounds must not be NaN")
        if not np.all(lb < ub):
            raise ValueError("Each lower bound must be strictly less than each upper bound.")     # scipy least_squares
        return lb, ub

    @staticmethod
    def _loss(loss, f_scale, bounds, policy):
        """scipy's loss= / f_scale= -> (code of lsqfit_b200.dense.LOSSES, f_scale), or None for 'linear'."""
        from .dense import LOSSES
        if loss not in LOSSES:
            raise ValueError("`loss` must be one of %s" % (LOSSES,))
        if loss == "linear":
            return None
        f_scale = float(f_scale)
        if not (np.isfinite(f_scale) and f_scale > 0):
            raise ValueError("f_scale must be finite and > 0")
        if bounds is not None:
            raise ValueError("a robust loss together with bounds is not built for batched fits")
        if POLICY[policy] == 1:
            raise ValueError("a robust loss is not built for the GSL policy (policy='gsl')")
        return LOSSES.index(loss), f_scale

    def _launch_with(self, bounds, loss, launch):
        """Run ``launch()`` with the box (b200lm_set_bounds) and the robust loss (b200lm_set_loss) set on the handle;
        the plan is cached and shared (the parent fit, other drivers), so both are cleared again afterwards."""
        if bounds is None and loss is None:
            return launch()
        try:
            if bounds is not None:
                lb, ub = bounds
                _cabi.check(_cabi.lib.b200lm_set_bounds(self._h, lb.ctypes.data, ub.ctypes.data), self._h)
            if loss is not None:
                _cabi.check(_cabi.lib.b200lm_set_loss(self._h, loss[0], loss[1]), self._h)
            return launch()
        finally:
            if loss is not None:
                _cabi.lib.b200lm_set_loss(self._h, 0, 1.0)
            if bounds is not None:
                _cabi.lib.b200lm_set_bounds(self._h, None, None)

    def _prepare(self, mean, sm, p0, sp, tol, maxit, scaler, polish, policy, bounds, want_cov, want_fJ, B=None,
                 loss="linear", f_scale=1.0):
        """What both launch entries check and compute.  mean [rows, N] (sm = N) or [N] (sm = 0), p0 likewise; with
        windows a row of means per copy and a start per window.  -> (B, solver arguments of the C entry, bounds as
        two host arrays or None, the loss as (code, f_scale) or None, shape and dtype of every output asked for, None
        for the others)."""
        xtol, gtol, ftol = normalize_tol(tol)
        sc = self._set_policy(policy, scaler)
        loss = self._loss(loss, f_scale, bounds, policy)
        if B is None:
            B = ((mean.shape[0] if sm else 1) * self.nwin if self.nwin else
                 (mean.shape[0] if sm else (p0.shape[0] if sp else 1)))
        rows_m, rows_p = (B // self.nwin, self.nwin) if self.nwin else (B, B)
        if (sm and mean.shape[0] != rows_m) or (sp and p0.shape[0] != rows_p):
            raise ValueError("mean and p0 disagree on the batch size")
        if bounds is not None:
            bounds = self._bounds(bounds)
            lo, hi = ((torch.as_tensor(b).to(p0.device) for b in bounds) if isinstance(p0, torch.Tensor) else bounds)
            if not bool(((p0 >= lo) & (p0 <= hi)).all()):             # one reduction (scipy: "`x0` is infeasible.")
                raise ValueError("`x0` is infeasible.")
        # 1-d shapes as B, not (B,): torch parses an int faster, and a launch of one fit is host bound
        f8, i4 = np.float64, np.int32
        shapes = dict(x=((B, self.np), f8), chi2=(B, f8), cov=((B, self.np, self.np), f8) if want_cov else None,
                      logdet=(B, f8), nit=(B, i4), status=(B, i4), f=((B, self.nchiv), f8) if want_fJ else None,
                      J=((B, self.nchiv, self.np), f8) if want_fJ else None)
        return B, (xtol, gtol, ftol, int(maxit), sc, int(polish)), bounds, loss, shapes

    def fit_batch(self, mean, p0, tol=1e-8, maxit=1000, scaler="more", B=None,
                  want_cov=True, want_fJ=False, out=None, polish=0, policy="trf", bounds=None,
                  loss="linear", f_scale=1.0):
        """Fit B problems on the device; inputs may be numpy arrays or device tensors.

        mean: [B, N] or [N] (shared);  p0: [B, np] or [np] (shared).
        bounds: None or (lb, ub) in device parameter order, scipy's ``bounds`` (±inf: none); p0 must lie in the box.
        loss, f_scale: scipy's robust loss ('linear' | 'huber' | 'soft_l1' | 'cauchy' | 'arctan') for every fit of the
        batch (b200lm_set_loss: cov from the rescaled rows, chi2 / f / J / logdet from the true ones; no polish; one
        warp per fit).  Not with bounds or policy='gsl'.
        Returns a BatchResult of device tensors (no host synchronisation)."""
        tm, sm = self._dev(mean, self.N)
        tp, sp = self._dev(p0, self.np)
        B, solver, bounds, loss, shapes = self._prepare(tm, sm, tp, sp, tol, maxit, scaler, polish, policy, bounds,
                                                        want_cov, want_fJ, B, loss, f_scale)
        if out is None:
            out = BatchResult(*[s and torch.empty(s[0], device=self.tdev,
                                                  dtype=torch.int32 if s[1] is np.int32 else torch.float64)
                                for s in shapes.values()])
        ptr = lambda t: t.data_ptr() if t is not None else None
        self._launch_with(bounds, loss, lambda: _cabi.check(_cabi.lib.b200lm_fit_batch(
            self._h, B, tm.data_ptr(), sm, tp.data_ptr(), sp, *solver,
            out.x.data_ptr(), out.chi2.data_ptr(), ptr(out.cov), out.logdet.data_ptr(),
            out.nit.data_ptr(), out.status.data_ptr(), ptr(out.f), ptr(out.J), self._stream()), self._h))
        out._keep = (tm, tp)        # keep inputs alive until the stream has consumed them
        return out

    def fit_batch_host(self, mean, p0, tol=1e-8, maxit=1000, scaler="more", want_cov=True,
                       want_fJ=False, out=None, polish=0, policy="trf", bounds=None, loss="linear", f_scale=1.0):
        """Same fit through the host-buffer C entry point: numpy in, numpy out.
        ``out`` may hold preallocated arrays (dict with keys x, chi2, cov, logdet, nit, status).
        ``bounds``, ``loss`` and ``f_scale`` as for fit_batch."""
        # the C entry point reads raw host pointers: dtype, contiguity and shapes are checked HERE
        # (np.ascontiguousarray is a no-op for conforming arrays)
        mean = np.ascontiguousarray(mean, dtype=np.float64)
        p0 = np.ascontiguousarray(p0, dtype=np.float64)
        if mean.ndim not in (1, 2) or mean.shape[-1] != self.N:
            raise ValueError("mean must be [N] or [B, N] with N = %d, got %s" % (self.N, mean.shape))
        if p0.ndim not in (1, 2) or p0.shape[-1] != self.np:
            raise ValueError("p0 must be [np] or [B, np] with np = %d, got %s" % (self.np, p0.shape))
        sm = 0 if mean.ndim == 1 else self.N
        sp = 0 if p0.ndim == 1 else self.np
        # every array of a given ``out`` is checked
        B, solver, bounds, loss, shapes = self._prepare(mean, sm, p0, sp, tol, maxit, scaler, polish, policy, bounds,
                                                        want_cov or out is not None, want_fJ or out is not None,
                                                        loss=loss, f_scale=f_scale)
        if out is None:
            out = dict((k, s and np.empty(*s)) for k, s in shapes.items())
        else:
            for k in ("x", "chi2", "logdet", "nit", "status"):
                if out.get(k) is None:
                    raise ValueError("out[%r] is required" % k)
            for k, (shp, dt) in shapes.items():
                a = out.get(k)
                if a is None:
                    continue
                shp = shp if isinstance(shp, tuple) else (shp,)
                if not (isinstance(a, np.ndarray) and a.dtype == dt and a.flags["C_CONTIGUOUS"]
                        and a.flags["WRITEABLE"] and tuple(a.shape) == shp):
                    raise ValueError("out[%r] must be a writable C-contiguous %s array of shape %s"
                                     % (k, np.dtype(dt).name, shp))
        ptr = lambda a: a.ctypes.data if a is not None else None
        self._launch_with(bounds, loss, lambda: _cabi.check(_cabi.lib.b200lm_fit_batch_host(
            self._h, B, mean.ctypes.data, sm, p0.ctypes.data, sp, *solver,
            ptr(out["x"]), ptr(out["chi2"]), ptr(out.get("cov")), ptr(out["logdet"]),
            ptr(out["nit"]), ptr(out["status"]), ptr(out.get("f")), ptr(out.get("J"))), self._h))
        return out

    def last_stats(self):
        """(function evaluations, Jacobian evaluations, Cholesky factorisations) of the
        last batch; synchronises."""
        buf = (C.c_ulonglong * 3)()
        _cabi.check(_cabi.lib.b200lm_last_stats(self._h, buf), self._h)
        return tuple(int(v) for v in buf)

    def last_stats_ex(self, n=16):
        """All diagnostic counters of the last batch (see b200lm_last_stats_ex); synchronises."""
        buf = (C.c_ulonglong * 16)()
        _cabi.check(_cabi.lib.b200lm_last_stats_ex(self._h, buf, int(n)), self._h)
        return [int(v) for v in buf[:n]]

    def set_order(self, mode):
        """Order of the work queue: None / -1 = default policy, 0 = input order, 1 = largest start-point chi2 first
        (b200lm_set_order: scheduling only, results unchanged)."""
        _cabi.check(_cabi.lib.b200lm_set_order(self._h, -1 if mode is None else int(mode)), self._h)

    def last_order(self):
        return int(_cabi.lib.b200lm_last_order(self._h))

    def set_team(self, team):
        """Kernel choice: 0/None = default policy (by problem shape), 1 = one warp per fit (saturated batches),
        2 / 4 = team kernel (lowest latency per trial point)."""
        _cabi.check(_cabi.lib.b200lm_set_team(self._h, int(team or 0)), self._h)

    def last_team(self):
        """Warps per fit of the last fit_batch launch (1 = one warp per fit, 2 / 4 = team kernel)."""
        return int(_cabi.lib.b200lm_last_team(self._h))

    def launch_count(self):
        return int(_cabi.lib.b200lm_launch_count(self._h))

    # ---- chiv(p) and its Jacobian ------------------------------------------------------
    def residual_jacobian(self, p, mean):
        tp, sp = self._dev(p, self.np)
        tm, sm = self._dev(mean, self.N)
        B = tp.shape[0] if sp else (tm.shape[0] if sm else 1)
        kw = dict(device=self.tdev, dtype=torch.float64)
        f = torch.empty((B, self.nchiv), **kw)
        J = torch.empty((B, self.nchiv, self.np), **kw)
        chi2 = torch.empty(B, **kw)
        _cabi.check(_cabi.lib.b200lm_residual_jacobian(
            self._h, B, tp.data_ptr(), sp, tm.data_ptr(), sm, f.data_ptr(), J.data_ptr(),
            chi2.data_ptr(), self._stream()), self._h)
        return f, J, chi2

    # ---- fit.p propagation -------------------------------------------------------------
    def propagate(self, x, cov, C_yp=None):
        """D = d p / d (y, prior)  [B, np, N]  and  cov(p) = D C D^T  [B, np, np]."""
        tx, _ = self._dev(np.atleast_2d(x) if not isinstance(x, torch.Tensor) else x, self.np)
        B = tx.shape[0]
        tc = (cov if isinstance(cov, torch.Tensor) else torch.as_tensor(np.asarray(cov, dtype=np.float64)))
        tc = tc.to(self.tdev, dtype=torch.float64).reshape(B, self.np, self.np).contiguous()
        kw = dict(device=self.tdev, dtype=torch.float64)
        D = torch.empty((B, self.np, self.N), **kw)
        covp = tC = None
        if C_yp is not None:
            tC = (C_yp if isinstance(C_yp, torch.Tensor) else torch.as_tensor(np.asarray(C_yp, dtype=np.float64)))
            tC = tC.to(self.tdev, dtype=torch.float64).contiguous()
            assert tuple(tC.shape) == (self.N, self.N)
            covp = torch.empty((B, self.np, self.np), **kw)
        _cabi.check(_cabi.lib.b200lm_propagate(
            self._h, B, tx.data_ptr(), tc.data_ptr(), tC.data_ptr() if tC is not None else None,
            D.data_ptr(), covp.data_ptr() if covp is not None else None, self._stream()), self._h)
        return D, covp

    def window_propagate(self, cov, J, C_in, dC=None):
        """fit.p of every window, jointly (windows set; b200lm_window_propagate).  cov [nwin, np, np] and J
        [nwin, nchiv, np]: the central batch's cov and J (``fit_batch(..., want_fJ=True)``); C_in [N, N]: the INPUT
        covariance of y (+) prior (None: D only); dC: every window's svd corrections as made by
        ``lsqfit_b200.windows.window_corrections`` (None: no window corrected).
        -> D [nwin, np, N] and the joint covariance [nwin, np, nwin, np] (or None): D_w C_in D_v^T between windows,
        D_w C_w D_w^T (C_w: window w's corrected covariance) within a window."""
        if not self.nwin:
            raise ValueError("window_propagate needs windows (set_windows)")
        nw, npar = self.nwin, self.np
        dev = lambda a: (a if isinstance(a, torch.Tensor) else torch.as_tensor(np.asarray(a, dtype=np.float64))).to(
            self.tdev, dtype=torch.float64).contiguous()
        tc = dev(cov).reshape(nw, npar, npar)
        tJ = dev(J).reshape(nw, self.nchiv, npar)
        kw = dict(device=self.tdev, dtype=torch.float64)
        D = torch.empty((nw, npar, self.N), **kw)
        tC = tdC = covp = None
        if C_in is not None:
            tC = dev(C_in)
            assert tuple(tC.shape) == (self.N, self.N)
            covp = torch.empty((nw, npar, nw, npar), **kw)
        if dC is not None:
            tdC = dev(dC).reshape(-1)
            if tdC.numel() != self._win_dC:
                raise ValueError("dC must hold %d doubles (one n_in x n_in block per correlated block of every window), "
                                 "got %d" % (self._win_dC, tdC.numel()))
        ptr = lambda t: t.data_ptr() if t is not None else None
        _cabi.check(_cabi.lib.b200lm_window_propagate(
            self._h, tc.data_ptr(), tJ.data_ptr(), ptr(tC), ptr(tdC), D.data_ptr(), ptr(covp), self._stream()),
            self._h)
        return D, covp
