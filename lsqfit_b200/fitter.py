"""``b200_lm`` -- the new ``fitter=`` plugin for ``lsqfit.nonlinear_fit``.

Plugin contract (reference src/lsqfit/__init__.py:662-682, mirrored from
src/lsqfit/_scipy.py:115-181 and src/lsqfit/_gsl.pyx:563-723):

    fit = b200_lm(x0, n, f, tol=tol, maxit=maxit, **fitterargs)

with attributes ``x cov f J nit tol stopping_criterion error results description``.
Non-convergence is reported through ``error`` / ``stopping_criterion``, never raised.

The reference hands the fitter an opaque callable ``f`` (a ``chiv`` instance).  The
device engine needs the model identity, ``x``, the mean vector and the whitening, so ``f``
must carry a ``b200`` attribute (a ``ChivSpec``) -- attached by
``lsqfit_b200.fit.nonlinear_fit`` or, for real lsqfit, by the ``_build_chiv_chivw`` hook
installed with ``lsqfit_b200.register()`` (see INTEGRATION.md).
"""
import numpy as np

from .engine import Plan, STOPPING_CRITERION, normalize_tol


class PlanCache(object):
    """Plans shared between fits that differ only in their means.

    The reference's iterators construct one ``nonlinear_fit`` per bootstrap copy (src/lsqfit/__init__.py:1612-1624)
    and each of them rebuilds chiv -- but model, x and whitening are the same for every copy, only the means move.
    A plan (device handle, uploaded x and weights, workspaces, stream) is therefore keyed by a digest of
    (functor, np, ny, x, i_invwgts, noprior, device): a copy then costs one launch, not a ``b200lm_create``."""

    def __init__(self, capacity=16):
        import collections
        self.capacity = int(capacity)
        self.plans = collections.OrderedDict()
        self.hits = self.misses = 0

    @staticmethod
    def key(functor, np_, ny, x, i_invwgts, noprior, device):
        import hashlib
        h = hashlib.blake2b(digest_size=16)
        h.update(("%s|%d|%d|%d|%d|%d" % (functor.name, functor.family, int(np_), int(ny), int(bool(noprior)), int(device))).encode())
        h.update(np.ascontiguousarray(functor.xrows(x, int(ny)), dtype=np.float64).tobytes())
        for idx, w in i_invwgts:
            h.update(np.ascontiguousarray(idx, dtype=np.int64).tobytes())
            h.update(np.ascontiguousarray(w, dtype=np.float64).tobytes())
        return h.hexdigest()

    def get(self, functor, np_, ny, x, i_invwgts, noprior, device):
        k = self.key(functor, np_, ny, x, i_invwgts, noprior, device)
        plan = self.plans.get(k)
        if plan is not None:
            self.hits += 1
            self.plans.move_to_end(k)
            return plan
        self.misses += 1
        plan = Plan(functor, np_, ny, x, i_invwgts, noprior=noprior, device=device)
        self.plans[k] = plan
        while len(self.plans) > self.capacity:
            _, old = self.plans.popitem(last=False)
            old.close()
        return plan

    def clear(self):
        for p in self.plans.values():
            p.close()
        self.plans.clear()
        self.hits = self.misses = 0


PLAN_CACHE = PlanCache()


class ChivSpec(object):
    """Everything the device needs to evaluate chiv: functor, x, whitening, means."""

    def __init__(self, functor, x, pdf, noprior, ny, np_, pperm=None):
        self.functor, self.x, self.pdf, self.noprior = functor, x, pdf, bool(noprior)
        self.ny, self.np = int(ny), int(np_)
        # pperm[k] = position in the CALLER's flat parameter buffer of device parameter k (composite functors fix
        # their own parameter order; lsqfit's buffer follows the prior dictionary); None = identical
        self.pperm = None if pperm is None else np.asarray(pperm, dtype=np.int64)
        self._plans = {}

    def _inv(self):
        inv = np.empty_like(self.pperm)
        inv[self.pperm] = np.arange(self.pperm.size)
        return inv

    @property
    def mean(self):
        """means of y (+) prior in DEVICE order"""
        m = np.asarray(self.pdf.mean, dtype=float)
        if self.pperm is None or self.noprior:
            return m
        return np.concatenate([m[:self.ny], m[self.ny:][self.pperm]])

    @property
    def i_invwgts(self):
        """the whitening with prior indices renumbered to the device's parameter order"""
        if self.pperm is None or self.noprior:
            return self.pdf.i_invwgts
        inv, ny = self._inv(), self.ny
        out = []
        for idx, w in self.pdf.i_invwgts:
            idx = np.asarray(idx, dtype=np.int64)
            out.append((np.where(idx >= ny, ny + inv[np.maximum(idx - ny, 0)], idx), w))
        return out

    def to_device(self, p):
        return np.asarray(p, dtype=float) if self.pperm is None else np.asarray(p, dtype=float)[..., self.pperm]

    def from_device(self, x=None, cov=None, J=None):
        """results in the caller's parameter order"""
        if self.pperm is None:
            return x, cov, J
        inv = self._inv()
        return (None if x is None else x[..., inv], None if cov is None else cov[..., inv, :][..., :, inv],
                None if J is None else J[..., inv])

    def plan(self, device=0):
        if device not in self._plans:
            self._plans[device] = PLAN_CACHE.get(self.functor, self.np, self.ny, self.x, self.i_invwgts,
                                                 self.noprior, device)
        return self._plans[device]


class DeviceChiv(object):
    """Callable ``chiv(p)`` evaluated on the device (reference src/lsqfit/_utilities.pyx:50-94)."""

    def __init__(self, spec, device=0):
        self.b200 = spec
        self.device = device

    def __call__(self, p):
        plan = self.b200.plan(self.device)
        f, _, _ = plan.residual_jacobian(self.b200.to_device(p).reshape(1, -1), self.b200.mean)
        return f[0].cpu().numpy()

    def jacobian(self, p):
        plan = self.b200.plan(self.device)
        _, J, _ = plan.residual_jacobian(self.b200.to_device(p).reshape(1, -1), self.b200.mean)
        return self.b200.from_device(J=J[0].cpu().numpy())[2]


class b200_lm(object):
    """B200 batched Levenberg-Marquardt fitter (single-fit plugin face).

    Args mirror the reference plugins: ``x0`` start, ``n`` number of residuals, ``f`` the chiv
    callable, ``tol`` = xtol or (xtol, gtol, ftol), ``maxit``.
    Extra ``fitterargs``:
      ``policy``  'trf' (default): the trust-region decisions of the solver behind ``lsqfit.scipy_least_squares``
                  (reference src/lsqfit/_scipy.py:156-161); ``nit`` and ``maxit`` count function evaluations (:167).
                  'gsl': those of ``lsqfit.gsl_multifit`` with ``alg='lm'`` (src/lsqfit/_gsl.pyx:563-723: Nielsen update
                  of the LM parameter, GSL's xtol/gtol tests); ``nit`` and ``maxit`` count iterations (:713), and the
                  reference's ``alg`` ('lm' only), ``solver`` ('qr' | 'cholesky' | 'svd': all served by the device's
                  LDL^T solve of the damped normal equations), ``factor_up``, ``factor_down``, ``avmax`` (read by GSL's
                  dogleg / lmaccel methods only) are accepted.
      ``scaler``  'more' (default) | 'levenberg' | 'marquardt' (gsl policy only)   (_gsl.pyx:621-653)
      ``bounds``  (lower, upper): scipy's bound constraints (``lsqfit.scipy_least_squares(bounds=...)``); such fits run on
                  the single-fit path (lsqfit_b200/dense.py) with scipy trf's reflective step selection; the batch
                  drivers of the fit (bootstrapped_fits, simulated_fits) fit their copies with the same box on the device.
      ``loss``, ``f_scale``  scipy's robust loss functions ('linear' | 'huber' | 'soft_l1' | 'cauchy' | 'arctan';
                  ``lsqfit.scipy_least_squares(loss=...)``, src/lsqfit/_scipy.py:77): also on the single-fit path.
      ``method``  None | 'trf' (scipy's other methods are different solvers and are refused).
      ``device``  CUDA index;  ``polish``  max Gauss-Newton refinement steps after the trust-region loop (default 0 =
                  stop where the reference's solver stops).
    """

    def __init__(self, x0, n, f, tol=(1e-8, 1e-10, 1e-10), maxit=1000, scaler="more", device=0,
                 polish=0, policy="trf", alg="lm", solver="qr", factor_up=3.0, factor_down=2.0, avmax=0.75,
                 bounds=None, loss="linear", f_scale=1.0, method=None, **extra_args):
        if extra_args:
            raise ValueError("b200_lm: unknown fitter arguments: " + ", ".join(sorted(extra_args)))
        if method not in (None, "trf"):
            # scipy's other methods ('dogbox', MINPACK 'lm': src/lsqfit/_scipy.py:56-71) are different solvers
            raise ValueError("b200_lm implements scipy's method='trf' (policy='trf') and GSL's 'lm' (policy='gsl') only; "
                             "got method=%r" % (method,))
        from .engine import POLICY, SCALER
        if policy not in POLICY:
            raise ValueError("b200_lm: unknown policy " + str(policy))
        gsl = POLICY[policy] == 1
        if alg != "lm":
            raise ValueError("unkown algorithm " + str(alg))                # _gsl.pyx:619 (only 'lm' runs on the device)
        if scaler not in SCALER or (SCALER[scaler] == 2 and not gsl):
            raise ValueError("unkown scaler " + str(scaler))                 # _gsl.pyx:628
        if solver not in ("qr", "cholesky", "svd"):
            raise ValueError("unkown solver " + str(solver))                 # _gsl.pyx:637
        spec = getattr(f, "b200", None)
        if spec is None:
            raise ValueError(
                "the b200_lm fitter needs a device functor: use lsqfit_b200.Functor(...) as fcn "
                "and install the hook with lsqfit_b200.register() (no CPU fallback exists)")
        self.tol = normalize_tol(tol)
        self.maxit = maxit
        self.n = n
        self.x0 = np.array(x0, dtype=float)
        self.policy, self.scaler = ("gsl" if gsl else "trf"), scaler
        if gsl:
            self.alg, self.solver, self.factor_up, self.factor_down, self.avmax = alg, solver, factor_up, factor_down, avmax
            self.description = "methods = {}/{}/{}    device = cuda:{}".format(alg, scaler, solver, device)
        else:
            self.description = "scaler = {}    device = cuda:{}".format(scaler, device)
        from ._cabi import B200LMError, functor_table
        if spec.np < 0:
            spec.np = self.x0.size
        robust = loss != "linear"
        if bounds is not None or robust or not any(fam == spec.functor.family and m == spec.np
                                                   for fam, m, _, _ in functor_table()):
            # no batched kernel for this parameter count, bound constraints (scipy's ``bounds``) or a robust loss
            # (scipy's ``loss`` / ``f_scale``): one fit over the whole GPU instead (lsqfit_b200/dense.py)
            if gsl:
                raise ValueError("b200_lm: policy='gsl' needs a batched kernel without bounds / loss (model %s, np=%d)"
                                 % (spec.functor.name, spec.np))
            from .dense import b200_dense
            d = b200_dense(x0, n, f, tol=tol, maxit=maxit, scaler=scaler, device=device, polish=polish, bounds=bounds,
                           loss=loss, f_scale=f_scale)
            for k in ("x", "cov", "f", "J", "nit", "logdet_JtJ", "results", "stopping_criterion", "error", "dense"):
                setattr(self, k, getattr(d, k))
            self.description = d.description
            return
        plan = spec.plan(device)
        if n != plan.nchiv:
            raise ValueError("b200_lm: n=%d does not match the whitening (%d residuals)" % (n, plan.nchiv))
        out = plan.fit_batch_host(spec.mean, spec.to_device(self.x0).reshape(1, -1), tol=self.tol, maxit=maxit,
                                  scaler=scaler, want_cov=True, want_fJ=True, polish=polish, policy=self.policy)
        self.x, self.cov, self.J = spec.from_device(out["x"][0].copy(), out["cov"][0].copy(), out["J"][0].copy())
        self.f = out["f"][0].copy()
        self.nit = int(out["nit"][0])
        self.logdet_JtJ = float(out["logdet"][0])
        status = int(out["status"][0])
        self.results = dict(status=status, nit=self.nit, chi2=float(out["chi2"][0]),
                            logdet_JtJ=self.logdet_JtJ)
        if not gsl:
            self.results["nfev"] = self.nit
        self.stopping_criterion = STOPPING_CRITERION[status]
        self.error = None
        if status == -1:
            self.error = "b200_lm: residuals are not finite at the starting point"
        elif status == 0:
            self.error = "b200_lm: no convergence in {} {}".format(maxit, "iterations" if gsl else "function evaluations")
        elif status == 14:
            self.error = "b200_lm can't improve on starting value; may have converged already."   # _gsl.pyx:714-715
        elif not np.all(np.isfinite(self.cov)):
            self.error = "b200_lm: J^T J is singular at the solution"
