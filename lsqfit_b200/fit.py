"""gvar-free host mirror of ``lsqfit.nonlinear_fit`` for the device hot path.

Real lsqfit needs gvar for every input.  This module offers the same operator
interface on plain arrays -- same argument names and meaning (``data``, ``fcn``,
``prior``, ``p0``, ``svdcut``, ``eps``, ``tol``, ``maxit``, ``fitter``, ``**fitterargs``),
same result attributes (``pmean psdev cov chi2 dof Q logGBF nit tol stopping_criterion
error residuals J svdn nblocks description fitter_results p0``), same iterators
(``bootstrapped_fit_iter``, ``simulated_fit_iter``) -- so that it is a drop-in for the
path  whiten -> chiv -> fitter -> fit.p  and so that the parity tests read like the
reference's own tests.  With real lsqfit + gvar installed use ``lsqfit_b200.register()``
instead and keep calling ``lsqfit.nonlinear_fit(..., fitter='b200_lm')``.

Array forms of the reference's GVar inputs:
  data  = (x, ymean, ycov | ysdev)     (the reference's 3-tuple form, __init__.py:1862-1866)
          or (ymean, ycov | ysdev) for ``fcn(p)`` models without x
  prior = (pmean, pcov | psdev) or None
  yp_cov= optional joint covariance of y (+) prior when data and prior are correlated

Reference lines followed: src/lsqfit/__init__.py:455-733 (constructor), :897-922 (_getp),
:1391-1469, 1471-1543 (simulated fits), :1548-1642 (bootstrap), :1947-1948 (default p0).
"""
import time

import numpy as np
import torch

from .engine import STOPPING_CRITERION, BatchResult
from .fitter import ChivSpec, DeviceChiv, b200_lm
from .functors import Functor
from .whiten import PDF


def gammaQ(a, x):
    """Q(a, x): the reference uses scipy.special.gammaincc too (src/lsqfit/_scipy.py:16-18)."""
    from scipy.special import gammaincc
    return gammaincc(a, x)


def _cov2(c, n):
    c = np.asarray(c, dtype=float)
    if c.ndim == 0:
        c = np.full(n, float(c))
    return np.diag(c ** 2) if c.ndim == 1 else c


def resolve_svdcut_eps(svdcut, eps):
    """The reference's defaults (src/lsqfit/__init__.py:470-479): neither given -> svdcut = 1e-12,
    eps = None; only ``eps`` given -> svdcut = None (the eps regulator is used); only ``svdcut`` given
    -> eps = None.  ``False`` is the "not given" sentinel, as in the reference."""
    if svdcut is False and eps is False:
        return 1e-12, None
    if svdcut is False:
        return None, eps
    if eps is False:
        return svdcut, None
    return svdcut, eps


def fresh_seed():
    """A new Philox key for unseeded calls (the reference draws from gvar's global RNG, so two
    unseeded calls never repeat the same noise)."""
    return int(np.random.SeedSequence().entropy) & (2 ** 64 - 1)


def _logGBF(logdet_JtJ, pdf_logdet, chi2, dof):
    """src/lsqfit/__init__.py:720-725"""
    return 0.5 * (-logdet_JtJ - pdf_logdet - chi2 - dof * np.log(2. * np.pi))


def _dense_plugin(*args, **kargs):
    from .dense import b200_dense
    return b200_dense(*args, **kargs)


class nonlinear_fit(object):
    FITTERS = {"b200_lm": b200_lm, "b200_dense": _dense_plugin}

    def __init__(self, data=None, fcn=None, prior=None, p0=None, svdcut=False, eps=False,
                 tol=1e-8, maxit=1000, fitter="b200_lm", yp_cov=None, _yp_pdf=None,
                 noise=False, noise_seed=None, **fitterargs):
        clock = time.perf_counter()
        svdcut, eps = resolve_svdcut_eps(svdcut, eps)
        # noise = (svd noise, prior noise), a bool meaning both (src/lsqfit/__init__.py:493-499, 516)
        self.noise = (bool(noise), bool(noise)) if isinstance(noise, (bool, np.bool_)) else tuple(bool(v) for v in noise)
        if len(self.noise) != 2:
            raise ValueError("noise must be a bool or a pair of bools")
        if any(self.noise) and noise_seed is None:
            noise_seed = fresh_seed()
        self.noise_seed = noise_seed
        if fitter not in nonlinear_fit.FITTERS:
            raise ValueError("unknown fitter: " + str(fitter))      # __init__.py:529-530
        if isinstance(fcn, str):
            fcn = Functor(fcn)
        if not isinstance(fcn, Functor):
            raise ValueError("fcn must be a lsqfit_b200.Functor (device model registry)")
        if not isinstance(data, tuple) or len(data) not in (2, 3):
            raise ValueError("data tuple wrong length: " + str(len(data) if isinstance(data, tuple) else data))
        if len(data) == 3:
            x, ymean, yerr = data
        else:
            x, (ymean, yerr) = False, data
        ymean = np.array(ymean, dtype=float).reshape(-1)
        ny = ymean.size
        self.fcn, self.fitter, self.fitterargs = fcn, fitter, dict(fitterargs)
        self.device = int(fitterargs.get("device", 0))
        self.x = x
        noprior = prior is None
        if noprior:
            if p0 is None:
                raise ValueError("need p0 if there is no prior")
            pmean = pcov = None
            npar = int(np.size(p0))
        else:
            pmean = np.array(prior[0], dtype=float).reshape(-1)
            npar = pmean.size
            pcov = _cov2(prior[1], npar)
            if self.noise[1]:
                # __init__.py:535-536: prior means fluctuate by one sample of the prior's own distribution
                # (device Philox normals; the factor of an np x np covariance is host work)
                from .bootstrap import normals
                Lp = np.linalg.cholesky(pcov) if np.count_nonzero(pcov - np.diag(np.diag(pcov))) else np.diag(np.sqrt(np.diag(pcov)))
                pmean = pmean + Lp @ normals(npar, int(noise_seed) ^ 0x9E3779B97F4A7C15,
                                             device=int(fitterargs.get("device", 0))).cpu().numpy()
        N = ny if noprior else ny + npar
        mean = ymean if noprior else np.concatenate([ymean, pmean])
        # ---- whitening (device) : __init__.py:539-561 ------------------------------
        if _yp_pdf is None:
            if yp_cov is None:
                yerr = np.asarray(yerr, dtype=float)
                pdiag = noprior or np.count_nonzero(pcov - np.diag(np.diag(pcov))) == 0
                if yerr.ndim <= 1 and pdiag:
                    sd = np.full(ny, float(yerr)) if yerr.ndim == 0 else yerr
                    yp_cov = sd if noprior else np.concatenate([sd, np.sqrt(np.diag(pcov))])
                else:
                    yp_cov = np.zeros((N, N))
                    yp_cov[:ny, :ny] = _cov2(yerr, ny)
                    if not noprior:
                        yp_cov[ny:, ny:] = pcov
            pdf = PDF(mean, yp_cov, svdcut=svdcut, eps=eps, device=self.device, noise=self.noise[0],
                      noise_seed=noise_seed)
            mean = pdf.mean                       # with the svd noise, if any (y.flat = yp_pdf.distribution, __init__.py:1896-1900)
            ymean = mean[:ny]
            if not noprior:
                pmean = mean[ny:]
        else:
            pdf = _yp_pdf.copy_with_mean(mean)
        self.yp_pdf = pdf
        self.svdcut, self.eps = pdf.svdcut, pdf.eps
        self.y = ymean
        self.prior = None if noprior else (pmean, pcov)
        self.svdn = pdf.nmod
        self.nblocks = pdf.nblocks
        # ---- p0 : __init__.py:562-565, 1947-1948 -------------------------------------
        if p0 is None:
            psd = np.sqrt(np.diag(pcov))
            p0 = np.where(pmean != 0.0, pmean, pmean + 0.1 * psd)
        self.p0 = np.array(p0, dtype=float).reshape(-1)
        if self.p0.size != npar:
            raise ValueError("p0 and prior shapes incompatible")
        # ---- chiv : __init__.py:571-575 ---------------------------------------------
        spec = ChivSpec(fcn, x, pdf, noprior, ny, npar)
        self._chiv = DeviceChiv(spec, self.device)
        nf = pdf.nchiv
        self.dof = nf - self.p0.size
        # ---- fit : __init__.py:657-682 ---------------------------------------------
        fit = nonlinear_fit.FITTERS[fitter](self.p0, nf, self._chiv, tol=tol, maxit=maxit, **fitterargs)
        self.error = fit.error
        self.cov = fit.cov
        self.chi2 = np.sum(fit.f ** 2)
        self.J = fit.J
        self.residuals = np.array(fit.f)
        self.Q = gammaQ(self.dof / 2., self.chi2 / 2.)
        self.nit = fit.nit
        self.tol = fit.tol
        self.maxit = maxit
        self.stopping_criterion = fit.stopping_criterion
        self.description = getattr(fit, "description", "")
        self.fitter_results = fit.results
        self.pmean = np.array(fit.x)
        self.psdev = np.sqrt(np.diag(fit.cov))
        self.palt = (self.pmean, self.psdev)
        self.logGBF = None if noprior else _logGBF(fit.logdet_JtJ, pdf.logdet, self.chi2, self.dof)
        self._p = None
        self._L = None
        self._dense = getattr(fit, "dense", None)            # single-fit path: its own propagation kernels
        self._spec = spec
        self.time = time.perf_counter() - clock

    # ---- fit.p : __init__.py:897-922 ---------------------------------------------------
    def _getp(self):
        if self._p is None and self._dense is not None:
            D, covp = self._dense.propagate()
            D, covp = D.cpu().numpy(), covp.cpu().numpy()
            if self._spec.pperm is not None:
                inv = self._spec._inv()
                D, covp = D[inv], covp[inv][:, inv]
            self._D, self._p = D, (self.pmean, covp)
        if self._p is None:
            plan = self._spec.plan(self.device)
            D, covp = plan.propagate(self.pmean.reshape(1, -1), self.cov.reshape(1, -1), self.yp_pdf.cov)
            self._D = D[0].cpu().numpy()
            self._p = (self.pmean, covp[0].cpu().numpy())
        return self._p

    p = property(_getp, doc="Best-fit parameters: (mean, covariance propagated as D C D^T).")

    @property
    def D(self):
        """d p[a] / d buf[i], buf = y (+) prior  (the derivative matrix of __init__.py:905-911)."""
        self._getp()
        return self._D

    @property
    def p_sdev(self):
        return np.sqrt(np.diag(self._getp()[1]))

    def check_roundoff(self, rtol=0.25, atol=1e-6):
        """__init__.py:884-895"""
        if not np.allclose(self.p_sdev, self.psdev, rtol=rtol, atol=atol):
            import warnings
            warnings.warn("Possible roundoff errors in fit.p; try svd cut.")

    # ---- batched drivers ---------------------------------------------------------------
    def _batch_args(self, kargs):
        """This fit's fitter arguments with ``kargs`` over them, as the batch drivers read them -> (the arguments of
        ``Plan.fit_batch``, kernel, loss, gsl).  tol and maxit default to this fit's; scipy's bounds=(lower, upper)
        in this fit's parameter order go to device order (as the single-fit path does).  kernel=: None (default, by
        problem shape), 1 / 2 / 4 warps per fit, or 32 / 'wave' -- the wave kernel, the fastest on saturated batches
        (10^5 ... 10^6 copies of a small model); see b200lm_set_team."""
        from .engine import POLICY
        args = dict(self.fitterargs, **kargs)
        bounds = args.get("bounds")
        if bounds is not None:
            bounds = tuple(self._spec.to_device(np.broadcast_to(np.asarray(b, dtype=float), (self._spec.np,)))
                           for b in bounds)
        fit = dict(tol=self.tol if args.get("tol") is None else args["tol"],
                   maxit=self.maxit if args.get("maxit") is None else args["maxit"],
                   scaler=args.get("scaler", "more"), polish=args.get("polish", 0), policy=args.get("policy", "trf"),
                   bounds=bounds)
        kernel = args.get("kernel")
        return fit, 32 if kernel == "wave" else kernel, args.get("loss", "linear"), POLICY.get(fit["policy"]) == 1

    def _batch(self, means, p0, tol=None, maxit=None, want_cov=True, **kargs):
        plan = self._spec.plan(self.device)
        args, kernel, loss, gsl = self._batch_args(dict(kargs, tol=tol, maxit=maxit))
        if loss != "linear":
            raise ValueError("batched fits with a robust loss (loss=%r) are not built: fit the copies one at a time "
                             "(fitter='b200_dense')" % (loss,))
        if gsl and args["bounds"] is not None:
            raise ValueError("b200_lm: policy='gsl' has no bound constraints")
        if kernel is not None:
            plan.set_team(int(kernel))
        try:
            out = plan.fit_batch(means, p0, want_cov=want_cov, **args)
        finally:
            if kernel is not None:
                plan.set_team(0)                 # (the plan is cached and shared: back to the default policy)
        return BatchFits(self, out)

    def bootstrap_means(self, n, seed=None, first=0):
        """Copies first .. first+n-1 of the bootstrap stream of y (+) prior means: mean + L z with
        L L^T = cov (gvar.bootstrap_iter as used at __init__.py:1615-1623), generated on the device
        by b200lm_bootstrap_means (counter-based Philox: any shard of copies is reproducible on its
        own, so ranks of a multi-GPU job generate only their slice)."""
        from .bootstrap import bootstrap_means
        if n is None:
            raise ValueError("n=None (the reference's endless iterator) is not supported: a batch is one launch; "
                             "pass the number of copies")
        if seed is None:
            seed = fresh_seed()
        self.last_seed = int(seed)
        if self._L is None:
            # L L^T = corrected covariance, from the device whitening's factors (no second eigen-decomposition on the host)
            self._L = self.yp_pdf.sqrt_cov()
        return bootstrap_means(self.yp_pdf.mean, self._L, n, int(seed), first=first,
                               device=self.device)

    def bootstrapped_fits(self, n=None, means=None, seed=None, **kargs):
        """All bootstrap fits in ONE launch (what bootstrapped_fit_iter loops over,
        __init__.py:1548-1642): p0 = self.pmean, means fluctuate, covariance fixed."""
        if means is None:
            means = self.bootstrap_means(n, seed)
        return self._batch(means, self.pmean, **kargs)

    def bootstrapped_fit_iter(self, n=None, datalist=None, seed=None, **kargs):
        """Iterator face of ``bootstrapped_fits`` (reference __init__.py:1548-1642).
        ``datalist`` yields mean vectors of y (+) prior (array form of the reference's data sets)."""
        if datalist is not None:
            # n = None: every data set of a FINITE datalist (an endless generator needs n)
            import itertools
            it = datalist if n is None else itertools.islice(datalist, int(n))
            means = np.array([np.asarray(m, dtype=float).reshape(-1) for m in it])
        else:
            means = None
        for f in self.bootstrapped_fits(n, means, seed, **kargs):
            yield f

    def simulated_means(self, n, pexact=None, add_priornoise=False, seed=None):
        """__init__.py:1471-1543: data means fcn(pexact) + noise, prior means fixed unless
        add_priornoise."""
        pexact = self.pmean if pexact is None else np.asarray(pexact, dtype=float)
        plan = self._spec.plan(self.device)
        # f(pexact) from the device functor: residuals with zero means and unit weights are
        # not available, so evaluate the registered host mirror (numpy) -- it is the same
        # call the reference makes on the host (__init__.py:1522).
        ny = self._spec.ny
        fexact = np.asarray(self.fcn(self.fcn.xrows(self.x, ny), pexact), dtype=float)
        means = self.bootstrap_means(n, seed)
        base = torch.as_tensor(self.yp_pdf.mean).to(means.device)
        noise = means - base[None, :]
        center = base.clone()
        center[:ny] = torch.as_tensor(fexact).to(means.device)
        if not add_priornoise and self.prior is not None:
            noise[:, ny:] = 0.0
        return center[None, :] + noise, pexact

    def simulated_fits(self, n, pexact=None, add_priornoise=False, seed=None, **kargs):
        """All simulated fits in ONE launch; whitening shared (``_yp_pdf``), p0 = pexact
        (__init__.py:1391-1469)."""
        means, pexact = self.simulated_means(n, pexact, add_priornoise, seed)
        bf = self._batch(means, pexact, **kargs)
        bf.pexact = pexact
        return bf

    def simulated_fit_iter(self, n=None, pexact=None, add_priornoise=False, seed=None, **kargs):
        for f in self.simulated_fits(n, pexact, add_priornoise, seed, **kargs):
            yield f

    def window_fits(self, masks, p0=None, **kargs):
        """Fit-window scan: the fits of the data windows ``masks`` (bool [nwin, ny]) in ONE launch.

        Window ``w`` is the fit ``nonlinear_fit(data=(x[m], y[m], ycov[m][:, m]), prior=self.prior, fcn=self.fcn,
        svdcut=self.svdcut, eps=self.eps, p0=p0)`` with ``m = masks[w]``: its y (+) prior covariance is this fit's input
        covariance restricted to its rows and the prior, whitened on its own.  ``p0``: [np] or [nwin, np], default this
        fit's ``pmean``.  Fitter arguments are this fit's unless given here (``tol``, ``maxit``, ``scaler``,
        ``polish``); ``kernel=`` is accepted and ignored (window batches run one warp per fit).  Returns a
        ``WindowScan``; its ``bootstrapped_fits`` fits every window's bootstrap copies in one more launch."""
        return WindowScan(self, masks, p0, **kargs)


class FitView(object):
    """One fit of a batch, with the attribute names of nonlinear_fit."""

    def __init__(self, parent, arrays, i):
        self.pmean = arrays["x"][i]
        self.cov = arrays["cov"][i] if arrays.get("cov") is not None else None
        self.psdev = np.sqrt(np.diag(self.cov)) if self.cov is not None else None
        self.chi2 = float(arrays["chi2"][i])
        self.dof = parent.dof
        self.nit = int(arrays["nit"][i])
        status = int(arrays["status"][i])
        self.stopping_criterion = STOPPING_CRITERION[status]
        self.error = None if status > 0 else "b200_lm: no convergence"
        self.logGBF = (None if parent.prior is None else
                       _logGBF(float(arrays["logdet"][i]), parent.yp_pdf.logdet, self.chi2, self.dof))
        self.tol = parent.tol
        self.svdn = parent.svdn

    @property
    def Q(self):
        return gammaQ(self.dof / 2., self.chi2 / 2.)


class BatchFits(object):
    """Results of a batch, resident on the device until asked for."""

    def __init__(self, parent, out):
        self.parent, self.out = parent, out
        self._np = None

    def arrays(self):
        if self._np is None:
            self._np = self.out.numpy()
        return self._np

    def __len__(self):
        return self.out.x.shape[0]

    def __iter__(self):
        a = self.arrays()
        for i in range(len(self)):
            yield FitView(self.parent, a, i)

    def pmean_stats(self):
        """Mean and covariance of the best-fit parameters over the batch, reduced on the
        device (the bootstrap estimate of fit.p, doc/source/testing.rst:419-432)."""
        ok = (self.out.status > 0)
        x = self.out.x[ok]
        m = x.mean(dim=0)
        d = x - m
        return m.cpu().numpy(), (d.T @ d / max(1, x.shape[0] - 1)).cpu().numpy()


class _Window(object):
    """What FitView and BatchFits read from the fit a result belongs to, for one window of a scan."""

    def __init__(self, parent, pdf, nchiv, np_):
        self.prior, self.tol = parent.prior, parent.tol
        self.yp_pdf, self.svdn = pdf, pdf.nmod
        self.dof = int(nchiv) - int(np_)


class WindowScan(object):
    """The central fits of a fit-window scan (``nonlinear_fit.window_fits``).

    Arrays over windows: ``pmean psdev`` [nwin, np], ``cov`` [nwin, np, np], ``chi2 dof Q logGBF svdn nit
    stopping_criterion error`` [nwin].  ``scan[w]`` has the attribute names of ``nonlinear_fit``; ``pdfs[w]`` is the
    window's whitening.  The scan owns its plan: the parent's (cached, shared) plan is left as it was.

    ``p``, ``D`` and ``p_sdev`` (computed on first access, like ``nonlinear_fit.p``): each window is its own fit of
    the same y (+) prior, so the windows' parameters are correlated.  ``D`` [nwin, np, N] is d pmean[w] / d (y, prior)
    (zero for data rows outside window w); ``p = (pmean, cov)`` with the joint covariance ``cov`` [nwin, np, nwin, np]:
    ``D[w] C D[v]^T`` between windows (C: this fit's input covariance of y (+) prior) and ``D[w] C_w D[w]^T`` within
    window w (C_w: its own svd-corrected covariance, so ``cov[w, :, w, :]`` is the window's own ``fit.p``
    covariance)."""

    def __init__(self, parent, masks, p0=None, **kargs):
        from .engine import Plan
        from .whiten import cov_blocks, whiten_blocks
        from .windows import check_masks, window_cov, window_weights
        # kernel= is ignored: window batches always run one warp per fit
        self.args, _, loss, gsl = parent._batch_args(kargs)
        refuse = lambda what: ValueError("b200_lm: %s not built for window scans" % what)
        if self.args["bounds"] is not None:
            raise refuse("bounds are")
        if loss != "linear":
            raise refuse("a robust loss is")
        if gsl:
            raise refuse("policy='gsl' is")
        if any(parent.noise):
            raise refuse("fits made with noise are")
        spec = parent._spec
        self.parent, self.device = parent, parent.device
        self.np, self.ny = spec.np, spec.ny
        self.masks = check_masks(masks, self.ny)
        self.nwin = self.masks.shape[0]
        pdf = parent.yp_pdf
        cov = pdf.cov_in if pdf.cov_in is not None else pdf.sdev_in
        wins = [window_cov(cov, self.ny, m) for m in self.masks]
        # the correlated blocks of every window, whitened in ONE call (b200lm_whiten: one CTA per block, and a block's
        # result depends on that block alone -- each window's whitening is bit for bit that of a PDF of its own)
        blocks = [cov_blocks(c)[1] if c.ndim == 2 else [] for _, c in wins]
        ns = [b.size for bl in blocks for b in bl]
        if ns:
            flat = np.concatenate([c[np.ix_(b, b)].reshape(-1) for (_, c), bl in zip(wins, blocks) for b in bl])
            W, Cc, nout, nmod, ld = whiten_blocks(np.array(ns), flat, pdf.svdcut, pdf.eps, self.device)
        self.pdfs = []
        o = k = 0
        for (sel, c), bl in zip(wins, blocks):
            nb, nel = len(bl), sum(b.size ** 2 for b in bl)
            part = (W[o:o + nel], Cc[o:o + nel], nout[k:k + nb], nmod[k:k + nb], ld[k:k + nb]) if nb else None
            self.pdfs.append(PDF(pdf.mean[sel], c, svdcut=pdf.svdcut, eps=pdf.eps, device=self.device,
                                 _whitened=part))
            o, k = o + nel, k + nb
        self.sels = [sel for sel, _ in wins]
        desc = window_weights(self.sels, [p.i_invwgts for p in self.pdfs])
        self.nchiv = desc["nchiv"]
        self.plan = Plan(spec.functor, spec.np, spec.ny, spec.x, spec.i_invwgts, noprior=spec.noprior,
                         device=self.device)
        self.plan.set_windows(desc)
        self.windows = [_Window(parent, p, n, self.np) for p, n in zip(self.pdfs, self.nchiv)]
        self.dof = np.array([w.dof for w in self.windows])
        self.svdn = np.array([w.svdn for w in self.windows])
        p0 = parent.pmean if p0 is None else np.asarray(p0, dtype=float)
        self.p0 = np.array(np.broadcast_to(p0, (self.nwin, self.np)))
        out = self._fit(spec.mean, self.p0, self.nwin)
        a = out.numpy()
        self.out, self._arrays = out, a
        self.pmean, self.cov, self.chi2, self.nit = a["x"], a["cov"], a["chi2"], a["nit"]
        self.psdev = np.sqrt(np.diagonal(self.cov, axis1=1, axis2=2))
        self.Q = gammaQ(self.dof / 2., self.chi2 / 2.)
        self.logGBF = (None if parent.prior is None else
                       np.array([_logGBF(a["logdet"][w], p.logdet, a["chi2"][w], d)
                                 for w, (p, d) in enumerate(zip(self.pdfs, self.dof))]))
        self.stopping_criterion = np.array([STOPPING_CRITERION[int(s)] for s in a["status"]])
        self.error = np.array([None if s > 0 else "b200_lm: no convergence" for s in a["status"]], dtype=object)
        self._p = None

    def _getp(self):
        if self._p is None:
            from .windows import window_corrections
            # J at the solutions: the central batch once more, with f and J (the same fits, so the same bits)
            J = self._fit(self.parent._spec.mean, self.p0, self.nwin, want_fJ=True).J
            pdf = self.parent.yp_pdf
            C = pdf.cov_in if pdf.cov_in is not None else np.diag(pdf.sdev_in ** 2)
            D, covp = self.plan.window_propagate(self.out.cov, J, C, window_corrections(self.pdfs))
            self._D = D.cpu().numpy()
            self._p = (self.pmean, covp.cpu().numpy())
        return self._p

    p = property(_getp, doc="(pmean [nwin, np], joint covariance [nwin, np, nwin, np] of every window's fit.p).")

    @property
    def D(self):
        """d pmean[w, a] / d buf[i], buf = y (+) prior: [nwin, np, N]."""
        self._getp()
        return self._D

    @property
    def p_sdev(self):
        """[nwin, np]: standard deviations of ``p``."""
        c = self._getp()[1].reshape(self.nwin * self.np, -1)
        return np.sqrt(np.diagonal(c)).reshape(self.nwin, self.np)

    def _fit(self, means, p0, B, want_fJ=False):
        return self.plan.fit_batch(means, p0, B=B, want_fJ=want_fJ, **self.args)

    def __len__(self):
        return self.nwin

    def __getitem__(self, w):
        return FitView(self.windows[w], self._arrays, w)

    def bootstrapped_fits(self, n=None, seed=None, means=None):
        """n bootstrap copies of every window in ONE launch (nwin * n fits).  The copies are the parent's
        ``bootstrap_means(n, seed)`` (or ``means`` [n, N]); every window of copy j reads its rows from the same row j,
        and the copies of window w start from the window's central ``pmean``."""
        if means is None:
            means = self.parent.bootstrap_means(n, seed)
        n = int(means.shape[0])
        return WindowBootstrap(self, self._fit(means, self.pmean, self.nwin * n), n)


class WindowBootstrap(object):
    """The bootstrap copies of a window scan: fit b is copy b % n of window b // n."""

    def __init__(self, scan, out, n):
        self.scan, self.out, self.n = scan, out, n

    def __len__(self):
        return self.out.x.shape[0]

    def arrays(self):
        return self.out.numpy()

    def window(self, w):
        """BatchFits of window w's copies (arrays(), iteration, pmean_stats())."""
        s = slice(w * self.n, (w + 1) * self.n)
        o = self.out
        part = BatchResult(*[None if t is None else t[s] for t in (o.x, o.chi2, o.cov, o.logdet, o.nit, o.status,
                                                                    o.f, o.J)])
        return BatchFits(self.scan.windows[w], part)


class WAvg(object):
    """Result of ``wavg``: ``mean``, ``cov``, ``sdev`` of the average plus the attributes the reference
    attaches (``chi2 dof Q time svdcorrection-free fit``; src/lsqfit/_extras.py:412-431)."""

    def __init__(self, fit):
        self.fit = fit
        self.mean, self.cov, self.sdev = fit.pmean, fit.cov, fit.psdev
        self.chi2, self.dof, self.Q, self.time = fit.chi2, fit.dof, fit.Q, fit.time
        self.svdn = fit.svdn


def wavg(means, cov, index=None, nparam=None, svdcut=False, eps=False, **fitterargs):
    """Weighted average of correlated estimates (array form of ``lsqfit.wavg``,
    src/lsqfit/_extras.py:358-516): a least-squares fit of the data ``means`` (flat, covariance ``cov``:
    matrix or vector of standard deviations) to ``f_i = p[index[i]]`` without a prior, started at the
    plain average of the inputs (:478-494) -- run on the device with the ``gather`` functor.

    ``means`` may be 2-d ``[M, np]`` (M estimates of np quantities; then ``index`` defaults to
    ``arange(np)`` tiled M times); ragged inputs pass a flat ``means`` and an explicit ``index``."""
    means = np.asarray(means, dtype=float)
    if index is None:
        if means.ndim != 2:
            means = means.reshape(-1, 1)
        M, npar = means.shape
        index = np.tile(np.arange(npar), M)
    index = np.asarray(index, dtype=int).reshape(-1)
    y = means.reshape(-1)
    if index.size != y.size:
        raise ValueError("index and means disagree on the number of data")
    npar = int(index.max()) + 1 if nparam is None else int(nparam)
    p0 = np.zeros(npar)
    cnt = np.zeros(npar)
    np.add.at(p0, index, y)
    np.add.at(cnt, index, 1.0)
    if np.any(cnt == 0):
        raise ValueError("every component of the average needs at least one datum")
    fit = nonlinear_fit(data=(index.astype(float), y, cov), fcn=Functor("gather"), p0=p0 / cnt, svdcut=svdcut, eps=eps,
                        **fitterargs)
    return WAvg(fit)
