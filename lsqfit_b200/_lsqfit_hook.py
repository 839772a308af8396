"""Hook for a real (unmodified) lsqfit installation.  Needs lsqfit + gvar; neither is
available in the build container, so this module is exercised only by the
skip-if-missing integration test (tests/test_lsqfit_integration.py).

Seams used (reference src/lsqfit/__init__.py):
  :110-128, 453   ``nonlinear_fit.FITTERS`` registry        -> add 'b200_lm'
  :571, 2074      ``lsqfit._build_chiv_chivw`` module global -> wrap, attach ChivSpec
  :1997-2012      flatfcn is a functools.partial whose keywords hold fcn, x, ...
"""
import functools

import numpy as np

from .fitter import ChivSpec, b200_lm
from .functors import Functor


class _ChivProxy(object):
    """Behaves like the reference's chiv object, plus the ``b200`` attribute."""

    def __init__(self, chiv, spec):
        self._chiv, self.b200 = chiv, spec

    def __call__(self, *args, **kargs):
        return self._chiv(*args, **kargs)


def _find_functor(flatfcn):
    """(functor, x, pperm) behind the reference's flatfcn (a functools.partial whose keywords hold fcn, x and the
    parameter / data buffers, src/lsqfit/__init__.py:1997-2012), or (None, None, None).  A MultiFitter closure
    (``_multifitfcn``, _extras.py:1816-1829) whose models are all device-backed maps onto one composite functor."""
    from .multifit import composite
    f = flatfcn
    while isinstance(f, functools.partial):
        kw = f.keywords or {}
        fcn = kw.get("fcn")
        if isinstance(fcn, Functor):
            return fcn, kw.get("x", False), None
        if hasattr(fcn, "flatmodels") and "po" in kw and "yo" in kw:
            c = composite(fcn, kw["po"], kw["yo"])
            if c is not None:
                return c
        f = f.func
    return None, None, None


def _prior_size(prior):
    """number of prior entries: a GVar array / BufferDict (``.size`` / ``.flat``), or the (mean, cov) pair of the
    array-form test double"""
    if isinstance(prior, tuple):
        m = prior[0]
        if isinstance(m, dict):
            return int(sum(np.size(v) for v in m.values()))
        return int(np.size(m))
    if hasattr(prior, "size"):
        return int(prior.size)
    return int(np.size(getattr(prior, "flat", prior)[:]))


def _prior_dist(prior):
    """(code, lo, hi) in the order of the flat prior buffer from the distribution keys of a dictionary prior (``log(E)``,
    ``sqrt(a)``, a ``BufferDict.uniform`` name), or None.  Each key's function is classified from a probe: a dictionary
    of the prior's own type holding one value under ``f(k)``, read under ``k`` -- names are not trusted.  A prior whose
    type does not resolve ``k`` (a plain dict) or a function the device does not have raises ValueError."""
    from . import pdist as P
    d = prior[0] if isinstance(prior, tuple) else prior
    if not hasattr(d, "keys"):
        return None
    keys = list(d.keys())
    if not any(P.parse_key(k)[0] is not None for k in keys):
        return None
    n = _prior_size(prior)
    code, lo, hi = np.zeros(n, dtype=np.int32), np.zeros(n), np.ones(n)
    cls, off = type(d), 0
    for k in keys:
        m = int(np.size(d[k]))
        sl = d.slice(k) if hasattr(d, "slice") else slice(off, off + m)
        off += m
        fname, base = P.parse_key(k)
        if fname is None:
            continue
        try:
            c, a, b = P.classify(lambda v, k=k, base=base: cls({k: v})[base])
        except ValueError as e:
            raise ValueError("prior key %r: %s" % (k, e))
        code[sl], lo[sl], hi[sl] = c, a, b
    return (code, lo, hi) if code.any() else None


def install(lsqfit):
    if getattr(lsqfit, "_b200lm_installed", False):
        return lsqfit
    reference_build = lsqfit._build_chiv_chivw

    def _build_chiv_chivw(yp_pdf, fcn, prior):
        cv, cvw = reference_build(yp_pdf=yp_pdf, fcn=fcn, prior=prior)
        functor, x, pperm = _find_functor(fcn)
        if functor is None:
            return cv, cvw                      # ordinary Python fcn: CPU fitters only
        noprior = prior is None
        N = len(yp_pdf.mean)
        npar = 0 if noprior else _prior_size(prior)
        ny = N - npar
        if noprior:
            npar = None                         # taken from p0 by the fitter
        spec = ChivSpec(functor, x, yp_pdf, noprior, ny, npar if npar is not None else -1, pperm=pperm)
        if not noprior:
            # distribution keys: the device fits them with codes; one it cannot fit is refused by the device fitters
            # only (the CPU fitters evaluate fcn on the prior's own dictionary and are not concerned)
            try:
                spec.pdist = _prior_dist(prior)
            except ValueError as e:
                spec.pdist_error = str(e)
        return _ChivProxy(cv, spec), cvw

    class b200_lm_plugin(b200_lm):
        def __init__(self, x0, n, f, **kargs):
            spec = getattr(f, "b200", None)
            if spec is not None and spec.np < 0:
                spec.np = len(x0)
            b200_lm.__init__(self, x0, n, f, **kargs)

    from .dense import b200_dense
    lsqfit._build_chiv_chivw = _build_chiv_chivw
    lsqfit.nonlinear_fit.FITTERS["b200_lm"] = b200_lm_plugin
    lsqfit.nonlinear_fit.FITTERS["b200_dense"] = b200_dense
    lsqfit.b200_lm = b200_lm_plugin
    lsqfit._b200lm_installed = True
    return lsqfit
