"""Parameter distributions: lsqfit's ``log(k)``, ``sqrt(k)`` and ``BufferDict.uniform`` prior keys (pure numpy).

In lsqfit a prior key ``f(k)`` makes the fit parameter ``p = f(q)``, and the model reads ``q = f^-1(p)`` under the key
``k``: ``log(E)`` keeps ``E = exp(p)`` positive, ``sqrt(a)`` gives ``a = p^2``, and a name made by
``gvar.BufferDict.uniform(fname, lo, hi)`` gives ``q = lo + (hi - lo) (1 + erf(p / sqrt 2)) / 2``, a parameter with a
uniform prior on (lo, hi).  The fit itself runs in p (prior residuals, p0, x, cov, fit.p, logGBF); only the model sees
``q = T(p)``, and its Jacobian columns pick up ``T'(p)``.

Codes, in device parameter order (``b200lm_set_param_dist``): 0 plain, 1 log, 2 sqrt, 3 uniform (with lo, hi).
The ``pdist=`` argument of ``lsqfit_b200.nonlinear_fit`` is the array form: one entry per parameter, each ``None``,
``'log'``, ``'sqrt'`` or ``('uniform', lo, hi)``.
"""
import math
import re

import numpy as np

PLAIN, LOG, SQRT, UNIFORM = 0, 1, 2, 3
NAMES = {None: PLAIN, "log": LOG, "sqrt": SQRT, "uniform": UNIFORM}

_KEY = re.compile(r"^([^()]+)\((.+)\)$")
_SQRT1_2 = 1.0 / math.sqrt(2.0)
_INV_SQRT_2PI = 1.0 / math.sqrt(2.0 * math.pi)


def parse_key(key):
    """``'f(k)'`` -> ``('f', 'k')``; any other key (not a string, or no ``f(...)`` form) -> ``(None, key)``.
    The same form gvar's ``BufferDict`` recognises for distribution keys."""
    if isinstance(key, str):
        m = _KEY.match(key)
        if m:
            return m.group(1), m.group(2)
    return None, key


def transform(code, lo, hi, p):
    """q = T(p) and T'(p) for arrays of codes, bounds and parameters (broadcast); the device computes the same
    (csrc/lm_kernel.cuh: param_transform)."""
    from scipy.special import erfc
    code, lo, hi, p = np.broadcast_arrays(np.asarray(code), np.asarray(lo, dtype=float), np.asarray(hi, dtype=float),
                                          np.asarray(p, dtype=float))
    q, dq = p.copy(), np.ones_like(p)
    e = np.exp(np.where(code == LOG, p, 0.0))
    q = np.where(code == LOG, e, q)
    dq = np.where(code == LOG, e, dq)
    q = np.where(code == SQRT, p * p, q)
    dq = np.where(code == SQRT, 2.0 * p, dq)
    w = hi - lo
    u = code == UNIFORM
    q = np.where(u, lo + w * (0.5 * erfc(-_SQRT1_2 * p)), q)
    dq = np.where(u, w * _INV_SQRT_2PI * np.exp(-0.5 * p * p), dq)
    return q, dq


def codes(pdist, np_):
    """The array form ``pdist`` (None, or one entry per parameter: None, 'log', 'sqrt' or ('uniform', lo, hi)) ->
    (code int32 [np], lo [np], hi [np]), or None when every entry is plain (such a fit is an ordinary fit)."""
    if pdist is None:
        return None
    pdist = list(pdist)
    if len(pdist) != np_:
        raise ValueError("pdist: one entry per parameter (%d), got %d" % (np_, len(pdist)))
    code = np.zeros(np_, dtype=np.int32)
    lo, hi = np.zeros(np_), np.ones(np_)
    for j, d in enumerate(pdist):
        if isinstance(d, tuple) and len(d) == 3 and d[0] == "uniform":
            a, b = float(d[1]), float(d[2])
            if not (np.isfinite(a) and np.isfinite(b) and a < b):
                raise ValueError("pdist[%d]: a uniform distribution needs finite lo < hi, got (%r, %r)" % (j, d[1], d[2]))
            code[j], lo[j], hi[j] = UNIFORM, a, b
        elif (d is None or isinstance(d, str)) and d in NAMES and d != "uniform":
            code[j] = NAMES[d]
        else:
            raise ValueError("pdist[%d]: unknown distribution %r (None, 'log', 'sqrt' or ('uniform', lo, hi))" % (j, d))
    if not code.any():
        return None
    return code, lo, hi


def entries(code, lo, hi):
    """(code, lo, hi) -> the array form of ``codes`` (one entry per parameter)."""
    out = []
    for c, a, b in zip(code, lo, hi):
        out.append(("uniform", float(a), float(b)) if c == UNIFORM else {PLAIN: None, LOG: "log", SQRT: "sqrt"}[int(c)])
    return out


# points the classifier probes a distribution function at (both signs, small and large |p|, no point where a
# square and an exponential could agree)
_PROBE = np.array([-3.1, -1.7, -0.9, -0.35, 0.15, 0.6, 1.3, 2.45])
_RTOL = 1e-13


def classify(g, rtol=_RTOL):
    """The code and bounds of the distribution function ``g`` (what gvar's ``BufferDict`` applies to the values stored
    under ``f(k)`` to give ``k``): ``(LOG, 0, 1)`` if g is exp, ``(SQRT, 0, 1)`` if g is the square, ``(UNIFORM, lo, hi)``
    with ``lo = g(-40)``, ``hi = g(40)`` if g is the uniform form of the module docstring.  g is checked at a spread of
    points to ``rtol`` relative; names are not trusted.  Anything else raises ValueError: the engine has no other
    transform, and a fit with a different function would be a different model."""
    def call(x):
        try:
            v = float(np.asarray(g(float(x)), dtype=float))
        except Exception as e:                                  # noqa: BLE001  (whatever g raises, it is not one of ours)
            raise ValueError("distribution function %r cannot be evaluated at %r: %s" % (g, x, e))
        return v
    vals = np.array([call(x) for x in _PROBE])
    close = lambda a, b, scale: bool(np.all(np.abs(a - b) <= rtol * scale))
    if np.all(np.isfinite(vals)):
        ex = np.exp(_PROBE)
        if close(vals, ex, ex):
            return LOG, 0.0, 1.0
        sq = _PROBE * _PROBE
        if close(vals, sq, sq):
            return SQRT, 0.0, 1.0
        lo, hi = call(-40.0), call(40.0)
        if np.isfinite(lo) and np.isfinite(hi) and lo < hi:
            q, _ = transform(UNIFORM, lo, hi, _PROBE)
            if close(vals, q, max(abs(lo), abs(hi), hi - lo)):
                return UNIFORM, lo, hi
    raise ValueError("distribution function %r is not one the device fit kernels have: log(k) (exp), sqrt(k) (square) "
                     "and BufferDict.uniform names are" % (g,))
