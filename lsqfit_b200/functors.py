"""Host-side mirror of the CUDA device-functor registry (csrc/functors.cuh).

In the reference the fit function is an arbitrary Python callable ``fcn(x, p)``
(src/lsqfit/__init__.py:566, 1997-2042).  The B200 engine instead evaluates the
model on the device, so the user picks a ``Functor`` from this registry.  A
``Functor`` is still a Python callable with the reference's ``fcn(x, p)`` signature,
written with numpy ufuncs only, so that unmodified lsqfit code which calls the fit
function on the host (``fit.format``, ``simulated_data_iter``, the CPU fitters, gvar
arithmetic -- src/lsqfit/__init__.py:615, 1352-1354, 1522) keeps working.
"""
import numpy as np

# family ids == enum FunctorFamily in csrc/functors.cuh
FAMILY = dict(
    multiexp=0, multiexp_de=1, simple=2, offset_exp=3, poly=4, exp_poly=5, xerr_logistic=6, gather=7,
    multiexp_shared2=8, multiexp_shared3=9,
    misra1a=10, chwirut=11, lanczos=12, gauss=13, danwood=14, misra1b=15, misra1c=16,
    misra1d=17, kirby2=18, hahn1=19, nelson=20, mgh17=21, roszman1=22, enso=23, mgh09=24,
    rat42=25, mgh10=26, eckerle4=27, rat43=28, bennett5=29, spline_poly=30,
)
NX = dict(simple=2, nelson=2, multiexp_shared2=2, multiexp_shared3=2, spline_poly=2)          # every other family reads one x column

# NIST StRD problem name -> functor family (examples/nist.py)
NIST_FORM = dict(
    misra1a="misra1a", boxbod="misra1a", chwirut1="chwirut", chwirut2="chwirut",
    lanczos1="lanczos", lanczos2="lanczos", lanczos3="lanczos",
    gauss1="gauss", gauss2="gauss", gauss3="gauss", danwood="danwood",
    misra1b="misra1b", misra1c="misra1c", misra1d="misra1d", kirby2="kirby2",
    hahn1="hahn1", thurber="hahn1", nelson="nelson", mgh17="mgh17",
    roszman1="roszman1", enso="enso", mgh09="mgh09", rat42="rat42",
    mgh10="mgh10", eckerle4="eckerle4", rat43="rat43", bennett5="bennett5",
)

_pi = np.pi


def _col(x, c=0):
    x = np.asarray(x)
    return x[:, c] if x.ndim == 2 else x


def _multiexp(x, p):
    t = _col(x)
    K = len(p) // 2
    return sum(p[k] * np.exp(-p[K + k] * t) for k in range(K))


def _multiexp_de(x, p):
    t = _col(x)
    K = len(p) // 2
    E = np.cumsum(p[K:])
    return sum(p[k] * np.exp(-E[k] * t) for k in range(K))


def _multiexp_shared(M):
    """M data sets with shared energies: x rows (t, m); p = [a^(0)(K), ..., a^(M-1)(K), E(K)]"""
    def f(x, p):
        x = np.asarray(x)
        t, m = x[:, 0], x[:, 1].astype(int)
        p = np.asarray(p)
        K = len(p) // (M + 1)
        a = p[:M * K].reshape(M, K)
        return sum(a[m, k] * np.exp(-p[M * K + k] * t) for k in range(K))
    return f


def _simple(x, p):
    x = np.asarray(x)
    t, kind = x[:, 0], x[:, 1]
    e = np.exp(p[0] + p[1] * t)
    return np.where(kind == 0, e, p[1] / p[0])


def _poly(x, p):
    t = _col(x)
    return sum(p[n] * t ** n for n in range(len(p)))


def _xerr(x, p):
    return p[0] / ((1.0 + np.exp(p[1] - p[2] * p[4:])) ** (1.0 / p[3]))


def _enso(x, b):
    t = _col(x)
    return (b[0] + b[1] * np.cos(2 * _pi * t / 12) + b[2] * np.sin(2 * _pi * t / 12)
            + b[4] * np.cos(2 * _pi * t / b[3]) + b[5] * np.sin(2 * _pi * t / b[3])
            + b[7] * np.cos(2 * _pi * t / b[6]) + b[8] * np.sin(2 * _pi * t / b[6]))


def _gauss(x, b):
    t = _col(x)
    return (b[0] * np.exp(-b[1] * t) + b[2] * np.exp(-(t - b[3]) ** 2 / b[4] ** 2)
            + b[5] * np.exp(-(t - b[6]) ** 2 / b[7] ** 2))


SPLINE_SHAPES = {13: (4, 5), 8: (4, 0), 12: (6, 0)}      # np -> (knots, polynomial coefficients): csrc/inst_misc_b.cu


def _spline_poly(x, p):
    """host mirror of csrc/functors.cuh: SplinePolyBody (Steffen's monotonic spline through the knots p[:NK], p[NK:2NK],
    end cubics continued outside, plus sum_i p[2NK+i] am^(2+2i); the model of reference examples/spline.py:50-60)"""
    x = np.asarray(x, dtype=float)
    p = np.asarray(p, dtype=float)
    nk, ncf = SPLINE_SHAPES[len(p)]
    xk, yk = p[:nk], p[nk:2 * nk]
    h = np.diff(xk)
    s = np.diff(yk) / h
    yp = np.zeros(nk)
    pi = (s[:-1] * h[1:] + s[1:] * h[:-1]) / (h[:-1] + h[1:])
    yp[1:-1] = (np.sign(s[:-1]) + np.sign(s[1:])) * np.minimum(np.minimum(np.abs(s[:-1]), np.abs(s[1:])), 0.5 * np.abs(pi))

    def end(s0, s1, h0, h1):
        r = h0 / (h0 + h1)
        pe = s0 * (1 + r) - s1 * r
        return 0.0 if pe * s0 <= 0 else (2 * s0 if abs(pe) > 2 * abs(s0) else pe)
    yp[0], yp[-1] = end(s[0], s[1], h[0], h[1]), end(s[-1], s[-2], h[-1], h[-2])
    m = x[:, 0]
    i = np.clip(np.searchsorted(xk[1:-1], m, side="left"), 0, nk - 2)
    t = m - xk[i]
    a = (yp[i] + yp[i + 1] - 2 * s[i]) / h[i] ** 2
    b = (3 * s[i] - 2 * yp[i] - yp[i + 1]) / h[i]
    f = ((a * t + b) * t + yp[i]) * t + yk[i]
    for k in range(ncf):
        f = f + p[2 * nk + k] * x[:, 1] ** (2 + 2 * k)
    return f


_HOST = dict(
    multiexp=_multiexp,
    multiexp_de=_multiexp_de,
    multiexp_shared2=_multiexp_shared(2),
    multiexp_shared3=_multiexp_shared(3),
    simple=_simple,
    offset_exp=lambda x, p: p[0] + p[1] * np.exp(-p[2] * _col(x)),
    poly=_poly,
    exp_poly=lambda x, p: np.exp(-_poly(x, p)),
    xerr_logistic=_xerr,
    gather=lambda x, p: np.asarray(p)[np.asarray(_col(x)).astype(int)],
    spline_poly=_spline_poly,
    misra1a=lambda x, b: b[0] * (1 - np.exp(-b[1] * _col(x))),
    chwirut=lambda x, b: np.exp(-b[0] * _col(x)) / (b[1] + b[2] * _col(x)),
    lanczos=lambda x, b: (b[0] * np.exp(-b[1] * _col(x)) + b[2] * np.exp(-b[3] * _col(x))
                          + b[4] * np.exp(-b[5] * _col(x))),
    gauss=_gauss,
    danwood=lambda x, b: b[0] * _col(x) ** b[1],
    misra1b=lambda x, b: b[0] * (1 - (1 + b[1] * _col(x) / 2) ** (-2)),
    misra1c=lambda x, b: b[0] * (1 - (1 + 2 * b[1] * _col(x)) ** (-.5)),
    misra1d=lambda x, b: b[0] * b[1] * _col(x) * ((1 + b[1] * _col(x)) ** (-1)),
    kirby2=lambda x, b: ((b[0] + b[1] * _col(x) + b[2] * _col(x) ** 2)
                         / (1 + b[3] * _col(x) + b[4] * _col(x) ** 2)),
    hahn1=lambda x, b: ((b[0] + b[1] * _col(x) + b[2] * _col(x) ** 2 + b[3] * _col(x) ** 3)
                        / (1 + b[4] * _col(x) + b[5] * _col(x) ** 2 + b[6] * _col(x) ** 3)),
    nelson=lambda x, b: b[0] - b[1] * _col(x, 0) * np.exp(-b[2] * _col(x, 1)),
    mgh17=lambda x, b: b[0] + b[1] * np.exp(-_col(x) * b[3]) + b[2] * np.exp(-_col(x) * b[4]),
    roszman1=lambda x, b: b[0] - b[1] * _col(x) - np.arctan(b[2] / (_col(x) - b[3])) / _pi,
    enso=_enso,
    mgh09=lambda x, b: b[0] * (_col(x) ** 2 + _col(x) * b[1]) / (_col(x) ** 2 + _col(x) * b[2] + b[3]),
    rat42=lambda x, b: b[0] / (1 + np.exp(b[1] - b[2] * _col(x))),
    mgh10=lambda x, b: b[0] * np.exp(b[1] / (_col(x) + b[2])),
    eckerle4=lambda x, b: (b[0] / b[1]) * np.exp(-0.5 * ((_col(x) - b[2]) / b[1]) ** 2),
    rat43=lambda x, b: b[0] / ((1 + np.exp(b[1] - b[2] * _col(x))) ** (1 / b[3])),
    bennett5=lambda x, b: b[0] * (b[1] + _col(x)) ** (-1 / b[2]),
)


# name -> UserFunctor of every model loaded at run time (lsqfit_b200/user_functor.py: cuda_functor)
USER = {}


class Functor(object):
    """A registered device model; also callable on the host as ``fcn(x, p)``.

    ``Functor('multiexp')`` works for any parameter count the device registry was
    compiled for (``lsqfit_b200.available()``); the count is taken from ``p0`` / the
    prior when a fit is set up.  The name of a model loaded with ``cuda_functor`` resolves too.
    """

    def __init__(self, name):
        if name in USER:
            u = USER[name]
            self.name, self.family, self.nx, self._host = u.name, u.family, u.nx, u._host
            return
        if name not in FAMILY:
            raise ValueError("unknown functor family: %s (known: %s)" % (name, ", ".join(sorted(FAMILY) + sorted(USER))))
        self.name = name
        self.family = FAMILY[name]
        self.nx = NX.get(name, 1)
        self._host = _HOST[name]

    def __call__(self, x, p):
        return self._host(x, p)

    def xrows(self, x, ny):
        """x as the row-major [ny][nx] float array the device functor reads."""
        if x is None or x is False:
            return np.zeros((ny, self.nx))
        x = np.asarray(x, dtype=float)
        if x.ndim == 1:
            x = x[:, None]
        if x.shape != (ny, self.nx):
            raise ValueError("x must have shape (%d, %d) for functor %s; got %s"
                             % (ny, self.nx, self.name, x.shape))
        return np.ascontiguousarray(x)

    def __repr__(self):
        return "Functor(%r)" % self.name
