"""Parameter distributions without a device: lsqfit's prior key forms, the classifier of distribution functions, the
transforms and their derivatives, an oracle fit with ``log(E)`` against scipy on an explicit chiv, and the refusals
that come before any device work."""
import math

import numpy as np
import pytest
from scipy.special import erf

from lsqfit_b200 import configs
from lsqfit_b200 import pdist as P
from oracle import dual as D
from oracle.models import multiexp


def uniform_form(lo, hi, c=1.0 / math.sqrt(2.0)):
    """gvar's documented BufferDict.uniform function (c: the constant in erf(p c))"""
    return lambda p: lo + (hi - lo) * (1.0 + erf(p * c)) / 2.0


def t_dual(code, lo, hi, p):
    """q = T(p) on the oracle's dual numbers (chain rule: dq = T'(p) dp)"""
    if isinstance(p, D.Dual):
        q, dq = P.transform(code, lo, hi, p.v)
        return D.Dual(q, dq[:, None] * p.d)
    return P.transform(code, lo, hi, p)[0]


def test_parse_key():
    assert P.parse_key("log(E)") == ("log", "E")
    assert P.parse_key("sqrt(a1)") == ("sqrt", "a1")
    assert P.parse_key("erfinv(50a)") == ("erfinv", "50a")
    assert P.parse_key("log(f(x))") == ("log", "f(x)")
    assert P.parse_key("E") == (None, "E")
    assert P.parse_key("(E)") == (None, "(E)")
    assert P.parse_key("log()") == (None, "log()")
    assert P.parse_key(("a", 1)) == (None, ("a", 1))


def test_classify_accepts():
    assert P.classify(np.exp) == (P.LOG, 0.0, 1.0)
    assert P.classify(lambda p: p * p) == (P.SQRT, 0.0, 1.0)
    assert P.classify(np.square) == (P.SQRT, 0.0, 1.0)
    for lo, hi in ((0.0, 1.0), (-2.5, 7.0), (1e-3, 2e-3), (-1e4, -10.0), (100.0, 1e6)):
        code, a, b = P.classify(uniform_form(lo, hi))
        assert code == P.UNIFORM
        assert abs(a - lo) <= 1e-13 * max(abs(lo), abs(hi)) and abs(b - hi) <= 1e-13 * max(abs(lo), abs(hi))


@pytest.mark.parametrize("g", [np.tanh, lambda p: 2.0 * p + 1.0, lambda p: p, np.sinh, np.expm1,
                               lambda p: np.exp(p) * (1 + 1e-11), lambda p: p * p * p, lambda p: abs(p),
                               uniform_form(0.0, 1.0, c=0.7071), uniform_form(-1.0, 3.0, c=0.5),
                               lambda p: uniform_form(0.0, 1.0)(p) * (1.0 + 1e-9 * p)])
def test_classify_refuses(g):
    with pytest.raises(ValueError):
        P.classify(g)


def test_classify_refuses_a_function_that_raises():
    def g(p):
        raise TypeError("no")
    with pytest.raises(ValueError):
        P.classify(g)


def test_derivative_matches_finite_differences():
    p = np.linspace(-3.0, 3.0, 25)
    h = 1e-6
    for code, lo, hi in ((P.PLAIN, 0, 1), (P.LOG, 0, 1), (P.SQRT, 0, 1), (P.UNIFORM, -2.0, 5.0), (P.UNIFORM, 1e2, 1e3)):
        q, dq = P.transform(code, lo, hi, p)
        fd = (P.transform(code, lo, hi, p + h)[0] - P.transform(code, lo, hi, p - h)[0]) / (2 * h)
        assert np.max(np.abs(dq - fd) / np.maximum(np.abs(dq), 1e-3 * max(1.0, hi - lo))) < 1e-7, code
    q, _ = P.transform(P.LOG, 0, 1, p)
    assert np.array_equal(q, np.exp(p))
    q, _ = P.transform(P.UNIFORM, 2.0, 4.0, p)
    assert np.allclose(q, uniform_form(2.0, 4.0)(p), rtol=1e-15, atol=4e-16)


def test_codes_array_form():
    c = P.codes([None, "log", "sqrt", ("uniform", -1.0, 2.0)], 4)
    assert list(c[0]) == [0, 1, 2, 3] and c[0].dtype == np.int32
    assert c[1][3] == -1.0 and c[2][3] == 2.0
    assert P.entries(*c) == [None, "log", "sqrt", ("uniform", -1.0, 2.0)]
    assert P.codes(None, 3) is None
    assert P.codes([None, None], 2) is None                     # all plain: an ordinary fit


@pytest.mark.parametrize("bad", [["log"], ["log", "exp"], ["log", ("uniform", 1.0, 1.0)],
                                 ["log", ("uniform", 0.0, np.inf)], ["log", ("uniform", 2.0, 1.0)],
                                 ["log", ("uniform", 0.0)], ["log", 3]])
def test_codes_refuses(bad):
    with pytest.raises(ValueError):
        P.codes(bad, 2)


def _explicit_problem(K=2):
    cfg = configs.correlator(K)
    ny, npar = cfg["ny"], cfg["np"]
    pm = cfg["prior_mean"].copy()
    ps = cfg["prior_sdev"].copy()
    # log(E): the prior of log E_k is log(0.5 k)(0.4)
    pm[K:] = np.log(cfg["ptrue"][K:])
    ps[K:] = 0.4
    code = np.array([0] * K + [1] * K, dtype=np.int32)
    y = cfg["f"] * (1.0 + 2e-3 * np.sin(np.arange(ny)))
    return cfg, y, pm, ps, code


def test_oracle_fit_with_log_energies_equals_scipy():
    """The oracle's fit of f(x, T(p)) with the chain-rule gradient is scipy least_squares on a chiv that applies exp to
    the energies explicitly."""
    import warnings
    from scipy.optimize import least_squares
    from oracle.fit import nonlinear_fit as ofit
    cfg, y, pm, ps, code = _explicit_problem()
    K, x = cfg["K"], cfg["x"]
    lo, hi = np.zeros(code.size), np.ones(code.size)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        fo = ofit(lambda x_, p: multiexp(x_, t_dual(code, lo, hi, p)), x, y, cfg["ycov"], prior_mean=pm, prior_cov=ps,
                  tol=(1e-14, 0.0, 0.0), maxit=2000, svdcut=1e-12)
    L = np.linalg.cholesky(np.linalg.inv(cfg["ycov"]))

    def chiv(p):
        q = np.concatenate([p[:K], np.exp(p[K:])])
        return np.concatenate([L.T @ (multiexp(x, q) - y), (p - pm) / ps])
    r = least_squares(chiv, pm, method="trf", x_scale="jac", xtol=1e-15, ftol=1e-15, gtol=1e-15, max_nfev=2000)
    sd = fo.psdev
    assert np.max(np.abs(fo.pmean - r.x) / sd) < 1e-6
    assert abs(fo.chi2 - 2 * r.cost) <= 1e-9 * fo.chi2
    # the oracle's J is the chain-rule Jacobian of the explicit chiv (the two whitenings differ by a rotation of the
    # data rows: compare J^T J)
    J = D.deriv(fo._chiv(D.Dual.variables(r.x)), r.x.size)
    h = 1e-7
    Jfd = np.array([(chiv(r.x + h * e) - chiv(r.x - h * e)) / (2 * h) for e in np.eye(r.x.size)]).T
    A, Afd = J.T @ J, Jfd.T @ Jfd
    s = np.sqrt(np.diag(A))
    assert np.max(np.abs(A - Afd) / (s[:, None] * s[None, :])) < 1e-6


def test_refusals_without_device():
    import lsqfit_b200 as lb
    cfg = configs.correlator(2)
    data = (cfg["x"], cfg["f"], cfg["ycov"])
    prior = (cfg["prior_mean"], cfg["prior_sdev"])
    with pytest.raises(ValueError, match="not built for fit sets"):
        lb.fit_set([data, data], prior=prior, fcn="multiexp", pdist=[None, None, "log", "log"])
    for bad in (["log"], [None, None, "log", "cosh"], [None, None, "log", ("uniform", 1.0, 0.0)]):
        with pytest.raises(ValueError, match="pdist"):
            lb.nonlinear_fit(data=data, prior=prior, fcn="multiexp", pdist=bad)
