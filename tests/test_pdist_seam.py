"""Distribution keys through the lsqfit seam: a dictionary prior with ``log(E)`` / ``sqrt(a)`` / uniform keys, read by the
``register()`` hook into distribution codes, ``Functor.__call__`` on a dictionary of parameters, and
``multifit.composite`` resolving a model key ``k`` to ``f(k)``.

``tests/lsqfit_double.py`` reproduces lsqfit's call protocol with plain dictionaries; here its dictionaries gain
BufferDict's distribution keys (``b['E'] = exp(b['log(E)'])``) through ``BDict`` below, so the double's own callers are
unchanged.  The CPU tests need no device; the others are marked gpu."""
import collections
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import lsqfit_double as L                                         # noqa: E402
from lsqfit_b200 import pdist as P                                # noqa: E402
from oracle import dual as D                                      # noqa: E402
from oracle import models as M                                    # noqa: E402


def _inverse(code, lo, hi):
    """q = T(p) for floats, arrays and the oracle's dual numbers"""
    def f(v):
        if isinstance(v, D.Dual):
            q, dq = P.transform(code, lo, hi, v.v)
            return D.Dual(q, dq[..., None] * v.d)
        return P.transform(code, lo, hi, v)[0]
    return f


class BDict(collections.OrderedDict):
    """The part of gvar.BufferDict the seam reads: values stored under ``f(k)`` are read under ``k`` through f's inverse
    (``log`` -> exp, ``sqrt`` -> square, names made by ``uniform``); iteration lists the stored keys."""
    DIST = {"log": _inverse(P.LOG, 0.0, 1.0), "sqrt": _inverse(P.SQRT, 0.0, 1.0)}

    def __missing__(self, k):
        for kk in list(self.keys()):
            f, base = P.parse_key(kk)
            if base == k and f in BDict.DIST:
                return BDict.DIST[f](dict.__getitem__(self, kk))
        raise KeyError(k)

    @staticmethod
    def uniform(fname, lo, hi):
        BDict.DIST[fname] = _inverse(P.UNIFORM, lo, hi)
        return fname


@pytest.fixture
def bufferdict(monkeypatch):
    """the double's parameter dictionaries with distribution keys"""
    monkeypatch.setattr(L._Flat, "unflatten",
                        lambda self, buf: BDict((k, buf[s]) for k, (s, shp) in self.slices.items()))


# ---- CPU ---------------------------------------------------------------------------------------------------------
def test_functor_reads_model_space_keys():
    import lsqfit_b200 as lb
    t = np.linspace(0.1, 3.0, 7)
    b = BDict([("a", np.array([0.5, 0.3])), ("log(E)", np.log([0.4, 1.1]))])
    ref = M.multiexp(t, np.array([0.5, 0.3, 0.4, 1.1]))
    assert np.allclose(lb.Functor("multiexp")(t, b), ref, rtol=1e-15, atol=0)
    plain = collections.OrderedDict([("a", np.array([0.5, 0.3])), ("E", np.array([0.4, 1.1]))])
    assert np.array_equal(lb.Functor("multiexp")(t, plain), lb.Functor("multiexp")(t, np.array([0.5, 0.3, 0.4, 1.1])))


def test_prior_dist_from_keys():
    from lsqfit_b200._lsqfit_hook import _prior_dist
    BDict.uniform("ufcn", -1.0, 3.0)
    pm = BDict([("sqrt(a)", np.ones(2)), ("ufcn(c)", 0.0), ("log(E)", np.zeros(3)), ("b", np.ones(2))])
    code, lo, hi = _prior_dist((pm, np.ones(8)))
    assert list(code) == [2, 2, 3, 1, 1, 1, 0, 0]
    assert lo[2] == -1.0 and hi[2] == 3.0
    # no distribution key: no codes (the double's existing callers)
    assert _prior_dist((collections.OrderedDict([("a", np.ones(2)), ("E", np.ones(2))]), np.ones(4))) is None
    assert _prior_dist((np.ones(3), np.ones(3))) is None
    # a dictionary that does not resolve k from f(k), or a function the device does not have: refused
    with pytest.raises(ValueError, match="log"):
        _prior_dist((collections.OrderedDict([("log(E)", np.zeros(2))]), np.ones(2)))
    BDict.DIST["tanh"] = np.tanh
    with pytest.raises(ValueError, match="tanh"):
        _prior_dist((BDict([("tanh(x)", np.zeros(2))]), np.ones(2)))


def test_composite_resolves_distribution_keys():
    from lsqfit_b200.multifit import SharedExpModel, composite
    t1, t2 = 0.25 * np.arange(1, 9), 0.25 * np.arange(2, 8)
    models = [SharedExpModel("G1", t1, "a1", "E"), SharedExpModel("G2", t2, "a2", "E")]
    yo = L._Flat(collections.OrderedDict([("G1", np.zeros(t1.size)), ("G2", np.zeros(t2.size))]))
    plain = L._Flat(collections.OrderedDict([("a1", np.ones(2)), ("E", np.ones(2)), ("a2", np.ones(2))]))
    logk = L._Flat(collections.OrderedDict([("a1", np.ones(2)), ("log(E)", np.ones(2)), ("a2", np.ones(2))]))
    f0, x0, p0 = composite(L._multifitfcn(models), plain, yo)
    f1, x1, p1 = composite(L._multifitfcn(models), logk, yo)
    assert f1.name == f0.name and np.array_equal(x1, x0) and np.array_equal(p1, p0)


# ---- GPU ---------------------------------------------------------------------------------------------------------
TIGHT = (1e-15, 0.0, 0.0)


def _install():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (no CPU fallback)")
    import lsqfit_b200 as lb
    lb.register(L)
    return lb


def _problem(K=2, ny=24, seed=3):
    from lsqfit_b200 import configs
    cfg = configs.correlator(K, ny=ny, dt=0.25, rel_err=1e-3)
    rng = np.random.default_rng(seed)
    y = cfg["f"] + np.linalg.cholesky(cfg["ycov"]) @ rng.standard_normal(ny)
    return cfg, y


@pytest.mark.gpu
def test_log_keys_through_the_double(bufferdict):
    """A dictionary prior with log(E) keys fitted with fitter='b200_lm' through the double = the mirror with pdist; the
    double's CPU scipy fitter on the same prior (fcn reading p['E']) agrees."""
    from parity_util import exact_minimum
    lb = _install()
    K = 2
    cfg, y = _problem(K)
    # (dictionary data: the double unflattens the parameters into a dictionary only for a dictionary fit function)
    data = (cfg["x"], collections.OrderedDict([("G", y)]), cfg["ycov"])
    am, lE = np.full(K, 0.5), np.log(cfg["ptrue"][K:])
    psd = np.concatenate([np.full(K, 0.4), np.full(K, 0.3)])
    prior = (BDict([("a", am), ("log(E)", lE)]), psd)
    dev = L.nonlinear_fit(data=data, prior=prior, fcn=lb.Functor("multiexp"), fitter="b200_lm", tol=TIGHT, maxit=2000,
                          polish=100)
    assert dev.error is None
    assert list(dev._chiv.b200.pdist[0]) == [0, 0, 1, 1]
    mir = lb.nonlinear_fit(data=(cfg["x"], y, cfg["ycov"]), prior=(np.concatenate([am, lE]), psd), fcn="multiexp",
                           pdist=[None] * K + ["log"] * K, svdcut=1e-12, tol=TIGHT, maxit=2000, polish=100)
    s = mir.psdev
    assert np.max(np.abs(dev.pmean - mir.pmean) / s) <= 1e-8
    assert abs(dev.chi2 - mir.chi2) <= 1e-9 * mir.chi2
    assert np.max(np.abs(dev.cov - mir.cov) / (s[:, None] * s[None, :])) <= 1e-8

    def fcn(x, p):
        return collections.OrderedDict([("G", M.multiexp(x, D.concatenate([p["a"], p["E"]])))])
    ref = L.nonlinear_fit(data=data, prior=prior, fcn=fcn, fitter="scipy_least_squares", tol=TIGHT, x_scale="jac")
    xe, f, J, cove = exact_minimum(ref)
    se = np.sqrt(np.diag(cove))
    assert np.max(np.abs(dev.pmean - xe) / se) <= 1e-8
    assert abs(dev.chi2 - f @ f) <= 1e-9 * (f @ f)
    assert np.max(np.abs(dev.cov - cove) / (se[:, None] * se[None, :])) <= 1e-8
    # a key whose function the device does not have: the device fitter refuses, the CPU fitter is not concerned
    BDict.DIST["tanh"] = np.tanh
    bad = (BDict([("a", am), ("tanh(E)", np.arctanh(cfg["ptrue"][K:] / 2))]), psd)
    with pytest.raises(ValueError, match="tanh"):
        L.nonlinear_fit(data=data, prior=bad, fcn=lb.Functor("multiexp"), fitter="b200_lm")


@pytest.mark.gpu
def test_multifitter_with_log_energies(bufferdict):
    """MultiFitter of shared-energy models with a log(E) prior key runs on the device (the composite functor with the
    codes carried through pperm) and agrees with the double's CPU MultiFitter."""
    from lsqfit_b200.multifit import SharedExpModel
    _install()
    K = 2
    rng = np.random.default_rng(5)
    t1, t2 = 0.25 * np.arange(1, 17), 0.25 * np.arange(2, 14)
    E = 0.5 * np.arange(1, K + 1)
    a1, a2 = np.full(K, 0.5), np.linspace(0.3, 0.8, K)
    data = collections.OrderedDict()
    for tag, t, a in (("G1", t1, a1), ("G2", t2, a2)):
        f = (a * np.exp(-np.outer(t, E))).sum(axis=1)
        sig = 1e-3 * f
        i = np.arange(f.size)
        cov = sig[:, None] * sig[None, :] * 0.8 ** np.abs(i[:, None] - i[None, :])
        data[tag] = (f + np.linalg.cholesky(cov) @ rng.standard_normal(f.size), cov)
    pm = BDict([("a1", a1.copy()), ("log(E)", np.log(E)), ("a2", a2.copy())])
    ps = collections.OrderedDict([("a1", np.full(K, 0.4)), ("log(E)", np.full(K, 0.3)), ("a2", np.full(K, 0.4))])
    models = [SharedExpModel("G1", t1, "a1", "E", exp=D.exp), SharedExpModel("G2", t2, "a2", "E", exp=D.exp)]
    ref = L.MultiFitter(models, fitter="scipy_least_squares", x_scale="jac", tol=TIGHT).lsqfit(data, (pm, ps))
    dev = L.MultiFitter(models, fitter="b200_lm", polish=100, tol=TIGHT).lsqfit(data, (pm, ps))
    assert dev.error is None
    spec = dev._chiv.b200
    assert spec.functor.name == "multiexp_shared2" and list(spec.pdist[0]) == [0, 0, 1, 1, 0, 0]
    assert list(spec.device_pdist[0]) == [0, 0, 0, 0, 1, 1]
    s = ref.psdev
    np.testing.assert_allclose(dev.pmean, ref.pmean, rtol=0, atol=2e-6 * np.max(s))
    np.testing.assert_allclose(dev.chi2, ref.chi2, rtol=1e-9)
    assert np.max(np.abs(dev.cov - ref.cov) / (s[:, None] * s[None, :])) < 1e-6
