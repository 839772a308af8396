"""Device path for simultaneous (MultiFitter) fits.

``lsqfit.MultiFitter`` hands ``nonlinear_fit`` a Python closure built from its models
(``_multifitfcn(flatmodels)``, reference src/lsqfit/_extras.py:1018-1028, 1816-1829): parameters arrive as a
dictionary, every model returns the values of its own data set.  A closure cannot run on the device, but a list of
models that are all device-backed can be mapped onto ONE composite device functor: here the shared-energy
correlator family (``multiexp_shared2/3``: M data sets, each  sum_k a^(m)_k exp(-E_k t), common energies E).

``SharedExpModel`` implements the reference's model interface (``datatag``, ``ncg``, ``fitfcn``, ``builddata``,
``buildprior``; src/lsqfit/_extras.py:518-640) with numpy, so it also works with the CPU fitters; ``composite``
turns the closure back into (functor, x rows, parameter permutation) for the ``_build_chiv_chivw`` hook.
"""
import collections

import numpy as np

from .functors import Functor


class SharedExpModel(object):
    """One correlator  G(t) = sum_k p[a][k] exp(-p[E][k] t)  of a simultaneous fit; ``a`` and ``E`` are the keys of
    its amplitudes and of the (shared) energies in the parameter dictionary."""

    def __init__(self, datatag, t, a, E, ncg=1, exp=np.exp):
        """``exp``: the exponential used by the CPU evaluation (``gvar.exp`` when a CPU fitter differentiates the
        model with GVars; the device path never calls it)."""
        self.datatag, self.t, self.a, self.E, self.ncg = datatag, np.asarray(t, dtype=float), a, E, ncg
        self.exp = exp

    def fitfcn(self, p):                                     # _extras.py:552-565
        a, E = p[self.a], p[self.E]
        ans = 0.0
        for k in range(len(a)):
            ans = ans + a[k] * self.exp(-E[k] * self.t)
        return ans

    def builddata(self, data):                               # _extras.py:595-606
        return data[self.datatag]

    def buildprior(self, prior, mopt=None):                  # _extras.py:608-640
        return collections.OrderedDict((k, prior[k]) for k in (self.a, self.E))


def _slices(buf):
    """key -> slice of a flat buffer, for a gvar.BufferDict (``.slice(k)``) or anything with ``.slices``."""
    if hasattr(buf, "slices"):
        return collections.OrderedDict((k, buf.slices[k][0] if isinstance(buf.slices[k], tuple) else buf.slices[k])
                                       for k in getattr(buf, "keys_", buf.slices.keys()))
    return collections.OrderedDict((k, buf.slice(k)) for k in buf.keys())


def composite(multifcn, po, yo):
    """(Functor, x rows [ny, 2], pperm) for a ``_multifitfcn`` whose models are all ``SharedExpModel`` with one common
    energy key, or None.  ``po`` / ``yo`` are the parameter / data buffers of the reference's flatfcn
    (src/lsqfit/__init__.py:2037-2042); ``pperm[k]`` is the position in lsqfit's flat parameter buffer of device
    parameter k (device order: amplitudes of data set 0, 1, ..., then the energies)."""
    models = getattr(multifcn, "flatmodels", None)
    if not models or not all(isinstance(m, SharedExpModel) for m in models):
        return None
    M = len(models)
    if M not in (2, 3) or len(set(m.E for m in models)) != 1 or len(set(m.a for m in models)) != M:
        return None
    ps, ys = _slices(po), _slices(yo)
    from .pdist import parse_key

    def key(k):
        """the prior key that holds model key k: k itself or a distribution key f(k) (its code: _lsqfit_hook)"""
        if k in ps:
            return k
        return next((kk for kk in ps if parse_key(kk)[0] is not None and parse_key(kk)[1] == k), k)

    def idx(s):
        return np.arange(s.start, s.stop) if isinstance(s, slice) else np.atleast_1d(np.asarray(s))
    if any(key(k) not in ps for k in [models[0].E] + [m.a for m in models]):
        return None
    E = idx(ps[key(models[0].E)])
    K = E.size
    amps = [idx(ps[key(m.a)]) for m in models]
    if any(a.size != K for a in amps) or sum(a.size for a in amps) + K != sum(idx(s).size for s in ps.values()):
        return None                                          # parameters the models do not use: no device mapping
    by_tag = dict((m.datatag, (i, m)) for i, m in enumerate(models))
    rows = []
    for tag, s in ys.items():
        if tag not in by_tag:
            return None
        i, m = by_tag[tag]
        if idx(s).size != m.t.size:
            return None
        rows.append(np.stack([m.t, np.full(m.t.size, float(i))], axis=1))
    x = np.concatenate(rows, axis=0)
    pperm = np.concatenate(amps + [E]).astype(np.int64)
    return Functor("multiexp_shared%d" % M), x, pperm


# ---------------------------------------------------------------------------------------------------------------
# MultiFitter for device-backed models: simultaneous fits, CHAINED fits with the posterior -> prior hand-off, and the
# batched bootstrap driver (reference src/lsqfit/_extras.py: lsqfit :1164-1212, chained_lsqfit :1214-1411,
# bootstrapped_fit_iter :1540-1586).  Data and priors are plain arrays: data[tag] = (mean, cov or sdev),
# prior = ({key: mean}, {key: sdev}).
# ---------------------------------------------------------------------------------------------------------------
class FunctorModel(object):
    """One data set fitted by a registered device functor: ``fitfcn(p) = Functor(fcn)(x, concat(p[k] for k in keys))``."""

    def __init__(self, datatag, fcn, x, keys):
        self.datatag, self.functor, self.keys = datatag, (fcn if isinstance(fcn, Functor) else Functor(fcn)), tuple(keys)
        self.x = np.asarray(x, dtype=float)

    def fitfcn(self, p):
        return self.functor(self.x, np.concatenate([np.ravel(p[k]) for k in self.keys]))


def _as_functor_model(m):
    if isinstance(m, FunctorModel):
        return m
    if isinstance(m, SharedExpModel):
        return FunctorModel(m.datatag, "multiexp", m.t, (m.a, m.E))
    raise ValueError("MultiFitter: models must be FunctorModel or SharedExpModel instances (device-backed)")


class ChainedFit(object):
    """Result of MultiFitter.chained_lsqfit: ``p`` (dictionary of means), ``pmean`` / ``pcov`` (flat, all keys, with the
    correlations between parameters of different links), ``chi2 dof logGBF Q`` summed over the links (as the reference's
    chained fit reports them), ``fits`` the per-link fit objects."""

    def __init__(self, keys, slices, mu, Sigma, fits):
        from .fit import gammaQ
        self.keys, self.slices, self.pmean, self.pcov, self.fits = keys, slices, mu, Sigma, fits
        self.psdev = np.sqrt(np.diag(Sigma))
        self.p = collections.OrderedDict((k, mu[s]) for k, s in slices.items())
        self.chi2 = float(sum(f.chi2 for f in fits))
        self.dof = int(sum(f.dof for f in fits))
        self.logGBF = float(sum(f.logGBF for f in fits))
        self.Q = float(gammaQ(self.dof / 2.0, self.chi2 / 2.0))
        self.nit = int(sum(f.nit for f in fits))
        self.error = next((f.error for f in fits if f.error is not None), None)


class MultiFitter(object):
    def __init__(self, models, **fitterargs):
        self.models, self.fitterargs = list(models), fitterargs
        self.fit = None

    @staticmethod
    def _flat_prior(prior):
        pm, ps = prior
        keys = list(pm.keys())
        slices, n = collections.OrderedDict(), 0
        for k in keys:
            m = int(np.size(pm[k]))
            slices[k] = slice(n, n + m)
            n += m
        mu = np.concatenate([np.ravel(np.asarray(pm[k], dtype=float)) for k in keys])
        if isinstance(ps, dict):
            Sigma = np.diag(np.concatenate([np.ravel(np.asarray(ps[k], dtype=float)) for k in keys]) ** 2)
        else:
            Sigma = np.array(ps, dtype=float)
            if Sigma.ndim == 1:
                Sigma = np.diag(Sigma ** 2)
        return keys, slices, mu, Sigma

    # ---- simultaneous fit (:1164-1212) -----------------------------------------------------------------------
    def lsqfit(self, data, prior, p0=None, **kargs):
        """One fit of all models together; needs a composite device functor (shared-energy correlators:
        ``SharedExpModel``s with one common energy key)."""
        from .fit import nonlinear_fit
        models = self.models
        if not all(isinstance(m, SharedExpModel) for m in models) or len(set(m.E for m in models)) != 1 \
                or len(models) not in (2, 3):
            raise ValueError("simultaneous device fits exist for 2 or 3 SharedExpModels with a common energy key; "
                             "use chained_lsqfit for other model lists")
        keys, slices, mu, Sigma = self._flat_prior(prior)
        M = len(models)
        order = [m.a for m in models] + [models[0].E]
        perm = np.concatenate([np.arange(slices[k].start, slices[k].stop) for k in order])
        x = np.concatenate([np.stack([m.t, np.full(m.t.size, float(i))], axis=1) for i, m in enumerate(models)], axis=0)
        ymean = np.concatenate([np.ravel(data[m.datatag][0]) for m in models])
        ny = ymean.size
        ycov = np.zeros((ny, ny))
        o = 0
        for m in models:
            c = np.asarray(data[m.datatag][1], dtype=float)
            c = np.diag(c ** 2) if c.ndim == 1 else c
            ycov[o:o + c.shape[0], o:o + c.shape[0]] = c
            o += c.shape[0]
        args = dict(self.fitterargs)
        args.update(kargs)
        pc = Sigma[np.ix_(perm, perm)]
        pc = np.sqrt(np.diag(pc)) if np.count_nonzero(pc - np.diag(np.diag(pc))) == 0 else pc
        fit = nonlinear_fit(data=(x, ymean, ycov), prior=(mu[perm], pc), fcn="multiexp_shared%d" % M,
                            p0=None if p0 is None else np.asarray(p0, dtype=float)[perm], **args)
        inv = np.empty_like(perm)
        inv[perm] = np.arange(perm.size)
        fit.pdict = collections.OrderedDict((k, fit.pmean[inv][s]) for k, s in slices.items())
        fit.pflat_order = inv                       # fit.pmean[inv] is in the prior dictionary's order
        self.fit = fit
        return fit

    def bootstrapped_fits(self, n, seed=None, **kargs):
        """n bootstrap copies of the last simultaneous fit in ONE launch (the reference refits copy by copy, :1540-1586)."""
        if self.fit is None:
            raise ValueError("call lsqfit first")
        return self.fit.bootstrapped_fits(n, seed=seed, **kargs)

    # ---- chained fit (:1214-1411) ----------------------------------------------------------------------------
    def chained_lsqfit(self, data, prior, **kargs):
        """The models are fitted one after the other; the best-fit parameters of each fit -- means, covariance AND their
        correlation with every parameter seen so far -- are the prior of the next one (reference :1365-1411, where gvar's
        correlated GVars carry this).  Here: the marginal prior of link k is a covariance MATRIX (whitened on the device
        like any correlated prior), and after the fit  cov(p_k, p_other) = D_prior . cov_old(p_k, p_other)  with
        D = d p / d (y, prior) from the device propagation kernel (b200lm_propagate; src/lsqfit/__init__.py:897-922)."""
        from .fit import nonlinear_fit
        keys, slices, mu, Sigma = self._flat_prior(prior)
        args = dict(self.fitterargs)
        args.update(kargs)
        fits = []
        for m in map(_as_functor_model, self.models):
            idx = np.concatenate([np.arange(slices[k].start, slices[k].stop) for k in m.keys])
            others = np.setdiff1d(np.arange(mu.size), idx)
            y, yc = data[m.datatag]
            y = np.ravel(np.asarray(y, dtype=float))
            pc = Sigma[np.ix_(idx, idx)]
            pc = np.sqrt(np.diag(pc)) if np.count_nonzero(pc - np.diag(np.diag(pc))) == 0 else pc
            fit = nonlinear_fit(data=(m.x, y, np.asarray(yc, dtype=float)), prior=(mu[idx], pc), fcn=m.functor, **args)
            covp = fit.p[1]
            Dpr = fit.D[:, y.size:]
            cross = Dpr @ Sigma[np.ix_(idx, others)]
            Sigma[np.ix_(idx, others)] = cross
            Sigma[np.ix_(others, idx)] = cross.T
            Sigma[np.ix_(idx, idx)] = covp
            mu[idx] = fit.pmean
            fits.append(fit)
        self.chained = ChainedFit(keys, slices, mu, Sigma, fits)
        return self.chained
