"""Fit sets without a device: the stacked description of lsqfit_b200.windows.set_description against the oracle.

Every problem is whitened by the oracle's PDF (gvar.PDF restated) on its own y (+) prior covariance, renumbered to the
stacked vector (every problem's data rows, then one prior slot per problem) by the product's builder, and applied to
a stacked vector as the window kernel applies it.  The result must be the oracle's chiv of the problem itself."""
import numpy as np
import pytest

from lsqfit_b200 import configs
from lsqfit_b200.functors import Functor
from lsqfit_b200.windows import set_description, window_weights
from oracle.chiv import Chiv
from oracle.models import multiexp
from oracle.whiten import PDF
from test_window_fits_cpu import apply_description

NEXP = 2


def problems(K, seed=5):
    """K problems of a 2-exponential model: ny 24 ... 64, each with its own x grid, data covariance (one dense block,
    two blocks, or a vector of standard deviations) and prior (correlated or a vector of standard deviations)."""
    rng = np.random.default_rng(seed)
    data, priors, full = [], [], []
    for k in range(K):
        ny = int(rng.integers(24, 65))
        cfg = configs.correlator(NEXP, ny=ny, dt=0.08 + 0.01 * k)
        y = cfg["f"] + np.linalg.cholesky(cfg["ycov"]) @ rng.standard_normal(ny)
        kind = k % 3
        if kind == 0:
            ycov = cfg["ycov"]
        elif kind == 1:
            ycov = cfg["ycov"].copy()
            h = ny // 2
            ycov[:h, h:] = ycov[h:, :h] = 0.0
        else:
            ycov = np.sqrt(np.diag(cfg["ycov"]))
        psd = cfg["prior_sdev"] * (1 + 0.1 * k)
        pmean = cfg["prior_mean"] * (1 + 0.05 * k)
        if k % 2:
            pc = 0.3 ** np.abs(np.subtract.outer(np.arange(2 * NEXP), np.arange(2 * NEXP)))
            prior = (pmean, psd[:, None] * psd[None, :] * pc)
        else:
            prior = (pmean, psd)
        data.append((cfg["x"], y, ycov))
        priors.append(prior)
        # the covariance nonlinear_fit whitens, restated: block diagonal over data and prior
        npar = 2 * NEXP
        c = np.zeros((ny + npar, ny + npar))
        c[:ny, :ny] = ycov if ycov.ndim == 2 else np.diag(ycov ** 2)
        c[ny:, ny:] = prior[1] if np.ndim(prior[1]) == 2 else np.diag(prior[1] ** 2)
        full.append(c)
    return data, priors, full


@pytest.mark.parametrize("svdcut", [1e-8, 0.05, -0.01])
def test_set_description_matches_oracle(svdcut):
    K = 10
    data, priors, full = problems(K)
    d = set_description(data, priors, Functor("multiexp"))
    npar = 2 * NEXP
    nys = [len(y) for _, y, _ in data]
    assert d["ny"] == sum(nys) and d["N"] == sum(nys) + K * npar and d["np"] == npar and not d["noprior"]
    assert len(set(nys)) > 3
    pdfs = []
    for k, (x, y, _) in enumerate(data):
        o = int(d["row_off"][k])
        assert o == sum(nys[:k]) and np.array_equal(d["x"][o:o + nys[k], 0], x[:, 0])
        sel = d["sels"][k]
        assert np.array_equal(sel[:nys[k]], np.arange(o, o + nys[k]))
        assert np.array_equal(sel[nys[k]:], d["ny"] + k * npar + np.arange(npar))
        assert np.array_equal(d["mean"][sel], np.concatenate([y, priors[k][0]]))
        c = d["covs"][k]
        assert np.array_equal(c if c.ndim == 2 else np.diag(c ** 2), full[k]), k
        pdfs.append(PDF(d["means"][k], c, svdcut=svdcut))
    # the three data covariance shapes, correlated and diagonal priors: 1x1 rows only, and 1, 2 or 3 blocks
    assert {len(p.i_invwgts) - 1 for p in pdfs} >= {0, 1, 2, 3}
    desc = window_weights(d["sels"], [p.i_invwgts for p in pdfs])
    if svdcut < 0:
        assert max(p.nmod for p in pdfs) > 0 and len(set(desc["nchiv"] - np.array(nys) - npar)) > 1
    rng = np.random.default_rng(11)
    ptrue = configs.correlator(NEXP)["ptrue"]
    nd, nb = desc["ndiag"], desc["nblk"]
    for k, pdf in enumerate(pdfs):
        assert desc["nchiv"][k] == pdf.nchiv
        # the rows mapped back to the problem's own indices are the oracle's whitening of the problem alone
        local = np.full(d["N"], -1)
        local[d["sels"][k]] = np.arange(d["sels"][k].size)
        o = int(nd[:k].sum())
        assert np.array_equal(local[desc["diag_idx"][o:o + nd[k]]], pdf.i_invwgts[0][0])
        assert np.array_equal(desc["diag_w"][o:o + nd[k]], pdf.i_invwgts[0][1])
        kb = int(nb[:k].sum())
        oi = int(desc["blk_nin"][:kb].sum())
        ow = int((desc["blk_nin"][:kb] * desc["blk_nout"][:kb]).sum())
        for j, (idx, W) in enumerate(pdf.i_invwgts[1:]):
            nin, nout = desc["blk_nin"][kb + j], desc["blk_nout"][kb + j]
            assert (nin, nout) == (idx.size, W.shape[0])
            assert np.array_equal(local[desc["blk_idx"][oi:oi + nin]], idx)
            assert np.array_equal(desc["blk_w"][ow:ow + nin * nout], W.reshape(-1))
            oi, ow = oi + nin, ow + nin * nout
    # the stacked chiv at random parameters of every problem is each problem's own chiv
    for _ in range(3):
        ps = [ptrue * (1 + 0.05 * rng.standard_normal(npar)) for _ in range(K)]
        delta = np.concatenate([multiexp(x[:, 0], p) for (x, _, _), p in zip(data, ps)] + ps) - d["mean"]
        for k, pdf in enumerate(pdfs):
            x = data[k][0][:, 0]
            chiv = Chiv(pdf, lambda p: multiexp(x, p), False)
            np.testing.assert_allclose(apply_description(desc, k, delta), chiv(ps[k]), rtol=1e-12, atol=1e-12)


def test_shared_prior_and_no_prior():
    data, priors, _ = problems(4)
    d = set_description(data, priors[0], Functor("multiexp"))
    for k in range(4):
        assert np.array_equal(d["pmeans"][k], priors[0][0]) and np.array_equal(d["pcovs"][k], np.diag(priors[0][1] ** 2))
    # (ymean, yerr) data without x and without a prior: N = ny, sels are the data rows
    d = set_description([(y, e) for _, y, e in data], None, Functor("multiexp"))
    assert d["noprior"] and d["N"] == d["ny"] and d["pmeans"] is None
    assert np.array_equal(np.concatenate(d["sels"]), np.arange(d["ny"]))
    assert not d["x"].any()


def test_refusals_without_device():
    import lsqfit_b200 as lb
    data, priors, _ = problems(3)
    f = Functor("multiexp")
    with pytest.raises(ValueError, match="not built for fit sets"):
        set_description([], None, f)
    with pytest.raises(ValueError, match="not built for fit sets"):
        set_description(data, [priors[0], None, priors[2]], f)
    with pytest.raises(ValueError, match="not built for fit sets"):
        set_description(data, [priors[0], priors[1], (np.ones(6), np.ones(6))], f)
    npar = 2 * NEXP
    for kw in (dict(bounds=(np.full(npar, -10.0), np.full(npar, 10.0))), dict(loss="huber"), dict(policy="gsl"),
               dict(noise=True), dict(yp_cov=np.eye(3))):
        with pytest.raises(ValueError, match="not built for fit sets"):
            lb.fit_set(data, priors, fcn="multiexp", **kw)
    with pytest.raises(ValueError, match="not built for fit sets"):
        lb.fit_set(data, priors, fcn="xerr_logistic")
    with pytest.raises(ValueError, match="not built for fit sets"):
        lb.fit_set([], None, fcn="multiexp", p0=np.ones(npar))
    with pytest.raises(ValueError, match="not built for fit sets"):
        lb.fit_set(data, priors, fcn="multiexp", p0=np.ones(npar + 1))          # p0 of another np
    with pytest.raises(ValueError, match="need p0"):
        lb.fit_set(data, None, fcn="multiexp")
    with pytest.raises(ValueError, match="unknown fitter arguments"):
        lb.fit_set(data, priors, fcn="multiexp", fitter_typo=1)
