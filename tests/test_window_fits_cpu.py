"""Fit-window scans without a device: the description builder of lsqfit_b200.windows against the oracle.

Each window is whitened by the oracle's PDF (gvar.PDF restated) on its own covariance, renumbered to the parent's full
y (+) prior vector by the product's builder, and applied to full-length vectors as the window kernel applies it.  The
result must be the oracle's chiv of the window problem itself."""
import numpy as np
import pytest

from lsqfit_b200 import configs
from lsqfit_b200.windows import check_masks, window_cov, window_rows, window_weights
from oracle.chiv import Chiv
from oracle.models import multiexp
from oracle.whiten import PDF


def apply_description(d, w, delta):
    """chiv of window w from a full-length delta = f (+) p - mean, as the device reads the description."""
    nd, nb = d["ndiag"], d["nblk"]
    o = int(nd[:w].sum())
    parts = [d["diag_w"][o:o + nd[w]] * delta[d["diag_idx"][o:o + nd[w]]]]
    kb = int(nb[:w].sum())
    oi = int(d["blk_nin"][:kb].sum())
    ow = int((d["blk_nin"][:kb] * d["blk_nout"][:kb]).sum())
    for k in range(kb, kb + nb[w]):
        nin, nout = d["blk_nin"][k], d["blk_nout"][k]
        W = d["blk_w"][ow:ow + nin * nout].reshape(nout, nin)
        parts.append(W @ delta[d["blk_idx"][oi:oi + nin]])
        oi += nin
        ow += nin * nout
    return np.concatenate(parts)


def _masks(ny, nwin, rng):
    out = [np.ones(ny, dtype=bool), np.arange(ny) < 8, np.arange(ny) >= ny - 8]
    while len(out) < nwin:
        lo = int(rng.integers(0, ny - 8))
        hi = int(rng.integers(lo + 8, ny + 1))
        m = (np.arange(ny) >= lo) & (np.arange(ny) < hi)
        if rng.random() < 0.3:
            m &= rng.random(ny) < 0.7              # holes: windows need not be ranges
            m[lo] = True
        out.append(m)
    return np.array(out)


@pytest.mark.parametrize("svdcut", [1e-8, -0.01])
@pytest.mark.parametrize("yp", [False, True])
def test_window_description_matches_oracle(svdcut, yp):
    cfg = configs.correlator(3, ny=32)
    ny, npar = cfg["ny"], cfg["np"]
    N = ny + npar
    cov = np.zeros((N, N))
    cov[:ny, :ny] = cfg["ycov"]
    cov[ny:, ny:] = np.diag(cfg["prior_sdev"] ** 2)
    if yp:                                     # data-prior correlation (yp_cov): one block over rows and prior
        s = np.sqrt(np.diag(cov))
        cov[:ny, ny] = cov[ny, :ny] = 0.2 * s[:ny] * s[ny]
    rng = np.random.default_rng(7)
    masks = _masks(ny, 20, rng)
    mean = np.concatenate([cfg["f"], cfg["prior_mean"]])
    x = cfg["x"][:, 0]
    sels, pdfs = [], []
    for m in masks:
        sel, c = window_cov(cov, ny, m)
        sels.append(sel)
        pdfs.append(PDF(mean[sel], c, svdcut=svdcut))
    d = window_weights(sels, [p.i_invwgts for p in pdfs])
    nmods = [p.nmod for p in pdfs]
    if svdcut < 0:
        # modes dropped: nchiv is not rows + np, and by how much differs by window
        assert len(set(d["nchiv"] - masks.sum(axis=1) - npar)) > 1 and max(nmods) > 0
    for w, (m, sel, pdf) in enumerate(zip(masks, sels, pdfs)):
        assert d["nchiv"][w] == pdf.nchiv
        chiv = Chiv(pdf, lambda p: multiexp(x[m], p), False)
        for _ in range(3):
            p = cfg["ptrue"] * (1 + 0.05 * rng.standard_normal(npar))
            full = np.concatenate([multiexp(x, p), p]) - mean     # the device reads every window from here
            np.testing.assert_allclose(apply_description(d, w, full), chiv(p), rtol=1e-12, atol=1e-12)
        # the same window whitened again: svdn and logdet are the window's own
        again = PDF(mean[sel], window_cov(cov, ny, m)[1], svdcut=svdcut)
        assert again.nmod == pdf.nmod and again.logdet == pdf.logdet


def test_uncorrelated_window():
    sd = np.linspace(1.0, 2.0, 10)
    m = np.zeros(10, dtype=bool)
    m[[2, 3, 7]] = True
    sel, c = window_cov(np.concatenate([sd, [0.5, 0.5]]), 10, m)
    assert list(sel) == [2, 3, 7, 10, 11] and np.array_equal(c, np.array([sd[2], sd[3], sd[7], 0.5, 0.5]))
    d = window_weights([sel], [[(np.arange(5), 1.0 / c)]])
    assert list(d["diag_idx"]) == [2, 3, 7, 10, 11] and d["nblk"][0] == 0 and d["nchiv"][0] == 5


def test_rows_and_refusals():
    assert list(window_rows(np.array([True, False, True]), 3, 5)) == [0, 2, 3, 4]
    ok = check_masks(np.ones((2, 5), dtype=bool), 5)
    assert ok.shape == (2, 5)
    assert check_masks(np.ones(5, dtype=bool), 5).shape == (1, 5)
    for bad in (np.ones((2, 4), dtype=bool), np.ones((2, 5), dtype=int), np.zeros((0, 5), dtype=bool),
                np.array([[True] * 5, [False] * 5]), np.ones((2, 5, 1), dtype=bool)):
        with pytest.raises(ValueError, match="not built for window scans"):
            check_masks(bad, 5)
