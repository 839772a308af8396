"""The svd corrections of a window scan's whitenings, packed for b200lm_window_propagate, without a device: each window's
PDF is built from the oracle's whitening of its own covariance, and the packed blocks must be the oracle's corrected
minus input covariance of that window, block after block in the order of ``window_weights``."""
import numpy as np
import pytest

from lsqfit_b200 import configs
from lsqfit_b200.whiten import PDF, cov_blocks
from lsqfit_b200.windows import window_corrections, window_cov, window_weights
from oracle.whiten import PDF as OPDF
from oracle.whiten import whiten_block_svd


def _pdf(mean, cov, svdcut):
    """lsqfit_b200's PDF with the oracle's block whitening in place of the device's"""
    if cov.ndim == 1:
        return PDF(mean, cov, svdcut=svdcut)
    _, blocks = cov_blocks(cov)
    if not blocks:
        return PDF(mean, cov, svdcut=svdcut)
    W, Cc, nout, nmod, ld = [], [], [], [], []
    for b in blocks:
        n = b.size
        w, logdet, nm, newblk = whiten_block_svd(cov[np.ix_(b, b)], svdcut)
        Wp = np.zeros((n, n))
        Wp[:w.shape[0]] = w
        W.append(Wp.reshape(-1)); Cc.append(np.asarray(newblk, dtype=float).reshape(-1))
        nout.append(w.shape[0]); nmod.append(nm); ld.append(logdet)
    return PDF(mean, cov, svdcut=svdcut, _whitened=(np.concatenate(W), np.concatenate(Cc), np.array(nout),
                                                     np.array(nmod), np.array(ld)))


def _problem(yp, two_blocks):
    cfg = configs.correlator(3, ny=32)
    ny, npar = cfg["ny"], cfg["np"]
    N = ny + npar
    cov = np.zeros((N, N))
    cov[:ny, :ny] = cfg["ycov"]
    cov[ny:, ny:] = np.diag(cfg["prior_sdev"] ** 2)
    s = np.sqrt(np.diag(cov))
    if yp:                                     # data-prior correlation: one block over the rows and a prior entry
        cov[:ny, ny] = cov[ny, :ny] = 0.2 * s[:ny] * s[ny]
    if two_blocks:                             # a second correlated block among the prior entries
        cov[ny + 1, ny + 2] = cov[ny + 2, ny + 1] = 0.3 * s[ny + 1] * s[ny + 2]
    mean = np.concatenate([cfg["f"], cfg["prior_mean"]])
    masks = np.zeros((5, ny), dtype=bool)
    for w, (lo, hi) in enumerate([(0, ny), (0, 8), (4, 20), (10, ny), (2, 30)]):
        masks[w, lo:hi] = True
    return cfg, cov, mean, masks


@pytest.mark.parametrize("svdcut", [0.05, -0.01])
@pytest.mark.parametrize("yp,two_blocks", [(False, False), (True, False), (False, True)])
def test_corrections_match_oracle(svdcut, yp, two_blocks):
    cfg, cov, mean, masks = _problem(yp, two_blocks)
    ny = cfg["ny"]
    pdfs, sels, ref = [], [], []
    for m in masks:
        sel, c = window_cov(cov, ny, m)
        pdfs.append(_pdf(mean[sel], c, svdcut))
        sels.append(sel)
        o = OPDF(mean[sel], c, svdcut=svdcut)
        for idx, _ in o.i_invwgts[1:]:
            ref.append(o.correction_cov[np.ix_(idx, idx)].reshape(-1))
    got = window_corrections(pdfs)
    assert got is not None and got.dtype == np.float64 and got.flags["C_CONTIGUOUS"]
    ref = np.concatenate(ref)
    assert got.shape == ref.shape
    assert np.max(np.abs(got - ref)) <= 1e-12 * np.max(np.abs(cov))
    assert np.abs(got).max() > 0
    # one n_in x n_in block per correlated block, in the order b200lm_set_windows reads the blocks
    d = window_weights(sels, [p.i_invwgts for p in pdfs])
    assert got.size == int(np.sum(d["blk_nin"].astype(np.int64) ** 2))
    assert len(d["blk_nin"]) == (2 if two_blocks else 1) * len(masks)


def test_no_corrections():
    cfg, cov, mean, masks = _problem(False, False)
    ny = cfg["ny"]
    # uncorrelated data: no correlated blocks
    sd = np.sqrt(np.diag(cov))
    assert window_corrections([_pdf(mean[s], c, 1e-12) for s, c in (window_cov(sd, ny, m) for m in masks)]) is None
    # correlated blocks that the cut leaves as they are: every correction exactly zero
    pdfs = [_pdf(mean[s], c, 0.0) for s, c in (window_cov(cov, ny, m) for m in masks)]
    assert all(len(p.i_invwgts) > 1 for p in pdfs)
    assert window_corrections(pdfs) is None
