"""Fit-window scans: the problem description of many data windows of one fit (pure numpy, no device).

A window is a boolean mask over the parent fit's ``ny`` data rows.  Window ``w`` is the fit of the rows
``m = masks[w]`` with the parent's prior: its y (+) prior vector is ``sel = rows(m) ++ prior``, and its covariance
is the parent's input covariance restricted to ``sel``.  Whitening that sub-matrix gives window-local
``i_invwgts`` (indices into the window's own y (+) prior vector); ``window_weights`` renumbers them to indices
of the parent's FULL y (+) prior vector and concatenates the windows in the layout of ``b200lm_set_windows``.
The device then reads every window's rows from the same full-length mean vector of a bootstrap copy.
"""
import numpy as np


def check_masks(masks, ny):
    """-> masks as a bool array [nwin, ny]; ValueError for a wrong shape, a non-boolean mask or an empty window."""
    m = np.asarray(masks)
    if m.ndim == 1:
        m = m[None, :]
    if m.ndim != 2 or m.shape[1] != ny or m.shape[0] < 1:
        raise ValueError("window masks must be a bool array [nwin, ny] with ny = %d, got shape %s: "
                         "masks of that shape are not built for window scans" % (ny, np.shape(masks)))
    if m.dtype != np.bool_:
        raise ValueError("window masks must be boolean (got dtype %s): other masks are not built for window scans"
                         % m.dtype)
    empty = np.nonzero(~m.any(axis=1))[0]
    if empty.size:
        raise ValueError("window %d is empty: empty windows are not built for window scans" % int(empty[0]))
    return m


def window_rows(mask, ny, N):
    """sel: the entries of the parent's y (+) prior vector that make up the window's, in the window's order."""
    return np.concatenate([np.nonzero(mask)[0], np.arange(ny, N)]).astype(np.intp)


def window_cov(cov, ny, mask):
    """(sel, covariance of the window's y (+) prior) from the parent's input covariance: a matrix [N, N] or a vector
    of standard deviations [N] (then the window's is the vector of its entries)."""
    cov = np.asarray(cov, dtype=float)
    sel = window_rows(mask, ny, cov.shape[0])
    return sel, (cov[sel] if cov.ndim == 1 else cov[np.ix_(sel, sel)])


def window_weights(sels, invwgts):
    """Concatenated description of nwin windows for ``b200lm_set_windows``.

    sels[w]: the window's entries of the full y (+) prior vector (``window_rows``); invwgts[w]: the window's own
    ``i_invwgts`` (local indices).  Returns a dict of contiguous arrays: ndiag, diag_idx, diag_w [per window, then
    concatenated], nblk, blk_nin, blk_nout, blk_idx, blk_w (row-major W of every block, window after window), and
    nchiv [nwin]."""
    nd, di, dw, nb, nin, nout, bi, bw, nchiv = [], [], [], [], [], [], [], [], []
    for sel, iw in zip(sels, invwgts):
        sel = np.asarray(sel, dtype=np.int64)
        idx0, w0 = iw[0]
        nd.append(len(idx0))
        di.append(sel[np.asarray(idx0, dtype=np.int64)])
        dw.append(np.asarray(w0, dtype=float).reshape(-1))
        nb.append(len(iw) - 1)
        n = len(idx0)
        for idx, W in iw[1:]:
            W = np.asarray(W, dtype=float)
            nin.append(len(idx))
            nout.append(W.shape[0])
            bi.append(sel[np.asarray(idx, dtype=np.int64)])
            bw.append(W.reshape(-1))
            n += W.shape[0]
        nchiv.append(n)
    cat = lambda a, dt: np.ascontiguousarray(np.concatenate(a) if a else np.zeros(0), dtype=dt)
    return dict(ndiag=np.array(nd, dtype=np.int32), diag_idx=cat(di, np.int32), diag_w=cat(dw, np.float64),
                nblk=np.array(nb, dtype=np.int32), blk_nin=np.array(nin, dtype=np.int32),
                blk_nout=np.array(nout, dtype=np.int32), blk_idx=cat(bi, np.int32), blk_w=cat(bw, np.float64),
                nchiv=np.array(nchiv, dtype=np.int64))


def window_corrections(pdfs):
    """Every window's svd correction for ``b200lm_window_propagate``: for each correlated block of each window's
    whitening ``pdfs[w]`` (a ``PDF``), in the block order of ``window_weights``, the block of its corrected covariance
    minus its input covariance, row-major n_in x n_in, concatenated.  None when no window has a correlated block or
    when every correction is exactly zero."""
    parts = [(cb - p.cov_in[np.ix_(b, b)]).reshape(-1) for p in pdfs for b, cb in p._corrected_blocks]
    if not parts:
        return None
    d = np.ascontiguousarray(np.concatenate(parts), dtype=np.float64)
    return d if d.any() else None
