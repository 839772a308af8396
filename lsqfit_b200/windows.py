"""Fit-window scans and fit sets: the problem description of many fits in one plan (pure numpy, no device).

A window is a boolean mask over the parent fit's ``ny`` data rows.  Window ``w`` is the fit of the rows
``m = masks[w]`` with the parent's prior: its y (+) prior vector is ``sel = rows(m) ++ prior``, and its covariance
is the parent's input covariance restricted to ``sel``.  Whitening that sub-matrix gives window-local
``i_invwgts`` (indices into the window's own y (+) prior vector); ``window_weights`` renumbers them to indices
of the parent's FULL y (+) prior vector and concatenates the windows in the layout of ``b200lm_set_windows``.
The device then reads every window's rows from the same full-length mean vector of a bootstrap copy.

A fit set (``set_description``) stacks K unrelated problems of one model the same way: the stacked y (+) prior
vector is every problem's data rows, problem after problem, then one prior slot of np entries per problem
(``b200lm_create_set``).  Problem k is the window ``sel_k = rows_k ++ slot_k`` of that vector.
"""
import numpy as np


def cov2(c, n):
    """A covariance matrix from a covariance matrix, a vector of n standard deviations or one shared one."""
    c = np.asarray(c, dtype=float)
    if c.ndim == 0:
        c = np.full(n, float(c))
    return np.diag(c ** 2) if c.ndim == 1 else c


def yp_cov(yerr, pcov, ny):
    """The covariance of y (+) prior that ``nonlinear_fit`` whitens, from the data's ``yerr`` (covariance matrix, vector
    of standard deviations or one shared one) and the prior covariance ``pcov`` (matrix; None: no prior): the vector of
    standard deviations when both are diagonal, else the block-diagonal matrix."""
    yerr = np.asarray(yerr, dtype=float)
    noprior = pcov is None
    pdiag = noprior or np.count_nonzero(pcov - np.diag(np.diag(pcov))) == 0
    if yerr.ndim <= 1 and pdiag:
        sd = np.full(ny, float(yerr)) if yerr.ndim == 0 else yerr
        return sd if noprior else np.concatenate([sd, np.sqrt(np.diag(pcov))])
    N = ny if noprior else ny + pcov.shape[0]
    c = np.zeros((N, N))
    c[:ny, :ny] = cov2(yerr, ny)
    if not noprior:
        c[ny:, ny:] = pcov
    return c


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


def _is_pair(prior):
    """True for one prior (pmean, pcov | psdev), False for a sequence of them."""
    if not isinstance(prior, tuple) or len(prior) != 2:
        return False
    try:
        return np.ndim(np.asarray(prior[0], dtype=float)) == 1
    except (TypeError, ValueError):
        return False


def set_description(data, prior, fcn):
    """The stacked problem of a fit set (``lsqfit_b200.fit_set``).

    data: a list of K data sets, each in a form ``nonlinear_fit`` accepts, (x, ymean, yerr) or (ymean, yerr); prior: a
    list of K priors (pmean, pcov | psdev), one prior shared by every problem, or None (no prior); fcn: the Functor.
    Returns a dict with ``x`` [ny, nx] (every problem's x rows, stacked as fcn.xrows reads them), ``mean`` [N] (the
    stacked y (+) prior means), ``ny`` (all data rows), ``N``, ``np``, ``noprior``, and per problem: ``nys``,
    ``row_off`` (first data row), ``sels`` (its y (+) prior entries in the stacked vector, in its own order: data rows,
    then its slot ``ny + k np ...``), ``means`` and ``covs`` (its own y (+) prior means and the covariance
    ``nonlinear_fit`` would whiten), ``pmeans`` and ``pcovs`` (None without a prior).  ValueError for an empty list,
    a mix of problems with and without a prior, and priors of different sizes."""
    refuse = lambda what: ValueError("%s not built for fit sets" % what)
    if not isinstance(data, (list, tuple)) or len(data) == 0:
        raise refuse("an empty list of problems is")
    K = len(data)
    if prior is None or _is_pair(prior):
        priors = [prior] * K
    else:
        priors = list(prior)
        if len(priors) != K:
            raise ValueError("%d priors for %d problems: priors of that number are not built for fit sets"
                             % (len(priors), K))
    noprior = priors[0] is None
    if any((p is None) != noprior for p in priors):
        raise refuse("a mix of problems with and without a prior is")
    xs, ys, yerrs = [], [], []
    for k, d in enumerate(data):
        if not isinstance(d, tuple) or len(d) not in (2, 3):
            raise ValueError("problem %d: data tuple wrong length" % k)
        x, ymean, yerr = d if len(d) == 3 else (False,) + tuple(d)
        ymean = np.array(ymean, dtype=float).reshape(-1)
        xs.append(fcn.xrows(x, ymean.size))
        ys.append(ymean)
        yerrs.append(yerr)
    nys = np.array([y.size for y in ys], dtype=np.int64)
    ny = int(nys.sum())
    row_off = np.concatenate([[0], np.cumsum(nys)[:-1]]).astype(np.int64)
    pmeans = pcovs = None
    if noprior:
        npar = -1
    else:
        pmeans = [np.array(p[0], dtype=float).reshape(-1) for p in priors]
        npar = pmeans[0].size
        if any(m.size != npar for m in pmeans):
            raise refuse("priors of different sizes (np %s) are" % sorted(set(m.size for m in pmeans)))
        pcovs = [cov2(p[1], npar) for p in priors]
    N = ny if noprior else ny + K * npar
    sels, means, covs = [], [], []
    for k in range(K):
        rows = np.arange(row_off[k], row_off[k] + nys[k])
        if noprior:
            sels.append(rows.astype(np.intp))
            means.append(ys[k])
        else:
            sels.append(np.concatenate([rows, ny + k * npar + np.arange(npar)]).astype(np.intp))
            means.append(np.concatenate([ys[k], pmeans[k]]))
        covs.append(yp_cov(yerrs[k], None if noprior else pcovs[k], int(nys[k])))
    mean = np.zeros(N)
    for sel, m in zip(sels, means):
        mean[sel] = m
    return dict(x=np.ascontiguousarray(np.concatenate(xs)), mean=mean, ny=ny, N=N, np=npar, noprior=noprior,
                nys=nys, row_off=row_off, sels=sels, means=means, covs=covs, pmeans=pmeans, pcovs=pcovs)
