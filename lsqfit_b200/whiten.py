"""Device whitening: the B200 replacement for ``gvar.PDF(y (+) prior, svdcut=, eps=)``.

The reference builds ``yp_pdf`` at src/lsqfit/__init__.py:1895,1898 and reads
``.mean .meanflat .nchiv .i_invwgts .logdet .nmod .nblocks .svdcut .eps`` from it
(src/lsqfit/__init__.py:549-561,574,723; src/lsqfit/_utilities.pyx:59-61).  ``PDF``
below offers the same attributes, but the eigen-decomposition / inverse-Cholesky of
every correlated block runs in the CUDA kernel behind ``b200lm_whiten``
(csrc/whiten.cu).  Finding the diagonal blocks of the covariance is integer
graph work on the non-zero pattern and stays on the host.
"""
import ctypes as C

import numpy as np
import torch

from . import _cabi


def cov_blocks(cov):
    """Diagonal blocks (connected components of the non-zero pattern) of ``cov``.

    Returns ``(idx_1x1, [idx_block, ...])`` with sorted index arrays, blocks ordered by
    their first index (cf. gvar.evalcov_blocks as used by gvar.PDF)."""
    cov = np.asarray(cov)
    n = cov.shape[0]
    offdiag = (cov != 0)
    np.fill_diagonal(offdiag, False)
    if not offdiag.any():
        return np.arange(n, dtype=np.intp), []
    # connected components of the non-zero pattern (compiled graph search; a Python DFS over a 7000 x 7000 pattern
    # took seconds); rows without off-diagonal entries are the 1x1 blocks
    from scipy.sparse import csr_matrix
    from scipy.sparse.csgraph import connected_components
    ncomp, comp = connected_components(csr_matrix(offdiag), directed=False)
    single = ~offdiag.any(axis=1)
    label = np.where(single, -1, comp).astype(np.int64)
    nlab = 0
    remap = {}
    for l in label[label >= 0]:
        if l not in remap:
            remap[l] = nlab
            nlab += 1
    label = np.array([remap[l] if l >= 0 else -1 for l in label], dtype=np.int64)
    diag = np.nonzero(label < 0)[0].astype(np.intp)
    blocks = [np.nonzero(label == l)[0].astype(np.intp) for l in range(nlab)]
    blocks.sort(key=lambda b: b[0])
    return diag, blocks


class PDF(object):
    """Whitened Gaussian distribution of y (+) prior (attribute-compatible with gvar.PDF
    as far as lsqfit reads it)."""

    def __init__(self, mean, cov, svdcut=1e-12, eps=None, device=0, noise=False, noise_seed=None, _whitened=None):
        """``_whitened``: the output of ``whiten_blocks`` for this covariance's correlated blocks, computed elsewhere
        (a window scan whitens the blocks of all its windows in one call; each block's result depends on that block
        alone)."""
        mean = np.array(mean, dtype=float).reshape(-1)
        cov = np.asarray(cov, dtype=float)
        if cov.ndim == 1:
            sd = cov
            cov = None
        N = mean.size
        if svdcut is not None:
            eps = None          # reference: eps ignored when svdcut is given (__init__.py:240-245)
        self.svdcut, self.eps = svdcut, eps
        self.mean = mean
        self.meanflat = mean
        self.size = N
        self.device = device
        self.nmod = 0
        self.nblocks = {}
        self.logdet = 0.0
        if cov is None:
            idx0, blocks = np.arange(N, dtype=np.intp), []
            sd0 = np.asarray(sd, dtype=float)
            self._cov_diag_only = sd0 ** 2
            self.sdev_in = sd0
        else:
            assert cov.shape == (N, N)
            idx0, blocks = cov_blocks(cov)
            sd0 = np.sqrt(cov[idx0, idx0])
            self._cov_diag_only = None
            self.sdev_in = None
        self.cov_in = cov
        self.i_invwgts = [(idx0, 1.0 / sd0)]
        if idx0.size:
            self.nblocks[1] = int(idx0.size)
        self.logdet += 2.0 * float(np.sum(np.log(sd0)))
        nchiv = int(idx0.size)
        self._corrected_blocks = []
        if blocks:
            ns = np.array([b.size for b in blocks], dtype=np.int32)
            flat = np.concatenate([cov[np.ix_(b, b)].reshape(-1) for b in blocks])
            W, Cc, nout, nmod, logdet = (whiten_blocks(ns, flat, svdcut, eps, device) if _whitened is None
                                         else _whitened)
            o = 0
            for k, b in enumerate(blocks):
                n = b.size
                Wk = W[o:o + n * n].reshape(n, n)[:nout[k]].copy()
                self.i_invwgts.append((b, Wk))
                self._corrected_blocks.append((b, Cc[o:o + n * n].reshape(n, n).copy()))
                self.nblocks[int(n)] = self.nblocks.get(int(n), 0) + 1
                self.logdet += float(logdet[k])
                self.nmod += int(nmod[k])
                nchiv += int(nout[k])
                o += n * n
        self.nchiv = nchiv
        self.noise = bool(noise)
        self.noise_seed = None
        if self.noise:
            # gvar.PDF(..., noise=True) as called at src/lsqfit/__init__.py:1895,1898: the means receive one random
            # sample of the uncertainty ADDED by the svd cut / eps regulator (covariance: corrected - original)
            from .fit import fresh_seed
            self.noise_seed = fresh_seed() if noise_seed is None else int(noise_seed)
            self.mean += self.svd_noise(1, self.noise_seed)[0]

    def svd_noise(self, n, seed, first=0):
        """[n, N] samples of N(0, corrected covariance - input covariance): the noise ``noise=True`` adds to the means
        (zero for entries the regulator did not touch).  Factor of the correction by Cholesky with a relative shift of
        1e-13 (the correction is positive semi-definite and usually of low rank), normals from the device Philox
        stream of ``seed``, the product by the bootstrap generator's GEMM."""
        from .bootstrap import bootstrap_means
        out = np.zeros((n, self.size))
        for k, (b, cb) in enumerate(self._corrected_blocks):
            d = cb - self.cov_in[np.ix_(b, b)]
            d = 0.5 * (d + d.T)
            scale = float(np.max(np.diag(cb)))
            if not np.any(np.abs(d) > 1e-15 * scale):
                continue
            L = _psd_factor(d, 1e-13 * scale, self.device)
            # one Philox key per block: the blocks' samples are independent
            out[:, b] = bootstrap_means(np.zeros(b.size), L, n, int(seed) + k, first=first, device=self.device).cpu().numpy()
        return out

    @property
    def cov(self):
        """Corrected covariance of y (+) prior (the reference's ``yp_pdf.distribution``)."""
        if getattr(self, "_cov_cache", None) is None:
            if self.cov_in is None:
                c = np.diag(self._cov_diag_only)
            else:
                c = self.cov_in.copy()
                for b, cb in self._corrected_blocks:
                    c[np.ix_(b, b)] = cb
            c.setflags(write=False)                      # shared between accesses: read-only
            self._cov_cache = c
        return self._cov_cache

    def sqrt_cov(self):
        """L [N, M] with L L^T = the corrected covariance, WITHOUT another eigen-decomposition: per block
        C_b W_b^T = D V Lambda^1/2 (W_b = Lambda^-1/2 V^T D^-1 from the device whitening); 1x1 entries: their sdev.
        Used by the bootstrap generator (mean + L z; reference src/lsqfit/__init__.py:1615-1623 via gvar.bootstrap_iter)."""
        idx0, w0 = self.i_invwgts[0]
        M = len(idx0) + sum(W.shape[0] for _, W in self.i_invwgts[1:])
        L = np.zeros((self.size, M))
        L[idx0, np.arange(len(idx0))] = 1.0 / np.asarray(w0, dtype=float)
        o = len(idx0)
        for (b, W), (_, Cb) in zip(self.i_invwgts[1:], self._corrected_blocks):
            L[np.ix_(b, np.arange(o, o + W.shape[0]))] = Cb @ W.T
            o += W.shape[0]
        return L

    def copy_with_mean(self, mean):
        """Simulated fits re-use the whitening and swap only the mean
        (src/lsqfit/__init__.py:545-552)."""
        import copy
        new = copy.copy(self)
        new.mean = np.array(mean, dtype=float).reshape(-1)
        new.meanflat = new.mean
        return new


def _psd_factor(d, shift, device):
    """L with L L^T = d + shift I for a positive semi-definite d: LAPACK on the host for small blocks, the library's own
    blocked Cholesky (b200lm_potrf) above that."""
    n = d.shape[0]
    if n <= 256:
        return np.linalg.cholesky(d + shift * np.eye(n))
    from .dense import _LA
    la = _LA(device)
    A = torch.as_tensor(np.ascontiguousarray(d)).to(la.tdev)
    L = la.empty(n, n)
    linv = la.empty(n, n)
    info = torch.zeros(1, dtype=torch.int32, device=la.tdev)
    if not la.potrf(A, shift, L, linv, info):
        raise ValueError("svd noise: the covariance correction is not positive semi-definite")
    return torch.tril(L)


def whiten_blocks(ns, cov_flat, svdcut, eps, device=0, as_torch=False):
    """Run b200lm_whiten on concatenated row-major blocks.  Returns numpy arrays
    (W_flat, cov_corrected_flat, nout, nmod, logdet); with ``as_torch`` the two matrices stay on
    the device as torch tensors."""
    if not torch.cuda.is_available():
        raise RuntimeError("lsqfit_b200.whiten: no CUDA device (there is no CPU fallback)")
    dev = torch.device("cuda", device)
    nblk = len(ns)
    ns = np.ascontiguousarray(ns, dtype=np.int32)
    d_cov = torch.as_tensor(np.ascontiguousarray(cov_flat, dtype=np.float64)).to(dev)
    d_w = torch.empty_like(d_cov)
    d_cc = torch.empty_like(d_cov)
    d_nout = torch.empty(nblk, dtype=torch.int32, device=dev)
    d_nmod = torch.empty(nblk, dtype=torch.int32, device=dev)
    d_ld = torch.empty(nblk, dtype=torch.float64, device=dev)
    use_eps = 1 if (svdcut is None and eps is not None) else 0
    stream = torch.cuda.current_stream(dev).cuda_stream
    _cabi.check(_cabi.lib.b200lm_whiten(
        device, nblk, ns.ctypes.data, d_cov.data_ptr(),
        float(svdcut) if svdcut is not None else 0.0, float(eps) if eps is not None else 0.0, use_eps,
        d_w.data_ptr(), d_cc.data_ptr(), d_nout.data_ptr(), d_nmod.data_ptr(), d_ld.data_ptr(),
        C.c_void_p(stream)))
    nmod_h = d_nmod.cpu().numpy()
    if use_eps and np.any(nmod_h < 0):
        k = int(np.nonzero(nmod_h < 0)[0][0])
        raise ValueError("eps regulator: block %d (n = %d) is not positive definite after the shift (pivot %d <= 0); "
                         "increase eps or use svdcut" % (k, int(ns[k]), -int(nmod_h[k]) - 1))
    if as_torch:
        return d_w, d_cc, d_nout.cpu().numpy(), d_nmod.cpu().numpy(), d_ld.cpu().numpy()
    return (d_w.cpu().numpy(), d_cc.cpu().numpy(), d_nout.cpu().numpy(), d_nmod.cpu().numpy(),
            d_ld.cpu().numpy())
