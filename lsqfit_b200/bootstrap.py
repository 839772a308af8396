"""Device generator of bootstrap / simulated copies (SURVEY.md section 8(f)-1).

``mean_b = mean + L z_b`` for a batch of copies in one call; the reference produces one copy per
Python iteration with ``gvar.bootstrap_iter`` / ``gvar.raniter`` (src/lsqfit/__init__.py:1532-1535,
1615-1624).  Philox4x32-10 normals and the DMMA GEMM behind ``b200lm_bootstrap_means``.
"""
import ctypes as C

import numpy as np
import torch

from . import _cabi


def normals(count, seed, first=0, device=0, raw=False):
    """Standard normals first .. first+count-1 of the stream keyed by ``seed`` (torch tensor)."""
    if not torch.cuda.is_available():
        raise RuntimeError("lsqfit_b200.bootstrap: no CUDA device (there is no CPU fallback)")
    dev = torch.device("cuda", device)
    z = torch.empty(count, dtype=torch.float64, device=dev)
    npair = ((first + count - 1) >> 1) - (first >> 1) + 1 if count else 0
    w = torch.zeros((npair, 4), dtype=torch.int32, device=dev) if raw else None
    _cabi.check(_cabi.lib.b200lm_normals(device, first, count, C.c_ulonglong(seed & (2 ** 64 - 1)), z.data_ptr(),
                                         w.data_ptr() if raw else None,
                                         C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
    return (z, w) if raw else z


def bootstrap_means(mean, L, n, seed, first=0, device=0, return_z=False):
    """[n, N] tensor of copies first .. first+n-1:  mean + L z  (L: N x M, L L^T = covariance)."""
    if not torch.cuda.is_available():
        raise RuntimeError("lsqfit_b200.bootstrap: no CUDA device (there is no CPU fallback)")
    dev = torch.device("cuda", device)
    N = int(np.shape(L)[0])
    out = torch.empty((n, N), dtype=torch.float64, device=dev)
    z = bootstrap_means_into(out, 0, mean, L, n, seed, first=first, device=device)
    return (out, z) if return_z else out


def bootstrap_means_into(out, col, mean, L, n, seed, first=0, device=0):
    """Copies first .. first+n-1 of mean + L z (L: N x M) into the columns col .. col+N-1 of the [n, *] device tensor
    ``out`` (b200lm_bootstrap_means with out_stride = out.shape[1]).  Returns the normals z [n, M]."""
    if not torch.cuda.is_available():
        raise RuntimeError("lsqfit_b200.bootstrap: no CUDA device (there is no CPU fallback)")
    dev = torch.device("cuda", device)
    tm = (mean if isinstance(mean, torch.Tensor) else torch.as_tensor(np.asarray(mean, dtype=np.float64))).to(dev)
    tm = tm.contiguous()
    tL = (L if isinstance(L, torch.Tensor) else torch.as_tensor(np.ascontiguousarray(L, dtype=np.float64))).to(dev)
    tL = tL.contiguous()
    N, M = tL.shape
    if out.dim() != 2 or out.shape[0] != n or not out.is_contiguous() or col < 0 or col + N > out.shape[1]:
        raise ValueError("out must be a contiguous [n, >= col + N] tensor")
    z = torch.empty((n, M), dtype=torch.float64, device=dev)
    _cabi.check(_cabi.lib.b200lm_bootstrap_means(
        device, n, first, N, M, tm.data_ptr(), tL.data_ptr(), M, C.c_ulonglong(seed & (2 ** 64 - 1)),
        z.data_ptr(), out.data_ptr() + 8 * col, out.shape[1], C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
    return z
