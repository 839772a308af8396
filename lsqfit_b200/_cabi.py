"""ctypes binding of libb200lm.so (the C ABI declared in include/b200lm.h).

There is no CPU fallback: if the library is missing, importing this module raises.
Build it with ``python lsqfit_b200/build.py`` (or ``__graft_entry__.build()``).
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B200LM_LIB") or os.path.join(HERE, "libb200lm.so")     # (override: A/B experiments)

OK, EINVAL, ENOFUNCTOR, ECUDA, ENOMEM, ESIZE = 0, -1, -2, -3, -4, -5


class B200LMError(RuntimeError):
    def __init__(self, code, msg):
        RuntimeError.__init__(self, "b200lm error %d: %s" % (code, msg))
        self.code = code


if not os.path.exists(LIB_PATH):
    raise ImportError(
        "lsqfit_b200: %s not found -- the CUDA extension must be built "
        "(python lsqfit_b200/build.py); there is no CPU fallback" % LIB_PATH)

lib = C.CDLL(LIB_PATH)

c_double_p = C.POINTER(C.c_double)
c_int_p = C.POINTER(C.c_int)
handle_t = C.c_void_p

# name -> (restype, argtypes); every symbol of include/b200lm.h
SIGNATURES = {
    "b200lm_version": (C.c_int, []),
    "b200lm_last_error": (C.c_char_p, [handle_t]),
    "b200lm_device_count": (C.c_int, []),
    "b200lm_functor_count": (C.c_int, []),
    "b200lm_functor_info": (C.c_int, [C.c_int, c_int_p, c_int_p, c_int_p, C.POINTER(C.c_char_p)]),
    "b200lm_functor_family": (C.c_int, [C.c_char_p]),
    "b200lm_load_functors": (C.c_int, [C.c_char_p, c_int_p]),
    "b200lm_create": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(handle_t)]),
    "b200lm_destroy": (None, [handle_t]),
    "b200lm_set_const": (C.c_int, [handle_t, C.c_void_p, C.c_int]),
    "b200lm_set_weights": (C.c_int, [handle_t, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200lm_nchiv": (C.c_int, [handle_t]),
    "b200lm_fit_batch": (C.c_int, [handle_t, C.c_int, C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong,
                                   C.c_double, C.c_double, C.c_double, C.c_int, C.c_int, C.c_int,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200lm_fit_batch_host": (C.c_int, [handle_t, C.c_int, C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong,
                                        C.c_double, C.c_double, C.c_double, C.c_int, C.c_int, C.c_int,
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200lm_last_stats": (C.c_int, [handle_t, C.POINTER(C.c_ulonglong)]),
    "b200lm_last_stats_ex": (C.c_int, [handle_t, C.POINTER(C.c_ulonglong), C.c_int]),
    "b200lm_last_team": (C.c_int, [handle_t]),
    "b200lm_set_team": (C.c_int, [handle_t, C.c_int]),
    "b200lm_set_order": (C.c_int, [handle_t, C.c_int]),
    "b200lm_last_order": (C.c_int, [handle_t]),
    "b200lm_comm_unique_id": (C.c_int, [C.c_char_p]),
    "b200lm_comm_init": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_char_p, C.POINTER(C.c_void_p)]),
    "b200lm_comm_destroy": (None, [C.c_void_p]),
    "b200lm_comm_rank": (C.c_int, [C.c_void_p]),
    "b200lm_comm_world": (C.c_int, [C.c_void_p]),
    "b200lm_gather": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p]),
    "b200lm_allreduce_sum": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p]),
    "b200lm_model_rows": (C.c_int, [handle_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "b200lm_normal_diag": (C.c_int, [handle_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200lm_set_policy": (C.c_int, [handle_t, C.c_int]),
    "b200lm_set_bounds": (C.c_int, [handle_t, C.c_void_p, C.c_void_p]),
    "b200lm_launch_count": (C.c_longlong, [handle_t]),
    "b200lm_residual_jacobian": (C.c_int, [handle_t, C.c_int, C.c_void_p, C.c_longlong, C.c_void_p,
                                           C.c_longlong, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200lm_whiten": (C.c_int, [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_double, C.c_double, C.c_int,
                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200lm_dgemm": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double,
                               C.c_void_p, C.c_longlong, C.c_int, C.c_void_p, C.c_longlong, C.c_int,
                               C.c_double, C.c_void_p, C.c_longlong, C.c_int, C.c_void_p]),
    "b200lm_multiexp_dense": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_int, C.c_void_p, C.c_void_p]),
    "b200lm_potrf": (C.c_int, [C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_double, C.c_void_p, C.c_int, C.c_void_p,
                               C.c_void_p, C.c_void_p]),
    "b200lm_trsm": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p,
                              C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    "b200lm_normals": (C.c_int, [C.c_int, C.c_longlong, C.c_longlong, C.c_ulonglong, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200lm_bootstrap_means": (C.c_int, [C.c_int, C.c_longlong, C.c_longlong, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                         C.c_int, C.c_ulonglong, C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p]),
    "b200lm_propagate": (C.c_int, [handle_t, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p]),
}

for _name, (_res, _args) in SIGNATURES.items():
    _f = getattr(lib, _name)          # AttributeError here == ABI mismatch: fail loudly
    _f.restype = _res
    _f.argtypes = _args


def last_error(handle=None):
    s = lib.b200lm_last_error(handle)
    return s.decode() if s else ""


def check(rc, handle=None):
    if rc != OK:
        raise B200LMError(rc, last_error(handle))
    return rc


def functor_table():
    """[(family, np, nx, name)] of every compiled device functor."""
    out = []
    fam, npar, nx, name = C.c_int(), C.c_int(), C.c_int(), C.c_char_p()
    for i in range(lib.b200lm_functor_count()):
        check(lib.b200lm_functor_info(i, C.byref(fam), C.byref(npar), C.byref(nx), C.byref(name)))
        out.append((fam.value, npar.value, nx.value, name.value.decode()))
    return out
