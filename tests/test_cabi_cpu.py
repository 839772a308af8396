"""CPU-only checks of the boundary: the shared library loads, exports every symbol that
include/b200lm.h declares, reports its functor registry, and fails loudly (no CPU
fallback) when no CUDA device is present.  No compute calls are made here."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _lib():
    from lsqfit_b200 import _cabi
    return _cabi


def test_library_exports_every_declared_symbol():
    cabi = _lib()
    hdr = open(os.path.join(ROOT, "include", "b200lm.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(b200lm_[a-z_]+)\s*\(", hdr))
    assert len(declared) >= 18
    for name in declared:
        assert hasattr(cabi.lib, name), "missing symbol " + name
    assert declared == set(cabi.SIGNATURES), declared ^ set(cabi.SIGNATURES)
    assert cabi.lib.b200lm_version() == 100


def test_functor_registry_matches_host_mirror():
    cabi = _lib()
    from lsqfit_b200.functors import FAMILY, NX
    table = cabi.functor_table()
    assert len(table) >= 40
    names = set()
    for fam, npar, nx, name in table:
        assert FAMILY[name] == fam
        assert NX.get(name, 1) == nx
        assert cabi.lib.b200lm_functor_family(name.encode()) == fam
        names.add(name)
    assert names == set(FAMILY)
    assert (0, 16, 1, "multiexp") in table and (0, 6, 1, "multiexp") in table
    assert cabi.lib.b200lm_functor_family(b"no_such_model") == cabi.ENOFUNCTOR


def test_no_cpu_fallback():
    """Without a GPU a plan cannot be created: the product path must fail loudly.  Where a GPU is present, the same
    checks run in a child process that sees no device (CUDA_VISIBLE_DEVICES empty)."""
    import torch
    if not torch.cuda.is_available():
        _no_device_checks()
        return
    code = "import sys; sys.path[:0] = [%r, %r]; import test_cabi_cpu; test_cabi_cpu._no_device_checks()" % (
        ROOT, os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]


def _no_device_checks():
    cabi = _lib()
    assert cabi.lib.b200lm_device_count() == 0
    h = cabi.handle_t()
    rc = cabi.lib.b200lm_create(0, 64, 16, 1, 0, 0, C.byref(h))
    assert rc == cabi.ECUDA and not h.value
    assert "no CPU fallback" in cabi.last_error()
    import lsqfit_b200 as lb
    with pytest.raises(RuntimeError):
        lb.Plan("multiexp", 16, 64, np.arange(64.), [(np.arange(80), np.ones(80))])
    with pytest.raises(RuntimeError):
        lb.PDF(np.zeros(2), np.array([[1.0, 0.5], [0.5, 1.0]]))
    # argument errors are reported before any device work
    rc = cabi.lib.b200lm_create(0, 64, 40, 1, 0, 0, C.byref(h))
    assert rc == cabi.ENOFUNCTOR


def test_product_does_not_import_oracle():
    """The oracle is test infrastructure: nothing under lsqfit_b200/ may reference it."""
    pkg = os.path.join(ROOT, "lsqfit_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f
                assert "from oracle" not in src and "import oracle" not in src, f


def test_host_mirror_functors(nist_problems):
    """The numpy face of each registered functor reproduces the reference's own fit functions
    (values recorded from examples/nist.py by tests/golden/make_golden.py)."""
    from lsqfit_b200 import Functor
    for pr in nist_problems:
        f = Functor(pr["form"])
        x = f.xrows(np.array(pr["x"]), len(pr["y"]))
        np.testing.assert_allclose(f(x, np.array(pr["p0"])), pr["f_p0"], rtol=1e-13)
        np.testing.assert_allclose(f(x, np.array(pr["certified"])), pr["f_cert"], rtol=1e-13)


def test_tol_normalisation_and_blocks():
    from lsqfit_b200 import normalize_tol, cov_blocks, STOPPING_CRITERION
    assert normalize_tol(1e-5) == (1e-5, 1e-10, 1e-10)            # _scipy.py:124-132
    assert normalize_tol((1e-5,)) == (1e-5, 1e-10, 1e-10)
    assert normalize_tol((1e-5, 1e-6)) == (1e-5, 1e-6, 1e-10)
    assert normalize_tol((1, 2, 3)) == (1.0, 2.0, 3.0)
    with pytest.raises(ValueError):
        normalize_tol((1, 2, 3, 4))
    assert {k: STOPPING_CRITERION[k] for k in (0, 1, 2, 3, 4, -1)} == {0: 0, 1: 2, 2: 3, 3: 1, 4: 1, -1: 0}     # _scipy.py:178-181
    assert {k: STOPPING_CRITERION[k] for k in (11, 12, 14)} == {11: 1, 12: 2, 14: 4}     # GSL policy: info 1, 2, 27 (_gsl.pyx:689-701)
    cov = np.diag([1., 2., 3., 4., 5.])
    cov[0, 3] = cov[3, 0] = 0.1
    cov[3, 4] = cov[4, 3] = 0.2
    d, b = cov_blocks(cov)
    assert list(d) == [1, 2] and [list(i) for i in b] == [[0, 3, 4]]
    d, b = cov_blocks(np.diag([1., 2.]))
    assert list(d) == [0, 1] and b == []


def test_config_generators():
    from lsqfit_b200 import configs
    c3 = configs.c3(B=16)
    assert c3["x"].shape == (64, 1) and c3["np"] == 16 and c3["ycov"].shape == (64, 64)
    m = configs.bootstrap_means(c3, 16, c3["seed"])
    assert m.shape == (16, 80)
    m2 = configs.bootstrap_means(c3, 16, c3["seed"])
    np.testing.assert_array_equal(m, m2)
    # SURVEY.md section 8(d): F_eval(C3) ~ 1.88e5, F_eval(C4) ~ 6.5e4
    assert abs(configs.eval_flops(64, 16, 8) - 1.88e5) < 2e3
    assert abs(configs.eval_flops(64, 6, 3) - 6.5e4) < 2e3


def test_philox_known_answers():
    """The numpy Philox4x32-10 that the GPU test compares the device generator with reproduces the
    known-answer vectors published with Random123 (Salmon et al., SC'11)."""
    from oracle.philox import philox4x32_10, normals
    def h(a):
        return " ".join("%08x" % x for x in a)
    assert h(philox4x32_10(np.array([0, 0, 0, 0]), (0, 0))) == "6627e8d5 e169c58d bc57ac4c 9b00dbd8"
    assert h(philox4x32_10(np.array([0xffffffff] * 4), (0xffffffff, 0xffffffff))) == "408f276d 41c83b0e a20bc7c6 6d5451fd"
    assert h(philox4x32_10(np.array([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344]),
                           (0xa4093822, 0x299f31d0))) == "d16cfe09 94fdcceb 5001e420 24126ea1"
    z, _ = normals(3, 200001, 12345)
    assert abs(z.mean()) < 0.02 and abs(z.std() - 1) < 0.01
    assert np.array_equal(normals(0, 1000, 5)[0][10:20], normals(10, 10, 5)[0])
