"""User-defined device models without a GPU: lsqfit_b200.cuda_functor generates a plug-in translation unit, nvcc
cross-compiles it for sm_100a, and b200lm_load_functors adds its entries to the registry (loading needs no device).
Covers registration, the cache, nvcc's diagnostics, the refusals of the loader, and that a body-form copy of a
built-in model compiles to the same machine code as the built-in."""
import concurrent.futures
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import lsqfit_b200 as lb
from lsqfit_b200 import _cabi, functors
from lsqfit_b200 import user_functor as uf

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TINY = "return b[0] * x[0];"


def rat43_body():
    """the text of Rat43Body in csrc/functors.cuh"""
    with open(os.path.join(ROOT, "lsqfit_b200", "csrc", "functors.cuh")) as fh:
        m = re.search(r"B200LM_BODY\(Rat43Body\) \{(.*?)\} \};", fh.read())
    return m.group(1).strip()


@pytest.fixture(scope="module")
def plugins():
    """the plug-ins of this module, compiled in parallel: a body-form copy of rat43, and three the loader refuses"""
    jobs = dict(
        rat43=("ut_rat43", rat43_body(), 4, ""),
        version=("ut_badabi", TINY, 1, "abi->version += 1;"),
        builtin=("rat43", TINY, 1, ""),
        np26=("ut_np26", TINY, 1, "kEntries[0].np = 26;"),
    )
    with concurrent.futures.ThreadPoolExecutor(len(jobs)) as ex:
        futs = dict((k, ex.submit(uf.build_plugin, name, src, n, _abi_patch=patch))
                    for k, (name, src, n, patch) in jobs.items())
        return dict((k, f.result()) for k, f in futs.items())


def _load_rc(path):
    fam = C.c_int(-7)
    rc = _cabi.lib.b200lm_load_functors(os.fsencode(path), C.byref(fam))
    return rc, fam.value, _cabi.last_error()


def test_body_plugin_registers(plugins, monkeypatch):
    before = _cabi.functor_table()
    builtin = [r for r in before if r[0] < 1000]
    assert before[:len(builtin)] == builtin and len(builtin) >= 40
    f = lb.cuda_functor("ut_rat43", rat43_body(), 4, host=functors._HOST["rat43"])
    assert isinstance(f, lb.Functor) and f.family >= 1000 and f.nx == 1 and f.path == plugins["rat43"]
    after = _cabi.functor_table()
    assert after[:len(before)] == before                     # built-in rows: same rows, same indices
    assert (f.family, 4, 1, "ut_rat43") in after[len(builtin):]
    assert lb.available() == after
    g = lb.Functor("ut_rat43")                               # the name resolves like a built-in one
    assert (g.name, g.family, g.nx) == ("ut_rat43", f.family, 1)
    x, p = np.linspace(1, 15, 15), np.array([700.0, 5.0, 0.75, 1.3])
    np.testing.assert_array_equal(g(x, p), functors._HOST["rat43"](x, p))
    # the same plug-in again: the same family, no new rows
    assert uf.load_plugin(f.path) == f.family
    assert _cabi.functor_table() == after
    # the same source again: a cache hit, nvcc is not started
    def no_nvcc(cmd):
        raise AssertionError("nvcc started on a cache hit")
    monkeypatch.setattr(uf, "_run_nvcc", no_nvcc)
    h = lb.cuda_functor("ut_rat43", rat43_body(), 4)
    assert h.family == f.family and _cabi.functor_table() == after
    with pytest.raises(ValueError, match="host"):            # no host implementation given this time
        h(x, p)
    # the same name from another source is refused
    monkeypatch.undo()
    with pytest.raises(ValueError, match="different plug-in"):
        lb.cuda_functor("ut_rat43", TINY, 1)


def test_nvcc_diagnostic_names_the_body_line(tmp_path, monkeypatch):
    monkeypatch.setenv("B200LM_FUNCTOR_CACHE", str(tmp_path))
    body = "const double t = x[0];\nreturn b[0] * t +;\n"
    with pytest.raises(ValueError) as e:
        lb.cuda_functor("ut_syntax", body, 2)
    assert re.search(r"ut_syntax\(2\): error", str(e.value)), str(e.value)
    assert not any(n.endswith(".so") for n in os.listdir(str(tmp_path)))


def test_loader_refusals(plugins):
    n0 = _cabi.lib.b200lm_functor_count()
    cases = [(plugins["version"], "version"), (plugins["builtin"], "built-in"), (plugins["np26"], "np must be"),
             (_cabi.LIB_PATH, "b200lm_plugin_entries")]         # a shared object without the entry symbol
    for path, what in cases:
        rc, fam, msg = _load_rc(path)
        assert rc == _cabi.EINVAL and what in msg, (path, rc, msg)
        with pytest.raises(ValueError, match=what):
            uf.load_plugin(path)
    assert _cabi.lib.b200lm_functor_count() == n0
    rc, _, _ = _load_rc(os.path.join(ROOT, "no_such_plugin.so"))
    assert rc == _cabi.EINVAL
    assert _cabi.lib.b200lm_load_functors(None, None) == _cabi.EINVAL
    # the Python interface refuses the same inputs before compiling anything
    for kw in (dict(name="rat43", np=4), dict(name="ut_x", np=26), dict(name="ut_x", np=0), dict(name="ut_x", np=(2, 2)),
               dict(name="ut_x", np=2, nx=9), dict(name="no good", np=2), dict(name="ut_x", np=2, form="python")):
        with pytest.raises(ValueError):
            lb.cuda_functor(source=TINY, **kw)
    assert _cabi.lib.b200lm_functor_count() == n0


def test_generated_source_forms():
    src = uf.generate("m", "return b[0];", (2, 18), 3)
    assert '#line 1 "m"' in src and "ADFunctor<Body, 2, 3>" in src and "ADFunctor<Body, 18, 3>" in src
    assert 'B200LM_ENTRY_TEAM(0, "m", ADFunctor<Body, 2, 3>)' in src      # team and wave kernels up to np 16
    assert 'B200LM_ENTRY(0, "m", ADFunctor<Body, 18, 3>)' in src
    src = uf.generate("m", "template <int NP> using Model = MultiExp<NP / 2>;", (16,), 1, form="functor")
    assert "struct Body" not in src and 'B200LM_ENTRY_TEAM(0, "m", Model<16>)' in src


# ---- the same machine code as the built-in model ----------------------------------------------------------------
KERNELS = {       # demangled kernel name pattern -> label; F is ADFunctor<..., 4, 1>
    r"fit_kernel<(.*), 0>": "fit0", r"fit_kernel<(.*), 1>": "fit1", r"fit_kernel<(.*), 2>": "fit2",
    r"fit_kernel<(.*), 3>": "fit3", r"resjac_kernel<(.*)>": "resjac", r"model_rows_kernel<(.*)>": "model_rows",
    r"normal_diag_kernel<(.*)>": "normal_diag",
}


def _sass(path, functor_pattern):
    """{label: normalised instruction list} of the kernels of the functor whose demangled type matches the pattern"""
    tool = "/usr/local/cuda/bin/"
    listing = subprocess.run([tool + "cuobjdump", "-res-usage", path], capture_output=True, text=True, check=True).stdout
    names = sorted(set(re.findall(r"Function (\S+):", listing)))
    dem = subprocess.run([tool + "cu++filt"], input="\n".join(names), capture_output=True, text=True,
                         check=True).stdout.split("\n")
    want = {}
    for name, d in zip(names, dem):
        d = d.replace("(int)", "")
        for pat, label in KERNELS.items():
            m = re.match(r"void b200lm::" + pat + r"\(", d)
            if m and re.search(functor_pattern, m.group(1)):
                want[name] = label
    out = subprocess.run([tool + "cuobjdump", "-sass", "-fun", ",".join(sorted(want)), path], capture_output=True,
                         text=True, check=True).stdout
    blocks = re.split(r"\n\s*Function : (\S+)\n", out)
    res = {}
    for name, body in zip(blocks[1::2], blocks[2::2]):
        ins = []
        for line in body.split("\n"):
            m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(.*?);", line)
            if m:
                ins.append(re.sub(r"0x[0-9a-f]+|(?<![\w.])-?\d+(\.\d+)?(e[+-]?\d+)?", "#", m.group(1)))
        res[want[name]] = ins
    return res


def test_body_plugin_has_the_builtin_machine_code(plugins):
    mine = _sass(plugins["rat43"], r"ADFunctor<b200lm::user_\w+::Body, 4, 1>")
    ref = _sass(_cabi.LIB_PATH, r"ADFunctor<b200lm::Rat43Body, 4, 1>")
    assert sorted(mine) == sorted(KERNELS.values()) and sorted(ref) == sorted(KERNELS.values())
    for k in sorted(KERNELS.values()):
        assert len(mine[k]) > 100 and mine[k] == ref[k], k


def test_prebuild_command(plugins, tmp_path):
    """python -m lsqfit_b200.user_functor MODULE.py builds (here: finds in the cache) every cuda_functor of the module"""
    import sys
    mod = tmp_path / "models.py"
    mod.write_text("import lsqfit_b200 as lb\nRAT = lb.cuda_functor('ut_rat43', %r, 4)\n"
                   "if __name__ == '__main__':\n    raise SystemExit('not run as __main__')\n" % rat43_body())
    env = dict(os.environ, PYTHONPATH=ROOT)
    r = subprocess.run([sys.executable, "-m", "lsqfit_b200.user_functor", str(mod)], capture_output=True, text=True,
                       env=env, cwd=str(tmp_path))
    assert r.returncode == 0, r.stderr
    assert "ut_rat43: %s" % plugins["rat43"] in r.stdout
