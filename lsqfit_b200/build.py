"""Build libb200lm.so in-tree with nvcc for sm_100a.

    python lsqfit_b200/build.py [--force]      (run as a script: importing the package needs the built library)

Every .cu under lsqfit_b200/csrc is compiled to an object file (in parallel) and
linked into lsqfit_b200/libb200lm.so.  nvcc cross-compiles without a GPU, so this
also runs in the CPU-only build container; the resulting .so travels to the GPU
box with the repo snapshot.
"""
import concurrent.futures
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
BUILD = os.path.join(HERE, "_build")
LIB = os.path.join(HERE, "libb200lm.so")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
CFLAGS = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC",
          "-I", INCLUDE] + os.environ.get("B200LM_EXTRA_CFLAGS", "").split()


def _sources():
    return sorted(f for f in os.listdir(CSRC) if f.endswith(".cu"))


def _headers_digest():
    h = hashlib.sha256()
    for d in (CSRC, INCLUDE):
        for f in sorted(os.listdir(d)):
            if f.endswith((".h", ".cuh")):
                with open(os.path.join(d, f), "rb") as fh:
                    h.update(fh.read())
    # the include path in its in-tree form: a tree built in one place and run from another keeps its digest
    h.update(" ".join(ARCH + CFLAGS).replace(INCLUDE, "include").encode())
    return h.hexdigest()


def digest_define(hdig):
    """the -D flag that compiles the headers digest into the library (capi.cu checks plug-ins against it) and into
    every functor plug-in (lsqfit_b200/user_functor.py)"""
    return '-DB200LM_HEADERS_DIGEST="%s"' % hdig


def _compile(src, hdig, force):
    obj = os.path.join(BUILD, src[:-3] + ".o")
    stamp = obj + ".stamp"
    with open(os.path.join(CSRC, src), "rb") as fh:
        dig = hashlib.sha256(fh.read() + hdig.encode()).hexdigest()
    if not force and os.path.exists(obj) and os.path.exists(stamp) and open(stamp).read() == dig:
        return obj, False
    cmd = [NVCC] + ARCH + CFLAGS + [digest_define(hdig), "-c", os.path.join(CSRC, src), "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, r.stdout, r.stderr))
    with open(stamp, "w") as fh:
        fh.write(dig)
    return obj, True


def build(force=False, verbose=True):
    os.makedirs(BUILD, exist_ok=True)
    hdig = _headers_digest()
    srcs = _sources()
    # largest translation units first, one nvcc per core
    srcs.sort(key=lambda f: -os.path.getsize(os.path.join(CSRC, f)) if not f.startswith("inst_") else -10 ** 9)
    with concurrent.futures.ThreadPoolExecutor(max_workers=min(os.cpu_count() or 8, len(srcs))) as ex:
        results = list(ex.map(lambda s: _compile(s, hdig, force), srcs))
    objs = [o for o, _ in results]
    rebuilt = any(ch for _, ch in results)
    if rebuilt or not os.path.exists(LIB):
        cmd = [NVCC] + ARCH + ["-shared", "-o", LIB] + objs
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
    if verbose:
        print("libb200lm.so: %s (%d objects, %s)" % (LIB, len(objs), "rebuilt" if rebuilt else "up to date"))
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv)
