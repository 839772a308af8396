"""Static guard on the team kernels' local memory (no GPU needed): the stack frame and the number of local-memory
instructions (LDL/STL) of fit_team_kernel<MultiExp<K>, 2|4>, K = 5..8, as the built library holds them.

The trial path of these kernels is latency bound and local memory on it goes to L2 under load.  The team context is
kept out of local memory by construction (no run-time index into its buffer pointers, no pointer to it held by the
evaluator, no context passed by reference to an out-of-line function); a change that brings it back shows up here
as a larger frame and more LDL/STL.  The limits are what the kernels compile to today with the flags of
lsqfit_b200/build.py (CUDA 12.9, sm_100a)."""
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "lsqfit_b200", "libb200lm.so")
CUDA_HOME = os.environ.get("CUDA_HOME", "/usr/local/cuda")
CUOBJDUMP = shutil.which("cuobjdump") or os.path.join(CUDA_HOME, "bin", "cuobjdump")

# (K, TW): (stack frame bytes, LDL + STL instructions of the kernel and the functions it calls)
LIMITS = {
    (5, 2): (464, 590), (5, 4): (448, 568),
    (6, 2): (408, 676), (6, 4): (392, 596),
    (7, 2): (408, 676), (7, 4): (400, 648),
    (8, 2): (480, 1038), (8, 4): (384, 617),
}

pytestmark = pytest.mark.skipif(not (os.path.exists(LIB) and os.path.exists(CUOBJDUMP)),
                                reason="needs the built library and cuobjdump")


def _mangled(k, tw):
    return "_ZN6b200lm15fit_team_kernelINS_8MultiExpILi%dEEELi%dEEEvNS_9FitParamsE" % (k, tw)


def _run(*args):
    return subprocess.run([CUOBJDUMP] + list(args) + [LIB], capture_output=True, text=True, check=True).stdout


@pytest.fixture(scope="module")
def stacks():
    out = _run("--dump-resource-usage")
    found = {}
    for name, stack in re.findall(r"Function (\S+):\s*\n\s*REG:\d+ STACK:(\d+)", out):
        found[name] = int(stack)
    return found


@pytest.mark.parametrize("k,tw", sorted(LIMITS))
def test_team_kernel_stack_frame(stacks, k, tw):
    name = _mangled(k, tw)
    assert name in stacks, "fit_team_kernel<MultiExp<%d>, %d> not in the library" % (k, tw)
    assert stacks[name] <= LIMITS[(k, tw)][0], "stack frame %d B > %d B" % (stacks[name], LIMITS[(k, tw)][0])


@pytest.mark.parametrize("k,tw", sorted(LIMITS))
def test_team_kernel_local_memory_instructions(k, tw):
    sass = _run("-sass", "-fun", _mangled(k, tw))
    n = len(re.findall(r"\b(?:LDL|STL)(?:\.\w+)*\s", sass))
    assert "fit_team_kernel" in sass
    assert n <= LIMITS[(k, tw)][1], "%d LDL/STL instructions > %d" % (n, LIMITS[(k, tw)][1])
