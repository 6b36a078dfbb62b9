"""Register spills of the step kernels' solve phase, read from ptxas (-Xptxas -v) for sm_100a.

The interior-point loop of the throughput kernels runs at 128 registers (T = 20: four blocks of four warps per SM).
Values spilled there are stored and reloaded on every iteration through an L1 that shares its 256 KB with ~200 KB of
shared memory, so a spill is a slowdown the results never show.  This cross-compiles jmpc.cu (no GPU needed) and
checks the spill bytes ptxas reports for every throughput instantiation of step_solve.
"""
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "av-simulation-at-intersections_b200", "csrc", "jmpc.cu")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")

# (T, G) -> largest (spill stores, spill loads) in bytes allowed for step_solve<T, G, false>.  T = 13 / 20 / 25 are
# spill-free; the T = 8 kernel (80 registers, six blocks per SM) and the generic runtime-T kernels (TT = 0) may not
# spill more than they did before the T = 20 loop was made spill-free.
LIMITS = {
    (20, 32): (0, 0),
    (13, 16): (0, 0),
    (25, 32): (0, 0),
    (8, 16): (562, 968),
    (0, 32): (236, 228),
    (0, 16): (290, 268),
}

_PROPS = re.compile(r"Function properties for (\S+)\s*\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, "
                    r"(\d+) bytes spill loads")
_SOLVE = re.compile(r"step_solveILi(\d+)ELi(\d+)ELb([01])E")


@pytest.fixture(scope="module")
def solve_spills(tmp_path_factory):
    if not os.path.exists(NVCC):
        pytest.skip(f"nvcc not found at {NVCC}")
    out = tmp_path_factory.mktemp("ptxas") / "jmpc.cubin"
    cmd = [NVCC, "-cubin", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
           "-Xptxas", "-v", "-o", str(out), SRC]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-4000:]
    spills = {}
    for m in _PROPS.finditer(res.stderr):
        s = _SOLVE.search(m.group(1))
        if s:
            spills[(int(s.group(1)), int(s.group(2)), s.group(3) == "1")] = (int(m.group(3)), int(m.group(4)))
    return spills


def test_t20_solve_phase_is_spill_free(solve_spills):
    assert solve_spills[(20, 32, False)] == (0, 0)


@pytest.mark.parametrize("T,G", sorted(LIMITS))
def test_throughput_solve_spills_within_limit(solve_spills, T, G):
    stores, loads = solve_spills[(T, G, False)]
    max_stores, max_loads = LIMITS[(T, G)]
    assert stores <= max_stores and loads <= max_loads, (T, G, stores, loads)


def test_every_throughput_solve_is_checked(solve_spills):
    assert {(T, G) for (T, G, lat) in solve_spills if not lat} == set(LIMITS)
