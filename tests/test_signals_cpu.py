"""Fixed-time traffic signals (BatchedEpisodes(signals=...), jmpc_signals), CPU side: hand-built cases of the signal
pass oracle, the host argument checks of SignalPlan, Trips.group and poisson_trips(groups=), struct jmpc_signal_plan
against its ctypes mirror, and the spill report of the new kernel from ptxas for sm_100a."""
import ctypes
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from oracle import signals as S

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "av-simulation-at-intersections_b200", "csrc", "jmpc.cu")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")


def _snap(**kw):
    """One vehicle, group 0 green in iterations 0 .. 4 of a 10-iteration cycle, stop line e = 20, margin 2 (L = 18),
    course index 5, dl 0.5, stop_decel 3: the stopping test's right-hand side is 2 * 3 * 12 * 0.5 = 36 exactly."""
    s = dict(iteration=7, cycle=10, green_start=[0], green_len=[5], margin=2, stop_decel=3.0, k=1, offset=None,
             owner=None, group=[0], zone=[[20, 30]], course_id=[0], course_n=[100], agent_idx=[5],
             state=[[0.0, 0.0, 4.0, 0.0]], dl=[0.5], done=[0], checked=True, course_len=[100], latch=[[-1, 0]],
             hold_steps=[0], go=[0])
    s.update(kw)
    return s


def _run(**kw):
    course_len, latch, hold, go = S.signal_pass(_snap(**kw))
    return course_len.tolist(), latch.tolist(), hold.tolist(), go.tolist()


def test_green_clears_the_latch_and_leaves_the_course():
    assert _run(iteration=3, course_len=[77], latch=[[0, 1]]) == ([77], [[-1, 0]], [0], [0])
    assert _run(iteration=13, course_len=[77], latch=[[0, 0]]) == ([77], [[-1, 0]], [0], [0])


def test_red_holds_a_vehicle_that_can_stop():
    assert _run() == ([18], [[0, 1]], [1], [0])


def test_stopping_test_at_equality_and_one_ulp_past_it():
    assert _run(state=[[0.0, 0.0, 6.0, 0.0]]) == ([18], [[0, 1]], [1], [0])           # 6 * 6 = 36 <= 36: hold
    v = float(np.nextafter(6.0, 7.0))
    assert v * v > 36.0
    assert _run(state=[[0.0, 0.0, v, 0.0]]) == ([100], [[0, 0]], [0], [1])            # cannot stop: a GO pass


def test_a_vehicle_past_the_line_goes_without_a_go_pass():
    for a in (18, 25):
        assert _run(agent_idx=[a]) == ([100], [[0, 0]], [0], [0])
    stopped = [[0.0, 0.0, 0.0, 0.0]]                            # L - 1 - a = 0: only a stopped vehicle holds
    assert _run(agent_idx=[17], state=stopped) == ([18], [[0, 1]], [1], [0])
    assert _run(agent_idx=[17], state=[[0.0, 0.0, 1e-9, 0.0]]) == ([100], [[0, 0]], [0], [1])


def test_unsignalised_group_or_course():
    assert _run(group=[-1], latch=[[0, 1]], course_len=[50]) == ([50], [[-1, 0]], [0], [0])
    assert _run(zone=[[-1, -1]], latch=[[0, 1]], course_len=[50]) == ([50], [[-1, 0]], [0], [0])


def test_a_held_vehicle_creeping_past_the_line_stays_held():
    assert _run(agent_idx=[19], latch=[[0, 1]], hold_steps=[4]) == ([20], [[0, 1]], [5], [0])
    # and a GO decision stays GO, even where a fresh test would hold
    assert _run(latch=[[0, 0]]) == ([100], [[0, 0]], [0], [0])
    # the hold never lengthens a shorter collision cut
    assert _run(course_len=[12]) == ([12], [[0, 1]], [1], [0])


def test_always_red_holds_for_good():
    kw = dict(green_len=[0], state=[[0.0, 0.0, 0.0, 0.0]])
    latch, hold = [[-1, 0]], [0]
    for i in range(0, 40, 3):
        cl, latch, hold, go = _run(iteration=i, latch=latch, hold_steps=hold, agent_idx=[5 + i], **kw)
        assert cl == [max(5 + i + 1, 18)] and latch == [[0, 1]] and go == [0]
    assert hold == [14]


def test_an_owner_change_resets_the_latch():
    kw = dict(owner=[3], group=[-1, -1, -1, 0], zone=[[-1, -1]] * 3 + [[20, 30]], hold_steps=[0] * 4, go=[0] * 4)
    fast = [[0.0, 0.0, 9.0, 0.0]]
    assert _run(latch=[[2, 1]], state=fast, **kw) == ([100], [[3, 0]], [0] * 4, [0, 0, 0, 1])   # decided afresh
    assert _run(latch=[[3, 1]], state=fast, **kw) == ([18], [[3, 1]], [0, 0, 0, 1], [0] * 4)    # trip 3's own hold


def test_green_uses_the_non_negative_modulus_with_offsets_and_wraps_the_cycle():
    # window (8, 4) of a 10-iteration cycle: green at phases 8, 9, 0, 1
    got = [bool(S.green(i, 0, 0, 10, [8], [4])) for i in range(14)]
    assert got == [True, True] + [False] * 6 + [True] * 4 + [False] * 2
    for i in range(-25, 25):
        for off in (-17, -10, -3, 0, 4, 13):
            assert bool(S.green(i, 0, off, 10, [8], [4])) == (((i + off - 8) % 10) < 4), (i, off)
    # per-scene offsets in the pass: k = 2, scene 0 offset -7, scene 1 offset 13, iteration 2
    # scene 0: (2 - 7 - 8) mod 10 = 7 -> red; scene 1: (2 + 13 - 8) mod 10 = 7 -> red; iteration 5: 0 / 0 -> green
    kw = dict(green_start=[8], green_len=[4], k=2, offset=[-7, 13], group=[0] * 4, zone=[[20, 30]] * 4,
              course_id=[0] * 4, agent_idx=[5] * 4, state=[[0.0, 0.0, 1.0, 0.0]] * 4, dl=[0.5] * 4, done=[0] * 4,
              course_len=[100] * 4, latch=[[-1, 0]] * 4, hold_steps=[0] * 4, go=[0] * 4)
    assert _run(iteration=2, **kw)[0] == [18] * 4
    assert _run(iteration=5, **kw)[0] == [100] * 4
    # scene 0 offset -8: (5 - 8 - 8) mod 10 = 9 -> red
    assert _run(iteration=5, **{**kw, "offset": [-8, 13]})[0] == [18, 18, 100, 100]


def test_without_a_collision_check_the_full_length_comes_back():
    # a previous hold left course_len at 18; no check ran: green restores the course, red re-cuts it
    assert _run(checked=False, iteration=2, course_len=[18], latch=[[0, 1]]) == ([100], [[-1, 0]], [0], [0])
    assert _run(checked=False, course_len=[18], latch=[[0, 1]], agent_idx=[30]) == ([31], [[0, 1]], [1], [0])
    assert _run(checked=False, group=[-1], course_len=[18]) == ([100], [[-1, 0]], [0], [0])
    # finished episodes are left alone
    assert _run(checked=False, done=[1], course_len=[18], latch=[[0, 1]]) == ([18], [[0, 1]], [0], [0])


# ---- host argument checks ------------------------------------------------------------------------------------------

def test_signal_plan_argument_checks():
    from junction_mpc.episodes import SignalPlan, signal_setup
    p = SignalPlan(300, [(0, 130), (150, 130)], (0.0, 0.0, 10.0))
    assert p.n_groups == 2 and p.margin is None and p.stop_decel == 3.0 and p.offset is None
    st = p.struct(9)
    assert (st.cycle, st.n_groups, st.margin, st.stop_decel) == (300, 2, 9, 3.0)
    assert list(st.green_start)[:2] == [0, 150] and list(st.green_len)[:2] == [130, 130]
    assert SignalPlan(5, [(0, 5)], (0, 0, 1), margin=3).struct(9).margin == 3
    J = (0.0, 0.0, 10.0)

    def bad(match, *a, **kw):
        with pytest.raises(ValueError, match=match):
            SignalPlan(*a, **kw)
    for c in (0, -1, 2.5, True, 2 ** 31):
        bad("cycle must be an integer >= 1", c, [(0, 1)], J)
    bad("1 to 8", 10, [], J)
    bad("1 to 8", 10, [(0, 1)] * 9, J)
    bad("1 to 8", 10, [(0, 1, 2)], J)
    bad("integers", 10, [(0.5, 1)], J)
    bad(r"start must be in \[0, 10\)", 10, [(10, 1)], J)
    bad(r"start must be in \[0, 10\)", 10, [(-1, 1)], J)
    bad(r"length must be in \[0, 10\]", 10, [(0, 11)], J)
    bad(r"length must be in \[0, 10\]", 10, [(0, -1)], J)
    bad("junction", 10, [(0, 1)], (0, 0, 0))
    bad("junction", 10, [(0, 1)], (0, 0))
    bad("junction", 10, [(0, 1)], (np.nan, 0, 1))
    bad("margin", 10, [(0, 1)], J, margin=-1)
    bad("margin", 10, [(0, 1)], J, margin=1.5)
    for d in (0.0, -1.0, np.inf, np.nan):
        bad("stop_decel", 10, [(0, 1)], J, stop_decel=d)
    bad("offset must be a 1-D integer", 10, [(0, 1)], J, offset=[0.5])
    bad("offset must be a 1-D integer", 10, [(0, 1)], J, offset=3)
    bad("offset must be within", 10, [(0, 1)], J, offset=[2 ** 31 - 1])
    # the per-episode groups and the offsets' shape
    assert signal_setup(None, None, 8, 4) is None
    g, off = signal_setup(p, [0, 1, -1, 0, 1, 1, 0, -1], 8, 4)
    assert g.dtype == np.int32 and off is None
    po = SignalPlan(300, [(0, 130)], J, offset=[3, -4])
    assert signal_setup(po, [0] * 8, 8, 4)[1].tolist() == [3, -4]

    def bad_setup(match, *a):
        with pytest.raises(ValueError, match=match):
            signal_setup(*a)
    bad_setup("signal_group is an argument of signals", None, [0] * 8, 8, 4)
    bad_setup("must be a SignalPlan", (300, [(0, 1)]), [0] * 8, 8, 4)
    bad_setup("need signal_group", p, None, 8, 4)
    bad_setup(r"signal_group must be \[8\]", p, [0] * 7, 8, 4)
    bad_setup(r"in \[-1, 2\)", p, [0] * 7 + [2], 8, 4)
    bad_setup(r"in \[-1, 2\)", p, [0] * 7 + [-2], 8, 4)
    bad_setup("1-D integer", p, [0.0] * 8, 8, 4)
    bad_setup(r"offset must be \[4\]", po, [0] * 8, 8, 2)


def test_trip_groups_and_poisson_groups():
    from junction_mpc.config import NPARAM
    from junction_mpc.episodes import SignalPlan, Trips, poisson_trips, trips_setup
    st = np.zeros((3, 4))
    tr = Trips([0, 0, 1], [0, 2, 1], [0, 1, 2], st, group=[0, -1, 1])
    assert tr.group.tolist() == [0, -1, 1]
    with pytest.raises(ValueError, match="group must be >= -1"):
        Trips([0], [0], [0], st[:1], group=[-2])
    with pytest.raises(ValueError, match=r"group must be \[1\]"):
        Trips([0], [0], [0], st[:1], group=[0, 0])
    with pytest.raises(ValueError, match="integer array"):
        Trips([0], [0], [0], st[:1], group=[0.5])
    p = SignalPlan(300, [(0, 130), (150, 130)], (0.0, 0.0, 10.0))
    ok = dict(n_scenes=2, k=2, n_courses=3, planned=False, n_extra=0, right_of_way=None, share_plans=False,
              params_default=np.zeros(NPARAM))
    trips_setup(tr, **ok, signals=p)
    with pytest.raises(ValueError, match="group is an argument of signals"):
        trips_setup(tr, **ok)
    with pytest.raises(ValueError, match="signals need Trips.group"):
        trips_setup(Trips([0], [0], [0], st[:1]), **ok, signals=p)
    with pytest.raises(ValueError, match=r"Trips.group must be in \[-1, 1\)"):
        trips_setup(tr, **ok, signals=SignalPlan(10, [(0, 5)], (0.0, 0.0, 10.0)))
    # the pass reads offset[scene] on the device: one offset per scene, and a plan object
    trips_setup(tr, **ok, signals=SignalPlan(300, [(0, 130), (150, 130)], (0.0, 0.0, 10.0), offset=[5, -3]))
    for off in ([0], [0, 1, 2]):
        with pytest.raises(ValueError, match=r"offset must be \[2\] \(one per scene\)"):
            trips_setup(tr, **ok, signals=SignalPlan(300, [(0, 130), (150, 130)], (0.0, 0.0, 10.0), offset=off))
    with pytest.raises(ValueError, match="signals must be a SignalPlan"):
        trips_setup(tr, **ok, signals=(300, [(0, 130)]))
    # poisson_trips: the approach's group, and the same draws as without groups
    routes = [[(3 * g + r, (10.0 * g, 0.0, 0.5 * r)) for r in range(3)] for g in range(4)]
    a = poisson_trips(50, routes, 300.0, 0.2, 600, 4.0, seed=3, groups=[0, 1, 0, -1])
    b = poisson_trips(50, routes, 300.0, 0.2, 600, 4.0, seed=3)
    for n in ("scene", "arrival", "course_id", "state"):
        assert np.array_equal(getattr(a, n), getattr(b, n)), n
    assert b.group is None
    assert np.array_equal(a.group, np.array([0, 1, 0, -1])[a.course_id // 3])
    for groups in ([0, 1, 0], [0, 1, 0, -2], [0.0, 1.0, 0.0, 1.0]):
        with pytest.raises(ValueError, match="groups must be 4 integers"):
            poisson_trips(2, routes, 300.0, 0.2, 60, groups=groups)


# ---- struct layout and the kernel's resources ----------------------------------------------------------------------

def test_signal_plan_struct_matches_the_header(tmp_path):
    from junction_mpc import _cabi
    with open(os.path.join(ROOT, "include", "jmpc.h")) as f:
        header = f.read()
    body = re.search(r"typedef struct jmpc_signal_plan \{(.*?)\} jmpc_signal_plan;", header, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = [re.sub(r"\[.*?\]", "", d.split()[-1]) for d in body.split(";") if d.strip()]
    assert names == [f[0] for f in _cabi.SignalPlan._fields_]
    assert int(re.search(r"#define JMPC_SIGNAL_MAX_GROUPS (\d+)", header).group(1)) == _cabi.SIGNAL_MAX_GROUPS
    cc = shutil.which("cc") or shutil.which("gcc")
    if cc is None:
        pytest.skip("no C compiler for the offset check")
    fields = ", ".join(f'(int)offsetof(jmpc_signal_plan, {n})' for n in names)
    src = tmp_path / "layout.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "jmpc.h"\n'
                   f"int main(void) {{ int o[] = {{{fields}}}; for (size_t i = 0; i < sizeof o / sizeof *o; ++i) "
                   'printf("%d ", o[i]); printf("%d\\n", (int)sizeof(jmpc_signal_plan)); return 0; }\n')
    exe = tmp_path / "layout"
    subprocess.run([cc, "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    want = [getattr(_cabi.SignalPlan, n).offset for n in names] + [ctypes.sizeof(_cabi.SignalPlan)]
    assert got == want


_PROPS = re.compile(r"Function properties for (\S+)\s*\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, "
                    r"(\d+) bytes spill loads")


def test_signal_kernel_is_spill_free(tmp_path):
    if not os.path.exists(NVCC):
        pytest.skip(f"nvcc not found at {NVCC}")
    out = tmp_path / "jmpc.cubin"
    cmd = [NVCC, "-cubin", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
           "-Xptxas", "-v", "-o", str(out), SRC]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-4000:]
    hits = [m.groups()[1:] for m in _PROPS.finditer(res.stderr) if re.fullmatch(r"_ZN4jmpc13signal_kernel.*",
                                                                                   m.group(1))]
    assert hits == [("0", "0", "0")], hits
