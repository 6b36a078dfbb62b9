"""Trips through scene slots (BatchedEpisodes.from_trips), CPU side: hand-built cases of the trips pass oracle, the host
argument checks, the Poisson demand generator, the trip-table helpers, struct jmpc_trips against its ctypes mirror, and
the register / spill report of the new kernels and the pinned ones from ptxas for sm_100a."""
import os
import re
import subprocess

import numpy as np
import pytest

from oracle import scene_trips as ST
from oracle.collision_oracle import CarGeometry

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "av-simulation-at-intersections_b200", "csrc", "jmpc.cu")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
GEO = CarGeometry()
W = ST.WAITING


def _pose(x, y, yaw=0.0, v=0.0):
    return [x, y, v, yaw]


def _pass(done, state, slot_trip, phase, arrival, usable, start, k, iteration=0, **kw):
    return ST.trips_pass(done, state, slot_trip, phase, [0, len(arrival)], arrival, usable, start, k, iteration, **kw)


def test_no_empty_slot_counts_slot_waits():
    r = _pass([0, 0], [_pose(0, 0), _pose(0, 50)], [0, 1], [1, 1, 0, 0], [0, 0, 0, 5], [1] * 4,
              [_pose(0, 0), _pose(0, 50), _pose(100, 0), _pose(200, 0)], k=2, iteration=3)
    assert r["admitted"] == [] and r["slot_waits"] == [2] and r["blocked_waits"] == []      # trip 3 is not due yet


def test_blocked_by_a_present_vehicle_at_the_gap():
    gap = 2.0
    at = gap + 2 * GEO.radius                    # side by side, same yaw: the closest circles are this far apart
    for d, admitted in ((at - 1e-9, False), (at + 1e-9, True)):
        assert (ST.start_clearance(_pose(0, 0), _pose(0, d), GEO) >= gap) == admitted
        r = _pass([0, W], [_pose(0, d), _pose(0, 0)], [0, -1], [1, 0], [0, 0], [1, 1], [_pose(0, d), _pose(0, 0)],
                  k=2, entry_gap=gap)
        assert (r["admitted"] == [(1, 1)]) == admitted and (r["blocked_waits"] == [1]) != admitted


def test_first_in_first_out_behind_an_earlier_pending_trip():
    # trips 0 and 1 start at the same pose; the slot holds a vehicle right there, so trip 0 is blocked and trip 1 waits
    # behind trip 0 even after the vehicle has moved on; trip 2 on another approach goes past both
    start = [_pose(0, 0), _pose(0, 0), _pose(50, 0)]
    r = _pass([0, W, W], [_pose(0, 1), _pose(0, 0), _pose(0, 0)], [9, -1, -1], [0, 0, 0], [0, 0, 0], [1] * 3, start, k=3)
    assert r["blocked_waits"] == [0, 1] and r["admitted"] == [(2, 1)]
    r = _pass([0, W, W], [_pose(0, 40), _pose(0, 0), _pose(0, 0)], [9, -1, -1], [0, 0, 0], [0, 0, 0], [1] * 3, start,
              k=3)
    assert r["admitted"] == [(0, 1), (2, 2)] and r["blocked_waits"] == [1]    # trip 1 is blocked by trip 0 just loaded


def test_unusable_course_is_closed_without_a_slot():
    r = _pass([W, W], np.zeros((2, 4)), [-1, -1], [0, 0, 0], [0, 0, 1], [0, 1, 1],
              [_pose(0, 0), _pose(0, 0), _pose(30, 0)], k=2)
    assert r["no_course"] == [0] and r["admitted"] == [(1, 0), (2, 1)]      # trip 0 blocks nothing


def test_lowest_empty_slot_is_taken():
    r = _pass([0, W, 2, W], [_pose(0, 100), _pose(0, 0), _pose(0, 200), _pose(0, 0)], [0, -1, 1, -1], [1, 1, 0],
              [0, 0, 4], [1] * 3, [_pose(0, 100), _pose(0, 200), _pose(0, 300)], k=4, iteration=3)
    assert r["admitted"] == [(2, 1)] and r["done"].tolist() == [0, 0, 2, W]


def test_close_and_readmit_into_the_same_slot_in_one_pass():
    r = _pass([ST.GOAL, 0], [_pose(0, 0), _pose(0, 60)], [0, 1], [1, 1, 0], [0, 0, 7], [1] * 3,
              [_pose(-30, 0), _pose(0, 60), _pose(-30, 0)], k=2, iteration=6)
    assert r["closed"] == [(0, 0)] and r["admitted"] == [(2, 0)] and r["entry"] == 7
    assert r["phase"].tolist() == [2, 1, 1] and r["slot_trip"].tolist() == [2, 1]


def test_a_trip_admitted_earlier_in_the_pass_blocks_a_later_one():
    # trips 0 and 1 at poses 3 m apart (clearance 3 - 2r < 2): trip 0 is admitted, trip 1 is blocked by it
    r = _pass([W, W, W], np.zeros((3, 4)), [-1, -1, -1], [0, 0], [0, 0], [1, 1], [_pose(0, 0), _pose(0, 3)], k=3,
              initial=True)
    assert r["admitted"] == [(0, 0)] and r["blocked_waits"] == [1] and r["entry"] == 0


def test_presence_from_the_trip_table():
    # slot 0: trip 0 in evaluations 0 .. 3 (goal at the top of iteration 3), trip 2 from evaluation 4; slot 1: trip 1
    p = ST.presence([0, 1, 0, -1], [0, 2, 4, -1], [3, 6, 6, -1], B=2, n=7)
    assert p[:, 0].all() and p[:, 1].tolist() == [0, 0, 1, 1, 1, 1, 1]
    c = ST.presence([0, 1, 0, -1], [0, 2, 4, -1], [3, 6, 6, -1], B=2, n=7, collision=True)
    assert c[:, 0].tolist() == [1, 1, 1, 0, 1, 1, 0]


def test_trip_holding_resolves_mate_slots():
    from junction_mpc.episodes import trip_holding
    # k = 3, scene 0: slot 0 holds trip 0 (evaluations 0 .. 5) then trip 3 (7 .. 9); slot 1 holds trip 1; slot 2 trip 2
    slot, entry, exit = [0, 1, 2, 0, -1], [0, 0, 1, 7, -1], [5, 9, 9, 9, -1]
    # trip 1 (slot 1): mate slot 0 is episode 0; trip 2 (slot 2): mate slot 1 is episode 1; obs 2 is an extra
    got = trip_holding(slot, entry, exit, 3, obs=[-1, 0, 1, 2, -1], evaluation=[0, 8, 4, 8, 0])
    assert got.tolist() == [-1, 3, 1, -1, -1]
    got = trip_holding(slot, entry, exit, 3, obs=[1, 0, 0, 0, 0], evaluation=[3, 6, 5, 3, 0])
    assert got.tolist() == [2, -1, 0, 1, -1]        # evaluation 6: slot 0 empty between its trips


def test_trip_argument_checks():
    from junction_mpc.config import NPARAM, PARAM_INDEX
    from junction_mpc.episodes import Trips, trips_setup
    st = np.zeros((4, 4))
    tr = Trips([0, 0, 1, 1], [0, 5, 3, 0], [0, 1, 2, 0], st)
    prm = np.zeros(NPARAM)
    prm[PARAM_INDEX["dt"]] = 0.2
    order, params, prio = trips_setup(tr, 2, 2, 3, False, 0, "fixed", False, prm)
    assert order.tolist() == [0, 1, 3, 2] and params.shape == (4, NPARAM) and prio.tolist() == [0, 1, 0, 1]
    ok = dict(n_scenes=2, k=2, n_courses=3, planned=False, n_extra=0, right_of_way=None, share_plans=False,
              params_default=prm)

    def bad(match, trips=tr, **kw):
        with pytest.raises(ValueError, match=match):
            trips_setup(trips, **{**ok, **kw})
    for k in (1, 10, 2.0, True):
        bad(r"agents_per_scene in \[2, 9\]", k=k)
    bad("exceed the 8 obstacle slots", k=4, n_extra=6)
    bad("scene out of range", n_scenes=1)
    bad("course_id out of range", n_courses=2)
    bad("give no state", planned=True)
    bad("need state", trips=Trips([0], [0], [0]))
    bad("priority is an argument of the fixed", trips=Trips([0], [0], [0], st[:1], priority=[1.0]))
    bad("depart / on_goal", depart=np.zeros(4, np.int32))
    bad("depart / on_goal", on_goal="leave")
    bad("obstacle_script", obstacle_script=np.zeros((1, 4, 1, 6)))
    p2 = np.repeat(prm[None], 4, axis=0)
    p2[1, PARAM_INDEX["dt"]] = 0.1
    bad("one dt per scene: scene 0", trips=Trips([0, 0, 1, 1], [0, 5, 3, 0], [0, 1, 2, 0], st, p2), share_plans=True)
    p2[3, PARAM_INDEX["dt"]] = 0.1                      # scene 1 (trips 1, 3) at 0.1 s, scene 0 at 0.2 s
    trips_setup(Trips([0, 1, 0, 1], [0, 5, 3, 0], [0, 1, 2, 0], st, p2), **{**ok, "share_plans": True})
    with pytest.raises(ValueError, match="arrival must be >= 0"):
        Trips([0], [-1], [0], st[:1])
    with pytest.raises(ValueError, match="int32"):
        Trips([0], [2 ** 40], [0], st[:1])
    with pytest.raises(ValueError, match="integer array"):
        Trips([0], [0.5], [0], st[:1])
    with pytest.raises(ValueError, match=r"state must be \[1, 4\]"):
        Trips([0], [0], [0], np.zeros((1, 3)))
    with pytest.raises(ValueError, match=r"arrival must be \[2\]"):
        Trips([0, 0], [0], [0, 0], st[:2])


def test_poisson_trips_are_seeded_and_have_the_requested_rate():
    from junction_mpc.episodes import poisson_trips
    routes = [[(3 * g + r, (10.0 * g, 0.0, 0.5 * r)) for r in range(3)] for g in range(4)]
    a = poisson_trips(200, routes, 300.0, 0.2, 600, 4.0, seed=3)
    b = poisson_trips(200, routes, 300.0, 0.2, 600, 4.0, seed=3)
    for n in ("scene", "arrival", "course_id", "state"):
        assert np.array_equal(getattr(a, n), getattr(b, n)), n
    assert not np.array_equal(poisson_trips(200, routes, 300.0, 0.2, 600, 4.0, seed=4).arrival[:50], a.arrival[:50])
    mean = 200 * 4 * 300.0 * 600 * 0.2 / 3600            # scenes x approaches x rate x horizon
    assert abs(a.n - mean) < 4 * np.sqrt(mean)
    assert (np.diff(a.scene) >= 0).all() and (a.arrival < 600).all() and (a.state[:, 2] == 4.0).all()
    group = a.course_id // 3
    assert np.array_equal(a.state[:, 0], 10.0 * group) and np.array_equal(a.state[:, 3], 0.5 * (a.course_id % 3))
    assert poisson_trips(2, [[(0, None)]], 3600.0, 0.2, 50, seed=0).state is None


def test_trips_struct_matches_the_header():
    from junction_mpc import _cabi
    with open(os.path.join(ROOT, "include", "jmpc.h")) as f:
        body = re.search(r"typedef struct jmpc_trips \{(.*?)\} jmpc_trips;", f.read(), re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = []
    for decl in body.split(";"):
        decl = re.sub(r"\b(const|int32_t|double)\b", "", decl)
        names += [n.strip(" *\n") for n in decl.split(",") if n.strip(" *\n")]
    assert names == [f[0] for f in _cabi.Trips._fields_]


_PROPS = re.compile(r"Function properties for (\S+)\s*\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, "
                    r"(\d+) bytes spill loads\s*\n[^\n]*Used (\d+) registers")


@pytest.fixture(scope="module")
def resources(tmp_path_factory):
    if not os.path.exists(NVCC):
        pytest.skip(f"nvcc not found at {NVCC}")
    out = tmp_path_factory.mktemp("ptxas") / "jmpc.cubin"
    cmd = [NVCC, "-cubin", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
           "-Xptxas", "-v", "-o", str(out), SRC]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-4000:]
    return {m.group(1): (int(m.group(3)), int(m.group(4)), int(m.group(5))) for m in _PROPS.finditer(res.stderr)}


def _one(resources, pattern):
    hits = [v for k, v in resources.items() if re.fullmatch(pattern, k)]
    assert len(hits) == 1, (pattern, sorted(resources))
    return hits[0]


def test_trip_kernels_are_spill_free(resources):
    for pattern in (r"_ZN4jmpc18scene_trips_kernel.*", r"_ZN4jmpc25scene_trips_finish_kernel.*"):
        stores, loads, _ = _one(resources, pattern)
        assert (stores, loads) == (0, 0), pattern


def test_pinned_kernels_unchanged(resources):
    # the register counts of the sm_100a build before trips were added: the scene, rule and outcome kernels' sources
    # are untouched (the same pins as before lifetimes, plus the lifetime kernels)
    pinned = {r"_ZN4jmpc16collision_kernelILb0EEEvNS_13CollisionArgsE": 64,
              r"_ZN4jmpc16collision_kernelILb1EEEvNS_13CollisionArgsE": 64,
              r"_ZN4jmpc23masked_collision_kernelILb0EEEvNS_13CollisionArgsEPKi": 64,
              r"_ZN4jmpc23masked_collision_kernelILb1EEEvNS_13CollisionArgsEPKi": 64,
              r"_ZN4jmpc19right_of_way_kernel.*": 31, r"_ZN4jmpc18scene_plans_kernel.*": 17,
              r"_ZN4jmpc21scene_exchange_kernel.*": 28, r"_ZN4jmpc22episode_outcome_kernelENS_11OutcomeArgsE": 56}
    for pattern, regs in pinned.items():
        assert _one(resources, pattern) == (0, 0, regs), pattern
    for pattern in (r"_ZN4jmpc18scene_enter_kernel.*", r"_ZN4jmpc21scene_presence_kernel.*",
                    r"_ZN4jmpc20scene_outcome_kernel.*", r"_ZN4jmpc19episode_post_kernel.*"):
        stores, loads, _ = _one(resources, pattern)
        assert (stores, loads) == (0, 0), pattern
