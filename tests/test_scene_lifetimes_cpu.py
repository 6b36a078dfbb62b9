"""Lifetimes of scene vehicles (BatchedEpisodes(depart=..., on_goal=...)), CPU side: hand-built cases of the presence
rule and the extended oracles, the host argument checks, the waiting code against include/jmpc.h, and the register /
spill report of the new kernels and the pinned ones from ptxas for sm_100a."""
import math
import os
import re
import subprocess

import numpy as np
import pytest

from oracle import scene_exchange as SX
from oracle import scene_lifetimes as SL
from oracle.collision_oracle import CarGeometry

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "av-simulation-at-intersections_b200", "csrc", "jmpc.cu")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")


def test_presence_at_entry_and_at_leaving():
    # vehicle 0: depart 0, goal after 3 steps (goal test at the top of iteration 3); vehicle 1: depart 2, 4 steps, goal;
    # vehicle 2: depart 1, index rule after 2 steps (done = 2); vehicle 3: depart 9, has not entered after 6 evaluations
    depart, steps, done = [0, 2, 1, 9], [3, 4, 2, 0], [1, 1, 2, 5]
    park = SL.presence(depart, steps, done, "park", 8)
    leave = SL.presence(depart, steps, done, "leave", 8)
    assert park[:, 0].all() and not (leave[:, 0] != [1, 1, 1, 1, 0, 0, 0, 0]).any()      # present at e = 3, gone at 4
    assert (park[:, 1] == [0, 0, 1, 1, 1, 1, 1, 1]).all()                                # enters at evaluation 2
    assert (leave[:, 1] == [0, 0, 1, 1, 1, 1, 1, 0]).all()                               # goal tested at 6, gone at 7
    # done = 2 has not reached its goal: parked and present under both settings
    assert (park[:, 2] == [0, 1, 1, 1, 1, 1, 1, 1]).all() and (leave[:, 2] == park[:, 2]).all()
    assert not park[:, 3].any() and not leave[:, 3].any()
    with pytest.raises(ValueError, match="unknown on_goal"):
        SL.presence(depart, steps, done, "stay", 8)


def test_presence_masks():
    present = np.array([True, False, True, True, False, False, True, True])
    m = SL.presence_masks(present, 4)
    # episode 0: mates 1, 2, 3 in slots 0, 1, 2 -> slot 0 cleared; episode 1: mates 0, 2, 3 all present; episodes 2
    # and 3: mate 1 in slot 1
    assert m[0] == ~1 and m[1] == -1 and m[2] == ~2 and m[3] == ~2
    # episode 5 (scene 1, j = 1): mates 4, 6, 7 -> slot 0 cleared; episode 4: mates 5, 6, 7 -> slot 0
    assert m[4] == ~1 and m[5] == ~1 and m[6] == ~3 and m[7] == ~3
    # the extras' bits (k - 1 ..) always stay set
    assert all((int(x) >> 3) & 0x1FFFFFFF == 0x1FFFFFFF for x in m)
    with pytest.raises(ValueError):
        SL.presence_masks(present[:7], 4)


def test_rows_before_entry_are_the_parked_start_pose():
    B = 2
    state0 = np.array([[1.0, 2.0, 3.0, 0.5], [10.0, 20.0, 4.0, -0.5]])
    R = 6
    history = np.full((R, B, 8), np.nan)
    # vehicle 0 drives from iteration 0 for 2 steps, vehicle 1 enters at iteration 3 and drives 2 steps (rows 3, 4)
    for i, b in ((0, 0), (1, 0), (3, 1), (4, 1)):
        history[i, b] = [i + 100 * b, i, 0.1 * i, 5.0 + i, 0.0, 0.2 * i, -0.3 * i, 0.0]
    rows = SL.vehicle_rows(state0, history, steps=[2, 2], done=[1, 1], max_steer=0.5, n_eval=8, depart=[0, 3])
    parked_start = [10.0, 20.0, 0.0, -0.5, 0.0, 0.0]
    for e in range(3):
        assert rows[e, 1].tolist() == parked_start, e
    assert rows[3, 1].tolist() == [10.0, 20.0, 4.0, -0.5, 0.0, 0.0]           # entry: the start row, speed kept
    for e in (4, 5):                                                           # History rows 3, 4: x, y, v, yaw, a, steer
        h = history[e - 1, 1]
        assert rows[e, 1].tolist() == [h[0], h[1], h[3], h[2], h[6], min(h[5], 0.5)], e
    assert rows[6, 1].tolist() == [104.0, 4.0, 0.0, 0.4, 0.0, 0.0]            # parked from depart + steps + 1 = 6
    # depart = 0 is today's rows, parked from steps + 1 = 3
    assert np.array_equal(rows[:, 0], SL.vehicle_rows(state0, history, [2, 2], [1, 1], 0.5, 8, depart=[0, 3])[:, 0])
    assert rows[3, 0].tolist() == [1.0, 1.0, 0.0, 0.1, 0.0, 0.0]
    mates = SL.mate_rows(state0, history, [2, 2], [1, 1], 0.5, 2, 8, depart=[0, 3])
    assert np.array_equal(mates[:, 0, 0], rows[:, 1]) and np.array_equal(mates[:, 1, 0], rows[:, 0])


def test_outcomes_skip_absent_slots_and_start_at_the_first_evaluation():
    geo = CarGeometry()
    history = np.array([[0.5, 0.0, 0.0, 2.0, 0.0, 0.0, 1.0, 0.1]])
    far = [50.0, 0.0, 0.0, 0.0, 0.0, 0.0]
    touching = [2.0, 0.0, 0.0, 0.0, 0.0, 0.0]
    nan = [math.nan] * 6
    # slot 1 is absent at both evaluations although it would touch: no contact, the clearance is slot 0's
    track = np.array([[far, nan], [far, nan]])
    o = SL.episode_outcomes([0.0, 0.0, 1.5, 0.0], history, [0], track, dt=0.2, L=2.5, max_steer=0.6, geo=geo, first=7)
    assert o["first_contact_eval"] == -1 and o["contact_evals"] == 0
    assert o["min_clearance_eval"] == 8 and o["min_clearance_obs"] == 0                # global index: first + 1
    # the same slot present at the second evaluation: contact there, counted from `first`
    track[1, 1] = touching
    o = SL.episode_outcomes([0.0, 0.0, 1.5, 0.0], history, [0], track, dt=0.2, L=2.5, max_steer=0.6, geo=geo, first=7)
    assert (o["first_contact_eval"], o["first_contact_obs"], o["contact_evals"]) == (8, 1, 1)
    assert (o["min_clearance_eval"], o["min_clearance_obs"]) == (8, 1)
    # every slot absent at every evaluation: the empty record's clearance columns
    o = SL.episode_outcomes([0.0, 0.0, 1.5, 0.0], history, [0], np.full((2, 2, 6), np.nan), dt=0.2, L=2.5,
                            max_steer=0.6, geo=geo, first=3)
    assert (o["min_clearance"], o["min_clearance_eval"], o["min_clearance_obs"]) == (math.inf, -1, -1)
    assert o["distance"] == 0.5 and o["max_abs_accel"] == 1.0


def test_lifetime_argument_checks():
    from junction_mpc.episodes import lifetime_setup
    assert lifetime_setup(None, "park", 4, 8) is None
    assert lifetime_setup(np.zeros(8, np.int64), "park", 4, 8) is None
    assert lifetime_setup([0] * 8, "park", 1, 8) is None
    dep, leave = lifetime_setup(None, "leave", 4, 8)
    assert dep.dtype == np.int32 and not dep.any() and leave
    dep, leave = lifetime_setup(np.arange(8, dtype=np.int16), "park", 1, 8)      # depart with one vehicle per scene
    assert dep.dtype == np.int32 and dep.tolist() == list(range(8)) and not leave
    with pytest.raises(ValueError, match="on_goal must be 'park' or 'leave'"):
        lifetime_setup(None, "stay", 4, 8)
    with pytest.raises(ValueError, match="on_goal must be 'park' or 'leave'"):
        lifetime_setup(None, None, 4, 8)
    with pytest.raises(ValueError, match="needs agents_per_scene > 1"):
        lifetime_setup(None, "leave", 1, 8)
    with pytest.raises(ValueError, match="integer array"):
        lifetime_setup(np.zeros(8), "park", 4, 8)
    with pytest.raises(ValueError, match="integer array"):
        lifetime_setup(np.zeros(8, bool), "park", 4, 8)
    with pytest.raises(ValueError, match=r"depart must be \[8\]"):
        lifetime_setup(np.zeros(4, np.int32), "park", 4, 8)
    with pytest.raises(ValueError, match=r"depart must be \[8\]"):
        lifetime_setup(np.zeros((8, 1), np.int32), "park", 4, 8)
    with pytest.raises(ValueError, match=">= 0"):
        lifetime_setup([0, 1, 2, -1, 0, 0, 0, 0], "park", 4, 8)
    with pytest.raises(ValueError, match="int32"):
        lifetime_setup([0, 1, 2, 2 ** 40, 0, 0, 0, 0], "park", 4, 8)


def test_waiting_code_matches_the_header():
    from junction_mpc import _cabi
    with open(os.path.join(ROOT, "include", "jmpc.h")) as f:
        text = f.read()
    body = re.search(r"enum jmpc_scene_lifetime \{(.*?)\};", text, re.S).group(1)
    assert dict(re.findall(r"JMPC_([A-Z_]+) = (\d+)", body)) == {"WAITING": str(_cabi.WAITING)}
    done = re.search(r"enum jmpc_done \{(.*?)\};", text, re.S).group(1)
    assert str(_cabi.WAITING) not in re.findall(r"= (\d+)", done)
    assert _cabi.WAITING not in SX.NEVER_STEPPED


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


def test_new_kernels_are_spill_free(resources):
    for pattern in (r"_ZN4jmpc24scene_depart_init_kernel.*", r"_ZN4jmpc18scene_enter_kernel.*",
                    r"_ZN4jmpc21scene_presence_kernel.*", r"_ZN4jmpc20scene_outcome_kernel.*"):
        stores, loads, _ = _one(resources, pattern)
        assert (stores, loads) == (0, 0), pattern


def test_pinned_kernels_unchanged(resources):
    # the register counts of the sm_100a build before lifetimes were added: these kernels' sources are untouched, and
    # the plain outcome kernel shares its body with scene_outcome_kernel through a template flag
    pinned = {r"_ZN4jmpc16collision_kernelILb0EEEvNS_13CollisionArgsE": 64,
              r"_ZN4jmpc16collision_kernelILb1EEEvNS_13CollisionArgsE": 64,
              r"_ZN4jmpc23masked_collision_kernelILb0EEEvNS_13CollisionArgsEPKi": 64,
              r"_ZN4jmpc23masked_collision_kernelILb1EEEvNS_13CollisionArgsEPKi": 64,
              r"_ZN4jmpc19right_of_way_kernel.*": 31, r"_ZN4jmpc18scene_plans_kernel.*": 17,
              r"_ZN4jmpc21scene_exchange_kernel.*": 28, r"_ZN4jmpc22episode_outcome_kernelENS_11OutcomeArgsE": 56}
    for pattern, regs in pinned.items():
        assert _one(resources, pattern) == (0, 0, regs), pattern


def test_without_lifetimes_the_extended_oracles_are_the_scene_oracles():
    from oracle import episode_outcomes as EO
    rng = np.random.default_rng(1)
    B, R = 8, 12
    state0 = rng.normal(size=(B, 4))
    history = rng.normal(size=(R, B, 8))
    steps = rng.integers(0, R + 1, B)
    done = rng.choice([0, 1, 2, 3, 4], B)
    steps[np.isin(done, SX.NEVER_STEPPED)] = 0
    for k in (1, 2, 4):
        assert np.array_equal(SL.mate_rows(state0, history, steps, done, 0.4, k, R + 1),
                              SX.mate_rows(state0, history, steps, done, 0.4, k, R + 1))
    track = rng.normal(scale=3.0, size=(R + 1, 3, 6))
    flags = rng.integers(-1, 2, R)
    assert SL.episode_outcomes(state0[0], history[:, 0], flags, track, 0.2, 2.5, 0.6) == \
        EO.episode_outcomes(state0[0], history[:, 0], flags, track, 0.2, 2.5, 0.6)
