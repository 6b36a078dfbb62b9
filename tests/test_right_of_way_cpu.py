"""Right-of-way rules (BatchedEpisodes(right_of_way=...)), CPU side: hand-built cases of oracle/right_of_way.py, the
host argument checks, and the register / spill report of the new and the existing collision kernels from ptxas for
sm_100a."""
import os
import re
import subprocess

import numpy as np
import pytest

from oracle import right_of_way as RW

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "av-simulation-at-intersections_b200", "csrc", "jmpc.cu")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
ALL = -1


def _bits(mask, k):
    """The mate slots 0 .. k - 2 whose bit is set; every bit above them must be set too (extras always considered)."""
    m = int(mask) & 0xFFFFFFFF
    assert m >> (k - 1) == 0xFFFFFFFF >> (k - 1), hex(m)
    return [s for s in range(k - 1) if (m >> s) & 1]


def test_zone_indices():
    xs = np.linspace(-20, 20, 401)
    course = np.stack([xs, np.full(401, 3.0), np.zeros(401)], axis=1)
    entry, exit_ = RW.zone_indices(course, (0.0, 0.0, 5.0))
    assert (entry, exit_) == (160, 240)                   # |x| <= 4 at y = 3: x = -4.0 .. 4.0
    assert RW.zone_indices(course, (0.0, 0.0, 2.9)) == (-1, -1)
    assert RW.zone_indices(course, (0.0, 3.0, 0.05)) == (200, 200)
    # the boundary: dx * dx + dy * dy <= r * r with separate roundings, exactly 5 m from the centre is inside
    assert RW.zone_indices(np.array([[3.0, 4.0], [3.0, 4.0 + 1e-12]]), (0.0, 0.0, 5.0)) == (0, 0)
    # a course that leaves and re-enters: the first and the last point inside
    course2 = np.concatenate([course, course[::-1]])
    assert RW.zone_indices(course2, (0.0, 0.0, 5.0)) == (160, 641)


def test_fixed_ties_broken_by_episode_index():
    a = np.zeros(8, np.int64)
    done = np.zeros(8, np.int64)
    # default priorities j: vehicle j yields to vehicles 0 .. j - 1 of its scene
    m = RW.consider_masks("fixed", 4, a, done, priority=np.arange(8) % 4)
    assert [_bits(x, 4) for x in m] == [[], [0], [0, 1], [0, 1, 2]] * 2
    # equal keys: the lower episode index goes first
    m = RW.consider_masks("fixed", 4, a, done, priority=np.full(8, 2.5))
    assert [_bits(x, 4) for x in m[:4]] == [[], [0], [0, 1], [0, 1, 2]]
    # a smaller key wins over the index: vehicle 3 first, then 1, 0 = 2 (tie -> 0 before 2)
    m = RW.consider_masks("fixed", 4, a[:4], done[:4], priority=[1.0, 0.5, 1.0, -3.0])
    # slots of b: its mates in episode order without b
    assert _bits(m[3], 4) == [] and _bits(m[1], 4) == [2]          # 1 yields to 3 (its slot 2)
    assert _bits(m[0], 4) == [0, 2] and _bits(m[2], 4) == [0, 1, 2]


def test_first_come_committed_ahead_of_approaching_and_past_ahead_of_inside():
    dl = 0.1
    # zone [100, 200] for every vehicle; vehicle 0 approaching 5 points out, 1 inside 30 points before the exit,
    # 2 past the zone, 3 approaching 50 points out
    zone = np.array([[100, 200]] * 4)
    a = np.array([95, 170, 230, 50])
    cls, key = RW.scene_keys("first_come", a, dl, zone)
    assert cls.tolist() == [1, 0, 0, 1]
    assert key.tolist() == [5 * dl, 30 * dl, -30 * dl, 50 * dl]
    m = RW.consider_masks("first_come", 4, a, np.zeros(4), dl, zone)
    # order: 2 (past), 1 (inside), 0 (approaching, closer), 3
    assert _bits(m[2], 4) == [] and _bits(m[1], 4) == [1] and _bits(m[0], 4) == [0, 1] and _bits(m[3], 4) == [0, 1, 2]
    # entering the zone is committed: a = entry gives class 0 with key (exit - entry) dl
    cls, key = RW.scene_keys("first_come", [100], dl, [[100, 200]])
    assert (cls[0], key[0]) == (0, 100 * dl)
    # the distances are course indices x each vehicle's own dl
    cls, key = RW.scene_keys("first_come", [90, 90], [0.1, 0.2], [[100, 150], [100, 150]])
    assert cls.tolist() == [1, 1] and key.tolist() == [10 * 0.1, 10 * 0.2]


def test_first_come_ties_and_a_course_that_never_enters():
    zone = np.array([[100, 200], [40, 140], [-1, -1], [-1, -1]])
    a = np.array([90, 30, 10, 70])                      # 0 and 1 both 10 points from their entry: a tie
    m = RW.consider_masks("first_come", 4, a, np.zeros(4), 0.1, zone)
    assert _bits(m[0], 4) == [] and _bits(m[1], 4) == [0]          # tie -> episode 0 first
    # the two that never enter yield to every moving mate, and between them the index decides
    assert _bits(m[2], 4) == [0, 1] and _bits(m[3], 4) == [0, 1, 2]
    cls, key = RW.scene_keys("first_come", a, 0.1, zone)
    assert cls.tolist() == [1, 1, 2, 2] and key[2] == key[3] == 0.0


def test_parked_mates_and_extras_always_considered():
    k = 3
    prio = np.array([0.0, 1.0, 2.0])
    # vehicle 0 has the highest priority; its mate 2 is parked (done = 1): 0 considers it, not the moving mate 1
    m = RW.consider_masks("fixed", k, np.zeros(3), [0, 0, 1], priority=prio)
    assert _bits(m[0], k) == [1] and _bits(m[1], k) == [0, 1]
    assert m[2] == ALL                                  # a finished episode: every bit
    # every parked code counts (goal, index rule, never stepped), and a parked mate ahead in the order too
    for code in (1, 2, 3, 4):
        m = RW.consider_masks("fixed", k, np.zeros(3), [0, code, 0], priority=prio)
        assert _bits(m[0], k) == [0] and _bits(m[2], k) == [0, 1]
    # the extras' bits (slots k - 1 ..) are set in every mask
    m = RW.consider_masks("first_come", k, [0, 0, 0], [0, 0, 0], 0.1, [[5, 9], [6, 9], [7, 9]])
    for x in m:
        assert all((int(x) >> s) & 1 for s in range(k - 1, 32))
    rows = np.arange(5 * 6, dtype=float).reshape(5, 6)
    assert [r[0] for r in RW.considered_rows(rows, m[0])] == [12.0, 18.0, 24.0]    # mates ignored, 3 extras kept


def test_top_vehicle_considers_only_parked_mates_and_extras():
    rng = np.random.default_rng(3)
    k, B = 5, 200
    for _ in range(20):
        zone = rng.integers(0, 300, (B, 2))
        zone.sort(axis=1)
        zone[rng.random(B) < 0.2] = -1
        a = rng.integers(0, 400, B)
        done = np.where(rng.random(B) < 0.3, rng.integers(1, 3, B), 0)
        dl = rng.choice([0.1, 0.2], B)
        for rule, kw in (("first_come", dict(dl=dl, zone=zone)), ("fixed", dict(priority=rng.integers(0, 3, B)))):
            m = RW.consider_masks(rule, k, a, done, **kw)
            cls, key = RW.scene_keys(rule, a, kw.get("dl"), kw.get("zone"), kw.get("priority"))
            for s in range(B // k):
                idx = [s * k + j for j in range(k)]
                moving = [b for b in idx if done[b] == 0]
                if not moving:
                    continue
                top = min(moving, key=lambda b: (cls[b], key[b], b))
                mates = [q for q in idx if q != top]
                assert _bits(m[top], k) == [slot for slot, q in enumerate(mates) if done[q] != 0]
                # total order: of any two moving vehicles exactly one considers the other
                for b in moving:
                    for q in moving:
                        if b < q:
                            sb = [x for x in idx if x != b].index(q)
                            sq = [x for x in idx if x != q].index(b)
                            assert ((int(m[b]) >> sb) & 1) + ((int(m[q]) >> sq) & 1) == 1


def test_oracle_argument_errors():
    with pytest.raises(ValueError):
        RW.consider_masks("fixed", 1, [0], [0], priority=[0.0])
    with pytest.raises(ValueError):
        RW.consider_masks("fixed", 3, [0] * 4, [0] * 4, priority=[0.0] * 4)
    with pytest.raises(ValueError, match="unknown rule"):
        RW.scene_keys("priority_to_the_right", [0])


def test_right_of_way_argument_checks():
    from junction_mpc import _cabi
    from junction_mpc.episodes import right_of_way_setup
    assert right_of_way_setup(None, 4, 8) is None
    assert right_of_way_setup(None, 1, 8) is None
    rule, prio, junc = right_of_way_setup("fixed", 4, 8)
    assert rule == _cabi.ROW_FIXED and prio.tolist() == [0, 1, 2, 3] * 2 and junc is None
    rule, prio, junc = right_of_way_setup("fixed", 4, 8, priority=np.arange(8)[::-1])
    assert prio.dtype == np.float64 and prio.tolist() == list(range(7, -1, -1))
    rule, prio, junc = right_of_way_setup("first_come", 4, 8, junction=(0.0, 0.0, 10.0))
    assert rule == _cabi.ROW_FIRST_COME and prio is None and junc.shape == (1, 3)
    assert right_of_way_setup("first_come", 4, 8, junction=[[0, 0, 10], [1, 1, 9]])[2].shape == (2, 3)
    with pytest.raises(ValueError, match="needs agents_per_scene > 1"):
        right_of_way_setup("fixed", 1, 8)
    with pytest.raises(ValueError, match="needs agents_per_scene > 1"):
        right_of_way_setup("first_come", 1, 8, junction=(0, 0, 10))
    with pytest.raises(ValueError, match="must be None, 'fixed' or 'first_come'"):
        right_of_way_setup("priority_to_the_right", 4, 8)
    with pytest.raises(ValueError, match="must be None, 'fixed' or 'first_come'"):
        right_of_way_setup(True, 4, 8)
    with pytest.raises(ValueError, match="needs junction"):
        right_of_way_setup("first_come", 4, 8)
    for bad in ((0, 0, 0.0), (0, 0, -1.0), (np.nan, 0, 10), (0, np.inf, 10), (0, 0, np.nan)):
        with pytest.raises(ValueError, match="finite with r > 0"):
            right_of_way_setup("first_come", 4, 8, junction=bad)
    with pytest.raises(ValueError, match="junction must be"):
        right_of_way_setup("first_come", 4, 8, junction=[[0, 0, 10]] * 3)
    with pytest.raises(ValueError, match="junction must be"):
        right_of_way_setup("first_come", 4, 8, junction=(0, 0))
    with pytest.raises(ValueError, match="takes no priority"):
        right_of_way_setup("first_come", 4, 8, priority=np.zeros(8), junction=(0, 0, 10))
    with pytest.raises(ValueError, match="takes no junction"):
        right_of_way_setup("fixed", 4, 8, junction=(0, 0, 10))
    with pytest.raises(ValueError, match="priority must be finite"):
        right_of_way_setup("fixed", 4, 8, priority=[0, 1, 2, np.nan, 0, 1, 2, 3])
    with pytest.raises(ValueError, match="priority must be finite"):
        right_of_way_setup("fixed", 4, 8, priority=[0, 1, 2, np.inf, 0, 1, 2, 3])
    with pytest.raises(ValueError, match=r"priority must be \[8\]"):
        right_of_way_setup("fixed", 4, 8, priority=np.zeros(4))
    with pytest.raises(ValueError, match=r"priority must be \[8\]"):
        right_of_way_setup("fixed", 4, 8, priority=np.zeros((8, 1)))
    with pytest.raises(ValueError, match="give right_of_way too"):
        right_of_way_setup(None, 4, 8, priority=np.zeros(8))
    with pytest.raises(ValueError, match="give right_of_way too"):
        right_of_way_setup(None, 4, 8, junction=(0, 0, 10))


def test_rule_enum_matches_python():
    from junction_mpc import _cabi
    with open(os.path.join(ROOT, "include", "jmpc.h")) as f:
        body = re.search(r"enum jmpc_right_of_way_rule \{(.*?)\};", f.read(), re.S).group(1)
    values = dict(re.findall(r"JMPC_ROW_([A-Z_]+) = (\d+)", body))
    assert values == {"FIXED": str(_cabi.ROW_FIXED), "FIRST_COME": str(_cabi.ROW_FIRST_COME)}


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
    for pattern in (r"_ZN4jmpc23masked_collision_kernelILb0EEEvNS_13CollisionArgsEPKi",
                    r"_ZN4jmpc23masked_collision_kernelILb1EEEvNS_13CollisionArgsEPKi",
                    r"_ZN4jmpc19right_of_way_kernel.*", r"_ZN4jmpc24right_of_way_init_kernel.*"):
        stores, loads, _ = _one(resources, pattern)
        assert (stores, loads) == (0, 0), pattern


def test_existing_collision_kernels_unchanged(resources):
    for flag in (0, 1):
        stores, loads, regs = _one(resources, rf"_ZN4jmpc16collision_kernelILb{flag}EEEvNS_13CollisionArgsE")
        assert (stores, loads) == (0, 0) and regs <= 64, flag
