"""Circle-centre tables rebuilt for a new car geometry after the courses are loaded (jmpc_set_car_geometry).

The collision kernel reads the ego's circle centres from per-course tables built when the courses are uploaded, and
computes the obstacles' circles and the reach from the handle's geometry.  A geometry set afterwards must rebuild the
tables, or the ego's circles stay where the old geometry put them and the flags and cut lengths drift from the
oracle's.  Flags and cut lengths are integers defined bit for bit by oracle/collision_oracle.py, so the checks are
exact."""
import numpy as np
import pytest

from helpers import load_planner_golden
from oracle import collision_oracle as C

pytestmark = pytest.mark.gpu

GEO = C.CarGeometry(width=1.8)
DS = 0.083                                  # point spacing of the recorded courses
MARGIN = C.cutoff_margin(GEO, DS)


def test_car_geometry_after_courses_matches_oracle(golden_dir):
    import __graft_entry__ as g
    g.build()
    from junction_mpc import synth
    from junction_mpc.batched import BatchedMPC
    from junction_mpc.config import PARAM_INDEX as PI
    z = load_planner_golden(golden_dir)
    courses = [np.array(z[f"{n}/trajectory"], dtype=np.float64) for n in z["variants"] if len(z[f"{n}/trajectory"])]
    for c in courses:
        synth.smooth_yaw_inplace(c[:, 2])
    assert len(courses) == 51
    B = 4096
    mpc = BatchedMPC(courses, dl=DS, T=13, max_batch=B)
    assert mpc.arc_table_flags().all()
    rng = np.random.default_rng(1808)
    cid = rng.integers(0, len(courses), B).astype(np.int32)
    a0 = np.array([rng.integers(0, len(courses[c])) for c in cid], dtype=np.int32)
    v = rng.uniform(0, 30 / 3.6, B)
    obs = np.zeros((B, 2, 6))
    for b in range(B):                      # scattered around the ego, the first one next to the path ahead
        c = courses[cid[b]]
        obs[b, :, :2] = c[a0[b], :2] + rng.uniform(-35, 35, (2, 2))
        obs[b, 0, :2] = c[min(a0[b] + int(rng.integers(0, 200)), len(c) - 1), :2] + rng.uniform(-8, 8, 2)
    obs[:, :, 2] = rng.uniform(0, 30 / 3.6, (B, 2))
    obs[:, :, 3] = rng.uniform(-np.pi, np.pi, (B, 2))
    obs[:, :, 5] = rng.uniform(-0.4, 0.4, (B, 2))
    run = lambda: mpc.collision_host(a0, v, obs, frame_window=20, margin=MARGIN, course_id=cid)   # noqa: E731
    default = run()

    before = mpc.launch_count
    mpc.set_car_geometry(*GEO.circle_offsets, GEO.radius)
    assert mpc.launch_count == before + 1   # the circle tables only: the arc-length tables stay
    flag, clen = run()
    p = mpc.default_params
    want = np.array([C.collision_cut(GEO, courses[cid[b]], int(a0[b]), float(v[b]), obs[b], dt=p[PI["dt"]], frame_window=20,
                                     max_accel=p[PI["max_accel"]], max_speed=p[PI["sim_max_speed"]], margin=MARGIN)
                     for b in range(B)], dtype=np.int64)
    bad = np.flatnonzero((flag != want[:, 0]) | (clen != want[:, 1]))
    assert len(bad) == 0, [(int(b), flag[b], clen[b], tuple(want[b])) for b in bad[:10]]
    assert 0.05 < (flag == 1).mean() < 0.95
    assert (clen != default[1]).sum() >= 100          # the geometry decides many of the cut lengths

    d = C.CarGeometry()                     # back to the default geometry: the first results again
    mpc.set_car_geometry(*d.circle_offsets, d.radius)
    assert all(np.array_equal(x, y) for x, y in zip(run(), default))
    mpc.close()
