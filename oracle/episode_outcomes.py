"""Numpy restatement of the per-episode outcome record (TEST INFRASTRUCTURE ONLY, see oracle/__init__.py).

Computes the public columns of enum jmpc_outcome (include/jmpc.h) for one episode from what a run with History returns:
the start state, the History rows (x, y, yaw, v, t, delta, a, xref_deviation; row i = the state after step i), the
collision flags of the executed steps, three parameters and a track of obstacle poses.  Evaluation e pairs the ego pose
of evaluation e (e = 0: the start state; e = i + 1: History row i) with track[e].  Circles as the collision check
draws them (collision_oracle.circle_tracks): clearance of (ego, obstacle) = min over the 4 circle pairs of dist - 2r,
contact <=> dist <= 2r for some pair (collision_oracle.check_collision's test).
"""
from __future__ import annotations

import math

import numpy as np

from .collision_oracle import CarGeometry, circle_tracks

COLUMNS = ("min_clearance", "min_clearance_eval", "min_clearance_obs", "first_contact_eval", "first_contact_obs",
           "contact_evals", "cut_steps", "limit_steps", "failed_solves", "max_abs_accel", "max_abs_jerk",
           "max_abs_steer_rate", "max_abs_lat_accel", "max_xref_dev", "sum_xref_dev", "distance")


def clearance_and_contact(ego_poses: np.ndarray, track: np.ndarray, geo: CarGeometry = CarGeometry()):
    """ego_poses [E, 3] (x, y, yaw), track [E, n_obs, >= 4] (x, y, v, yaw, ...) -> clearance [E, n_obs] and contact
    [E, n_obs] (bool)."""
    E, n_obs = track.shape[0], track.shape[1]
    reach = 2 * geo.radius
    ego = circle_tracks(np.asarray(ego_poses, np.float64), geo)                 # (2, E, 2)
    clear = np.empty((E, n_obs))
    hit = np.zeros((E, n_obs), bool)
    for k in range(n_obs):
        obs = circle_tracks(track[:, k][:, [0, 1, 3]], geo)                     # (2, E, 2)
        diff = ego[:, None] - obs[None, :]                                      # (ego circle, obs circle, E, 2)
        dist = np.sqrt(diff[..., 0] * diff[..., 0] + diff[..., 1] * diff[..., 1])
        clear[:, k] = (dist - reach).min(axis=(0, 1))
        hit[:, k] = (dist <= reach).any(axis=(0, 1))
    return clear, hit


def episode_outcomes(state0, history, flags, track, dt: float, L: float, max_steer: float,
                     geo: CarGeometry = CarGeometry()) -> dict:
    """state0 [4] x, y, v, yaw; history [n, 8] the episode's executed steps; flags [n]; track [n + 1, n_obs, 6].
    Returns a dict of the public columns (python floats / ints)."""
    history = np.asarray(history, np.float64).reshape(-1, 8)
    n = len(history)
    flags = np.asarray(flags).reshape(-1)[:n]
    track = np.asarray(track, np.float64)
    if track.ndim != 3 or track.shape[0] != n + 1:
        raise ValueError(f"track must be [{n + 1}, n_obs, 6]")
    x0, y0, v0, yaw0 = (float(s) for s in state0)
    out = dict(min_clearance=math.inf, min_clearance_eval=-1, min_clearance_obs=-1, first_contact_eval=-1,
               first_contact_obs=-1, contact_evals=0)
    poses = np.vstack([[[x0, y0, yaw0]], history[:, :3]])
    if track.shape[1] > 0:
        clear, hit = clearance_and_contact(poses, track, geo)
        flat = clear.reshape(-1)
        j = int(np.argmin(flat))                         # first occurrence: earliest evaluation, then lowest obstacle
        out.update(min_clearance=float(flat[j]), min_clearance_eval=j // clear.shape[1],
                   min_clearance_obs=j % clear.shape[1])
        any_hit = hit.any(axis=1)
        out["contact_evals"] = int(any_hit.sum())
        if any_hit.any():
            e = int(np.argmax(any_hit))
            out.update(first_contact_eval=e, first_contact_obs=int(np.argmax(hit[e])))
    out["cut_steps"] = int((flags == 1).sum())
    out["limit_steps"] = int((flags == -1).sum())
    dev = history[:, 7]
    ok = np.isfinite(dev)                                # History column 7 is NaN after a failed solve
    out["failed_solves"] = int(n - ok.sum())
    a = history[:, 6]
    steer = np.clip(history[:, 5], -max_steer, max_steer)
    v_before = np.concatenate([[v0], history[:-1, 3]]) if n else np.zeros(0)
    lat = v_before * ((v_before / L) * np.tan(steer))
    m = lambda z: float(np.abs(z).max()) if len(z) else 0.0       # noqa: E731
    out["max_abs_accel"] = m(a)
    out["max_abs_jerk"] = m((a[1:] - a[:-1]) / dt)
    out["max_abs_steer_rate"] = m((steer[1:] - steer[:-1]) / dt)
    out["max_abs_lat_accel"] = m(lat)
    total = 0.0
    for d in dev[ok]:                                    # sequential, as the record accumulates it
        total += float(d)
    out["max_xref_dev"] = float(dev[ok].max()) if ok.any() else 0.0
    out["sum_xref_dev"] = total
    dist = 0.0
    for i in range(n):
        dist += math.hypot(poses[i + 1, 0] - poses[i, 0], poses[i + 1, 1] - poses[i, 1])
    out["distance"] = dist
    return out
