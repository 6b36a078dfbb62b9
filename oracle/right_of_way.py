"""Numpy restatement of the right-of-way rules (TEST INFRASTRUCTURE ONLY, see oracle/__init__.py).

Which scene mates a vehicle yields to (jmpc_right_of_way_init / jmpc_right_of_way in include/jmpc.h):
  * zone_indices: the first and last point of a course inside the junction zone;
  * scene_keys: every vehicle's key (class, key), compared lexicographically and then by episode index;
  * consider_masks: the consider mask of every episode at one evaluation, from a snapshot of agent_idx / done / params.
The masked collision cut needs no oracle of its own: it is collision_oracle.collision_cut on the considered rows only,
because dropping rows keeps the reference's row order of the others.
"""
from __future__ import annotations

import numpy as np

FIXED, FIRST_COME = "fixed", "first_come"


def zone_indices(course, junction):
    """course [N, >= 2] (x, y, ...); junction (x, y, r).  Returns (entry, exit): the first and last index with
    dx * dx + dy * dy <= r * r (numpy: separate products and sum, no fused multiply-add), or (-1, -1)."""
    course = np.asarray(course, np.float64)
    x, y, r = (float(c) for c in junction)
    dx, dy = course[:, 0] - x, course[:, 1] - y
    inside = np.flatnonzero(dx * dx + dy * dy <= r * r)
    if len(inside) == 0:
        return -1, -1
    return int(inside[0]), int(inside[-1])


def scene_keys(rule: str, agent_idx, dl=None, zone=None, priority=None):
    """(cls [B] int64, key [B] float64) of every episode.  fixed: (0, priority).  first_come, a = agent_idx, zone
    [B, 2] (entry, exit), dl [B]: committed (a >= entry) (0, (exit - a) dl), approaching (1, (entry - a) dl), a course
    that never enters the zone (entry < 0) (2, 0)."""
    agent_idx = np.asarray(agent_idx, np.int64)
    B = len(agent_idx)
    if rule == FIXED:
        return np.zeros(B, np.int64), np.asarray(priority, np.float64).copy()
    if rule != FIRST_COME:
        raise ValueError(f"unknown rule {rule!r}")
    zone = np.asarray(zone, np.int64)
    dl = np.broadcast_to(np.asarray(dl, np.float64), (B,))
    entry, exit_ = zone[:, 0], zone[:, 1]
    cls = np.where(entry < 0, 2, np.where(agent_idx >= entry, 0, 1))
    key = np.where(cls == 0, (exit_ - agent_idx).astype(np.float64) * dl,
                   np.where(cls == 1, (entry - agent_idx).astype(np.float64) * dl, 0.0))
    return cls, key


def consider_masks(rule: str, k: int, agent_idx, done, dl=None, zone=None, priority=None) -> np.ndarray:
    """int32 [B]: every bit set except the mate slots s (0 .. k - 2, the mates in episode order without b) whose mate
    is moving (done = 0) and does not come before b in (cls, key, episode index); -1 for a finished b."""
    done = np.asarray(done, np.int64)
    B = len(done)
    if k < 2 or B % k:
        raise ValueError(f"need k >= 2 dividing B = {B}")
    cls, key = scene_keys(rule, agent_idx, dl, zone, priority)
    order = lambda m: (int(cls[m]), float(key[m]), m)     # noqa: E731
    out = np.full(B, -1, np.int64)
    for b in range(B):
        if done[b]:
            continue
        s, j = divmod(b, k)
        mask = 0xFFFFFFFF
        for slot, m in enumerate(s * k + q for q in range(k) if q != j):
            if done[m] == 0 and not order(m) < order(b):
                mask &= ~(1 << slot)
        out[b] = mask - (1 << 32) if mask >= 1 << 31 else mask
    return out.astype(np.int32)


def considered_rows(rows, mask: int):
    """The obstacle rows [n_obs, 6] of one episode whose bit is set in its consider mask, in slot order."""
    return [r for s, r in enumerate(rows) if (int(mask) >> s) & 1]
