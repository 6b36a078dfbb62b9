"""Numpy restatement of the scene exchange (TEST INFRASTRUCTURE ONLY, see oracle/__init__.py).

Rebuilds, from what a run with History returns, the obstacle rows that the vehicles of a scene see of each other at
every evaluation (jmpc_scene_exchange in include/jmpc.h).  Episode b = s * k + j is vehicle j of scene s; its first
k - 1 obstacle slots hold its mates in episode order, skipping itself.  Evaluation e = 0 is the start; e = i + 1 follows
loop iteration i, where History row i is the state after a vehicle's step i.  A vehicle that executed n steps and
ended with `done`:
  * e <= n and not a never-stepped vehicle (done 3 / 4): moving, row (x, y, v, yaw, a, clamp(delta, +-max_steer)) of
    History row e - 1 (a = History column 6: MAX_DECEL after a failed solve; delta = column 5), or
    (x, y, v, yaw, 0, 0) of the start state at e = 0;
  * otherwise parked: its last pose (History row n - 1, or the start state) with v = a = steer = 0.
A vehicle stops stepping (goal, index rule) in the iteration after its last step, so the first parked row is n + 1.
"""
from __future__ import annotations

import numpy as np

NEVER_STEPPED = (3, 4)        # JMPC_DONE_NO_COURSE, JMPC_DONE_MATE_NO_COURSE


def vehicle_rows(state0, history, steps, done, max_steer, n_eval: int) -> np.ndarray:
    """state0 [B, 4] x, y, v, yaw; history [R, B, 8] (x, y, yaw, v, t, delta, a, xref_dev); steps, done [B];
    max_steer scalar or [B].  Returns [n_eval, B, 6]: the row every vehicle presents to its mates at evaluations
    0 .. n_eval - 1."""
    state0 = np.asarray(state0, np.float64)
    history = np.asarray(history, np.float64)
    steps, done = np.asarray(steps, np.int64), np.asarray(done, np.int64)
    B = len(state0)
    max_steer = np.broadcast_to(np.asarray(max_steer, np.float64), (B,))
    if history.ndim != 3 or history.shape[1:] != (B, 8):
        raise ValueError(f"history must be [rows, {B}, 8]")
    if (steps > len(history)).any():
        raise ValueError("history holds fewer rows than a vehicle executed steps")
    cols = lambda h: np.stack([h[..., 0], h[..., 1], h[..., 3], h[..., 2]], axis=-1)   # noqa: E731  x, y, v, yaw
    bs = np.arange(B)
    last = np.where((steps == 0)[:, None], state0, cols(history[np.maximum(steps - 1, 0), bs]) if len(history) else state0)
    parked_from = np.where(np.isin(done, NEVER_STEPPED), 0, steps + 1)
    out = np.empty((n_eval, B, 6))
    for e in range(n_eval):
        if e == 0:
            row = np.concatenate([state0, np.zeros((B, 2))], axis=1)
        else:
            h = history[min(e - 1, len(history) - 1)] if len(history) else np.full((B, 8), np.nan)
            steer = np.maximum(np.minimum(h[:, 5], max_steer), -max_steer)
            row = np.concatenate([cols(h), h[:, 6:7], steer[:, None]], axis=1)
        parked = np.concatenate([last[:, :2], np.zeros((B, 1)), last[:, 3:4], np.zeros((B, 2))], axis=1)
        out[e] = np.where((e >= parked_from)[:, None], parked, row)
    return out


def mate_rows(state0, history, steps, done, max_steer, k: int, n_eval: int) -> np.ndarray:
    """[n_eval, B, k - 1, 6]: the scene-mate slots of every episode at evaluations 0 .. n_eval - 1."""
    rows = vehicle_rows(state0, history, steps, done, max_steer, n_eval)
    B = rows.shape[1]
    if k < 1 or B % k:
        raise ValueError(f"B = {B} is not a multiple of k = {k}")
    out = np.empty((n_eval, B, k - 1, 6))
    for b in range(B):
        s, j = divmod(b, k)
        mates = [s * k + m for m in range(k) if m != j]
        out[:, b] = rows[:, mates]
    return out
