"""Numpy restatement of vehicle lifetimes in scenes (TEST INFRASTRUCTURE ONLY, see oracle/__init__.py).

BatchedEpisodes(depart=..., on_goal=...): vehicle b takes its first step in loop iteration depart[b] and, with
on_goal = "leave", is absent once its goal test has fired (jmpc_scene_depart_init / jmpc_scene_enter /
jmpc_scene_presence / jmpc_episode_outcomes_scene in include/jmpc.h).  This module extends oracle/scene_exchange.py
and oracle/episode_outcomes.py, which describe scenes whose vehicles are all present from evaluation 0, without
changing them:
  * vehicle_rows / mate_rows: a vehicle with depart d and n executed steps (History rows d .. d + n - 1, global
    iteration indices) presents its parked start pose at e < d, its start row at e = d, History row e - 1 up to
    e = d + n, and is parked from d + n + 1 on.  depart = 0 is scene_exchange.vehicle_rows.
  * presence: which vehicles a mate sees at all at each evaluation.
  * episode_outcomes: the outcome record of one vehicle whose record starts at evaluation `first`, with NaN track rows
    for absent obstacles (they add no clearance and no contact).
"""
from __future__ import annotations

import math

import numpy as np

from .collision_oracle import CarGeometry
from .episode_outcomes import clearance_and_contact
from .episode_outcomes import episode_outcomes as _outcomes_all_present
from .scene_exchange import NEVER_STEPPED

ON_GOAL = ("park", "leave")


def vehicle_rows(state0, history, steps, done, max_steer, n_eval: int, depart=None) -> np.ndarray:
    """state0 [B, 4] x, y, v, yaw; history [R, B, 8] (x, y, yaw, v, t, delta, a, xref_dev); steps, done [B];
    max_steer scalar or [B]; depart [B] entry iterations or None (all 0).  Returns [n_eval, B, 6]: the row every
    vehicle presents to its mates at evaluations 0 .. n_eval - 1."""
    state0 = np.asarray(state0, np.float64)
    history = np.asarray(history, np.float64)
    steps, done = np.asarray(steps, np.int64), np.asarray(done, np.int64)
    B = len(state0)
    depart = np.zeros(B, np.int64) if depart is None else np.asarray(depart, np.int64)
    max_steer = np.broadcast_to(np.asarray(max_steer, np.float64), (B,))
    if history.ndim != 3 or history.shape[1:] != (B, 8):
        raise ValueError(f"history must be [rows, {B}, 8]")
    if (depart + steps > len(history)).any():
        raise ValueError("history holds fewer rows than a vehicle executed steps")
    cols = lambda h: np.stack([h[..., 0], h[..., 1], h[..., 3], h[..., 2]], axis=-1)   # noqa: E731  x, y, v, yaw
    bs = np.arange(B)
    last = np.where((steps == 0)[:, None], state0,
                    cols(history[np.maximum(depart + steps - 1, 0), bs]) if len(history) else state0)
    parked_from = np.where(np.isin(done, NEVER_STEPPED), 0, depart + steps + 1)
    start = np.concatenate([state0, np.zeros((B, 2))], axis=1)
    waiting = np.concatenate([state0[:, :2], np.zeros((B, 1)), state0[:, 3:4], np.zeros((B, 2))], axis=1)
    parked = np.concatenate([last[:, :2], np.zeros((B, 1)), last[:, 3:4], np.zeros((B, 2))], axis=1)
    out = np.empty((n_eval, B, 6))
    for e in range(n_eval):
        if e == 0:
            row = start
        else:
            h = history[min(e - 1, len(history) - 1)] if len(history) else np.full((B, 8), np.nan)
            steer = np.maximum(np.minimum(h[:, 5], max_steer), -max_steer)
            row = np.concatenate([cols(h), h[:, 6:7], steer[:, None]], axis=1)
            row = np.where((e == depart)[:, None], start, row)
        row = np.where((e >= parked_from)[:, None], parked, row)
        out[e] = np.where((e < depart)[:, None], waiting, row)
    return out


def _mates(B: int, k: int):
    if k < 1 or B % k:
        raise ValueError(f"B = {B} is not a multiple of k = {k}")
    for b in range(B):
        s, j = divmod(b, k)
        yield b, [s * k + m for m in range(k) if m != j]


def mate_rows(state0, history, steps, done, max_steer, k: int, n_eval: int, depart=None) -> np.ndarray:
    """[n_eval, B, k - 1, 6]: the scene-mate slots of every episode at evaluations 0 .. n_eval - 1."""
    rows = vehicle_rows(state0, history, steps, done, max_steer, n_eval, depart)
    out = np.empty((n_eval, rows.shape[1], k - 1, 6))
    for b, mates in _mates(rows.shape[1], k):
        out[:, b] = rows[:, mates]
    return out


def presence(depart, steps, done, on_goal: str, n_eval: int) -> np.ndarray:
    """[n_eval, B] bool: vehicle m is present at evaluation e iff depart[m] <= e and not (on_goal == "leave",
    done[m] == 1 and e > depart[m] + steps[m]).  A goal test that fires at the top of iteration g = depart + steps sees
    the state of evaluation g, so the vehicle is still present there.  (A vehicle of a scene that is not driven,
    done 3 / 4, never waits on the device; no vehicle of such a scene is measured, so its presence is never read.)"""
    if on_goal not in ON_GOAL:
        raise ValueError(f"unknown on_goal {on_goal!r}")
    depart, steps, done = (np.asarray(a, np.int64) for a in (depart, steps, done))
    e = np.arange(n_eval)[:, None]
    gone = (on_goal == "leave") & (done == 1)[None, :] & (e > (depart + steps)[None, :])
    return (depart[None, :] <= e) & ~gone


def presence_masks(present, k: int) -> np.ndarray:
    """present [B] bool (one instant) -> [B] int32 masks: bit s of mask[b] cleared for every absent mate in slot s
    (jmpc_scene_presence with combine = 0)."""
    present = np.asarray(present, bool)
    out = np.full(len(present), -1, np.int64)
    for b, mates in _mates(len(present), k):
        for slot, m in enumerate(mates):
            if not present[m]:
                out[b] &= ~(1 << slot)
    return out.astype(np.int32)


def episode_outcomes(state0, history, flags, track, dt: float, L: float, max_steer: float,
                     geo: CarGeometry = CarGeometry(), first: int = 0) -> dict:
    """state0 [4] x, y, v, yaw; history [n, 8] the vehicle's executed steps; flags [n]; track [n + 1, n_obs, 6] with
    NaN rows for absent obstacles; first: the global index of the record's first evaluation (the *_eval columns add
    it).  Returns a dict of the public columns of enum jmpc_outcome (python floats / ints)."""
    history = np.asarray(history, np.float64).reshape(-1, 8)
    track = np.asarray(track, np.float64)
    if track.ndim != 3 or track.shape[0] != len(history) + 1:
        raise ValueError(f"track must be [{len(history) + 1}, n_obs, 6]")
    # the step columns do not depend on the obstacles
    out = _outcomes_all_present(state0, history, flags, np.zeros((len(history) + 1, 0, 6)), dt, L, max_steer, geo)
    if track.shape[1] == 0:
        return out
    poses = np.vstack([[[float(state0[0]), float(state0[1]), float(state0[3])]], history[:, :3]])
    clear, hit = clearance_and_contact(poses, track, geo)
    absent = np.isnan(track[:, :, 0])
    clear[absent], hit[absent] = math.inf, False
    flat = clear.reshape(-1)
    j = int(np.argmin(flat))                             # first occurrence: earliest evaluation, then lowest obstacle
    if flat[j] < math.inf:
        out.update(min_clearance=float(flat[j]), min_clearance_eval=first + j // clear.shape[1],
                   min_clearance_obs=j % clear.shape[1])
    any_hit = hit.any(axis=1)
    out["contact_evals"] = int(any_hit.sum())
    if any_hit.any():
        e = int(np.argmax(any_hit))
        out.update(first_contact_eval=first + e, first_contact_obs=int(np.argmax(hit[e])))
    return out
