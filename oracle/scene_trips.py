"""Numpy restatement of trips through scene slots (TEST INFRASTRUCTURE ONLY, see oracle/__init__.py).

BatchedEpisodes.from_trips: scenes of k slots fed from a stream of timed trips (jmpc_scene_trips /
jmpc_scene_trips_finish in include/jmpc.h).  This module extends oracle/scene_lifetimes.py without changing it:
  * trips_pass: the close / admit / load decision of one pass on a snapshot, with the clearance arithmetic of
    oracle/episode_outcomes.clearance_and_contact;
  * presence: which slots hold a trip at each evaluation (and at each collision check), from the trip table;
  * trip_outcomes: a trip's outcome record, scene_lifetimes.episode_outcomes on its slot's rows of its window.
Trip indices here are positions in the scene-sorted layout the pass walks (scene, then arrival, then trip index).
"""
from __future__ import annotations

import numpy as np

from .collision_oracle import CarGeometry
from .episode_outcomes import clearance_and_contact
from .scene_lifetimes import episode_outcomes

WAITING, GOAL, NO_COURSE = 5, 1, 3
PENDING, IN_SLOT, CLOSED = 0, 1, 2


def start_clearance(p, q, geo: CarGeometry = CarGeometry()) -> float:
    """Clearance of two poses p, q (x, y, v, yaw): min over the 4 circle pairs of dist - 2r."""
    clear, _ = clearance_and_contact(np.array([[p[0], p[1], p[3]]], np.float64),
                                     np.asarray(q, np.float64)[None, None, :4], geo)
    return float(clear[0, 0])


def trips_pass(done, state, slot_trip, phase, scene_start, arrival, usable, start, k: int, iteration: int,
               initial: bool = False, entry_gap: float = 2.0, geo: CarGeometry = CarGeometry()) -> dict:
    """One trips pass on a snapshot taken where the pass runs in loop iteration `iteration` (initial: before
    evaluation 0).  done, state [B] / [B, 4] and slot_trip [B] of the slots; phase [N] (0 pending, 1 in a slot, 2 closed),
    scene_start [S + 1], arrival, usable [N], start [N, 4] of the trips.  Returns the decisions and the state after the
    pass: closed [(trip, slot)], no_course [trip], admitted [(trip, slot)], slot_waits [trip], blocked_waits [trip],
    entry, and done / slot_trip / phase updated (a loaded slot's state is its trip's start)."""
    done, state = np.array(done, np.int64), np.array(state, np.float64)
    slot_trip, phase = np.array(slot_trip, np.int64), np.array(phase, np.int64)
    start = np.asarray(start, np.float64)
    entry = 0 if initial else iteration + 1
    out = dict(closed=[], no_course=[], admitted=[], slot_waits=[], blocked_waits=[], entry=entry)
    for s in range(len(scene_start) - 1):
        b0 = s * k
        for b in range(b0, b0 + k):
            if done[b] == GOAL:
                out["closed"].append((int(slot_trip[b]), b))
                phase[slot_trip[b]] = CLOSED
                slot_trip[b], done[b] = -1, WAITING
        empty = [b for b in range(b0, b0 + k) if done[b] == WAITING]
        waiting = []                                        # earlier pending trips of this walk
        for t in range(scene_start[s], scene_start[s + 1]):
            if arrival[t] > entry:
                break
            if phase[t] != PENDING:
                continue
            if not usable[t]:
                out["no_course"].append(t)
                phase[t] = CLOSED
                continue
            if not empty:
                out["slot_waits"].append(t)
                waiting.append(t)
                continue
            others = [state[b] for b in range(b0, b0 + k) if done[b] != WAITING] + [start[u] for u in waiting]
            if any(start_clearance(start[t], q, geo) < entry_gap for q in others):
                out["blocked_waits"].append(t)
                waiting.append(t)
                continue
            b = empty.pop(0)
            out["admitted"].append((t, b))
            state[b], done[b], slot_trip[b], phase[t] = start[t], 0, t, IN_SLOT
    out.update(done=done, state=state, slot_trip=slot_trip, phase=phase)
    return out


def presence(slot, entry, exit, B: int, n: int, collision: bool = False) -> np.ndarray:
    """[n, B] bool from the trip table (slot, entry, exit [N]): slot b holds a trip at evaluation e iff some trip of b
    has entry <= e <= exit (a trip whose goal test fired at the top of iteration exit is still present in evaluation
    exit); with collision=True at the collision check of iteration e: entry <= e < exit."""
    out = np.zeros((n, B), bool)
    e = np.arange(n)
    for b, a, x in zip(slot, entry, exit):
        if b < 0:
            continue
        out[:, b] |= (e >= a) & ((e < x) if collision else (e <= x))
    return out


def trip_outcomes(start, history, flags, obstacle_history, slot: int, entry: int, steps: int, dt: float, L: float,
                  max_steer: float, geo: CarGeometry = CarGeometry()) -> dict:
    """The outcome record of a trip that entered slot `slot` at evaluation `entry` and executed `steps` steps: its
    slot's History / flags rows entry .. entry + steps - 1 and obstacle_history rows entry .. entry + steps (NaN rows
    for absent mates)."""
    h = history[entry:entry + steps, slot]
    f = flags[entry:entry + steps, slot]
    track = obstacle_history[entry:entry + steps + 1, slot]
    return episode_outcomes(start, h, f, track, dt=dt, L=L, max_steer=max_steer, geo=geo, first=entry)
