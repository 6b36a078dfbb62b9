"""Numpy restatement of fixed-time traffic signals (TEST INFRASTRUCTURE ONLY, see oracle/__init__.py).

BatchedEpisodes(signals=SignalPlan(...)): a red light is one more course cut at the stop line, decided once per red
phase and owner (jmpc_signals in include/jmpc.h).  This module adds to the oracle without changing any other module:
  * green: whether a signal group is green in a loop iteration of a scene;
  * signal_pass: the pass on a snapshot of its inputs, taken where it runs (after the collision check, before the
    step), returning what it writes.
The stopping test is evaluated left to right with every product rounded once, as the kernel does without fused
multiply-adds, so the two agree bit for bit.
"""
from __future__ import annotations

import numpy as np

RUNNING = 0


def green(i, group, offset, cycle: int, green_start, green_len):
    """Whether `group` is green in loop iteration i of a scene with `offset`: ((i + offset - green_start[g]) mod C) <
    green_len[g] with the non-negative modulus.  group, offset and i broadcast; group must be in [0, G)."""
    group = np.asarray(group, np.int64)
    start, length = np.asarray(green_start, np.int64), np.asarray(green_len, np.int64)
    phase = np.mod(np.asarray(i, np.int64) + np.asarray(offset, np.int64) - start[group], int(cycle))
    return phase < length[group]


def signal_pass(snap: dict):
    """One signal pass on a snapshot.  snap keys:
      iteration, cycle, green_start [G], green_len [G], margin, stop_decel, k, offset [B / k] or None;
      owner [B] or None (owner = b), group [n_owner], zone [n_owner, 2];
      course_id [B], course_n [n_courses], agent_idx [B], state [B, 4], dl [B], done [B], checked (bool);
      course_len [B], latch [B, 2], hold_steps [n_owner], go [n_owner] as they are before the pass.
    Returns (course_len, latch, hold_steps, go) after the pass, as new arrays."""
    B = len(snap["done"])
    course_len = np.array(snap["course_len"], np.int64)
    latch = np.array(snap["latch"], np.int64).reshape(B, 2)
    hold_steps, go = np.array(snap["hold_steps"], np.int64), np.array(snap["go"], np.int64)
    run = np.asarray(snap["done"]) == RUNNING
    b = np.arange(B)
    if not snap["checked"]:
        full = np.asarray(snap["course_n"], np.int64)[np.asarray(snap["course_id"], np.int64)]
        course_len[run] = full[run]
    owner = b if snap["owner"] is None else np.asarray(snap["owner"], np.int64)
    o = np.where(run, owner, 0)
    g = np.asarray(snap["group"], np.int64)[o]
    e = np.asarray(snap["zone"], np.int64).reshape(-1, 2)[o, 0]
    G = len(snap["green_start"])
    signalised = run & (g >= 0) & (g < G) & (e >= 0)
    k = int(snap["k"])
    offset = np.zeros(B, np.int64) if snap["offset"] is None else np.asarray(snap["offset"], np.int64)[b // k]
    red = signalised.copy()
    red[signalised] = ~green(int(snap["iteration"]), g[signalised], offset[signalised], snap["cycle"],
                             snap["green_start"], snap["green_len"])
    clear = run & ~red
    latch[clear] = (-1, 0)
    a = np.asarray(snap["agent_idx"], np.int64)
    L = e - int(snap["margin"])
    known = red & (latch[:, 0] == o)
    decide = red & ~known
    v = np.asarray(snap["state"], np.float64).reshape(B, 4)[:, 2]
    reach = 2.0 * float(snap["stop_decel"]) * (L - 1 - a).astype(np.float64) * np.asarray(snap["dl"], np.float64)
    fresh = (a < L) & (v * v <= reach)
    hold = np.where(known, latch[:, 1] == 1, fresh) & red
    latch[decide, 0] = o[decide]
    latch[decide, 1] = fresh[decide]
    passed = decide & ~fresh & (a < L)
    np.add.at(go, o[passed], 1)
    course_len[hold] = np.minimum(course_len[hold], np.maximum(a[hold] + 1, L[hold]))
    np.add.at(hold_steps, o[hold], 1)
    return course_len, latch, hold_steps, go
