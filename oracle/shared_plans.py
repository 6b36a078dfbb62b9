"""Numpy restatement of shared plans (TEST INFRASTRUCTURE ONLY, see oracle/__init__.py).

Scene mates predicted along their own MPC plans (jmpc_scene_plans / jmpc_collision_planned in include/jmpc.h):
  * predict_obstacle_plan: collision_oracle.predict_obstacle fed a sequence of (a, steer) inputs;
  * collision_cut: collision_oracle.collision_cut with an optional input sequence per obstacle;
  * mate_plans: the inputs that predict every mate slot at one evaluation, from a snapshot of the warm-start arrays
    and the obstacle rows of that evaluation.
"""
from __future__ import annotations

import math
from typing import Sequence, Tuple

import numpy as np

from .collision_oracle import CarGeometry, check_collision, cut_index, ego_prediction, predict_obstacle


def predict_obstacle_plan(x, y, v, yaw, inputs, dt: float, L: float, horizon: float = 7.0) -> np.ndarray:
    """predict_obstacle fed a sequence of inputs: step k uses inputs[min(k, len(inputs) - 1)] = (a, steer), so past
    the plan the last input is held.  With every input equal this is predict_obstacle, bit for bit."""
    inputs = [(float(a), float(s)) for a, s in inputs]
    if not inputs:
        raise ValueError("a plan needs at least one input")
    n = len(np.arange(0, horizon, dt))
    out = np.zeros((n, 4))
    for k in range(n):
        a, steer = inputs[min(k, len(inputs) - 1)]
        x += v * math.cos(yaw) * dt
        y += v * math.sin(yaw) * dt
        v += a * dt
        yaw += (v / L) * math.tan(steer) * dt
        out[k] = (x, y, yaw, k * dt)
    return out


def collision_cut(geo: CarGeometry, path_full: np.ndarray, agent_idx: int, v: float,
                  obstacles: Sequence[Sequence[float]], dt: float, frame_window: int, max_accel: float,
                  max_speed: float, margin: int, horizon: float = 7.0, plans=None) -> Tuple[bool, int]:
    """collision_oracle.collision_cut where obstacle i is predicted from plans[i], a sequence of (a, steer) inputs
    (predict_obstacle_plan), instead of its row's constant input; plans None, or an entry None, keeps the row's."""
    plans = [None] * len(obstacles) if plans is None else list(plans)
    if len(plans) != len(obstacles):
        raise ValueError("plans needs one entry (or None) per obstacle")
    path = path_full[agent_idx:]
    ego = ego_prediction(path, v, dt, max_accel, max_speed)
    preds = [predict_obstacle(*o, dt=dt, L=geo.L, horizon=horizon) if p is None else
             predict_obstacle_plan(*o[:4], p, dt=dt, L=geo.L, horizon=horizon) for o, p in zip(obstacles, plans)]
    hit = check_collision(geo, ego, path, preds, frame_window)
    if hit is None:
        return False, len(path_full)
    k = cut_index(path_full, hit[0], hit[1]) - margin
    return True, max(agent_idx + 1, k)


def mate_plans(oa, od, warm, done, rows, max_steer, k: int) -> np.ndarray:
    """oa, od [B, T]: every vehicle's last plan (oa / od after its last solve); warm, done [B]; rows [B, n_obs, 6]: the
    obstacle rows of the same evaluation (slots 0 .. k - 2 the mates); max_steer scalar or [B].  Returns
    [B, k - 1, T - 1, 2]: for mate m and step t, (oa[m, t + 1], clip(od[m, t + 1], +-max_steer[m])) when m is running
    (done = 0) with a warm start (warm != 0), else its row's (a, steer) repeated."""
    oa, od = np.asarray(oa, np.float64), np.asarray(od, np.float64)
    warm, done = np.asarray(warm, np.int64), np.asarray(done, np.int64)
    rows = np.asarray(rows, np.float64)
    B, T = oa.shape
    if k < 2 or B % k or T < 2 or rows.shape[:1] != (B,) or rows.shape[1] < k - 1:
        raise ValueError(f"need k >= 2 dividing B = {B}, T >= 2 and rows [B, >= k - 1, 6]")
    max_steer = np.broadcast_to(np.asarray(max_steer, np.float64), (B,))
    out = np.empty((B, k - 1, T - 1, 2))
    for b in range(B):
        s, j = divmod(b, k)
        for slot, m in enumerate(s * k + q for q in range(k) if q != j):
            if done[m] == 0 and warm[m] != 0:
                out[b, slot, :, 0] = oa[m, 1:]
                out[b, slot, :, 1] = np.maximum(np.minimum(od[m, 1:], max_steer[m]), -max_steer[m])
            else:
                out[b, slot, :, :] = rows[b, slot, 4:6]
    return out
