"""Planned scenarios from scene to goal on the device: main/scenarios/mpc_intersection.py:27-163 for a batch.

The reference script plans a course with MotionPrimitiveSearch (:63-66), derives dl from its first segment (:73), builds
an MPC on it (yaw smoothed in place, mpc.py:260), starts the ego at trajectory_full[0] with v = 0 (:76-79) and runs the
closed loop against its scripted obstacles (:99-163).  `run_planned_scenarios` does the same for many (scene, start,
goal, weights) at once: the searches, the course ingestion and the loop all run in libjmpc.so kernels and the planned
courses never leave the GPU.
"""
from __future__ import annotations

from typing import Optional, Sequence

from .batched import BatchedMPC
from .config import MPCConfig
from .episodes import BatchedEpisodes, scripted_obstacles
from .planner import BatchedPlanner


def run_planned_scenarios(scenes: Sequence[Sequence], start, goal_point, goal_area, allowed_dtheta, scene_id=None,
                          weights=None, obstacles: Optional[Sequence[Sequence[dict]]] = None, frame_window: int = 10,
                          T: Optional[int] = None, config: Optional[MPCConfig] = None, dt: float = 0.2,
                          max_steps: int = 256, max_expansions: int = 4096, max_path: int = 48,
                          max_N: Optional[int] = None, planner: Optional[BatchedPlanner] = None, device: int = 0,
                          outcomes: bool = False, record_history: bool = True, agents_per_scene: int = 1,
                          share_plans: bool = False, right_of_way=None, priority=None, junction=None) -> dict:
    """One episode per search.  scenes / start / goal_point / goal_area / allowed_dtheta / scene_id / weights as in
    `BatchedPlanner.plan`; obstacles: per episode a list of the reference's scripted-obstacle dicts (see
    `episodes.scripted_obstacles`), or None for an empty road; frame_window: FRAME_WINDOW of the script (10 for the
    intersection, 20 for the roundabout).  Returns `BatchedEpisodes.run`'s dict (steps, done -- 3 where the search
    found no course --, state, history, flags, plan_status, plan_cost, expansions) plus the episodes' `dl` and
    `margin`.  outcomes=True adds the per-episode outcome record (`BatchedEpisodes(outcomes=True)`); with
    record_history=False no History is kept on the device at all, which is what a large study wants.

    agents_per_scene = k > 1: searches [s k, (s + 1) k) are the k MPC-driven vehicles of scene s, which see each other
    as moving obstacles (`BatchedEpisodes(agents_per_scene=k)`); `obstacles` is then given per scene (len = B / k) and
    replicated to its vehicles.  A scene with a failed search is not driven: that vehicle gets done = 3, its mates
    done = 4.  share_plans=True: the vehicles of a scene predict each other along their MPC plans
    (`BatchedEpisodes(share_plans=True)`).  right_of_way / priority / junction: a rule that decides which mates each
    vehicle yields to (`BatchedEpisodes(right_of_way=...)`); priority per search, junction once or per scene."""
    import torch
    k = int(agents_per_scene)
    if obstacles is not None and k > 1:
        if len(start) % k or len(obstacles) != len(start) // k:
            raise ValueError(f"with agents_per_scene = {k}, obstacles must hold one list per scene ({len(start)} // {k})")
        obstacles = [specs for specs in obstacles for _ in range(k)]
    planner = planner or BatchedPlanner(device=device)
    plans = planner.plan_device(start, goal_point, goal_area, allowed_dtheta, scenes, scene_id=scene_id, weights=weights,
                                max_expansions=max_expansions, max_path=max_path)
    engine = BatchedMPC.from_plans(plans, T=T, config=config, dt=dt, max_N=max_N, max_batch=len(plans), device=device)
    try:
        program = None if obstacles is None else scripted_obstacles(obstacles)
        ep = BatchedEpisodes.from_plans(engine, plans, obstacle_program=program, frame_window=frame_window,
                                        max_steps=max_steps, record_history=record_history, outcomes=outcomes,
                                        agents_per_scene=k, share_plans=share_plans, right_of_way=right_of_way,
                                        priority=priority, junction=junction)
        res = ep.run(max_steps=max_steps)
        res.update(dl=engine.course_dl.cpu().numpy(), margin=ep.margin)
        torch.cuda.synchronize(engine.device)
        return res
    finally:
        engine.close()
