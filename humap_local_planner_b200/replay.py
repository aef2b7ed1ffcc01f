"""Closed-loop replay harness (BASELINE.json config 5): consecutive planning cycles with moving people and the
init -> move -> adjust -> stop state sequence, measuring the latency of the planning cycle through the C ABI.

Only what SURVEY.md Appendix F lists is restated, minimally and without ROS: the state sequence of
`PlannerState` (src/planner_state.cpp:43-210) driven by three predicates (position reached within
0.65 * xy_goal_tolerance, goal reached incl. yaw tolerance, pointing towards the goal within 30 deg), rotation in
place for INIT / ADJUST (LatchedStopRotateController, src/latched_stop_rotate_controller.cpp:203-287, reduced to an
acceleration-limited proportional turn), the command integration `computeNextPoseBaseVel`
(src/utils/transformations.cpp:16-30) and constant-velocity people. Recovery predicates are stubbed false (no obstacle
is placed inside the footprint), the yield-way / group-intrusion detectors are not modelled. The MOVE state is the
only one that enters the hot path (src/humap_planner.cpp:390).
"""
from __future__ import annotations

import math
import time
from dataclasses import dataclass, field
from typing import List, Optional

import numpy as np

from . import config, scenes
from .capi import HmpObstacle, HmpPerson, HmpResult, HmpWorld, Planner

XY_TOL, YAW_TOL = 0.1, 0.2     # src/humap_config_ros.cpp:63-64


@dataclass
class ReplayLog:
    states: List[str] = field(default_factory=list)
    plan_ms: List[float] = field(default_factory=list)       # wall time of the full C-ABI cycle (MOVE cycles)
    gpu_ms: List[float] = field(default_factory=list)
    best: List[int] = field(default_factory=list)
    poses: List[tuple] = field(default_factory=list)
    goals_reached: int = 0
    recoveries: int = 0                                       # cycles without a valid trajectory (the host backs off)
    escalated: int = 0                                        # plans redone as an exact FP64 sweep (hmp_set_escalation)
    parity_checked: int = 0
    parity_mismatch: int = 0
    last_result: Optional[HmpResult] = None                   # HmpResult of the last MOVE cycle


def _wrap(a):
    return math.atan2(math.sin(a), math.cos(a))


def run_replay(planner: Planner, n_cycles: int = 1000, period: float = 0.05, seed: int = 0, cfg_name: str = "cfg0",
               sampling_axes: Optional[dict] = None, on_plan=None, on_plan_every: int = 0,
               device_mapgrids: bool = True) -> ReplayLog:
    """`on_plan(params, scene, sampling, result) -> bool` (optional) is called on every `on_plan_every`-th MOVE cycle with
    a `capi.Scene` of that cycle's inputs; tests use it to compare the selection with their checker. It returns True
    when the selection is accepted."""
    cfg = scenes.CONFIGS[cfg_name]
    base = scenes.make_scene(cfg, seed)
    params = scenes.make_params(cfg)
    params.general.sim_period = period
    smp = config.make_sampling(sampling_axes if sampling_axes is not None else cfg.sampling)
    planner.set_params(params)
    planner.set_costmap(base.cells, base.origin_x, base.origin_y, base.resolution)
    planner.set_footprint(base.footprint)
    rng = np.random.default_rng(seed + 1000)
    n_static = base.world.n_obstacles - base.world.n_people
    static_obs = [base.world.obstacles[i] for i in range(n_static)]
    people = [[base.world.people[i].x, base.world.people[i].y, base.world.people[i].vx, base.world.people[i].vy,
               base.world.people[i].cov_xx] for i in range(base.world.n_people)]
    r_robot, r_person = config.ROBOT_INSCRIBED_RADIUS, config.PERSON_MODEL_RADIUS
    L = params.limits
    x, y, th = 0.0, 0.0, 0.0
    vx, vth = 0.0, 0.0
    goals = [(3.0, 0.0, 0.0), (0.0, 0.0, math.pi)]     # shuttle inside the free corridor of the scene
    gi = 0
    state = "init"
    log = ReplayLog()
    # highest_valid_cost_ of the MapGrid critics: prepare() of cycle k + 1 moves cycle k's value into highest_valid_cost_prev_
    # (src/map_grid_cost_function.cpp:76-77), which the unreachable-cell heuristic returns (:135-138)
    hv_prev = [0.0, 0.0, 0.0, 0.0]
    for cyc in range(n_cycles):
        gx, gy, gyaw = goals[gi]
        dist = math.hypot(gx - x, gy - y)
        head_err = _wrap(math.atan2(gy - y, gx - x) - th)
        # ---- PlannerState::update (reduced) ------------------------------------------------------------------
        if state == "init" and abs(head_err) <= math.radians(30.0):
            state = "move"
        elif state == "move" and dist <= 0.65 * XY_TOL:
            state = "adjust"
        elif state == "adjust" and abs(_wrap(gyaw - th)) <= YAW_TOL and abs(vx) < 0.01 and abs(vth) < 0.01:
            state = "stop"
        elif state == "stop":
            gi = (gi + 1) % len(goals)
            log.goals_reached += 1
            state = "init"
        log.states.append(state)
        cmd_x, cmd_th = 0.0, 0.0
        if state == "move":
            # ---- environment model for this cycle (createEnvironmentModel, reduced to points + circles) --------
            obs = []
            for o in static_obs:
                d = math.hypot(o.obj_x - x, o.obj_y - y)
                h = HmpObstacle()
                h.robot_x, h.robot_y, h.robot_yaw = x + r_robot * (o.obj_x - x) / d, y + r_robot * (o.obj_y - y) / d, th
                h.obj_x, h.obj_y = o.obj_x, o.obj_y
                obs.append(h)
            ppl = []
            for p in people:
                d = max(math.hypot(p[0] - x, p[1] - y), 1e-6)
                ux, uy = (p[0] - x) / d, (p[1] - y) / d
                h = HmpObstacle()
                h.robot_x, h.robot_y, h.robot_yaw = x + r_robot * ux, y + r_robot * uy, th
                h.obj_x, h.obj_y = p[0] - r_person * ux, p[1] - r_person * uy
                h.vx, h.vy, h.force_dynamic = p[2], p[3], 1
                obs.append(h)
                q = HmpPerson()
                q.x, q.y, q.vx, q.vy = p[0], p[1], p[2], p[3]
                q.yaw = math.atan2(p[3], p[2])
                q.cov_xx = q.cov_yy = p[4]
                ppl.append(q)
            w = HmpWorld()
            w.robot_x, w.robot_y, w.robot_yaw = x, y, th
            w.vel_x, w.vel_th = vx, vth
            lg = min(dist, 2.5)
            w.goal_local_x, w.goal_local_y = x + lg * (gx - x) / max(dist, 1e-9), y + lg * (gy - y) / max(dist, 1e-9)
            w.goal_x, w.goal_y, w.goal_yaw = gx, gy, gyaw
            oa = (HmpObstacle * max(1, len(obs)))(*obs)
            pa = (HmpPerson * max(1, len(ppl)))(*ppl)
            w.obstacles, w.people, w.n_obstacles, w.n_people, w.n_groups = oa, pa, len(obs), len(ppl), 0
            plan = np.array([[x + s * (w.goal_local_x - x) / max(lg, 1e-9), y + s * (w.goal_local_y - y) / max(lg, 1e-9)]
                             for s in np.arange(0.0, lg + 1e-9, 0.1)] + [[w.goal_local_x, w.goal_local_y]])
            fwd = min(0.325, lg)
            front = plan[: max(1, int(fwd / 0.1) + 1)]
            t0 = time.perf_counter()
            planner.set_costmap(base.cells, base.origin_x, base.origin_y, base.resolution)
            grids = None
            if device_mapgrids:
                planner.compute_mapgrid(0, plan, False, hv_prev[0])
                planner.compute_mapgrid(1, plan, True, hv_prev[1])
                planner.compute_mapgrid(2, plan, False, hv_prev[2])
                planner.compute_mapgrid(3, front, True, hv_prev[3])
            else:
                grids = [scenes.mapgrid_wavefront(base.cells, base.origin_x, base.origin_y, base.resolution, pl_, lg_)
                         for pl_, lg_ in ((plan, False), (plan, True), (plan, False), (front, True))]
                for g in range(4):
                    planner.set_mapgrid(g, grids[g], hv_prev[g])
            planner.set_footprint(base.footprint)
            res, _ = planner.plan(w, smp, want_poses=False)
            log.plan_ms.append(1e3 * (time.perf_counter() - t0))
            log.gpu_ms.append(res.gpu_ms)
            log.best.append(res.best_index)
            log.last_result = res
            if hasattr(planner, "last_escalated") and planner.last_escalated() == 1:
                log.escalated += 1
            if res.status == 0:
                cmd_x, cmd_th = res.xv, res.thetav
            else:
                # no valid trajectory: what RecoveryManager does on the host in the reference (src/recovery_manager.cpp) is out
                # of scope here; the harness backs off along the heading at min_vel_x and turns slowly until a plan exists again
                log.recoveries += 1
                cmd_x = max(min(L.min_vel_x, 0.0), vx - L.acc_lim_x * period) if L.min_vel_x < 0 else 0.0
                cmd_th = min(L.min_vel_theta, vth + L.acc_lim_theta * period)
            if on_plan is not None and on_plan_every and (on_plan_every == 1 or len(log.plan_ms) % on_plan_every == 1):
                if grids is None:
                    grids = [planner.get_mapgrid(g, base.cells.shape) for g in range(4)]
                from .capi import Scene
                sc = Scene(w, oa, pa, None, base.cells, base.origin_x, base.origin_y, base.resolution, grids, base.footprint,
                           tuple(hv_prev))
                log.parity_checked += 1
                if not on_plan(params, sc, smp, res):
                    log.parity_mismatch += 1
            hv_prev = [float(v) for v in res.highest_valid_cost]
        elif state in ("init", "adjust"):
            err = head_err if state == "init" else _wrap(gyaw - th)
            want = math.copysign(min(max(abs(err), L.min_vel_theta), L.max_vel_theta), err)
            want = math.copysign(min(abs(want), math.sqrt(2.0 * L.acc_lim_theta * abs(err))), err)
            if state == "adjust" and abs(err) <= 0.5 * YAW_TOL:
                want = 0.0     # inside the yaw tolerance: stop rotating (LatchedStopRotateController::isGoalReached)
            cmd_th = min(max(want, vth - L.acc_lim_theta * period), vth + L.acc_lim_theta * period)
            cmd_x = max(vx - L.acc_lim_x * period, 0.0)
        # ---- apply the command for one period (computeNextPoseBaseVel), move the people ----------------------------
        x += cmd_x * math.cos(th) * period
        y += cmd_x * math.sin(th) * period
        th = _wrap(th + cmd_th * period)
        vx, vth = cmd_x, cmd_th
        for p in people:
            p[0] += p[2] * period
            p[1] += p[3] * period
            if math.hypot(p[0], p[1]) > 5.5:     # keep the crowd inside the window: re-enter from the opposite side
                p[0], p[1] = -p[0] * 0.9, -p[1] * 0.9
        log.poses.append((x, y, th))
    return log


def summarize(log: ReplayLog) -> dict:
    ms = np.array(log.plan_ms) if log.plan_ms else np.zeros(1)
    g = np.array(log.gpu_ms) if log.gpu_ms else np.zeros(1)
    seq = [s for i, s in enumerate(log.states) if i == 0 or s != log.states[i - 1]]
    return {"cycles": len(log.states), "move_cycles": len(log.plan_ms), "goals_reached": log.goals_reached,
            "p50_cycle_ms": float(np.percentile(ms, 50)), "p99_cycle_ms": float(np.percentile(ms, 99)),
            "p50_gpu_ms": float(np.percentile(g, 50)), "p99_gpu_ms": float(np.percentile(g, 99)),
            "state_sequence_head": seq[:12], "parity_checked": log.parity_checked, "parity_mismatch": log.parity_mismatch,
            "escalated_plans": log.escalated,
            "recoveries": log.recoveries}


def bench_line(args, rank, local_rank, world, barrier, dump: Optional[dict] = None) -> Optional[dict]:
    """`bench.py --cfg cfg4`: BASELINE config 5 -- consecutive 20 Hz planning cycles with moving people and the
    init -> move -> adjust -> stop sequence; p50 / p99 latency of the full C-ABI cycle (costmap upload, four device wave
    fronts, footprint, plan in the configured precision mode, result read back) for the stock sampling (72 candidates) and
    for the 64k-candidate grid. --steps = cycles per run. One process per GPU runs the same replay. A dict passed as
    `dump` receives the 64k replay's outputs: the last plan's HmpResult, the winner of every MOVE cycle, the robot poses."""
    cycles = args.steps
    pl = Planner(local_rank)
    pl.set_precision(int(args.precise))
    pl.set_sweep_layout(int(args.layout))
    run_replay(pl, n_cycles=60)   # warm-up (allocations, module load)
    barrier()
    l0 = pl.launch_count()
    small = summarize(run_replay(pl, cycles))
    big_log = run_replay(pl, cycles, sampling_axes=config.SAMPLING_64K)
    big = summarize(big_log)
    launches = pl.launch_count() - l0
    if dump is not None:
        dump["replay_last_result"] = big_log.last_result
        dump["replay_best_index"] = np.array(big_log.best, dtype=np.float64)
        dump["replay_robot_poses"] = np.array(big_log.poses, dtype=np.float64).reshape(-1, 3)
    barrier()
    pl.close()
    if rank != 0:
        return None
    return {
        "metric": "p50 planning-cycle latency at 64k candidates (closed-loop replay)", "value": big["p50_cycle_ms"], "unit": "ms",
        "n_gpus": world, "steps": cycles, "warmup": 60, "ms_per_step": big["p50_cycle_ms"], "higher_is_better": False, "scaling": "weak",
        "vs_baseline": None, "dtype": {0: "f32", 1: "f64", 2: "f32 sweep + f64 refinement of the leaders"}[int(args.precise)],
        "data": "synthetic",
        "config": {"workload": f"closed-loop replay (BASELINE config 5): {cycles} consecutive 20 Hz cycles, cfg0 world (4 moving people, 30 obstacle "
                               "points), states init -> move -> adjust -> stop, full C-ABI cycle per MOVE cycle",
                   "timing": "wall clock of the C-ABI calls of one cycle (host buffers in, result out)"},
        "p50_cycle_ms_64k": big["p50_cycle_ms"], "p99_cycle_ms_64k": big["p99_cycle_ms"], "p50_gpu_ms_64k": big["p50_gpu_ms"],
        "p99_gpu_ms_64k": big["p99_gpu_ms"], "move_cycles_64k": big["move_cycles"], "goals_reached_64k": big["goals_reached"],
        "p50_cycle_ms_cfg0": small["p50_cycle_ms"], "p99_cycle_ms_cfg0": small["p99_cycle_ms"], "p50_gpu_ms_cfg0": small["p50_gpu_ms"],
        "p99_gpu_ms_cfg0": small["p99_gpu_ms"], "move_cycles_cfg0": small["move_cycles"], "goals_reached_cfg0": small["goals_reached"],
        "escalated_plans_64k": big["escalated_plans"], "escalated_plans_cfg0": small["escalated_plans"],
        "state_sequence_head": small["state_sequence_head"],
        "e2e": {"value": big["p50_cycle_ms"], "unit": "ms", "h2d_bytes_per_step": 40000 + 4 * 400 + 4096, "d2h_bytes_per_step": 1416},
        "gpu_launches": int(launches),
    }


if __name__ == "__main__":
    import argparse
    import json
    ap = argparse.ArgumentParser()
    ap.add_argument("--cycles", type=int, default=1000)
    ap.add_argument("--candidates", default="cfg0", choices=["cfg0", "64k"])
    a = ap.parse_args()
    pl = Planner(0)
    axes = None if a.candidates == "cfg0" else config.SAMPLING_64K
    out = summarize(run_replay(pl, a.cycles, sampling_axes=axes))
    out["candidates"] = a.candidates
    print(json.dumps(out))
