#!/usr/bin/env python
"""Benchmark of the trajectory sampling + scoring hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--cfg cfg2|cfg1|cfg0|cfg3|cfg4]

A "step" is one planning cycle: every candidate of the workload rolled out, scored by all critics and the
argmin selected. The default workload is BASELINE.json configs[2] ("crowd stress": 65 536 candidates x
50 people x 8 F-formation groups x 500 obstacle points, 5 s horizon) -- the configuration the metric's
"p50 planning-cycle latency at 64k candidates" is quoted on; it fits one GPU.

  value  candidates/s with the scene already resident in HBM (hmp_replan_resident), timed with CUDA events
         on the library's launching stream (HmpResult.gpu_ms), max over ranks.
  e2e    the same metric through the public C-ABI calls a planner makes every cycle, host buffers in, host
         result out: hmp_set_costmap + 4 x hmp_set_mapgrid + hmp_set_footprint + hmp_plan (wall clock).
  seeds  the timed steps are spread over the synthetic worlds of seeds 0..9; value / ms_per_step are the median over them.
  N > 1  BASELINE config 4: 4096 independent worlds x 4096 candidates (seed = world index), world s -> rank s mod N, one
         hmp_plan_batch per rank per step, host gather of the argmins, no collective on the data path: STRONG scaling.
         The same measurement at one GPU is nested in the default line as "config4".

`--impl reference` times the reference's CPU implementation of the path (oracle/_ref: its own sources compiled in
place; falls back to the oracle restatement if that library is absent), FP64, all host threads, on a bounded candidate
sample of the same workload.

`--steps K` is the number of timed steps of the workload (default 40; cfg4: replay cycles, default 1000).
`--dump-outputs DIR` writes, after the timed steps, what the timed path returned in its last step as DIR/<name>.npy
(float64): every field of the HmpResult records (result_<field>, leading axis = scene; timings left out) and the
per-candidate totals (explored_totals, or a fixed seeded sample of them with its flat indices where they exceed 2^20).
The inputs are seeded, so two builds run with the same arguments can be compared output for output. In a multi-GPU run
of the batched workload (cfg3) the file holds rank 0's share of the worlds (s mod N == 0, in that order).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "candidate trajectories scored/sec"
UNIT = "candidates/s"


DUMP_MAX_BYTES = 64 << 20
DUMP_MAX_TOTALS = 1 << 20


def _result_arrays(results) -> dict:
    """HmpResult records -> one float64 array per field (leading axis = scene); timings and padding are left out."""
    from humap_local_planner_b200 import capi
    out = {}
    for name, _ in capi.HmpResult._fields_:
        if name not in ("gpu_ms", "gpu_ms_select", "_pad"):
            out["result_" + name] = np.array([np.array(getattr(r, name), dtype=np.float64) for r in results])
    return out


def _totals_arrays(totals: np.ndarray) -> dict:
    """Per-candidate totals, or a fixed seeded sample of them (and its flat indices) where there are more than DUMP_MAX_TOTALS."""
    if totals.size <= DUMP_MAX_TOTALS:
        return {"explored_totals": totals}
    idx = np.sort(np.random.default_rng(0).choice(totals.size, DUMP_MAX_TOTALS, replace=False))
    return {"explored_totals_sample": totals[idx], "explored_totals_sample_index": idx.astype(np.float64)}


def _write_outputs(path: str, arrays: dict):
    arrays = {k: np.ascontiguousarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_MAX_BYTES}-byte limit")
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def algorithmic_flops_per_candidate(cfg, params, n_static, n_dynamic, fis_on, T, K=8, V=16, c_cells=45):
    """SURVEY.md section 8d: W = 294 + 86 S + 103 D + 185 P + 45 G + (K+1)(16 V + 6 c) [+ 2900 D with FIS] per step."""
    P, G = cfg.n_people, cfg.n_groups
    W = 294 + 86 * n_static + 103 * n_dynamic + 185 * P + 45 * G + (K + 1) * (16 * V + 6 * c_cells)
    if fis_on:
        W += 2900 * n_dynamic
    return T * W + 60, W


class ClockSampler:
    """Samples SM clocks / throttle reasons with nvidia-smi while the timed region runs."""

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.1)

    def start(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join(timeout=6)
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        smax = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if "Active" in r[3 + i] and "Not" not in r[3 + i]})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": reasons, "samples": len(sm)}


def cpu_baseline(cfg, scene, params, sampling, seconds_budget=12.0):
    """The reference path on the host cores, bounded sample, all host threads.

    kind "reference": oracle/_ref/libhmp_ref.so -- the reference's own first-party sources for the path (generator, SFM,
    World, FIS, conductor, critics) compiled in place against the stand-in third-party headers of oracle/ref_shim/ --
    when that library was built (it travels to the GPU box with the snapshot); kind "port": the oracle restatement."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_binding as ob
    import concurrent.futures as cf
    cores = os.cpu_count() or 1
    impl = "ref" if os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libhmp_ref.so")) else "oracle"
    kind = "reference" if impl == "ref" else "port"
    Cn = ob.num_candidates(sampling)
    # calibrate on a few candidates, then size the sample for ~seconds_budget of wall time
    probe = np.unique(np.linspace(0, Cn - 1, 4).astype(int))
    t0 = time.perf_counter()
    for i in probe:
        ob.plan(params, scene, sampling, cand_range=(int(i), int(i) + 1), want=("totals",), impl=impl)
    per = (time.perf_counter() - t0) / len(probe)
    n = int(min(Cn, max(cores, seconds_budget / per * cores)))
    idx = np.unique(np.linspace(0, Cn - 1, n).astype(int))
    chunks = np.array_split(idx, cores * 2)

    def work(ch):
        for i in ch:
            ob.plan(params, scene, sampling, cand_range=(int(i), int(i) + 1), want=("totals",), impl=impl)
        return len(ch)

    t0 = time.perf_counter()
    with cf.ThreadPoolExecutor(cores) as ex:
        done = sum(ex.map(work, chunks))
    dt = time.perf_counter() - t0
    what = ("reference first-party sources compiled in place (oracle/_ref, stand-in third-party headers)" if impl == "ref"
            else "oracle restatement (oracle/hmp_oracle.cpp)")
    return {"value": done / dt, "unit": UNIT, "cores": cores, "kind": kind,
            "sample": f"{done} of {Cn} candidates of {cfg.name} (evenly spaced over the sampling grid), {dt:.1f} s wall, "
                      f"single-thread rate {1.0 / per:.1f} candidates/s; {what}"}, dt, done


def run_reference(args, rank, world):
    """`--impl reference`: the reference's CPU path (oracle/_ref, else the oracle port), bounded sample per step, rank 0 only."""
    if rank != 0:
        return
    from humap_local_planner_b200 import scenes
    cfg = scenes.CONFIGS[args.cfg]
    scene = scenes.make_scene(cfg, 0)
    params = scenes.make_params(cfg, fis=bool(args.fis))
    sampling = scenes.make_sampling(cfg)
    per_step = max(3.0, min(20.0, 120.0 / max(1, args.steps + args.warmup)))
    times, counts = [], []
    base = None
    for s in range(args.warmup + args.steps):
        base, dt, done = cpu_baseline(cfg, scene, params, sampling, seconds_budget=per_step)
        if s >= args.warmup:
            times.append(dt)
            counts.append(done)
    value = sum(counts) / sum(times)
    base["value"] = value
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / len(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": _workload_name(cfg, args), "candidates_per_step_sample": int(np.mean(counts))},
        "cpu_baseline": base,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def _workload_name(cfg, args):
    return (f"{cfg.name}: {cfg.n_people} people, {cfg.n_groups} F-formation groups, {cfg.n_obstacles} obstacle points, "
            f"{cfg.size}x{cfg.size} costmap @ {cfg.resolution} m, horizon {cfg.sim_time} s @ {cfg.sim_granularity} s, "
            f"FIS {'on' if args.fis else 'off'}")


def _make_scene_job(a):
    """One world of config 4 (worker process): everything hmp_plan_batch / hmp_compute_mapgrid_batch need, as plain bytes and
    arrays; the four MapGrids are NOT computed here (the device does that from the plans)."""
    from humap_local_planner_b200 import scenes
    name, seed = a
    sc = scenes.make_scene(scenes.CONFIGS[name], seed, with_grids=False)
    w = sc.world
    return dict(world=[w.robot_x, w.robot_y, w.robot_yaw, w.vel_x, w.vel_y, w.vel_th, w.goal_local_x, w.goal_local_y,
                       w.goal_local_yaw, w.goal_x, w.goal_y, w.goal_yaw],
                obstacles=bytes(memoryview(sc._obstacles))[: w.n_obstacles * 80], n_obstacles=w.n_obstacles,
                people=bytes(memoryview(sc._people))[: w.n_people * 80], n_people=w.n_people,
                groups=bytes(memoryview(sc._groups))[: w.n_groups * 64], n_groups=w.n_groups,
                cells=sc.cells, plans=[np.asarray(p, dtype=np.float64).reshape(-1, 2) for p, _ in sc.plans],
                local_goal=[bool(lg) for _, lg in sc.plans], hv=sc.hv_prev)


def run_batched(args, rank, local_rank, world, barrier, steps, warmup, n_scenes, dump=None):
    """BASELINE config 4: n_scenes independent worlds (seed = world index) x cfg3's 4096 candidates each, scene s -> rank
    s mod N, one hmp_plan_batch launch per rank per step, host gather of the per-scene argmins (no collective on the data
    path). Total work is fixed, so this is STRONG scaling. Returns the JSON line (rank 0) or None. A dict passed as `dump`
    receives the outputs of this rank's last timed step.

      value  resident: costmaps, MapGrids and worlds already in HBM, hmp_replan_resident, CUDA events
      e2e    host buffers through the C ABI every step: hmp_compute_mapgrid_batch (uploads the costmaps -- 1 byte per cell --
             and the plans, the 4 x n wave fronts run on the device) + hmp_plan_batch (packs and uploads the worlds, reads
             the per-scene results back); wall clock, max over ranks"""
    import ctypes as Cc
    import multiprocessing as mp
    import torch
    from humap_local_planner_b200 import Planner, scenes, capi
    from humap_local_planner_b200.sharding import scenes_for_rank, gather_scene_results
    cfg = scenes.CONFIGS["cfg3"]
    S = n_scenes
    mine = scenes_for_rank(S, rank, world)
    t_gen = time.perf_counter()
    procs = max(1, min(32, (os.cpu_count() or 1) // max(1, world)))
    with mp.get_context("fork").Pool(procs) as pool:
        flats = pool.map(_make_scene_job, [("cfg3", s) for s in mine], chunksize=8)
    t_gen = time.perf_counter() - t_gen
    n_local = len(mine)
    worlds = (capi.HmpWorld * n_local)()
    keep = []
    for k, f in enumerate(flats):
        w = worlds[k]
        (w.robot_x, w.robot_y, w.robot_yaw, w.vel_x, w.vel_y, w.vel_th, w.goal_local_x, w.goal_local_y, w.goal_local_yaw,
         w.goal_x, w.goal_y, w.goal_yaw) = f["world"]
        ob = (capi.HmpObstacle * max(1, f["n_obstacles"])).from_buffer_copy(f["obstacles"].ljust(80 * max(1, f["n_obstacles"]), b"\0"))
        pe = (capi.HmpPerson * max(1, f["n_people"])).from_buffer_copy(f["people"].ljust(80 * max(1, f["n_people"]), b"\0"))
        gr = (capi.HmpGroup * max(1, f["n_groups"])).from_buffer_copy(f["groups"].ljust(64 * max(1, f["n_groups"]), b"\0"))
        w.obstacles, w.people, w.groups = ob, pe, gr
        w.n_obstacles, w.n_people, w.n_groups = f["n_obstacles"], f["n_people"], f["n_groups"]
        keep.append((ob, pe, gr))
    # the per-cycle inputs live in page-locked memory (hmp_host_alloc), as a planner host would keep its staging buffers
    cells_pin = capi.PinnedArray((n_local,) + flats[0]["cells"].shape, np.uint8)
    cells = cells_pin.array
    for k, f in enumerate(flats):
        cells[k] = f["cells"]
    plans = []
    for g in range(4):
        xy = [f["plans"][g] for f in flats]
        plans.append((np.concatenate(xy), np.concatenate([[0], np.cumsum([len(a) for a in xy])]).astype(np.int32)))
    local_goal = flats[0]["local_goal"]
    hv = np.array([f["hv"] for f in flats])
    first = scenes.make_scene(cfg, mine[0], with_grids=False)
    params = scenes.make_params(cfg, fis=bool(args.fis))
    sampling = scenes.make_sampling(cfg)
    pl = Planner(local_rank)
    pl.set_precision(int(args.precise))
    pl.set_sweep_layout(int(args.layout))
    pl.set_params(params)
    pl.set_costmap(first.cells, first.origin_x, first.origin_y, first.resolution)
    pl.set_footprint(first.footprint)

    split_ms = []

    def full_batch():
        # per step, from host buffers: costmaps + plans in, wave fronts on the device, worlds in, per-scene results out
        t0 = time.perf_counter()
        pl.compute_mapgrid_batch(cells, plans, local_goal)
        t1 = time.perf_counter()
        r = pl.plan_batch(worlds, None, None, sampling, hv_prev=hv)
        split_ms.append((1e3 * (t1 - t0), 1e3 * (time.perf_counter() - t1)))
        return r

    res = full_batch()
    C = res[0].n_candidates
    for _ in range(max(1, warmup - 1)):
        pl.replan_resident()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = pl.launch_count()
    dev_ms = []
    for _ in range(steps):
        torch.cuda.synchronize()
        last = pl.replan_resident()
        dev_ms.append(last[0].gpu_ms)   # per-step inputs (n_local x 680 kB) exceed the 126 MB L2
    barrier()
    launches = pl.launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    if dump is not None:
        dump.update(_result_arrays(last))
        dump.update(_totals_arrays(pl.explored_totals(n_local * C)))
    t_dev = torch.tensor([sum(dev_ms) * 1e-3], dtype=torch.float64, device="cuda")
    e2e_t = []
    n_e2e = max(1, min(steps, 5))
    for _ in range(n_e2e):
        torch.cuda.synchronize()
        barrier()
        t0 = time.perf_counter()
        res = full_batch()
        e2e_t.append(time.perf_counter() - t0)
    barrier()
    t_e2e = torch.tensor([statistics.mean(e2e_t)], dtype=torch.float64, device="cuda")
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(t_dev, op=dist.ReduceOp.MAX)
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
    # host gather of the per-scene argmins (16 bytes per scene)
    gathered = gather_scene_results({s: (r.best_index, r.best_total) for s, r in zip(mine, res)}, S)
    line = None
    if rank == 0:
        n_cells = cells[0].size
        h2d = int(cells.nbytes + sum(p[0].nbytes + p[1].nbytes for p in plans) +
                  sum(f["n_obstacles"] * 80 + f["n_people"] * 64 + f["n_groups"] * 32 + 256 for f in flats))
        # fixture check: worlds 0..7 of config 4 against the compiled reference's full-grid winners
        sel = _check_batched_selection(gathered)
        line = {
            "metric": METRIC, "value": S * C * steps / float(t_dev.item()), "unit": UNIT, "n_gpus": world, "steps": steps,
            "warmup": warmup, "ms_per_step": 1e3 * float(t_dev.item()) / steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": {0: "f32", 1: "f64", 2: "f32 sweep + f64 refinement of the leaders"}[int(args.precise)],
            "data": "synthetic",
            "config": {"workload": f"batched scenes (BASELINE config 4): {S} independent worlds (seed = world index) x {C} candidates "
                                   f"({_workload_name(cfg, args)})",
                       "parallelism": f"scene s -> rank s mod {world}, one hmp_plan_batch launch per rank, host gather of argmins, no collective",
                       "l2": f"resident inputs per step ({n_local} scenes x {(n_cells * 17) // 1024} kB) exceed L2",
                       "timing": "CUDA events on the launching stream, max over ranks"},
            "e2e": {"value": S * C / float(t_e2e.item()), "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": int(n_local * Cc.sizeof(capi.HmpResult)), "steps": n_e2e,
                    "ms_mapgrids_then_plan_rank0": [round(statistics.mean(x[0] for x in split_ms[-n_e2e:]), 2),
                                                    round(statistics.mean(x[1] for x in split_ms[-n_e2e:]), 2)],
                    "what": "hmp_compute_mapgrid_batch (costmaps + plans up, wave fronts on the device) + hmp_plan_batch (worlds up, results down), wall clock"},
            "gpu_launches": int(launches), "clocks": clocks,
            "scenes_with_valid_winner": int(sum(1 for b, _ in gathered if b >= 0)),
            "selection_matches_reference": sel, "scene_generation_s": round(t_gen, 1),
        }
    pl.close()
    return line


def _check_batched_selection(gathered):
    """Worlds 0..7 of config 4 against tests/golden/ref_full_cfg3_s0-7.npz (the compiled reference's full-grid winners)."""
    path = os.path.join(ROOT, "tests", "golden", "ref_full_cfg3_s0-7.npz")
    if not os.path.exists(path) or len(gathered) < 8:
        return None
    g = np.load(path)
    ok = True
    for k, s in enumerate(g["seeds"]):
        bi, bt = gathered[int(s)]
        t = g["totals"][k]
        v = np.sort(t[t >= 0])
        close = len(v) > 1 and (v[1] - v[0]) <= 1e-4 * abs(v[0])
        ok &= bool(bi == int(g["best_index"][k]) or close)
        ok &= bool(abs(bt - float(g["best_total"][k])) <= 1e-4 * abs(float(g["best_total"][k])))
    return {"checked_worlds": [int(x) for x in g["seeds"]], "ok": bool(ok)}


def _check_selection(cfg_name, seed, res):
    """The cycle's winner against the compiled reference's full-grid fixture (tests/golden/ref_full_<cfg>_s<seed>.npz):
    north_star's gate -- identical candidate unless the reference's two best totals are within 1e-4 relative."""
    path = os.path.join(ROOT, "tests", "golden", f"ref_full_{cfg_name}_s{seed}.npz")
    if not os.path.exists(path):
        return None
    g = np.load(path)
    t = g["totals"]
    v = np.sort(t[t >= 0])
    close = len(v) > 1 and (v[1] - v[0]) <= 1e-4 * abs(v[0])
    same = int(res.best_index) == int(g["best_index"])
    total_ok = abs(res.best_total - float(g["best_total"])) <= 1e-4 * abs(float(g["best_total"]))
    return bool((same or close) and total_ok)


def _ncu_counts():
    """Executed-instruction counts of the dominant kernel from the latest committed ncu capture (profiles/*_ncu_counts.json,
    written by tools/make_profiles.py): thread-level FFMA / FMUL / FADD (packed FFMA2 etc. counted twice), MUFU, issue-active."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "*_ncu_counts.json")))
    if not files:
        return None
    try:
        d = json.load(open(files[-1]))
        d["file"] = os.path.basename(files[-1])
        return d
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 40; cfg4: replay cycles, default 1000)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cfg", default=None, help="workload: cfg2 (default at 1 GPU: BASELINE config 3, the headline), cfg1, cfg0, "
                                                "cfg3 (BASELINE config 4, batched scenes: the default at N > 1), cfg4 (config 5: closed-loop replay)")
    ap.add_argument("--fis", type=int, default=1)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--scenes", type=int, default=4096, help="config 4: independent worlds in total, sharded over the ranks")
    ap.add_argument("--seeds", type=int, default=10, help="single-scene workloads: synthetic worlds (seeds 0 .. n-1) the timed steps are "
                                                          "spread over; value = candidates / median cycle time over the seeds (SURVEY 8d)")
    ap.add_argument("--no-exact", action="store_true", help="1 GPU: skip the nested exact-mode (FP64, precision 1) measurement")
    ap.add_argument("--no-config4", action="store_true", help="1 GPU: skip the nested config-4 (batched scenes) measurement")
    ap.add_argument("--precise", type=int, default=2, help="hmp_set_precision mode: 0 FP32 object loops, 1 FP64 (exact-parity mode), 2 FP32 sweep + FP64 refinement of the leaders")
    ap.add_argument("--layout", type=int, default=0, help="hmp_set_sweep_layout: 0 automatic, 1 one warp per candidate, 2 one thread per candidate")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path returned in its last step to DIR/<name>.npy (float64, at most 64 MB); "
                         "cfg3 on N > 1 GPUs: rank 0's share of the worlds")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.cfg is None:
        # 1 GPU: the configuration the metric is quoted on (64k candidates, one planning cycle = one GPU by design);
        # N > 1: the only configuration that shards (independent worlds), BASELINE config 4
        args.cfg = "cfg2" if world == 1 else "cfg3"
    if args.steps is None:
        args.steps = 1000 if args.cfg == "cfg4" else 40
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    dump = {} if args.dump_outputs else None

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from humap_local_planner_b200 import Planner, scenes

    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if args.cfg == "cfg4":
        from humap_local_planner_b200 import replay
        line = replay.bench_line(args, rank, local_rank, world, barrier, dump=dump)
        if rank == 0 and line is not None:
            if dump is not None:
                last = dump.pop("replay_last_result")
                dump.update(_result_arrays([] if last is None else [last]))
                _write_outputs(args.dump_outputs, dump)
            print(json.dumps(line))
        if world > 1:
            dist.destroy_process_group()
        return

    if args.cfg == "cfg3":
        line = run_batched(args, rank, local_rank, world, barrier, args.steps, args.warmup, args.scenes, dump=dump)
        if rank == 0:
            if dump is not None:
                _write_outputs(args.dump_outputs, dump)
            print(json.dumps(line))
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- single-scene workloads (cfg2 headline, cfg1, cfg0): one planning cycle per step ---------------------------------
    # N > 1 (only on request, --cfg cfg2 under torchrun): every rank plans the same seeds -- replicas, weak scaling
    cfg = scenes.CONFIGS[args.cfg]
    n_seeds = max(1, min(args.seeds, args.steps))
    per_seed = [args.steps // n_seeds + (1 if k < args.steps % n_seeds else 0) for k in range(n_seeds)]   # sums to --steps
    params = scenes.make_params(cfg, fis=bool(args.fis))
    sampling = scenes.make_sampling(cfg)
    pl = Planner(local_rank)
    pl.set_precision(int(args.precise))
    pl.set_sweep_layout(int(args.layout))
    pl.set_params(params)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")  # > 126 MB L2
    sampler = ClockSampler(local_rank)
    started = False
    launches = 0
    seed_rows = []
    dev_all, sel_all, e2e_all, e2e_dev_all = [], [], [], []
    escalated_plans = 0   # e2e plans that hmp_plan redid as an exact FP64 sweep (hmp_set_escalation; none expected on these worlds)
    selection = {}
    scene0 = None
    t_dev_sum = 0.0
    t_e2e_sum = 0.0
    wall_resident = 0.0
    for seed in range(n_seeds):
        scene = scenes.make_scene(cfg, seed=seed)
        if seed == 0:
            scene0 = scene

        def full_cycle():
            # what HumapPlanner does every control cycle before and at the seam (humap_planner.cpp:1054-1141, :1294-1377)
            pl.set_costmap(scene.cells, scene.origin_x, scene.origin_y, scene.resolution)
            for g in range(4):
                pl.set_mapgrid(g, scene.grids[g], scene.hv_prev[g])
            pl.set_footprint(scene.footprint)
            return pl.plan(scene.world, sampling, want_poses=True)

        def full_cycle_device_grids():
            # variant: MapGridCostFunction::prepare() replaced as well (wave fronts computed on the device from the plan poses)
            pl.set_costmap(scene.cells, scene.origin_x, scene.origin_y, scene.resolution)
            for g, (plan, local_goal) in enumerate(scene.plans):
                pl.compute_mapgrid(g, plan, local_goal, scene.hv_prev[g])
            pl.set_footprint(scene.footprint)
            return pl.plan(scene.world, sampling, want_poses=True)

        res, _ = full_cycle()
        C = res.n_candidates
        T = pl.num_steps()
        chk = _check_selection(cfg.name, seed, res) if int(args.precise) != 0 else None
        if chk is not None:
            selection[seed] = chk
        # ---- value: inputs resident in HBM, CUDA-event time of the kernels on the launching stream ------------------
        for _ in range(args.warmup):
            flush.zero_()
            pl.replan_resident()
        barrier()
        if rank == 0 and not started:
            sampler.start()
            started = True
        l0 = pl.launch_count()
        dev_ms, sel_ms = [], []
        t_w0 = time.perf_counter()
        for _ in range(per_seed[seed]):
            flush.zero_()          # L2 flush between timed iterations (not inside the event-timed region)
            torch.cuda.synchronize()
            r = pl.replan_resident()[0]
            dev_ms.append(r.gpu_ms)
            sel_ms.append(r.gpu_ms_select)
        barrier()
        wall_resident += time.perf_counter() - t_w0
        launches += pl.launch_count() - l0
        if dump is not None and seed == n_seeds - 1:
            # read before the e2e cycles below plan again
            dump.update(_result_arrays([r]))
            dump.update(_totals_arrays(pl.explored_totals(C)))
        # ---- e2e: host buffers through the public C-ABI, every step uploads the cycle's inputs and reads the result ----
        full_cycle()
        barrier()
        e2e_times = []
        for _ in range(per_seed[seed]):
            flush.zero_()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r, poses = full_cycle()
            e2e_times.append(time.perf_counter() - t0)
            escalated_plans += 1 if pl.last_escalated() == 1 else 0
        unreliable = pl.last_unreliable_leaders()
        barrier()
        full_cycle_device_grids()
        e2e_dev_times = []
        for _ in range(min(per_seed[seed], 3)):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r_dev, _ = full_cycle_device_grids()
            e2e_dev_times.append(time.perf_counter() - t0)
        assert r_dev.best_index == r.best_index and r_dev.best_total == r.best_total, "device wave front changed the selection"
        barrier()
        td = torch.tensor([sum(dev_ms) * 1e-3, sum(e2e_times)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(td, op=dist.ReduceOp.MAX)
        t_dev_sum += float(td[0].item())
        t_e2e_sum += float(td[1].item())
        dev_all += dev_ms
        sel_all += sel_ms
        e2e_all += e2e_times
        e2e_dev_all += e2e_dev_times
        seed_rows.append({"seed": seed, "cycle_ms": statistics.mean(dev_ms), "sweep_ms": statistics.mean(sel_ms),
                          "e2e_ms": 1e3 * statistics.mean(e2e_times), "best_index": int(r.best_index), "best_total": float(r.best_total),
                          "n_valid": int(r.n_valid), "leaders": pl.last_num_leaders(), "unreliable_leaders": int(unreliable)})
    clocks = sampler.stop() if rank == 0 else None
    scene = scene0

    if rank == 0:
        import ctypes as Cc
        from humap_local_planner_b200 import capi
        # SURVEY 8d: seeds 0..9, the median is reported. value = candidates per second at the median cycle time over the seeds
        # (each seed's cycle time = mean over its share of the --steps timed steps); ms_per_step is that median.
        med_cycle = statistics.median([row["cycle_ms"] for row in seed_rows])
        med_sweep = statistics.median([row["sweep_ms"] for row in seed_rows])
        med_e2e = statistics.median([row["e2e_ms"] for row in seed_rows])
        n_cells = scene.cells.size
        h2d = n_cells + 4 * n_cells * 4 + Cc.sizeof(capi.HmpParams) + scene.world.n_obstacles * 64 + scene.world.n_people * 64 + \
            scene.world.n_groups * 32 + 10 * 64 * 8
        d2h = (14 + 3 + 3 * T + 1) * 8 + 8 + 64
        nd = sum(1 for i in range(scene.world.n_obstacles) if scene.world.obstacles[i].force_dynamic or
                 (scene.world.obstacles[i].vx ** 2 + scene.world.obstacles[i].vy ** 2) ** 0.5 > 0.035)
        ns = scene.world.n_obstacles - nd
        flops_cand, W = algorithmic_flops_per_candidate(cfg, params, ns, nd, bool(args.fis), T)
        sel_s = med_sweep * 1e-3
        achieved = C * flops_cand / sel_s / 1e12
        # INSTRUMENTED operation count of the reference formulation (tools/count_flops.py: the oracle over a counting scalar, a
        # 512-candidate sample per seed, committed as profiles/r02_flop_count.json -- only the JSON is read here): flop one cycle
        # of the CPU path executes for this world, rejections included, over this run's sweep time of the same seed
        instrumented = None
        try:
            fc = json.load(open(os.path.join(ROOT, "profiles", "r02_flop_count.json")))
            per_seed_flop = {r["seed"]: r for r in fc["rows"] if r["config"] == args.cfg}
            tf_rows = [per_seed_flop[row["seed"]]["flop_per_cycle"] / (row["sweep_ms"] * 1e-3) / 1e12
                       for row in seed_rows if row["seed"] in per_seed_flop]
            if tf_rows and bool(args.fis):
                med = fc["median_over_seeds"][args.cfg]
                instrumented = {"flop_per_candidate_step": med["flop_per_candidate_step"], "flop_per_cycle": med["flop_per_cycle"],
                                "tflops": statistics.median(tf_rows), "seeds": len(tf_rows),
                                "survey_estimate_over_instrumented": W / med["flop_per_candidate_step"],
                                "source": "profiles/r02_flop_count.json (tools/count_flops.py)"}
        except Exception:
            instrumented = None
        mode = pl.last_sweep_mode()
        sweep_name = (f"sweep_tpc_kernel{'<double>' if int(args.precise) == 1 else ''} (one thread per candidate, {mode} threads per block)" if mode
                      else ("plan_kernel<false,double> (one warp per candidate, FP64)" if int(args.precise) == 1
                            else "plan_kernel<false,float> (one warp per candidate)"))
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        traffic = None
        try:   # DRAM bytes per launch of the dominant kernel from the latest committed ncu --set full capture
            import glob
            tf = sorted(glob.glob(os.path.join(ROOT, "profiles", "*_traffic.json")))[-1]
            tj = json.load(open(tf))
            if args.cfg == "cfg2" and int(args.precise) != 1:
                traffic = int(tj["dram_bytes_read"]) + int(tj["dram_bytes_write"])
        except Exception:
            pass
        sm_max = float(peaks.get("sm_max_mhz", 1965.0))
        peak_fp32 = 148 * 128 * 2 * sm_max * 1e6 / 1e12
        peak_fp32_measured = pl.measure_fp32_peak()       # FFMA micro-benchmark on this GPU, same launch shape as the sweep
        hbm_peak = float(peaks.get("hbm_gbs", 0.0)) or None
        counts = _ncu_counts() if (args.cfg == "cfg2" and int(args.precise) != 1) else None
        executed = None
        if counts:
            # flop the kernel EXECUTED per launch (ncu, thread-level, predicated-on): FFMA = 2, FMUL / FADD = 1, MUFU = 1;
            # divided by the live launch time of this run
            ex_flop = 2.0 * counts["ffma"] + counts["fmul"] + counts["fadd"] + counts.get("mufu", 0.0)
            executed = {"flop_per_launch": ex_flop, "tflops": ex_flop / sel_s / 1e12,
                        "frac": ex_flop / sel_s / 1e12 / peak_fp32, "issue_active": counts.get("issue_active"),
                        "fma_pipe": counts.get("fma_pipe"), "alu_pipe": counts.get("alu_pipe"), "xu_pipe": counts.get("xu_pipe"),
                        "source": counts.get("file")}
        line = {
            "metric": METRIC, "value": world * C / (med_cycle * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": med_cycle, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": {0: "f32", 1: "f64", 2: "f32 sweep + f64 refinement of the leaders"}[int(args.precise)], "data": "synthetic",
            "config": {"workload": _workload_name(cfg, args), "candidates": C, "steps_per_rollout": T,
                       "seeds": f"synthetic worlds of seeds 0..{n_seeds - 1}, {args.steps} timed steps spread over them; value and "
                                "ms_per_step are the MEDIAN over the seeds (SURVEY 8d)",
                       "parallelism": ("one planning cycle = one scene on one GPU" if world == 1 else
                                       f"replicas: every one of the {world} ranks plans the same worlds, no collective"),
                       "l2": "flushed with a 256 MiB write between timed iterations", "timing": "CUDA events on the launching stream"},
            "value_mean_over_all_steps": world * C * args.steps / t_dev_sum,
            "p50_cycle_ms": statistics.median(dev_all), "p99_cycle_ms": sorted(dev_all)[min(len(dev_all) - 1, int(0.99 * len(dev_all)))],
            "p50_cycle_ms_e2e": 1e3 * statistics.median(e2e_all),
            "p50_cycle_ms_e2e_device_mapgrids": 1e3 * statistics.median(e2e_dev_all),
            "wall_ms_per_step_resident": 1e3 * wall_resident / args.steps,
            "per_seed": seed_rows,
            "e2e": {"value": world * C / (med_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "value_mean_over_all_steps": world * C * args.steps / t_e2e_sum},
            "gpu_launches": int(launches),
            "escalated_plans": int(escalated_plans),
            "clocks": clocks,
            "selection_matches_reference": (all(selection.values()) if selection else None),
            "selection_checked_seeds": sorted(selection),
            # frac = FP32 flop the kernel EXECUTED (ncu thread-level counts of the committed capture of this very kernel) over the
            # live launch time, against the nominal CUDA-core peak. The algorithmic estimate of SURVEY 8d (what the reference's
            # statements would cost) is reported beside it: the exact prunings (obstacle critic deferred and walked largest bound
            # first, people-critic bounds) and the reformulations of DESIGN 3b skip most of it, so it can exceed the peak.
            "roofline": {"bound": "fp32-cuda-core",
                         "achieved": executed["tflops"] if executed else achieved,
                         "peak": peak_fp32, "unit": "TFLOP/s",
                         "frac": (executed["frac"] if executed else achieved / peak_fp32),
                         "frac_is": "executed FP32 flop (ncu) / nominal peak" if executed else "algorithmic estimate / nominal peak",
                         "traffic": traffic,
                         "executed_fp32_frac": executed["frac"] if executed else None,
                         "issue_active": executed["issue_active"] if executed else None,
                         "executed": executed,
                         "algorithmic_frac": (instrumented["tflops"] if instrumented else achieved) / peak_fp32,
                         "algorithmic_frac_is": ("instrumented flop count of the reference formulation / sweep time / nominal peak"
                                                 if instrumented else "SURVEY 8d estimate / sweep time / nominal peak"),
                         "algorithmic": {"instrumented": instrumented,
                                         "survey_estimate": {"flop_per_candidate_step": W, "tflops": achieved,
                                                             "over_nominal_peak": achieved / peak_fp32,
                                                             "over_measured_peak": achieved / peak_fp32_measured}},
                         "peak_measured": peak_fp32_measured,
                         "frac_of_measured": (executed["tflops"] / peak_fp32_measured) if executed else achieved / peak_fp32_measured,
                         "hbm": {"achieved_gbs": (traffic / sel_s / 1e9) if traffic else None, "peak_gbs": hbm_peak},
                         "note": f"dominant kernel {sweep_name}, live launch time (median over seeds) {1e3 * sel_s:.3f} ms. executed: thread-level "
                                 f"FFMA x2 + FMUL + FADD + MUFU of the committed ncu capture ({executed['source'] if executed else 'none'}); "
                                 f"issue_active: ncu smsp__issue_active of that capture. algorithmic.instrumented: flop the CPU formulation executes "
                                 f"per cycle, counted by running the oracle over a counting scalar (add, mul, div, sqrt, exp, trig, atan2 one "
                                 f"each), over the sweep time -- how much of the literal formulation's work per second the kernel delivers, not a "
                                 f"utilisation (prunings and reformulations skip part of it); survey_estimate: W={W} flop per candidate-step "
                                 f"(SURVEY.md 8d, read off the reference's statements; 1.4-1.9x the instrumented count). peak = nominal 148 SM x 128 lanes x 2 x {sm_max:.0f} MHz; peak_measured = FFMA probe "
                                 "of this run (MEASURED_PEAKS.json has no FP32 CUDA-core entry; the path is neither HBM- nor tensor-bound: "
                                 "traffic is the DRAM bytes of the capture)"},
            "best_index": int(seed_rows[0]["best_index"]), "best_total": float(seed_rows[0]["best_total"]), "n_valid": int(seed_rows[0]["n_valid"]),
        }
        if not args.no_cpu_baseline:
            base, _, _ = cpu_baseline(cfg, scene, params, sampling, seconds_budget=12.0)
            line["cpu_baseline"] = base
    if world == 1 and args.cfg == "cfg2" and int(args.precise) == 2 and not args.no_exact:
        # The same workload in the exact-parity mode (hmp_set_precision 1: every candidate rolled out with FP64 object loops and
        # FIS, the oracle's selection by construction) -- north_star's 50 ms budget has to hold for it too. Seeds 0..2 (the ones
        # with frozen reference winners), resident inputs, CUDA events, L2 flushed between the steps.
        try:
            pl.set_precision(1)
            ex_rows, ex_ok = [], []
            for seed in range(n_seeds):   # selection checked where a frozen reference winner exists (seeds 0..2)
                sc = scenes.make_scene(cfg, seed=seed)
                pl.set_costmap(sc.cells, sc.origin_x, sc.origin_y, sc.resolution)
                for g in range(4):
                    pl.set_mapgrid(g, sc.grids[g], sc.hv_prev[g])
                pl.set_footprint(sc.footprint)
                r1, _ = pl.plan(sc.world, sampling, want_poses=True)
                chk = _check_selection(cfg.name, seed, r1)
                if chk is not None:
                    ex_ok.append(bool(chk))
                ms = []
                for _ in range(2):
                    flush.zero_()
                    torch.cuda.synchronize()
                    ms.append(pl.replan_resident()[0].gpu_ms)
                ex_rows.append({"seed": seed, "cycle_ms": statistics.median(ms), "best_index": int(r1.best_index),
                                "best_total": float(r1.best_total)})
            ex_mode = pl.last_sweep_mode()
            ex_med = statistics.median([r["cycle_ms"] for r in ex_rows])
            line["exact_mode"] = {"dtype": "f64", "ms_per_step": ex_med, "value": C / (ex_med * 1e-3), "unit": UNIT,
                                  "max_cycle_ms": max(r["cycle_ms"] for r in ex_rows), "min_cycle_ms": min(r["cycle_ms"] for r in ex_rows),
                                  "seeds_within_50ms": sum(1 for r in ex_rows if r["cycle_ms"] <= 50.0), "seeds": len(ex_rows),
                                  "selection_matches_reference": (all(ex_ok) if ex_ok else None), "per_seed": ex_rows,
                                  "kernel": (f"sweep_tpc_kernel<double> (one thread per candidate, {ex_mode} threads per block)" if ex_mode
                                             else "plan_kernel<false,double> (one warp per candidate)"),
                                  "what": "hmp_set_precision(1): FP64 object loops, literal FIS and scalar section for every candidate; "
                                          "resident inputs, CUDA events, median of 2 steps per seed, ms_per_step = median over the seeds"}
        except Exception as e:   # the headline line must not depend on it
            line["exact_mode"] = {"error": repr(e)}
    pl.close()
    del flush
    torch.cuda.empty_cache()
    if world == 1 and args.cfg == "cfg2" and not args.no_config4 and int(args.precise) == 2:
        # BASELINE config 4 (batched scenes) at one GPU, nested: the N = 1 point of the strong-scaling curve `--gpus N` reports
        try:
            c4 = run_batched(args, rank, local_rank, world, barrier, steps=3, warmup=2, n_scenes=args.scenes)
            line["config4"] = {k: c4[k] for k in ("value", "unit", "ms_per_step", "steps", "scaling", "config", "e2e", "gpu_launches",
                                                  "scenes_with_valid_winner", "selection_matches_reference", "scene_generation_s")}
        except Exception as e:   # the headline line must not depend on it
            line["config4"] = {"error": repr(e)}
    if rank == 0:
        if dump is not None:
            _write_outputs(args.dump_outputs, dump)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
