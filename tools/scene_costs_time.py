"""What a per-scene cost table (hmp_set_scene_costs) costs a BASELINE config-4 batch: 4096 worlds x 4096 candidates, built by
bench.py's config-4 world builder, planned without and with a table in one process, the two variants alternating.

  resident  hmp_replan_resident (worlds, costmaps and MapGrids already in HBM), wall clock around the call, which includes the
            host-side build and upload of the 4096 DevParams copies; the device time of the cycle (CUDA events) beside it
  e2e       hmp_compute_mapgrid_batch + hmp_plan_batch from host buffers, wall clock

The table is config.local_scene_costs of every world (the per-cycle values of updateLocalCosts). Prints one JSON line with
the card name and power limit.

    python tools/scene_costs_time.py [--scenes 4096] [--rounds 5] [--replans 5]
"""
import argparse
import json
import multiprocessing as mp
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from bench import _make_scene_job  # noqa: E402
from humap_local_planner_b200 import Planner, capi, config, scenes  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scenes", type=int, default=4096)
    ap.add_argument("--rounds", type=int, default=5, help="alternations of the two variants")
    ap.add_argument("--replans", type=int, default=5, help="resident re-plans per variant and round")
    ap.add_argument("--precise", type=int, default=2)
    args = ap.parse_args()
    S = args.scenes
    cfg = scenes.CONFIGS["cfg3"]
    with mp.get_context("fork").Pool(max(1, min(32, os.cpu_count() or 1))) as pool:
        flats = pool.map(_make_scene_job, [("cfg3", s) for s in range(S)], chunksize=8)
    worlds = (capi.HmpWorld * S)()
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
    params = scenes.make_params(cfg)
    sampling = scenes.make_sampling(cfg)
    table = [config.local_scene_costs(params, worlds[s], [(worlds[s].people[i].x, worlds[s].people[i].y) for i in range(worlds[s].n_people)])
             for s in range(S)]
    cells_pin = capi.PinnedArray((S,) + flats[0]["cells"].shape, np.uint8)
    cells = cells_pin.array
    for k, f in enumerate(flats):
        cells[k] = f["cells"]
    plans = []
    for g in range(4):
        xy = [f["plans"][g] for f in flats]
        plans.append((np.concatenate(xy), np.concatenate([[0], np.cumsum([len(a) for a in xy])]).astype(np.int32)))
    local_goal = flats[0]["local_goal"]
    hv = np.array([f["hv"] for f in flats])
    first = scenes.make_scene(cfg, 0, with_grids=False)
    pl = Planner(0)
    pl.set_precision(args.precise)
    pl.set_params(params)
    pl.set_costmap(first.cells, first.origin_x, first.origin_y, first.resolution)
    pl.set_footprint(first.footprint)

    variants = {"no_table": None, "table": table}
    t = {v: {"resident_wall_ms": [], "resident_gpu_ms": [], "e2e_ms": []} for v in variants}
    winners = {}

    def full_batch():
        pl.compute_mapgrid_batch(cells, plans, local_goal)
        return pl.plan_batch(worlds, None, None, sampling, hv_prev=hv)

    for v, tab in variants.items():   # warm-up of both variants
        pl.set_scene_costs(tab)
        full_batch()
        pl.replan_resident()
    for _ in range(args.rounds):
        for v, tab in variants.items():
            pl.set_scene_costs(tab)
            t0 = time.perf_counter()
            res = full_batch()
            t[v]["e2e_ms"].append(1e3 * (time.perf_counter() - t0))
            winners[v] = [r.best_index for r in res]
            for _ in range(args.replans):
                t0 = time.perf_counter()
                r = pl.replan_resident()
                t[v]["resident_wall_ms"].append(1e3 * (time.perf_counter() - t0))
                t[v]["resident_gpu_ms"].append(r[0].gpu_ms)
    pl.close()
    try:
        smi = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
    except Exception as e:   # noqa: BLE001
        smi = f"nvidia-smi unavailable: {e}"
    out = {"scenes": S, "candidates_per_scene": res[0].n_candidates, "precise": args.precise, "gpu": smi,
           "rounds": args.rounds, "replans_per_round": args.replans,
           "table_bytes_uploaded": S * 1952, "worlds_whose_winner_changes_with_the_table":
               int(sum(a != b for a, b in zip(winners["no_table"], winners["table"])))}
    for v in variants:
        out[v] = {k: {"median": round(statistics.median(x), 3), "min": round(min(x), 3), "max": round(max(x), 3)} for k, x in t[v].items()}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
