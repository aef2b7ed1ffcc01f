#!/usr/bin/env python
"""Freezes the COMPILED REFERENCE's full-grid explored totals + winner record of the headline configurations.

    python tools/make_ref_golden_full.py [cfg2:0 cfg2:1 cfg2:2 cfg3:0-7]

oracle/_ref/libhmp_ref.so (the reference's own sources compiled in place, oracle/Makefile target `ref`) scores EVERY
candidate of the sampling grid without the early exit of SimpleScoredSamplingPlanner (full sums, so that the fixture also
ranks the losers); the winner (first strict minimum = the reference's rule, humap_planner.cpp:1367) is then evaluated
once more alone for its record (raw critics, seed twist, poses). Needs HMP_REFERENCE_DIR (a checkout of the reference); the
fixtures let the tests run without one: tests/golden/ref_full_<cfg>_s<seed>.npz (cfg2: 65 536 totals, ~3.6 min on 16 threads each) and
tests/golden/ref_full_cfg3_s0-7.npz (8 worlds x 4096). One process per candidate chunk (the stand-in MapGrid fill hook is a
process-wide pointer, so threads are avoided here).
"""
import multiprocessing as mp
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

CHUNK = 128


def _chunk(a):
    import oracle_binding as ob
    from humap_local_planner_b200 import scenes
    name, seed, lo, hi = a
    cfg = scenes.CONFIGS[name]
    sc = scenes.make_scene(cfg, seed)
    r = ob.plan(scenes.make_params(cfg), sc, scenes.make_sampling(cfg), cand_range=(lo, hi), impl="ref", want=("totals",))
    return lo, hi, r["totals"][lo:hi].copy()


def full_cycle(pool, name, seed):
    import oracle_binding as ob
    from humap_local_planner_b200 import scenes
    from golden_cases import scene_fingerprint
    cfg = scenes.CONFIGS[name]
    sc = scenes.make_scene(cfg, seed)
    params, smp = scenes.make_params(cfg), scenes.make_sampling(cfg)
    Cn = ob.num_candidates(smp)
    totals = np.full(Cn, np.nan)
    jobs = [(name, seed, lo, min(Cn, lo + CHUNK)) for lo in range(0, Cn, CHUNK)]
    for lo, hi, t in pool.imap_unordered(_chunk, jobs, chunksize=1):
        totals[lo:hi] = t
    assert not np.isnan(totals).any()
    valid = totals >= 0
    best = int(np.flatnonzero(valid)[np.argmin(totals[valid])]) if valid.any() else -1   # argmin = FIRST minimum
    out = dict(totals=totals, C=Cn, T=ob.num_steps(params, sc.world), best_index=best, n_valid=int(valid.sum()),
               n_generated=int((totals != -1.0).sum()),
               fingerprint=np.frombuffer(scene_fingerprint(sc, params, smp), dtype=np.uint8))
    if best >= 0:
        w = ob.plan(params, sc, smp, cand_range=(best, best + 1), impl="ref")
        assert w["totals"][best] == totals[best]
        out.update(best_total=totals[best], best_costs=w["costs"][best], best_seed=w["seeds"][best],
                   best_poses=w["poses"][best][: int(w["n_poses"][best])])
    return out


def main():
    import oracle_binding as ob
    ob.ref_lib()   # builds oracle/_ref if needed, before the workers fork
    specs = sys.argv[1:] or ["cfg2:0", "cfg2:1", "cfg2:2", "cfg3:0-7"]
    gold = os.path.join(ROOT, "tests", "golden")
    with mp.get_context("fork").Pool(os.cpu_count() or 1) as pool:
        for spec in specs:
            name, seeds = spec.split(":")
            t0 = time.time()
            if "-" in seeds:
                a, b = (int(x) for x in seeds.split("-"))
                per = [full_cycle(pool, name, s) for s in range(a, b + 1)]
                path = os.path.join(gold, f"ref_full_{name}_s{a}-{b}.npz")
                np.savez_compressed(path, seeds=np.arange(a, b + 1), totals=np.stack([p["totals"] for p in per]),
                                    best_index=np.array([p["best_index"] for p in per]),
                                    best_total=np.array([p.get("best_total", -7.0) for p in per]),
                                    n_valid=np.array([p["n_valid"] for p in per]),
                                    n_generated=np.array([p["n_generated"] for p in per]),
                                    fingerprint=np.stack([p["fingerprint"] for p in per]),
                                    best_costs=np.stack([p["best_costs"] for p in per]),
                                    best_seed=np.stack([p["best_seed"] for p in per]))
            else:
                out = full_cycle(pool, name, int(seeds))
                path = os.path.join(gold, f"ref_full_{name}_s{int(seeds)}.npz")
                np.savez_compressed(path, **out)
            print(path, os.path.getsize(path), "bytes", f"{time.time() - t0:.0f} s", flush=True)


if __name__ == "__main__":
    main()
