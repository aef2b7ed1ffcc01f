#!/usr/bin/env python
"""Generates tests/golden/ref_*.npz from the REFERENCE'S OWN sources.

oracle/_ref/libhmp_ref.so is the reference's first-party code for the path (generator, SFM, World, FIS, conductor, the
eleven first-party critics) compiled where it lies in the checkout HMP_REFERENCE_DIR names, against the stand-in
third-party headers of oracle/ref_shim/ (oracle/Makefile, target `ref`; driver oracle/ref_driver.cpp). Its outputs on the
seeded synthetic scenes of humap_local_planner_b200/scenes.py are frozen as small fixtures so that the tests need no
checkout; tests/test_ref_golden.py (CPU: oracle vs fixtures) and tests/test_gpu_parity.py (GPU: CUDA path vs fixtures)
read them. Re-run after changing scenes.py / config.py defaults:

    HMP_REFERENCE_DIR=<checkout> python tools/make_ref_golden.py          # tests/golden/ref_cycle_*.npz, ref_fis.npz
    HMP_REFERENCE_DIR=<checkout> python tools/make_ref_golden.py --live   # tests/golden/ref_live_*.npz

--live runs the comparisons of tests/test_ref_golden.py that have no fixture of their own with HMP_WRITE_REF_GOLDEN=1:
each stores the compiled reference's outputs for its case, which the test reads where oracle/_ref is absent.
"""
import hashlib
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import oracle_binding as ob  # noqa: E402
from humap_local_planner_b200 import scenes  # noqa: E402
from golden_cases import CYCLE_CASES, FIS_SEED, FIS_N, fixture_path, scene_fingerprint, sample_indices, fis_inputs  # noqa: E402


def main():
    os.makedirs(os.path.join(ROOT, "tests", "golden"), exist_ok=True)
    L = ob.ref_lib()
    for name, seed, n_sample in CYCLE_CASES:
        cfg = scenes.CONFIGS[name]
        sc = scenes.make_scene(cfg, seed)
        params = scenes.make_params(cfg)
        smp = scenes.make_sampling(cfg)
        Cn = ob.num_candidates(smp)
        idx = sample_indices(Cn, n_sample)
        out = {k: [] for k in ("totals", "costs", "seeds", "poses", "n_poses", "generated")}
        for i in idx:
            r = ob.plan(params, sc, smp, cand_range=(int(i), int(i) + 1), impl="ref")
            for k in out:
                out[k].append(r[k][int(i)])
        arrs = {k: np.array(v) for k, v in out.items()}
        extra = {}
        if Cn <= 4096:
            # whole cycle with the reference's early exit: the selection the robot would execute
            full = ob.plan(params, sc, smp, early_exit=True, impl="ref", want=("totals",))
            res = full["result"]
            extra = dict(best_index=res.best_index, best_total=res.best_total, n_generated=res.n_generated,
                         n_valid=res.n_valid, best_costs=np.array(list(res.costs)), best_seed=np.array([res.xv, res.yv, res.thetav]),
                         best_poses=full["best_poses"], hv=np.array(list(res.highest_valid_cost)))
        path = fixture_path(name, seed, n_sample)
        np.savez_compressed(path, idx=idx, fingerprint=np.frombuffer(scene_fingerprint(sc, params, smp), dtype=np.uint8),
                            T=ob.num_steps(params, sc.world), C=Cn, **arrs, **extra)
        print(path, os.path.getsize(path), "bytes; generated", int(arrs["generated"].sum()), "of", len(idx))
    # fuzzy inference: fuzz::Processor::process on random tuples
    x = fis_inputs()
    out3 = np.zeros((FIS_N, 3))
    import ctypes as C
    for i in range(FIS_N):
        L.ref_fis_process(x[i, 0], x[i, 1], x[i, 2], x[i, 3], out3[i].ctypes.data_as(C.c_void_p))
    path = os.path.join(ROOT, "tests", "golden", "ref_fis.npz")
    np.savez_compressed(path, inputs=x, outputs=out3)
    print(path, os.path.getsize(path), "bytes; fired", int(out3[:, 2].sum()), "of", FIS_N)


def main_live():
    if not ob.ref_available():
        sys.exit("oracle/_ref is not built and HMP_REFERENCE_DIR names no checkout of the reference")
    env = dict(os.environ, HMP_WRITE_REF_GOLDEN="1")
    subprocess.run([sys.executable, "-m", "pytest", "-q", os.path.join(ROOT, "tests", "test_ref_golden.py"), "-k", "compiled_reference"],
                   check=True, env=env)


if __name__ == "__main__":
    main_live() if "--live" in sys.argv[1:] else main()
