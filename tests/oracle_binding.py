"""ctypes binding of the CPU oracle (oracle/hmp_oracle.cpp). TEST INFRASTRUCTURE: only tests/,
__graft_entry__.smoke() and bench.py's CPU-baseline legs import this module."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from humap_local_planner_b200.capi import (HmpParams, HmpWorld, HmpSampling, HmpSample, HmpResult, HmpEquisampled,
                                           NUM_COSTS, NUM_MAPGRIDS, NUM_AMPLIFIERS, Scene)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_LIB = os.path.join(ROOT, "oracle", "_build", "libhmp_oracle.so")
_REF_LIB = os.path.join(ROOT, "oracle", "_ref", "libhmp_ref.so")
# Optional checkout of the original humap_local_planner: the live comparisons compile its own sources where they lie
# (oracle/Makefile and tests/Makefile read the same variable). Without it they skip.
REFERENCE_DIR = os.environ.get("HMP_REFERENCE_DIR", "")
_d, _i = C.c_double, C.c_int32
_lib = None
_ref_lib = None


class OrcPlanInput(C.Structure):
    _fields_ = [
        ("params", C.POINTER(HmpParams)), ("world", C.POINTER(HmpWorld)), ("sampling", C.POINTER(HmpSampling)),
        ("extra", C.c_void_p), ("n_extra", _i),
        ("size_x", _i), ("size_y", _i), ("cells", C.c_void_p),
        ("origin_x", _d), ("origin_y", _d), ("resolution", _d),
        ("target_dist", C.c_void_p * NUM_MAPGRIDS), ("highest_valid_cost_prev", _d * NUM_MAPGRIDS),
        ("footprint_xy", C.c_void_p), ("n_footprint", _i),
        ("early_exit", _i), ("cand_begin", _i), ("cand_end", _i),
        ("equisampled", C.c_void_p),
    ]


class OrcPlanOutput(C.Structure):
    _fields_ = [
        ("result", HmpResult),
        ("totals", C.c_void_p), ("costs", C.c_void_p), ("seeds", C.c_void_p), ("poses", C.c_void_p),
        ("n_poses", C.c_void_p), ("generated", C.c_void_p), ("best_poses", C.c_void_p), ("forces", C.c_void_p),
        ("forces_candidate", _i), ("_pad", _i),
    ]


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB):
            subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle")], check=True)
        _lib = C.CDLL(_LIB)
        _lib.orc_plan.argtypes = [C.POINTER(OrcPlanInput), C.POINTER(OrcPlanOutput)]
        _lib.orc_plan.restype = C.c_int
        _lib.orc_num_candidates.argtypes = [C.POINTER(HmpSampling), C.c_int]
        _lib.orc_num_steps.argtypes = [C.POINTER(HmpParams), C.POINTER(HmpWorld)]
        for name, res in (("orc_wrap", _d), ("orc_yaw_roundtrip", _d), ("orc_factor_fov", _d),
                          ("orc_behaviour_strength_exp", _d), ("orc_passing_speed", _d), ("orc_direction", _d),
                          ("orc_len3", _d), ("orc_theta_alpha_beta_2011", _d), ("orc_theta_alpha_beta_2014", _d),
                          ("orc_relative_speed", _d), ("orc_personal_space", _d), ("orc_formation_space", _d),
                          ("orc_heading_disturbance", _d)):
            getattr(_lib, name).restype = res
        _lib.orc_wrap.argtypes = [_d]
        _lib.orc_yaw_roundtrip.argtypes = [_d]
        _lib.orc_factor_fov.argtypes = [_d, _d, C.c_int]
        _lib.orc_behaviour_strength_exp.argtypes = [_d, _d, _d, _d]
        _lib.orc_passing_speed.argtypes = [_d, _d, _d, _d]
    return _lib


def reference_has(sub: str) -> bool:
    """True when HMP_REFERENCE_DIR names a checkout of the original project that has `sub` (src, include)."""
    return bool(REFERENCE_DIR) and os.path.isdir(os.path.join(REFERENCE_DIR, sub))


def ref_available() -> bool:
    """True when oracle/_ref/libhmp_ref.so (the reference's own sources compiled against oracle/ref_shim) exists or can
    be built from the checkout HMP_REFERENCE_DIR names."""
    return os.path.exists(_REF_LIB) or reference_has("src")


def ref_lib() -> C.CDLL:
    global _ref_lib
    if _ref_lib is None:
        lib()  # libhmp_oracle.so first: the stand-ins' orc_tp_* hooks resolve against it
        if reference_has("src"):   # incremental; without the checkout a prebuilt library is used as is
            subprocess.run(["make", "-s", "-j8", "-C", os.path.join(ROOT, "oracle"), "ref"], check=True)
        _ref_lib = C.CDLL(_REF_LIB)
        _ref_lib.ref_plan.argtypes = [C.POINTER(OrcPlanInput), C.POINTER(OrcPlanOutput)]
        _ref_lib.ref_plan.restype = C.c_int
        _ref_lib.ref_fis_process.argtypes = [_d, _d, _d, _d, C.c_void_p]
        _ref_lib.ref_fis_process.restype = None
        _ref_lib.ref_num_candidates.argtypes = [C.POINTER(HmpSampling), C.c_int]
    return _ref_lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def num_candidates(sampling: HmpSampling, n_extra: int = 0) -> int:
    return lib().orc_num_candidates(C.byref(sampling), n_extra)


def equisampled_samples(params: HmpParams, world: HmpWorld, eq: HmpEquisampled) -> np.ndarray:
    """Velocity samples (vx, vy, vth) of the equisampled generator for this cycle, in generator order."""
    L = lib()
    L.orc_equisampled_samples.argtypes = [C.POINTER(HmpParams), C.POINTER(HmpWorld), C.POINTER(HmpEquisampled), C.c_void_p, C.c_int]
    n = L.orc_equisampled_samples(C.byref(params), C.byref(world), C.byref(eq), None, 0)
    out = np.zeros((max(n, 1), 3))
    L.orc_equisampled_samples(C.byref(params), C.byref(world), C.byref(eq), _p(out), n)
    return out[:n]


def num_equisampled(params: HmpParams, world: HmpWorld, eq: HmpEquisampled) -> int:
    return equisampled_samples(params, world, eq).shape[0]


def num_steps(params: HmpParams, world: HmpWorld) -> int:
    return lib().orc_num_steps(C.byref(params), C.byref(world))


def _make_input(params, scene, sampling, ex, n_extra, early_exit, cand_range, equisampled=None):
    inp = OrcPlanInput()
    inp.equisampled = C.addressof(equisampled) if equisampled is not None else None
    inp.params = C.pointer(params)
    inp.world = C.pointer(scene.world)
    inp.sampling = C.pointer(sampling)
    inp.extra = _p(ex)
    inp.n_extra = n_extra
    inp.size_x, inp.size_y = scene.size_x, scene.size_y
    inp.cells = _p(scene.cells)
    inp.origin_x, inp.origin_y, inp.resolution = scene.origin_x, scene.origin_y, scene.resolution
    for g in range(NUM_MAPGRIDS):
        inp.target_dist[g] = scene.grids[g].ctypes.data
        inp.highest_valid_cost_prev[g] = scene.hv_prev[g]
    inp.footprint_xy = _p(scene.footprint)
    inp.n_footprint = scene.footprint.shape[0]
    inp.early_exit = 1 if early_exit else 0
    inp.cand_begin, inp.cand_end = cand_range
    return inp


def score_trajectory(params: HmpParams, scene: Scene, sampling: HmpSampling, poses: np.ndarray, seed):
    """All critics of the oracle on an externally supplied trajectory. Returns (raw costs[14], total, hv[4])."""
    L = lib()
    L.orc_score_trajectory.argtypes = [C.POINTER(OrcPlanInput), C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p]
    inp = _make_input(params, scene, sampling, None, 0, False, (0, 0))
    poses = np.ascontiguousarray(poses, dtype=np.float64).reshape(-1, 3)
    sd = np.ascontiguousarray(seed, dtype=np.float64)
    raw = np.zeros(NUM_COSTS)
    total = np.zeros(1)
    hv = np.zeros(NUM_MAPGRIDS)
    L.orc_score_trajectory(C.byref(inp), _p(poses), poses.shape[0], _p(sd), _p(raw), _p(total), _p(hv))
    return raw, float(total[0]), hv


def plan(params: HmpParams, scene: Scene, sampling: HmpSampling, extra=None, early_exit: bool = False,
         cand_range=(0, 0), want=("totals", "costs", "seeds", "poses", "n_poses", "generated"), forces_candidate: int = -1,
         impl: str = "oracle", equisampled: HmpEquisampled = None):
    """Runs orc_plan (impl="oracle") or ref_plan (impl="ref": the reference's own sources, oracle/ref_driver.cpp) and
    returns a dict of numpy arrays (+ 'result': HmpResult)."""
    L = lib()
    fn = L.orc_plan if impl == "oracle" else ref_lib().ref_plan
    ex = None
    n_extra = 0
    if extra is not None:
        ex = np.ascontiguousarray(extra, dtype=np.float64).reshape(-1, NUM_AMPLIFIERS)
        n_extra = ex.shape[0]
    Cn = num_candidates(sampling, n_extra)
    if equisampled is not None and impl == "oracle":
        Cn += num_equisampled(params, scene.world, equisampled)
    T = num_steps(params, scene.world)
    inp = _make_input(params, scene, sampling, ex, n_extra, early_exit, cand_range, equisampled if impl == "oracle" else None)
    out = OrcPlanOutput()
    arrs = {}
    if "totals" in want:
        arrs["totals"] = np.full(Cn, np.nan)
        out.totals = _p(arrs["totals"])
    if "costs" in want:
        arrs["costs"] = np.full((Cn, NUM_COSTS), np.nan)
        out.costs = _p(arrs["costs"])
    if "seeds" in want:
        arrs["seeds"] = np.zeros((Cn, 3))
        out.seeds = _p(arrs["seeds"])
    if "poses" in want:
        arrs["poses"] = np.zeros((Cn, T, 3))
        out.poses = _p(arrs["poses"])
    if "n_poses" in want:
        arrs["n_poses"] = np.zeros(Cn, dtype=np.int32)
        out.n_poses = _p(arrs["n_poses"])
    if "generated" in want:
        arrs["generated"] = np.zeros(Cn, dtype=np.int32)
        out.generated = _p(arrs["generated"])
    arrs["best_poses"] = np.zeros((T, 3))
    out.best_poses = _p(arrs["best_poses"])
    out.forces_candidate = forces_candidate
    if forces_candidate >= 0:
        arrs["forces"] = np.zeros((T, 8))
        out.forces = _p(arrs["forces"])
    rc = fn(C.byref(inp), C.byref(out))
    assert rc == 0
    res = HmpResult()
    C.memmove(C.byref(res), C.byref(out.result), C.sizeof(HmpResult))
    arrs["result"] = res
    arrs["T"] = T
    arrs["C"] = Cn
    return arrs


def build_environment(env, robot_pose, pose_ref, shapes, vertices, people, groups):
    """orc_build_environment: same return as Planner.build_environment."""
    from humap_local_planner_b200.capi import _build_environment, HmpEnvParams
    L = lib()
    L.orc_build_environment.argtypes = [C.POINTER(HmpEnvParams), C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32,
                                        C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p]
    L.orc_build_environment.restype = C.c_int

    def check(rc):
        assert rc == 0

    return _build_environment(L.orc_build_environment, None, check, env, robot_pose, pose_ref, shapes, vertices, people, groups)


def force_grid(params: HmpParams, env, world: HmpWorld, positions, shapes, vertices) -> np.ndarray:
    from humap_local_planner_b200.capi import HmpEnvParams
    L = lib()
    L.orc_force_grid.argtypes = [C.POINTER(HmpParams), C.POINTER(HmpEnvParams), C.POINTER(HmpWorld), C.c_void_p, C.c_int32, C.c_void_p,
                                 C.c_int32, C.c_void_p, C.c_int32, C.c_void_p]
    L.orc_force_grid.restype = C.c_int
    pos = np.ascontiguousarray(positions, dtype=np.float64).reshape(-1, 2)
    verts = np.ascontiguousarray(vertices, dtype=np.float64).reshape(-1, 2)
    out = np.zeros((pos.shape[0], 8))
    ns = len(shapes) if shapes is not None else 0
    assert L.orc_force_grid(C.byref(params), C.byref(env), C.byref(world), _p(pos), pos.shape[0], C.cast(shapes, C.c_void_p) if ns else None,
                            ns, _p(verts) if verts.size else None, verts.shape[0], _p(out)) == 0
    return out


def cost_cloud(params: HmpParams, scene: Scene, sampling: HmpSampling, impl: str = "oracle"):
    """HumapPlanner::computeCellCost per cell: (cloud [size_y][size_x][6] float32, valid [size_y][size_x] bool)."""
    L = lib() if impl == "oracle" else ref_lib()
    fn = L.orc_cost_cloud if impl == "oracle" else L.ref_cost_cloud
    fn.argtypes = [C.POINTER(OrcPlanInput), C.c_void_p, C.c_void_p]
    fn.restype = C.c_int
    inp = _make_input(params, scene, sampling, None, 0, False, (0, 0))
    n = scene.size_x * scene.size_y
    out = np.zeros((n, 6), dtype=np.float32)
    valid = np.zeros(n, dtype=np.uint8)
    assert fn(C.byref(inp), _p(out), _p(valid)) == 0
    return out.reshape(scene.size_y, scene.size_x, 6), valid.reshape(scene.size_y, scene.size_x).astype(bool)


def plan_sampled(params, scene, sampling, indices, equisampled=None):
    """Oracle results for an explicit list of candidate indices (one orc_plan call per candidate)."""
    out = {"totals": [], "costs": [], "poses": [], "seeds": [], "n_poses": []}
    for i in indices:
        r = plan(params, scene, sampling, cand_range=(int(i), int(i) + 1), equisampled=equisampled)
        for k in out:
            out[k].append(r[k][int(i)])
    return {k: np.array(v) for k, v in out.items()}


def plan_all_threaded(params, scene, sampling, n_threads=None, want=("totals",)):
    """Full-grid oracle totals, split over host threads (ctypes releases the GIL during orc_plan)."""
    import concurrent.futures as cf
    import os as _os
    Cn = num_candidates(sampling)
    n_threads = n_threads or min(64, _os.cpu_count() or 1)
    bounds = np.linspace(0, Cn, n_threads * 4 + 1).astype(int)
    totals = np.full(Cn, np.nan)

    def work(k):
        a, b = int(bounds[k]), int(bounds[k + 1])
        if b > a:
            r = plan(params, scene, sampling, cand_range=(a, b), want=("totals",))
            totals[a:b] = r["totals"][a:b]

    with cf.ThreadPoolExecutor(n_threads) as ex_:
        list(ex_.map(work, range(len(bounds) - 1)))
    return totals


OP_NAMES = ("add", "mul", "div", "sqrt", "exp", "trig", "atan2", "cmp", "rnd")
_count_lib = None


def count_ops(params, scene, sampling, indices):
    """Instrumented floating-point operation count of the oracle (oracle/hmp_oracle_count.cpp: the oracle's source text over a
    counting scalar) for the listed social candidates. Returns a dict: ops_rollout / ops_scoring (name -> count, summed over
    the candidates), steps_rolled, n_generated, totals (bit-identical to orc_plan's)."""
    global _count_lib
    if _count_lib is None:
        path = os.path.join(ROOT, "oracle", "_build", "libhmp_oracle_count.so")
        if not os.path.exists(path):
            subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle")], check=True)
        _count_lib = C.CDLL(path)
        _count_lib.orc_count_plan.restype = C.c_int
        _count_lib.orc_count_plan.argtypes = [C.POINTER(OrcPlanInput), C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                              C.c_void_p, C.c_void_p]
        assert _count_lib.orc_count_num_ops() == len(OP_NAMES)
    idx = np.ascontiguousarray(indices, dtype=np.int32)
    inp = _make_input(params, scene, sampling, None, 0, False, (0, 0), None)
    ro = np.zeros(len(OP_NAMES), dtype=np.uint64)
    sc = np.zeros(len(OP_NAMES), dtype=np.uint64)
    steps = np.zeros(1, dtype=np.uint64)
    ngen = np.zeros(1, dtype=np.int32)
    totals = np.full(len(idx), np.nan)
    rc = _count_lib.orc_count_plan(C.byref(inp), _p(idx), len(idx), _p(ro), _p(sc), _p(steps), _p(ngen), _p(totals))
    assert rc == 0
    return {"ops_rollout": {n: int(v) for n, v in zip(OP_NAMES, ro)}, "ops_scoring": {n: int(v) for n, v in zip(OP_NAMES, sc)},
            "steps_rolled": int(steps[0]), "n_generated": int(ngen[0]), "totals": totals}
