"""ctypes binding of the C ABI in include/hmp_planner.h (the drop-in boundary of the sampling + scoring path).

The structures mirror the header field by field; `Planner` is a thin convenience wrapper over the
`hmp_*` entry points used by tests/ and bench.py. The library is CUDA-only: loading fails loudly
if the shared object is missing and `Planner()` raises if no sm_100 device is usable. There is no
CPU fallback anywhere in this package.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Sequence

import numpy as np

NUM_AMPLIFIERS = 10
MAX_AMP_VALUES = 64
NUM_COSTS = 14
NUM_MAPGRIDS = 4
MAX_FOOTPRINT = 64
MAX_STEPS = 512

COST_NAMES = (
    "obstacle", "path", "goal", "alignment", "goal_front", "unsaturated", "backward", "ttc",
    "heading_change", "vel_smoothness", "heading_dist", "personal_space", "fformation", "passing_speed",
)
AMP_NAMES = ("speed", "an", "bn", "cn", "ap", "bp", "cp", "aw", "bw", "as")

HMP_OK, HMP_E_INVALID, HMP_E_CUDA, HMP_E_NOT_READY, HMP_E_CAPACITY = 0, -1, -2, -3, -4

_d, _i = C.c_double, C.c_int32


class HmpLimits(C.Structure):
    _fields_ = [(n, _d) for n in (
        "max_vel_trans", "min_vel_trans", "max_vel_x", "min_vel_x", "max_vel_y", "min_vel_y",
        "max_vel_theta", "min_vel_theta", "acc_lim_x", "acc_lim_y", "acc_lim_theta",
        "twist_rotation_compensation")] + [("maintain_vel_components_rate", _i), ("_pad", _i)]


class HmpGeneral(C.Structure):
    _fields_ = [(n, _d) for n in ("sim_time", "sim_granularity", "angular_sim_granularity", "sim_period",
                                  "people_prediction_dt")] + [("discretize_by_time", _i), ("_pad", _i)]


class HmpSfm(C.Structure):
    _fields_ = [(n, _d) for n in (
        "fov", "mass", "internal_force_factor", "static_interaction_force_factor",
        "dynamic_interaction_force_factor", "min_force", "max_force", "speed_desired", "relaxation_time",
        "an", "bn", "cn", "ap", "bp", "cp", "aw", "bw")] + [
        ("fov_factor_method", _i), ("filter_forces", _i), ("disable_interaction_forces", _i), ("_pad", _i)]


class HmpFis(C.Structure):
    _fields_ = [("force_factor", _d), ("human_action_range", _d), ("fov", _d), ("fov_factor_method", _i), ("_pad", _i)]


class HmpCosts(C.Structure):
    _fields_ = [
        ("scale", _d * NUM_COSTS),
        ("occdist_separation", _d), ("occdist_separation_kernel", _i), ("occdist_sum_scores", _i),
        ("xshift", _d * NUM_MAPGRIDS), ("yshift", _d * NUM_MAPGRIDS), ("stop_on_failure", _i * NUM_MAPGRIDS),
        ("neighbour_kernel_size", _i * NUM_MAPGRIDS), ("neighbour_cost_multiplier", _d * NUM_MAPGRIDS),
        ("unsat_max_trans_vel", _d), ("unsat_max_vel_x", _d), ("unsat_max_vel_y", _d),
        ("backward_penalty", _d), ("ttc_rollout_time", _d), ("ttc_collision_distance", _d),
        ("hd_fov_person", _d), ("hd_person_model_radius", _d), ("hd_robot_circumradius", _d), ("hd_max_speed", _d),
        ("ps_max_speed", _d), ("ps_min_dist", _d),
        ("unsat_whole_horizon", _i), ("hd_whole_horizon", _i), ("psi_whole_horizon", _i),
        ("fsi_whole_horizon", _i), ("ps_whole_horizon", _i), ("_pad", _i),
    ]


class HmpParams(C.Structure):
    _fields_ = [("limits", HmpLimits), ("general", HmpGeneral), ("sfm", HmpSfm), ("fis", HmpFis), ("costs", HmpCosts)]


class HmpObstacle(C.Structure):
    _fields_ = [(n, _d) for n in ("robot_x", "robot_y", "robot_yaw", "obj_x", "obj_y", "obj_yaw", "vx", "vy", "vth")] + [
        ("force_dynamic", _i), ("_pad", _i)]


class HmpPerson(C.Structure):
    _fields_ = [(n, _d) for n in ("x", "y", "yaw", "vx", "vy", "vth", "cov_xx", "cov_xy", "cov_yx", "cov_yy")]


class HmpGroup(C.Structure):
    _fields_ = [(n, _d) for n in ("x", "y", "yaw", "span_x", "span_y", "cov_xx", "cov_xy", "cov_yy")]


class HmpWorld(C.Structure):
    _fields_ = [(n, _d) for n in (
        "robot_x", "robot_y", "robot_yaw", "vel_x", "vel_y", "vel_th",
        "goal_local_x", "goal_local_y", "goal_local_yaw", "goal_x", "goal_y", "goal_yaw")] + [
        ("obstacles", C.POINTER(HmpObstacle)), ("people", C.POINTER(HmpPerson)), ("groups", C.POINTER(HmpGroup)),
        ("n_obstacles", _i), ("n_people", _i), ("n_groups", _i), ("_pad", _i)]


class HmpSampling(C.Structure):
    _fields_ = [("amp_min", _d * NUM_AMPLIFIERS), ("amp_max", _d * NUM_AMPLIFIERS),
                ("amp_granularity", _d * NUM_AMPLIFIERS)]


class HmpSample(C.Structure):
    _fields_ = [("amp", _d * NUM_AMPLIFIERS)]


class HmpSceneCosts(C.Structure):
    """Per-world scales and MapGrid shifts of a batch (hmp_set_scene_costs); same meaning as the fields of HmpCosts."""
    _fields_ = [("scale", _d * NUM_COSTS), ("xshift", _d * NUM_MAPGRIDS), ("yshift", _d * NUM_MAPGRIDS)]


class HmpResult(C.Structure):
    _fields_ = [
        ("status", _i), ("best_index", _i), ("n_candidates", _i), ("n_generated", _i), ("n_valid", _i), ("n_poses", _i),
        ("best_total", _d), ("costs", _d * NUM_COSTS), ("xv", _d), ("yv", _d), ("thetav", _d), ("time_delta", _d),
        ("amplifiers", _d * NUM_AMPLIFIERS), ("highest_valid_cost", _d * NUM_MAPGRIDS),
        ("gpu_ms", _d), ("gpu_ms_select", _d),
        ("n_social", _i), ("_pad", _i),
    ]


class HmpShape(C.Structure):
    """One obstacle of the costmap_converter container (teb point / circle / line / polygon)."""
    _fields_ = [("type", _i), ("n_vertices", _i), ("first_vertex", _i), ("_pad", _i), ("x", _d), ("y", _d), ("x2", _d), ("y2", _d),
                ("radius", _d), ("vx", _d), ("vy", _d)]


MAX_ENV_POLYGON = 16


class HmpEnvParams(C.Structure):
    _fields_ = [("robot_model", _i), ("obstacles_closest_num", _i), ("people_closest_num", _i), ("groups_closest_num", _i),
                ("robot_radius", _d), ("person_model_radius", _d), ("obstacle_extension_multiplier", _d),
                ("ttc_collision_distance", _d), ("person_containment_rate", _d), ("obstacles_force_dynamic", _i),
                ("people_force_dynamic", _i), ("two_circles", _d * 4), ("line_xy", _d * 4), ("n_polygon", _i), ("_pad", _i),
                ("polygon_xy", _d * (2 * MAX_ENV_POLYGON))]


SHAPE_POINT, SHAPE_CIRCLE, SHAPE_LINE, SHAPE_POLYGON = 0, 1, 2, 3
ROBOT_POINT, ROBOT_CIRCULAR, ROBOT_TWO_CIRCLES, ROBOT_LINE, ROBOT_POLYGON = 0, 1, 2, 3, 4


class HmpEquisampled(C.Structure):
    """TrajectoryGeneration's equisampled-velocity generator (humap_config.h:154-174)."""
    _fields_ = [("enabled", _i), ("vx_samples", _i), ("vy_samples", _i), ("vth_samples", _i), ("min_vel_x", _d),
                ("continued_acceleration", _i), ("_pad", _i)]


# Every symbol include/hmp_planner.h declares (checked by tests/test_capi_symbols.py)
ABI_SYMBOLS = (
    "hmp_create", "hmp_destroy", "hmp_last_error", "hmp_abi_version", "hmp_set_params", "hmp_set_costmap",
    "hmp_set_mapgrid", "hmp_set_footprint", "hmp_plan", "hmp_plan_batch", "hmp_replan_resident",
    "hmp_get_explored_totals", "hmp_explain", "hmp_debug_world_to_map", "hmp_debug_footprint_cost",
    "hmp_debug_fis", "hmp_debug_last_forces", "hmp_num_steps", "hmp_launch_count", "hmp_set_precision", "hmp_compute_mapgrid", "hmp_get_mapgrid",
    "hmp_set_refinement", "hmp_last_num_leaders", "hmp_set_equisampled", "hmp_compute_cost_cloud", "hmp_build_environment", "hmp_compute_force_grid", "hmp_debug_measure_fp32_peak",
    "hmp_set_sweep_layout", "hmp_last_sweep_mode", "hmp_last_num_leaders_round2",
    "hmp_compute_mapgrid_batch", "hmp_set_mapgrids_batch_f32", "hmp_last_num_scenes", "hmp_last_fallback_rounds",
    "hmp_debug_sweep_candidate", "hmp_host_alloc", "hmp_host_free",
    "hmp_set_escalation", "hmp_last_unreliable_leaders", "hmp_last_escalated", "hmp_set_scene_costs",
)

_LIB_PATH = os.environ.get("HMP_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib", "libhmp_planner.so")
_lib = None


def lib_path() -> str:
    return _LIB_PATH


def load_library() -> C.CDLL:
    """Loads lib/libhmp_planner.so (built by __graft_entry__.build()). Raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise RuntimeError(
            f"{_LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'`. "
            "humap_local_planner_b200 has no CPU fallback.")
    lib = C.CDLL(_LIB_PATH)
    P = C.POINTER
    lib.hmp_create.restype = C.c_void_p
    lib.hmp_create.argtypes = [C.c_int]
    lib.hmp_destroy.restype = None
    lib.hmp_destroy.argtypes = [C.c_void_p]
    lib.hmp_last_error.restype = C.c_char_p
    lib.hmp_last_error.argtypes = []
    lib.hmp_abi_version.restype = C.c_int
    lib.hmp_set_params.argtypes = [C.c_void_p, P(HmpParams)]
    lib.hmp_set_costmap.argtypes = [C.c_void_p, C.c_void_p, _i, _i, _d, _d, _d]
    lib.hmp_set_mapgrid.argtypes = [C.c_void_p, _i, C.c_void_p, _d]
    lib.hmp_set_footprint.argtypes = [C.c_void_p, C.c_void_p, _i]
    lib.hmp_plan.argtypes = [C.c_void_p, P(HmpWorld), P(HmpSampling), C.c_void_p, _i, P(HmpResult), C.c_void_p, _i]
    lib.hmp_plan_batch.argtypes = [C.c_void_p, P(HmpWorld), _i, C.c_void_p, C.c_void_p, C.c_void_p, P(HmpSampling),
                                   P(HmpResult)]
    lib.hmp_replan_resident.argtypes = [C.c_void_p, P(HmpResult), _i]
    lib.hmp_compute_mapgrid_batch.argtypes = [C.c_void_p, _i, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.hmp_compute_mapgrid_batch.restype = C.c_int
    lib.hmp_set_mapgrids_batch_f32.argtypes = [C.c_void_p, _i, C.c_void_p]
    lib.hmp_set_mapgrids_batch_f32.restype = C.c_int
    lib.hmp_set_escalation.argtypes = [C.c_void_p, _i]
    lib.hmp_set_escalation.restype = C.c_int
    lib.hmp_set_scene_costs.argtypes = [C.c_void_p, C.c_void_p, _i]
    lib.hmp_set_scene_costs.restype = C.c_int
    for name in ("hmp_last_num_scenes", "hmp_last_fallback_rounds", "hmp_last_num_leaders_round2", "hmp_last_unreliable_leaders",
                 "hmp_last_escalated"):
        getattr(lib, name).argtypes = [C.c_void_p]
        getattr(lib, name).restype = C.c_int
    lib.hmp_get_explored_totals.argtypes = [C.c_void_p, C.c_void_p, _i]
    lib.hmp_explain.argtypes = [C.c_void_p, C.c_void_p, _i, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.hmp_debug_world_to_map.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, _i, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.hmp_debug_footprint_cost.argtypes = [C.c_void_p, C.c_void_p, _i, C.c_void_p]
    lib.hmp_debug_fis.argtypes = [C.c_void_p, C.c_void_p, _i, C.c_void_p]
    lib.hmp_debug_last_forces.argtypes = [C.c_void_p, _i, C.c_void_p]
    lib.hmp_num_steps.argtypes = [C.c_void_p]
    lib.hmp_set_precision.argtypes = [C.c_void_p, _i]
    lib.hmp_compute_mapgrid.argtypes = [C.c_void_p, _i, C.c_void_p, _i, _i, _d]
    lib.hmp_compute_mapgrid.restype = C.c_int
    lib.hmp_get_mapgrid.argtypes = [C.c_void_p, _i, C.c_void_p]
    lib.hmp_get_mapgrid.restype = C.c_int
    lib.hmp_set_precision.restype = C.c_int
    lib.hmp_set_refinement.argtypes = [C.c_void_p, _d, _i]
    lib.hmp_set_sweep_layout.argtypes = [C.c_void_p, _i]
    lib.hmp_set_sweep_layout.restype = C.c_int
    lib.hmp_last_sweep_mode.argtypes = [C.c_void_p]
    lib.hmp_last_sweep_mode.restype = C.c_int
    lib.hmp_set_refinement.restype = C.c_int
    lib.hmp_set_equisampled.argtypes = [C.c_void_p, C.c_void_p]
    lib.hmp_set_equisampled.restype = C.c_int
    lib.hmp_build_environment.argtypes = [C.c_void_p, P(HmpEnvParams), C.c_void_p, C.c_void_p, C.c_void_p, _i, C.c_void_p, _i,
                                          C.c_void_p, _i, C.c_void_p, _i, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_void_p]
    lib.hmp_build_environment.restype = C.c_int
    lib.hmp_compute_force_grid.argtypes = [C.c_void_p, P(HmpEnvParams), P(HmpWorld), C.c_void_p, _i, C.c_void_p, _i, C.c_void_p, _i,
                                           C.c_void_p]
    lib.hmp_compute_force_grid.restype = C.c_int
    lib.hmp_debug_measure_fp32_peak.argtypes = [C.c_void_p, C.c_void_p]
    lib.hmp_debug_measure_fp32_peak.restype = C.c_int
    lib.hmp_compute_cost_cloud.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    lib.hmp_compute_cost_cloud.restype = C.c_int
    lib.hmp_last_num_leaders.argtypes = [C.c_void_p]
    lib.hmp_last_num_leaders.restype = C.c_int
    lib.hmp_launch_count.restype = C.c_int64
    lib.hmp_launch_count.argtypes = [C.c_void_p]
    for name in ("hmp_set_params", "hmp_set_costmap", "hmp_set_mapgrid", "hmp_set_footprint", "hmp_plan",
                 "hmp_plan_batch", "hmp_replan_resident", "hmp_get_explored_totals", "hmp_explain",
                 "hmp_debug_world_to_map", "hmp_debug_footprint_cost", "hmp_debug_fis", "hmp_debug_last_forces",
                 "hmp_num_steps"):
        getattr(lib, name).restype = C.c_int
    _lib = lib
    return lib


class PinnedArray:
    """numpy view of page-locked host memory (hmp_host_alloc); keep the object alive as long as the array is used."""

    def __init__(self, shape, dtype):
        lib = load_library()
        lib.hmp_host_alloc.restype = C.c_void_p
        lib.hmp_host_alloc.argtypes = [C.c_size_t]
        lib.hmp_host_free.restype = None
        lib.hmp_host_free.argtypes = [C.c_void_p]
        self._lib = lib
        dt = np.dtype(dtype)
        n = int(np.prod(shape)) * dt.itemsize
        self._ptr = lib.hmp_host_alloc(n)
        if not self._ptr:
            raise MemoryError(lib.hmp_last_error().decode())
        buf = (C.c_char * max(n, 1)).from_address(self._ptr)
        self.array = np.frombuffer(buf, dtype=dt, count=int(np.prod(shape))).reshape(shape)

    def __del__(self):
        try:
            if getattr(self, "_ptr", None):
                self.array = None
                self._lib.hmp_host_free(self._ptr)
                self._ptr = None
        except Exception:
            pass


class HmpError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"hmp error {code}: {message}")
        self.code = code


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class Scene:
    """Host-side container of one planning cycle's inputs; keeps the ctypes arrays alive."""

    def __init__(self, world: HmpWorld, obstacles, people, groups, cells: np.ndarray, origin_x: float, origin_y: float,
                 resolution: float, grids: Sequence[np.ndarray], footprint: np.ndarray,
                 hv_prev: Sequence[float] = (0.0, 0.0, 0.0, 0.0)):
        self.world = world
        self._obstacles, self._people, self._groups = obstacles, people, groups
        self.cells = np.ascontiguousarray(cells, dtype=np.uint8)
        self.size_y, self.size_x = self.cells.shape
        self.origin_x, self.origin_y, self.resolution = float(origin_x), float(origin_y), float(resolution)
        self.grids = [np.ascontiguousarray(g, dtype=np.float64) for g in grids]
        self.footprint = np.ascontiguousarray(footprint, dtype=np.float64)
        self.hv_prev = tuple(float(v) for v in hv_prev)


def _build_environment(fn, ctx, check, env, robot_pose, pose_ref, shapes, vertices, people, groups):
    """Shared marshalling of hmp_build_environment / orc_build_environment (same argument list after the context)."""
    rp = np.ascontiguousarray(robot_pose, dtype=np.float64)
    pr = np.ascontiguousarray(pose_ref, dtype=np.float64)
    verts = np.ascontiguousarray(vertices, dtype=np.float64).reshape(-1, 2)
    ns = len(shapes) if shapes is not None else 0
    n_p = len(people) if people is not None else 0
    n_g = len(groups) if groups is not None else 0
    cap = ns + n_p
    out = (HmpObstacle * max(1, cap))()
    n_out = C.c_int32(cap)
    psel = np.zeros(max(1, n_p), dtype=np.int32)
    gsel = np.zeros(max(1, n_g), dtype=np.int32)
    n_ps, n_gs = C.c_int32(0), C.c_int32(0)
    args = [C.byref(env), _ptr(rp), _ptr(pr), C.cast(shapes, C.c_void_p) if ns else None, ns, _ptr(verts) if verts.size else None,
            verts.shape[0], C.cast(people, C.c_void_p) if n_p else None, n_p, C.cast(groups, C.c_void_p) if n_g else None, n_g,
            C.cast(out, C.c_void_p), C.byref(n_out), _ptr(psel), C.byref(n_ps), _ptr(gsel), C.byref(n_gs)]
    rc = fn(ctx, *args) if ctx is not None else fn(*args)
    check(rc)
    return out, n_out.value, psel[:n_ps.value].copy(), gsel[:n_gs.value].copy()


class Planner:
    """One GPU context (hmp_create). Not re-entrant, like the reference (it plans under cfg_->getMutex())."""

    def __init__(self, device: int = 0):
        self._lib = load_library()
        self._ctx = self._lib.hmp_create(int(device))
        if not self._ctx:
            raise HmpError(HMP_E_CUDA, self._lib.hmp_last_error().decode())
        self.device = device

    def close(self):
        if getattr(self, "_ctx", None):
            self._lib.hmp_destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc != 0:
            raise HmpError(rc, self._lib.hmp_last_error().decode())

    # ---- configuration -------------------------------------------------------------------------
    def set_params(self, params: HmpParams):
        self._check(self._lib.hmp_set_params(self._ctx, C.byref(params)))

    def set_precision(self, mode):
        """False / 0: FP32 object loops; True / 1: FP64 (parity mode); 2: FP32 sweep + FP64 refinement of the leaders."""
        self._check(self._lib.hmp_set_precision(self._ctx, int(mode)))

    def set_refinement(self, rel_window: float = 0.02, max_leaders: int = 0):
        self._check(self._lib.hmp_set_refinement(self._ctx, float(rel_window), int(max_leaders)))

    def set_sweep_layout(self, layout: int = 0):
        """FP32 sweep: 0 automatic, 1 one warp per candidate, 2 one thread per candidate."""
        self._check(self._lib.hmp_set_sweep_layout(self._ctx, int(layout)))

    def last_num_leaders_round2(self) -> int:
        """Candidates re-scored by the second refinement round of the last single-scene plan in mode 2."""
        return int(self._lib.hmp_last_num_leaders_round2(self._ctx))

    def set_escalation(self, min_unreliable_leaders: int = 0):
        """Mode 2: redo a plan as an exact FP64 sweep when at least this many leaders contradict their FP32 totals (0: never)."""
        self._check(self._lib.hmp_set_escalation(self._ctx, int(min_unreliable_leaders)))

    def last_unreliable_leaders(self) -> int:
        return int(self._lib.hmp_last_unreliable_leaders(self._ctx))

    def last_escalated(self) -> int:
        return int(self._lib.hmp_last_escalated(self._ctx))

    def last_fallback_rounds(self) -> int:
        """Extra refinement rounds the last plan needed because FP64 rejected every leader (mode 2)."""
        return int(self._lib.hmp_last_fallback_rounds(self._ctx))

    def last_num_scenes(self) -> int:
        return int(self._lib.hmp_last_num_scenes(self._ctx))

    def last_sweep_mode(self) -> int:
        """0 = the last main sweep ran one warp per candidate, else the block size of the thread-per-candidate kernel."""
        return int(self._lib.hmp_last_sweep_mode(self._ctx))

    def set_equisampled(self, eq: Optional["HmpEquisampled"]):
        """Second generator of the pool (equisampled velocities); None turns it off."""
        self._check(self._lib.hmp_set_equisampled(self._ctx, C.byref(eq) if eq is not None else None))

    def cost_cloud(self):
        """HumapPlanner::computeCellCost for every cell: (cloud [size_y][size_x][6] float32, valid [size_y][size_x] bool)."""
        n = self._size_y * self._size_x
        out = np.zeros((n, 6), dtype=np.float32)
        valid = np.zeros(n, dtype=np.uint8)
        self._check(self._lib.hmp_compute_cost_cloud(self._ctx, _ptr(out), _ptr(valid)))
        return out.reshape(self._size_y, self._size_x, 6), valid.reshape(self._size_y, self._size_x).astype(bool)

    def build_environment(self, env: HmpEnvParams, robot_pose, pose_ref, shapes, vertices: np.ndarray, people, groups):
        """HumapPlanner::createEnvironmentModel on the device. shapes / people / groups: ctypes arrays (or None).
        Returns (obstacles ctypes array, n_obstacles, selected people indices, selected group indices)."""
        return _build_environment(self._lib.hmp_build_environment, self._ctx, self._check, env, robot_pose, pose_ref, shapes, vertices,
                                  people, groups)

    def force_grid(self, env: HmpEnvParams, world: HmpWorld, positions: np.ndarray, shapes, vertices: np.ndarray) -> np.ndarray:
        """HumapPlanner::computeForceAtPosition for every position: [n][8] (internal, dynamic, static, human-action xy)."""
        pos = np.ascontiguousarray(positions, dtype=np.float64).reshape(-1, 2)
        verts = np.ascontiguousarray(vertices, dtype=np.float64).reshape(-1, 2)
        out = np.zeros((pos.shape[0], 8))
        ns = len(shapes) if shapes is not None else 0
        self._check(self._lib.hmp_compute_force_grid(self._ctx, C.byref(env), C.byref(world), _ptr(pos), pos.shape[0],
                                                     C.cast(shapes, C.c_void_p) if ns else None, ns,
                                                     _ptr(verts) if verts.size else None, verts.shape[0], _ptr(out)))
        return out

    def measure_fp32_peak(self) -> float:
        """Measured FP32 FFMA throughput of this GPU in TFLOP/s (independent FMA chains, 2 x 256 threads per SM)."""
        out = C.c_double(0.0)
        self._check(self._lib.hmp_debug_measure_fp32_peak(self._ctx, C.byref(out)))
        return float(out.value)

    def last_num_leaders(self) -> int:
        return int(self._lib.hmp_last_num_leaders(self._ctx))

    def set_costmap(self, cells: np.ndarray, origin_x: float, origin_y: float, resolution: float):
        cells = np.ascontiguousarray(cells, dtype=np.uint8)
        sy, sx = cells.shape
        self._size_y, self._size_x = sy, sx
        self._check(self._lib.hmp_set_costmap(self._ctx, _ptr(cells), sx, sy, origin_x, origin_y, resolution))

    def set_mapgrid(self, grid: int, target_dist: np.ndarray, hv_prev: float = 0.0):
        t = np.ascontiguousarray(target_dist, dtype=np.float64)
        self._check(self._lib.hmp_set_mapgrid(self._ctx, grid, _ptr(t), float(hv_prev)))

    def compute_mapgrid(self, grid: int, plan_xy: np.ndarray, local_goal: bool, hv_prev: float = 0.0):
        p = np.ascontiguousarray(plan_xy, dtype=np.float64).reshape(-1, 2)
        self._check(self._lib.hmp_compute_mapgrid(self._ctx, grid, _ptr(p), p.shape[0], 1 if local_goal else 0, float(hv_prev)))

    def get_mapgrid(self, grid: int, shape) -> np.ndarray:
        out = np.zeros(shape, dtype=np.float64)
        self._check(self._lib.hmp_get_mapgrid(self._ctx, grid, _ptr(out)))
        return out

    def set_footprint(self, xy: np.ndarray):
        xy = np.ascontiguousarray(xy, dtype=np.float64).reshape(-1, 2)
        self._check(self._lib.hmp_set_footprint(self._ctx, _ptr(xy), xy.shape[0]))

    def set_scene(self, scene: Scene):
        self.set_costmap(scene.cells, scene.origin_x, scene.origin_y, scene.resolution)
        for g in range(NUM_MAPGRIDS):
            self.set_mapgrid(g, scene.grids[g], scene.hv_prev[g])
        self.set_footprint(scene.footprint)

    # ---- hot path ------------------------------------------------------------------------------
    def plan(self, world: HmpWorld, sampling: HmpSampling, extra: Optional[np.ndarray] = None, want_poses: bool = True):
        res = HmpResult()
        n_extra = 0
        ex = None
        if extra is not None:
            ex = np.ascontiguousarray(extra, dtype=np.float64).reshape(-1, NUM_AMPLIFIERS)
            n_extra = ex.shape[0]
        poses = np.zeros((MAX_STEPS, 3), dtype=np.float64) if want_poses else None
        self._check(self._lib.hmp_plan(self._ctx, C.byref(world), C.byref(sampling), _ptr(ex), n_extra, C.byref(res),
                                       _ptr(poses), MAX_STEPS if want_poses else 0))
        return res, (poses[: max(res.n_poses, 0)] if want_poses else None)

    def set_scene_costs(self, costs):
        """Per-world scales / MapGrid shifts of the following plan_batch calls: a sequence (or ctypes array) of HmpSceneCosts,
        entry s for scene s. None or an empty sequence clears the table: every world uses the scales / shifts of set_params."""
        n = 0 if costs is None else len(costs)
        arr = None
        if n:
            arr = costs if isinstance(costs, C.Array) else (HmpSceneCosts * n)(*costs)
        self._check(self._lib.hmp_set_scene_costs(self._ctx, arr, n))

    def plan_batch(self, worlds, cells: Optional[np.ndarray], grids: Optional[Sequence[np.ndarray]],
                   sampling: HmpSampling, hv_prev: Optional[np.ndarray] = None, scene_costs=None):
        """worlds: sequence of HmpWorld or a ctypes HmpWorld array; cells: [n][size_y][size_x] uint8 or None (costmaps of an
        earlier batch call stay); grids: 4 arrays [n][size_y][size_x] float64, or None (grids left resident by
        compute_mapgrid_batch / set_mapgrids_batch_f32 / an earlier batch). scene_costs: if given, set_scene_costs(scene_costs)
        first; the table then stays for later batches until it is set again or cleared."""
        if scene_costs is not None:
            self.set_scene_costs(scene_costs)
        n = len(worlds)
        arr = worlds if isinstance(worlds, C.Array) else (HmpWorld * n)(*worlds)
        cells = None if cells is None else np.ascontiguousarray(cells, dtype=np.uint8)
        gp = None
        if grids is not None:
            gs = [np.ascontiguousarray(g, dtype=np.float64) for g in grids]
            gp = (C.c_void_p * NUM_MAPGRIDS)(*[g.ctypes.data for g in gs])
        hv = None if hv_prev is None else np.ascontiguousarray(hv_prev, dtype=np.float64)
        res = (HmpResult * n)()
        self._check(self._lib.hmp_plan_batch(self._ctx, arr, n, _ptr(cells), gp, _ptr(hv), C.byref(sampling), res))
        return list(res)

    def compute_mapgrid_batch(self, cells: Optional[np.ndarray], plans, local_goal: Sequence[bool], n_scenes: Optional[int] = None):
        """Wave fronts of n_scenes x 4 grids on the device. plans[g] = (plan_xy [total poses][2], plan_start [n_scenes + 1])."""
        if cells is not None:
            cells = np.ascontiguousarray(cells, dtype=np.uint8)
            n_scenes = cells.shape[0]
        xy = [np.ascontiguousarray(p[0], dtype=np.float64).reshape(-1, 2) for p in plans]
        st = [np.ascontiguousarray(p[1], dtype=np.int32) for p in plans]
        assert all(s.shape[0] == n_scenes + 1 for s in st)
        xp = (C.c_void_p * NUM_MAPGRIDS)(*[a.ctypes.data for a in xy])
        sp = (C.c_void_p * NUM_MAPGRIDS)(*[a.ctypes.data for a in st])
        lg = np.ascontiguousarray([1 if b else 0 for b in local_goal], dtype=np.int32)
        self._check(self._lib.hmp_compute_mapgrid_batch(self._ctx, int(n_scenes), _ptr(cells), xp, sp, _ptr(lg)))

    def set_mapgrids_batch_f32(self, grids: Sequence[np.ndarray]):
        """grids: 4 float32 arrays [n][size_y][size_x] (ideally in pinned memory), uploaded without conversion."""
        gs = [np.ascontiguousarray(g, dtype=np.float32) for g in grids]
        gp = (C.c_void_p * NUM_MAPGRIDS)(*[g.ctypes.data for g in gs])
        self._check(self._lib.hmp_set_mapgrids_batch_f32(self._ctx, int(gs[0].shape[0]), gp))

    def replan_resident(self, n_scenes: Optional[int] = None):
        """Re-runs the last plan on the resident scene data; returns one HmpResult per scene of that plan."""
        n_last = self.last_num_scenes()
        if n_last < 0:
            raise HmpError(HMP_E_NOT_READY, "no previous plan to re-run")
        if n_scenes is not None and n_scenes != n_last:
            raise HmpError(HMP_E_INVALID, f"the last plan had {n_last} scene(s), not {n_scenes}")
        res = (HmpResult * n_last)()
        self._check(self._lib.hmp_replan_resident(self._ctx, res, n_last))
        return list(res)

    # ---- diagnostics ---------------------------------------------------------------------------
    def explored_totals(self, n: int) -> np.ndarray:
        out = np.zeros(n, dtype=np.float64)
        self._check(self._lib.hmp_get_explored_totals(self._ctx, _ptr(out), n))
        return out

    def num_steps(self) -> int:
        return int(self._lib.hmp_num_steps(self._ctx))

    def explain(self, indices: Sequence[int], with_forces: bool = False):
        idx = np.ascontiguousarray(indices, dtype=np.int32)
        n = idx.shape[0]
        T = self.num_steps()
        costs = np.zeros((n, NUM_COSTS))
        seeds = np.zeros((n, 3))
        poses = np.zeros((n, T, 3))
        nsteps = np.zeros(n, dtype=np.int32)
        self._check(self._lib.hmp_explain(self._ctx, _ptr(idx), n, _ptr(costs), _ptr(seeds), _ptr(poses), _ptr(nsteps)))
        out = {"costs": costs, "seeds": seeds, "poses": poses, "n_poses": nsteps}
        if with_forces:
            forces = np.zeros((n, T, 8))
            self._check(self._lib.hmp_debug_last_forces(self._ctx, n, _ptr(forces)))
            out["forces"] = forces
        return out

    def debug_world_to_map(self, wx: np.ndarray, wy: np.ndarray):
        wx = np.ascontiguousarray(wx, dtype=np.float64)
        wy = np.ascontiguousarray(wy, dtype=np.float64)
        n = wx.shape[0]
        mx, my, ok = (np.zeros(n, dtype=np.int32) for _ in range(3))
        self._check(self._lib.hmp_debug_world_to_map(self._ctx, _ptr(wx), _ptr(wy), n, _ptr(mx), _ptr(my), _ptr(ok)))
        return mx, my, ok

    def debug_footprint_cost(self, xyt: np.ndarray) -> np.ndarray:
        xyt = np.ascontiguousarray(xyt, dtype=np.float64).reshape(-1, 3)
        out = np.zeros(xyt.shape[0])
        self._check(self._lib.hmp_debug_footprint_cost(self._ctx, _ptr(xyt), xyt.shape[0], _ptr(out)))
        return out

    def debug_fis(self, in4: np.ndarray) -> np.ndarray:
        in4 = np.ascontiguousarray(in4, dtype=np.float64).reshape(-1, 4)
        out = np.zeros((in4.shape[0], 2))
        self._check(self._lib.hmp_debug_fis(self._ctx, _ptr(in4), in4.shape[0], _ptr(out)))
        return out

    def debug_sweep_candidate(self, candidate: int) -> np.ndarray:
        """What the thread-per-candidate sweep computed for one candidate of the last plan: 14 raw critics, seed (x, w), last pose."""
        out = np.zeros(19)
        self._lib.hmp_debug_sweep_candidate.argtypes = [C.c_void_p, _i, C.c_void_p]
        self._lib.hmp_debug_sweep_candidate.restype = C.c_int
        self._check(self._lib.hmp_debug_sweep_candidate(self._ctx, int(candidate), _ptr(out)))
        return out

    def launch_count(self) -> int:
        return int(self._lib.hmp_launch_count(self._ctx))
