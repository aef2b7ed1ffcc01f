"""humap_local_planner_b200/adapter/from_reference.h: the reference-side binding (converters from the reference's own
types + a generator with SocialTrajectoryGenerator's setParameters / initialise signatures).

CPU: flat inputs -> the reference's objects (World built with its own addObstacle calls, HumapConfig, Person / Group,
TrajectorySamplingParams) -> converters -> flat outputs == inputs (round trip through oracle/_ref's objects).
GPU: HumapPlanner's call sequence on the reference's types, through the adapter, returns what a direct hmp_plan returns."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from humap_local_planner_b200 import scenes, config
from humap_local_planner_b200.capi import HmpParams, HmpWorld, HmpSampling, HmpObstacle, HmpPerson, HmpGroup, HmpResult, NUM_MAPGRIDS

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "tests", "_build", "libfrom_reference_test.so")


def _lib():
    import oracle_binding as ob
    if ob.reference_has("include"):
        ob.ref_lib()   # oracle/_ref/libhmp_ref.so
        from humap_local_planner_b200 import build as b
        b.build_library()
        subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "tests")], check=True)
    if not os.path.exists(LIB):
        pytest.skip("tests/_build/libfrom_reference_test.so is built from the original project's headers (HMP_REFERENCE_DIR)")
    return C.CDLL(LIB)


def _bytes(s):
    return C.string_at(C.addressof(s), C.sizeof(s))


@pytest.mark.parametrize("name,seed", [("cfg0", 0), ("cfg0", 3), ("cfg1", 1), ("cfg2", 0)])
def test_converters_round_trip(name, seed):
    L = _lib()
    cfg = scenes.CONFIGS[name]
    sc = scenes.make_scene(cfg, seed)
    params = scenes.make_params(cfg)
    smp = scenes.make_sampling(cfg)
    w = sc.world
    p_out, s_out, w_out = HmpParams(), HmpSampling(), HmpWorld()
    ob_out = (HmpObstacle * max(1, w.n_obstacles))()
    pe_out = (HmpPerson * max(1, w.n_people))()
    gr_out = (HmpGroup * max(1, w.n_groups))()
    L.fr_roundtrip.argtypes = [C.c_void_p] * 3 + [C.c_double, C.c_double] + [C.c_void_p] * 6
    rc = L.fr_roundtrip(C.byref(params), C.byref(w), C.byref(smp), sc.resolution, config.ROBOT_INSCRIBED_RADIUS, C.byref(p_out),
                        C.byref(s_out), C.byref(w_out), ob_out, pe_out, gr_out)
    assert rc == 0
    # sampling: exact
    assert _bytes(s_out) == _bytes(smp)
    # parameters: every field of limits / general / sfm / fis; costs field by field (MapGrid scales go x resolution / resolution)
    for blk in ("limits", "general", "sfm", "fis"):
        assert _bytes(getattr(p_out, blk)) == _bytes(getattr(params, blk)), blk
    for fname, _t in params.costs._fields_:
        a, b = getattr(p_out.costs, fname), getattr(params.costs, fname)
        a, b = (list(a), list(b)) if hasattr(a, "__len__") else ([a], [b])
        assert np.allclose(a, b, rtol=1e-15, atol=0), (fname, a, b)
    # world: robot, goals
    for f in ("robot_x", "robot_y", "vel_x", "vel_y", "vel_th", "goal_local_x", "goal_local_y", "goal_x", "goal_y"):
        assert getattr(w_out, f) == getattr(w, f), f
    for f in ("robot_yaw", "goal_local_yaw", "goal_yaw"):   # through the reference's quaternion
        assert abs(getattr(w_out, f) - getattr(w, f)) < 1e-15
    assert (w_out.n_obstacles, w_out.n_people, w_out.n_groups) == (w.n_obstacles, w.n_people, w.n_groups)
    # obstacles: World::addObstacle sorted them into dynamic (forced or moving) and static; the converter emits dynamic first
    def key(o, static_zero_vel):
        v = (0.0, 0.0, 0.0) if static_zero_vel else (o.vx, o.vy, o.vth)
        return (o.robot_x, o.robot_y, o.obj_x, o.obj_y) + v
    dyn_in = [o for o in (w.obstacles[i] for i in range(w.n_obstacles)) if o.force_dynamic or (o.vx ** 2 + o.vy ** 2 + o.vth ** 2) ** 0.5 > 0.035]
    sta_in = [o for o in (w.obstacles[i] for i in range(w.n_obstacles)) if not (o.force_dynamic or (o.vx ** 2 + o.vy ** 2 + o.vth ** 2) ** 0.5 > 0.035)]
    got = [ob_out[i] for i in range(w_out.n_obstacles)]
    assert [key(o, False) for o in got[:len(dyn_in)]] == [key(o, False) for o in dyn_in]
    assert all(o.force_dynamic == 1 for o in got[:len(dyn_in)])
    assert [key(o, False) for o in got[len(dyn_in):]] == [key(o, True) for o in sta_in]
    assert all(o.force_dynamic == 0 for o in got[len(dyn_in):])
    for i in range(w.n_obstacles):
        assert abs(got[i].robot_yaw - ([*dyn_in, *sta_in][i]).robot_yaw) < 1e-15
    for i in range(w.n_people):
        a, b = pe_out[i], w.people[i]
        assert (a.x, a.y, a.vx, a.vy, a.vth, a.cov_xx, a.cov_xy, a.cov_yx, a.cov_yy) == (b.x, b.y, b.vx, b.vy, b.vth, b.cov_xx, b.cov_xy, b.cov_yx, b.cov_yy)
        assert abs(a.yaw - b.yaw) < 1e-15
    for i in range(w.n_groups):
        a, b = gr_out[i], w.groups[i]
        assert (a.x, a.y, a.span_x, a.span_y, a.cov_xx, a.cov_xy, a.cov_yy) == (b.x, b.y, b.span_x, b.span_y, b.cov_xx, b.cov_xy, b.cov_yy)
        assert abs(a.yaw - b.yaw) < 1e-15


@pytest.mark.gpu
@pytest.mark.parametrize("name,seed", [("cfg0", 0), ("cfg1", 0)])
def test_reference_call_sequence_equals_direct_plan(planner, name, seed):
    L = _lib()
    cfg = scenes.CONFIGS[name]
    sc = scenes.make_scene(cfg, seed)
    params = scenes.make_params(cfg)
    smp = scenes.make_sampling(cfg)
    planner.set_precision(2)
    planner.set_params(params)
    planner.set_scene(sc)
    res, _ = planner.plan(sc.world, smp)
    planner.set_precision(0)
    out = HmpResult()
    cost = C.c_double(0.0)
    npts = C.c_int(0)
    gp = (C.c_void_p * NUM_MAPGRIDS)(*[g.ctypes.data for g in sc.grids])
    hv = np.array(sc.hv_prev, dtype=np.float64)
    L.fr_plan.argtypes = [C.c_void_p] * 4 + [C.c_int, C.c_int, C.c_double, C.c_double, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                          C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]
    rc = L.fr_plan(C.byref(params), C.byref(sc.world), C.byref(smp), sc.cells.ctypes.data, sc.size_x, sc.size_y, sc.origin_x, sc.origin_y,
                   sc.resolution, gp, hv.ctypes.data, sc.footprint.ctypes.data, sc.footprint.shape[0], config.ROBOT_INSCRIBED_RADIUS,
                   C.byref(out), C.byref(cost), C.byref(npts))
    assert rc == 0
    assert out.n_candidates == res.n_candidates and out.n_generated == res.n_generated
    assert out.best_index == res.best_index
    # the World's object order (dynamic first) differs from the flat call order: force sums differ by FP64 rounding only
    assert abs(out.best_total - res.best_total) <= 1e-9 * abs(res.best_total)
    assert cost.value == out.best_total and npts.value == res.n_poses
    assert abs(out.xv - res.xv) < 1e-9 and abs(out.thetav - res.thetav) < 1e-9
