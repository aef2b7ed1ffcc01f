"""Per-world critic scales and MapGrid shifts of a batched plan (hmp_set_scene_costs): every robot of a batch gets the values
HumapPlanner::updateLocalCosts (src/humap_planner.cpp:1054-1141) derives from its own state, and the batch selects what a
single-scene plan with those values in HmpParams selects."""
import ctypes as C
import json
import math
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

from humap_local_planner_b200 import capi, config, scenes
from humap_local_planner_b200.capi import HmpError, HmpParams, HmpSceneCosts, NUM_COSTS, NUM_MAPGRIDS

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OBSTACLE, PATH, GOAL, ALIGNMENT, GOAL_FRONT, UNSAT, TTC, HEADING_CHANGE, PERSONAL_SPACE, FFORMATION = (
    0, 1, 2, 3, 4, 5, 7, 8, 11, 12)


def _shared(params) -> HmpSceneCosts:
    """The table entry that repeats the shared values of params."""
    t = HmpSceneCosts()
    for k in range(NUM_COSTS):
        t.scale[k] = params.costs.scale[k]
    for g in range(NUM_MAPGRIDS):
        t.xshift[g], t.yshift[g] = params.costs.xshift[g], params.costs.yshift[g]
    return t


def _params_with(params, t: HmpSceneCosts) -> HmpParams:
    """params with one table entry's values in HmpCosts: what a single-scene plan of that world is given."""
    p = HmpParams.from_buffer_copy(params)
    for k in range(NUM_COSTS):
        p.costs.scale[k] = t.scale[k]
    for g in range(NUM_MAPGRIDS):
        p.costs.xshift[g], p.costs.yshift[g] = t.xshift[g], t.yshift[g]
    return p


def _people_xy(w):
    return [(w.people[i].x, w.people[i].y) for i in range(w.n_people)]


# ---------------------------------------------------------------------------------------------------------------
# CPU: ABI layout and the restated updateLocalCosts
# ---------------------------------------------------------------------------------------------------------------
def test_scene_costs_size_matches_the_c_layout():
    src = '#include <stdio.h>\n#include "hmp_planner.h"\nint main(){printf("%zu\\n",sizeof(HmpSceneCosts));return 0;}\n'
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "s.c"), "w").write(src)
        subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), "-o", os.path.join(d, "s"), os.path.join(d, "s.c")], check=True)
        size = int(subprocess.run([os.path.join(d, "s")], capture_output=True, text=True, check=True).stdout)
    assert C.sizeof(HmpSceneCosts) == size == 8 * (NUM_COSTS + 2 * NUM_MAPGRIDS)


def _world(goal_dist=8.0):
    w = capi.HmpWorld()
    w.robot_x, w.robot_y, w.robot_yaw = 1.0, -2.0, 0.3
    w.goal_x, w.goal_y = w.robot_x + goal_dist * math.cos(0.3), w.robot_y + goal_dist * math.sin(0.3)
    return w


def test_local_scene_costs_closed_form():
    params = config.default_params()
    base = params.costs
    r, fpd = config.ROBOT_INSCRIBED_RADIUS, 0.325
    # an empty world far from its goal: the shared values
    t = config.local_scene_costs(params, _world(), None)
    assert list(t.scale) == list(base.scale) and list(t.xshift) == list(base.xshift) and list(t.yshift) == list(base.yshift)
    # goal within forward_point_distance: no alignment; unsaturated ramp 6 / (3 r) * d
    t = config.local_scene_costs(params, _world(0.3), [])
    assert t.scale[ALIGNMENT] == 0.0
    assert t.scale[UNSAT] == pytest.approx(base.scale[UNSAT] / (3 * r) * 0.3, rel=1e-12)
    # goal at 0.4 m: alignment stays, the ramp value
    t = config.local_scene_costs(params, _world(0.4), [])
    assert t.scale[ALIGNMENT] == base.scale[ALIGNMENT]
    assert t.scale[UNSAT] == pytest.approx(base.scale[UNSAT] / (3 * r) * 0.4, rel=1e-12)
    assert list(t.xshift) == list(base.xshift)
    # a person 0.8 m away: xshift of alignment + goal front = 0.8 - (0.4 + 0.275); path / goal untouched
    w = _world()
    t = config.local_scene_costs(params, w, [(w.robot_x + 0.8, w.robot_y), (w.robot_x - 3.0, w.robot_y)])
    assert t.xshift[2] == pytest.approx(0.125, abs=1e-12) and t.xshift[3] == pytest.approx(0.125, abs=1e-12)
    assert t.xshift[0] == base.xshift[0] and t.xshift[1] == base.xshift[1]
    # ... 0.5 m away: the gap is clamped at 0
    t = config.local_scene_costs(params, w, [(w.robot_x, w.robot_y + 0.5)])
    assert t.xshift[2] == 0.0 and t.xshift[3] == 0.0
    # ... 3 m away: forward_point_distance
    t = config.local_scene_costs(params, w, [(w.robot_x, w.robot_y + 3.0)])
    assert t.xshift[2] == fpd and t.xshift[3] == fpd
    # goal inside a group, 1.2 m from its edge: F-formation x (1 - e^(-0.7 (1.2 - r)))
    t = config.local_scene_costs(params, w, None, goal_within_group=True, dist_to_group_edge=1.2)
    assert t.scale[FFORMATION] == pytest.approx(base.scale[FFORMATION] * (1.0 - math.exp(-0.7 * (1.2 - r))), rel=1e-12)
    t = config.local_scene_costs(params, w, None, goal_within_group=True, dist_to_group_edge=0.1)
    assert t.scale[FFORMATION] == 0.0
    # nothing else changes
    for k in range(NUM_COSTS):
        if k not in (ALIGNMENT, UNSAT, FFORMATION):
            assert t.scale[k] == base.scale[k]


# ---------------------------------------------------------------------------------------------------------------
# GPU: batch with a table == single-scene plans with the same values
# ---------------------------------------------------------------------------------------------------------------
@pytest.fixture(params=[1, 2], ids=["warp", "thread"])
def layout(request, planner):
    planner.set_sweep_layout(request.param)
    yield request.param
    planner.set_sweep_layout(0)


def _six_worlds(params):
    """Six cfg3 worlds whose per-cycle values all differ from the shared ones (and from each other)."""
    cfg = scenes.CONFIGS["cfg3"]
    scs = [scenes.make_scene(cfg, s) for s in range(6)]
    table = []
    w = scs[0].world   # goal 0.2 m ahead: no alignment critic, unsaturated-translation ramp
    w.goal_x, w.goal_y = w.robot_x + 0.2, w.robot_y
    table.append(config.local_scene_costs(params, w, _people_xy(w)))
    w = scs[1].world   # goal 0.6 m ahead: alignment on, ramp
    w.goal_x, w.goal_y = w.robot_x + 0.6, w.robot_y
    table.append(config.local_scene_costs(params, w, _people_xy(w)))
    w = scs[2].world   # a person 0.8 m to the side: forward point 0.125 m
    scs[2]._people[0].x, scs[2]._people[0].y = w.robot_x, w.robot_y + 0.8
    table.append(config.local_scene_costs(params, w, _people_xy(w)))
    w = scs[3].world   # goal inside an F-formation, 1 m from its edge
    table.append(config.local_scene_costs(params, w, _people_xy(w), goal_within_group=True, dist_to_group_edge=1.0))
    w = scs[4].world   # obstacle, goal-grid, TTC and personal-space critics off
    t = config.local_scene_costs(params, w, _people_xy(w))
    for k in (OBSTACLE, GOAL, TTC, PERSONAL_SPACE):
        t.scale[k] = 0.0
    table.append(t)
    t = _shared(params)   # shifts on all four grids
    for g, (dx, dy) in enumerate([(0.1, 0.05), (-0.15, -0.1), (0.2, 0.15), (0.05, -0.05)]):
        t.xshift[g], t.yshift[g] = dx, dy
    table.append(t)
    return scs, table


def _stack(scs):
    return (np.stack([sc.cells for sc in scs]), [np.stack([sc.grids[g] for sc in scs]) for g in range(4)],
            np.array([sc.hv_prev for sc in scs]))


def _singles(planner, params, scs, table, smp):
    out = []
    for sc, t in zip(scs, table):
        planner.set_params(_params_with(params, t) if t is not None else params)
        planner.set_scene(sc)
        r, _ = planner.plan(sc.world, smp, want_poses=False)
        out.append((r, planner.explored_totals(r.n_candidates)))
    return out


def _close(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    if not np.array_equal(np.isnan(a), np.isnan(b)):
        return False
    m = ~np.isnan(b)
    return bool(np.all(np.abs(a[m] - b[m]) <= 1e-12 * np.maximum(1.0, np.abs(b[m]))))


def _check_equal(res, tot, singles, mode, hv=True):
    for s, (r, (q, q_tot)) in enumerate(zip(res, singles)):
        assert (r.best_index, r.n_generated, r.n_valid) == (q.best_index, q.n_generated, q.n_valid), (s, r.best_index, q.best_index)
        if mode == 0:
            assert r.best_total == q.best_total, s
            assert np.array_equal(tot[s], q_tot), s
        else:
            assert abs(r.best_total - q.best_total) <= 1e-12 * max(1.0, abs(q.best_total)), s
        if hv and mode in (0, 1):
            assert list(r.highest_valid_cost) == list(q.highest_valid_cost), s
        assert _close(r.costs, q.costs), (s, list(r.costs), list(q.costs))
        assert _close([r.xv, r.yv, r.thetav], [q.xv, q.yv, q.thetav]), s


def _batch(planner, params, scs, smp, table):
    cells, grids, hv = _stack(scs)
    planner.set_params(params)
    planner.set_scene(scs[0])
    res = planner.plan_batch([sc.world for sc in scs], cells, grids, smp, hv_prev=hv, scene_costs=table)
    return res, planner.explored_totals(len(scs) * res[0].n_candidates).reshape(len(scs), -1)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1, 2], ids=["fp32", "fp64", "refine"])
def test_batch_with_scene_costs_equals_single_plans(planner, mode, layout):
    cfg = scenes.CONFIGS["cfg3"]
    params, smp = scenes.make_params(cfg), scenes.make_sampling(cfg)
    scs, table = _six_worlds(params)
    planner.set_precision(mode)
    try:
        singles = _singles(planner, params, scs, table, smp)
        res, tot = _batch(planner, params, scs, smp, table)
        _check_equal(res, tot, singles, mode)
        # the zero scales of world 4 are skipped there (NaN) and nowhere else; without the table the critics run
        assert res[4].best_index >= 0
        for k in (OBSTACLE, GOAL, TTC, PERSONAL_SPACE):
            assert math.isnan(res[4].costs[k]) and not math.isnan(res[5].costs[k]), k
        plain = planner.plan_batch([sc.world for sc in scs], None, None, smp, hv_prev=_stack(scs)[2], scene_costs=[])
        assert plain[4].best_index >= 0 and not any(math.isnan(plain[4].costs[k]) for k in (OBSTACLE, GOAL, TTC, PERSONAL_SPACE))
        assert any(plain[s].best_index != res[s].best_index or plain[s].best_total != res[s].best_total for s in range(6))
    finally:
        planner.set_scene_costs(None)
        planner.set_precision(False)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 2], ids=["fp32", "refine"])
def test_mixed_obstacle_scale(planner, mode, layout):
    """One world without the obstacle critic, the others with it: the launch keeps the obstacle machinery (dilated map, the
    deferred-critic instance of the thread-per-candidate sweep) for the others, and that world skips the critic."""
    cfg = scenes.CONFIGS["cfg3"]
    params, smp = scenes.make_params(cfg), scenes.make_sampling(cfg)
    scs = [scenes.make_scene(cfg, 20 + s) for s in range(4)]
    table = [_shared(params) for _ in scs]
    table[1].scale[OBSTACLE] = 0.0
    planner.set_precision(mode)
    try:
        singles = _singles(planner, params, scs, table, smp)
        res, tot = _batch(planner, params, scs, smp, table)
        _check_equal(res, tot, singles, mode)
        assert math.isnan(res[1].costs[OBSTACLE]) and not math.isnan(res[0].costs[OBSTACLE])
    finally:
        planner.set_scene_costs(None)
        planner.set_precision(False)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 2], ids=["fp32", "refine"])
def test_table_of_shared_values_changes_nothing(planner, mode, layout):
    cfg = scenes.CONFIGS["cfg3"]
    params, smp = scenes.make_params(cfg), scenes.make_sampling(cfg)
    scs = [scenes.make_scene(cfg, 40 + s) for s in range(6)]
    planner.set_precision(mode)
    try:
        planner.set_scene_costs(None)
        res0, tot0 = _batch(planner, params, scs, smp, None)
        res1, tot1 = _batch(planner, params, scs, smp, [_shared(params) for _ in scs])
    finally:
        planner.set_scene_costs(None)
        planner.set_precision(False)
    for a, b in zip(res0, res1):
        assert (a.best_index, a.best_total, a.n_generated, a.n_valid, a.n_poses) == (b.best_index, b.best_total, b.n_generated, b.n_valid, b.n_poses)
        assert list(a.highest_valid_cost) == list(b.highest_valid_cost) and (a.xv, a.yv, a.thetav) == (b.xv, b.yv, b.thetav)
        assert np.array_equal(np.array(a.costs), np.array(b.costs), equal_nan=True)
    assert np.array_equal(tot0, tot1)


@pytest.mark.gpu
@pytest.mark.parametrize("precise", [1, 2], ids=["fp64", "refine"])
def test_scene_costs_with_equisampled_pool(planner, precise, layout):
    cfg = scenes.CONFIGS["cfg0"]
    params, smp = scenes.make_params(cfg), scenes.make_sampling(cfg)
    vels = [(0.3, 0.0, 0.0), (0.9, 0.0, -0.4), (0.0, 0.0, 0.0), (0.05, 0.0, 0.1), (1.2, 0.0, 0.2)]
    scs = [scenes.make_scene(cfg, 10 + k, base_vel=v) for k, v in enumerate(vels)]
    table = []
    for k, sc in enumerate(scs):
        t = config.local_scene_costs(params, sc.world, _people_xy(sc.world), goal_within_group=(k == 3), dist_to_group_edge=0.9)
        t.scale[HEADING_CHANGE] *= 1.0 + 0.3 * k
        t.xshift[2], t.yshift[3] = 0.05 * k, -0.03 * k
        table.append(t)
    eq = capi.HmpEquisampled()
    eq.enabled, eq.vx_samples, eq.vy_samples, eq.vth_samples, eq.min_vel_x, eq.continued_acceleration = 1, 5, 1, 10, 0.1, 0
    planner.set_precision(precise)
    try:
        planner.set_equisampled(eq)
        singles = _singles(planner, params, scs, table, smp)
        res, tot = _batch(planner, params, scs, smp, table)
    finally:
        planner.set_scene_costs(None)
        planner.set_equisampled(None)
        planner.set_precision(False)
    _check_equal(res, tot, singles, precise, hv=False)   # as the batch test with this pool: selection and record


@pytest.mark.gpu
def test_table_persists_and_clears(planner, layout):
    cfg = scenes.CONFIGS["cfg3"]
    params, smp = scenes.make_params(cfg), scenes.make_sampling(cfg)
    scs, table = _six_worlds(params)
    hv = _stack(scs)[2]
    worlds = [sc.world for sc in scs]
    key = lambda rs: [(r.best_index, r.best_total, r.n_valid, list(r.highest_valid_cost)) for r in rs]   # noqa: E731
    planner.set_precision(False)
    try:
        planner.set_scene_costs(None)
        shared, _ = _batch(planner, params, scs, smp, None)
        res, _ = _batch(planner, params, scs, smp, table)
        assert key(res) != key(shared)
        assert key(planner.replan_resident()) == key(res)            # the table of the last plan
        planner.set_params(params)                                     # does not clear the table
        assert key(planner.plan_batch(worlds, None, None, smp, hv_prev=hv)) == key(res)
        planner.set_scene_costs([_shared(params)] * 6)                 # a new table does not change what the last plan re-runs with
        assert key(planner.replan_resident()) == key(res)
        planner.set_scene_costs(None)
        assert key(planner.replan_resident()) == key(res)
        assert key(planner.plan_batch(worlds, None, None, smp, hv_prev=hv)) == key(shared)   # cleared: the shared values
        assert key(planner.replan_resident()) == key(shared)
        # a larger table serves a smaller batch; hmp_plan ignores the table
        planner.set_scene_costs(table)
        assert key(planner.plan_batch(worlds[:3], None, None, smp, hv_prev=hv[:3])) == key(res[:3])
        planner.set_scene(scs[5])
        r_table, _ = planner.plan(scs[5].world, smp, want_poses=False)
        planner.set_scene_costs(None)
        r_plain, _ = planner.plan(scs[5].world, smp, want_poses=False)
        assert (r_table.best_index, r_table.best_total) == (r_plain.best_index, r_plain.best_total)
    finally:
        planner.set_scene_costs(None)


@pytest.mark.gpu
def test_scene_costs_against_oracle(planner, layout):
    """Two cfg0 worlds in mode 1: selection and the early-exit highest_valid_cost_ equal the oracle's with each world's params."""
    import oracle_binding as ob
    cfg = scenes.CONFIGS["cfg0"]
    params, smp = scenes.make_params(cfg), scenes.make_sampling(cfg)
    scs = [scenes.make_scene(cfg, 2), scenes.make_scene(cfg, 5)]
    w = scs[0].world
    w.goal_x, w.goal_y = w.robot_x + 0.3, w.robot_y
    table = [config.local_scene_costs(params, w, _people_xy(w)),
             config.local_scene_costs(params, scs[1].world, [(scs[1].world.robot_x + 0.85, scs[1].world.robot_y)])]
    table[1].yshift[0], table[1].scale[TTC] = 0.1, 0.0
    planner.set_precision(1)
    try:
        res, _ = _batch(planner, params, scs, smp, table)
    finally:
        planner.set_scene_costs(None)
        planner.set_precision(False)
    for sc, t, r in zip(scs, table, res):
        p = _params_with(params, t)
        o = ob.plan(p, sc, smp, early_exit=True, want=("totals",))
        full = ob.plan(p, sc, smp, early_exit=False, want=("totals",))["totals"]
        valid = np.sort(full[full >= 0])
        q = o["result"]
        top2_close = len(valid) > 1 and (valid[1] - valid[0]) <= 1e-4 * abs(valid[0])
        assert r.best_index == q.best_index or top2_close, (r.best_index, q.best_index)
        if q.best_index >= 0:
            assert abs(r.best_total - q.best_total) <= 1e-6 * abs(q.best_total)
        assert np.allclose(np.array(r.highest_valid_cost), np.array(q.highest_valid_cost))


@pytest.mark.gpu
def test_scene_cost_errors():
    cfg = scenes.CONFIGS["cfg3"]
    params, smp = scenes.make_params(cfg), scenes.make_sampling(cfg)
    scs = [scenes.make_scene(cfg, s, with_grids=False) for s in range(3)]
    cells = np.stack([sc.cells for sc in scs])
    pl = capi.Planner(0)
    try:
        def code(fn, *a, **k):
            with pytest.raises(HmpError) as e:
                fn(*a, **k)
            return e.value.code
        lib = capi.load_library()
        assert lib.hmp_set_scene_costs(pl._ctx, None, -1) == capi.HMP_E_INVALID
        assert lib.hmp_set_scene_costs(pl._ctx, None, 2) == capi.HMP_E_INVALID
        assert lib.hmp_set_scene_costs(pl._ctx, None, 0) == capi.HMP_OK
        for bad in (float("nan"), float("inf")):
            t = [_shared(params) for _ in range(3)]
            t[2].yshift[1] = bad
            assert code(pl.set_scene_costs, t) == capi.HMP_E_INVALID
        # MapGrid critics off in the shared params but on in the table: the grids must be resident for every scene
        p = HmpParams.from_buffer_copy(params)
        for g in range(NUM_MAPGRIDS):
            p.costs.scale[PATH + g] = 0.0
        pl.set_params(p)
        pl.set_costmap(scs[0].cells, scs[0].origin_x, scs[0].origin_y, scs[0].resolution)
        pl.set_footprint(scs[0].footprint)
        t = [_shared(p) for _ in range(3)]
        t[1].scale[GOAL_FRONT] = 0.4
        pl.set_scene_costs(t)
        assert code(pl.plan_batch, [sc.world for sc in scs], cells, None, smp) == capi.HMP_E_NOT_READY
        # too few entries for the batch
        pl.set_scene_costs(t[:2])
        assert code(pl.plan_batch, [sc.world for sc in scs], cells, None, smp) == capi.HMP_E_INVALID
    finally:
        pl.close()


SNIPPET = r'''
import json, sys
import numpy as np
sys.path.insert(0, %(root)r)
sys.path.insert(0, %(tests)r)
from humap_local_planner_b200 import Planner, scenes
import test_scene_costs as t
cfg = scenes.CONFIGS["cfg3"]
params, smp = scenes.make_params(cfg), scenes.make_sampling(cfg)
scs, table = t._six_worlds(params)
scs, table = scs[2:], table[2:]
out = {}
pl = Planner(0)
for mode, lay in ((2, 2), (0, 1), (0, 2), (1, 2)):
    pl.set_precision(mode); pl.set_sweep_layout(lay)
    res, tot = t._batch(pl, params, scs, smp, table)
    out["%%d-%%d" %% (mode, lay)] = [[r.best_index, r.best_total, r.n_valid, [c if c == c else None for c in r.costs]] for r in res] + [float(tot.sum())]
pl.close()
print("RESULT " + json.dumps(out))
'''


def _run(lib):
    env = dict(os.environ)
    if lib:
        env["HMP_LIB"] = lib
    return subprocess.run([sys.executable, "-c", SNIPPET % {"root": ROOT, "tests": os.path.join(ROOT, "tests")}], capture_output=True,
                          text=True, timeout=900, env=env)


@pytest.mark.gpu
def test_scene_costs_in_the_bounds_checked_build():
    from humap_local_planner_b200 import build as b
    lib = b.LIB_CHECK
    if not os.path.exists(lib):
        lib = b.build_library(check=True)
    r = _run(lib)
    assert "HMP_CHECK failed" not in r.stdout + r.stderr, (r.stdout + r.stderr)[-2000:]
    assert r.returncode == 0, (r.stdout + r.stderr)[-2000:]
    checked = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("RESULT ")][-1][7:])
    r0 = _run(None)
    assert r0.returncode == 0, (r0.stdout + r0.stderr)[-2000:]
    plain = json.loads([ln for ln in r0.stdout.splitlines() if ln.startswith("RESULT ")][-1][7:])
    assert checked == plain
