"""MapGrid wave fronts whose shared-memory frontier queue overflows (DESIGN 6b): the block finishes the BFS itself with scans
of the grid from the level it reached. An open costmap and a serpentine plan along the cell centres of every k-th row give
either more distinct seed cells than the queue holds, or a first level (distance 1) larger than the queue; both for the
padded kernel (200 x 200 window, queue of 16384 cells) and for the queue kernel (256 x 256, queue of 12288 cells). Each case
is checked against the oracle's queue BFS (base_local_planner::MapGrid::computeTargetDistance) cell for cell, through a plan
on the device grids against one on the oracle grids, through a batch whose scene 0 overflows, and in the bounds-checked build."""
import ctypes as C
import dataclasses
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

import oracle_binding as ob
from humap_local_planner_b200 import Planner, scenes

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TESTS = os.path.dirname(os.path.abspath(__file__))
RES = 0.05
# name: (window size, every k-th row of the serpentine, distance whose cell count exceeds the queue, queue capacity)
CASES = {
    "padded-seeds": (200, 2, 0, 16384),
    "padded-frontier": (200, 4, 1, 16384),
    "queue-seeds": (256, 2, 0, 12288),
    "queue-frontier": (256, 8, 1, 12288),
}
LOCAL_GOAL = (False, True, False, True)   # MapGridCostFunction flags of the four grids (path, goal, alignment, goal front)


def serpentine(size, step, origin):
    """Cell centres of rows 0, step, 2 step, ... walked alternately left to right and back, joined at the row ends."""
    pts = []
    for k, r in enumerate(range(0, size, step)):
        cols = list(range(size)) if k % 2 == 0 else list(range(size - 1, -1, -1))
        if k > 0:
            pts += [(cols[0], rr) for rr in range(r - step + 1, r)]
        pts += [(c, r) for c in cols]
    return origin + (np.array(pts, dtype=np.float64) + 0.5) * RES


def oracle_grid(cells, origin, plan, local_goal):
    L = ob.lib()
    L.orc_mapgrid_compute.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double, C.c_void_p,
                                      C.c_int, C.c_int, C.c_void_p]
    L.orc_mapgrid_compute.restype = None
    plan = np.ascontiguousarray(plan, dtype=np.float64)
    out = np.zeros(cells.shape, dtype=np.float64)
    sy, sx = cells.shape
    L.orc_mapgrid_compute(cells.ctypes.data, sx, sy, origin, origin, RES, plan.ctypes.data, plan.shape[0], 1 if local_goal else 0,
                          out.ctypes.data)
    return out


def make_case(name):
    """Scene 0 on the open costmap with the serpentine (grids 0 and 2: every cell of it is a seed; 1 and 3 take a local goal),
    two ordinary scenes of the same window for the batch, and the oracle grids of all three."""
    size, step, dist, qcap = CASES[name]
    cfg = dataclasses.replace(scenes.CONFIGS["cfg0"], size=size)
    scs = [scenes.make_scene(cfg, seed, with_grids=False) for seed in range(3)]
    scs[0].cells = np.zeros((size, size), dtype=np.uint8)
    origin = scs[0].origin_x
    serp = serpentine(size, step, origin)
    plans = [[(serp, False), (serp, True), (serp, False), scs[0].plans[3]]] + [list(sc.plans) for sc in scs[1:]]
    refs = [[oracle_grid(sc.cells, origin, p, lg) for p, lg in four] for sc, four in zip(scs, plans)]
    # the case must really overflow the queue: seed cells (distance 0) or the first level (distance 1) of the serpentine
    assert (refs[0][0] == dist).sum() > qcap, (name, int((refs[0][0] == dist).sum()))
    return dict(name=name, scenes=scs, plans=plans, refs=refs, params=scenes.make_params(cfg), sampling=scenes.make_sampling(cfg))


@pytest.fixture(scope="module")
def pl():
    p = Planner(0)
    yield p
    p.close()


@pytest.fixture(scope="module", params=list(CASES))
def case(request):
    return make_case(request.param)


def setup_scene(pl, case):
    sc = case["scenes"][0]
    pl.set_params(case["params"])
    pl.set_costmap(sc.cells, sc.origin_x, sc.origin_y, sc.resolution)
    pl.set_footprint(sc.footprint)


def device_grids(pl, case):
    """compute_mapgrid of scene 0's four grids, then a plan that joins them; returns (grids, plan result, explored totals)."""
    setup_scene(pl, case)
    sc = case["scenes"][0]
    for g, (plan, lg) in enumerate(case["plans"][0]):
        pl.compute_mapgrid(g, plan, lg, sc.hv_prev[g])
    res, _ = pl.plan(sc.world, case["sampling"])
    tot = pl.explored_totals(res.n_candidates)
    return [pl.get_mapgrid(g, sc.cells.shape) for g in range(4)], res, tot


def batch_plans(case):
    plans = []
    for g in range(4):
        xy = [np.asarray(p[g][0], dtype=np.float64).reshape(-1, 2) for p in case["plans"]]
        plans.append((np.concatenate(xy), np.concatenate([[0], np.cumsum([len(a) for a in xy])]).astype(np.int32)))
    return plans


def device_grids_batch(pl, case):
    """compute_mapgrid_batch of the three scenes, then plan_batch on the resident grids; returns (scene 0's grids, results, totals)."""
    setup_scene(pl, case)
    scs = case["scenes"]
    pl.compute_mapgrid_batch(np.stack([sc.cells for sc in scs]), batch_plans(case), LOCAL_GOAL)
    res = pl.plan_batch([sc.world for sc in scs], None, None, case["sampling"], hv_prev=np.array([sc.hv_prev for sc in scs]))
    tot = pl.explored_totals(len(scs) * res[0].n_candidates)
    return [pl.get_mapgrid(g, scs[0].cells.shape) for g in range(4)], res, tot


def test_overflowing_wavefront_equals_the_oracle(pl, case):
    grids, _, _ = device_grids(pl, case)
    for g in range(4):
        ref = case["refs"][0][g]
        assert np.array_equal(grids[g], ref), (case["name"], g, int((grids[g] != ref).sum()))


def test_plan_on_overflowing_wavefronts_equals_uploaded_grids(pl, case):
    _, r1, t1 = device_grids(pl, case)
    sc = case["scenes"][0]
    for g in range(4):
        pl.set_mapgrid(g, case["refs"][0][g], sc.hv_prev[g])
    r2, _ = pl.plan(sc.world, case["sampling"])
    t2 = pl.explored_totals(r2.n_candidates)
    assert (r1.best_index, r1.best_total) == (r2.best_index, r2.best_total)
    assert np.array_equal(t1, t2)


def test_batch_with_an_overflowing_scene_equals_uploaded_grids(pl, case):
    grids, r1, t1 = device_grids_batch(pl, case)
    for g in range(4):
        ref = case["refs"][0][g]
        assert np.array_equal(grids[g], ref), (case["name"], g, int((grids[g] != ref).sum()))
    scs = case["scenes"]
    oracle = [np.stack([refs[g] for refs in case["refs"]]) for g in range(4)]
    r2 = pl.plan_batch([sc.world for sc in scs], np.stack([sc.cells for sc in scs]), oracle, case["sampling"],
                       hv_prev=np.array([sc.hv_prev for sc in scs]))
    t2 = pl.explored_totals(len(scs) * r2[0].n_candidates)
    assert [(r.best_index, r.best_total) for r in r1] == [(r.best_index, r.best_total) for r in r2]
    assert np.array_equal(t1, t2)


def test_single_wavefront_after_a_batch_equals_the_oracle(pl, case):
    """A batch of wave fronts, an uploaded grid in slot 0, then a single-grid wave front in slot 1 while the batch may still run
    on its side stream: slot 1 is the single grid's (the serpentine: two short levels), not the batch's (a local goal: hundreds
    of levels), and the plan equals one on the uploaded oracle grids."""
    setup_scene(pl, case)
    scs = case["scenes"]
    sc, refs = scs[0], case["refs"][0]
    pl.compute_mapgrid_batch(np.stack([s.cells for s in scs]), batch_plans(case), LOCAL_GOAL)
    pl.set_mapgrid(0, refs[0], sc.hv_prev[0])
    pl.compute_mapgrid(1, case["plans"][0][0][0], False, sc.hv_prev[1])
    r1, _ = pl.plan(sc.world, case["sampling"])
    t1 = pl.explored_totals(r1.n_candidates)
    expect = [refs[0], refs[0], refs[2], refs[3]]
    for g in range(4):
        got = pl.get_mapgrid(g, sc.cells.shape)
        assert np.array_equal(got, expect[g]), (case["name"], g, int((got != expect[g]).sum()))
    for g in range(4):
        pl.set_mapgrid(g, expect[g], sc.hv_prev[g])
    r2, _ = pl.plan(sc.world, case["sampling"])
    assert (r1.best_index, r1.best_total) == (r2.best_index, r2.best_total)
    assert np.array_equal(t1, pl.explored_totals(r2.n_candidates))


SNIPPET = r'''
import sys
import numpy as np
sys.path.insert(0, %(root)r)
sys.path.insert(0, %(tests)r)
import test_wavefront_overflow as t
from humap_local_planner_b200 import Planner
pl = Planner(0)
out = {}
for name in t.CASES:
    case = t.make_case(name)
    out[name] = np.stack(t.device_grids(pl, case)[0])
    out[name + "-batch"] = np.stack(t.device_grids_batch(pl, case)[0])
pl.close()
np.savez(%(out)r, **out)
'''


def test_overflowing_wavefronts_in_the_bounds_checked_build():
    from humap_local_planner_b200 import build as b
    lib = b.LIB_CHECK
    if not os.path.exists(lib):
        lib = b.build_library(check=True)
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "grids.npz")
        r = subprocess.run([sys.executable, "-c", SNIPPET % {"root": ROOT, "tests": TESTS, "out": path}], capture_output=True,
                           text=True, timeout=900, env=dict(os.environ, HMP_LIB=lib))
        assert "HMP_CHECK failed" not in r.stdout + r.stderr, (r.stdout + r.stderr)[-2000:]
        assert r.returncode == 0, (r.stdout + r.stderr)[-2000:]
        got = dict(np.load(path))
    for name in CASES:
        refs = np.stack(make_case(name)["refs"][0])
        assert np.array_equal(got[name], refs), name
        assert np.array_equal(got[name + "-batch"], refs), name
