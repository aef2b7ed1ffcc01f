"""Pins the CPU oracle against the known-answer tests of the reference's own test suite.

Every case below is transcribed from the reference's test/*.cpp (file:line cited per test); the
numbers are the reference's golden values (most of them produced by the author's MATLAB prototypes in
scripts/). These tests run on CPU (`-m "not gpu"`).
"""
import ctypes as C
import math

import numpy as np
import pytest

import oracle_binding as ob
from humap_local_planner_b200.capi import HmpFis, HmpObstacle, HmpWorld

PI = math.pi
STRICT = 1e-9


def _v3(*a):
    return (C.c_double * 3)(*a)


def _out(n=3):
    return (C.c_double * n)()


@pytest.fixture(scope="module")
def L():
    lib = ob.lib()
    lib.orc_theta_alpha_beta_2011.argtypes = [C.c_void_p, C.c_void_p]
    lib.orc_theta_alpha_beta_2014.argtypes = [C.c_void_p, C.c_void_p]
    lib.orc_relative_speed.argtypes = [C.c_void_p, C.c_void_p]
    lib.orc_direction.argtypes = [C.c_void_p]
    lib.orc_len3.argtypes = [C.c_void_p]
    return lib


# ---- test/test_geometry_angle.cpp:21-25, :48-71 -----------------------------------------------------------
def test_angle_normalisation(L):
    assert L.orc_direction(_v3(0.0, 0.0, 0.0)) == 0.0                      # atan2 of the zero vector
    assert L.orc_wrap(0.0) == 0.0
    assert L.orc_wrap(PI / 2) == pytest.approx(PI / 2, abs=1e-15)
    assert L.orc_wrap(3 * PI / 2) == pytest.approx(-PI / 2, abs=1e-12)     # wrap-around at +pi
    assert L.orc_wrap(-3 * PI / 2) == pytest.approx(PI / 2, abs=1e-12)     # wrap-around at -pi
    assert L.orc_wrap(2 * PI + 0.25) == pytest.approx(0.25, abs=1e-12)
    assert abs(L.orc_wrap(PI)) == pytest.approx(PI, abs=1e-12)


# ---- test/test_geometry_pose.cpp / test_geometry_quaternion.cpp: yaw survives the quaternion round trip ----
@pytest.mark.parametrize("yaw", [0.0, PI / 4, -PI / 2, 3 * PI / 4, -3 * PI / 4, 0.463647609000806, -2.9])
def test_pose_yaw_roundtrip(L, yaw):
    assert L.orc_yaw_roundtrip(yaw) == pytest.approx(yaw, abs=1e-12)


# ---- test/test_geometry_vector.cpp: 3-D length (SURVEY App. A #4) -------------------------------------------
def test_vector_length_is_3d(L):
    assert L.orc_len3(_v3(3.0, 4.0, 12.0)) == pytest.approx(13.0, abs=1e-12)


# ---- test/test_velocity_conversions.cpp:15-58 ----------------------------------------------------------------
@pytest.mark.parametrize("yaw,expect", [
    (0.0, (0.15, 0.0, 0.25)),
    (PI / 4, (0.106066017177982, 0.106066017177982, 0.25)),
    (-PI / 2, (9.18485099360515e-18, -0.15, 0.25)),
    (PI / 2, (9.184850993605149e-18, 0.15, 0.25)),
])
def test_compute_velocity_global(L, yaw, expect):
    out = _out()
    L.orc_velocity_global(_v3(0.15, 0.0, 0.25), C.c_double(yaw), out)
    assert np.allclose(list(out), expect, atol=STRICT, rtol=0)


# ---- test/test_velocity_conversions.cpp:60-109 ---------------------------------------------------------------
def test_compute_twist(L):
    L.orc_compute_twist.argtypes = [C.c_void_p, C.c_void_p] + [C.c_double] * 5 + [C.c_void_p]
    pose = _v3(0.0, 0.0, 0.0)
    out = _out()
    args = (1.0, 0.0, 1.5, 2.0, 0.0)   # mass, min_vel_x, max_vel_x, max_rot_vel, twist_rotation_compensation
    L.orc_compute_twist(pose, _v3(0.0, 0.0, 0.0), *args, out)
    assert list(out) == [0.0, 0.0, 0.0]
    L.orc_compute_twist(pose, _v3(1.0, 0.0, 0.0), *args, out)
    assert list(out) == [1.0, 0.0, 0.0]
    L.orc_compute_twist(pose, _v3(-0.5, -0.5, 0.0), *args, out)
    assert out[0] == 0.0 and out[1] == 0.0 and out[2] < 0.0


# ---- test/test_velocity_conversions.cpp:111-237 --------------------------------------------------------------
@pytest.mark.parametrize("vg,yaw,holo,expect", [
    ((1.0, 0.0, 0.0), 0.0, 0, (1.0, 0.0, 0.0)),
    ((0.0, 1.0, 0.0), PI / 2, 0, (1.0, 0.0, 0.0)),
    ((0.0, -1.0, 0.0), -PI / 2, 0, (1.0, 0.0, 0.0)),
    ((-1.0, 0.0, 0.0), PI, 0, (1.0, 0.0, 0.0)),
    ((-1.0, 0.0, 0.0), 0.0, 0, (-1.0, 0.0, 0.0)),
    ((1.0, 1.0, 0.0), PI / 4, 0, (1.414213562373095, 0.0, 0.0)),
    ((-1.0, -1.0, 0.0), PI / 4, 0, (-1.414213562373095, 0.0, 0.0)),
    ((-1.0, -1.0, -PI / 2), -3 * PI / 4, 0, (1.414213562373095, 0.0, -PI / 2)),
    ((1.0, 1.0, PI / 2), 0.0, 1, (1.0, 1.0, 1.570796326794897)),
    ((-1.0, -1.0, PI / 2), 0.0, 1, (-1.0, -1.0, 1.570796326794897)),
    ((0.5, 0.6, PI / 4), PI / 4, 1, (0.777817459305202, 0.070710678118655, 0.785398163397448)),
    ((0.7, 0.5, PI / 4), -PI / 4, 1, (0.141421356237310, 0.848528137423857, 0.785398163397448)),
])
def test_compute_velocity_local(L, vg, yaw, holo, expect):
    out = _out()
    L.orc_velocity_local(_v3(*vg), C.c_double(yaw), holo, out)
    assert np.allclose(list(out), expect, atol=STRICT, rtol=0)


# ---- test/test_velocity_conversions.cpp:239-405: two 25-step acceleration-limit sequences --------------------
CMD_LOOP = [(0.00, 0.0, 0.40)] + [(0.35, 0.0, 0.40)] * 3 + [(0.0, 0.0, 0.0)] * 3 + [(0.50, 0.0, 0.00)] + \
           [(0.50, 0.0, 0.50)] * 3 + [(0.60, 0.0, 0.00)] * 3 + [(0.0, 0.0, 0.0)] * 2 + [(-0.1, 0.0, 1.00)] * 4 + \
           [(0.0, 0.0, 0.0)] * 5
RESULTS_MAINTAIN = [
    (0.2700, 0, 0.1020), (0.0322, 0, 0.3645), (0.2822, 0, 0.3924), (0.3500, 0, 0.4000), (0.3500, 0, 0.4000),
    (0.1203, 0, 0.1375), (0, 0, 0), (0, 0, 0), (0.2500, 0, 0), (0.3812, 0, 0.2625), (0.5000, 0, 0.5000),
    (0.5000, 0, 0.5000), (0.5000, 0, 0.5000), (0.5000, 0, 0.5000), (0.5000, 0, 0.5000), (0.2500, 0, 0.2500),
    (0, 0, 0), (-0.0263, 0, 0.2625), (-0.0525, 0, 0.5250), (-0.0788, 0, 0.7875), (-0.1000, 0, 1.0000),
    (-0.0738, 0, 0.7375), (-0.0475, 0, 0.4750), (-0.0213, 0, 0.2125), (0, 0, 0), (0, 0, 0)]
RESULTS_TRIM = [
    (0.2700, 0, 0.1020), (0.0200, 0, 0.3645), (0.2700, 0, 0.4000), (0.3500, 0, 0.4000), (0.3500, 0, 0.4000),
    (0.1000, 0, 0.1375), (0, 0, 0), (0, 0, 0), (0.2500, 0, 0), (0.5000, 0, 0.2625), (0.5000, 0, 0.5000),
    (0.5000, 0, 0.5000), (0.5000, 0, 0.2375), (0.5000, 0, 0), (0.5000, 0, 0), (0.2500, 0, 0), (0, 0, 0),
    (-0.1000, 0, 0.2625), (-0.1000, 0, 0.5250), (-0.1000, 0, 0.7875), (-0.1000, 0, 1.0000), (0, 0, 0.7375),
    (0, 0, 0.4750), (0, 0, 0.2125), (0, 0, 0), (0, 0, 0)]


@pytest.mark.parametrize("maintain,expected", [(1, RESULTS_MAINTAIN), (0, RESULTS_TRIM)])
def test_adjust_twist_with_acc_limits_sequences(L, maintain, expected):
    L.orc_adjust_twist_acc.argtypes = [C.c_void_p] * 4 + [C.c_double, C.c_void_p, C.c_int, C.c_void_p]
    acc, vmin, vmax = _v3(1.0, 0.0, 1.05), _v3(-0.1, 0.0, -1.05), _v3(0.50, 0.0, 1.05)
    seq = [(0.27, 0.0, 0.102)]
    assert len(CMD_LOOP) == 25
    for cmd in CMD_LOOP:
        out = _out()
        L.orc_adjust_twist_acc(_v3(*seq[-1]), acc, vmin, vmax, 0.25, _v3(*cmd), maintain, out)
        seq.append(tuple(out))
    assert len(seq) == len(expected)
    assert np.allclose(np.array(seq), np.array(expected, dtype=float), atol=1e-4, rtol=0)


# ---- test/test_sfm.cpp:50-84 -----------------------------------------------------------------------------------
def test_sfm_internal_force(L):
    L.orc_internal_force.argtypes = [C.c_void_p, C.c_void_p, C.c_double, C.c_double, C.c_double, C.c_void_p]
    out = _out()
    L.orc_internal_force(_v3(0, 0, 0), _v3(5.0, 0.0, 0.0), 100.0, 1.0, 0.5, out)
    assert math.atan2(out[1], out[0]) == 0.0
    L.orc_internal_force(_v3(-1.0, -1.0, 0.0), _v3(-5.0, -5.0, 3 * PI / 4), 1.0, 10.0, 2.0, out)
    assert math.atan2(out[1], out[0]) == pytest.approx(-3 * PI / 4, abs=1e-12)
    L.orc_internal_force(_v3(0.5, -1.0, 0.0), _v3(5.0, -10.0, -PI / 2), 1.0, 10.0, 2.0, out)
    assert math.atan2(out[1], out[0]) == pytest.approx(-1.1071, abs=1e-4)
    L.orc_internal_force(_v3(0.5, -1.0, 0.0), _v3(5.0, -10.0, -PI / 2), 0.0, 10.0, 2.0, out)
    assert np.allclose(list(out), 0.0, atol=1e-6)


# ---- test/test_sfm.cpp:86-130 ----------------------------------------------------------------------------------
def test_sfm_theta_alpha_beta(L):
    assert math.isnan(L.orc_theta_alpha_beta_2011(_v3(0, 0, 0), _v3(1.0, -1.0, 0.0)))
    assert L.orc_theta_alpha_beta_2011(_v3(2.0, 3.0, 0.3), _v3(1.0, -1.0, 0.0)) == pytest.approx(1.7675, abs=1e-4)
    assert L.orc_theta_alpha_beta_2011(_v3(1.0, -1.0, 0.0), _v3(2.0, 3.0, 0.3)) == pytest.approx(1.7675, abs=1e-4)
    assert L.orc_theta_alpha_beta_2014(_v3(1.0, 0.0, 0.0), _v3(2.0, 3.0, 1.0)) == pytest.approx(-0.9828, abs=1e-4)
    n2 = _v3(math.cos(-PI / 4), math.sin(-PI / 4), 0.0)
    d2 = _v3(math.cos(PI / 2), math.sin(PI / 2), 0.0)
    assert L.orc_theta_alpha_beta_2014(n2, d2) == pytest.approx(L.orc_wrap(-PI / 4 - PI / 2), abs=1e-4)


# ---- test/test_sfm.cpp:132-158 ---------------------------------------------------------------------------------
@pytest.mark.parametrize("yaw,desc,expect", [
    (PI / 4, 1, PI / 4 + PI), (3 * PI / 4, 1, 3 * PI / 4 + PI), (3 * PI / 4, 0, 3 * PI / 4), (-PI / 2, 0, -PI / 2)])
def test_sfm_normal_alpha(L, yaw, desc, expect):
    L.orc_normal_alpha.argtypes = [C.c_double, C.c_int, C.c_void_p]
    out = _out()
    L.orc_normal_alpha(yaw, desc, out)
    assert L.orc_direction(out) == pytest.approx(L.orc_wrap(expect), abs=1e-12)


# ---- test/test_sfm.cpp:160-197: sign table of p_alpha (RelativeLocation: RIGHT = 1, LEFT = 2) -------------------
@pytest.mark.parametrize("n_angle,rel_loc,desc,rot", [
    (0.0, 1, 0, PI / 2), (0.0, 1, 1, -PI / 2), (-PI / 4, 2, 0, -PI / 2), (-PI / 4, 2, 1, PI / 2)])
def test_sfm_perpendicular_to_normal(L, n_angle, rel_loc, desc, rot):
    L.orc_perpendicular.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    n = (math.cos(n_angle), math.sin(n_angle), 0.0)
    out = _out()
    L.orc_perpendicular(_v3(*n), rel_loc, desc, out)
    expect = (n[0] * math.cos(rot) - n[1] * math.sin(rot), n[0] * math.sin(rot) + n[1] * math.cos(rot), 0.0)
    assert np.allclose(list(out), expect, atol=1e-6)


# ---- test/test_sfm.cpp:199-225 ---------------------------------------------------------------------------------
def test_sfm_relative_speed(L):
    assert L.orc_relative_speed(_v3(1.25, 1.25, 0), _v3(-1.25, -1.25, 0)) == pytest.approx(math.hypot(2.5, 2.5), abs=1e-4)
    assert L.orc_relative_speed(_v3(2.75, 2.75, 0), _v3(2.5, 2.5, 0)) == pytest.approx(math.hypot(0.25, 0.25), abs=1e-4)
    # the angular component is ignored
    assert L.orc_relative_speed(_v3(2.75, 2.75, PI / 4), _v3(2.5, 2.5, PI / 4)) == pytest.approx(math.hypot(0.25, 0.25), abs=1e-4)


# ---- test/test_world_generation.cpp:16-134 ---------------------------------------------------------------------
def _world(pose, vel, goal_local, goal, obstacles=()):
    w = HmpWorld()
    w.robot_x, w.robot_y, w.robot_yaw = pose
    w.vel_x, w.vel_y, w.vel_th = vel
    w.goal_local_x, w.goal_local_y, w.goal_local_yaw = goal_local
    w.goal_x, w.goal_y, w.goal_yaw = goal
    arr = (HmpObstacle * max(1, len(obstacles)))()
    for i, (rp, op, v) in enumerate(obstacles):
        arr[i].robot_x, arr[i].robot_y, arr[i].robot_yaw = rp
        arr[i].obj_x, arr[i].obj_y, arr[i].obj_yaw = op
        arr[i].vx, arr[i].vy, arr[i].vth = v
    w.obstacles = arr
    w.n_obstacles = len(obstacles)
    w._keep = arr
    return w


def _predict(L, w, vels, dt):
    L.orc_world_predict_sequence.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_double, C.c_void_p]
    v = np.ascontiguousarray(vels, dtype=np.float64).reshape(-1, 3)
    out = np.zeros((v.shape[0] + 1, 14))
    L.orc_world_predict_sequence(C.byref(w), v.ctypes.data, v.shape[0], dt, out.ctypes.data)
    return out


def test_world_target_distances(L):
    w = _world((1.0, 0.0, 0.0), (0, 0, 0), (2.0, 0.0, 0.0), (3.0, 0.0, 0.0))
    s = _predict(L, w, np.zeros((0, 3)), 1.0)[0]
    assert s[6] == 1.0 and s[7] == 2.0 and s[8] == pytest.approx(0.0, abs=1e-7)
    w = _world((0.0, 0.0, math.radians(90.0)), (0, 0, 0), (5.0, 5.0, 0.0), (10.0, 10.0, math.radians(180.0)))
    s = _predict(L, w, np.zeros((0, 3)), 1.0)[0]
    assert s[6] == math.sqrt(50.0) and s[7] == math.sqrt(200.0) and s[8] == pytest.approx(math.radians(45.0), abs=1e-6)


def test_world_predict_one_step(L):
    w = _world((1.0, 0.0, 0.0), (0.5, 0.0, 0.0), (2.0, 0.0, 0.0), (3.0, 0.0, 0.0),
               [((1.0, 0.0, 0.0), (2.0, 0.0, 0.0), (-0.25, 0.0, 0.0))])
    s = _predict(L, w, [(0.5, 0.0, 0.0)], 1.0)
    assert s[1][0] == 1.5 and s[1][1] == 0.0            # centroid + vel
    assert s[1][10] == 1.0 and s[1][9] == 0.0           # one dynamic object, no static
    assert s[1][11] == 1.75 and s[1][12] == 0.0         # obstacle + its velocity


def test_world_predict_sequence(L):
    # robot follows a trajectory with local velocity (0.6, -0.1, 0.0), dt = 0.1; the World velocity of each
    # state is the velocity that led to it (test_world_generation.cpp:75-134)
    w = _world((1.0, 0.0, 0.0), (0.5, 0.0, 0.0), (2.0, 0.0, 0.0), (3.0, 0.0, 0.0),
               [((1.0, 0.0, 0.0), (2.0, 0.0, 0.0), (-0.25, 0.0, 0.0))])
    vl = (0.6, -0.1, 0.0)
    L.orc_next_pose.argtypes = [C.c_void_p, C.c_void_p, C.c_double, C.c_int, C.c_void_p]
    p2, p3 = _out(), _out()
    L.orc_next_pose(_v3(1.0, 0.0, 0.0), _v3(*vl), 0.1, 1, p2)
    L.orc_next_pose(p2, _v3(*vl), 0.1, 1, p3)
    s = _predict(L, w, [vl, vl], 0.1)     # yaw stays 0 so the global velocities equal the local ones
    assert s.shape[0] == 3
    assert np.allclose(s[0][:2], (1.0, 0.0), atol=STRICT) and np.allclose(s[0][3:6], (0.5, 0.0, 0.0), atol=STRICT)
    assert np.allclose(s[1][:2], list(p2)[:2], atol=STRICT) and np.allclose(s[1][3:6], vl, atol=STRICT)
    assert np.allclose(s[2][:2], list(p3)[:2], atol=STRICT) and np.allclose(s[2][3:6], vl, atol=STRICT)


# ---- test/test_trajectory.cpp:15-120: constant-velocity person prediction ----------------------------------------
@pytest.mark.parametrize("vel,dt,expect_last", [((1.0, 1.0, 0.0), 1.0, (4.0, 4.0)), ((1.0, -0.33, 0.0), 0.1, (0.4, -0.132))])
def test_person_prediction(L, vel, dt, expect_last):
    L.orc_predict_object.argtypes = [C.c_void_p, C.c_void_p, C.c_double, C.c_int, C.c_void_p]
    L.orc_predict_object.restype = C.c_int
    yaw = math.atan2(vel[1], vel[0])
    poses = np.zeros((5, 3))
    nv = L.orc_predict_object(_v3(0.0, 0.0, yaw), _v3(*vel), dt, 5, poses.ctypes.data)
    assert nv == 4
    for i in range(5):
        assert poses[i][0] == pytest.approx(i * dt * vel[0], abs=1e-12)
        assert poses[i][1] == pytest.approx(i * dt * vel[1], abs=1e-12)
        assert poses[i][2] == pytest.approx(yaw, abs=1e-12)
    assert np.allclose(poses[4][:2], expect_last, atol=1e-12)


# ---- test/test_trajectory.cpp:122-379: base_local_planner::Trajectory -> poses + velocities ----------------------
def _traj_vels(L, pts, seed, dt, glob):
    L.orc_trajectory_velocities.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_double, C.c_int, C.c_void_p, C.c_void_p]
    L.orc_trajectory_velocities.restype = C.c_int
    p = np.ascontiguousarray(pts, dtype=np.float64)
    vels = np.zeros((len(pts), 3))
    poses = np.zeros((len(pts), 3))
    n = L.orc_trajectory_velocities(p.ctypes.data, len(pts), _v3(*seed), dt, glob, vels.ctypes.data, poses.ctypes.data)
    return vels[:n], poses


def test_trajectory_from_blp_linear(L):
    pts = [(0, 0, -0.785398163397448), (0, -0.353553390593274, -0.785398163397448),
           (0, -0.707106781186548, -0.785398163397448), (0, -1.06066017177982, -0.785398163397448)]
    vg, poses = _traj_vels(L, pts, (1.0, -1.0, 0.0), 0.25, 1)
    assert len(vg) == 3
    assert np.allclose(vg, [(0.0, -1.414213562373095, 0.0)] * 3, atol=STRICT)
    assert np.allclose(poses, pts, atol=STRICT)
    vl, _ = _traj_vels(L, pts, (1.0, -1.0, 0.0), 0.25, 0)
    assert np.allclose(vl, [(1.0, -1.0, 0.0)] * 3, atol=STRICT)


def test_trajectory_from_blp_angular(L):
    pts = [(0.0, 0.0, 0.463647609000806), (0.670820393249937, 0.894427190999916, 0.213647609000806),
           (1.542071433324901, 1.595085185436783, -0.036352390999194),
           (2.559582950388867, 2.058410462798365, -0.286352390999194),
           (3.660091006547741, 2.255595701417830, -0.536352390999194)]
    vg, poses = _traj_vels(L, pts, (1.0, 0.5, -0.25), 1.0, 1)
    expect = [(0.670820393249937, 0.894427190999916, -0.25), (0.871251040074964, 0.700657994436868, -0.25),
              (1.017511517063966, 0.463325277361582, -0.25), (1.100508056158875, 0.197185238619465, -0.25)]
    assert np.allclose(vg, expect, atol=STRICT)
    assert np.allclose(poses, pts, atol=STRICT)
    vl, _ = _traj_vels(L, pts, (1.0, 0.5, -0.25), 1.0, 0)
    assert np.allclose(vl, [(1.0, 0.5, -0.25)] * 4, atol=STRICT)


# ---- test/test_fuzzy_social_conductor.cpp:20-68 --------------------------------------------------------------------
def test_behaviour_strength_exponential(L):
    assert L.orc_behaviour_strength_exp(4.0, 4.1, 1.0, 1.0) == 0.0          # beyond the action range
    assert L.orc_behaviour_strength_exp(4.0, 2.0, 0.0, 0.0) == 0.0          # nobody moves
    assert L.orc_behaviour_strength_exp(4.0, 2.0, 1.0, 1.0) == pytest.approx(0.8647, abs=1e-3)
    assert L.orc_behaviour_strength_exp(4.0, 2.0, 2.0, 2.0) == pytest.approx(7.2537, abs=1e-3)


# ---- test/test_fuzzy_social_conductor.cpp:70-145 -------------------------------------------------------------------
def test_behaviour_force_orientation(L):
    L.orc_behaviour_force.argtypes = [C.c_void_p, C.c_double, C.c_void_p, C.c_double, C.c_int] + [C.c_void_p] * 6
    cfg = HmpFis()
    cfg.force_factor, cfg.human_action_range, cfg.fov, cfg.fov_factor_method = 1.0, 4.0, 2.0, 2   # NONE
    out = _out()
    arr = lambda *a: np.array(a, dtype=np.float64)
    speed = math.hypot(0.5, 0.5)
    v, m, sp, d, rl = arr(-PI / 4), arr(1.0), arr(speed), arr(2.0), arr(0.0)
    L.orc_behaviour_force(C.byref(cfg), 1.0, _v3(0.0, 0.0, PI / 4), speed, 1, v.ctypes.data, m.ctypes.data,
                          sp.ctypes.data, d.ctypes.data, rl.ctypes.data, out)
    assert math.atan2(out[1], out[0]) == pytest.approx(PI / 4 - PI / 4, abs=1e-6)
    # additivity of the unit vectors
    v, m, sp, d, rl = arr(-PI / 4, -3 * PI / 4), arr(1.0, 1.0), arr(0.5, 0.5), arr(3.6, 3.6), arr(0.0, 0.0)
    L.orc_behaviour_force(C.byref(cfg), 1.0, _v3(0.0, 0.0, 0.0), 0.5, 2, v.ctypes.data, m.ctypes.data,
                          sp.ctypes.data, d.ctypes.data, rl.ctypes.data, out)
    expect = math.atan2(math.sin(-PI / 4) + math.sin(-3 * PI / 4), math.cos(-PI / 4) + math.cos(-3 * PI / 4))
    assert math.atan2(out[1], out[0]) == pytest.approx(expect, abs=1e-12)


# ---- test/test_fuzzy_trapezoids_dynamic.cpp:203-330: rectangular trapezoids (0 deg flanks), cases 1 and 2 ---------
def _loc_dep(L, side, gs, ge, isect=0.0):
    L.orc_trapezoid_loc_dep.argtypes = [C.c_double, C.c_int, C.c_double, C.c_double, C.c_void_p]
    out = _out(8)
    L.orc_trapezoid_loc_dep(isect, side, gs, ge, out)
    return list(out)


def _loc_indep(L, centre, isect=0.0, length=0.0):
    L.orc_trapezoid_loc_indep.argtypes = [C.c_double, C.c_double, C.c_double, C.c_void_p]
    out = _out(8)
    L.orc_trapezoid_loc_indep(isect, length, centre, out)
    return list(out)


def _is_nan4(v):
    return all(math.isnan(x) for x in v)


def test_trapezoids_rectangular_case1(L):
    # robot1 yaw -30 deg, object1 at (5, 2.88675): gamma_eq -30, gamma_opp 150, gamma_cc -150, object on the LEFT (2)
    eq, opp, cc = math.radians(-30.0), math.radians(150.0), L.orc_wrap(math.atan2(2.88675, 5.0) + PI)
    assert math.degrees(cc) == pytest.approx(-150.0, abs=1e-3)
    t = _loc_dep(L, 2, opp, eq)                                   # outwards
    assert np.allclose(t[:4], [eq, eq, opp, opp], atol=1e-5) and _is_nan4(t[4:])
    t = _loc_dep(L, 2, eq, cc)                                    # cross_front
    assert np.allclose(t[:4], [cc, cc, eq, eq], atol=1e-5)
    t = _loc_dep(L, 2, cc, opp)                                   # cross_behind: wraps through +-pi
    assert np.allclose(t[:4], [opp, opp, PI, PI], atol=1e-5)
    assert np.allclose(t[4:], [-PI, -PI, cc, cc], atol=1e-5)
    t = _loc_indep(L, eq)                                         # equal
    assert np.allclose(t[:4], [eq] * 4, atol=1e-3) and _is_nan4(t[4:])
    t = _loc_indep(L, opp)                                        # opposite
    assert np.allclose(t[:4], [opp] * 4, atol=1e-3) and _is_nan4(t[4:])


def test_trapezoids_rectangular_case2(L):
    # robot2 yaw -30 deg, object2 at (5, -5): gamma_cc +135, object on the RIGHT (1)
    eq, opp, cc = math.radians(-30.0), math.radians(150.0), L.orc_wrap(math.atan2(-5.0, 5.0) + PI)
    assert math.degrees(cc) == pytest.approx(135.0, abs=1e-3)
    t = _loc_dep(L, 1, opp, eq)                                   # outwards: wraps
    assert np.allclose(t[:4], [opp, opp, PI, PI], atol=1e-5)
    assert np.allclose(t[4:], [-PI, -PI, eq, eq], atol=1e-5)
    t = _loc_dep(L, 1, eq, cc)                                    # cross_front
    assert np.allclose(t[:4], [eq, eq, cc, cc], atol=1e-5)


# ---- test/test_fuzzy_inference_system.cpp:120-379 pins only the SIGN / RANGE / TERM of the output ---------------
FIS_TERMS = ["accelerate", "turn_right_accelerate", "turn_right", "turn_right_decelerate", "decelerateA", "stopA",
             "decelerateB", "stopB", "turn_left_decelerate", "turn_left", "turn_left_accelerate"]


def _fis(L, dir_alpha, dir_beta, rel_loc, dist_angle):
    L.orc_fis_process.argtypes = [C.c_double] * 4 + [C.c_void_p] * 3
    out = _out(3)
    L.orc_fis_process(dir_alpha, dir_beta, rel_loc, dist_angle, out, None, None)
    return out[0], out[1], int(out[2])


# (object x, y, yaw) with the robot at (0, 0, 0) -> (value lower bound, upper bound, accepted term substrings)
FIS_LAYOUTS = [
    ((2.0, 0.0, PI), (-PI, 0.0), ("turn_right",)),                          # front / opposite         :131-143
    ((2.0, 0.0, -PI / 2), (-PI, 0.0), ("=turn_right",)),                    # front / cross front      :150-161
    ((1.0, -2.0, 3 * PI / 4), (0.0, PI), ("=turn_left",)),                  # front right / cross behind :166-177
    ((2.0, -2.0, PI), (0.0, PI), ("=turn_left",)),                          # front right / opposite   :182-193
    ((2.0, -2.0, -PI), (0.0, PI), ("=turn_left",)),                         # front right / outwards   :198-209
    ((2.0, -2.0, 0.0), (0.0, PI / 2), ("turn_left", "accelerate")),         # front right / equal      :214-230
    ((2.0, -2.0, PI / 4), (-PI, 0.0), ("=turn_right",)),                    # front right / cross front :235-246
    ((-2.0, -2.0, PI / 2), (0.0, PI / 2), ("=turn_left_accelerate",)),      # back right / cross behind :251-265
    ((-2.0, -2.0, PI), (-PI, 0.0), None),                                   # back right / opposite    :267-281
    ((-2.0, -2.0, 0.0), (-PI / 2, 0.0), ("=turn_right_accelerate",)),       # back right / equal       :283-295
    ((-2.0, -2.0, PI / 8), (-PI / 2, PI / 2), ("accelerate",)),             # back right / cross front :297-309
    ((-2.0, 2.0, -PI / 2), (-PI / 2, PI / 2), ("accelerate",)),             # back left / cross behind :311-323
    ((2.0, 2.0, -5.0 / 6.0 * PI), (-PI, 0.0), ("=turn_right",)),            # front left / cross behind :325-337
    ((2.0, 2.0, -PI / 2), (-PI / 2, 0.0), ("=turn_right_accelerate",)),     # front left / cross front :339-351
]


@pytest.mark.parametrize("obj,bounds,terms", FIS_LAYOUTS)
def test_fis_output_terms(L, obj, bounds, terms):
    # fuzzyfy() helper of the reference test (:457-475): dir_beta = object yaw, rel_loc = wrap(dist_angle - robot yaw)
    dist_angle = math.atan2(obj[1], obj[0])
    v, mu, term = _fis(L, 0.0, L.orc_wrap(obj[2]), L.orc_wrap(dist_angle - 0.0), dist_angle)
    assert term >= 0 and mu > 0.0
    assert bounds[0] <= v <= bounds[1]
    name = FIS_TERMS[term]
    if name[-1] in "AB":
        name = name[:-1]
    if terms is not None:
        assert any((name == t[1:]) if t.startswith("=") else (t in name) for t in terms), name
