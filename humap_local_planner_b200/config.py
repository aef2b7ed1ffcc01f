"""Default parameter sets of the sampling + scoring path as flat `HmpParams`.

`default_params()` reproduces the values that win at runtime in the reference: the
dynamic_reconfigure defaults of cfg/HumapPlanner.cfg and the TIAGo limits of
src/humap_config_ros.cpp:51-67 (SURVEY.md Appendix C, ".cfg" column), with the scale / parameter
wiring of HumapPlanner::updateCostParameters (src/humap_planner.cpp:868-928).
"""
from __future__ import annotations

import math

from .capi import (COST_NAMES, HmpParams, HmpSampling, HmpSceneCosts, NUM_AMPLIFIERS, NUM_COSTS, NUM_MAPGRIDS)

ROBOT_INSCRIBED_RADIUS = 0.275
PERSON_MODEL_RADIUS = 0.4
PERSON_FOV_HALF = 3.31613 / 2.0


def default_params(resolution: float = 0.05, sim_time: float = 3.5, sim_granularity: float = 0.1,
                   fis: bool = True) -> HmpParams:
    p = HmpParams()
    L = p.limits  # src/humap_config_ros.cpp:51-67
    L.max_vel_trans, L.min_vel_trans = 1.5, 0.1
    L.max_vel_x, L.min_vel_x = 1.5, -0.1
    L.max_vel_y, L.min_vel_y = 0.0, 0.0
    L.max_vel_theta, L.min_vel_theta = 2.0, 0.4
    L.acc_lim_x, L.acc_lim_y, L.acc_lim_theta = 2.5, 0.0, 3.2
    L.twist_rotation_compensation = 0.40          # cfg/HumapPlanner.cfg:15
    L.maintain_vel_components_rate = 0            # cfg/HumapPlanner.cfg:16
    g = p.general
    g.sim_time, g.sim_granularity, g.angular_sim_granularity = sim_time, sim_granularity, 0.1
    g.sim_period = 0.1                            # 10 Hz controller_frequency, humap_config_ros.cpp:27-29
    g.people_prediction_dt = sim_granularity      # humap_planner_ros.cpp:530-531
    g.discretize_by_time = 1                      # planMovingRobot, humap_planner.cpp:1313
    s = p.sfm  # cfg/HumapPlanner.cfg:45-78
    s.fov, s.mass = 2.0, 14.5
    s.internal_force_factor, s.static_interaction_force_factor, s.dynamic_interaction_force_factor = 0.75, 4.9, 10.0
    s.min_force, s.max_force = 5.0, 300.0
    s.speed_desired, s.relaxation_time = 1.29, 0.54
    s.an, s.bn, s.cn, s.ap, s.bp, s.cp, s.aw, s.bw = -2.092, 2.013, 3.2421, 1.5375, 0.9876, 0.4568, 40.39, 0.22452
    s.fov_factor_method, s.filter_forces, s.disable_interaction_forces = 0, 0, 0
    f = p.fis  # cfg/HumapPlanner.cfg:96-103; fis.fov = general.person_fov (humap_config_ros.cpp:150)
    f.force_factor = 100.0 if fis else 0.0
    f.human_action_range, f.fov, f.fov_factor_method = 8.0, PERSON_FOV_HALF, 0
    c = p.costs  # cfg/HumapPlanner.cfg:197-243; MapGrid scales x resolution (humap_planner.h:462-466)
    scales = [0.05, 15.0 * resolution, 25.5 * resolution, 8.5 * resolution, 8.0 * resolution, 6.0, 0.08, 3.0, 10.0,
              17.0, 20.0, 30.0, 7.5, 10.0]
    for k, v in enumerate(scales):
        c.scale[k] = v
    c.occdist_separation, c.occdist_separation_kernel, c.occdist_sum_scores = 0.025, 1, 0
    fwd = 0.325  # forward_point_distance
    for gidx in range(NUM_MAPGRIDS):
        c.xshift[gidx] = fwd if gidx >= 2 else 0.0      # alignment + goal_front (humap_planner.cpp:900-901)
        c.yshift[gidx] = 0.0
        c.stop_on_failure[gidx] = 0                      # humap_planner.cpp:58-61
        c.neighbour_kernel_size[gidx] = 3 if gidx >= 2 else 0   # humap MapGridCostFunction vs upstream class
        c.neighbour_cost_multiplier[gidx] = 3.0
    c.unsat_max_trans_vel, c.unsat_max_vel_x, c.unsat_max_vel_y = L.max_vel_trans, L.max_vel_x, L.max_vel_y
    c.backward_penalty = 25.0
    c.ttc_rollout_time, c.ttc_collision_distance = 0.0, 0.05
    c.hd_fov_person = 2.0 * PERSON_FOV_HALF
    c.hd_person_model_radius = PERSON_MODEL_RADIUS
    c.hd_robot_circumradius = ROBOT_INSCRIBED_RADIUS
    c.hd_max_speed = L.max_vel_trans
    c.ps_max_speed, c.ps_min_dist = L.max_vel_trans, ROBOT_INSCRIBED_RADIUS
    c.unsat_whole_horizon, c.hd_whole_horizon, c.psi_whole_horizon = 0, 1, 1
    c.fsi_whole_horizon, c.ps_whole_horizon = 1, 1
    return p


_ALIGNMENT, _UNSATURATED, _FFORMATION = (COST_NAMES.index(n) for n in ("alignment", "unsaturated", "fformation"))
_GRID_ALIGNMENT, _GRID_GOAL_FRONT = 2, 3   # HmpMapGridIndex


def local_scene_costs(params: HmpParams, world, people_xy=None, goal_within_group: bool = False, dist_to_group_edge: float = 0.0,
                      inscribed_radius: float = ROBOT_INSCRIBED_RADIUS,
                      person_model_radius: float = PERSON_MODEL_RADIUS) -> HmpSceneCosts:
    """The per-cycle setScale / setXShift calls of HumapPlanner::updateLocalCosts (src/humap_planner.cpp:1054-1141) for one
    robot, restated from adapter/from_reference.h (applyLocalCosts + minGapHumanRobot); one entry of Planner.set_scene_costs.

    `params` holds the base values, as toHmpParams / default_params leave them: scale[] (MapGrid scales x resolution) and
    forward_point_distance as the xshift of the goal-front grid. `world` gives pose_ and goal_; people_xy: [n][2] positions of
    the people of people_env_model_ (None: no people). GroupIntrusionDetector is not restated: whether the goal lies inside an
    F-formation and its distance to that group's edge are inputs."""
    c = params.costs
    out = HmpSceneCosts()
    for k in range(NUM_COSTS):
        out.scale[k] = c.scale[k]
    for g in range(NUM_MAPGRIDS):
        out.xshift[g], out.yshift[g] = c.xshift[g], c.yshift[g]
    forward_point_distance = c.xshift[_GRID_GOAL_FRONT]
    min_gap = float("inf")   # std::numeric_limits<double>::max() without people, :1068-1083
    for px, py in ([] if people_xy is None else people_xy):
        gap = math.hypot(px - world.robot_x, py - world.robot_y) - person_model_radius - inscribed_radius
        min_gap = min(max(0.0, gap), min_gap)
    fwd = min(min_gap, forward_point_distance)                                   # :1085
    out.xshift[_GRID_GOAL_FRONT] = fwd                                           # :1104
    out.xshift[_GRID_ALIGNMENT] = fwd                                            # :1112
    dist_to_goal = math.hypot(world.goal_x - world.robot_x, world.goal_y - world.robot_y)   # :1056
    out.scale[_ALIGNMENT] = 0.0 if dist_to_goal <= forward_point_distance else c.scale[_ALIGNMENT]   # :1107-1111
    if goal_within_group:                                                        # :1116-1127
        dist_to_group = max(dist_to_group_edge - inscribed_radius, 0.0)
        out.scale[_FFORMATION] = (1.0 - math.exp(-0.7 * dist_to_group)) * c.scale[_FFORMATION]
    threshold = 3.0 * inscribed_radius                                           # :1130-1140
    if dist_to_goal <= threshold:
        lin_val = c.scale[_UNSATURATED] / threshold * dist_to_goal
        out.scale[_UNSATURATED] = min(max(lin_val, 0.0), c.scale[_UNSATURATED])
    return out


def amplifier_samples(amp_min: float, amp_max: float, granularity: float):
    """SocialTrajectoryGenerator::computeAmplifierSamples (src/social_trajectory_generator.cpp:465-498)."""
    out = []
    n = math.ceil((amp_max - amp_min) / granularity)
    for i in range(n + 1):
        v = amp_min + granularity * i
        if v > amp_max:
            out.append(amp_max)
            break
        out.append(v)
    return out or [0.0]


def make_sampling(axes: dict) -> HmpSampling:
    """axes: name -> (min, max, granularity); unspecified axes are {1.0}."""
    from .capi import AMP_NAMES
    s = HmpSampling()
    for a in range(NUM_AMPLIFIERS):
        lo, hi, gr = axes.get(AMP_NAMES[a], (1.0, 1.0, 1.0))
        s.amp_min[a], s.amp_max[a], s.amp_granularity[a] = lo, hi, gr
    return s


def count_candidates(s: HmpSampling) -> int:
    n = 1
    for a in range(NUM_AMPLIFIERS):
        n *= len(amplifier_samples(s.amp_min[a], s.amp_max[a], s.amp_granularity[a]))
    return n


# cfg/HumapPlanner.cfg:123-189 -> 3 x 3 x 2 x 2 x 2 = 72 candidates
SAMPLING_CFG_DEFAULT = {
    "an": (-0.4, 1.0, 0.7), "cn": (-0.5, 2.5, 1.5), "ap": (-0.5, 1.5, 2.0), "aw": (0.5, 1.0, 0.5), "bw": (1.0, 4.5, 3.5),
}
# 4 values per axis inside the "meaningful ranges" named next to each axis in the .cfg
_AXES4 = {
    "speed": (0.4, 1.0, 0.2), "an": (-0.5, 1.0, 0.5), "cn": (-0.5, 2.5, 1.0), "ap": (-0.5, 4.0, 1.5),
    "aw": (0.5, 2.0, 0.5), "bw": (1.0, 4.0, 1.0), "as": (0.5, 2.0, 0.5), "bn": (0.5, 2.0, 0.5),
}
SAMPLING_4K = {k: _AXES4[k] for k in ("speed", "an", "cn", "ap", "aw", "bw")}          # 4^6
SAMPLING_16K = {k: _AXES4[k] for k in ("speed", "an", "cn", "ap", "aw", "bw", "as")}   # 4^7
SAMPLING_64K = dict(_AXES4)                                                             # 4^8
