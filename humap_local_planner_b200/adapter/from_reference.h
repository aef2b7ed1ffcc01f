/*
 * from_reference.h -- the reference-side binding as code: converters from humap_local_planner's OWN types to the flat
 * structs of the C ABI (include/hmp_planner.h), and a generator class whose setParameters / initialise have the
 * signatures of humap_local_planner::SocialTrajectoryGenerator, so that HumapPlanner's call sites compile unchanged.
 *
 * Header-only; needs the reference's headers on the include path (include/humap_local_planner/...). It is NOT part of
 * libhmp_planner.so and uses no CUDA header. Compiled and tested against $HMP_REFERENCE_DIR/include + the stand-in
 * third-party headers of oracle/ref_shim (tests/from_reference_test.cpp, tests/test_from_reference.py).
 *
 *   toHmpSampling(TrajectorySamplingParams)            humap_config.h:176-224 -> HmpSampling
 *   toHmpSample(SampleAmplifierSet)                    social_trajectory_generator.h:28-52 -> HmpSample
 *   toHmpWorld(World, vel_local, people, groups, out)  world.h:92-247 (what World::addObstacle stored, src/world.cpp:43-63),
 *                                                      person.h, group.h -> HmpWorld + storage
 *   toHmpParams(HumapConfig, resolution, radius)       HumapPlanner::reconfigure -> generator_social_.setParameters
 *                                                      (src/humap_planner.cpp:177-226) + updateCostParameters (:868-928, scales
 *                                                      of the MapGrid critics x costmap resolution, humap_planner.h:452-472)
 *                                                      + the constructor's fixed settings (:56-63)
 *   applyLocalCosts(params, cfg, inputs)               the per-cycle setScale / setXShift of updateLocalCosts (:1054-1141)
 *   GpuSocialTrajectoryGeneratorRef                    setParameters(...) / initialise(world_model_, vel_, sampling, limits,
 *                                                      mass, discretize_by_time) exactly as called at :205-226 and :1307-1314
 */
#pragma once

#include <cmath>
#include <limits>
#include <memory>
#include <vector>

#include <humap_local_planner/group.h>
#include <humap_local_planner/humap_config.h>
#include <humap_local_planner/person.h>
#include <humap_local_planner/social_trajectory_generator.h>
#include <humap_local_planner/world.h>

#include "gpu_social_trajectory_generator.h"

namespace humap_local_planner_b200 {

namespace hlp = humap_local_planner;

/// TrajectorySamplingParams -> HmpSampling (axis order HmpAmplifierIndex = nesting order of the generator's loops,
/// src/social_trajectory_generator.cpp:166-175)
inline HmpSampling toHmpSampling(const hlp::TrajectorySamplingParams& ts) {
	HmpSampling s;
	const double v[HMP_NUM_AMPLIFIERS][3] = {
	    {ts.sfm_desired_speed_amplifier_min, ts.sfm_desired_speed_amplifier_max, ts.sfm_desired_speed_amplifier_granularity},
	    {ts.sfm_an_amplifier_min, ts.sfm_an_amplifier_max, ts.sfm_an_amplifier_granularity},
	    {ts.sfm_bn_amplifier_min, ts.sfm_bn_amplifier_max, ts.sfm_bn_amplifier_granularity},
	    {ts.sfm_cn_amplifier_min, ts.sfm_cn_amplifier_max, ts.sfm_cn_amplifier_granularity},
	    {ts.sfm_ap_amplifier_min, ts.sfm_ap_amplifier_max, ts.sfm_ap_amplifier_granularity},
	    {ts.sfm_bp_amplifier_min, ts.sfm_bp_amplifier_max, ts.sfm_bp_amplifier_granularity},
	    {ts.sfm_cp_amplifier_min, ts.sfm_cp_amplifier_max, ts.sfm_cp_amplifier_granularity},
	    {ts.sfm_aw_amplifier_min, ts.sfm_aw_amplifier_max, ts.sfm_aw_amplifier_granularity},
	    {ts.sfm_bw_amplifier_min, ts.sfm_bw_amplifier_max, ts.sfm_bw_amplifier_granularity},
	    {ts.fis_as_amplifier_min, ts.fis_as_amplifier_max, ts.fis_as_amplifier_granularity},
	};
	for (int a = 0; a < HMP_NUM_AMPLIFIERS; ++a) {
		s.amp_min[a] = v[a][0];
		s.amp_max[a] = v[a][1];
		s.amp_granularity[a] = v[a][2];
	}
	return s;
}

inline HmpSample toHmpSample(const hlp::SocialTrajectoryGenerator::SampleAmplifierSet& a) {
	HmpSample s;
	s.amp[HMP_AMP_SPEED] = a.sfm_speed_desired_amplifier;
	s.amp[HMP_AMP_AN] = a.sfm_an_amplifier;
	s.amp[HMP_AMP_BN] = a.sfm_bn_amplifier;
	s.amp[HMP_AMP_CN] = a.sfm_cn_amplifier;
	s.amp[HMP_AMP_AP] = a.sfm_ap_amplifier;
	s.amp[HMP_AMP_BP] = a.sfm_bp_amplifier;
	s.amp[HMP_AMP_CP] = a.sfm_cp_amplifier;
	s.amp[HMP_AMP_AW] = a.sfm_aw_amplifier;
	s.amp[HMP_AMP_BW] = a.sfm_bw_amplifier;
	s.amp[HMP_AMP_AS] = a.fis_as_amplifier;
	return s;
}

/// HmpWorld points into these vectors; keep the storage alive as long as the world is used
struct HmpWorldStorage {
	HmpWorld world{};
	std::vector<HmpObstacle> obstacles;
	std::vector<HmpPerson> people;
	std::vector<HmpGroup> groups;
};

/**
 * The World as the generator receives it (generator_social_.initialise(world_model_, vel_, ...), :1307-1314) plus the
 * people / groups the social critics hold references to (people_env_model_, groups_env_model_, :37-40).
 *
 * World::addObstacle sorted every object into obstacle_dynamic_ (forced, or |v|_3 > 0.035) or obstacle_static_ (velocity
 * dropped) (src/world.cpp:43-63); that classification is what the rollout starts from, so it is reproduced literally:
 * dynamic objects first (force_dynamic = 1, their velocity kept -- an object that was only FORCED dynamic turns static after
 * the first World::predict, src/world.cpp:101-110, which the device handles), then the static ones with zero velocity.
 * robot_local_vel is vel_ (base frame): World only keeps the global velocity.
 */
inline void toHmpWorld(const hlp::World& world_model, const hlp::geometry::Vector& robot_local_vel, const std::vector<hlp::Person>& people,
                       const std::vector<hlp::Group>& groups, HmpWorldStorage& out) {
	const hlp::Robot& r = world_model.getRobotData();
	HmpWorld& w = out.world;
	w = HmpWorld{};
	w.robot_x = r.centroid.getX();
	w.robot_y = r.centroid.getY();
	w.robot_yaw = r.centroid.getYaw();
	w.vel_x = robot_local_vel.getX();
	w.vel_y = robot_local_vel.getY();
	w.vel_th = robot_local_vel.getZ();
	w.goal_local_x = r.target.object.getX();
	w.goal_local_y = r.target.object.getY();
	w.goal_local_yaw = r.target.object.getYaw();
	w.goal_x = r.goal.object.getX();
	w.goal_y = r.goal.object.getY();
	w.goal_yaw = r.goal.object.getYaw();
	out.obstacles.clear();
	for (const auto& d : world_model.getDynamicObjectsData()) {
		HmpObstacle o{};
		o.robot_x = d.robot.getX();
		o.robot_y = d.robot.getY();
		o.robot_yaw = d.robot.getYaw();
		o.obj_x = d.object.getX();
		o.obj_y = d.object.getY();
		o.obj_yaw = d.object.getYaw();
		o.vx = d.vel.getX();
		o.vy = d.vel.getY();
		o.vth = d.vel.getZ();
		o.force_dynamic = 1;
		out.obstacles.push_back(o);
	}
	for (const auto& s : world_model.getStaticObjectsData()) {
		HmpObstacle o{};
		o.robot_x = s.robot.getX();
		o.robot_y = s.robot.getY();
		o.robot_yaw = s.robot.getYaw();
		o.obj_x = s.object.getX();
		o.obj_y = s.object.getY();
		o.obj_yaw = s.object.getYaw();
		out.obstacles.push_back(o);
	}
	out.people.clear();
	for (const auto& p : people) {
		const hlp::geometry::Pose pose(p.getPose());   // as humap_local_planner::Trajectory reads it (trajectory.h:160-170)
		HmpPerson q{};
		q.x = pose.getX();
		q.y = pose.getY();
		q.yaw = pose.getYaw();
		q.vx = p.getVelocityX();
		q.vy = p.getVelocityY();
		q.vth = p.getVelocityTheta();
		q.cov_xx = p.getCovariancePoseXX();
		q.cov_xy = p.getCovariancePoseXY();
		q.cov_yx = p.getCovariancePoseYX();
		q.cov_yy = p.getCovariancePoseYY();
		out.people.push_back(q);
	}
	out.groups.clear();
	for (const auto& g : groups) {
		const hlp::geometry::Pose pose(g.getPose());
		HmpGroup q{};
		q.x = pose.getX();
		q.y = pose.getY();
		q.yaw = pose.getYaw();
		q.span_x = g.getSpanX();
		q.span_y = g.getSpanY();
		q.cov_xx = g.getCovariancePoseXX();
		q.cov_xy = g.getCovariancePoseXY();
		q.cov_yy = g.getCovariancePoseYY();
		out.groups.push_back(q);
	}
	w.obstacles = out.obstacles.data();
	w.people = out.people.data();
	w.groups = out.groups.data();
	w.n_obstacles = (int32_t)out.obstacles.size();
	w.n_people = (int32_t)out.people.size();
	w.n_groups = (int32_t)out.groups.size();
}

inline HmpLimits toHmpLimits(const hlp::PlannerLimitsParams& l) {
	HmpLimits h{};
	h.max_vel_trans = l.max_vel_trans;
	h.min_vel_trans = l.min_vel_trans;
	h.max_vel_x = l.max_vel_x;
	h.min_vel_x = l.min_vel_x;
	h.max_vel_y = l.max_vel_y;
	h.min_vel_y = l.min_vel_y;
	h.max_vel_theta = l.max_vel_theta;
	h.min_vel_theta = l.min_vel_theta;
	h.acc_lim_x = l.acc_lim_x;
	h.acc_lim_y = l.acc_lim_y;
	h.acc_lim_theta = l.acc_lim_theta;
	h.twist_rotation_compensation = l.twist_rotation_compensation;
	h.maintain_vel_components_rate = l.maintain_vel_components_rate ? 1 : 0;
	return h;
}

inline HmpSfm toHmpSfm(const hlp::SfmParams& s) {
	HmpSfm h{};
	h.fov = s.fov;
	h.mass = s.mass;
	h.internal_force_factor = s.internal_force_factor;
	h.static_interaction_force_factor = s.static_interaction_force_factor;
	h.dynamic_interaction_force_factor = s.dynamic_interaction_force_factor;
	h.min_force = s.min_force;
	h.max_force = s.max_force;
	h.speed_desired = s.speed_desired;
	h.relaxation_time = s.relaxation_time;
	h.an = s.an;
	h.bn = s.bn;
	h.cn = s.cn;
	h.ap = s.ap;
	h.bp = s.bp;
	h.cp = s.cp;
	h.aw = s.aw;
	h.bw = s.bw;
	h.fov_factor_method = (int32_t)s.fov_factor_method;
	h.filter_forces = s.filter_forces ? 1 : 0;
	h.disable_interaction_forces = s.disable_interaction_forces ? 1 : 0;
	return h;
}

inline HmpFis toHmpFis(const hlp::FisParams& f) {
	HmpFis h{};
	h.force_factor = f.force_factor;
	h.human_action_range = f.human_action_range;
	h.fov = f.fov;
	h.fov_factor_method = (int32_t)f.fov_factor_method;
	return h;
}

/**
 * Everything HumapPlanner::reconfigure (src/humap_planner.cpp:177-226) + updateCostParameters (:868-928) + the constructor
 * (:56-63) push into the generator and the 14 critics. `costmap_resolution` = planner_util_->getCostmap()->getResolution(),
 * `inscribed_radius` = robot_model_->getInscribedRadius(). scale[] holds getScale() of every critic: the four MapGrid
 * scales are multiplied by the resolution (ScalesCmCostFunctions, humap_planner.h:452-472). The per-cycle changes of
 * updateLocalCosts are applied on top by applyLocalCosts().
 */
inline HmpParams toHmpParams(const hlp::HumapConfig& cfg, double costmap_resolution, double inscribed_radius) {
	HmpParams p{};
	const auto& L = *cfg.getLimits();
	const auto& G = *cfg.getGeneral();
	const auto& C = *cfg.getCost();
	p.limits = toHmpLimits(L);
	p.general.sim_time = G.sim_time;
	p.general.sim_granularity = G.sim_granularity;
	p.general.angular_sim_granularity = G.angular_sim_granularity;
	p.general.sim_period = G.sim_period;
	p.general.people_prediction_dt = G.sim_granularity;   // src/humap_planner_ros.cpp:530
	p.general.discretize_by_time = 1;                     // planMovingRobot passes true (:1313); initialise() overrides
	p.sfm = toHmpSfm(*cfg.getSfm());
	p.fis = toHmpFis(*cfg.getFis());
	HmpCosts& c = p.costs;
	c.scale[HMP_COST_OBSTACLE] = C.occdist_scale;
	c.scale[HMP_COST_PATH] = C.path_distance_scale * costmap_resolution;
	c.scale[HMP_COST_GOAL] = C.goal_distance_scale * costmap_resolution;
	c.scale[HMP_COST_ALIGNMENT] = C.alignment_scale * costmap_resolution;
	c.scale[HMP_COST_GOAL_FRONT] = C.goal_front_scale * costmap_resolution;
	c.scale[HMP_COST_UNSATURATED] = C.unsaturated_translation_scale;
	c.scale[HMP_COST_BACKWARD] = C.backward_scale;
	c.scale[HMP_COST_TTC] = C.ttc_scale;
	c.scale[HMP_COST_HEADING_CHANGE] = C.heading_change_smoothness_scale;
	c.scale[HMP_COST_VEL_SMOOTHNESS] = C.velocity_smoothness_scale;
	c.scale[HMP_COST_HEADING_DIST] = C.heading_dir_scale;
	c.scale[HMP_COST_PERSONAL_SPACE] = C.personal_space_scale;
	c.scale[HMP_COST_FFORMATION] = C.fformation_space_scale;
	c.scale[HMP_COST_PASSING_SPEED] = C.passing_speed_scale;
	c.occdist_separation = C.occdist_separation;
	c.occdist_separation_kernel = (int32_t)C.occdist_separation_kernel;
	c.occdist_sum_scores = C.occdist_sum_scores ? 1 : 0;
	for (int g = 0; g < HMP_NUM_MAPGRIDS; ++g) {
		c.xshift[g] = 0.0;
		c.yshift[g] = 0.0;
		c.stop_on_failure[g] = 0;   // constructor, :56-60
		// n_kernel_size_ / n_cost_multiplier_ defaults of the customised critic (src/map_grid_cost_function.cpp:57-58); the
		// upstream class behind path / goal has no neighbour heuristic
		const bool custom = (g == HMP_GRID_ALIGNMENT || g == HMP_GRID_GOAL_FRONT);
		c.neighbour_kernel_size[g] = custom ? 3 : 0;
		c.neighbour_cost_multiplier[g] = 3.0;
	}
	c.xshift[HMP_GRID_GOAL_FRONT] = C.forward_point_distance;   // :900-901
	c.xshift[HMP_GRID_ALIGNMENT] = C.forward_point_distance;
	c.unsat_max_trans_vel = L.max_vel_trans;
	c.unsat_max_vel_x = L.max_vel_x;
	c.unsat_max_vel_y = L.max_vel_y;
	c.unsat_whole_horizon = C.unsaturated_translation_compute_whole_horizon ? 1 : 0;
	c.backward_penalty = C.backward_penalty;
	c.ttc_rollout_time = C.ttc_rollout_time;
	c.ttc_collision_distance = C.ttc_collision_distance;
	c.hd_fov_person = 2.0 * G.person_fov;
	c.hd_person_model_radius = G.person_model_radius;
	c.hd_robot_circumradius = inscribed_radius;
	c.hd_max_speed = L.max_vel_trans;
	c.hd_whole_horizon = C.heading_dir_compute_whole_horizon ? 1 : 0;
	c.psi_whole_horizon = C.personal_space_compute_whole_horizon ? 1 : 0;
	c.fsi_whole_horizon = C.fformation_space_compute_whole_horizon ? 1 : 0;
	c.ps_max_speed = L.max_vel_trans;
	c.ps_min_dist = inscribed_radius;
	c.ps_whole_horizon = C.passing_speed_compute_whole_horizon ? 1 : 0;
	return p;
}

/// What updateLocalCosts (src/humap_planner.cpp:1054-1141) derives from the cycle's state before it touches the critics
struct LocalCostInputs {
	double dist_to_goal = std::numeric_limits<double>::max();        ///< |goal_ - pose_| (:1056)
	double min_gap_human_robot = std::numeric_limits<double>::max(); ///< result of the loop over people_env_model_ (:1069-1083)
	bool goal_within_group = false;                                  ///< group_intrusion_.isGlobalGoalWithinGroup() (:1116)
	double dist_to_group_edge = 0.0;                                 ///< group_intrusion_.getDistanceToGroupEdgeGoalWithin() (:1121)
};

/// min_gap_human_robot of :1068-1083
inline double minGapHumanRobot(const std::vector<hlp::Person>& people, double robot_x, double robot_y, double person_model_radius,
                               double inscribed_radius) {
	double min_gap = std::numeric_limits<double>::max();
	for (const auto& person : people) {
		const double distance = std::hypot(person.getPositionX() - robot_x, person.getPositionY() - robot_y);
		const double gap = distance - person_model_radius - inscribed_radius;
		min_gap = std::min(std::max(0.0, gap), min_gap);
	}
	return min_gap;
}

/// The per-cycle setXShift / setScale calls of updateLocalCosts applied to params (start from toHmpParams every cycle)
inline void applyLocalCosts(HmpParams& p, const hlp::HumapConfig& cfg, double costmap_resolution, double inscribed_radius,
                            const LocalCostInputs& in) {
	const auto& C = *cfg.getCost();
	const double forward_point_distance = std::min(in.min_gap_human_robot, C.forward_point_distance);   // :1085
	p.costs.xshift[HMP_GRID_GOAL_FRONT] = forward_point_distance;                                       // :1104
	p.costs.xshift[HMP_GRID_ALIGNMENT] = forward_point_distance;                                        // :1112
	p.costs.scale[HMP_COST_ALIGNMENT] = (in.dist_to_goal <= C.forward_point_distance) ? 0.0 : C.alignment_scale * costmap_resolution;   // :1107-1111
	if (!in.goal_within_group) {
		p.costs.scale[HMP_COST_FFORMATION] = C.fformation_space_scale;
	} else {
		const double dist_to_group = std::max(in.dist_to_group_edge - inscribed_radius, 0.0);
		p.costs.scale[HMP_COST_FFORMATION] = (1.0 - std::exp(-0.7 * dist_to_group)) * C.fformation_space_scale;   // :1118-1127
	}
	const double threshold = 3.0 * inscribed_radius;
	if (in.dist_to_goal > threshold) {
		p.costs.scale[HMP_COST_UNSATURATED] = C.unsaturated_translation_scale;
	} else {
		const double lin_val = C.unsaturated_translation_scale / threshold * in.dist_to_goal;
		p.costs.scale[HMP_COST_UNSATURATED] = std::min(std::max(lin_val, 0.0), C.unsaturated_translation_scale);   // :1130-1140
	}
}

/// TrajectoryGeneration -> the equisampled generator's settings (generator_vel_space_.setParameters, :196-203)
inline HmpEquisampled toHmpEquisampled(const hlp::TrajectoryGeneration& t) {
	HmpEquisampled e{};
	e.enabled = t.use_equisampled_velocities_generator ? 1 : 0;
	e.vx_samples = (int32_t)t.equisampled_vx;
	e.vy_samples = (int32_t)t.equisampled_vy;
	e.vth_samples = (int32_t)t.equisampled_vth;
	e.min_vel_x = t.equisampled_min_vel_x;
	e.continued_acceleration = t.equisampled_continued_acceleration ? 1 : 0;
	return e;
}

/**
 * GpuSocialTrajectoryGenerator with the member signatures of humap_local_planner::SocialTrajectoryGenerator, so that
 *     generator_social_.setParameters(cfg_->getSfm(), cfg_->getFis(), sim_time, ...)                    (:205-226)
 *     generator_social_.initialise(world_model_, vel_, *cfg_->getTrajectorySampling(), cfg_->getLimits(), mass, true)   (:1307-1314)
 * compile unchanged against a member of this type. It keeps references to the people / groups containers exactly like the
 * social critics do (heading_disturbance_costs_(people_env_model_), ... :37-40), and a copy of the critic parameters
 * (setCostParameters, from toHmpParams + applyLocalCosts) since on this path the critics live behind the same C ABI.
 */
class GpuSocialTrajectoryGeneratorRef : public GpuSocialTrajectoryGenerator {
public:
	GpuSocialTrajectoryGeneratorRef(const std::vector<hlp::Person>& people, const std::vector<hlp::Group>& groups, int device_id = 0)
	    : GpuSocialTrajectoryGenerator(device_id), people_(people), groups_(groups) {}

	/// SocialTrajectoryGenerator::setParameters (social_trajectory_generator.h:135-147); the log flags have no device side
	void setParameters(std::shared_ptr<const hlp::SfmParams> sfm_params_ptr, std::shared_ptr<const hlp::FisParams> fis_params_ptr,
	                   double sim_time, double sim_granularity, double angular_sim_granularity, double sim_period,
	                   bool maintain_vel_components_rate, bool = false, bool = false, bool = false, bool = false) {
		params_.sfm = toHmpSfm(*sfm_params_ptr);
		params_.fis = toHmpFis(*fis_params_ptr);
		params_.general.sim_time = sim_time;
		params_.general.sim_granularity = sim_granularity;
		params_.general.angular_sim_granularity = angular_sim_granularity;
		params_.general.sim_period = sim_period;
		params_.general.people_prediction_dt = sim_granularity;
		maintain_rate_ = maintain_vel_components_rate;
		dirty_ = true;
	}

	/// limits / general / costs of a toHmpParams(+ applyLocalCosts) result (updateCostParameters, updateLocalCosts)
	void setCostParameters(const HmpParams& p) {
		params_.costs = p.costs;
		dirty_ = true;
	}

	/// SocialTrajectoryGenerator::initialise (social_trajectory_generator.h:188-195)
	void initialise(const hlp::World& world_model, const hlp::geometry::Vector& robot_local_vel, const hlp::TrajectorySamplingParams& limits_amplifiers,
	                std::shared_ptr<const hlp::PlannerLimitsParams> limits_lp_ptr, const double& robot_mass, bool discretize_by_time = false,
	                bool explore_all = false) {
		params_.limits = toHmpLimits(*limits_lp_ptr);
		params_.limits.maintain_vel_components_rate = maintain_rate_ ? 1 : 0;   // setParameters' flag is the one the generator uses
		params_.sfm.mass = robot_mass;
		params_.general.discretize_by_time = discretize_by_time ? 1 : 0;
		GpuSocialTrajectoryGenerator::setParameters(params_);
		dirty_ = false;
		toHmpWorld(world_model, robot_local_vel, people_, groups_, storage_);
		GpuSocialTrajectoryGenerator::initialise(storage_.world, toHmpSampling(limits_amplifiers), explore_all);
	}

	const HmpParams& params() const { return params_; }
	const HmpWorldStorage& lastWorld() const { return storage_; }

private:
	const std::vector<hlp::Person>& people_;
	const std::vector<hlp::Group>& groups_;
	HmpParams params_{};
	HmpWorldStorage storage_;
	bool maintain_rate_ = false;
	bool dirty_ = true;
};

}  // namespace humap_local_planner_b200
