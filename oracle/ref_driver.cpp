/*
 * ref_driver.cpp -- TEST INFRASTRUCTURE. Drives the reference's OWN first-party sources (compiled where they lie under
 * $HMP_REFERENCE_DIR by oracle/Makefile, target _ref/libhmp_ref.so, against the stand-in third-party headers of
 * oracle/ref_shim/) through the same flat inputs as the oracle's orc_plan, so that tests can compare
 *     reference sources  <->  oracle restatement (hmp_oracle.cpp)  <->  CUDA path
 * on identical scenes. Nothing under humap_local_planner_b200/ may include, link or load this.
 *
 * What is wired here follows HumapPlanner (reference src/humap_planner.cpp): critic list and order :68-82, parameter
 * pushes of updateCostParameters :868-928, world construction :365-370, generator_social_.initialise :1307-1314 and the
 * SimpleScoredSamplingPlanner loop of :1367 (scoreTrajectory / findBestTrajectory semantics, here with the raw critic
 * outputs recorded per candidate).
 */
#include <humap_local_planner/social_trajectory_generator.h>
#include <humap_local_planner/obstacle_separation_cost_function.h>
#include <humap_local_planner/map_grid_cost_function.h>
#include <humap_local_planner/unsaturated_translation_cost_function.h>
#include <humap_local_planner/ttc_cost_function.h>
#include <humap_local_planner/heading_change_smoothness_cost_function.h>
#include <humap_local_planner/velocity_smoothness_cost_function.h>
#include <humap_local_planner/heading_disturbance_cost_function.h>
#include <humap_local_planner/personal_space_intrusion_cost_function.h>
#include <humap_local_planner/fformation_space_intrusion_cost_function.h>
#include <humap_local_planner/passing_speed_cost_function.h>
#include <humap_local_planner/person.h>
#include <humap_local_planner/group.h>
#include <humap_local_planner/fuzz/processor.h>

#include <base_local_planner/map_grid_cost_function.h>
#include <base_local_planner/prefer_forward_cost_function.h>

#include <cstring>

#include "hmp_oracle.h"

namespace hlp = humap_local_planner;
using hlp::geometry::Pose;
using hlp::geometry::Vector;

namespace {

// Exposes the generator's sample list so that a candidate sub-range can be evaluated (multi-threaded CPU baseline).
class RefGenerator : public hlp::SocialTrajectoryGenerator {
public:
	size_t numSamples() const { return sample_amplifier_params_v_.size(); }
	const SampleAmplifierSet& sample(size_t i) const { return sample_amplifier_params_v_[i]; }
	void seek(unsigned int index) { next_sample_index_ = index; }
	unsigned int position() const { return next_sample_index_; }
	int steps(double speed_linear, double speed_angular) { return computeStepsNumber(speed_linear, speed_angular); }
};

// Access to highest_valid_cost_ of the customised MapGrid critic (map_grid_cost_function.cpp:78-79,87,135).
class RefMapGridCost : public hlp::MapGridCostFunction {
public:
	using hlp::MapGridCostFunction::MapGridCostFunction;
	void seedHighestValidCost(double v) { highest_valid_cost_ = v; }  // prepare() moves it to highest_valid_cost_prev_
	double highestValidCost() const { return highest_valid_cost_; }
};

thread_local const double* g_fill_grids[HMP_NUM_MAPGRIDS];
thread_local int g_fill_next = 0;

void fillGrid(base_local_planner::MapGrid& grid, const costmap_2d::Costmap2D& cm, const std::vector<geometry_msgs::PoseStamped>&, bool) {
	const double* src = g_fill_grids[g_fill_next++ % HMP_NUM_MAPGRIDS];
	for (unsigned int y = 0; y < cm.getSizeInCellsY(); ++y) {
		for (unsigned int x = 0; x < cm.getSizeInCellsX(); ++x) {
			grid(x, y).target_dist = src[(size_t)y * cm.getSizeInCellsX() + x];
		}
	}
}

}  // namespace

extern "C" {

// Same contract as orc_plan (oracle/hmp_oracle.h). out->forces is not filled.
int ref_plan(const OrcPlanInput* in, OrcPlanOutput* out) {
	const HmpParams& P = *in->params;
	const HmpWorld& hw = *in->world;

	// ---- configuration structs (humap_config.h) ------------------------------------------------
	auto sfm = std::make_shared<hlp::SfmParams>();
	sfm->fov = P.sfm.fov;
	sfm->fov_factor_method = (unsigned int)P.sfm.fov_factor_method;
	sfm->mass = P.sfm.mass;
	sfm->internal_force_factor = P.sfm.internal_force_factor;
	sfm->static_interaction_force_factor = P.sfm.static_interaction_force_factor;
	sfm->dynamic_interaction_force_factor = P.sfm.dynamic_interaction_force_factor;
	sfm->min_force = P.sfm.min_force;
	sfm->max_force = P.sfm.max_force;
	sfm->heterogenous_population = false;
	sfm->filter_forces = P.sfm.filter_forces != 0;
	sfm->disable_interaction_forces = P.sfm.disable_interaction_forces != 0;
	sfm->speed_desired = P.sfm.speed_desired;
	sfm->relaxation_time = P.sfm.relaxation_time;
	sfm->an = P.sfm.an;
	sfm->bn = P.sfm.bn;
	sfm->cn = P.sfm.cn;
	sfm->ap = P.sfm.ap;
	sfm->bp = P.sfm.bp;
	sfm->cp = P.sfm.cp;
	sfm->aw = P.sfm.aw;
	sfm->bw = P.sfm.bw;
	auto fis = std::make_shared<hlp::FisParams>();
	fis->force_factor = P.fis.force_factor;
	fis->human_action_range = P.fis.human_action_range;
	fis->fov = P.fis.fov;
	fis->fov_factor_method = (unsigned int)P.fis.fov_factor_method;
	auto limits = std::make_shared<hlp::PlannerLimitsParams>();
	limits->max_vel_trans = P.limits.max_vel_trans;
	limits->min_vel_trans = P.limits.min_vel_trans;
	limits->max_vel_x = P.limits.max_vel_x;
	limits->min_vel_x = P.limits.min_vel_x;
	limits->max_vel_y = P.limits.max_vel_y;
	limits->min_vel_y = P.limits.min_vel_y;
	limits->max_vel_theta = P.limits.max_vel_theta;
	limits->min_vel_theta = P.limits.min_vel_theta;
	limits->acc_lim_x = P.limits.acc_lim_x;
	limits->acc_lim_y = P.limits.acc_lim_y;
	limits->acc_lim_theta = P.limits.acc_lim_theta;
	limits->twist_rotation_compensation = P.limits.twist_rotation_compensation;
	limits->maintain_vel_components_rate = P.limits.maintain_vel_components_rate != 0;
	hlp::TrajectorySamplingParams ts;
	double* ts_fields[HMP_NUM_AMPLIFIERS][3] = {
	    {&ts.sfm_desired_speed_amplifier_min, &ts.sfm_desired_speed_amplifier_max, &ts.sfm_desired_speed_amplifier_granularity},
	    {&ts.sfm_an_amplifier_min, &ts.sfm_an_amplifier_max, &ts.sfm_an_amplifier_granularity},
	    {&ts.sfm_bn_amplifier_min, &ts.sfm_bn_amplifier_max, &ts.sfm_bn_amplifier_granularity},
	    {&ts.sfm_cn_amplifier_min, &ts.sfm_cn_amplifier_max, &ts.sfm_cn_amplifier_granularity},
	    {&ts.sfm_ap_amplifier_min, &ts.sfm_ap_amplifier_max, &ts.sfm_ap_amplifier_granularity},
	    {&ts.sfm_bp_amplifier_min, &ts.sfm_bp_amplifier_max, &ts.sfm_bp_amplifier_granularity},
	    {&ts.sfm_cp_amplifier_min, &ts.sfm_cp_amplifier_max, &ts.sfm_cp_amplifier_granularity},
	    {&ts.sfm_aw_amplifier_min, &ts.sfm_aw_amplifier_max, &ts.sfm_aw_amplifier_granularity},
	    {&ts.sfm_bw_amplifier_min, &ts.sfm_bw_amplifier_max, &ts.sfm_bw_amplifier_granularity},
	    {&ts.fis_as_amplifier_min, &ts.fis_as_amplifier_max, &ts.fis_as_amplifier_granularity},
	};
	for (int a = 0; a < HMP_NUM_AMPLIFIERS; ++a) {
		*ts_fields[a][0] = in->sampling->amp_min[a];
		*ts_fields[a][1] = in->sampling->amp_max[a];
		*ts_fields[a][2] = in->sampling->amp_granularity[a];
	}
	std::vector<hlp::SocialTrajectoryGenerator::SampleAmplifierSet> extra;
	for (int i = 0; i < in->n_extra; ++i) {
		hlp::SocialTrajectoryGenerator::SampleAmplifierSet s;
		const double* a = in->extra[i].amp;
		s.sfm_speed_desired_amplifier = a[HMP_AMP_SPEED];
		s.sfm_an_amplifier = a[HMP_AMP_AN];
		s.sfm_bn_amplifier = a[HMP_AMP_BN];
		s.sfm_cn_amplifier = a[HMP_AMP_CN];
		s.sfm_ap_amplifier = a[HMP_AMP_AP];
		s.sfm_bp_amplifier = a[HMP_AMP_BP];
		s.sfm_cp_amplifier = a[HMP_AMP_CP];
		s.sfm_aw_amplifier = a[HMP_AMP_AW];
		s.sfm_bw_amplifier = a[HMP_AMP_BW];
		s.fis_as_amplifier = a[HMP_AMP_AS];
		extra.push_back(s);
	}

	// ---- world, people, groups (humap_planner.cpp:365-370, humap_planner_ros.cpp:525-554) -------
	Pose pose(hw.robot_x, hw.robot_y, hw.robot_yaw);
	Vector vel(hw.vel_x, hw.vel_y, hw.vel_th);
	Vector vel_glob;
	hlp::computeVelocityGlobal(vel, pose, vel_glob);
	hlp::World world(pose, vel_glob, Pose(hw.goal_local_x, hw.goal_local_y, hw.goal_local_yaw), Pose(hw.goal_x, hw.goal_y, hw.goal_yaw));
	for (int i = 0; i < hw.n_obstacles; ++i) {
		const HmpObstacle& o = hw.obstacles[i];
		world.addObstacle(Pose(o.robot_x, o.robot_y, o.robot_yaw), Pose(o.obj_x, o.obj_y, o.obj_yaw), Vector(o.vx, o.vy, o.vth),
		                  o.force_dynamic != 0);
	}
	const unsigned int prediction_steps = (unsigned int)std::ceil(P.general.sim_time / P.general.sim_granularity);
	std::vector<hlp::Person> people;
	for (int i = 0; i < hw.n_people; ++i) {
		const HmpPerson& p = hw.people[i];
		people.push_back(hlp::Person(people_msgs_utils::Person(p.x, p.y, p.yaw, p.vx, p.vy, p.vth, p.cov_xx, p.cov_xy, p.cov_yx, p.cov_yy),
		                             P.general.people_prediction_dt, prediction_steps));
	}
	std::vector<hlp::Group> groups;
	for (int i = 0; i < hw.n_groups; ++i) {
		const HmpGroup& g = hw.groups[i];
		groups.push_back(hlp::Group(people_msgs_utils::Group(g.x, g.y, g.yaw, g.span_x, g.span_y, g.cov_xx, g.cov_xy, g.cov_yy),
		                            P.general.people_prediction_dt, prediction_steps));
	}

	// ---- critics (humap_planner.cpp:24-40, 58-82, 868-928) -------------------------------------
	costmap_2d::Costmap2D costmap(in->cells, (unsigned)in->size_x, (unsigned)in->size_y, in->resolution, in->origin_x, in->origin_y);
	const HmpCosts& C = P.costs;
	hlp::ObstacleSeparationCostFunction obstacle_costs(&costmap);
	base_local_planner::MapGridCostFunction path_costs(&costmap);
	base_local_planner::MapGridCostFunction goal_costs(&costmap, 0.0, 0.0, true);
	RefMapGridCost alignment_costs(&costmap);
	RefMapGridCost goal_front_costs(&costmap, 0.0, 0.0, true);
	hlp::UnsaturatedTranslationCostFunction unsaturated_trans_costs;
	base_local_planner::PreferForwardCostFunction backward_costs(0.0);
	hlp::TTCCostFunction ttc_costs(world);
	hlp::HeadingChangeSmoothnessCostFunction heading_change_smoothness_costs(vel);
	hlp::VelocitySmoothnessCostFunction velocity_smoothness_costs(vel);
	hlp::HeadingDisturbanceCostFunction heading_disturbance_costs(people);
	hlp::PersonalSpaceIntrusionCostFunction personal_space_costs(people);
	hlp::FformationSpaceIntrusionCostFunction fformation_space_costs(groups);
	hlp::PassingSpeedCostFunction passing_speed_costs(people);

	std::vector<geometry_msgs::Point> footprint;
	for (int i = 0; i < in->n_footprint; ++i) {
		geometry_msgs::Point p;
		p.x = in->footprint_xy[2 * i];
		p.y = in->footprint_xy[2 * i + 1];
		footprint.push_back(p);
	}
	obstacle_costs.setParams(P.limits.max_vel_trans, 0.2, 0.25, C.occdist_separation, (unsigned short)C.occdist_separation_kernel);
	obstacle_costs.setSumScores(C.occdist_sum_scores != 0);
	obstacle_costs.setFootprint(footprint);
	path_costs.setStopOnFailure(C.stop_on_failure[HMP_GRID_PATH] != 0);
	path_costs.setXShift(C.xshift[HMP_GRID_PATH]);
	path_costs.setYShift(C.yshift[HMP_GRID_PATH]);
	goal_costs.setStopOnFailure(C.stop_on_failure[HMP_GRID_GOAL] != 0);
	goal_costs.setXShift(C.xshift[HMP_GRID_GOAL]);
	goal_costs.setYShift(C.yshift[HMP_GRID_GOAL]);
	RefMapGridCost* custom[2] = {&alignment_costs, &goal_front_costs};
	const int custom_slot[2] = {HMP_GRID_ALIGNMENT, HMP_GRID_GOAL_FRONT};
	for (int k = 0; k < 2; ++k) {
		int g = custom_slot[k];
		custom[k]->setStopOnFailure(C.stop_on_failure[g] != 0);
		custom[k]->setXShift(C.xshift[g]);
		custom[k]->setYShift(C.yshift[g]);
		custom[k]->setKernelSize((unsigned int)C.neighbour_kernel_size[g]);
		custom[k]->setNeighborCellCostMultiplier(C.neighbour_cost_multiplier[g]);
		custom[k]->seedHighestValidCost(in->highest_valid_cost_prev[g]);
	}
	unsaturated_trans_costs.setParameters(C.unsat_max_trans_vel, C.unsat_max_vel_x, C.unsat_max_vel_y, C.unsat_whole_horizon != 0);
	backward_costs.setPenalty(C.backward_penalty);
	ttc_costs.setParameters(C.ttc_rollout_time, C.ttc_collision_distance);
	heading_disturbance_costs.setParameters(C.hd_fov_person, C.hd_person_model_radius, C.hd_robot_circumradius, C.hd_max_speed,
	                                        C.hd_whole_horizon != 0);
	personal_space_costs.setParameters(C.psi_whole_horizon != 0);
	fformation_space_costs.setParameters(C.fsi_whole_horizon != 0);
	passing_speed_costs.setParameters(C.ps_max_speed, C.ps_min_dist, C.ps_whole_horizon != 0);

	// order == HmpCostIndex == humap_planner.cpp:68-82
	std::vector<base_local_planner::TrajectoryCostFunction*> critics = {
	    &obstacle_costs, &path_costs, &goal_costs, &alignment_costs, &goal_front_costs, &unsaturated_trans_costs, &backward_costs,
	    &ttc_costs, &heading_change_smoothness_costs, &velocity_smoothness_costs, &heading_disturbance_costs, &personal_space_costs,
	    &fformation_space_costs, &passing_speed_costs};
	for (int k = 0; k < HMP_NUM_COSTS; ++k) critics[k]->setScale(C.scale[k]);

	// ---- generator (humap_planner.cpp:177-226, 1307-1314) ----------------------------------------
	RefGenerator generator;
	generator.setParameters(sfm, fis, P.general.sim_time, P.general.sim_granularity, P.general.angular_sim_granularity,
	                        P.general.sim_period, P.limits.maintain_vel_components_rate != 0, false, false, false, false);
	generator.initialise(world, vel, ts, limits, extra, P.sfm.mass, P.general.discretize_by_time != 0);

	// ---- SimpleScoredSamplingPlanner::findBestTrajectory semantics -----------------------------
	// prepare() in critic order; the MapGrid stand-in takes its cells from the caller's grids in that same order
	// (path, goal, alignment, goal_front = HmpMapGridIndex)
	for (int g = 0; g < HMP_NUM_MAPGRIDS; ++g) g_fill_grids[g] = in->target_dist[g];
	g_fill_next = 0;
	base_local_planner::MapGrid::fillHook() = fillGrid;
	ttc_costs.reset();  // updateLocalCosts, humap_planner.cpp:1115
	for (auto* c : critics) {
		if (!c->prepare()) return -1;
	}

	const int Cn = (int)generator.numSamples();
	const int c_begin = std::max(0, in->cand_begin);
	const int c_end = (in->cand_end <= 0) ? Cn : std::min(Cn, in->cand_end);
	const int T = generator.steps(std::hypot(hw.vel_x, hw.vel_y), hw.vel_th);
	const double NaN = std::numeric_limits<double>::quiet_NaN();

	base_local_planner::Trajectory loop_traj, best_traj;
	double best_cost = -1;
	int best_idx = -1, n_generated = 0, n_valid = 0;
	double best_raw[HMP_NUM_COSTS];
	generator.seek((unsigned)c_begin);
	while (generator.hasMoreTrajectories() && (int)generator.position() < c_end) {
		const int ci = (int)generator.position();
		bool ok = generator.nextTrajectory(loop_traj);
		if (out->generated) out->generated[ci] = ok ? 1 : 0;
		if (out->n_poses) out->n_poses[ci] = (int)loop_traj.getPointsSize();
		if (out->poses) {
			for (unsigned int i = 0; i < loop_traj.getPointsSize() && (int)i < T; ++i) {
				double* p = out->poses + ((size_t)ci * T + i) * 3;
				loop_traj.getPoint(i, p[0], p[1], p[2]);
			}
		}
		if (out->seeds) {
			out->seeds[3 * ci + 0] = loop_traj.xv_;
			out->seeds[3 * ci + 1] = loop_traj.yv_;
			out->seeds[3 * ci + 2] = loop_traj.thetav_;
		}
		double raw[HMP_NUM_COSTS];
		for (int k = 0; k < HMP_NUM_COSTS; ++k) raw[k] = NaN;
		if (!ok) {
			if (out->totals) out->totals[ci] = -1.0;
			if (out->costs) std::memcpy(out->costs + (size_t)ci * HMP_NUM_COSTS, raw, sizeof(raw));
			continue;
		}
		n_generated++;
		// scoreTrajectory(traj, best_traj_cost)
		double traj_cost = 0;
		for (int k = 0; k < HMP_NUM_COSTS; ++k) {
			if (critics[k]->getScale() == 0) continue;
			double cost = critics[k]->scoreTrajectory(loop_traj);
			raw[k] = cost;
			if (cost < 0) {
				traj_cost = cost;
				break;
			}
			if (cost != 0) cost *= critics[k]->getScale();
			traj_cost += cost;
			if (in->early_exit && best_cost > 0 && traj_cost > best_cost) break;
		}
		if (out->totals) out->totals[ci] = traj_cost;
		if (out->costs) std::memcpy(out->costs + (size_t)ci * HMP_NUM_COSTS, raw, sizeof(raw));
		if (traj_cost >= 0) {
			n_valid++;
			if (best_cost < 0 || traj_cost < best_cost) {
				best_cost = traj_cost;
				best_idx = ci;
				best_traj = loop_traj;
				std::memcpy(best_raw, raw, sizeof(raw));
			}
		}
		// the TTC critic keeps every predicted world of every scored trajectory for visualisation
		// (ttc_cost_function.cpp:66-70,83-85); drop them so that large candidate counts fit in memory
		ttc_costs.reset();
	}
	base_local_planner::MapGrid::fillHook() = nullptr;

	HmpResult& r = out->result;
	std::memset(&r, 0, sizeof(r));
	r.n_candidates = Cn;
	r.n_social = Cn;   // the second generator of the pool is third-party code (base_local_planner): not part of this build
	r.n_generated = n_generated;
	r.n_valid = n_valid;
	r.best_index = best_idx;
	r.status = best_idx >= 0 ? 0 : 1;
	r.best_total = best_idx >= 0 ? best_cost : -7.0;
	r.time_delta = P.general.sim_time / T;
	r.highest_valid_cost[HMP_GRID_ALIGNMENT] = alignment_costs.highestValidCost();
	r.highest_valid_cost[HMP_GRID_GOAL_FRONT] = goal_front_costs.highestValidCost();
	r.highest_valid_cost[HMP_GRID_PATH] = NaN;  // the upstream class has no such member
	r.highest_valid_cost[HMP_GRID_GOAL] = NaN;
	if (best_idx >= 0) {
		std::memcpy(r.costs, best_raw, sizeof(best_raw));
		r.xv = best_traj.xv_;
		r.yv = best_traj.yv_;
		r.thetav = best_traj.thetav_;
		r.time_delta = best_traj.time_delta_;
		r.n_poses = (int)best_traj.getPointsSize();
		const auto& s = generator.sample((size_t)best_idx);
		const double amps[HMP_NUM_AMPLIFIERS] = {s.sfm_speed_desired_amplifier, s.sfm_an_amplifier, s.sfm_bn_amplifier,
		                                         s.sfm_cn_amplifier, s.sfm_ap_amplifier, s.sfm_bp_amplifier, s.sfm_cp_amplifier,
		                                         s.sfm_aw_amplifier, s.sfm_bw_amplifier, s.fis_as_amplifier};
		std::memcpy(r.amplifiers, amps, sizeof(amps));
		if (out->best_poses) {
			for (unsigned int i = 0; i < best_traj.getPointsSize(); ++i) {
				best_traj.getPoint(i, out->best_poses[3 * i], out->best_poses[3 * i + 1], out->best_poses[3 * i + 2]);
			}
		}
	}
	return 0;
}

// HumapPlanner::computeCellCost (reference src/humap_planner.cpp:535-576, restated here because humap_planner.cpp itself is
// not part of this build) over the reference's own critics: humap MapGridCostFunction::getCellCosts,
// ObstacleSeparationCostFunction::getFootprintCost(px, py). Same contract as orc_cost_cloud.
int ref_cost_cloud(const OrcPlanInput* in, float* cloud6, uint8_t* valid) {
	const HmpCosts& C = in->params->costs;
	costmap_2d::Costmap2D costmap(in->cells, (unsigned)in->size_x, (unsigned)in->size_y, in->resolution, in->origin_x, in->origin_y);
	hlp::ObstacleSeparationCostFunction obstacle_costs(&costmap);
	base_local_planner::MapGridCostFunction path_costs(&costmap);
	base_local_planner::MapGridCostFunction goal_costs(&costmap, 0.0, 0.0, true);
	RefMapGridCost alignment_costs(&costmap);
	RefMapGridCost goal_front_costs(&costmap, 0.0, 0.0, true);
	std::vector<geometry_msgs::Point> footprint;
	for (int i = 0; i < in->n_footprint; ++i) {
		geometry_msgs::Point p;
		p.x = in->footprint_xy[2 * i];
		p.y = in->footprint_xy[2 * i + 1];
		footprint.push_back(p);
	}
	obstacle_costs.setParams(in->params->limits.max_vel_trans, 0.2, 0.25, C.occdist_separation, (unsigned short)C.occdist_separation_kernel);
	obstacle_costs.setFootprint(footprint);
	RefMapGridCost* custom[2] = {&alignment_costs, &goal_front_costs};
	const int slot[2] = {HMP_GRID_ALIGNMENT, HMP_GRID_GOAL_FRONT};
	for (int k = 0; k < 2; ++k) {
		custom[k]->setKernelSize((unsigned int)C.neighbour_kernel_size[slot[k]]);
		custom[k]->setNeighborCellCostMultiplier(C.neighbour_cost_multiplier[slot[k]]);
		custom[k]->seedHighestValidCost(in->highest_valid_cost_prev[slot[k]]);
	}
	path_costs.setScale(C.scale[HMP_COST_PATH]);
	goal_costs.setScale(C.scale[HMP_COST_GOAL]);
	obstacle_costs.setScale(C.scale[HMP_COST_OBSTACLE]);
	alignment_costs.setScale(C.scale[HMP_COST_ALIGNMENT]);
	goal_front_costs.setScale(C.scale[HMP_COST_GOAL_FRONT]);
	for (int g = 0; g < HMP_NUM_MAPGRIDS; ++g) g_fill_grids[g] = in->target_dist[g];
	g_fill_next = 0;
	base_local_planner::MapGrid::fillHook() = fillGrid;
	path_costs.prepare();
	goal_costs.prepare();
	alignment_costs.prepare();
	goal_front_costs.prepare();
	base_local_planner::MapGrid::fillHook() = nullptr;
	for (int cy = 0; cy < in->size_y; ++cy) {
		for (int cx = 0; cx < in->size_x; ++cx) {
			const size_t c = (size_t)cy * in->size_x + cx;
			float path_cost = path_costs.getCellCosts(cx, cy);
			float goal_cost = goal_costs.getCellCosts(cx, cy);
			float occ_cost = obstacle_costs.getFootprintCost((unsigned)cx, (unsigned)cy);
			float align_cost = alignment_costs.getCellCosts(cx, cy);
			float goal_front_cost = goal_front_costs.getCellCosts(cx, cy);
			bool cell_unreachable = path_cost == path_costs.obstacleCosts() || path_cost == path_costs.unreachableCellCosts() ||
			                        goal_cost == goal_costs.obstacleCosts() || goal_cost == goal_costs.unreachableCellCosts() ||
			                        occ_cost >= costmap_2d::LETHAL_OBSTACLE || occ_cost < costmap_2d::FREE_SPACE ||
			                        align_cost == alignment_costs.obstacleCosts() || align_cost == alignment_costs.unreachableCellCosts() ||
			                        goal_front_cost == goal_front_costs.obstacleCosts() ||
			                        goal_front_cost == goal_front_costs.unreachableCellCosts();
			valid[c] = cell_unreachable ? 0 : 1;
			float* o = cloud6 + c * 6;
			if (cell_unreachable) {
				for (int k = 0; k < 6; ++k) o[k] = 0.0f;
				continue;
			}
			path_cost *= path_costs.getScale();
			goal_cost *= goal_costs.getScale();
			occ_cost *= obstacle_costs.getScale();
			align_cost *= alignment_costs.getScale();
			goal_front_cost *= goal_front_costs.getScale();
			o[0] = path_cost + goal_cost + occ_cost + align_cost + goal_front_cost;
			o[1] = path_cost;
			o[2] = goal_cost;
			o[3] = occ_cost;
			o[4] = align_cost;
			o[5] = goal_front_cost;
		}
	}
	return 0;
}

// fuzz::Processor::process for one tuple; out3 = (value, membership, 1 if a term fired else 0). Same contract as
// orc_fis_process.
void ref_fis_process(double dir_alpha, double dir_beta, double rel_loc, double dist_angle, double out3[3]) {
	static thread_local hlp::fuzz::Processor proc;
	out3[0] = out3[1] = out3[2] = 0.0;
	if (!proc.process(dir_alpha, {dir_beta}, {rel_loc}, {dist_angle})) return;
	auto o = proc.getOutput();
	if (o.empty()) return;
	out3[0] = o[0].value;
	out3[1] = o[0].membership;
	out3[2] = (o[0].term_name == "none") ? 0.0 : 1.0;
}

int ref_num_candidates(const HmpSampling* s, int n_extra) {
	size_t total = 1;
	for (int a = 0; a < HMP_NUM_AMPLIFIERS; ++a) {
		total *= hlp::SocialTrajectoryGenerator::computeAmplifierSamples(s->amp_min[a], s->amp_max[a], s->amp_granularity[a], "").size();
	}
	return (int)(total + n_extra);
}

}  // extern "C"
