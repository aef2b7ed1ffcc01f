/*
 * hmp_planner.h -- C ABI of the B200-native trajectory sampling + scoring hot path.
 *
 * This is the drop-in boundary for ONE path of rayvburn/humap_local_planner: the call
 *     scored_sampling_planner_.findBestTrajectory(result_traj_, &traj_explored_)
 * at reference src/humap_planner.cpp:1367, i.e. SocialTrajectoryGenerator rollouts
 * (src/social_trajectory_generator.cpp:292-462) -> 14 TrajectoryCostFunction critics
 * (src/humap_planner.cpp:68-82) -> weighted total -> first strict minimum.
 *
 * Conventions (mirroring the reference, SURVEY.md section 8b):
 *  - plain C, plain pointers and sizes, no ownership transfer: every pointer argument is a
 *    caller-owned HOST buffer that is only read (or written, for outputs) during the call;
 *  - every function returns an int status: 0 ok, < 0 error (HMP_E_*); nothing throws;
 *  - one context per host thread and per GPU; a context is not re-entrant (the reference holds
 *    cfg_->getMutex() for the whole cycle, src/humap_planner.cpp:357);
 *  - negative COSTS are the reference's "invalid trajectory" codes and are preserved:
 *      -1  generator rejected the sample (velocity limits), social_trajectory_generator.cpp:319,411
 *      -4  MapGrid point off the map, map_grid_cost_function.cpp:166-170
 *      -6  footprint touches lethal / unknown / leaves the map, obstacle_separation_cost_function.cpp:225
 *      -7  trajectory centre off the map, obstacle_separation_cost_function.cpp:231
 *      -9  empty footprint, obstacle_separation_cost_function.cpp:92
 *      -10 / -12 TTC preconditions, ttc_cost_function.cpp:32,38
 *  - there is NO CPU fallback behind this ABI: if no CUDA device / kernel image is usable the
 *    calls fail with HMP_E_CUDA.
 */
#ifndef HMP_PLANNER_H_
#define HMP_PLANNER_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HMP_ABI_VERSION 2

/* ---- status codes ------------------------------------------------------------------------ */
#define HMP_OK            0
#define HMP_E_INVALID    -1   /* bad argument (null pointer, negative size, inconsistent sizes) */
#define HMP_E_CUDA       -2   /* CUDA runtime error or no usable device; see hmp_last_error()  */
#define HMP_E_NOT_READY  -3   /* a required hmp_set_* call is missing                           */
#define HMP_E_CAPACITY   -4   /* problem does not fit the configured limits (see HMP_MAX_*)     */

/* ---- compile-time limits ------------------------------------------------------------------ */
#define HMP_NUM_AMPLIFIERS      10     /* SampleAmplifierSet, social_trajectory_generator.h:28-52 */
#define HMP_MAX_AMP_VALUES      64     /* values per amplifier axis                                */
#define HMP_NUM_COSTS           14     /* critics, humap_planner.cpp:68-82                          */
#define HMP_NUM_MAPGRIDS        4
#define HMP_MAX_FOOTPRINT       64     /* footprint polygon vertices                                */
#define HMP_MAX_STEPS           512    /* rollout steps per candidate                               */

/* Critic order == evaluation order of the reference (src/humap_planner.cpp:68-82). */
enum HmpCostIndex {
	HMP_COST_OBSTACLE = 0,        /* ObstacleSeparationCostFunction           */
	HMP_COST_PATH = 1,            /* MapGridCostFunction path_costs_          */
	HMP_COST_GOAL = 2,            /* MapGridCostFunction goal_costs_          */
	HMP_COST_ALIGNMENT = 3,       /* MapGridCostFunction alignment_costs_     */
	HMP_COST_GOAL_FRONT = 4,      /* MapGridCostFunction goal_front_costs_    */
	HMP_COST_UNSATURATED = 5,     /* UnsaturatedTranslationCostFunction       */
	HMP_COST_BACKWARD = 6,        /* base_local_planner::PreferForwardCostFunction */
	HMP_COST_TTC = 7,             /* TTCCostFunction                          */
	HMP_COST_HEADING_CHANGE = 8,  /* HeadingChangeSmoothnessCostFunction      */
	HMP_COST_VEL_SMOOTHNESS = 9,  /* VelocitySmoothnessCostFunction           */
	HMP_COST_HEADING_DIST = 10,   /* HeadingDisturbanceCostFunction           */
	HMP_COST_PERSONAL_SPACE = 11, /* PersonalSpaceIntrusionCostFunction       */
	HMP_COST_FFORMATION = 12,     /* FformationSpaceIntrusionCostFunction     */
	HMP_COST_PASSING_SPEED = 13   /* PassingSpeedCostFunction                 */
};

/* Order of the MapGrid slots used by hmp_set_mapgrid. */
enum HmpMapGridIndex {
	HMP_GRID_PATH = 0,
	HMP_GRID_GOAL = 1,
	HMP_GRID_ALIGNMENT = 2,
	HMP_GRID_GOAL_FRONT = 3
};

/* Order of the amplifier axes == nesting order of the 10 loops, outermost first
 * (src/social_trajectory_generator.cpp:166-175). Candidate index c decodes as a mixed-radix
 * number with HMP_AMP_SPEED the most significant digit and HMP_AMP_AS the least significant. */
enum HmpAmplifierIndex {
	HMP_AMP_SPEED = 0, HMP_AMP_AN = 1, HMP_AMP_BN = 2, HMP_AMP_CN = 3, HMP_AMP_AP = 4,
	HMP_AMP_BP = 5, HMP_AMP_CP = 6, HMP_AMP_AW = 7, HMP_AMP_BW = 8, HMP_AMP_AS = 9
};

/* ---- parameters (flattened HumapConfig, include/humap_local_planner/humap_config.h) -------- */

/* PlannerLimitsParams (humap_config.h:13-24) + base_local_planner::LocalPlannerLimits fields used on the path */
typedef struct HmpLimits {
	double max_vel_trans, min_vel_trans;
	double max_vel_x, min_vel_x;
	double max_vel_y, min_vel_y;
	double max_vel_theta, min_vel_theta;
	double acc_lim_x, acc_lim_y, acc_lim_theta;
	double twist_rotation_compensation;
	int32_t maintain_vel_components_rate;
	int32_t _pad;
} HmpLimits;

/* GeneralParams subset (humap_config.h:26-58) */
typedef struct HmpGeneral {
	double sim_time;
	double sim_granularity;
	double angular_sim_granularity;
	double sim_period;
	/* dt of the constant-velocity people/group predictions (humap_planner_ros.cpp:530): the
	 * reference uses sim_granularity; kept separate because the robot uses sim_time / steps. */
	double people_prediction_dt;
	int32_t discretize_by_time;   /* planMovingRobot passes true (humap_planner.cpp:1313) */
	int32_t _pad;
} HmpGeneral;

/* SfmParams (humap_config.h:78-130). Equation parameters are doubles here; they are truncated to
 * float after multiplication by the amplifier exactly where the reference does it
 * (sfm/social_force_model.h:422-446 float members, social_trajectory_generator.cpp:627-637). */
typedef struct HmpSfm {
	double fov;                   /* HALF of the robot's field of view */
	double mass;
	double internal_force_factor;
	double static_interaction_force_factor;
	double dynamic_interaction_force_factor;
	double min_force, max_force;
	double speed_desired, relaxation_time;
	double an, bn, cn, ap, bp, cp, aw, bw;
	int32_t fov_factor_method;    /* 0 Gaussian, 1 linear (sfm::FovCalculationMethod) */
	int32_t filter_forces;
	int32_t disable_interaction_forces;
	int32_t _pad;
} HmpSfm;

/* FisParams (humap_config.h:137-152). `as` is not here: the reference never reads it (SURVEY App. A #13). */
typedef struct HmpFis {
	double force_factor;          /* <= 0 disables the fuzzy human-action force (social_conductor.cpp:30-35) */
	double human_action_range;
	double fov;                   /* passed as the FULL fov argument of computeFactorFOV (social_conductor.cpp:181-190) */
	int32_t fov_factor_method;    /* 0 Gaussian, 1 linear, other: factor 1.0 */
	int32_t _pad;
} HmpFis;

/* CostParams (humap_config.h:226-287) + the per-cycle values HumapPlanner pushes into its critics
 * (updateCostParameters humap_planner.cpp:868-928, updateLocalCosts :1054-1141). */
typedef struct HmpCosts {
	/* Effective scale of every critic as returned by getScale() when findBestTrajectory is
	 * entered (MapGrid scales already multiplied by the costmap resolution, dynamic per-cycle
	 * scales already applied). A zero scale skips the critic (SimpleScoredSamplingPlanner). */
	double scale[HMP_NUM_COSTS];
	/* ObstacleSeparationCostFunction */
	double occdist_separation;
	int32_t occdist_separation_kernel;   /* 0 CROSS, 1 RECTANGLE, else none */
	int32_t occdist_sum_scores;
	/* MapGridCostFunction x4, slots HmpMapGridIndex */
	double xshift[HMP_NUM_MAPGRIDS];
	double yshift[HMP_NUM_MAPGRIDS];
	int32_t stop_on_failure[HMP_NUM_MAPGRIDS];
	/* customised MapGrid heuristic (map_grid_cost_function.h: n_kernel_size_, n_cost_multiplier_);
	 * applies to HMP_GRID_ALIGNMENT and HMP_GRID_GOAL_FRONT only (the humap_local_planner class);
	 * path/goal use the upstream base_local_planner class. */
	int32_t neighbour_kernel_size[HMP_NUM_MAPGRIDS];
	double neighbour_cost_multiplier[HMP_NUM_MAPGRIDS];
	/* UnsaturatedTranslationCostFunction::setParameters */
	double unsat_max_trans_vel, unsat_max_vel_x, unsat_max_vel_y;
	/* PreferForwardCostFunction */
	double backward_penalty;
	/* TTCCostFunction::setParameters */
	double ttc_rollout_time, ttc_collision_distance;
	/* HeadingDisturbanceCostFunction::setParameters */
	double hd_fov_person;          /* FULL fov (2 * person_fov) */
	double hd_person_model_radius;
	double hd_robot_circumradius;
	double hd_max_speed;
	/* PassingSpeedCostFunction::setParameters */
	double ps_max_speed, ps_min_dist;
	int32_t unsat_whole_horizon;
	int32_t hd_whole_horizon;
	int32_t psi_whole_horizon;
	int32_t fsi_whole_horizon;
	int32_t ps_whole_horizon;
	int32_t _pad;
} HmpCosts;

typedef struct HmpParams {
	HmpLimits limits;
	HmpGeneral general;
	HmpSfm sfm;
	HmpFis fis;
	HmpCosts costs;
} HmpParams;

/* ---- per-cycle scene ---------------------------------------------------------------------- */

/* One World::addObstacle() call (src/world.cpp:43-63): closest-point pair + object velocity. */
typedef struct HmpObstacle {
	double robot_x, robot_y, robot_yaw;   /* pose of the robot-footprint point closest to the object */
	double obj_x, obj_y, obj_yaw;         /* pose of the object point closest to the robot          */
	double vx, vy, vth;                   /* object velocity, global frame                           */
	int32_t force_dynamic;                /* addObstacle(..., force_dynamic_type)                    */
	int32_t _pad;
} HmpObstacle;

/* humap_local_planner::Person = people_msgs_utils::Person + constant-velocity prediction (person.h) */
typedef struct HmpPerson {
	double x, y, yaw;
	double vx, vy, vth;
	double cov_xx, cov_xy, cov_yx, cov_yy;
} HmpPerson;

/* humap_local_planner::Group (group.h); groups are static over the horizon (group.h:18-21) */
typedef struct HmpGroup {
	double x, y, yaw;
	double span_x, span_y;
	double cov_xx, cov_xy, cov_yy;
} HmpGroup;

typedef struct HmpWorld {
	double robot_x, robot_y, robot_yaw;   /* pose_ (humap_planner.cpp:369)                     */
	double vel_x, vel_y, vel_th;          /* vel_: current BASE-frame velocity (:360)          */
	double goal_local_x, goal_local_y, goal_local_yaw;   /* goal_local_                         */
	double goal_x, goal_y, goal_yaw;      /* goal_                                              */
	const HmpObstacle* obstacles;         /* in World::addObstacle call order                   */
	const HmpPerson* people;              /* people_env_model_                                  */
	const HmpGroup* groups;               /* groups_env_model_                                  */
	int32_t n_obstacles, n_people, n_groups;
	int32_t _pad;
} HmpWorld;

/* TrajectorySamplingParams (humap_config.h:176-224): per axis {min, max, granularity}. */
typedef struct HmpSampling {
	double amp_min[HMP_NUM_AMPLIFIERS];
	double amp_max[HMP_NUM_AMPLIFIERS];
	double amp_granularity[HMP_NUM_AMPLIFIERS];
} HmpSampling;

/* Explicit sample, appended after the grid (initialise(..., additional_samples, ...),
 * social_trajectory_generator.cpp:51-70). Axis order HmpAmplifierIndex. */
typedef struct HmpSample {
	double amp[HMP_NUM_AMPLIFIERS];
} HmpSample;

/* The second generator of HumapPlanner's pool: base_local_planner::SimpleTrajectoryGenerator fed with equisampled
 * velocities (TrajectoryGeneration, humap_config.h:154-174; wiring src/humap_planner.cpp:196-203, :1317-1361). Its
 * candidates are appended after the social ones (generator_list order, humap_planner.cpp:85-88) and compete in the
 * same selection. Candidate index: [0, n_social) social grid + extra samples, [n_social, n_candidates) equisampled,
 * in the generator's own order (vx outermost, vth innermost). */
typedef struct HmpEquisampled {
	int32_t enabled;                 /* use_equisampled_velocities_generator                                     */
	int32_t vx_samples, vy_samples, vth_samples;   /* equisampled_vx / vy / vth                                   */
	double min_vel_x;                /* equisampled_min_vel_x                                                    */
	int32_t continued_acceleration;  /* equisampled_continued_acceleration (setParameters gets use_dwa = !this)   */
	int32_t _pad;
} HmpEquisampled;

/* ---- environment model (SURVEY 8f rank 3): inputs of HumapPlanner::createEnvironmentModel ------------------------- */
/* One obstacle of the ObstContainer the planner receives from costmap_converter (teb_local_planner obstacle types
 * wrapped by include/humap_local_planner/obstacles.h). Polygon vertices live in a shared pool (xy interleaved). */
enum HmpShapeType { HMP_SHAPE_POINT = 0, HMP_SHAPE_CIRCLE = 1, HMP_SHAPE_LINE = 2, HMP_SHAPE_POLYGON = 3 };
typedef struct HmpShape {
	int32_t type;                 /* HmpShapeType                                                     */
	int32_t n_vertices;           /* polygon: vertices in the pool; others: ignored                   */
	int32_t first_vertex;         /* polygon: index of its first vertex in the pool                   */
	int32_t _pad;
	double x, y;                  /* point / circle centre / line start                               */
	double x2, y2;                /* line end                                                         */
	double radius;                /* circle                                                           */
	double vx, vy;                /* getCentroidVelocity()                                            */
} HmpShape;
#define HMP_MAX_ENV_POLYGON 16       /* vertices of a PolygonRobotFootprint */
enum HmpRobotModel {
	HMP_ROBOT_POINT = 0,          /* PointRobotFootprint, robot_footprint_model.h:55-95        */
	HMP_ROBOT_CIRCULAR = 1,       /* CircularRobotFootprint, :98-140                           */
	HMP_ROBOT_TWO_CIRCLES = 2,    /* TwoCirclesRobotFootprint, :143-226                        */
	HMP_ROBOT_LINE = 3,           /* LineRobotFootprint, :228-294                              */
	HMP_ROBOT_POLYGON = 4         /* PolygonRobotFootprint, :296-346                           */
};
typedef struct HmpEnvParams {
	int32_t robot_model;          /* HmpRobotModel */
	int32_t obstacles_closest_num, people_closest_num, groups_closest_num;   /* GeneralParams, -1 = all   */
	double robot_radius;          /* getInscribedRadius()                                             */
	double person_model_radius;   /* GeneralParams::person_model_radius                               */
	double obstacle_extension_multiplier;   /* GeneralParams                                          */
	double ttc_collision_distance;           /* CostParams (enlargeObstacle threshold = 1.05 x this)   */
	double person_containment_rate;          /* HumapPlanner::PERSON_POLYGON_CONTAINMENT_RATE = 0.667  */
	int32_t obstacles_force_dynamic;         /* static_obj_interaction == INTERACTION_REPULSIVE_EVASIVE */
	int32_t people_force_dynamic;            /* SfmParams::human_force_formulation_dynamic              */
	/* footprint geometry of the non-circular models, robot frame (robot_radius stays getInscribedRadius() of the model) */
	double two_circles[4];                   /* front_offset, front_radius, rear_offset, rear_radius    */
	double line_xy[4];                       /* line_start (x, y), line_end (x, y)                      */
	int32_t n_polygon;                       /* vertices of the polygon model, <= HMP_MAX_ENV_POLYGON   */
	int32_t _pad;
	double polygon_xy[2 * HMP_MAX_ENV_POLYGON];
} HmpEnvParams;

/* ---- result ------------------------------------------------------------------------------- */
typedef struct HmpResult {
	int32_t status;                /* 0: a valid trajectory was found; 1: none valid (cost < 0)   */
	int32_t best_index;            /* index into the generator's sample list; -1 if none          */
	int32_t n_candidates;          /* samples in the list                                          */
	int32_t n_generated;           /* nextTrajectory() returned true                               */
	int32_t n_valid;               /* total cost >= 0                                              */
	int32_t n_poses;               /* poses of the winner written to `poses`                       */
	double best_total;             /* result_traj_.cost_ (weighted); -7 if none (humap_planner.cpp:1364) */
	double costs[HMP_NUM_COSTS];   /* RAW (unscaled) critic outputs of the winner, NaN if the critic was skipped */
	double xv, yv, thetav;         /* seed twist = twist of step 0 (social_trajectory_generator.cpp:415-419)   */
	double time_delta;             /* traj.time_delta_                                                         */
	double amplifiers[HMP_NUM_AMPLIFIERS];  /* the winner's SampleAmplifierSet                                */
	double highest_valid_cost[HMP_NUM_MAPGRIDS];  /* highest_valid_cost_ after the cycle (map_grid_cost_function.cpp:87,135) */
	double gpu_ms;                 /* device time of the cycle (CUDA events on the launching stream), milliseconds */
	double gpu_ms_select;          /* ... of the rollout + scoring + selection kernel alone                        */
	int32_t n_social;              /* candidates of the social generator (grid + extra); best_index >= n_social means the
	                                  winner came from the equisampled generator (amplifiers are NaN then)          */
	int32_t _pad;
} HmpResult;

typedef struct HmpContext HmpContext;

/* ---- lifecycle ---------------------------------------------------------------------------- */
/* Creates a context bound to CUDA device `device_id`. Returns NULL on failure (hmp_last_error()). */
HmpContext* hmp_create(int device_id);
void hmp_destroy(HmpContext* ctx);
/* Text of the last error on this thread (never NULL). */
const char* hmp_last_error(void);
int hmp_abi_version(void);

/* ---- configuration: replaces HumapPlanner::reconfigure -> generator_social_.setParameters +
 *      updateCostParameters (humap_planner.cpp:177-226, :868-928) and the per-cycle setScale /
 *      setXShift calls of updateLocalCosts (:1054-1141) ----------------------------------------- */
int hmp_set_params(HmpContext* ctx, const HmpParams* params);

/* Arithmetic of the per-object loops (static / dynamic interaction forces, fuzzy inference): 0 = FP32 (the fast
 * path), 1 = FP64 (parity mode: reproduces the FP64 reference to rounding noise; about 2x slower),
 * 2 (default) = FP32 sweep + FP64 refinement: all candidates are ranked in FP32, the leaders (valid candidates whose total is
 * within the window of hmp_set_refinement of the best) are rolled out and scored again in FP64, and the winner is the
 * first strict minimum of the refined totals -- the selection, the seed twist, the poses and the critic values returned
 * in HmpResult are then those of the FP64 path at a few percent of extra time.
 * Pose integration, twist / limit arithmetic, cell indexing and the weighted total are FP64 in every mode. */
int hmp_set_precision(HmpContext* ctx, int32_t fp64);
/* Mode 2 only: relative window above the best FP32 total (default 0.02) and the cap on leaders per scene (rounded up to a
 * multiple of 8; batches use at most 32). Until this is called (and for max_leaders = 0) the cap is the SM count of the device, so that the leaders
 * of a single-scene plan are one wave of block-cooperative FP64 rollouts. If more candidates fall inside the window it
 * shrinks to the widest window that holds at most the cap; fewer than 16 widens it (DESIGN.md 4b). No reference counterpart. */
int hmp_set_refinement(HmpContext* ctx, double rel_window, int32_t max_leaders);
/* Leaders re-scored in FP64 by the last plan of scene 0 (0 in modes 0 / 1), -1 if there is no plan. */
int hmp_last_num_leaders(HmpContext* ctx);
/* Single-scene plans in mode 2 run a second refinement round: the window is taken once more above the REFINED best of the
 * first round and the candidates between the two thresholds are refined as well, so that every candidate whose FP32 total
 * lies within the window of the final (FP64) best has been re-scored even when the FP32 best was a rollout with a large
 * FP32 error. Returns how many candidates that second round re-scored in the last plan (almost always 0). */
int hmp_last_num_leaders_round2(HmpContext* ctx);
/* Mode 2: when the FP64 evaluation rejects EVERY leader (e.g. the footprint of each touches a lethal cell by a margin FP32
 * missed), the FP32 selection is not handed out: the best of the remaining valid FP32 totals is taken and refined, up to 8
 * more rounds; if none yields a valid FP64 winner the plan reports status 1 / best_index -1 (no valid trajectory).
 * Returns how many such extra rounds the last plan needed (0 almost always). */
int hmp_last_fallback_rounds(HmpContext* ctx);
/* Mode 2, single-scene plans: the refinement knows both the FP32 and the FP64 total of every leader. A leader is UNRELIABLE when
 * the two differ by more than 1 % or disagree on validity; in an ordinary plan that is none or one of 1184, around a robot that
 * spins at its yaw-rate limit (chaotic rollouts, DESIGN.md 4b) it is dozens -- and then the true winner can sit far outside the
 * refined ranks. From `min_unreliable_leaders` such leaders on (default 24; 0 = never; HMP_ESCALATE in the environment presets
 * it) hmp_plan redoes the plan as an exact FP64 sweep (the mode-1 path on the resident inputs) and returns that result; the
 * leader counters keep describing the mode-2 pass. Batches (hmp_plan_batch) and hmp_replan_resident do not escalate.
 * hmp_last_unreliable_leaders / hmp_last_escalated report the count and whether the last plan was redone. No reference counterpart. */
int hmp_set_escalation(HmpContext* ctx, int32_t min_unreliable_leaders);
int hmp_last_unreliable_leaders(HmpContext* ctx);
int hmp_last_escalated(HmpContext* ctx);
/* Work layout of the FP32 sweep (modes 0 and 2): 0 (default) = automatic, 1 = one warp per candidate (lanes stride over the
 * objects; shortest latency for a few thousand candidates), 2 = one thread per candidate (a warp rolls out 32 candidates,
 * the per-step scalar section is issued once per 32; highest throughput from ~16k candidates per launch). Both layouts
 * evaluate the same FP32 arithmetic; only the summation order of the interaction forces differs. The environment variable
 * HMP_SWEEP_LAYOUT presets it at hmp_create. No reference counterpart. */
int hmp_set_sweep_layout(HmpContext* ctx, int32_t layout);
/* Layout the last plan's main sweep ran with: 0 = warp per candidate, else the block size of the thread-per-candidate kernel. */
int hmp_last_sweep_mode(HmpContext* ctx);

/* Replaces the costmap_2d::Costmap2D* every critic holds (row-major, index = my * size_x + mx). */
int hmp_set_costmap(HmpContext* ctx, const uint8_t* cells, int32_t size_x, int32_t size_y,
                    double origin_x, double origin_y, double resolution);

/* Replaces MapGridCostFunction::prepare() output (map_grid_cost_function.cpp:67-79): the wave-front
 * grid map_(x, y).target_dist of slot `grid`, row-major, size_x * size_y doubles, together with
 * highest_valid_cost_prev_ of that critic. Values are integers < 2^24 (cell counts, obstacleCosts(),
 * unreachableCellCosts()), which is checked. */
int hmp_set_mapgrid(HmpContext* ctx, int32_t grid, const double* target_dist, double highest_valid_cost_prev);

/* Replaces MapGridCostFunction::setTargetPoses + prepare() (map_grid_cost_function.cpp:63-79 ->
 * base_local_planner::MapGrid::setTargetCells / setLocalGoal + computeTargetDistance): computes the wave-front grid of
 * slot `grid` ON THE DEVICE from the plan poses (xy interleaved, map frame) and the costmap set by hmp_set_costmap, so
 * that neither the host wave front nor the 4-byte-per-cell upload is needed. local_goal = is_local_goal_function_. */
int hmp_compute_mapgrid(HmpContext* ctx, int32_t grid, const double* plan_xy, int32_t n_plan, int32_t local_goal,
                        double highest_valid_cost_prev);
/* Reads a MapGrid slot back (row-major doubles); diagnostics / parity tests. */
int hmp_get_mapgrid(HmpContext* ctx, int32_t grid, double* target_dist_out);

/* Replaces generator_vel_space_.setParameters (humap_planner.cpp:196-203) + the per-cycle initialise (:1317-1361) of the
 * equisampled generator for the following hmp_plan / hmp_plan_batch calls (NULL or enabled = 0 turns it off, which
 * is the state after hmp_create; in a batch every world gets its own velocity window and samples). The velocity window is derived per cycle from HmpLimits, HmpGeneral (sim_time,
 * sim_period), the robot velocity and the goal of the HmpWorld, as the reference does. */
int hmp_set_equisampled(HmpContext* ctx, const HmpEquisampled* eq);
/* Replaces ObstacleSeparationCostFunction::setFootprint (humap_planner.cpp:1059); xy interleaved. */
int hmp_set_footprint(HmpContext* ctx, const double* xy, int32_t n_points);

/* ---- the hot path: replaces generator_social_.initialise(...) (humap_planner.cpp:1307-1314) +
 *      scored_sampling_planner_.findBestTrajectory(...) (:1367) for the social generator.
 *      `extra`/`n_extra` may be NULL/0. `poses_out` (3 doubles per pose: x, y, yaw) may be NULL;
 *      at most poses_capacity poses are written. ------------------------------------------------ */
int hmp_plan(HmpContext* ctx, const HmpWorld* world, const HmpSampling* sampling,
             const HmpSample* extra, int32_t n_extra,
             HmpResult* result, double* poses_out, int32_t poses_capacity);

/* Same, for a batch of independent scenes that share params, costmap geometry and sampling but
 * have their own world, costmap cells and MapGrids (BASELINE config "batched scenes"); with hmp_set_scene_costs each scene
 * also has its own critic scales and MapGrid shifts. Scene s uses
 * worlds[s], cells + s * size_x * size_y, target_dist[g] + s * size_x * size_y. One launch.
 * cells = NULL reuses the costmaps of an earlier batch call, target_dist = NULL the grids left resident by
 * hmp_compute_mapgrid_batch / hmp_set_mapgrids_batch_f32 / an earlier batch; HMP_E_NOT_READY / HMP_E_INVALID if they do
 * not cover n_scenes scenes. target_dist values are checked like hmp_set_mapgrid's. */
int hmp_plan_batch(HmpContext* ctx, const HmpWorld* worlds, int32_t n_scenes,
                   const uint8_t* cells, const double* const target_dist[HMP_NUM_MAPGRIDS],
                   const double* highest_valid_cost_prev /* [n_scenes][4] or NULL */,
                   const HmpSampling* sampling, HmpResult* results);

/* Batch variant of hmp_compute_mapgrid (MapGridCostFunction::setTargetPoses + prepare(), src/map_grid_cost_function.cpp:63-79,
 * for every scene of a batch): the four wave-front grids of n_scenes scenes are computed on the device in one launch from
 * the per-scene costmaps and plans, and stay resident for the following hmp_plan_batch call (pass cells = NULL and
 * target_dist = NULL there). cells: n_scenes costmaps (scene s = cells + s * size_x * size_y), or NULL to reuse the costmaps
 * of an earlier batch call. plan_xy[g]: the poses (xy interleaved, map frame) of slot g of all scenes back to back;
 * plan_start[g][s] .. plan_start[g][s + 1] is scene s's range of POSES in it (n_scenes + 1 entries). local_goal[g] =
 * is_local_goal_function_ of slot g. This replaces the upload of 4 x 4 bytes per cell and scene by 1 byte per cell. */
int hmp_compute_mapgrid_batch(HmpContext* ctx, int32_t n_scenes, const uint8_t* cells, const double* const plan_xy[HMP_NUM_MAPGRIDS],
                              const int32_t* const plan_start[HMP_NUM_MAPGRIDS], const int32_t local_goal[HMP_NUM_MAPGRIDS]);
/* Uploads the wave-front grids of a batch as FLOATS (cell counts are exact in FP32 below 2^24) straight from the caller's
 * buffers, target_dist[g] + s * size_x * size_y = grid g of scene s; no conversion pass, full PCIe rate from pinned memory.
 * They stay resident for hmp_plan_batch(..., target_dist = NULL, ...). */
int hmp_set_mapgrids_batch_f32(HmpContext* ctx, int32_t n_scenes, const float* const target_dist[HMP_NUM_MAPGRIDS]);

/* Page-locked host memory for the buffers handed to the batch entry points every cycle (costmaps, plans, float grids): copies
 * from it run asynchronously at the full PCIe rate (the driver stages copies from pageable memory). NULL on failure. */
void* hmp_host_alloc(size_t bytes);
void hmp_host_free(void* p);

/* Per-world values of the per-cycle setScale / setXShift / setYShift calls (updateLocalCosts, humap_planner.cpp:1054-1141):
 * each robot of a batch derives them from its own state (distance to its goal, gap to the nearest person, goal inside a
 * group). */
typedef struct HmpSceneCosts {
	double scale[HMP_NUM_COSTS];      /* same meaning as HmpCosts.scale (MapGrid scales already x resolution); 0 skips the critic */
	double xshift[HMP_NUM_MAPGRIDS];  /* same meaning as HmpCosts.xshift / yshift                                               */
	double yshift[HMP_NUM_MAPGRIDS];
} HmpSceneCosts;
/* Sets the per-scene cost table of the following hmp_plan_batch calls: scene s uses costs[s] in place of HmpCosts.scale /
 * xshift / yshift; every other field of HmpParams stays shared. The table is copied. costs = NULL or n_scenes = 0 clears it,
 * which is the state after hmp_create. hmp_set_params does not clear it; hmp_plan ignores it; hmp_plan_batch with more
 * scenes than the table holds returns HMP_E_INVALID; hmp_replan_resident re-runs with the table the last plan used.
 * HMP_E_INVALID for a negative count, a NULL table with n_scenes > 0 or a non-finite value. */
int hmp_set_scene_costs(HmpContext* ctx, const HmpSceneCosts* costs, int32_t n_scenes);

/* Re-runs the last hmp_plan / hmp_plan_batch on the scene data still resident in device memory (only
 * the few-KB parameter block is re-sent and the result read back). `results` must hold results_capacity >=
 * hmp_last_num_scenes() records. No reference counterpart: it exists so that benchmarks can time the kernels with inputs
 * already in HBM. */
int hmp_replan_resident(HmpContext* ctx, HmpResult* results, int32_t results_capacity);
/* Scenes of the last plan (1 for hmp_plan), -1 if there is none. */
int hmp_last_num_scenes(HmpContext* ctx);

/* ---- diagnostics of the LAST hmp_plan (traj_explored_, humap_planner.cpp:1367,1969-2084) ------ */
/* Weighted total per candidate (negative = reference error code); n must equal n_candidates. */
int hmp_get_explored_totals(HmpContext* ctx, double* totals, int32_t n);
/* Re-runs the given candidates with full write-back: raw per-critic costs [n][HMP_NUM_COSTS]
 * (NaN where the reference would not have evaluated the critic), seed twist [n][3], and the poses
 * [n][n_steps][3]. Any output pointer may be NULL. Used by the parity tests and by the adapter for
 * traj_explored_. */
int hmp_explain(HmpContext* ctx, const int32_t* candidate_indices, int32_t n,
                double* costs_out, double* seeds_out, double* poses_out, int32_t* n_steps_out);

/* ---- diagnostics grids (SURVEY 8f rank 4) ------------------------------------------------------------------------ */
/* Replaces the per-cell loop of HumapPlannerROS::createCostGridPcl (src/humap_planner_ros.cpp:923-969) over
 * HumapPlanner::computeCellCost (src/humap_planner.cpp:535-576): for every costmap cell c = cy * size_x + cx,
 * cloud6[c] = {total, path, goal, layered (occ), alignment, goal_front} (scaled, FP32 like the reference's floats) and
 * valid[c] = 1, or valid[c] = 0 where computeCellCost returns false (a MapGrid value is obstacle / unreachable, or the
 * footprint at the cell centre with yaw 0 is in collision). Uses the costmap, MapGrids, footprint and scales currently
 * set. The caller emits the valid cells in the reference's order (cx outer, cy inner) to build the point cloud. */
int hmp_compute_cost_cloud(HmpContext* ctx, float* cloud6, uint8_t* valid);

/* Replaces HumapPlanner::createEnvironmentModel (src/humap_planner.cpp:930-1052 with extractNonPeopleObstacles :760-801,
 * selectRelevant humap_planner.h:387-427, calculateClosestPoints robot_footprint_model.h:89-140, enlargeObstacle
 * :681-758): filters obstacles that are really people, keeps the N closest obstacles / people / groups (metric relative to
 * robot_pose = pose_), and computes on the device, for the robot placed at pose_ref, the closest-point pair of every kept
 * obstacle (enlarged) and of every kept person (a circle of person_model_radius). Output = the World::addObstacle call
 * sequence (obstacles first, then people) ready for HmpWorld.obstacles, plus the indices of the kept people / groups
 * (people_env_model_, groups_env_model_). *n_obstacles_out holds the capacity on entry. Ties of the N-closest metric are
 * resolved by input order (the reference's std::sort leaves them unspecified). All five footprint models of
 * robot_footprint_model.h (point, circular, two circles, line, polygon); their calculateClosestPoints are restated as written,
 * including that the two-circle model returns the shortest VECTOR as the robot-side "pose" (:203-223) and that the polygon
 * model measures against the footprint's robot-frame vertices (:340-344). */
int hmp_build_environment(HmpContext* ctx, const HmpEnvParams* env, const double robot_pose[3], const double pose_ref[3],
                          const HmpShape* shapes, int32_t n_shapes, const double* vertices_xy, int32_t n_vertices,
                          const HmpPerson* people, int32_t n_people, const HmpGroup* groups, int32_t n_groups,
                          HmpObstacle* obstacles_out, int32_t* n_obstacles_out, int32_t* people_selected,
                          int32_t* n_people_selected, int32_t* groups_selected, int32_t* n_groups_selected);
/* Replaces the loop of Visualization::publishGrid (src/visualization.cpp:246-286) over
 * HumapPlanner::computeForceAtPosition (src/humap_planner.cpp:652-678): for each of the n positions the robot is placed
 * there with the yaw of robot_pose, the environment model is rebuilt (as above; the N-closest selection stays relative to
 * robot_pose), and the social force model + fuzzy conductor are evaluated once with unit amplifiers and dt = sim_period
 * (generateTrajectoryWithoutPlanning, social_trajectory_generator.cpp:504-527). forces_out[i] = {internal.xy, dynamic.xy,
 * static.xy, human-action.xy}; the reference's force_total is their sum. world carries vel_, goal_local_, goal_. */
int hmp_compute_force_grid(HmpContext* ctx, const HmpEnvParams* env, const HmpWorld* world, const double* positions_xy,
                           int32_t n_positions, const HmpShape* shapes, int32_t n_shapes, const double* vertices_xy,
                           int32_t n_vertices, double* forces_out);

/* ---- device-side helpers exposed for bit-exact parity tests (no reference counterpart) -------- */
/* costmap_2d::Costmap2D::worldToMap on the device for n points; ok[i] = 0/1. */
int hmp_debug_world_to_map(HmpContext* ctx, const double* wx, const double* wy, int32_t n,
                           int32_t* mx, int32_t* my, int32_t* ok);
/* CostmapModel::footprintCost on the device for n poses (x, y, yaw) with the configured footprint. */
int hmp_debug_footprint_cost(HmpContext* ctx, const double* xyt, int32_t n, double* cost);

/* fuzz::Processor::process (src/fuzz/processor.cpp:200-271) on the device for n tuples
 * (dir_alpha, dir_beta, rel_loc, dist_angle); out2 = (crisp direction, membership of the winning term). */
int hmp_debug_fis(HmpContext* ctx, const double* in4, int32_t n, double* out2);
/* Per-step forces of the candidates of the last hmp_explain call: [n][T][8] doubles
 * (internal.xy, dynamic.xy, static.xy, human-action.xy), social_trajectory_generator.cpp:701-704. */
int hmp_debug_last_forces(HmpContext* ctx, int32_t n, double* forces_out);
/* FP32 FFMA throughput of the device measured with independent FMA chains at the main sweep's launch shape (TFLOP/s): the
 * measured denominator of the roofline fraction bench.py reports beside the nominal one. */
int hmp_debug_measure_fp32_peak(HmpContext* ctx, double* tflops_out);
/* Re-runs the last single-scene plan and returns what the thread-per-candidate SWEEP itself computed for one social candidate:
 * out19 = the 14 raw critic values, the seed twist (x, w) and the pose after the last step (x, y, yaw); all NaN if the sweep
 * ran in the warp-per-candidate layout. hmp_explain always runs one warp per candidate, so only this hook can show a deviation
 * of the sweep's own arithmetic. */
int hmp_debug_sweep_candidate(HmpContext* ctx, int32_t candidate, double* out19);
/* Rollout steps of the last plan (SocialTrajectoryGenerator::computeStepsNumber), -1 if none. */
int hmp_num_steps(HmpContext* ctx);

/* Number of kernels this library launched on the context since creation (bench.py's gpu_launches). */
int64_t hmp_launch_count(HmpContext* ctx);

#ifdef __cplusplus
}
#endif
#endif /* HMP_PLANNER_H_ */
