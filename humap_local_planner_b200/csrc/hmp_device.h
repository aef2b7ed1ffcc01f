/*
 * hmp_device.h -- device-side data layout shared by the host code (hmp_api.cu) and the kernels
 * (hmp_kernels.cu). Everything here is plain-old-data that is memcpy'd to the GPU.
 *
 * Coordinates: the host translates the scene into a robot-centred frame (origin = robot position at
 * t = 0, NO rotation) before narrowing to FP32, so FP32 magnitudes stay below the costmap half-width
 * no matter where in the map frame the robot is. The absolute pose is carried in FP64 beside it for
 * costmap / MapGrid cell indexing (reference: costmap_2d::Costmap2D::worldToMap).
 */
#ifndef HMP_DEVICE_H_
#define HMP_DEVICE_H_

#include <stdint.h>

#include "../../include/hmp_planner.h"

#define HMP_DEV_MAX_KERNEL_PTS 9   /* centre + 8 offsets (RECTANGLE kernel) */
#ifndef HMP_WARPS_PER_BLOCK
#define HMP_WARPS_PER_BLOCK 8
#endif
#define HMP_THREADS_PER_BLOCK (32 * HMP_WARPS_PER_BLOCK)
#ifndef HMP_MIN_BLOCKS
#define HMP_MIN_BLOCKS 2
#endif
#ifndef HMP_F64_STATIC_UNROLL
#define HMP_F64_STATIC_UNROLL 2   /* static objects in flight per lane in the FP64 instances */
#endif
#ifndef HMP_F64_SWEEP_MIN_BLOCKS
#define HMP_F64_SWEEP_MIN_BLOCKS 2   /* resident blocks per SM the FP64 sweep (precision mode 1) is register-budgeted for */
#endif

/* Rollout-invariant record of one object treated with the STATIC interaction formulation
 * (reference StaticObject, world.h:24-41). d0 = object point - robot-side point at t = 0; during the
 * rollout dist_v = d0 - (c - c0) because World::predict only translates the robot-side point with the
 * centroid (world.cpp:107-110, SURVEY App. A #6). */
struct DevStatic {
	double d0x, d0y;
};

/* One object treated with the DYNAMIC formulation (DynamicObject, world.h:43-59). Geometry is FP64: the
 * dynamic interaction force can reach 1e4..1e6 N for amplified parameter sets and the twist amplifies any
 * rounding of its direction by |F| / m per step. */
struct DevDynamic {
	double d0x, d0y;  /* object point - robot-side point at t = 0                     */
	double vx, vy;    /* object velocity (global)                                     */
	double psi0;      /* yaw of the robot-side closest-point pose at t = 0            */
	double dir_beta;  /* wrap(direction(vel)), world.cpp:183                          */
	double speed;     /* |vel_xy|, world.cpp:180-181                                  */
	double _pad;
};

/* humap_local_planner::Person prediction source (person.h, trajectory.h:160-193) + covariances +
 * the speed-dependent personal-space variances (personal_space_intrusion_cost_function.cpp:55-58). */
struct DevPerson {
	float x, y, yaw, vth;      /* pose at t = 0 in the robot-centred frame, yaw rate     */
	float vx, vy, cos0, sin0;  /* velocity (global), cos/sin of yaw at t = 0             */
	float cxx, cxy, cyx, cyy;  /* position covariance                                    */
	float var_front, var_rear, var_side;
	float radius_eff;          /* person_model_radius + sqrt((cxx + cyy) / 2), heading-disturbance occupancy circle */
};

/* Group: static over the horizon (group.h:18-21) so the inverse covariance of the O-space Gaussian
 * (fformation_space_intrusion_cost_function.cpp:60-61 + pose covariance) is precomputed on the host:
 * q = ia dx^2 + 2 ib dx dy + ic dy^2, cost = exp(-q / 2). */
struct DevGroup {
	float x, y, ia, ib;
	float ic, _p0, _p1, _p2;
};

/* Per-scene header. Arrays follow in one blob; offsets are in bytes from the blob start. */
struct alignas(16) DevScene {
	double x0, y0, yaw0;          /* robot pose at t = 0 (absolute, map frame)                         */
	double u0x_d, u0y_d, u0w_d;   /* robot global velocity at t = 0 (computeVelocityGlobal(vel_, pose_)) */
	double glx_d, gly_d, gx_d, gy_d;  /* goal_local_ and goal_ relative to (x0, y0)                     */
	float u0x, u0y, u0w;          /* robot global velocity at t = 0 (computeVelocityGlobal(vel_, pose_)) */
	float vlx, vly, vlw;          /* vel_: current base-frame velocity (smoothness critics)            */
	float glx, gly;               /* goal_local_ - (x0, y0)                                            */
	float gx, gy;                 /* goal_       - (x0, y0)                                            */
	int32_t n_static0;            /* objects static at step 0                                          */
	int32_t n_static;             /* ... from step 1 on (adds objects re-classified by World::predict, App. A #5) */
	int32_t n_dynamic;            /* objects dynamic at step 0                                         */
	int32_t n_dynamic_later;      /* ... from step 1 on (prefix of the dynamic array)                  */
	int32_t n_people, n_groups;
	uint32_t off_static, off_dynamic, off_people, off_groups;
	uint32_t blob_bytes;          /* header + arrays, multiple of 16                                   */
	int32_t _pad;
	double hv_prev[HMP_NUM_MAPGRIDS];   /* highest_valid_cost_prev_ per MapGrid critic                    */
	/* equisampled generator (SimpleTrajectoryGenerator): Eigen::Vector3f pos_ of this scene (float stores of the UNWRAPPED pose;
	 * vel_ is vlx / vly / vlw above) and the number of its velocity samples -- the scenes of a batch share n_equi of DevParams
	 * (the largest count); candidates beyond a scene's own count are padding and count as rejected by the generator */
	float equi_px, equi_py, equi_pth;
	int32_t n_equi;
};

/* Flattened HumapConfig for the device: FP32 where the arithmetic is FP32, FP64 where the reference's
 * doubles decide an integer (cell index) or the final weighted sum. */
struct alignas(16) DevParams {
	/* --- time discretisation (social_trajectory_generator.cpp:324-328) */
	int32_t T;                    /* num_steps                                      */
	int32_t n_ttc_extra;          /* iterations of the TTC look-ahead loop (ttc_cost_function.cpp:100) */
	double dt_d;                  /* sim_time / T                                   */
	double ttc_rollout_time_d;
	float dt;
	float people_dt;
	/* --- limits (FP64: the twist / limit arithmetic of every step is done in double) */
	double max_vel_x, min_vel_x, max_vel_y, min_vel_y, max_vel_theta, min_vel_theta;
	double max_vel_trans, min_vel_trans;
	double acc_x, acc_y, acc_th, acc_decel;     /* acc_decel = hypot(acc_x, acc_y)  */
	double rot_comp;
	double back_max;               /* (min_vel_x < 0) ? |min_vel_x| : 0              */
	/* --- SFM */
	double mass, m_over_tau;
	double k_int, k_stat, k_dyn, min_force, max_force;
	double fov_half_d;             /* linear method: half angle = cfg.fov                */
	double fov_gauss_scale_d;      /* 1 / (sigma sqrt(2 pi)), sigma = cfg.fov            */
	double fov_neg_inv_2var_d;     /* -1 / (2 sigma^2)                                   */
	float fov_half, fov_gauss_scale, fov_neg_inv_2var;   /* FP32 copies for the static-object loop */
	int32_t maintain_rate;
	int32_t fov_method, filter_forces, disable_interaction;
	int32_t _pads;
	float base[9];                /* (float)cfg.{speed_desired, an, bn, cn, ap, bp, cp, aw, bw}: SFM float members */
	/* --- FIS */
	int32_t fis_on, fis_fov_method;
	double fis_force_factor_d, fis_range_d;
	double fis_fov_half_d;        /* linear method: cfg.fov / 2                        */
	double fis_gauss_scale_d, fis_neg_inv_2var_d;
	/* --- candidates */
	int32_t amp_n[HMP_NUM_AMPLIFIERS];
	int32_t n_grid;               /* product of amp_n                                  */
	int32_t n_candidates;         /* n_social + n_equi                                 */
	int32_t n_social;             /* n_grid + n_extra: candidates of the social generator */
	int32_t n_equi;               /* equisampled-velocity candidates appended after them (SimpleTrajectoryGenerator) */
	int32_t equi_continued;       /* continued_acceleration_                           */
	int32_t _pade;
	float equi_pos[3], equi_vel[3], equi_acc[3];   /* Eigen::Vector3f pos_, vel_, getAccLimits() of the generator */
	float _padq[3];
	/* --- costmap geometry */
	int32_t size_x, size_y;
	double origin_x, origin_y, resolution, inv_resolution;
	/* --- critics */
	double scale[HMP_NUM_COSTS];
	int32_t n_footprint;
	int32_t n_kernel_pts;         /* 1, 5 (CROSS) or 9 (RECTANGLE)                     */
	double kernel_dx[HMP_DEV_MAX_KERNEL_PTS];   /* offset of placement k in the robot frame: sep * (cos a_k, sin a_k) */
	double kernel_dy[HMP_DEV_MAX_KERNEL_PTS];
	double footprint_x[HMP_MAX_FOOTPRINT];
	double footprint_y[HMP_MAX_FOOTPRINT];
	int32_t occdist_sum;
	int32_t mg_stop_on_failure[HMP_NUM_MAPGRIDS];
	int32_t mg_kernel[HMP_NUM_MAPGRIDS];
	int32_t _padc;
	double mg_xshift[HMP_NUM_MAPGRIDS], mg_yshift[HMP_NUM_MAPGRIDS];
	float unsat_max_trans, unsat_max_x, unsat_max_y;
	float backward_penalty;
	float ttc_collision_distance, _padf;
	float hd_neg_inv_2var_fov, hd_dmin, hd_inv_max_speed;
	float ps_min_dist, ps_inv_max_speed;
	int32_t unsat_whole, hd_whole, psi_whole, fsi_whole, ps_whole;
};

/* Kernel argument block (passed by value). */
struct KernelArgs {
	const DevParams* params;         /* device; scene s reads the block params_stride * s bytes further on */
	const double* amp_values;        /* [10][HMP_MAX_AMP_VALUES] device                           */
	const double* extra_samples;     /* [n_extra][10] device, or null                             */
	const double* equi_samples;      /* [n_scenes][n_equi][3] target velocities (float values), or null */
	const uint8_t* scenes;           /* n_scenes blobs, stride scene_stride bytes                  */
	uint32_t scene_stride;
	int32_t n_scenes;
	const uint8_t* costmaps;         /* n_scenes costmaps, stride costmap_stride bytes (mult of 16) */
	uint32_t costmap_stride;
	int32_t costmap_in_smem;
	int32_t precise;                 /* 1: object loops and the FIS in FP64 (parity mode), 0: FP32 (fast mode) */
	int32_t cand_list_stride;        /* scene s reads cand_list + s * cand_list_stride (0: one list for all scenes) */
	const float* mapgrids;           /* [n_scenes][4][size_y * size_x]                            */
	/* selection */
	const int32_t* cand_list;        /* explicit candidate indices (detail mode) or null          */
	int32_t n_work;                  /* candidates per scene to evaluate                          */
	int32_t use_best_index;          /* detail mode: candidate = (int)best_out[scene][1]          */
	double* totals;                  /* [n_scenes][n_candidates] or null                          */
	unsigned long long* block_best;  /* scratch [n_scenes][gridDim.x][2] (cost bits, index)       */
	unsigned int* counters;          /* [n_scenes][4]: work ticket, done ticket, n_generated, n_valid */
	unsigned int* hv_out;            /* [n_scenes][4] highest_valid_cost (float bits, atomicMax)  */
	double* best_out;                /* [n_scenes][2]: best total, best index (as double)         */
	/* detail outputs (DETAIL kernel only) */
	double* d_costs;                 /* [n_work][14]                                               */
	double* d_seeds;                 /* [n_work][3]                                                */
	double* d_poses;                 /* [n_work][T][3]                                             */
	double* d_forces;                /* [n_work][T][8] or null                                     */
	int32_t* d_nposes;               /* [n_work] poses recorded (T, or fewer when the generator rejected) */
	const uint8_t* dilated;          /* [n_scenes] maps, stride costmap_stride: max costmap cost over the disc that contains every
	                                    cell the footprint critic can touch from a centre in that cell (255 outside the map), or
	                                    null: lets the obstacle critic skip poses that cannot raise its running maximum        */
	int32_t cand_offset;             /* sweep launches: candidate = work index + cand_offset (the equisampled sweep starts at n_social) */
	int32_t no_prune;                /* 1: the exact prunings of the max-type critics (obstacle: dilated map, people: distance bounds) are off (A/B) */
	const double* best_init;         /* [n_scenes][2] (total, index) of an earlier sweep over other candidates of the same pool, merged
	                                    into best_out by the last block (ties: lower index wins), or null                */
	int32_t forces_only;             /* detail launches of the force-field grid: rollout arithmetic only, no critic touches the costmap / MapGrids */
	int32_t _padf2;
	int32_t warps_per_ticket;        /* candidates a block takes per ticket (1..HMP_WARPS_PER_BLOCK, 0 = all): the refinement
	                                    pass spreads few candidates over many SMs to cut the latency of a rollout       */
	int32_t debug_cand;              /* thread-per-candidate sweep, parity hook: when d_costs is set, the raw critic values [14], the
	                                    seed twist (x, w) and the last pose (x, y, yaw) of this candidate are written there [19]      */
	/* highest_valid_cost_ with the reference's early-exit semantics (hv_early_exit_kernel): per candidate and MapGrid critic g,
	 * the weighted partial sum of the critics BEFORE g (what SimpleScoredSamplingPlanner::scoreTrajectory compares with the best
	 * so far; -1 if scoring cannot reach g: generator rejected the sample, an earlier critic was negative, or g has scale 0) and
	 * the largest valid cell value g looked up along the trajectory. Sweep launches only; null: not recorded. */
	double* hv_pre;                  /* [n_scenes][n_candidates][4] */
	float* hv_val;                   /* [n_scenes][n_candidates][4] */
	/* Thread-per-candidate sweep, deferred obstacle critic: scratch for the poses (x, y, yaw as three planes of blockDim.x doubles per
	 * step) of one ticket per block, [pose_n_slots][T][3][blockDim.x]; null: the critic walks the footprint inside the rollout
	 * loop. Needs `dilated`, the max aggregation and T * blockDim.x bytes of dynamic shared memory behind the packed static objects. */
	double* pose_scratch;
	/* ... one scratch SLOT per resident block, not per block of the grid: a block takes a free slot when it starts (atomicCAS on
	 * pose_slots, zeroed by the host before the launch; probing starts at its linear block index) and gives it back when it ends.
	 * pose_n_slots >= blocks that can be resident at once, so a free slot always exists. */
	unsigned int* pose_slots;
	int32_t pose_n_slots;
	uint32_t params_stride;          /* 0: one DevParams for every scene; sizeof(DevParams): one per scene (hmp_set_scene_costs) */
};

#endif
