/*
 * hmp_api.cu -- host side of the C ABI declared in include/hmp_planner.h.
 *
 * Flattens HumapConfig-like parameters and the per-cycle World into the device layout of hmp_device.h,
 * uploads them, launches the rollout+scoring+selection kernel (hmp_kernels.cu) and reads back the
 * winner. There is NO CPU implementation of the path in this library: if CUDA is unavailable every
 * entry point fails with HMP_E_CUDA.
 */
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <limits>
#include <new>
#include <numeric>
#include <thread>
#include <vector>

#include "hmp_device.h"

static_assert(sizeof(DevParams) % 16 == 0, "DevParams is copied with cp.async.bulk (16-byte granules)");
static_assert(sizeof(DevScene) % 16 == 0, "DevScene header must keep the arrays 16-byte aligned");
static_assert(sizeof(DevDynamic) == 64 && sizeof(DevPerson) == 64 && sizeof(DevGroup) == 32 && sizeof(DevStatic) == 16,
              "device record sizes are relied upon by the float4 loads in the kernel");

extern "C" size_t hmp_dev_smem_bytes(uint32_t scene_stride, uint32_t costmap_stride, int costmap_in_smem);
extern "C" cudaError_t hmp_dev_configure(size_t max_smem);
extern "C" cudaError_t hmp_dev_occupancy(size_t smem, int precise, int* blocks_per_sm);
extern "C" cudaError_t hmp_dev_occupancy_tpc(size_t smem, int threads, int rich, int* blocks_per_sm);
extern "C" cudaError_t hmp_dev_occupancy_tpc64(size_t smem, int threads, int* blocks_per_sm);
extern "C" int hmp_dev_tpc_max_threads();
extern "C" int hmp_dev_tpc64_max_threads();
extern "C" size_t hmp_dev_tpc_extra_smem(uint32_t scene_stride);
extern "C" cudaError_t hmp_dev_launch_plan(const KernelArgs* args, int blocks_x, int detail, size_t smem, cudaStream_t stream);
extern "C" cudaError_t hmp_dev_launch_env_filter(const HmpShape* shapes, int n_shapes, const double* verts, const HmpPerson* people, int n_people,
                                                 double person_radius, double containment_rate, double rx, double ry, int32_t* keep,
                                                 double* metric, cudaStream_t stream);
extern "C" cudaError_t hmp_dev_launch_env_closest(const HmpShape* shapes, const double* verts, const HmpPerson* people, const int32_t* objects,
                                                  const int32_t* counts, int row_stride, const double* positions_xy, int n_positions, double yaw,
                                                  const HmpEnvParams* env, HmpObstacle* out, cudaStream_t stream);
extern "C" cudaError_t hmp_dev_launch_env_select(const int32_t* keep, const double* metric, int n_shapes, const HmpPerson* people, int n_people,
                                                 const HmpGroup* groups, int n_groups, double rx, double ry, int n_obst_max, int n_people_max,
                                                 int n_groups_max, double* scratch_metric, int32_t* objects_out, int32_t* people_out,
                                                 int32_t* groups_out, int32_t* counts_out, cudaStream_t stream);
extern "C" cudaError_t hmp_dev_launch_dilate(const uint8_t* cm, int sx, int sy, uint32_t stride, float radius, uint8_t* out,
                                             int n_scenes, cudaStream_t stream);
extern "C" cudaError_t hmp_dev_launch_collect_leaders(const double* totals, int C, const double* best_out, double rel_window, int K,
                                                      int32_t* leaders, int32_t* count, const double* thr_lo, double* thr_out,
                                                      int min_leaders, int n_scenes, const int32_t* active, cudaStream_t stream);
extern "C" cudaError_t hmp_dev_launch_hv_early_exit(const double* totals, const double* hv_pre, const float* hv_val, int C,
                                                    unsigned int* hv_out, int n_scenes, cudaStream_t stream);
extern "C" cudaError_t hmp_dev_launch_collect_topk(const double* totals, int C, const double* best_out, int K, double round2_window,
                                                   int32_t* leaders, int32_t* count, double* thr_out, int n_scenes, const int32_t* active,
                                                   cudaStream_t stream);
extern "C" cudaError_t hmp_dev_launch_fill_leaders(int32_t* leaders, int K, int C, int32_t* count, cudaStream_t stream);
extern "C" cudaError_t hmp_dev_launch_reselect(const double* totals, int C, double* best_out, const int32_t* active, int n_scenes,
                                               cudaStream_t stream);
extern "C" cudaError_t hmp_dev_launch_refine_select(const int32_t* leaders, int K, int C, int T, const double* r_totals,
                                                    const double* r_costs, const double* r_seeds, const double* r_poses,
                                                    const int32_t* r_nposes, double* totals_full, double* best_out, double* o_costs,
                                                    double* o_seeds, double* o_poses, double* o_total, int32_t* o_nposes,
                                                    int n_scenes, int merge, const int32_t* active, int32_t* unreliable_out, cudaStream_t stream);
extern "C" cudaError_t hmp_dev_launch_world_to_map(const DevParams* P, const double* wx, const double* wy, int n, int* mx,
                                                   int* my, int* ok, cudaStream_t stream);
extern "C" cudaError_t hmp_dev_launch_footprint_cost(const DevParams* P, const uint8_t* cm, const double* xyt, int n,
                                                     double* cost, cudaStream_t stream);
extern "C" size_t hmp_dev_wavefront_smem(int sx, int sy);
extern "C" cudaError_t hmp_dev_launch_wavefront(const uint8_t* cms, uint32_t cm_stride, int sx, int sy, const int* seeds,
                                                const int* seed_off, float* dist, int n_grids, int n_scenes, cudaStream_t stream);
extern "C" cudaError_t hmp_dev_launch_fis(const double* in4, int n, double* out2, int precise, cudaStream_t stream);
extern "C" cudaError_t hmp_dev_launch_ffma_peak(int blocks, int iters, float* sink, cudaStream_t stream);
extern "C" cudaError_t hmp_dev_launch_cost_cloud(const DevParams* P, int n_cells, const uint8_t* cm, const float* mapgrids, const double* hv,
                                                 float* out, uint8_t* valid, cudaStream_t stream);

namespace {

thread_local char g_err[512] = "";

void set_err(const char* fmt, ...) {
	va_list ap;
	va_start(ap, fmt);
	vsnprintf(g_err, sizeof(g_err), fmt, ap);
	va_end(ap);
}

#define CU(call)                                                                              \
	do {                                                                                      \
		cudaError_t e__ = (call);                                                             \
		if (e__ != cudaSuccess) {                                                             \
			set_err("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
			return HMP_E_CUDA;                                                                \
		}                                                                                     \
	} while (0)

constexpr double PI = 3.14159265358979323846;
inline double wrap(double a) { return std::atan2(std::sin(a), std::cos(a)); }

// A device buffer that only grows.
struct DevBuf {
	void* p = nullptr;
	size_t cap = 0;
	int ensure(size_t bytes) {
		if (bytes <= cap) return HMP_OK;
		if (p) cudaFree(p);
		p = nullptr;
		cap = 0;
		size_t want = std::max<size_t>(bytes, 256);
		CU(cudaMalloc(&p, want));
		cap = want;
		return HMP_OK;
	}
	void release() {
		if (p) cudaFree(p);
		p = nullptr;
		cap = 0;
	}
};
struct HostBuf {  // pinned
	void* p = nullptr;
	size_t cap = 0;
	int ensure(size_t bytes) {
		if (bytes <= cap) return HMP_OK;
		if (p) cudaFreeHost(p);
		p = nullptr;
		cap = 0;
		size_t want = std::max<size_t>(bytes, 256);
		CU(cudaMallocHost(&p, want));
		cap = want;
		return HMP_OK;
	}
	void release() {
		if (p) cudaFreeHost(p);
		p = nullptr;
		cap = 0;
	}
};

// SocialTrajectoryGenerator::computeAmplifierSamples, social_trajectory_generator.cpp:465-498
int amplifier_samples(double amp_min, double amp_max, double granularity, double* out, int cap) {
	int n = 0;
	double span = (amp_max - amp_min) / granularity;
	if (!(span == span) || std::fabs(span) > 1e9) return -1;
	int num = (int)std::ceil(span);
	for (int i = 0; i <= num; i++) {
		double v = amp_min + granularity * i;
		if (n >= cap) return -1;
		if (v > amp_max) {
			out[n++] = amp_max;
			break;
		}
		out[n++] = v;
	}
	if (n == 0) out[n++] = 0.0;
	return n;
}

}  // namespace

struct HmpContext {
	int device = 0;
	int sm_count = 0;
	size_t max_smem_optin = 0;
	cudaStream_t stream = nullptr;
	cudaStream_t stream2 = nullptr;   // FP64 rollouts of a small pool, beside the FP32 sweep (run_cycle)
	cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
	cudaEvent_t ev0 = nullptr, ev1 = nullptr, evm = nullptr;
	int64_t launches = 0;

	HmpParams params{};
	bool have_params = false;
	int size_x = 0, size_y = 0;
	double origin_x = 0, origin_y = 0, resolution = 0;
	bool have_costmap = false;
	bool have_grid[HMP_NUM_MAPGRIDS] = {false, false, false, false};
	double hv_prev[HMP_NUM_MAPGRIDS] = {0, 0, 0, 0};
	std::vector<double> footprint;
	std::vector<uint8_t> h_cells;   // host copy of the single-scene costmap (scene 0 after a batch): seed test of the device wave front
	int costmap_scenes = 0;         // scenes whose costmap is resident in d_costmaps (1 after hmp_set_costmap, n after a batch upload)
	int batch_grid_scenes = 0;      // scenes whose four MapGrids are resident in d_mapgrids from a batch call (0: single-scene slots only)
	bool have_footprint = false;
	int precise = 2;                 // 0 FP32, 1 FP64, 2 (default) FP32 sweep + FP64 refinement of the leaders
	double refine_window = 0.02;     // leaders: FP32 total <= best * (1 + window)
	int refine_max_leaders = 0;      // per scene; 0 (default) = the SM count (single-scene plans: one block-cooperative FP64 rollout
	                                 // per SM, a single wave); batches use min(this or 256, 32)
	int last_n_leaders = 0;
	int last_n_leaders2 = 0;        // ... of the second round (single-scene plans)
	int last_explain_n = 0, last_explain_T = 0;   // shape of the forces hmp_explain left in h_out (0: overwritten since)
	int debug_cand = -1;            // hmp_debug_sweep_candidate
	int last_unreliable = 0;        // leaders of the last plan whose FP32 total was off by > 1 % or whose validity differed (mode 2, round 1)
	int escalate_min = 24;          // hmp_set_escalation: from this many unreliable leaders the plan is redone in FP64 (0: never)
	int last_escalated = 0;         // the last plan was redone in FP64 for that reason
	int last_fallback_rounds = 0;   // extra refinement rounds of the last plan because FP64 rejected every leader (mode 2)
	std::vector<HmpSceneCosts> scene_costs;   // per-scene scales / shifts of hmp_plan_batch (hmp_set_scene_costs); empty: shared params
	HmpEquisampled equi{};           // second generator of the pool (hmp_set_equisampled); enabled = 0 after hmp_create
	std::vector<double> last_equi;   // its velocity samples of the last plan ([n][3])
	bool dilated_dirty = true;       // costmap cells, footprint or separation changed since the dilated map was built
	int dilated_scenes = 0;
	int prune_obstacle = 1;          // HMP_NO_PRUNE=1 in the environment disables the dilated-map pruning (A/B timing)
	HostBuf h_grid_stage[2];         // pinned staging of hmp_plan_batch's MapGrids (float), double-buffered
	cudaEvent_t grid_stage_ev[2] = {nullptr, nullptr};
	int sweep_layout = 0;            // FP32 sweep: 0 auto, 1 one warp per candidate, 2 one thread per candidate (hmp_set_sweep_layout)
	int tpc_bps = 0;                 // resident blocks per SM of the last thread-per-candidate launch shape (launch_main)
	int tpc_defer = 0;               // the last launch_main reserved shared memory for the deferred obstacle critic of the thread-per-candidate sweep
	int last_sweep_mode = 0;         // launch mode of the last main sweep (0 warp per candidate, else threads per block of the thread-per-candidate kernel)

	DevBuf d_seeds[HMP_NUM_MAPGRIDS];
	HostBuf h_seeds[HMP_NUM_MAPGRIDS];
	cudaEvent_t seeds_event[HMP_NUM_MAPGRIDS] = {nullptr, nullptr, nullptr, nullptr};
	cudaStream_t wf_stream[HMP_NUM_MAPGRIDS] = {nullptr, nullptr, nullptr, nullptr};   // the four wave fronts of a cycle run side by side
	cudaEvent_t wf_done[HMP_NUM_MAPGRIDS] = {nullptr, nullptr, nullptr, nullptr};
	bool seeds_event_valid[HMP_NUM_MAPGRIDS] = {false, false, false, false};
	bool wavefront_pending[HMP_NUM_MAPGRIDS] = {false, false, false, false};   // slot 0 also stands for a hmp_compute_mapgrid_batch
	// wf_done[g] was last recorded by a batch of wave fronts (on wf_stream[0]), which writes slot g too: the next single-grid wave
	// front of the slot waits for it on the device. A join does not clear this, it orders ctx->stream only.
	bool wf_after_batch[HMP_NUM_MAPGRIDS] = {false, false, false, false};
	DevBuf d_params, d_amp, d_extra, d_scenes, d_costmaps, d_mapgrids, d_totals, d_block_best, d_ctrl, d_detail, d_dbg, d_refine, d_dilated, d_equi, d_env, d_mask, d_hvrec, d_posescr, d_poseslots;
	HostBuf h_stage, h_out;
	HostBuf h_params;  // pinned staging of the per-scene DevParams copies of a batch with a cost table
	HostBuf h_small;   // pinned words read back inside a cycle: [0..1] leader counts of the two refinement rounds, [2] unreliable leaders
	HostBuf h_grid[HMP_NUM_MAPGRIDS];   // pinned staging of hmp_set_mapgrid, one per slot
	uint32_t costmap_stride = 0;

	// last plan
	int last_n_candidates = 0, last_T = 0, last_n_scenes = 0;
	uint32_t last_scene_stride = 0;
	DevParams last_dev_params{};
	std::vector<HmpSceneCosts> last_scene_costs;   // the table the last plan ran with (empty: none)
	std::vector<double> last_amp_table;
	std::vector<HmpSample> last_extra;
	bool last_valid = false;
};

namespace {

// ---- flattening ------------------------------------------------------------------------------------
int compute_steps(const HmpGeneral& g, double speed_linear, double speed_angular) {
	// SocialTrajectoryGenerator::computeStepsNumber, social_trajectory_generator.cpp:584-599
	if (g.discretize_by_time) return (int)std::ceil(g.sim_time / g.sim_granularity);
	double sd = speed_linear * g.sim_time;
	double sa = std::fabs(speed_angular) * g.sim_time;
	return (int)std::ceil(std::max(sd / g.sim_granularity, sa / g.angular_sim_granularity));
}

int build_dev_params(const HmpContext* ctx, const HmpSampling* sampling, int n_extra, int T, DevParams& D,
                     std::vector<double>& amp_table) {
	const HmpParams& P = ctx->params;
	std::memset(&D, 0, sizeof(D));
	D.T = T;
	D.dt_d = P.general.sim_time / T;
	D.dt = (float)D.dt_d;
	D.people_dt = (float)P.general.people_prediction_dt;
	D.ttc_rollout_time_d = P.costs.ttc_rollout_time;
	{
		int n = 0;  // iterations of `for (double t = 0.0; t < ttc_rollout_time_; t += dt)`, ttc_cost_function.cpp:100
		for (double t = 0.0; t < P.costs.ttc_rollout_time; t += D.dt_d) {
			if (++n > 100000) break;
		}
		D.n_ttc_extra = n;
	}
	const HmpLimits& L = P.limits;
	D.max_vel_x = L.max_vel_x;
	D.min_vel_x = L.min_vel_x;
	D.max_vel_y = L.max_vel_y;
	D.min_vel_y = L.min_vel_y;
	D.max_vel_theta = L.max_vel_theta;
	D.min_vel_theta = L.min_vel_theta;
	D.max_vel_trans = L.max_vel_trans;
	D.min_vel_trans = L.min_vel_trans;
	D.acc_x = L.acc_lim_x;
	D.acc_y = L.acc_lim_y;
	D.acc_th = L.acc_lim_theta;
	D.acc_decel = std::hypot(L.acc_lim_x, L.acc_lim_y);
	D.rot_comp = L.twist_rotation_compensation;
	D.back_max = (L.min_vel_x < 0.0) ? std::fabs(L.min_vel_x) : 0.0;
	D.maintain_rate = L.maintain_vel_components_rate != 0;

	const HmpSfm& S = P.sfm;
	D.fov_method = S.fov_factor_method;
	D.filter_forces = S.filter_forces != 0;
	D.disable_interaction = S.disable_interaction_forces != 0;
	D.mass = S.mass;
	D.m_over_tau = S.mass * (1 / (double)(float)S.relaxation_time);
	D.k_int = S.internal_force_factor;
	D.k_stat = S.static_interaction_force_factor;
	D.k_dyn = S.dynamic_interaction_force_factor;
	D.min_force = S.min_force;
	D.max_force = S.max_force;
	// computeFactorFOV(angle, 2 * cfg.fov, gaussian): half angle cfg.fov, variance cfg.fov^2, PDF not normalised to 1
	D.fov_half_d = S.fov;
	D.fov_gauss_scale_d = 1.0 / (std::sqrt(S.fov * S.fov) * std::sqrt(2.0 * PI));
	D.fov_neg_inv_2var_d = -1.0 / (2.0 * S.fov * S.fov);
	D.fov_half = (float)D.fov_half_d;
	D.fov_gauss_scale = (float)D.fov_gauss_scale_d;
	D.fov_neg_inv_2var = (float)D.fov_neg_inv_2var_d;
	const double base[9] = {S.speed_desired, S.an, S.bn, S.cn, S.ap, S.bp, S.cp, S.aw, S.bw};
	for (int i = 0; i < 9; ++i) D.base[i] = (float)base[i];

	const HmpFis& F = P.fis;
	D.fis_on = (!D.disable_interaction && !(F.force_factor <= 0.0)) ? 1 : 0;
	D.fis_fov_method = F.fov_factor_method;
	D.fis_force_factor_d = F.force_factor;
	D.fis_range_d = F.human_action_range;
	D.fis_fov_half_d = F.fov / 2.0;
	{
		double var = (F.fov / 2.0) * (F.fov / 2.0);
		D.fis_gauss_scale_d = 1.0 / (std::sqrt(var) * std::sqrt(2.0 * PI));
		D.fis_neg_inv_2var_d = -1.0 / (2.0 * var);
	}

	// amplifier lists
	amp_table.assign((size_t)HMP_NUM_AMPLIFIERS * HMP_MAX_AMP_VALUES, 0.0);
	long long total = 1;
	for (int a = 0; a < HMP_NUM_AMPLIFIERS; ++a) {
		int n = amplifier_samples(sampling->amp_min[a], sampling->amp_max[a], sampling->amp_granularity[a],
		                          &amp_table[(size_t)a * HMP_MAX_AMP_VALUES], HMP_MAX_AMP_VALUES);
		if (n <= 0) {
			set_err("amplifier axis %d yields more than %d values or is malformed", a, HMP_MAX_AMP_VALUES);
			return HMP_E_CAPACITY;
		}
		D.amp_n[a] = n;
		total *= n;
		if (total > (1ll << 30)) {
			set_err("sampling grid has more than 2^30 candidates");
			return HMP_E_CAPACITY;
		}
	}
	D.n_grid = (int)total;
	D.n_social = (int)total + n_extra;
	D.n_equi = 0;
	D.n_candidates = D.n_social;

	D.size_x = ctx->size_x;
	D.size_y = ctx->size_y;
	D.origin_x = ctx->origin_x;
	D.origin_y = ctx->origin_y;
	D.resolution = ctx->resolution;
	D.inv_resolution = 1.0 / ctx->resolution;

	const HmpCosts& C = P.costs;
	for (int k = 0; k < HMP_NUM_COSTS; ++k) D.scale[k] = C.scale[k];
	D.n_footprint = (int)ctx->footprint.size() / 2;
	for (int i = 0; i < D.n_footprint; ++i) {
		D.footprint_x[i] = ctx->footprint[2 * i];
		D.footprint_y[i] = ctx->footprint[2 * i + 1];
	}
	// separation kernel, obstacle_separation_cost_function.cpp:183-219
	D.n_kernel_pts = 1;
	D.kernel_dx[0] = D.kernel_dy[0] = 0.0;
	if (!(std::fabs(C.occdist_separation) < 1e-03)) {
		static const double cross[4] = {0.0, M_PI_2, M_PI, -M_PI_2};
		static const double rect[8] = {0.0, M_PI_4, M_PI_2, 3.0 * M_PI_4, M_PI, -3.0 * M_PI_4, -M_PI_2, -M_PI_4};
		const double* ang = nullptr;
		int n = 0;
		if (C.occdist_separation_kernel == 0) {
			ang = cross;
			n = 4;
		} else if (C.occdist_separation_kernel == 1) {
			ang = rect;
			n = 8;
		}
		for (int i = 0; i < n; ++i) {
			D.kernel_dx[1 + i] = C.occdist_separation * std::cos(ang[i]);
			D.kernel_dy[1 + i] = C.occdist_separation * std::sin(ang[i]);
		}
		D.n_kernel_pts = 1 + n;
	}
	D.occdist_sum = C.occdist_sum_scores != 0;
	for (int g = 0; g < HMP_NUM_MAPGRIDS; ++g) {
		D.mg_stop_on_failure[g] = C.stop_on_failure[g] != 0;
		D.mg_kernel[g] = C.neighbour_kernel_size[g];
		D.mg_xshift[g] = C.xshift[g];
		D.mg_yshift[g] = C.yshift[g];
	}
	D.unsat_max_trans = (float)C.unsat_max_trans_vel;
	D.unsat_max_x = (float)C.unsat_max_vel_x;
	D.unsat_max_y = (float)C.unsat_max_vel_y;
	D.backward_penalty = (float)C.backward_penalty;
	D.ttc_collision_distance = (float)C.ttc_collision_distance;
	{
		double var = (C.hd_fov_person / 2.0) * (C.hd_fov_person / 2.0);
		D.hd_neg_inv_2var_fov = (float)(-1.0 / (2.0 * var));
	}
	D.hd_dmin = (float)(C.hd_robot_circumradius + C.hd_person_model_radius);
	D.hd_inv_max_speed = (float)(1.0 / C.hd_max_speed);
	D.ps_min_dist = (float)C.ps_min_dist;
	D.ps_inv_max_speed = (float)(1.0 / C.ps_max_speed);
	D.unsat_whole = C.unsat_whole_horizon != 0;
	D.hd_whole = C.hd_whole_horizon != 0;
	D.psi_whole = C.psi_whole_horizon != 0;
	D.fsi_whole = C.fsi_whole_horizon != 0;
	D.ps_whole = C.ps_whole_horizon != 0;
	return HMP_OK;
}

size_t scene_blob_bytes(const HmpWorld& w) {
	// worst case: every obstacle appears in both the dynamic and the static array (App. A #5)
	size_t b = sizeof(DevScene);
	b += (size_t)w.n_obstacles * sizeof(DevStatic);
	b += (size_t)w.n_obstacles * sizeof(DevDynamic);
	b += (size_t)w.n_people * sizeof(DevPerson);
	b += (size_t)w.n_groups * sizeof(DevGroup);
	return (b + 15) / 16 * 16;
}

// Packs one World (+ people / groups) into `out` (scene_blob_bytes(w) bytes, zero-filled by the caller).
void pack_scene(const HmpContext* ctx, const HmpWorld& w, const double* hv_prev, double dt, unsigned char* out, int n_equi = 0) {
	const HmpParams& P = ctx->params;
	DevScene H;
	std::memset(&H, 0, sizeof(H));
	H.x0 = w.robot_x;
	H.y0 = w.robot_y;
	H.yaw0 = wrap(w.robot_yaw);
	// computeVelocityGlobal(vel_, pose_), humap_planner.cpp:366-369
	double cy = std::cos(H.yaw0), sy = std::sin(H.yaw0);
	H.u0x_d = w.vel_x * cy - w.vel_y * sy;
	H.u0y_d = w.vel_x * sy + w.vel_y * cy;
	H.u0w_d = w.vel_th;
	H.u0x = (float)H.u0x_d;
	H.u0y = (float)H.u0y_d;
	H.u0w = (float)H.u0w_d;
	H.glx_d = w.goal_local_x - w.robot_x;
	H.gly_d = w.goal_local_y - w.robot_y;
	H.gx_d = w.goal_x - w.robot_x;
	H.gy_d = w.goal_y - w.robot_y;
	H.vlx = (float)w.vel_x;
	H.vly = (float)w.vel_y;
	H.vlw = (float)w.vel_th;
	H.glx = (float)(w.goal_local_x - w.robot_x);
	H.gly = (float)(w.goal_local_y - w.robot_y);
	H.gx = (float)(w.goal_x - w.robot_x);
	H.gy = (float)(w.goal_y - w.robot_y);
	for (int g = 0; g < HMP_NUM_MAPGRIDS; ++g) H.hv_prev[g] = hv_prev ? hv_prev[g] : 0.0;
	H.equi_px = (float)w.robot_x;   // Eigen::Vector3f pos_ of the equisampled generator (humap_planner.cpp:1317-1361)
	H.equi_py = (float)w.robot_y;
	H.equi_pth = (float)w.robot_yaw;
	H.n_equi = n_equi;

	std::vector<DevStatic> st_always, st_later;
	std::vector<DevDynamic> dy_always, dy_first;
	for (int i = 0; i < w.n_obstacles; ++i) {
		const HmpObstacle& o = w.obstacles[i];
		double len3 = std::sqrt(o.vx * o.vx + o.vy * o.vy + o.vth * o.vth);  // Vector::calculateLength is 3-D (App. A #4)
		bool moving = len3 > 0.035;                                          // world.h:110
		bool dyn0 = (o.force_dynamic != 0) || moving;                        // world.cpp:49
		double d0x = o.obj_x - o.robot_x, d0y = o.obj_y - o.robot_y;
		if (!dyn0) {
			st_always.push_back({d0x, d0y});
			continue;
		}
		DevDynamic d;
		d.d0x = d0x;
		d.d0y = d0y;
		d.vx = o.vx;
		d.vy = o.vy;
		d.psi0 = wrap(o.robot_yaw);
		d.dir_beta = wrap(std::atan2(o.vy, o.vx));
		d.speed = std::hypot(o.vx, o.vy);
		d._pad = 0.0;
		if (moving) {
			dy_always.push_back(d);
		} else {
			// dynamic at step 0 only: advanced once by v dt in the first World::predict, then static (world.cpp:101-110)
			dy_first.push_back(d);
			st_later.push_back({d0x + o.vx * dt, d0y + o.vy * dt});
		}
	}
	H.n_static0 = (int)st_always.size();
	H.n_static = (int)(st_always.size() + st_later.size());
	H.n_dynamic_later = (int)dy_always.size();
	H.n_dynamic = (int)(dy_always.size() + dy_first.size());
	H.n_people = w.n_people;
	H.n_groups = w.n_groups;
	uint32_t off = sizeof(DevScene);
	H.off_static = off;
	off += (uint32_t)((size_t)H.n_static * sizeof(DevStatic));
	H.off_dynamic = off;
	off += (uint32_t)((size_t)H.n_dynamic * sizeof(DevDynamic));
	H.off_people = off;
	off += (uint32_t)((size_t)H.n_people * sizeof(DevPerson));
	H.off_groups = off;
	off += (uint32_t)((size_t)H.n_groups * sizeof(DevGroup));
	H.blob_bytes = (off + 15) / 16 * 16;

	std::memcpy(out, &H, sizeof(H));
	DevStatic* ps = reinterpret_cast<DevStatic*>(out + H.off_static);
	for (size_t i = 0; i < st_always.size(); ++i) ps[i] = st_always[i];
	for (size_t i = 0; i < st_later.size(); ++i) ps[st_always.size() + i] = st_later[i];
	DevDynamic* pd = reinterpret_cast<DevDynamic*>(out + H.off_dynamic);
	for (size_t i = 0; i < dy_always.size(); ++i) pd[i] = dy_always[i];
	for (size_t i = 0; i < dy_first.size(); ++i) pd[dy_always.size() + i] = dy_first[i];

	DevPerson* pp = reinterpret_cast<DevPerson*>(out + H.off_people);
	for (int i = 0; i < w.n_people; ++i) {
		const HmpPerson& p = w.people[i];
		DevPerson d;
		d.x = (float)(p.x - w.robot_x);
		d.y = (float)(p.y - w.robot_y);
		double yaw = wrap(p.yaw);
		d.yaw = (float)yaw;
		d.vth = (float)p.vth;
		d.vx = (float)p.vx;
		d.vy = (float)p.vy;
		d.cos0 = (float)std::cos(yaw);
		d.sin0 = (float)std::sin(yaw);
		d.cxx = (float)p.cov_xx;
		d.cxy = (float)p.cov_xy;
		d.cyx = (float)p.cov_yx;
		d.cyy = (float)p.cov_yy;
		// personal_space_intrusion_cost_function.cpp:55-58
		double vel_lin = std::hypot(p.vx, p.vy);
		double var_front = std::max(2.0 * vel_lin, 0.5);
		d.var_front = (float)var_front;
		d.var_side = (float)((2.0 / 3.0) * var_front);
		d.var_rear = (float)((1.0 / 2.0) * var_front);
		d.radius_eff = (float)(P.costs.hd_person_model_radius + std::sqrt(0.5 * (p.cov_xx + p.cov_yy)));
		pp[i] = d;
	}
	DevGroup* pg = reinterpret_cast<DevGroup*>(out + H.off_groups);
	for (int i = 0; i < w.n_groups; ++i) {
		const HmpGroup& g = w.groups[i];
		// fformation_space_intrusion_cost_function.cpp:60-61: variance = (span / 2 / 2)^2 along the group's axes
		double var_x = std::pow((g.span_x / 2.0) / 2.0, 2), var_y = std::pow((g.span_y / 2.0) / 2.0, 2);
		double yaw = wrap(g.yaw);
		double c = std::cos(yaw), s = std::sin(yaw);
		double a = var_x * c * c + var_y * s * s + g.cov_xx;
		double b = (var_x - var_y) * c * s + g.cov_xy;
		double cc = var_x * s * s + var_y * c * c + g.cov_yy;
		double det = a * cc - b * b;
		DevGroup d;
		std::memset(&d, 0, sizeof(d));
		d.x = (float)(g.x - w.robot_x);
		d.y = (float)(g.y - w.robot_y);
		d.ia = (float)(cc / det);
		d.ib = (float)(-b / det);
		d.ic = (float)(a / det);
		pg[i] = d;
	}
}

// Velocity samples of the equisampled generator for one cycle: src/humap_planner.cpp:1317-1361 (min_vel_x rule) +
// base_local_planner::SimpleTrajectoryGenerator::initialise / VelocityIterator [RECALLED]. Eigen::Vector3f state: float stores.
void velocity_iterator(double vmin, double vmax, int num_samples, std::vector<double>& out) {
	out.clear();
	if (vmin == vmax) {
		out.push_back(vmin);
		return;
	}
	num_samples = std::max(2, num_samples);
	const double step = (vmax - vmin) / double(std::max(1, num_samples - 1));
	double next = vmin;
	for (int j = 0; j < num_samples - 1; ++j) {
		const double current = next;
		next += step;
		out.push_back(current);
		if (current < 0 && next > 0) out.push_back(0.0);
	}
	out.push_back(vmax);
}

void equisampled_samples(const HmpParams& P, const HmpWorld& w, const HmpEquisampled& eq, DevParams& D, std::vector<double>& samples) {
	samples.clear();
	const HmpLimits& L = P.limits;
	const double sim_time = P.general.sim_time, sim_period = P.general.sim_period;
	const double from_min = std::max(std::max(eq.min_vel_x, L.min_vel_x), std::max(eq.min_vel_x, w.vel_x - L.acc_lim_x * sim_period));
	const double min_vel_x = std::min(from_min, L.max_vel_x);
	double max_vel_x = L.max_vel_x, max_vel_y = L.max_vel_y;
	const double min_vel_y = L.min_vel_y, max_vel_th = L.max_vel_theta, min_vel_th = -L.max_vel_theta;
	const float pos[3] = {(float)w.robot_x, (float)w.robot_y, (float)w.robot_yaw};
	const float vel[3] = {(float)w.vel_x, (float)w.vel_y, (float)w.vel_th};
	const float acc[3] = {(float)L.acc_lim_x, (float)L.acc_lim_y, (float)L.acc_lim_theta};
	for (int k = 0; k < 3; ++k) {
		D.equi_pos[k] = pos[k];
		D.equi_vel[k] = vel[k];
		D.equi_acc[k] = acc[k];
	}
	D.equi_continued = eq.continued_acceleration ? 1 : 0;
	const float vs[3] = {(float)eq.vx_samples, (float)eq.vy_samples, (float)eq.vth_samples};
	if (!(vs[0] * vs[1] * vs[2] > 0)) return;
	const double window = eq.continued_acceleration ? sim_time : sim_period;   // use_dwa = !continued_acceleration
	if (eq.continued_acceleration) {
		const float gx = (float)w.goal_x, gy = (float)w.goal_y;
		const double dist = std::hypot(gx - pos[0], gy - pos[1]);
		max_vel_x = std::max(std::min(max_vel_x, dist / sim_time), min_vel_x);
		max_vel_y = std::max(std::min(max_vel_y, dist / sim_time), min_vel_y);
	}
	const float hi[3] = {(float)std::min(max_vel_x, vel[0] + acc[0] * window), (float)std::min(max_vel_y, vel[1] + acc[1] * window),
	                     (float)std::min(max_vel_th, vel[2] + acc[2] * window)};
	const float lo[3] = {(float)std::max(min_vel_x, vel[0] - acc[0] * window), (float)std::max(min_vel_y, vel[1] - acc[1] * window),
	                     (float)std::max(min_vel_th, vel[2] - acc[2] * window)};
	std::vector<double> xs, ys, ts;
	velocity_iterator(lo[0], hi[0], (int)vs[0], xs);
	velocity_iterator(lo[1], hi[1], (int)vs[1], ys);
	velocity_iterator(lo[2], hi[2], (int)vs[2], ts);
	for (double vx : xs)
		for (double vy : ys)
			for (double vt : ts) {
				samples.push_back((double)(float)vx);
				samples.push_back((double)(float)vy);
				samples.push_back((double)(float)vt);
			}
}

struct CtrlLayout {  // d_ctrl: counters [n][4] u32 | hv_out [n][4] u32 | best_out [n][2] f64 | best of the equisampled sweep [n][2] f64
	                   // | work ticket of a refinement that runs beside the sweep [n][4] u32
	size_t off_counters, off_hv, off_best, off_best2, off_counters2, total;
};
CtrlLayout ctrl_layout(int n_scenes) {
	CtrlLayout c;
	c.off_counters = 0;
	c.off_hv = (size_t)n_scenes * 4 * sizeof(unsigned int);
	c.off_best = c.off_hv + (size_t)n_scenes * 4 * sizeof(unsigned int);
	c.off_best = (c.off_best + 15) / 16 * 16;
	c.off_best2 = c.off_best + (size_t)n_scenes * 2 * sizeof(double);
	c.off_counters2 = c.off_best2 + (size_t)n_scenes * 2 * sizeof(double);
	c.total = c.off_counters2 + (size_t)n_scenes * 4 * sizeof(unsigned int);
	return c;
}

int check_ready(const HmpContext* ctx) {
	if (!ctx) {
		set_err("null context");
		return HMP_E_INVALID;
	}
	if (!ctx->have_params) {
		set_err("hmp_set_params has not been called");
		return HMP_E_NOT_READY;
	}
	if (!ctx->have_costmap) {
		set_err("hmp_set_costmap has not been called");
		return HMP_E_NOT_READY;
	}
	return HMP_OK;
}

// Common part of hmp_plan / hmp_plan_batch: scenes, costmaps and mapgrids are already on the device.
struct PlanLaunch {
	int n_scenes;
	uint32_t scene_stride;
	int n_extra;
	int T;
	const HmpSceneCosts* scene_costs = nullptr;   // n_scenes entries (hmp_set_scene_costs), or null: every scene uses D's
};

// Whether critic k is evaluated in any scene of a launch: host decisions that serve all scenes at once (inputs the critic
// needs, shared-memory reservations) follow the union over the scenes; the kernels skip the critic per scene.
bool scale_on(const double* shared_scale, const HmpSceneCosts* scene_costs, int n_scenes, int k) {
	if (!scene_costs) return shared_scale[k] != 0.0;
	for (int s = 0; s < n_scenes; ++s)
		if (scene_costs[s].scale[k] != 0.0) return true;
	return false;
}

int launch_main(HmpContext* ctx, const DevParams& D, const PlanLaunch& pl, int* blocks_x_out, size_t* smem_out,
                int* costmap_in_smem_out, int* sweep_mode_out = nullptr, size_t* smem_sweep_out = nullptr) {
	const int C = D.n_social;
	size_t cm_bytes = (size_t)ctx->costmap_stride;
	int in_smem = 1;
	size_t smem = hmp_dev_smem_bytes(pl.scene_stride, (uint32_t)cm_bytes, 1);
	if (smem > ctx->max_smem_optin || cm_bytes > (1u << 19)) {
		in_smem = 0;
		smem = hmp_dev_smem_bytes(pl.scene_stride, (uint32_t)cm_bytes, 0);
		if (smem > ctx->max_smem_optin) {
			set_err("scene does not fit shared memory (%zu bytes needed, %zu available)", smem, ctx->max_smem_optin);
			return HMP_E_CAPACITY;
		}
	}
	// Layout of the FP32 sweep. One warp per candidate (plan_kernel) has the shortest latency for a few thousand
	// candidates; one thread per candidate (sweep_tpc_kernel) issues the per-step scalar section once per 32 candidates
	// and wins as soon as the launch holds enough candidates to give every SM sub-partition a warp.
	// The exact-parity sweep (precision mode 1) has the same two layouts; its thread-per-candidate instance is compiled for one
	// block per SM (225 registers, no spills).
	int tpc_threads = 0;
	const bool f64 = ctx->precise == 1;
	if (sweep_mode_out) {
		const long long total = (long long)C * pl.n_scenes;
		const bool want = ctx->sweep_layout == 2 || (ctx->sweep_layout == 0 && total >= 16384);
		if (want) {
			tpc_threads = hmp_dev_tpc_max_threads();
			// few candidates: smaller blocks so that every SM gets one
			while (tpc_threads > 64 && ((long long)C + tpc_threads - 1) / tpc_threads * pl.n_scenes * 10 < (long long)ctx->sm_count * 9)
				tpc_threads = (tpc_threads > 128) ? 128 : 64;
		}
	}
	if (tpc_threads && f64) tpc_threads = std::min(tpc_threads, hmp_dev_tpc64_max_threads());   // launch bound of the FP64 instance
	size_t smem_sweep = smem;
	ctx->tpc_defer = 0;
	if (tpc_threads) {
		smem_sweep = smem + hmp_dev_tpc_extra_smem(pl.scene_stride);
		if (smem_sweep > ctx->max_smem_optin) {
			tpc_threads = 0;
			smem_sweep = smem;
		}
	}
	// few warps per SM sub-partition anyway (<= 2): the register-rich instance of the thread-per-candidate sweep
	int tpc_rich = 0;
	if (tpc_threads && !f64) {
		const long long warps = (((long long)C + tpc_threads - 1) / tpc_threads) * pl.n_scenes * (tpc_threads / 32);
		tpc_rich = (warps <= (long long)ctx->sm_count * 8) ? 1 : 0;
	}
	if (tpc_threads && ctx->prune_obstacle && scale_on(D.scale, pl.scene_costs, pl.n_scenes, HMP_COST_OBSTACLE) && D.n_footprint > 0 && !D.occdist_sum &&
	    !getenv("HMP_NO_DEFER")) {
		// deferred obstacle critic: one byte per pose and thread behind the packed static objects; taken when it costs no
		// resident block (the pose scratch in global memory is one slot per resident block, run_cycle)
		const size_t with = ((smem_sweep + 15) & ~(size_t)15) + (size_t)pl.T * tpc_threads;
		int b0 = 0, b1 = 0;
		auto occ = [&](size_t bytes, int* b) {
			return f64 ? hmp_dev_occupancy_tpc64(bytes, tpc_threads, b) : hmp_dev_occupancy_tpc(bytes, tpc_threads, tpc_rich, b);
		};
		if (with <= ctx->max_smem_optin && occ(smem_sweep, &b0) == cudaSuccess && occ(with, &b1) == cudaSuccess && b1 >= b0 && b1 >= 1) {
			smem_sweep = with;
			ctx->tpc_defer = 1;
		}
	}
	int bps = 0;
	if (tpc_threads && f64) CU(hmp_dev_occupancy_tpc64(smem_sweep, tpc_threads, &bps));
	else if (tpc_threads) CU(hmp_dev_occupancy_tpc(smem_sweep, tpc_threads, tpc_rich, &bps));
	if (tpc_threads) ctx->tpc_bps = bps;
	else CU(hmp_dev_occupancy(smem, ctx->precise == 1, &bps));
	if (bps < 1) {
		set_err("kernel cannot be resident with %zu bytes of shared memory", smem);
		return HMP_E_CUDA;
	}
	// persistent blocks: fill the GPU once; with many scenes give each scene fewer blocks
	long long resident = (long long)ctx->sm_count * bps;
	const long long per_block = tpc_threads ? tpc_threads : HMP_WARPS_PER_BLOCK;   // candidates a block takes per ticket
	long long need = ((long long)C + per_block - 1) / per_block;
	// blocks per scene: one scene fills the GPU once; with several scenes per launch pick the split p that minimises the
	// number of block waves times the work per block, ceil(n_scenes * p / resident) / p (ties: the finer split)
	long long per_scene = std::max<long long>(1, std::min<long long>(need, resident));
	if (pl.n_scenes > 1) {
		double best_t = 1e300;
		for (long long p = 1; p <= std::min<long long>(need, 8); ++p) {
			const double t = (double)((pl.n_scenes * p + resident - 1) / resident) / (double)p;
			if (t <= best_t * (1.0 + 1e-12)) {
				best_t = t;
				per_scene = p;
			}
		}
	}
	if (getenv("HMP_DEBUG")) fprintf(stderr, "[hmp] smem %zu B/block, %d blocks/SM resident, %lld blocks per scene, %d scenes, sweep mode %d\n", smem, bps, per_scene, pl.n_scenes, tpc_threads);
	if (sweep_mode_out) *sweep_mode_out = tpc_threads ? (tpc_threads | (tpc_rich ? 1024 : 0)) : 0;
	if (smem_sweep_out) *smem_sweep_out = smem_sweep;
	*blocks_x_out = (int)per_scene;
	*smem_out = smem;
	*costmap_in_smem_out = in_smem;
	return HMP_OK;
}

}  // namespace

// ====================================================================================================
extern "C" {

const char* hmp_last_error(void) { return g_err; }
int hmp_abi_version(void) { return HMP_ABI_VERSION; }

HmpContext* hmp_create(int device_id) {
	int n = 0;
	cudaError_t e = cudaGetDeviceCount(&n);
	if (e != cudaSuccess || n <= 0) {
		set_err("no usable CUDA device (%s); this library has no CPU fallback", e != cudaSuccess ? cudaGetErrorString(e) : "count 0");
		return nullptr;
	}
	if (device_id < 0 || device_id >= n) {
		set_err("device %d out of range (%d devices)", device_id, n);
		return nullptr;
	}
	if ((e = cudaSetDevice(device_id)) != cudaSuccess) {
		set_err("cudaSetDevice(%d): %s", device_id, cudaGetErrorString(e));
		return nullptr;
	}
	cudaDeviceProp prop;
	if ((e = cudaGetDeviceProperties(&prop, device_id)) != cudaSuccess) {
		set_err("cudaGetDeviceProperties: %s", cudaGetErrorString(e));
		return nullptr;
	}
	if (prop.major != 10) {
		set_err("device %d is sm_%d%d; this library carries sm_100a code only", device_id, prop.major, prop.minor);
		return nullptr;
	}
	HmpContext* ctx = new (std::nothrow) HmpContext();
	if (!ctx) {
		set_err("out of memory");
		return nullptr;
	}
	ctx->device = device_id;
	ctx->prune_obstacle = getenv("HMP_NO_PRUNE") ? 0 : 1;
	if (const char* e = getenv("HMP_ESCALATE")) ctx->escalate_min = std::max(0, atoi(e));
	if (const char* e = getenv("HMP_SWEEP_LAYOUT")) ctx->sweep_layout = std::max(0, std::min(2, atoi(e)));
	ctx->sm_count = prop.multiProcessorCount;
	ctx->max_smem_optin = prop.sharedMemPerBlockOptin - 1024;  // static __shared__ of the kernel comes out of the same budget
	if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess ||
	    cudaStreamCreateWithFlags(&ctx->stream2, cudaStreamNonBlocking) != cudaSuccess ||
	    cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
	    cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming) != cudaSuccess ||
	    cudaEventCreate(&ctx->ev0) != cudaSuccess || cudaEventCreate(&ctx->ev1) != cudaSuccess ||
	    cudaEventCreate(&ctx->evm) != cudaSuccess || cudaEventCreateWithFlags(&ctx->seeds_event[0], cudaEventDisableTiming) != cudaSuccess ||
	    cudaEventCreateWithFlags(&ctx->seeds_event[1], cudaEventDisableTiming) != cudaSuccess ||
	    cudaEventCreateWithFlags(&ctx->seeds_event[2], cudaEventDisableTiming) != cudaSuccess ||
	    cudaEventCreateWithFlags(&ctx->seeds_event[3], cudaEventDisableTiming) != cudaSuccess ||
	    cudaStreamCreateWithFlags(&ctx->wf_stream[0], cudaStreamNonBlocking) != cudaSuccess ||
	    cudaStreamCreateWithFlags(&ctx->wf_stream[1], cudaStreamNonBlocking) != cudaSuccess ||
	    cudaStreamCreateWithFlags(&ctx->wf_stream[2], cudaStreamNonBlocking) != cudaSuccess ||
	    cudaStreamCreateWithFlags(&ctx->wf_stream[3], cudaStreamNonBlocking) != cudaSuccess ||
	    cudaEventCreateWithFlags(&ctx->wf_done[0], cudaEventDisableTiming) != cudaSuccess ||
	    cudaEventCreateWithFlags(&ctx->wf_done[1], cudaEventDisableTiming) != cudaSuccess ||
	    cudaEventCreateWithFlags(&ctx->wf_done[2], cudaEventDisableTiming) != cudaSuccess ||
	    cudaEventCreateWithFlags(&ctx->wf_done[3], cudaEventDisableTiming) != cudaSuccess ||
	    hmp_dev_configure(ctx->max_smem_optin) != cudaSuccess) {
		set_err("context setup failed: %s", cudaGetErrorString(cudaGetLastError()));
		delete ctx;
		return nullptr;
	}
	return ctx;
}

void hmp_destroy(HmpContext* ctx) {
	if (!ctx) return;
	cudaSetDevice(ctx->device);
	if (ctx->stream) cudaStreamSynchronize(ctx->stream);
	for (int g = 0; g < HMP_NUM_MAPGRIDS; ++g) {
		ctx->d_seeds[g].release();
		ctx->h_seeds[g].release();
		ctx->h_grid[g].release();
		if (ctx->seeds_event[g]) cudaEventDestroy(ctx->seeds_event[g]);
		if (ctx->wf_stream[g]) {
			cudaStreamSynchronize(ctx->wf_stream[g]);
			cudaStreamDestroy(ctx->wf_stream[g]);
		}
		if (ctx->wf_done[g]) cudaEventDestroy(ctx->wf_done[g]);
	}
	DevBuf* bufs[] = {&ctx->d_params, &ctx->d_amp, &ctx->d_extra, &ctx->d_scenes, &ctx->d_costmaps, &ctx->d_mapgrids,
	                  &ctx->d_totals, &ctx->d_block_best, &ctx->d_ctrl, &ctx->d_detail, &ctx->d_dbg, &ctx->d_refine, &ctx->d_dilated, &ctx->d_equi, &ctx->d_env, &ctx->d_mask, &ctx->d_hvrec, &ctx->d_posescr, &ctx->d_poseslots};
	for (DevBuf* b : bufs) b->release();
	ctx->h_stage.release();
	ctx->h_params.release();
	for (int b = 0; b < 2; ++b) {
		ctx->h_grid_stage[b].release();
		if (ctx->grid_stage_ev[b]) cudaEventDestroy(ctx->grid_stage_ev[b]);
	}
	ctx->h_out.release();
	ctx->h_small.release();
	if (ctx->ev0) cudaEventDestroy(ctx->ev0);
	if (ctx->ev1) cudaEventDestroy(ctx->ev1);
	if (ctx->evm) cudaEventDestroy(ctx->evm);
	if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
	if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
	if (ctx->stream2) {
		cudaStreamSynchronize(ctx->stream2);
		cudaStreamDestroy(ctx->stream2);
	}
	if (ctx->stream) cudaStreamDestroy(ctx->stream);
	delete ctx;
}

int hmp_set_params(HmpContext* ctx, const HmpParams* params) {
	if (!ctx || !params) {
		set_err("null argument");
		return HMP_E_INVALID;
	}
	if (!(params->general.sim_time > 0.0) || !(params->general.sim_granularity > 0.0)) {
		set_err("sim_time and sim_granularity must be positive");
		return HMP_E_INVALID;
	}
	if (!ctx->have_params || params->costs.occdist_separation != ctx->params.costs.occdist_separation ||
	    params->costs.occdist_separation_kernel != ctx->params.costs.occdist_separation_kernel)
		ctx->dilated_dirty = true;
	ctx->params = *params;
	ctx->have_params = true;
	ctx->last_valid = false;
	return HMP_OK;
}

// Device wave fronts (hmp_compute_mapgrid[_batch]) run on side streams and finish on the device whatever their frontiers hold:
// the plan stream waits for their events, the host does not. Work queued on ctx->stream after the join sees their grids.
static int join_wavefronts(HmpContext* ctx) {
	for (int g = 0; g < HMP_NUM_MAPGRIDS; ++g) {
		if (!ctx->wavefront_pending[g]) continue;
		CU(cudaStreamWaitEvent(ctx->stream, ctx->wf_done[g], 0));
		ctx->wavefront_pending[g] = false;
	}
	return HMP_OK;
}

int hmp_set_costmap(HmpContext* ctx, const uint8_t* cells, int32_t size_x, int32_t size_y, double origin_x, double origin_y,
                    double resolution) {
	if (!ctx || !cells || size_x <= 0 || size_y <= 0 || !(resolution > 0.0)) {
		set_err("bad costmap arguments");
		return HMP_E_INVALID;
	}
	if ((long long)size_x * size_y >= (1ll << 24)) {
		set_err("costmap has 2^24 cells or more: MapGrid distances would not be exact in FP32");
		return HMP_E_CAPACITY;
	}
	CU(cudaSetDevice(ctx->device));
	for (int g = 0; g < HMP_NUM_MAPGRIDS; ++g)   // a wave front still reading the old cells must finish first
		if (ctx->wavefront_pending[g]) CU(cudaStreamSynchronize(ctx->wf_stream[g]));
	if (size_x != ctx->size_x || size_y != ctx->size_y) {
		for (bool& b : ctx->have_grid) b = false;
	}
	size_t cells_n = (size_t)size_x * size_y;
	uint32_t stride = (uint32_t)((cells_n + 127) / 128 * 128);
	int rc = ctx->d_costmaps.ensure(stride);
	if (rc) return rc;
	rc = ctx->d_mapgrids.ensure(cells_n * HMP_NUM_MAPGRIDS * sizeof(float));
	if (rc) return rc;
	rc = ctx->h_stage.ensure(std::max<size_t>(stride, cells_n * sizeof(float)));
	if (rc) return rc;
	CU(cudaStreamSynchronize(ctx->stream));
	ctx->h_cells.assign(cells, cells + cells_n);
	std::memcpy(ctx->h_stage.p, cells, cells_n);
	std::memset((unsigned char*)ctx->h_stage.p + cells_n, 0, stride - cells_n);
	CU(cudaMemcpyAsync(ctx->d_costmaps.p, ctx->h_stage.p, stride, cudaMemcpyHostToDevice, ctx->stream));
	CU(cudaStreamSynchronize(ctx->stream));
	ctx->costmap_stride = stride;
	ctx->size_x = size_x;
	ctx->size_y = size_y;
	ctx->origin_x = origin_x;
	ctx->origin_y = origin_y;
	ctx->resolution = resolution;
	ctx->have_costmap = true;
	ctx->costmap_scenes = 1;
	ctx->batch_grid_scenes = 0;
	ctx->last_valid = false;
	ctx->dilated_dirty = true;
	return HMP_OK;
}

int hmp_set_mapgrid(HmpContext* ctx, int32_t grid, const double* target_dist, double highest_valid_cost_prev) {
	if (!ctx || !target_dist || grid < 0 || grid >= HMP_NUM_MAPGRIDS) {
		set_err("bad mapgrid arguments");
		return HMP_E_INVALID;
	}
	if (!ctx->have_costmap) {
		set_err("hmp_set_costmap must precede hmp_set_mapgrid");
		return HMP_E_NOT_READY;
	}
	CU(cudaSetDevice(ctx->device));
	int rc = join_wavefronts(ctx);   // the upload lands after any device wave front still writing this slot
	if (rc) return rc;
	size_t n = (size_t)ctx->size_x * ctx->size_y;
	// one pinned staging buffer per slot: the four uploads of a cycle queue on the stream without a host synchronisation
	// (the previous cycle's plan has synchronised, so the buffer is free); the conversion loop is branch-free so that the
	// host compiler vectorises it (it used to be a third of the e2e overhead of a cycle)
	if (n * sizeof(float) > ctx->h_grid[grid].cap) CU(cudaStreamSynchronize(ctx->stream));
	rc = ctx->h_grid[grid].ensure(n * sizeof(float));
	if (rc) return rc;
	float* f = (float*)ctx->h_grid[grid].p;
	const double limit = (double)n + 1.0;
	int bad = 0;
	for (size_t i = 0; i < n; ++i) {
		const double v = target_dist[i];
		const int iv = (int)v;   // NaN / out-of-range convert to INT_MIN on x86-64 and fail the round trip below
		bad |= ((double)iv != v) | (iv < 0) | (v > limit);
		f[i] = (float)iv;
	}
	if (bad) {
		for (size_t i = 0; i < n; ++i) {
			const double v = target_dist[i];
			if (!(v >= 0.0) || v > limit || v != std::floor(v)) {
				set_err("target_dist[%zu] = %g is not a cell count in [0, size_x*size_y+1]", i, v);
				return HMP_E_INVALID;
			}
		}
	}
	CU(cudaMemcpyAsync((float*)ctx->d_mapgrids.p + (size_t)grid * n, f, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
	ctx->have_grid[grid] = true;
	ctx->batch_grid_scenes = 0;
	ctx->hv_prev[grid] = highest_valid_cost_prev;
	ctx->last_valid = false;
	return HMP_OK;
}

// Host part of base_local_planner::MapGrid::setTargetCells / setLocalGoal [RECALLED, SURVEY App. B]: densify the plan
// to the costmap resolution (adjustPlanResolution) and collect the seed cells of the wave front (every on-map,
// known plan cell up to the first gap; the local-goal variant seeds only the last one of them).
static void collect_seeds(const HmpContext* ctx, const uint8_t* cells, const double* plan_xy, int n_plan, int local_goal,
                          std::vector<int>& seeds) {
	seeds.clear();
	if (n_plan <= 0) return;
	const int sx = ctx->size_x, sy = ctx->size_y;
	auto world_to_map = [&](double wx, double wy, int& mx, int& my) {
		if (wx < ctx->origin_x || wy < ctx->origin_y) return false;
		mx = (int)((wx - ctx->origin_x) / ctx->resolution);
		my = (int)((wy - ctx->origin_y) / ctx->resolution);
		return mx < sx && my < sy;
	};
	std::vector<double> px, py;
	double last_x = plan_xy[0], last_y = plan_xy[1];
	px.push_back(last_x);
	py.push_back(last_y);
	const double min_sq = ctx->resolution * ctx->resolution;
	for (int i = 1; i < n_plan; ++i) {
		double lx = plan_xy[2 * i], ly = plan_xy[2 * i + 1];
		double sq = (lx - last_x) * (lx - last_x) + (ly - last_y) * (ly - last_y);
		if (sq > min_sq) {
			int steps = (int)std::ceil(std::sqrt(sq) / ctx->resolution);
			double dx = (lx - last_x) / steps, dy = (ly - last_y) / steps;
			for (int j = 1; j < steps; ++j) {
				px.push_back(last_x + j * dx);
				py.push_back(last_y + j * dy);
			}
		}
		px.push_back(lx);
		py.push_back(ly);
		last_x = lx;
		last_y = ly;
	}
	bool started = false;
	int goal = -1;
	for (size_t i = 0; i < px.size(); ++i) {
		int mx, my;
		if (world_to_map(px[i], py[i], mx, my) && cells[(size_t)my * sx + mx] != 255) {
			if (local_goal) goal = my * sx + mx;
			else seeds.push_back(my * sx + mx);
			started = true;
		} else if (started) {
			break;
		}
	}
	if (local_goal && goal >= 0) seeds.push_back(goal);
}

// Replaces MapGridCostFunction::setTargetPoses + prepare(): seeds on the host (collect_seeds), wave front on the device.
int hmp_compute_mapgrid(HmpContext* ctx, int32_t grid, const double* plan_xy, int32_t n_plan, int32_t local_goal,
                        double highest_valid_cost_prev) {
	if (!ctx || grid < 0 || grid >= HMP_NUM_MAPGRIDS || n_plan < 0 || (n_plan > 0 && !plan_xy)) {
		set_err("bad mapgrid arguments");
		return HMP_E_INVALID;
	}
	if (!ctx->have_costmap) {
		set_err("hmp_set_costmap must precede hmp_compute_mapgrid");
		return HMP_E_NOT_READY;
	}
	CU(cudaSetDevice(ctx->device));
	const int sx = ctx->size_x, sy = ctx->size_y;
	const size_t n = (size_t)sx * sy;
	if (hmp_dev_wavefront_smem(sx, sy) > ctx->max_smem_optin) {
		set_err("costmap too large for the on-device wave front (%zu bytes of shared memory needed, %zu available)",
		        hmp_dev_wavefront_smem(sx, sy), ctx->max_smem_optin);
		return HMP_E_CAPACITY;
	}
	// the costmap cells are needed for the NO_INFORMATION test of the seeds: keep a host copy from hmp_set_costmap
	if (ctx->h_cells.size() != n) {
		set_err("host copy of the costmap is missing");
		return HMP_E_NOT_READY;
	}
	std::vector<int> seeds;
	collect_seeds(ctx, ctx->h_cells.data(), plan_xy, n_plan, local_goal, seeds);
	// per-slot staging so that the four grids of a cycle queue on the stream without a host synchronisation, laid out like a
	// batch of one: [0] [1] seed offsets, [2..] seed cells
	const size_t need = (2 + std::max<size_t>(1, seeds.size())) * sizeof(int);
	int rc = ctx->d_seeds[grid].ensure(need);
	if (rc) return rc;
	// the previous upload from this staging buffer (slot 0: possibly a batch's) has been consumed
	if (ctx->seeds_event_valid[grid]) CU(cudaEventSynchronize(ctx->seeds_event[grid]));
	if (need > ctx->h_seeds[grid].cap) {
		CU(cudaStreamSynchronize(ctx->stream));
		if ((rc = ctx->h_seeds[grid].ensure(need * 2))) return rc;
	}
	int* hs = (int*)ctx->h_seeds[grid].p;
	hs[0] = 0;
	hs[1] = (int)seeds.size();
	if (!seeds.empty()) std::memcpy(hs + 2, seeds.data(), seeds.size() * sizeof(int));
	// each grid has its own stream: hmp_set_costmap has synchronised (the cells are on the device), the previous plan has
	// synchronised (nobody reads the MapGrid buffer), so the four single-block wave fronts of a cycle can overlap
	cudaStream_t st = ctx->wf_stream[grid];
	if (ctx->wf_after_batch[grid]) {   // a batch of wave fronts may still be writing this slot
		CU(cudaStreamWaitEvent(st, ctx->wf_done[grid], 0));
		ctx->wf_after_batch[grid] = false;
	}
	int* dsd = (int*)ctx->d_seeds[grid].p;
	CU(cudaMemcpyAsync(dsd, hs, need, cudaMemcpyHostToDevice, st));
	CU(cudaEventRecord(ctx->seeds_event[grid], st));
	ctx->seeds_event_valid[grid] = true;
	float* out = (float*)ctx->d_mapgrids.p + (size_t)grid * n;
	CU(hmp_dev_launch_wavefront((const uint8_t*)ctx->d_costmaps.p, ctx->costmap_stride, sx, sy, dsd + 2, dsd, out, 1, 1, st));
	CU(cudaEventRecord(ctx->wf_done[grid], st));
	ctx->launches++;
	ctx->wavefront_pending[grid] = true;
	ctx->have_grid[grid] = true;
	ctx->batch_grid_scenes = 0;
	ctx->hv_prev[grid] = highest_valid_cost_prev;
	ctx->last_valid = false;
	return HMP_OK;
}

int hmp_get_mapgrid(HmpContext* ctx, int32_t grid, double* target_dist_out) {
	if (!ctx || grid < 0 || grid >= HMP_NUM_MAPGRIDS || !target_dist_out || !ctx->have_grid[grid]) {
		set_err("bad arguments or grid not set");
		return HMP_E_INVALID;
	}
	CU(cudaSetDevice(ctx->device));
	{
		int rc = join_wavefronts(ctx);
		if (rc) return rc;
	}
	const size_t n = (size_t)ctx->size_x * ctx->size_y;
	std::vector<float> tmp(n);
	CU(cudaMemcpyAsync(tmp.data(), (const float*)ctx->d_mapgrids.p + (size_t)grid * n, n * sizeof(float), cudaMemcpyDeviceToHost,
	                   ctx->stream));
	CU(cudaStreamSynchronize(ctx->stream));
	for (size_t i = 0; i < n; ++i) target_dist_out[i] = tmp[i];
	return HMP_OK;
}

int hmp_set_footprint(HmpContext* ctx, const double* xy, int32_t n_points) {
	if (!ctx || n_points < 0 || (n_points > 0 && !xy)) {
		set_err("bad footprint arguments");
		return HMP_E_INVALID;
	}
	if (n_points > HMP_MAX_FOOTPRINT) {
		set_err("footprint has %d vertices, limit %d", n_points, HMP_MAX_FOOTPRINT);
		return HMP_E_CAPACITY;
	}
	ctx->footprint.assign(xy, xy + 2 * (size_t)n_points);
	ctx->have_footprint = true;
	ctx->last_valid = false;
	ctx->dilated_dirty = true;
	return HMP_OK;
}

static int validate_world(const HmpWorld* w) {
	if (!w || w->n_obstacles < 0 || w->n_people < 0 || w->n_groups < 0 || (w->n_obstacles > 0 && !w->obstacles) ||
	    (w->n_people > 0 && !w->people) || (w->n_groups > 0 && !w->groups)) {
		set_err("bad world arguments");
		return HMP_E_INVALID;
	}
	return HMP_OK;
}

// Runs the selection kernel + the winner's detail pass for scenes already resident on the device.
static int run_cycle(HmpContext* ctx, const DevParams& D, const std::vector<double>& amp_table, const HmpSample* extra,
                     int n_extra, const std::vector<double>& equi, const PlanLaunch& pl, HmpResult* results, double* poses_out,
                     int32_t poses_capacity) {
	const int C = D.n_candidates;
	const int T = D.T;
	const int NS = pl.n_scenes;
	int rc;
	// with a per-scene cost table: one DevParams per scene, D with that scene's scales / shifts (scene 0 first, so that launches
	// that read the first block, e.g. hmp_explain after a one-scene batch, see scene 0's values)
	const size_t params_bytes = sizeof(DevParams) * (pl.scene_costs ? (size_t)NS : 1);
	if ((rc = ctx->d_params.ensure(params_bytes))) return rc;
	if ((rc = ctx->d_amp.ensure(amp_table.size() * sizeof(double)))) return rc;
	if ((rc = ctx->d_extra.ensure(std::max<size_t>(1, (size_t)n_extra) * sizeof(HmpSample)))) return rc;
	if ((rc = ctx->d_equi.ensure(std::max<size_t>(1, equi.size()) * sizeof(double)))) return rc;
	if ((rc = ctx->d_totals.ensure((size_t)NS * C * sizeof(double)))) return rc;
	// per candidate and MapGrid critic: partial sum before the critic (f64) + largest valid cell value (f32), for the
	// early-exit semantics of highest_valid_cost_ (hv_early_exit_kernel)
	const size_t hv_items = (size_t)NS * C * HMP_NUM_MAPGRIDS;
	if ((rc = ctx->d_hvrec.ensure(hv_items * (sizeof(double) + sizeof(float))))) return rc;
	const CtrlLayout cl = ctrl_layout(NS);
	if ((rc = ctx->d_ctrl.ensure(cl.total))) return rc;
	// detail buffer per scene: costs[14] seeds[3] poses[T][3] totals[1] (f64) + nposes (i32, padded to 8)
	const size_t det_doubles = (size_t)HMP_NUM_COSTS + 3 + (size_t)T * 3 + 1;
	const size_t det_bytes = (det_doubles * sizeof(double) + 8) * NS;
	if ((rc = ctx->d_detail.ensure(det_bytes))) return rc;
	if ((rc = ctx->h_out.ensure(det_bytes + cl.total))) return rc;
	ctx->last_explain_n = 0;   // h_out is reused below

	int blocks_x = 0, in_smem = 0, sweep_mode = 0;
	size_t smem = 0, smem_sweep = 0;
	if ((rc = launch_main(ctx, D, pl, &blocks_x, &smem, &in_smem, &sweep_mode, &smem_sweep))) return rc;
	ctx->last_sweep_mode = sweep_mode;
	// per-block argmin scratch: the main sweep's blocks, then (its own region) the blocks of the equisampled sweep
	const int equi_blocks = D.n_equi > 0 ? (D.n_equi + HMP_WARPS_PER_BLOCK - 1) / HMP_WARPS_PER_BLOCK : 0;
	if ((rc = ctx->d_block_best.ensure((size_t)NS * ((size_t)blocks_x + equi_blocks) * 2 * sizeof(unsigned long long)))) return rc;

	cudaStream_t st = ctx->stream;
	if (pl.scene_costs) {
		if ((rc = ctx->h_params.ensure(params_bytes))) return rc;
		CU(cudaStreamSynchronize(st));   // no copy from the staging buffer is still in flight
		DevParams* hp = (DevParams*)ctx->h_params.p;
		for (int s = 0; s < NS; ++s) {
			const HmpSceneCosts& sc = pl.scene_costs[s];
			hp[s] = D;
			std::memcpy(hp[s].scale, sc.scale, sizeof(hp[s].scale));
			std::memcpy(hp[s].mg_xshift, sc.xshift, sizeof(hp[s].mg_xshift));
			std::memcpy(hp[s].mg_yshift, sc.yshift, sizeof(hp[s].mg_yshift));
		}
		CU(cudaMemcpyAsync(ctx->d_params.p, hp, params_bytes, cudaMemcpyHostToDevice, st));
	} else {
		CU(cudaMemcpyAsync(ctx->d_params.p, &D, sizeof(DevParams), cudaMemcpyHostToDevice, st));
	}
	CU(cudaMemcpyAsync(ctx->d_amp.p, amp_table.data(), amp_table.size() * sizeof(double), cudaMemcpyHostToDevice, st));
	if (n_extra > 0) CU(cudaMemcpyAsync(ctx->d_extra.p, extra, (size_t)n_extra * sizeof(HmpSample), cudaMemcpyHostToDevice, st));
	if (!equi.empty()) CU(cudaMemcpyAsync(ctx->d_equi.p, equi.data(), equi.size() * sizeof(double), cudaMemcpyHostToDevice, st));
	CU(cudaMemsetAsync(ctx->d_ctrl.p, 0, cl.total, st));

	unsigned char* ctrl = (unsigned char*)ctx->d_ctrl.p;
	KernelArgs A;
	std::memset(&A, 0, sizeof(A));
	A.params = (const DevParams*)ctx->d_params.p;
	A.params_stride = pl.scene_costs ? (uint32_t)sizeof(DevParams) : 0u;
	A.amp_values = (const double*)ctx->d_amp.p;
	A.extra_samples = (const double*)ctx->d_extra.p;
	A.equi_samples = (const double*)ctx->d_equi.p;
	A.scenes = (const uint8_t*)ctx->d_scenes.p;
	A.scene_stride = pl.scene_stride;
	A.n_scenes = NS;
	A.costmaps = (const uint8_t*)ctx->d_costmaps.p;
	A.costmap_stride = ctx->costmap_stride;
	A.costmap_in_smem = in_smem;
	A.precise = (ctx->precise == 1) ? 1 : 0;
	A.mapgrids = (const float*)ctx->d_mapgrids.p;
	A.n_work = D.n_social;
	A.totals = (double*)ctx->d_totals.p;
	A.block_best = (unsigned long long*)ctx->d_block_best.p;
	A.counters = (unsigned int*)(ctrl + cl.off_counters);
	A.hv_out = (unsigned int*)(ctrl + cl.off_hv);
	A.best_out = (double*)(ctrl + cl.off_best);
	A.no_prune = ctx->prune_obstacle ? 0 : 1;
	A.hv_pre = (double*)ctx->d_hvrec.p;
	A.hv_val = (float*)((double*)ctx->d_hvrec.p + hv_items);
	A.debug_cand = -1;
	if (ctx->debug_cand >= 0) {   // hmp_debug_sweep_candidate: the thread-per-candidate sweep writes this candidate's raw critics
		if ((rc = ctx->d_dbg.ensure(32 * sizeof(double)))) return rc;
		CU(cudaMemsetAsync(ctx->d_dbg.p, 0xff, 32 * sizeof(double), ctx->stream));
		A.debug_cand = ctx->debug_cand;
		A.d_costs = (double*)ctx->d_dbg.p;
	}

	CU(cudaEventRecord(ctx->ev0, st));
	// dilated max-cost map for the exact pruning of the obstacle critic (rebuilt when costmap / footprint / separation change)
	if (ctx->prune_obstacle && scale_on(D.scale, pl.scene_costs, NS, HMP_COST_OBSTACLE) && D.n_footprint > 0) {
		if (ctx->dilated_dirty || ctx->dilated_scenes != NS) {
			if ((rc = ctx->d_dilated.ensure((size_t)ctx->costmap_stride * NS))) return rc;
			double r_fp = 0.0, r_k = 0.0;
			for (int i = 0; i < D.n_footprint; ++i) r_fp = std::max(r_fp, std::hypot(D.footprint_x[i], D.footprint_y[i]));
			for (int k = 0; k < D.n_kernel_pts; ++k) r_k = std::max(r_k, std::hypot(D.kernel_dx[k], D.kernel_dy[k]));
			// vertex cells lie within |d| / res + sqrt(2) of the centre cell, rasterised cells within 0.5 of the segment between
			// two vertex cells: radius (r_fp + r_k) / res + 2 covers them all
			const float radius = (float)((r_fp + r_k) / D.resolution + 2.0);
			CU(hmp_dev_launch_dilate((const uint8_t*)ctx->d_costmaps.p, D.size_x, D.size_y, ctx->costmap_stride, radius,
			                         (uint8_t*)ctx->d_dilated.p, NS, st));
			ctx->launches++;
			ctx->dilated_dirty = false;
			ctx->dilated_scenes = NS;
		}
		A.dilated = (const uint8_t*)ctx->d_dilated.p;
	}
	if (D.n_equi > 0) {
		// the second generator of the pool first (a few dozen kinematic rollouts): its best is merged by the main sweep's last block
		KernelArgs E = A;
		E.n_work = D.n_equi;
		E.cand_offset = D.n_social;
		E.best_out = (double*)(ctrl + cl.off_best2);
		E.block_best = A.block_best + (size_t)NS * blocks_x * 2;
		CU(hmp_dev_launch_plan(&E, equi_blocks, 2, smem, st));
		ctx->launches++;
		// work / done tickets of every scene back to zero; the counts (the other two words of a scene's four) accumulate
		CU(cudaMemset2DAsync(ctrl + cl.off_counters, 4 * sizeof(unsigned int), 0, 2 * sizeof(unsigned int), (size_t)NS, st));
		A.best_init = E.best_out;
	}
	if (sweep_mode && ctx->tpc_defer && A.dilated) {
		// deferred obstacle critic: one pose-scratch slot per block that can be resident at once (24 bytes per pose of one ticket)
		const long long grid_blocks = (long long)NS * blocks_x;
		const int n_slots = (int)std::min<long long>(grid_blocks, (long long)ctx->sm_count * std::max(1, ctx->tpc_bps));
		const size_t scr = (size_t)n_slots * (size_t)(sweep_mode & 1023) * T * 3 * sizeof(double);
		if ((rc = ctx->d_posescr.ensure(scr))) return rc;
		if ((rc = ctx->d_poseslots.ensure((size_t)n_slots * sizeof(unsigned int)))) return rc;
		CU(cudaMemsetAsync(ctx->d_poseslots.p, 0, (size_t)n_slots * sizeof(unsigned int), st));
		A.pose_scratch = (double*)ctx->d_posescr.p;
		A.pose_slots = (unsigned int*)ctx->d_poseslots.p;
		A.pose_n_slots = n_slots;
	}
	// Small pools in mode 2 (at most one block-cooperative FP64 wave, e.g. the stock 72 + 30 samples): every candidate is a leader
	// whatever the FP32 sweep says, so the FP64 rollouts do not depend on it and run BESIDE it on a second stream; the FP32
	// sweep still supplies the counters and the highest_valid_cost_ records. (K as in the refinement below.)
	const int k_all = std::max(8, (C + 7) / 8 * 8);
	const bool overlap = ctx->precise == 2 && NS == 1 && ctx->refine_max_leaders <= 0 &&
	                     k_all + blocks_x + equi_blocks <= ctx->sm_count;
	if (overlap) {
		CU(cudaEventRecord(ctx->ev_fork, st));   // inputs of the cycle are on the device (uploads, wave fronts, dilated map)
		CU(cudaStreamWaitEvent(ctx->stream2, ctx->ev_fork, 0));
	}
	CU(hmp_dev_launch_plan(&A, blocks_x, sweep_mode, smem_sweep, st));
	A.pose_scratch = nullptr;   // the detail / refinement launches derived from A do not use it
	A.pose_slots = nullptr;
	ctx->launches++;
	CU(cudaEventRecord(ctx->evm, st));
	// snapshot the counters (n_generated, n_valid) before the detail pass reuses the work ticket
	CU(cudaMemcpyAsync((unsigned char*)ctx->h_out.p + det_bytes, ctrl, cl.total, cudaMemcpyDeviceToHost, st));
	CU(cudaMemsetAsync(ctrl + cl.off_counters, 0, (size_t)NS * 4 * sizeof(unsigned int), st));

	A.d_costs = nullptr;
	KernelArgs B = A;
	B.hv_pre = nullptr;   // detail / refinement launches do not record (the sweep's records stand)
	B.hv_val = nullptr;
	double* det = (double*)ctx->d_detail.p;
	B.d_costs = det;
	B.d_seeds = det + (size_t)NS * HMP_NUM_COSTS;
	B.d_poses = B.d_seeds + (size_t)NS * 3;
	B.totals = B.d_poses + (size_t)NS * T * 3;
	B.d_nposes = (int32_t*)(B.totals + NS);
	B.d_forces = nullptr;
	std::function<int(int, const int32_t*)> refine_round;   // set in mode 2; also drives the fallback rounds below
	int32_t* r_count_dev[2] = {nullptr, nullptr};
	if (ctx->precise != 2) {
		// winner's detail pass: one warp per scene re-runs the best candidate with write-back
		B.n_work = 1;
		B.use_best_index = 1;
		CU(hmp_dev_launch_plan(&B, 1, 1, smem, st));
		ctx->launches++;
		ctx->last_n_leaders = 0;
	} else {
		// selection refinement: leaders of the FP32 sweep -> FP64 rollouts -> winner among the refined totals
		// Leaders per scene. Single-scene plans: the K best-ranked candidates, K = one wave of warp-per-candidate FP64 rollouts
		// (8 per SM: 1184 on a B200; a wave costs the latency of ONE FP64 rollout whatever its size) -- or every candidate when
		// the pool is smaller, in which case the plan is simply the FP64 result. Batches: the 32 best-ranked per scene.
		const int k_cap = (NS == 1) ? (ctx->refine_max_leaders > 0 ? ctx->refine_max_leaders : ctx->sm_count * HMP_WARPS_PER_BLOCK)
		                            : std::min(ctx->refine_max_leaders > 0 ? ctx->refine_max_leaders : 32, 256);
		const int K = std::max(8, (std::min(k_cap, C) + 7) / 8 * 8);
		const bool want_poses = (NS == 1);
		const size_t nk = (size_t)NS * K;
		const size_t r_doubles = nk * (HMP_NUM_COSTS + 3 + 1) + (want_poses ? nk * T * 3 : 0);
		const size_t r_bytes = r_doubles * sizeof(double) + (nk * 2 + 2 * NS) * sizeof(int32_t) + 8;   // one round's buffers, 8-byte aligned
		const size_t r_set = (r_bytes + 15) / 16 * 16;
		// single-scene plans run a second round (below): a second set of buffers + the first round's threshold
		// (not when round 1 already holds every candidate of the pool, C <= K: nothing is left for a second list)
		const int rounds = (NS == 1 && C > K) ? 2 : 1;
		if ((rc = ctx->d_refine.ensure(r_set * rounds + 2 * NS * sizeof(double)))) return rc;   // + (threshold, effective window) of round 1
		double* r_thr = (double*)((unsigned char*)ctx->d_refine.p + r_set * rounds);
		constexpr int REFINE_MIN_LEADERS = 16;   // collect_leaders_kernel: the best-ranked candidates a window-based FIRST round always lists
		refine_round = [=, &r_count_dev](int round, const int32_t* active) -> int {
			unsigned char* base = (unsigned char*)ctx->d_refine.p + r_set * round;
			double* r_costs = (double*)base;
			double* r_seeds = r_costs + nk * HMP_NUM_COSTS;
			double* r_totals = r_seeds + nk * 3;
			double* r_poses = want_poses ? r_totals + nk : nullptr;
			int32_t* r_leaders = (int32_t*)((double*)base + r_doubles);
			int32_t* r_nposes = r_leaders + nk;
			int32_t* r_count = r_nposes + nk;
			int32_t* r_unrel = r_count + NS;   // per scene: leaders whose FP32 total the FP64 evaluation contradicts
			// round 1: rank-based (the K lowest FP32 totals); round 2: everything not yet refined whose FP32 total lies within the
			// window above the REFINED best (at most K, the lowest first)
			const bool beside = overlap && round == 0 && !active;   // first pass of a small pool: see `overlap` above
			cudaStream_t rs = beside ? ctx->stream2 : st;
			if (beside)
				CU(hmp_dev_launch_fill_leaders(r_leaders, K, C, r_count, rs));
			else if (round == 0)
				CU(hmp_dev_launch_collect_topk(A.totals, C, A.best_out, K, ctx->refine_window, r_leaders, r_count, r_thr, NS, active, st));
			else
				CU(hmp_dev_launch_collect_leaders(A.totals, C, A.best_out, ctx->refine_window, K, r_leaders, r_count, r_thr, nullptr,
				                                  REFINE_MIN_LEADERS, NS, active, st));
			KernelArgs Rf = A;
			Rf.hv_pre = nullptr;
			Rf.hv_val = nullptr;
			Rf.precise = 1;
			Rf.cand_list = r_leaders;
			Rf.cand_list_stride = K;
			Rf.n_work = K;
			Rf.use_best_index = 0;
			Rf.d_costs = r_costs;
			Rf.d_seeds = r_seeds;
			Rf.d_poses = r_poses;
			Rf.totals = r_totals;
			Rf.d_nposes = r_nposes;
			Rf.d_forces = nullptr;
			if (beside) Rf.counters = (unsigned int*)(ctrl + cl.off_counters2);   // its own work ticket: the sweep is pulling from A.counters
			// single scene: few candidates, many SMs -> one candidate per BLOCK (block-cooperative instance), as many blocks as
			// the GPU holds; batches have enough leaders in total to keep one warp per candidate
			// The block-cooperative instance finishes a wave of <= sm_count leaders in ~0.85 ms (cfg2), the warp-per-candidate
			// instance any number up to 2 x sm_count in ~1.4 ms; the count is only known on the device, so the choice follows
			// the previous cycle's count (consecutive control cycles have similar leader sets). The second round's list is
			// almost always empty (its blocks find no candidate and leave): one warp per candidate, two per block.
			if (NS == 1 && round == 0 && K <= ctx->sm_count) {
				CU(hmp_dev_launch_plan(&Rf, K, 3, smem, rs));   // a small pool: one block-cooperative FP64 rollout per SM
				if (beside) {
					CU(cudaEventRecord(ctx->ev_join, rs));
					CU(cudaStreamWaitEvent(st, ctx->ev_join, 0));
				}
			} else if (NS == 1) {
				// one wave: every SM takes ceil(K / SMs) candidates, one per warp (round 2 is almost always empty: its blocks leave)
				const int wpt = std::max(1, std::min(HMP_WARPS_PER_BLOCK, (K + ctx->sm_count - 1) / ctx->sm_count));
				Rf.warps_per_ticket = wpt;
				CU(hmp_dev_launch_plan(&Rf, (K + wpt - 1) / wpt, 1, smem, st));
			} else {
				Rf.warps_per_ticket = HMP_WARPS_PER_BLOCK;
				CU(hmp_dev_launch_plan(&Rf, (K + HMP_WARPS_PER_BLOCK - 1) / HMP_WARPS_PER_BLOCK, 1, smem, st));
			}
			CU(hmp_dev_launch_refine_select(r_leaders, K, C, T, r_totals, r_costs, r_seeds, r_poses, r_nposes, A.totals, A.best_out,
			                                B.d_costs, B.d_seeds, B.d_poses, B.totals, B.d_nposes, NS, round, active, r_unrel, st));
			ctx->launches += 3;
			r_count_dev[round] = r_count;   // read back after the last round (a copy to pageable memory here would stall the
			                                // host, and with it the launches of the next round, until this round has finished)
			return HMP_OK;
		};
		// Round 1: leaders within the window of the FP32 best. Round 2: the window above the REFINED best of round 1, minus
		// what round 1 covered -- empty unless the FP32 best was a candidate whose FP32 total is far too low (a chaotic
		// rollout): then the candidates between the two thresholds could beat its FP64 total and are refined too. After
		// round 2 every candidate whose FP32 total lies within the window of the final (FP64) best has been refined.
		// The work ticket is reset between the rounds (both rollouts pull candidates from it).
		ctx->last_n_leaders2 = 0;
		if ((rc = refine_round(0, nullptr))) return rc;
		if (rounds == 2) {
			CU(cudaMemsetAsync(ctrl + cl.off_counters, 0, (size_t)NS * 4 * sizeof(unsigned int), st));
			if ((rc = refine_round(1, nullptr))) return rc;
		}
		// leader counts: into pinned words (a copy to pageable memory would block the host until the stream has drained, i.e.
		// before the hv pass and the result copies are even queued); picked up after the final synchronisation
		if ((rc = ctx->h_small.ensure(64))) return rc;
		int32_t* hw = (int32_t*)ctx->h_small.p;
		hw[0] = hw[1] = hw[2] = 0;
		CU(cudaMemcpyAsync(&hw[0], r_count_dev[0], sizeof(int32_t), cudaMemcpyDeviceToHost, st));
		CU(cudaMemcpyAsync(&hw[2], r_count_dev[0] + NS, sizeof(int32_t), cudaMemcpyDeviceToHost, st));   // r_unrel of scene 0
		if (r_count_dev[1]) CU(cudaMemcpyAsync(&hw[1], r_count_dev[1], sizeof(int32_t), cudaMemcpyDeviceToHost, st));
	}
	// highest_valid_cost_ of the MapGrid critics as the reference's sequential, early-exiting loop would leave it: needs the final
	// explored totals (refined leaders included) for the best-so-far every candidate was scored against
	auto hv_pass = [&]() -> int {
		CU(hmp_dev_launch_hv_early_exit(A.totals, A.hv_pre, A.hv_val, C, A.hv_out, NS, st));
		ctx->launches++;
		return HMP_OK;
	};
	if ((rc = hv_pass())) return rc;
	CU(cudaEventRecord(ctx->ev1, st));
	auto read_back = [&]() -> int {
		CU(cudaMemcpyAsync(ctx->h_out.p, det, det_bytes, cudaMemcpyDeviceToHost, st));
		CU(cudaMemcpyAsync((unsigned char*)ctx->h_out.p + det_bytes + cl.off_hv, ctrl + cl.off_hv, (size_t)NS * 4 * sizeof(unsigned int),
		                   cudaMemcpyDeviceToHost, st));
		if (ctx->precise == 2)   // the refinement may have replaced (best total, best index) after the control-block snapshot
			CU(cudaMemcpyAsync((unsigned char*)ctx->h_out.p + det_bytes + cl.off_best, ctrl + cl.off_best, (size_t)NS * 2 * sizeof(double),
			                   cudaMemcpyDeviceToHost, st));
		CU(cudaStreamSynchronize(st));
		return HMP_OK;
	};
	if ((rc = read_back())) return rc;
	if (ctx->precise == 2) {
		ctx->last_n_leaders = ((const int32_t*)ctx->h_small.p)[0];
		ctx->last_n_leaders2 = ((const int32_t*)ctx->h_small.p)[1];
		ctx->last_unreliable = ((const int32_t*)ctx->h_small.p)[2];
	} else {
		ctx->last_unreliable = 0;
	}
	float ms = 0.f;
	CU(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
	float ms_main = 0.f;
	CU(cudaEventElapsedTime(&ms_main, ctx->ev0, ctx->evm));

	ctx->last_fallback_rounds = 0;
	std::vector<int32_t> unresolved(NS, 0);
	if (ctx->precise == 2) {
		// A scene is UNRESOLVED when the authoritative FP64 evaluation rejected every leader (the published record is the FP32
		// best's, with a negative FP64 total): the FP32 selection must not be handed out. The refined (negative) totals are in
		// the explored-totals array by now, so the best of the remaining valid totals becomes the new FP32 best and another
		// refinement round runs around it -- until a refined winner exists, no valid candidate is left, or 8 rounds have passed
		// (then the scene reports "no valid trajectory", the conservative answer). Rare: costs one host round trip per round.
		const double* h_tot = (const double*)ctx->h_out.p + (size_t)NS * (HMP_NUM_COSTS + 3 + (size_t)T * 3);
		const double* h_b = (const double*)((const unsigned char*)ctx->h_out.p + det_bytes + cl.off_best);
		for (int iter = 0; iter < 8; ++iter) {
			bool any = false;
			for (int s = 0; s < NS; ++s) {
				unresolved[s] = ((int)h_b[2 * s + 1] >= 0 && h_tot[s] < 0.0) ? 1 : 0;
				any |= unresolved[s] != 0;
			}
			if (!any) break;
			if ((rc = ctx->d_mask.ensure((size_t)NS * sizeof(int32_t)))) return rc;
			CU(cudaMemcpyAsync(ctx->d_mask.p, unresolved.data(), (size_t)NS * sizeof(int32_t), cudaMemcpyHostToDevice, st));
			CU(hmp_dev_launch_reselect(A.totals, C, A.best_out, (const int32_t*)ctx->d_mask.p, NS, st));
			ctx->launches++;
			CU(cudaMemsetAsync(ctrl + cl.off_counters, 0, (size_t)NS * 4 * sizeof(unsigned int), st));
			if ((rc = refine_round(0, (const int32_t*)ctx->d_mask.p))) return rc;
			if ((rc = hv_pass())) return rc;
			if ((rc = read_back())) return rc;
			ctx->last_fallback_rounds = iter + 1;
		}
		for (int s = 0; s < NS; ++s) unresolved[s] = ((int)h_b[2 * s + 1] >= 0 && h_tot[s] < 0.0) ? 1 : 0;
	}

	const double* h_det = (const double*)ctx->h_out.p;
	const double* h_costs = h_det;
	const double* h_seeds = h_det + (size_t)NS * HMP_NUM_COSTS;
	const double* h_poses = h_seeds + (size_t)NS * 3;
	const int32_t* h_nposes = (const int32_t*)(h_poses + (size_t)NS * T * 3 + NS);
	const unsigned char* h_ctrl = (const unsigned char*)ctx->h_out.p + det_bytes;
	const unsigned int* h_counters = (const unsigned int*)(h_ctrl + cl.off_counters);
	const unsigned int* h_hv = (const unsigned int*)(h_ctrl + cl.off_hv);
	const double* h_best = (const double*)(h_ctrl + cl.off_best);
	for (int s = 0; s < NS; ++s) {
		HmpResult& r = results[s];
		std::memset(&r, 0, sizeof(r));
		int best = (int)h_best[2 * s + 1];
		if (unresolved[s]) best = -1;   // FP64 rejected every candidate the fallback rounds reached
		r.best_index = best;
		r.status = best >= 0 ? 0 : 1;
		r.n_candidates = C;
		r.n_social = D.n_social;
		r.n_generated = (int)h_counters[4 * s + 2];
		r.n_valid = (int)h_counters[4 * s + 3];
		r.best_total = best >= 0 ? h_best[2 * s] : -7.0;  // caller pre-sets cost_ = -7, humap_planner.cpp:1364
		if (best >= 0 && ctx->precise == 1 && sweep_mode) {
			// exact mode through the thread-per-candidate sweep: its FP32 critics are evaluated in another (equivalent) form than the
			// winner's detail pass, 1e-8 relative apart. The published total is the detail pass's -- the number that goes with the
			// published critics, and the one mode 2 reports for the same candidate.
			const double det_total = (h_det + (size_t)NS * (HMP_NUM_COSTS + 3 + (size_t)T * 3))[s];
			if (det_total >= 0.0) r.best_total = det_total;
		}
		r.time_delta = D.dt_d;
		r.gpu_ms = ms;
		r.gpu_ms_select = ms_main;
		for (int g = 0; g < HMP_NUM_MAPGRIDS; ++g) {
			float f;
			std::memcpy(&f, &h_hv[4 * s + g], sizeof(f));
			r.highest_valid_cost[g] = f;
		}
		for (int k = 0; k < HMP_NUM_COSTS; ++k) r.costs[k] = std::numeric_limits<double>::quiet_NaN();
		if (best >= 0) {
			for (int k = 0; k < HMP_NUM_COSTS; ++k) r.costs[k] = h_costs[(size_t)s * HMP_NUM_COSTS + k];
			r.xv = h_seeds[3 * s];
			r.yv = h_seeds[3 * s + 1];
			r.thetav = h_seeds[3 * s + 2];
			r.n_poses = h_nposes[s];
			if (best < D.n_grid) {
				int rem = best;
				for (int a = HMP_NUM_AMPLIFIERS - 1; a >= 0; --a) {
					int n = D.amp_n[a];
					r.amplifiers[a] = amp_table[(size_t)a * HMP_MAX_AMP_VALUES + rem % n];
					rem /= n;
				}
			} else if (best < D.n_social && extra) {
				for (int a = 0; a < HMP_NUM_AMPLIFIERS; ++a) r.amplifiers[a] = extra[best - D.n_grid].amp[a];
			} else {
				for (int a = 0; a < HMP_NUM_AMPLIFIERS; ++a) r.amplifiers[a] = std::numeric_limits<double>::quiet_NaN();
			}
			if (poses_out && s == 0) {
				int n = std::min<int>(r.n_poses, poses_capacity);
				std::memcpy(poses_out, h_poses + (size_t)s * T * 3, (size_t)n * 3 * sizeof(double));
			}
		}
	}
	ctx->last_n_candidates = C;
	ctx->last_T = T;
	ctx->last_n_scenes = NS;
	ctx->last_scene_stride = pl.scene_stride;
	ctx->last_dev_params = D;
	if (!pl.scene_costs) ctx->last_scene_costs.clear();
	else if (pl.scene_costs != ctx->last_scene_costs.data()) ctx->last_scene_costs.assign(pl.scene_costs, pl.scene_costs + NS);
	if (&amp_table != &ctx->last_amp_table) ctx->last_amp_table = amp_table;
	if (extra != ctx->last_extra.data()) ctx->last_extra.assign(extra, extra + n_extra);
	if (&equi != &ctx->last_equi) ctx->last_equi = equi;
	ctx->last_valid = true;
	return HMP_OK;
}

int hmp_plan(HmpContext* ctx, const HmpWorld* world, const HmpSampling* sampling, const HmpSample* extra, int32_t n_extra,
             HmpResult* result, double* poses_out, int32_t poses_capacity) {
	int rc = check_ready(ctx);
	if (rc) return rc;
	if (!sampling || !result || n_extra < 0 || (n_extra > 0 && !extra) || (poses_out && poses_capacity < 0)) {
		set_err("bad plan arguments");
		return HMP_E_INVALID;
	}
	if ((rc = validate_world(world))) return rc;
	for (int g = 0; g < HMP_NUM_MAPGRIDS; ++g) {
		if (!ctx->have_grid[g] && ctx->params.costs.scale[HMP_COST_PATH + g] != 0.0) {
			set_err("hmp_set_mapgrid(%d) has not been called for the current costmap", g);
			return HMP_E_NOT_READY;
		}
	}
	if (!ctx->have_footprint && ctx->params.costs.scale[HMP_COST_OBSTACLE] != 0.0) {
		set_err("hmp_set_footprint has not been called");
		return HMP_E_NOT_READY;
	}
	CU(cudaSetDevice(ctx->device));
	int T = compute_steps(ctx->params.general, std::hypot(world->vel_x, world->vel_y), world->vel_th);
	if (T < 1 || T > HMP_MAX_STEPS) {
		set_err("rollout has %d steps, supported 1..%d", T, HMP_MAX_STEPS);
		return HMP_E_CAPACITY;
	}
	DevParams D;
	std::vector<double> amp_table;
	if ((rc = build_dev_params(ctx, sampling, n_extra, T, D, amp_table))) return rc;

	size_t blob = scene_blob_bytes(*world);
	if ((rc = ctx->d_scenes.ensure(blob))) return rc;
	if ((rc = ctx->h_stage.ensure(blob))) return rc;
	CU(cudaStreamSynchronize(ctx->stream));
	std::memset(ctx->h_stage.p, 0, blob);
	std::vector<double> equi;
	if (ctx->equi.enabled) {
		equisampled_samples(ctx->params, *world, ctx->equi, D, equi);
		D.n_equi = (int)(equi.size() / 3);
		D.n_candidates = D.n_social + D.n_equi;
	}
	pack_scene(ctx, *world, ctx->hv_prev, D.dt_d, (unsigned char*)ctx->h_stage.p, D.n_equi);
	uint32_t used = reinterpret_cast<DevScene*>(ctx->h_stage.p)->blob_bytes;
	// device wave fronts of this cycle (hmp_compute_mapgrid) have been running on their side streams while the host packed the
	// world; the plan stream joins them here
	if ((rc = join_wavefronts(ctx))) return rc;
	CU(cudaMemcpyAsync(ctx->d_scenes.p, ctx->h_stage.p, used, cudaMemcpyHostToDevice, ctx->stream));
	PlanLaunch pl{1, used, n_extra, T};
	if ((rc = run_cycle(ctx, D, amp_table, extra, n_extra, equi, pl, result, poses_out, poses_capacity))) return rc;
	// Escalation (hmp_set_escalation): the refinement has just compared the FP32 and FP64 totals of the leaders. When many of them
	// disagree by more than 1 % the FP32 ranking of THIS plan is unreliable (chaotic rollouts around a spinning robot: the true
	// winner can sit thousands of ranks down, DESIGN 4b) -- the plan is redone as an exact FP64 sweep on the resident inputs.
	ctx->last_escalated = 0;
	if (ctx->precise == 2 && ctx->escalate_min > 0 && ctx->last_unreliable >= ctx->escalate_min) {
		const int unreliable = ctx->last_unreliable, leaders = ctx->last_n_leaders, leaders2 = ctx->last_n_leaders2;
		const int fallback = ctx->last_fallback_rounds;
		ctx->precise = 1;
		rc = run_cycle(ctx, D, amp_table, extra, n_extra, equi, pl, result, poses_out, poses_capacity);
		ctx->precise = 2;
		ctx->last_unreliable = unreliable;   // the counters keep describing the mode-2 pass that asked for the escalation
		ctx->last_n_leaders = leaders;
		ctx->last_n_leaders2 = leaders2;
		ctx->last_fallback_rounds = fallback;
		ctx->last_escalated = 1;
		if (rc) return rc;
	}
	return HMP_OK;
}

// Uploads the per-scene costmaps of a batch (scene s = cells + s * size_x * size_y) into the padded device layout.
static int upload_batch_costmaps(HmpContext* ctx, const uint8_t* cells, int n_scenes) {
	const size_t n = (size_t)ctx->size_x * ctx->size_y;
	int rc;
	if ((rc = ctx->d_costmaps.ensure((size_t)ctx->costmap_stride * n_scenes))) return rc;
	CU(cudaMemcpy2DAsync(ctx->d_costmaps.p, ctx->costmap_stride, cells, n, n, n_scenes, cudaMemcpyHostToDevice, ctx->stream));
	CU(cudaStreamSynchronize(ctx->stream));
	ctx->h_cells.assign(cells, cells + n);   // scene 0 is what a later single-scene call sees
	ctx->costmap_scenes = n_scenes;
	ctx->dilated_dirty = true;
	ctx->last_valid = false;
	return HMP_OK;
}

// MapGridCostFunction::setTargetPoses + prepare() for n_scenes x 4 grids in ONE launch: seeds on the host, the wave fronts on
// the device (one block per grid, hmp_dev_launch_wavefront), so that a batch uploads 1 byte per cell (the costmap)
// instead of 17 (costmap + four float grids).
int hmp_compute_mapgrid_batch(HmpContext* ctx, int32_t n_scenes, const uint8_t* cells, const double* const plan_xy[HMP_NUM_MAPGRIDS],
                              const int32_t* const plan_start[HMP_NUM_MAPGRIDS], const int32_t local_goal[HMP_NUM_MAPGRIDS]) {
	int rc = check_ready(ctx);
	if (rc) return rc;
	if (n_scenes <= 0 || !plan_xy || !plan_start || !local_goal) {
		set_err("bad batch mapgrid arguments");
		return HMP_E_INVALID;
	}
	for (int g = 0; g < HMP_NUM_MAPGRIDS; ++g) {
		if (!plan_xy[g] || !plan_start[g]) {
			set_err("plan_xy[%d] / plan_start[%d] is null", g, g);
			return HMP_E_INVALID;
		}
		for (int s = 0; s < n_scenes; ++s)
			if (plan_start[g][s] < 0 || plan_start[g][s + 1] < plan_start[g][s]) {
				set_err("plan_start[%d] is not a non-decreasing prefix array at scene %d", g, s);
				return HMP_E_INVALID;
			}
	}
	CU(cudaSetDevice(ctx->device));
	if ((rc = join_wavefronts(ctx))) return rc;
	const int sx = ctx->size_x, sy = ctx->size_y;
	const size_t n = (size_t)sx * sy;
	if (hmp_dev_wavefront_smem(sx, sy) > ctx->max_smem_optin) {
		set_err("costmap too large for the on-device wave front");
		return HMP_E_CAPACITY;
	}
	if (cells) {
		if ((rc = upload_batch_costmaps(ctx, cells, n_scenes))) return rc;
	} else if (ctx->costmap_scenes < n_scenes) {
		set_err("hmp_compute_mapgrid_batch needs the per-scene costmap cells (%d scenes resident, %d asked)", ctx->costmap_scenes, n_scenes);
		return HMP_E_NOT_READY;
	}
	// seeds of all (scene, grid) pairs on the host threads: [offsets n_items + 1][seeds ...]
	const size_t items = (size_t)n_scenes * HMP_NUM_MAPGRIDS;
	std::vector<std::vector<int>> seeds(items);
	std::vector<uint8_t> cells_dev;   // only when the cells are not passed again (seed test needs them): read back
	const uint8_t* cells_h = cells;
	if (!cells_h) {
		cells_dev.resize(n * n_scenes);
		CU(cudaMemcpy2D(cells_dev.data(), n, ctx->d_costmaps.p, ctx->costmap_stride, n, n_scenes, cudaMemcpyDeviceToHost));
		cells_h = cells_dev.data();
	}
	{
		const unsigned nt = (unsigned)std::max<size_t>(1, std::min<size_t>(std::min(16u, std::max(1u, std::thread::hardware_concurrency())), items / 64 + 1));
		auto work = [&](unsigned t) {
			for (size_t it = t; it < items; it += nt) {
				const int s = (int)(it / HMP_NUM_MAPGRIDS), g = (int)(it % HMP_NUM_MAPGRIDS);
				const int a = plan_start[g][s], b = plan_start[g][s + 1];
				collect_seeds(ctx, cells_h + (size_t)s * n, plan_xy[g] + 2 * (size_t)a, b - a, local_goal[g], seeds[it]);
			}
		};
		std::vector<std::thread> pool;
		for (unsigned t = 1; t < nt; ++t) pool.emplace_back(work, t);
		work(0);
		for (auto& th : pool) th.join();
	}
	size_t total = 0;
	for (auto& v : seeds) total += v.size();
	const size_t words = (items + 1) + std::max<size_t>(1, total);
	if ((rc = ctx->d_seeds[0].ensure(words * sizeof(int)))) return rc;
	CU(cudaStreamSynchronize(ctx->stream));
	if ((rc = ctx->h_seeds[0].ensure(words * sizeof(int)))) return rc;
	int* off = (int*)ctx->h_seeds[0].p;
	int* sd = off + items + 1;
	size_t pos = 0;
	for (size_t it = 0; it < items; ++it) {
		off[it] = (int)pos;
		if (!seeds[it].empty()) std::memcpy(sd + pos, seeds[it].data(), seeds[it].size() * sizeof(int));
		pos += seeds[it].size();
	}
	off[items] = (int)pos;
	if ((rc = ctx->d_mapgrids.ensure(n * HMP_NUM_MAPGRIDS * sizeof(float) * n_scenes))) return rc;
	// The wave fronts run on slot 0's side stream and are NOT waited for here: the caller's next step (hmp_plan_batch packs and
	// uploads the worlds) overlaps them; join_wavefronts() orders them before the first kernel that reads the grids. The
	// costmaps are on the device already (upload_batch_costmaps synchronised).
	cudaStream_t st = ctx->wf_stream[0];
	int* d = (int*)ctx->d_seeds[0].p;
	CU(cudaMemcpyAsync(d, off, words * sizeof(int), cudaMemcpyHostToDevice, st));
	CU(cudaEventRecord(ctx->seeds_event[0], st));   // slot 0's staging buffer: hmp_compute_mapgrid(0) waits for this copy
	ctx->seeds_event_valid[0] = true;
	CU(hmp_dev_launch_wavefront((const uint8_t*)ctx->d_costmaps.p, ctx->costmap_stride, sx, sy, d + items + 1, d, (float*)ctx->d_mapgrids.p,
	                            HMP_NUM_MAPGRIDS, n_scenes, st));
	ctx->launches++;
	for (int g = 0; g < HMP_NUM_MAPGRIDS; ++g) {   // the batch writes every slot of scene 0
		CU(cudaEventRecord(ctx->wf_done[g], st));
		ctx->wf_after_batch[g] = true;
	}
	ctx->wavefront_pending[0] = true;
	for (bool& b : ctx->have_grid) b = true;
	ctx->batch_grid_scenes = n_scenes;
	ctx->last_valid = false;
	return HMP_OK;
}

// Uploads n_scenes x 4 wave-front grids that are already FLOAT (cell counts are exact in FP32 below 2^24) straight from the
// caller's buffers -- pinned memory makes the copy asynchronous at full PCIe rate -- without the double -> float pass of
// hmp_plan_batch's target_dist argument. Values are the caller's responsibility here (hmp_set_mapgrid states the contract).
int hmp_set_mapgrids_batch_f32(HmpContext* ctx, int32_t n_scenes, const float* const target_dist[HMP_NUM_MAPGRIDS]) {
	int rc = check_ready(ctx);
	if (rc) return rc;
	if (n_scenes <= 0 || !target_dist || !target_dist[0] || !target_dist[1] || !target_dist[2] || !target_dist[3]) {
		set_err("bad batch mapgrid arguments");
		return HMP_E_INVALID;
	}
	CU(cudaSetDevice(ctx->device));
	if ((rc = join_wavefronts(ctx))) return rc;
	const size_t n = (size_t)ctx->size_x * ctx->size_y;
	if ((rc = ctx->d_mapgrids.ensure(n * HMP_NUM_MAPGRIDS * sizeof(float) * n_scenes))) return rc;
	for (int g = 0; g < HMP_NUM_MAPGRIDS; ++g)   // [scene][grid][cells] on the device, [scene][cells] per grid on the host
		CU(cudaMemcpy2DAsync((float*)ctx->d_mapgrids.p + (size_t)g * n, n * HMP_NUM_MAPGRIDS * sizeof(float), target_dist[g], n * sizeof(float),
		                     n * sizeof(float), n_scenes, cudaMemcpyHostToDevice, ctx->stream));
	CU(cudaStreamSynchronize(ctx->stream));
	for (bool& b : ctx->have_grid) b = true;
	ctx->batch_grid_scenes = n_scenes;
	ctx->last_valid = false;
	return HMP_OK;
}

int hmp_plan_batch(HmpContext* ctx, const HmpWorld* worlds, int32_t n_scenes, const uint8_t* cells,
                   const double* const target_dist[HMP_NUM_MAPGRIDS], const double* highest_valid_cost_prev,
                   const HmpSampling* sampling, HmpResult* results) {
	int rc = check_ready(ctx);
	if (rc) return rc;
	if (!worlds || n_scenes <= 0 || !sampling || !results) {
		set_err("bad batch arguments");
		return HMP_E_INVALID;
	}
	if (!ctx->scene_costs.empty() && (size_t)n_scenes > ctx->scene_costs.size()) {
		set_err("the per-scene cost table holds %zu scenes, the batch has %d", ctx->scene_costs.size(), n_scenes);
		return HMP_E_INVALID;
	}
	const HmpSceneCosts* table = ctx->scene_costs.empty() ? nullptr : ctx->scene_costs.data();
	const double* scale = ctx->params.costs.scale;
	if (!ctx->have_footprint && scale_on(scale, table, n_scenes, HMP_COST_OBSTACLE)) {
		set_err("hmp_set_footprint has not been called");
		return HMP_E_NOT_READY;
	}
	CU(cudaSetDevice(ctx->device));
	const size_t n = (size_t)ctx->size_x * ctx->size_y;
	int T = -1;
	size_t stride = 0;
	for (int s = 0; s < n_scenes; ++s) {
		if ((rc = validate_world(&worlds[s]))) return rc;
		int Ts = compute_steps(ctx->params.general, std::hypot(worlds[s].vel_x, worlds[s].vel_y), worlds[s].vel_th);
		if (T < 0) T = Ts;
		if (Ts != T) {
			set_err("scenes of one batch must share the step count (scene %d: %d vs %d)", s, Ts, T);
			return HMP_E_INVALID;
		}
		stride = std::max(stride, scene_blob_bytes(worlds[s]));
	}
	if (T < 1 || T > HMP_MAX_STEPS) {
		set_err("rollout has %d steps, supported 1..%d", T, HMP_MAX_STEPS);
		return HMP_E_CAPACITY;
	}
	// what the kernels will index must be resident for EVERY scene: costmaps and (if a MapGrid critic is on) the four grids
	const bool any_grid = target_dist && (target_dist[0] || target_dist[1] || target_dist[2] || target_dist[3]);
	if (any_grid) {
		for (int g = 0; g < HMP_NUM_MAPGRIDS; ++g) {
			if (!target_dist[g]) {
				set_err("target_dist[%d] is null", g);
				return HMP_E_INVALID;
			}
		}
	} else {
		for (int g = 0; g < HMP_NUM_MAPGRIDS; ++g) {
			if (!scale_on(scale, table, n_scenes, HMP_COST_PATH + g)) continue;
			if (n_scenes == 1 ? !ctx->have_grid[g] : ctx->batch_grid_scenes < n_scenes) {
				set_err("MapGrid %d is not resident for %d scene(s): pass target_dist or call hmp_compute_mapgrid_batch / hmp_set_mapgrids_batch_f32 first", g,
				        n_scenes);
				return HMP_E_NOT_READY;
			}
		}
	}
	if (!cells && ctx->costmap_scenes < n_scenes) {
		set_err("hmp_plan_batch needs per-scene costmap cells (%d scene(s) resident, %d asked)", ctx->costmap_scenes, n_scenes);
		return HMP_E_INVALID;
	}
	DevParams D;
	std::vector<double> amp_table;
	if ((rc = build_dev_params(ctx, sampling, 0, T, D, amp_table))) return rc;
	if ((rc = ctx->d_scenes.ensure(stride * n_scenes))) return rc;
	if (any_grid) {
		if ((rc = ctx->d_mapgrids.ensure(n * HMP_NUM_MAPGRIDS * sizeof(float) * n_scenes))) return rc;
	}
	size_t stage = std::max(stride * n_scenes, std::max((size_t)ctx->costmap_stride, n * sizeof(float)));
	if ((rc = ctx->h_stage.ensure(stage))) return rc;
	CU(cudaStreamSynchronize(ctx->stream));
	unsigned char* hs = (unsigned char*)ctx->h_stage.p;
	std::memset(hs, 0, stride * n_scenes);
	std::vector<std::vector<double>> equi_scene;
	std::vector<double> equi_all;
	{
		// scene blobs packed by the host threads (a 4096-world batch is ~12 MB of records)
		const unsigned nt = (unsigned)std::max(1, std::min<int>(std::min(16u, std::max(1u, std::thread::hardware_concurrency())), n_scenes / 64 + 1));
		// second generator of the pool (hmp_set_equisampled): every world has its own velocity window, hence its own samples and,
		// where the window spans zero, its own sample count; the batch takes the largest count and pads (DevScene.n_equi)
		const bool with_equi = ctx->equi.enabled != 0;
		if (with_equi) equi_scene.resize((size_t)n_scenes);
		auto work = [&](unsigned t) {
			DevParams Dt = D;   // equisampled_samples also fills the (shared) acceleration limits; the per-thread copy is discarded
			for (int s = (int)t; s < n_scenes; s += (int)nt) {
				int ne = 0;
				if (with_equi) {
					equisampled_samples(ctx->params, worlds[s], ctx->equi, Dt, equi_scene[(size_t)s]);
					ne = (int)(equi_scene[(size_t)s].size() / 3);
				}
				pack_scene(ctx, worlds[s], highest_valid_cost_prev ? highest_valid_cost_prev + 4 * (size_t)s : nullptr, D.dt_d, hs + stride * s, ne);
			}
		};
		std::vector<std::thread> pool;
		for (unsigned t = 1; t < nt; ++t) pool.emplace_back(work, t);
		work(0);
		for (auto& th : pool) th.join();
		if (with_equi) {
			std::vector<double> dummy;
			equisampled_samples(ctx->params, worlds[0], ctx->equi, D, dummy);   // acceleration limits / continued flag into D
			size_t ne_max = 0;
			for (const auto& v : equi_scene) ne_max = std::max(ne_max, v.size() / 3);
			equi_all.assign((size_t)n_scenes * ne_max * 3, 0.0);
			for (int s = 0; s < n_scenes; ++s)
				std::copy(equi_scene[(size_t)s].begin(), equi_scene[(size_t)s].end(), equi_all.begin() + (size_t)s * ne_max * 3);
			D.n_equi = (int)ne_max;
			D.n_candidates = D.n_social + D.n_equi;
		}
	}
	CU(cudaMemcpyAsync(ctx->d_scenes.p, hs, stride * n_scenes, cudaMemcpyHostToDevice, ctx->stream));
	CU(cudaStreamSynchronize(ctx->stream));
	// device wave fronts still in flight (hmp_compute_mapgrid[_batch]) ran beside the packing above; join them now
	if ((rc = join_wavefronts(ctx))) return rc;
	if (cells) {
		if ((rc = upload_batch_costmaps(ctx, cells, n_scenes))) return rc;
	}
	if (any_grid) {
		// double -> float conversion of n_scenes x 4 grids (328 MB for 512 scenes of 200 x 200) by all host threads into two
		// pinned staging buffers; the copy of one chunk of scenes overlaps the conversion of the next. Values must be cell
		// counts in [0, size_x * size_y + 1] (the contract of hmp_set_mapgrid), checked on the way.
		const size_t scene_floats = n * HMP_NUM_MAPGRIDS;
		const int chunk = (int)std::max<size_t>(1, std::min<size_t>((size_t)n_scenes, ((size_t)48 << 20) / (scene_floats * sizeof(float))));
		if ((rc = ctx->h_grid_stage[0].ensure((size_t)chunk * scene_floats * sizeof(float)))) return rc;
		if ((rc = ctx->h_grid_stage[1].ensure((size_t)chunk * scene_floats * sizeof(float)))) return rc;
		for (int b = 0; b < 2; ++b)
			if (!ctx->grid_stage_ev[b]) CU(cudaEventCreateWithFlags(&ctx->grid_stage_ev[b], cudaEventDisableTiming));
		const unsigned hw = std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
		const double limit = (double)n + 1.0;
		int buf = 0;
		int bad_any = 0;
		for (int s0 = 0; s0 < n_scenes; s0 += chunk, buf ^= 1) {
			const int ns = std::min(chunk, n_scenes - s0);
			if (s0 >= 2 * chunk) CU(cudaEventSynchronize(ctx->grid_stage_ev[buf]));   // the copy that last read this buffer
			float* f = (float*)ctx->h_grid_stage[buf].p;
			const size_t items = (size_t)ns * HMP_NUM_MAPGRIDS;   // (scene, grid) pairs of this chunk
			const unsigned nt = (unsigned)std::min<size_t>(hw, items);
			std::vector<int> bad_t(nt, 0);
			auto work = [&](unsigned t) {
				int bad = 0;
				for (size_t it = t; it < items; it += nt) {
					const int s = s0 + (int)(it / HMP_NUM_MAPGRIDS), g = (int)(it % HMP_NUM_MAPGRIDS);
					const double* src = target_dist[g] + (size_t)s * n;
					float* dst = f + it * n;
					for (size_t i = 0; i < n; ++i) {
						const double v = src[i];
						const int iv = (int)v;   // NaN / out-of-range convert to INT_MIN on x86-64 and fail the round trip
						bad |= ((double)iv != v) | (iv < 0) | (v > limit);
						dst[i] = (float)iv;
					}
				}
				bad_t[t] = bad;
			};
			std::vector<std::thread> pool;
			for (unsigned t = 1; t < nt; ++t) pool.emplace_back(work, t);
			work(0);
			for (auto& th : pool) th.join();
			for (int b : bad_t) bad_any |= b;
			if (bad_any) break;
			CU(cudaMemcpyAsync((float*)ctx->d_mapgrids.p + (size_t)s0 * scene_floats, f, items * n * sizeof(float), cudaMemcpyHostToDevice,
			                   ctx->stream));
			CU(cudaEventRecord(ctx->grid_stage_ev[buf], ctx->stream));
		}
		if (bad_any) {
			CU(cudaStreamSynchronize(ctx->stream));
			ctx->batch_grid_scenes = 0;
			for (bool& b : ctx->have_grid) b = false;
			set_err("a target_dist value is not a cell count in [0, size_x*size_y+1]");
			return HMP_E_INVALID;
		}
		for (bool& b : ctx->have_grid) b = true;
		ctx->batch_grid_scenes = n_scenes;
	}
	PlanLaunch pl{n_scenes, (uint32_t)stride, 0, T, table};
	return run_cycle(ctx, D, amp_table, nullptr, 0, equi_all, pl, results, nullptr, 0);
}

// Re-runs the selection of the last plan on the data still resident on the device (no host<->device
// traffic except the 16-byte result): used to time the kernels with inputs already in HBM.
int hmp_replan_resident(HmpContext* ctx, HmpResult* results, int32_t results_capacity) {
	if (!ctx || !results || !ctx->last_valid) {
		set_err("no previous plan to re-run");
		return HMP_E_NOT_READY;
	}
	if (results_capacity < ctx->last_n_scenes) {
		set_err("results holds %d records, the last plan had %d scenes", results_capacity, ctx->last_n_scenes);
		return HMP_E_INVALID;
	}
	CU(cudaSetDevice(ctx->device));
	PlanLaunch pl{ctx->last_n_scenes, ctx->last_scene_stride, (int)ctx->last_extra.size(), ctx->last_T,
	              ctx->last_scene_costs.empty() ? nullptr : ctx->last_scene_costs.data()};
	return run_cycle(ctx, ctx->last_dev_params, ctx->last_amp_table, pl.n_extra ? ctx->last_extra.data() : nullptr, pl.n_extra,
	                 ctx->last_equi, pl, results, nullptr, 0);
}

int hmp_get_explored_totals(HmpContext* ctx, double* totals, int32_t n) {
	if (!ctx || !totals || !ctx->last_valid) {
		set_err("no previous plan");
		return HMP_E_NOT_READY;
	}
	if (n != ctx->last_n_candidates * ctx->last_n_scenes) {
		set_err("n = %d, expected %d", n, ctx->last_n_candidates * ctx->last_n_scenes);
		return HMP_E_INVALID;
	}
	CU(cudaSetDevice(ctx->device));
	CU(cudaMemcpyAsync(totals, ctx->d_totals.p, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
	CU(cudaStreamSynchronize(ctx->stream));
	return HMP_OK;
}

int hmp_explain(HmpContext* ctx, const int32_t* candidate_indices, int32_t n, double* costs_out, double* seeds_out,
                double* poses_out, int32_t* n_steps_out) {
	if (!ctx || !candidate_indices || n <= 0 || !ctx->last_valid) {
		set_err("no previous plan or bad arguments");
		return HMP_E_NOT_READY;
	}
	if (ctx->last_n_scenes != 1) {
		set_err("hmp_explain works on single-scene plans");
		return HMP_E_INVALID;
	}
	CU(cudaSetDevice(ctx->device));
	const DevParams& D = ctx->last_dev_params;
	const int T = D.T;
	const size_t doubles = (size_t)n * (HMP_NUM_COSTS + 3 + (size_t)T * 3 + (size_t)T * 8);
	const size_t bytes = doubles * sizeof(double) + (size_t)n * 2 * sizeof(int32_t);
	int rc;
	if ((rc = ctx->d_dbg.ensure(bytes))) return rc;
	if ((rc = ctx->h_out.ensure(bytes))) return rc;
	double* base = (double*)ctx->d_dbg.p;
	int32_t* d_idx = (int32_t*)(base + doubles);
	int32_t* d_np = d_idx + n;
	cudaStream_t st = ctx->stream;
	CU(cudaMemcpyAsync(d_idx, candidate_indices, (size_t)n * sizeof(int32_t), cudaMemcpyHostToDevice, st));
	const CtrlLayout cl = ctrl_layout(1);
	unsigned char* ctrl = (unsigned char*)ctx->d_ctrl.p;
	CU(cudaMemsetAsync(ctrl + cl.off_counters, 0, 4 * sizeof(unsigned int), st));
	int blocks_x = 0, in_smem = 0;
	size_t smem = 0;
	PlanLaunch pl{1, ctx->last_scene_stride, 0, T};
	if ((rc = launch_main(ctx, D, pl, &blocks_x, &smem, &in_smem))) return rc;
	KernelArgs A;
	std::memset(&A, 0, sizeof(A));
	A.params = (const DevParams*)ctx->d_params.p;
	A.amp_values = (const double*)ctx->d_amp.p;
	A.extra_samples = (const double*)ctx->d_extra.p;
	A.equi_samples = (const double*)ctx->d_equi.p;
	A.scenes = (const uint8_t*)ctx->d_scenes.p;
	A.scene_stride = ctx->last_scene_stride;
	A.n_scenes = 1;
	A.costmaps = (const uint8_t*)ctx->d_costmaps.p;
	A.costmap_stride = ctx->costmap_stride;
	A.costmap_in_smem = in_smem;
	A.precise = (ctx->precise == 1) ? 1 : 0;
	A.mapgrids = (const float*)ctx->d_mapgrids.p;
	A.cand_list = d_idx;
	A.n_work = n;
	A.counters = (unsigned int*)(ctrl + cl.off_counters);
	A.hv_out = (unsigned int*)(ctrl + cl.off_hv);
	A.best_out = (double*)(ctrl + cl.off_best);
	A.d_costs = base;
	A.d_seeds = A.d_costs + (size_t)n * HMP_NUM_COSTS;
	A.d_poses = A.d_seeds + (size_t)n * 3;
	A.d_forces = A.d_poses + (size_t)n * T * 3;
	A.d_nposes = d_np;
	int bx = (int)std::min<long long>(((long long)n + HMP_WARPS_PER_BLOCK - 1) / HMP_WARPS_PER_BLOCK, (long long)ctx->sm_count * 4);
	CU(cudaMemsetAsync(base, 0, doubles * sizeof(double), st));
	CU(hmp_dev_launch_plan(&A, bx, 1, smem, st));
	ctx->launches++;
	CU(cudaMemcpyAsync(ctx->h_out.p, base, bytes, cudaMemcpyDeviceToHost, st));
	CU(cudaStreamSynchronize(st));
	const double* h = (const double*)ctx->h_out.p;
	if (costs_out) std::memcpy(costs_out, h, (size_t)n * HMP_NUM_COSTS * sizeof(double));
	if (seeds_out) std::memcpy(seeds_out, h + (size_t)n * HMP_NUM_COSTS, (size_t)n * 3 * sizeof(double));
	if (poses_out) std::memcpy(poses_out, h + (size_t)n * (HMP_NUM_COSTS + 3), (size_t)n * T * 3 * sizeof(double));
	if (n_steps_out) std::memcpy(n_steps_out, (const int32_t*)(h + doubles) + n, (size_t)n * sizeof(int32_t));
	ctx->last_explain_n = n;   // h_out holds this call's forces until another call reuses it (hmp_debug_last_forces)
	ctx->last_explain_T = T;
	return HMP_OK;
}

// Per-step forces of the candidates of the last hmp_explain call: [n][T][8] doubles
// (internal.xy, dynamic.xy, static.xy, human-action.xy). Parity-test hook.
int hmp_debug_last_forces(HmpContext* ctx, int32_t n, double* forces_out) {
	if (!ctx || !forces_out || !ctx->last_valid || n <= 0) {
		set_err("bad arguments");
		return HMP_E_INVALID;
	}
	if (n != ctx->last_explain_n || ctx->last_dev_params.T != ctx->last_explain_T) {
		set_err("the last hmp_explain call covered %d candidates x %d steps, not %d x %d (or another call reused its buffer)",
		        ctx->last_explain_n, ctx->last_explain_T, n, ctx->last_dev_params.T);
		return HMP_E_NOT_READY;
	}
	const int T = ctx->last_dev_params.T;
	const double* h = (const double*)ctx->h_out.p;
	std::memcpy(forces_out, h + (size_t)n * (HMP_NUM_COSTS + 3 + (size_t)T * 3), (size_t)n * T * 8 * sizeof(double));
	return HMP_OK;
}

int hmp_num_steps(HmpContext* ctx) { return (ctx && ctx->last_valid) ? ctx->last_T : -1; }

// ---- parity hooks ------------------------------------------------------------------------------------
static int debug_params(HmpContext* ctx, DevParams& D) {
	HmpSampling s;
	for (int a = 0; a < HMP_NUM_AMPLIFIERS; ++a) {
		s.amp_min[a] = s.amp_max[a] = 1.0;
		s.amp_granularity[a] = 1.0;
	}
	std::vector<double> amp;
	int rc = build_dev_params(ctx, &s, 0, 1, D, amp);
	if (rc) return rc;
	if ((rc = ctx->d_params.ensure(sizeof(DevParams)))) return rc;
	CU(cudaMemcpyAsync(ctx->d_params.p, &D, sizeof(D), cudaMemcpyHostToDevice, ctx->stream));
	ctx->last_valid = false;
	return HMP_OK;
}

int hmp_debug_world_to_map(HmpContext* ctx, const double* wx, const double* wy, int32_t n, int32_t* mx, int32_t* my,
                           int32_t* ok) {
	int rc = check_ready(ctx);
	if (rc) return rc;
	if (!wx || !wy || !mx || !my || !ok || n <= 0) {
		set_err("bad arguments");
		return HMP_E_INVALID;
	}
	CU(cudaSetDevice(ctx->device));
	DevParams D;
	if ((rc = debug_params(ctx, D))) return rc;
	size_t bytes = (size_t)n * (2 * sizeof(double) + 3 * sizeof(int32_t));
	if ((rc = ctx->d_dbg.ensure(bytes))) return rc;
	double* dwx = (double*)ctx->d_dbg.p;
	double* dwy = dwx + n;
	int32_t* dmx = (int32_t*)(dwy + n);
	int32_t* dmy = dmx + n;
	int32_t* dok = dmy + n;
	cudaStream_t st = ctx->stream;
	CU(cudaMemcpyAsync(dwx, wx, (size_t)n * sizeof(double), cudaMemcpyHostToDevice, st));
	CU(cudaMemcpyAsync(dwy, wy, (size_t)n * sizeof(double), cudaMemcpyHostToDevice, st));
	CU(hmp_dev_launch_world_to_map((const DevParams*)ctx->d_params.p, dwx, dwy, n, dmx, dmy, dok, st));
	ctx->launches++;
	CU(cudaMemcpyAsync(mx, dmx, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
	CU(cudaMemcpyAsync(my, dmy, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
	CU(cudaMemcpyAsync(ok, dok, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
	CU(cudaStreamSynchronize(st));
	return HMP_OK;
}

int hmp_debug_footprint_cost(HmpContext* ctx, const double* xyt, int32_t n, double* cost) {
	int rc = check_ready(ctx);
	if (rc) return rc;
	if (!xyt || !cost || n <= 0 || !ctx->have_footprint) {
		set_err("bad arguments or footprint missing");
		return HMP_E_INVALID;
	}
	CU(cudaSetDevice(ctx->device));
	DevParams D;
	if ((rc = debug_params(ctx, D))) return rc;
	size_t bytes = (size_t)n * 4 * sizeof(double);
	if ((rc = ctx->d_dbg.ensure(bytes))) return rc;
	double* dx = (double*)ctx->d_dbg.p;
	double* dc = dx + 3 * (size_t)n;
	cudaStream_t st = ctx->stream;
	CU(cudaMemcpyAsync(dx, xyt, (size_t)n * 3 * sizeof(double), cudaMemcpyHostToDevice, st));
	CU(hmp_dev_launch_footprint_cost((const DevParams*)ctx->d_params.p, (const uint8_t*)ctx->d_costmaps.p, dx, n, dc, st));
	ctx->launches++;
	CU(cudaMemcpyAsync(cost, dc, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, st));
	CU(cudaStreamSynchronize(st));
	return HMP_OK;
}

// HumapPlanner::computeCellCost for every cell of the costmap (diagnostics; see cost_cloud_kernel)
int hmp_compute_cost_cloud(HmpContext* ctx, float* cloud6, uint8_t* valid) {
	int rc = check_ready(ctx);
	if (rc) return rc;
	if (!cloud6 || !valid) {
		set_err("null output");
		return HMP_E_INVALID;
	}
	for (int g = 0; g < HMP_NUM_MAPGRIDS; ++g) {
		if (!ctx->have_grid[g]) {
			set_err("hmp_set_mapgrid(%d) has not been called for the current costmap", g);
			return HMP_E_NOT_READY;
		}
	}
	CU(cudaSetDevice(ctx->device));
	if ((rc = join_wavefronts(ctx))) return rc;
	DevParams D;
	if ((rc = debug_params(ctx, D))) return rc;
	const size_t n = (size_t)ctx->size_x * ctx->size_y;
	if ((rc = ctx->d_dbg.ensure(n * 6 * sizeof(float) + n))) return rc;
	float* d_out = (float*)ctx->d_dbg.p;
	uint8_t* d_valid = (uint8_t*)(d_out + n * 6);
	cudaStream_t st = ctx->stream;
	CU(hmp_dev_launch_cost_cloud((const DevParams*)ctx->d_params.p, (int)n, (const uint8_t*)ctx->d_costmaps.p,
	                             (const float*)ctx->d_mapgrids.p, ctx->hv_prev, d_out, d_valid, st));
	ctx->launches++;
	CU(cudaMemcpyAsync(cloud6, d_out, n * 6 * sizeof(float), cudaMemcpyDeviceToHost, st));
	CU(cudaMemcpyAsync(valid, d_valid, n, cudaMemcpyDeviceToHost, st));
	CU(cudaStreamSynchronize(st));
	return HMP_OK;
}

// ---- environment model ---------------------------------------------------------------------------------------------
namespace {

struct EnvSelection {
	// host copies, valid after the caller's stream synchronisation (env_select queues their read-back)
	std::vector<int32_t> objects;          // >= 0 shape index, < 0 person -(index + 1); World::addObstacle order (first counts[0] + counts[1])
	std::vector<int32_t> people, groups;   // people_env_model_, groups_env_model_ (first counts[1] / counts[2] entries)
	int32_t counts[3] = {0, 0, 0};         // selected shapes, people, groups
	int row_stride = 0;                    // capacity of one position's row of closest-point records (shapes + people)
	// device pointers into ctx->d_env (valid until the next call)
	const HmpShape* d_shapes = nullptr;
	const double* d_verts = nullptr;
	const HmpPerson* d_people = nullptr;
	int32_t* d_objects = nullptr;
	int32_t* d_counts = nullptr;
	int32_t* d_psel = nullptr;
	int32_t* d_gsel = nullptr;
	int n_people = 0, n_groups = 0;
	double* d_positions = nullptr;
	HmpObstacle* d_out = nullptr;
};

size_t align16(size_t v) { return (v + 15) / 16 * 16; }

// Uploads the inputs, then on the device: extractNonPeopleObstacles + the N-closest metric (env_filter_kernel) and
// selectRelevant for obstacles / people / groups (env_select_kernel). Nothing is waited for: the selection stays on the device
// for env_closest_points_kernel, its read-back into `sel` is queued and becomes valid with the caller's synchronisation.
int env_select(HmpContext* ctx, const HmpEnvParams& env, const double robot_pose[3], const HmpShape* shapes, int n_shapes,
               const double* verts, int n_verts, const HmpPerson* people, int n_people, const HmpGroup* groups, int n_groups,
               int n_positions, EnvSelection& sel) {
	if (env.robot_model < HMP_ROBOT_POINT || env.robot_model > HMP_ROBOT_POLYGON) {
		set_err("robot_model %d: unknown footprint model (0 point, 1 circular, 2 two circles, 3 line, 4 polygon)", env.robot_model);
		return HMP_E_INVALID;
	}
	if (env.robot_model == HMP_ROBOT_POLYGON && (env.n_polygon < 1 || env.n_polygon > HMP_MAX_ENV_POLYGON)) {
		set_err("polygon footprint model with %d vertices (1..%d supported)", env.n_polygon, HMP_MAX_ENV_POLYGON);
		return HMP_E_INVALID;
	}
	for (int i = 0; i < n_shapes; ++i) {
		const HmpShape& s = shapes[i];
		if (s.type < HMP_SHAPE_POINT || s.type > HMP_SHAPE_POLYGON ||
		    (s.type == HMP_SHAPE_POLYGON && (s.n_vertices < 1 || s.first_vertex < 0 || s.first_vertex + s.n_vertices > n_verts))) {
			set_err("shape %d is malformed", i);
			return HMP_E_INVALID;
		}
	}
	const size_t n_obj_max = (size_t)n_shapes + n_people;
	const size_t b_shapes = align16(std::max(1, n_shapes) * sizeof(HmpShape));
	const size_t b_verts = align16(std::max(1, n_verts) * 2 * sizeof(double));
	const size_t b_people = align16(std::max(1, n_people) * sizeof(HmpPerson));
	const size_t b_groups = align16(std::max(1, n_groups) * sizeof(HmpGroup));
	const size_t b_keep = align16(std::max(1, n_shapes) * sizeof(int32_t));
	const size_t b_metric = align16(std::max(1, n_shapes) * sizeof(double));
	const size_t b_scratch = align16(std::max(1, std::max(n_people, n_groups)) * sizeof(double));
	const size_t b_objects = align16(std::max<size_t>(1, n_obj_max) * sizeof(int32_t));
	const size_t b_psel = align16(std::max(1, n_people) * sizeof(int32_t));
	const size_t b_gsel = align16(std::max(1, n_groups) * sizeof(int32_t));
	const size_t b_counts = 16;
	const size_t b_pos = align16(std::max(1, n_positions) * 2 * sizeof(double));
	const size_t b_out = align16(std::max<size_t>(1, n_obj_max * n_positions) * sizeof(HmpObstacle));
	int rc;
	if ((rc = ctx->d_env.ensure(b_shapes + b_verts + b_people + b_groups + b_keep + b_metric + b_scratch + b_objects + b_psel + b_gsel + b_counts +
	                            b_pos + b_out)))
		return rc;
	unsigned char* q = (unsigned char*)ctx->d_env.p;
	auto take = [&](size_t bytes) {
		unsigned char* r = q;
		q += bytes;
		return r;
	};
	HmpShape* d_shapes = (HmpShape*)take(b_shapes);
	double* d_verts = (double*)take(b_verts);
	HmpPerson* d_people = (HmpPerson*)take(b_people);
	HmpGroup* d_groups = (HmpGroup*)take(b_groups);
	int32_t* d_keep = (int32_t*)take(b_keep);
	double* d_metric = (double*)take(b_metric);
	double* d_scratch = (double*)take(b_scratch);
	sel.d_objects = (int32_t*)take(b_objects);
	int32_t* d_psel = (int32_t*)take(b_psel);
	int32_t* d_gsel = (int32_t*)take(b_gsel);
	sel.d_counts = (int32_t*)take(b_counts);
	sel.d_positions = (double*)take(b_pos);
	sel.d_out = (HmpObstacle*)take(b_out);
	sel.d_shapes = d_shapes;
	sel.d_verts = d_verts;
	sel.d_people = d_people;
	sel.row_stride = (int)n_obj_max;
	cudaStream_t st = ctx->stream;
	if (n_shapes > 0) CU(cudaMemcpyAsync(d_shapes, shapes, (size_t)n_shapes * sizeof(HmpShape), cudaMemcpyHostToDevice, st));
	if (n_verts > 0) CU(cudaMemcpyAsync(d_verts, verts, (size_t)n_verts * 2 * sizeof(double), cudaMemcpyHostToDevice, st));
	if (n_people > 0) CU(cudaMemcpyAsync(d_people, people, (size_t)n_people * sizeof(HmpPerson), cudaMemcpyHostToDevice, st));
	if (n_groups > 0) CU(cudaMemcpyAsync(d_groups, groups, (size_t)n_groups * sizeof(HmpGroup), cudaMemcpyHostToDevice, st));
	if (n_shapes > 0) {
		CU(hmp_dev_launch_env_filter(d_shapes, n_shapes, d_verts, d_people, n_people, env.person_model_radius, env.person_containment_rate,
		                             robot_pose[0], robot_pose[1], d_keep, d_metric, st));
		ctx->launches++;
	}
	CU(hmp_dev_launch_env_select(d_keep, d_metric, n_shapes, d_people, n_people, d_groups, n_groups, robot_pose[0], robot_pose[1],
	                             env.obstacles_closest_num, env.people_closest_num, env.groups_closest_num, d_scratch, sel.d_objects, d_psel,
	                             d_gsel, sel.d_counts, st));
	ctx->launches++;
	sel.d_psel = d_psel;
	sel.d_gsel = d_gsel;
	sel.n_people = n_people;
	sel.n_groups = n_groups;
	return HMP_OK;
}

// Reads the selection and n_positions rows of closest-point records back through the pinned staging buffer: ONE synchronisation.
int env_read_back(HmpContext* ctx, EnvSelection& sel, int n_positions, std::vector<HmpObstacle>& records) {
	const size_t cap = (size_t)sel.row_stride;
	const size_t o_counts = 0, o_objects = 16, o_people = o_objects + align16(std::max<size_t>(1, cap) * 4);
	const size_t o_groups = o_people + align16(std::max(1, sel.n_people) * 4), o_rec = o_groups + align16(std::max(1, sel.n_groups) * 4);
	const size_t total = o_rec + std::max<size_t>(1, cap * n_positions) * sizeof(HmpObstacle);
	int rc;
	if ((rc = ctx->h_out.ensure(total))) return rc;
	ctx->last_explain_n = 0;   // h_out is reused
	unsigned char* h = (unsigned char*)ctx->h_out.p;
	cudaStream_t st = ctx->stream;
	CU(cudaMemcpyAsync(h + o_counts, sel.d_counts, 3 * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
	if (cap > 0) CU(cudaMemcpyAsync(h + o_objects, sel.d_objects, cap * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
	if (sel.n_people > 0) CU(cudaMemcpyAsync(h + o_people, sel.d_psel, (size_t)sel.n_people * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
	if (sel.n_groups > 0) CU(cudaMemcpyAsync(h + o_groups, sel.d_gsel, (size_t)sel.n_groups * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
	if (cap > 0) CU(cudaMemcpyAsync(h + o_rec, sel.d_out, cap * n_positions * sizeof(HmpObstacle), cudaMemcpyDeviceToHost, st));
	CU(cudaStreamSynchronize(st));
	std::memcpy(sel.counts, h + o_counts, 3 * sizeof(int32_t));
	sel.objects.assign((const int32_t*)(h + o_objects), (const int32_t*)(h + o_objects) + cap);
	sel.people.assign((const int32_t*)(h + o_people), (const int32_t*)(h + o_people) + sel.n_people);
	sel.groups.assign((const int32_t*)(h + o_groups), (const int32_t*)(h + o_groups) + sel.n_groups);
	records.assign((const HmpObstacle*)(h + o_rec), (const HmpObstacle*)(h + o_rec) + cap * n_positions);
	return HMP_OK;
}

}  // namespace

int hmp_build_environment(HmpContext* ctx, const HmpEnvParams* env, const double robot_pose[3], const double pose_ref[3],
                          const HmpShape* shapes, int32_t n_shapes, const double* vertices_xy, int32_t n_vertices,
                          const HmpPerson* people, int32_t n_people, const HmpGroup* groups, int32_t n_groups,
                          HmpObstacle* obstacles_out, int32_t* n_obstacles_out, int32_t* people_selected,
                          int32_t* n_people_selected, int32_t* groups_selected, int32_t* n_groups_selected) {
	if (!ctx || !env || !robot_pose || !pose_ref || n_shapes < 0 || n_vertices < 0 || n_people < 0 || n_groups < 0 ||
	    (n_shapes > 0 && !shapes) || (n_vertices > 0 && !vertices_xy) || (n_people > 0 && !people) || (n_groups > 0 && !groups) ||
	    !obstacles_out || !n_obstacles_out || !people_selected || !n_people_selected || !groups_selected || !n_groups_selected) {
		set_err("bad environment arguments");
		return HMP_E_INVALID;
	}
	CU(cudaSetDevice(ctx->device));
	EnvSelection sel;
	int rc = env_select(ctx, *env, robot_pose, shapes, n_shapes, vertices_xy, n_vertices, people, n_people, groups, n_groups, 1, sel);
	if (rc) return rc;
	// one launch over the capacity (the counts stay on the device), one synchronisation for selection + records
	cudaStream_t st = ctx->stream;
	std::vector<HmpObstacle> records;
	CU(cudaMemcpyAsync(sel.d_positions, pose_ref, 2 * sizeof(double), cudaMemcpyHostToDevice, st));
	if (sel.row_stride > 0) {
		CU(hmp_dev_launch_env_closest(sel.d_shapes, sel.d_verts, sel.d_people, sel.d_objects, sel.d_counts, sel.row_stride, sel.d_positions, 1,
		                              pose_ref[2], env, sel.d_out, st));
		ctx->launches++;
	}
	if ((rc = env_read_back(ctx, sel, 1, records))) return rc;
	const int n_obj = sel.counts[0] + sel.counts[1];
	if (n_obj > *n_obstacles_out) {
		set_err("environment model has %d objects, capacity %d", n_obj, *n_obstacles_out);
		return HMP_E_CAPACITY;
	}
	std::copy(records.begin(), records.begin() + n_obj, obstacles_out);
	*n_obstacles_out = n_obj;
	std::copy(sel.people.begin(), sel.people.begin() + sel.counts[1], people_selected);
	*n_people_selected = sel.counts[1];
	std::copy(sel.groups.begin(), sel.groups.begin() + sel.counts[2], groups_selected);
	*n_groups_selected = sel.counts[2];
	return HMP_OK;
}

int hmp_compute_force_grid(HmpContext* ctx, const HmpEnvParams* env, const HmpWorld* world, const double* positions_xy,
                           int32_t n_positions, const HmpShape* shapes, int32_t n_shapes, const double* vertices_xy,
                           int32_t n_vertices, double* forces_out) {
	int rc = check_ready(ctx);
	if (rc) return rc;
	if (!env || !world || !positions_xy || n_positions <= 0 || n_shapes < 0 || n_vertices < 0 || (n_shapes > 0 && !shapes) ||
	    (n_vertices > 0 && !vertices_xy) || !forces_out || world->n_people < 0 || world->n_groups < 0 ||
	    (world->n_people > 0 && !world->people) || (world->n_groups > 0 && !world->groups)) {
		set_err("bad force-grid arguments");
		return HMP_E_INVALID;
	}
	CU(cudaSetDevice(ctx->device));
	const double robot_pose[3] = {world->robot_x, world->robot_y, world->robot_yaw};
	EnvSelection sel;
	if ((rc = env_select(ctx, *env, robot_pose, shapes, n_shapes, vertices_xy, n_vertices, world->people, world->n_people, world->groups,
	                     world->n_groups, n_positions, sel)))
		return rc;
	cudaStream_t st = ctx->stream;
	const int cap = sel.row_stride;
	std::vector<HmpObstacle> records;
	if (cap > 0) {
		CU(cudaMemcpyAsync(sel.d_positions, positions_xy, (size_t)n_positions * 2 * sizeof(double), cudaMemcpyHostToDevice, st));
		CU(hmp_dev_launch_env_closest(sel.d_shapes, sel.d_verts, sel.d_people, sel.d_objects, sel.d_counts, cap, sel.d_positions, n_positions,
		                              world->robot_yaw, env, sel.d_out, st));
		ctx->launches++;
	}
	if ((rc = env_read_back(ctx, sel, n_positions, records))) return rc;
	const int n_obj = sel.counts[0] + sel.counts[1];
	// one world per position: the robot there with the yaw of pose_, velocity vel_ rotated by pose_ (computeVelocityGlobal(vel_,
	// pose_), humap_planner.cpp:654-656 -- the yaw is the same), goals unchanged; the motion model runs once with
	// SampleAmplifierSet() and dt = sim_period (social_trajectory_generator.cpp:504-527)
	HmpSampling unit;
	for (int a = 0; a < HMP_NUM_AMPLIFIERS; ++a) {
		unit.amp_min[a] = unit.amp_max[a] = 1.0;
		unit.amp_granularity[a] = 1.0;
	}
	DevParams D;
	std::vector<double> amp_table;
	if ((rc = build_dev_params(ctx, &unit, 0, 1, D, amp_table))) return rc;
	D.dt_d = ctx->params.general.sim_period;
	D.dt = (float)D.dt_d;
	std::vector<HmpWorld> worlds((size_t)n_positions, *world);
	size_t stride = 0;
	for (int i = 0; i < n_positions; ++i) {
		HmpWorld& w = worlds[i];
		w.robot_x = positions_xy[2 * i];
		w.robot_y = positions_xy[2 * i + 1];
		w.obstacles = n_obj > 0 ? records.data() + (size_t)i * cap : nullptr;
		w.n_obstacles = n_obj;
		w.people = nullptr;
		w.n_people = 0;
		w.groups = nullptr;
		w.n_groups = 0;
		stride = std::max(stride, scene_blob_bytes(w));
	}
	if ((rc = ctx->d_scenes.ensure(stride * n_positions))) return rc;
	if ((rc = ctx->h_stage.ensure(stride * n_positions))) return rc;
	unsigned char* hs = (unsigned char*)ctx->h_stage.p;
	std::memset(hs, 0, stride * n_positions);
	for (int i = 0; i < n_positions; ++i) pack_scene(ctx, worlds[i], nullptr, D.dt_d, hs + stride * i);
	CU(cudaMemcpyAsync(ctx->d_scenes.p, hs, stride * n_positions, cudaMemcpyHostToDevice, st));
	if ((rc = ctx->d_params.ensure(sizeof(DevParams)))) return rc;
	if ((rc = ctx->d_amp.ensure(amp_table.size() * sizeof(double)))) return rc;
	const CtrlLayout cl = ctrl_layout(n_positions);
	if ((rc = ctx->d_ctrl.ensure(cl.total))) return rc;
	const size_t f_bytes = (size_t)n_positions * 8 * sizeof(double);
	if ((rc = ctx->d_dbg.ensure(f_bytes))) return rc;
	CU(cudaMemcpyAsync(ctx->d_params.p, &D, sizeof(DevParams), cudaMemcpyHostToDevice, st));
	CU(cudaMemcpyAsync(ctx->d_amp.p, amp_table.data(), amp_table.size() * sizeof(double), cudaMemcpyHostToDevice, st));
	CU(cudaMemsetAsync(ctx->d_ctrl.p, 0, cl.total, st));
	CU(cudaMemsetAsync(ctx->d_dbg.p, 0, f_bytes, st));
	const size_t smem = hmp_dev_smem_bytes((uint32_t)stride, 0, 0);
	if (smem > ctx->max_smem_optin) {
		set_err("scene does not fit shared memory");
		return HMP_E_CAPACITY;
	}
	unsigned char* ctrl = (unsigned char*)ctx->d_ctrl.p;
	KernelArgs A;
	std::memset(&A, 0, sizeof(A));
	A.params = (const DevParams*)ctx->d_params.p;
	A.amp_values = (const double*)ctx->d_amp.p;
	A.scenes = (const uint8_t*)ctx->d_scenes.p;
	A.scene_stride = (uint32_t)stride;
	A.n_scenes = n_positions;
	A.costmaps = (const uint8_t*)ctx->d_costmaps.p;   // untouched: forces_only
	A.costmap_stride = 0;
	A.costmap_in_smem = 0;
	A.precise = 1;                                    // diagnostics: FP64 object loops
	A.mapgrids = (const float*)ctx->d_mapgrids.p;
	A.n_work = 1;
	A.forces_only = 1;
	A.counters = (unsigned int*)(ctrl + cl.off_counters);
	A.hv_out = (unsigned int*)(ctrl + cl.off_hv);
	A.best_out = (double*)(ctrl + cl.off_best);
	A.d_forces = (double*)ctx->d_dbg.p;
	CU(hmp_dev_launch_plan(&A, 1, 1, smem, st));
	ctx->launches++;
	CU(cudaMemcpyAsync(forces_out, ctx->d_dbg.p, f_bytes, cudaMemcpyDeviceToHost, st));
	CU(cudaStreamSynchronize(st));
	ctx->last_valid = false;
	return HMP_OK;
}

// Measured FP32 FFMA throughput of this device at the main sweep's launch shape (2 x 256 threads per SM): the denominator of
// bench.py's roofline next to the nominal SMs x 128 lanes x 2 x clock. Best of 5 timed launches of ~2 ms.
int hmp_debug_measure_fp32_peak(HmpContext* ctx, double* tflops_out) {
	if (!ctx || !tflops_out) {
		set_err("bad arguments");
		return HMP_E_INVALID;
	}
	CU(cudaSetDevice(ctx->device));
	int rc = ctx->d_dbg.ensure(64);
	if (rc) return rc;
	const int blocks = ctx->sm_count * 2, iters = 1 << 16;
	cudaStream_t st = ctx->stream;
	CU(hmp_dev_launch_ffma_peak(blocks, iters, (float*)ctx->d_dbg.p, st));   // warm-up
	double best_ms = 1e30;
	for (int k = 0; k < 5; ++k) {
		CU(cudaEventRecord(ctx->ev0, st));
		CU(hmp_dev_launch_ffma_peak(blocks, iters, (float*)ctx->d_dbg.p, st));
		CU(cudaEventRecord(ctx->ev1, st));
		CU(cudaStreamSynchronize(st));
		float ms = 0.f;
		CU(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
		best_ms = std::min(best_ms, (double)ms);
		ctx->launches++;
	}
	*tflops_out = (double)blocks * 256.0 * (double)iters * 8.0 * 2.0 / (best_ms * 1e-3) / 1e12;
	return HMP_OK;
}

// fuzz::Processor::process on the device for n input tuples (dir_alpha, dir_beta, rel_loc, dist_angle);
// out: (value, membership) per tuple.
int hmp_debug_fis(HmpContext* ctx, const double* in4, int32_t n, double* out2) {
	if (!ctx || !in4 || !out2 || n <= 0) {
		set_err("bad arguments");
		return HMP_E_INVALID;
	}
	CU(cudaSetDevice(ctx->device));
	int rc;
	if ((rc = ctx->d_dbg.ensure((size_t)n * 6 * sizeof(double)))) return rc;
	double* din = (double*)ctx->d_dbg.p;
	double* dout = din + (size_t)n * 4;
	cudaStream_t st = ctx->stream;
	CU(cudaMemcpyAsync(din, in4, (size_t)n * 4 * sizeof(double), cudaMemcpyHostToDevice, st));
	CU(hmp_dev_launch_fis(din, n, dout, ctx->precise == 1, st));
	ctx->launches++;
	CU(cudaMemcpyAsync(out2, dout, (size_t)n * 2 * sizeof(double), cudaMemcpyDeviceToHost, st));
	CU(cudaStreamSynchronize(st));
	return HMP_OK;
}

// 0: FP32 object loops and FIS -- the fast path. 1: the same kernel instantiated with FP64 object loops and
// FIS (vertex quantisation included) -- parity mode used to separate restatement errors from FP32 rounding.
// 2 (default): FP32 sweep over all candidates, then the leaders (hmp_set_refinement) are rolled out again in FP64 and the winner
// is chosen among the refined totals: the selection, the command and the winner's record are those of the FP64 path.
int hmp_set_precision(HmpContext* ctx, int32_t fp64) {
	if (!ctx) {
		set_err("null context");
		return HMP_E_INVALID;
	}
	ctx->precise = (fp64 == 2) ? 2 : (fp64 ? 1 : 0);
	ctx->last_valid = false;
	return HMP_OK;
}

int hmp_set_sweep_layout(HmpContext* ctx, int32_t layout) {
	if (!ctx || layout < 0 || layout > 2) {
		set_err("bad sweep layout (0 auto, 1 warp per candidate, 2 thread per candidate)");
		return HMP_E_INVALID;
	}
	ctx->sweep_layout = layout;
	return HMP_OK;
}

int hmp_last_sweep_mode(HmpContext* ctx) { return ctx ? (ctx->last_sweep_mode & 1023) : -1; }   // bit 10 = register-rich instance

int hmp_set_equisampled(HmpContext* ctx, const HmpEquisampled* eq) {
	if (!ctx) {
		set_err("null context");
		return HMP_E_INVALID;
	}
	if (eq && eq->enabled && (eq->vx_samples < 0 || eq->vy_samples < 0 || eq->vth_samples < 0 ||
	                          (long long)(eq->vx_samples + 1) * (eq->vy_samples + 1) * (eq->vth_samples + 1) > (1 << 20))) {
		set_err("bad equisampled sample counts");
		return HMP_E_INVALID;
	}
	if (eq) ctx->equi = *eq;
	else ctx->equi.enabled = 0;
	ctx->last_valid = false;
	return HMP_OK;
}

int hmp_set_scene_costs(HmpContext* ctx, const HmpSceneCosts* costs, int32_t n_scenes) {
	if (!ctx || n_scenes < 0 || (n_scenes > 0 && !costs)) {
		set_err("bad scene cost arguments (null context, negative count or null table)");
		return HMP_E_INVALID;
	}
	if (!costs || n_scenes == 0) {
		ctx->scene_costs.clear();
		return HMP_OK;
	}
	for (int s = 0; s < n_scenes; ++s) {
		const double* v = (const double*)&costs[s];
		for (size_t i = 0; i < sizeof(HmpSceneCosts) / sizeof(double); ++i)
			if (!std::isfinite(v[i])) {
				set_err("scene %d: non-finite scale or shift", s);
				return HMP_E_INVALID;
			}
	}
	ctx->scene_costs.assign(costs, costs + n_scenes);
	return HMP_OK;
}

int hmp_set_refinement(HmpContext* ctx, double rel_window, int32_t max_leaders) {
	if (!ctx || !(rel_window >= 0.0) || max_leaders < 0 || max_leaders > 4096) {
		set_err("bad refinement arguments (window >= 0, 0 <= max_leaders <= 4096; 0 = the SM count)");
		return HMP_E_INVALID;
	}
	ctx->refine_window = rel_window;
	ctx->refine_max_leaders = (max_leaders + 7) / 8 * 8;   // 0 stays 0: automatic
	return HMP_OK;
}

int hmp_last_num_leaders(HmpContext* ctx) { return (ctx && ctx->last_valid) ? ctx->last_n_leaders : -1; }

int hmp_last_num_leaders_round2(HmpContext* ctx) { return (ctx && ctx->last_valid) ? ctx->last_n_leaders2 : -1; }

// Parity hook: re-runs the last plan and returns what the thread-per-candidate SWEEP computed for one social candidate: the 14
// raw critic values, the seed twist (x, w) and the pose after the last step (the detail / explain passes always run one warp
// per candidate, so they cannot show a deviation of the sweep's own arithmetic). out19: 19 doubles (NaN: sweep ran another layout).
int hmp_debug_sweep_candidate(HmpContext* ctx, int32_t candidate, double* out19) {
	if (!ctx || !out19 || !ctx->last_valid || candidate < 0 || candidate >= ctx->last_dev_params.n_social) {
		set_err("bad arguments or no previous plan");
		return HMP_E_INVALID;
	}
	std::vector<HmpResult> res((size_t)ctx->last_n_scenes);
	ctx->debug_cand = candidate;
	int rc = hmp_replan_resident(ctx, res.data(), ctx->last_n_scenes);
	ctx->debug_cand = -1;
	if (rc) return rc;
	CU(cudaMemcpy(out19, ctx->d_dbg.p, 19 * sizeof(double), cudaMemcpyDeviceToHost));
	return HMP_OK;
}

// Page-locked host memory for the buffers a caller hands to the batch entry points every cycle (costmaps, plans, float
// grids): copies from it run at the full PCIe rate and asynchronously; from pageable memory the driver stages them.
void* hmp_host_alloc(size_t bytes) {
	void* p = nullptr;
	if (cudaMallocHost(&p, std::max<size_t>(bytes, 1)) != cudaSuccess) {
		set_err("cudaMallocHost(%zu) failed: %s", bytes, cudaGetErrorString(cudaGetLastError()));
		return nullptr;
	}
	return p;
}
void hmp_host_free(void* p) {
	if (p) cudaFreeHost(p);
}

int hmp_last_fallback_rounds(HmpContext* ctx) { return (ctx && ctx->last_valid) ? ctx->last_fallback_rounds : -1; }

int hmp_set_escalation(HmpContext* ctx, int32_t min_unreliable_leaders) {
	if (!ctx || min_unreliable_leaders < 0) {
		set_err("bad escalation threshold");
		return HMP_E_INVALID;
	}
	ctx->escalate_min = min_unreliable_leaders;
	return HMP_OK;
}
int hmp_last_unreliable_leaders(HmpContext* ctx) { return (ctx && ctx->last_valid) ? ctx->last_unreliable : -1; }
int hmp_last_escalated(HmpContext* ctx) { return (ctx && ctx->last_valid) ? ctx->last_escalated : -1; }

int hmp_last_num_scenes(HmpContext* ctx) { return (ctx && ctx->last_valid) ? ctx->last_n_scenes : -1; }

int64_t hmp_launch_count(HmpContext* ctx) { return ctx ? ctx->launches : 0; }

}  // extern "C"
