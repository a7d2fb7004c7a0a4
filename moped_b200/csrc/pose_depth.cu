// pose_depth.cu — moped3d's depth-aware POSE stages (SURVEY.md §8f row 4):
//   variant 0  POSE_RANSAC_LM_DIFF_BACKPROJECTION_DEPTH_CPU (moped3d/libmoped/src/pose/POSE_RANSAC_LM_DIFF_BACKPROJECTION_DEPTH_CPU.hpp:57-470)
//   variant 1  POSE_RANSAC_LM_DIFF_REPROJECTION_DEPTH_CPU   (moped3d/libmoped/src/pose/POSE_RANSAC_LM_DIFF_REPROJECTION_DEPTH_CPU.hpp:57-435)
// and, with the same machinery, the moped2 stage in "exact order" mode (mc_set_option "pose_exact_order"):
//   variant 2  POSE_RANSAC_LM_DIFF_REPROJECTION_CPU         (moped2/libmoped/src/pose/POSE_RANSAC_LM_DIFF_REPROJECTION_CPU.hpp:57-307)
//
// One WARP owns one RANSAC test (sample fit -> inlier test -> refit on the inliers) through depth_pose.cuh /
// lm_exact.cuh: an LM whose every sum runs in levmar's order, so the poses are those of the strict-IEEE build of the
// reference bit for bit (the stage is too ill-conditioned in fp32 for a tolerance to mean much — DESIGN.md §2, §4.9).
// This file is compiled with -fmad=false (products and sums round separately, like the oracle's -ffp-contract=off)
// and -ftz=true (the reference process runs FTZ/DAZ).
// The LM work arrays (5 vectors + the Jacobian, 11 floats per residual) live in a per-warp slice of a global scratch
// buffer: a warp touches only its own slice, which stays in the SM's L1/L2.
#include "common.cuh"
#include "ransac_sample.cuh"
#include "depth_pose.cuh"

#include <algorithm>

namespace mc {

static_assert(sizeof(lmx::Cam) == sizeof(Camera), "lmx::Cam must mirror mc::Camera");

constexpr int kDepthWarps = 4;                 // warps (= concurrent RANSAC tests) per CTA
constexpr int kNoSuccess = 0x7fffffff;

__host__ __device__ inline size_t depth_slice_floats(int n_max, int R) {
	// LM work + selection list + count word (hypothesis_scratch_floats) + inlier mask bytes, rounded to 128 B
	const size_t f = ((size_t)R * n_max) * (4 + lmx::M) + 64 + (size_t)n_max + 16 + ((size_t)n_max + 3) / 4 + 1;
	return (f + 31) & ~(size_t)31;
}

__device__ __forceinline__ lmx::Cluster cluster_view(const int32_t *cluster_offsets, int c, const float *xy, const float *xyz, const float *world,
                                                     const float *cauchy, const int32_t *image, const Camera *cams, float alpha) {
	const int lo = cluster_offsets[c];
	lmx::Cluster v;
	v.n = cluster_offsets[c + 1] - lo;
	v.xy = xy + 2 * (size_t)lo; v.xyz = xyz + 3 * (size_t)lo; v.world = world ? world + 3 * (size_t)lo : nullptr; v.cauchy = cauchy ? cauchy + lo : nullptr; v.image = image + lo;
	v.cams = reinterpret_cast<const lmx::Cam *>(cams); v.alpha = alpha;
	return v;
}

// ---- explicit hypotheses: persistent grid, one TEAM of W lanes per (sample set, initial quaternion) ----
// W = 32: a warp per hypothesis (default). W = 8: four hypotheses per warp (mc_set_option "depth_team_lanes", 8) — a 10-row sample fit
// leaves most of a warp idle, but teams of one warp that take different LM paths serialise; which wins is a measurement.
template <int V, int W>
__global__ void __launch_bounds__(32 * kDepthWarps)
k_depth_hypotheses(const int32_t *__restrict__ cluster_offsets, const float *__restrict__ xy, const float *__restrict__ xyz,
                   const float *__restrict__ world, const float *__restrict__ cauchy, const int32_t *__restrict__ image,
                   const Camera *__restrict__ cams, float alpha, const int32_t *__restrict__ hyp_cluster, const int32_t *__restrict__ sample_pos,
                   const float *__restrict__ init_quat, int n_hyp, int n_align, int max_lm, float thr, int min_npts, int finite_check,
                   float *__restrict__ scratch, size_t slice, int n_max, const int64_t *__restrict__ mask_offsets, int32_t *__restrict__ n_inliers,
                   float *__restrict__ pose_lm_out, float *__restrict__ pose_refit_out, float *__restrict__ lm_err_out, uint8_t *__restrict__ mask_out) {
	constexpr int R = lmx::DepthResiduals<V>::R;
	constexpr int kTeams = 32 / W;                                  // teams per warp
	const int lane = threadIdx.x & 31;
	const int team_id = (blockIdx.x * kDepthWarps + (threadIdx.x >> 5)) * kTeams + lane / W, n_teams = gridDim.x * kDepthWarps * kTeams;
	float *my = scratch + (size_t)team_id * slice;
	uint8_t *my_mask = reinterpret_cast<uint8_t *>(my + lmx::hypothesis_scratch_floats(n_max, R));
	lmx::Team<W> team;
	team.init(lane);
	for (int h = team_id; h < n_hyp; h += n_teams) {
		const lmx::Cluster c = cluster_view(cluster_offsets, hyp_cluster[h], xy, xyz, world, cauchy, image, cams, alpha);
		uint8_t *mask = mask_out ? mask_out + mask_offsets[h] : my_mask;
		const float quat[4] = { init_quat[4 * h], init_quat[4 * h + 1], init_quat[4 * h + 2], init_quat[4 * h + 3] };
		float pose_lm[7] = { 0, 0, 0, 0, 0, 0, 0 }, pose_refit[7] = { 0, 0, 0, 0, 0, 0, 0 }, err2[2];
		// the LM work area is laid out for THIS cluster's size (hypothesis() carves it with c.n), inside the slice sized for n_max
		const int cnt = lmx::hypothesis<V, W>(team, c, sample_pos + (size_t)h * n_align, n_align, quat, max_lm, thr, min_npts, my, mask,
		                                      finite_check != 0, pose_lm, pose_refit, err2);
		if (team.lane == 0) {
			n_inliers[h] = cnt;
			lm_err_out[2 * h] = err2[0]; lm_err_out[2 * h + 1] = err2[1];
			for (int j = 0; j < 7; j++) { pose_lm_out[7 * h + j] = pose_lm[j]; pose_refit_out[7 * h + j] = pose_refit[j]; }
		}
		team.sync();
	}
}

// ---- RANSAC: one CTA per (cluster, try) task, one warp per test, rounds of kDepthWarps consecutive tests ----
// Reference semantics (RANSAC(), …BACKPROJECTION_DEPTH_CPU.hpp:278-314): sequential tests, return at the FIRST one whose
// consistent set exceeds MinNPtsObject, refitted on that set. The lowest successful index of a round is that test.
// kDevCount: the cluster count is read from the device (*n_clusters_p, at most n_clusters_cap); tasks past it find nothing
template <int V, bool kDevCount>
__global__ void __launch_bounds__(32 * kDepthWarps)
k_depth_ransac(const int32_t *__restrict__ cluster_offsets, int n_clusters_cap, const int32_t *__restrict__ n_clusters_p, const float *__restrict__ xy, const float *__restrict__ xyz,
               const float *__restrict__ world, const float *__restrict__ cauchy, const int32_t *__restrict__ image,
               const int32_t *__restrict__ tie, const Camera *__restrict__ cams, float alpha, int max_obj, int max_ransac, int max_lm, int n_align,
               int min_npts, float thr, uint64_t seed, int finite_check, float *__restrict__ scratch, size_t slice, int n_max,
               int n_tasks, uint8_t *__restrict__ found, float *__restrict__ pose_out, int32_t *__restrict__ n_tests) {
	constexpr int R = lmx::DepthResiduals<V>::R;
	__shared__ int s_first, s_fail;
	__shared__ float s_pose[kDepthWarps][7];           // refitted pose of each warp's successful test of the current round
	const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
	// persistent grid over the tasks: the LM scratch is one slice per warp of the RESIDENT CTAs, not of every task
	float *my = scratch + ((size_t)blockIdx.x * kDepthWarps + w) * slice;
	uint8_t *my_mask = reinterpret_cast<uint8_t *>(my + lmx::hypothesis_scratch_floats(n_max, R));
	lmx::Team<32> team;
	team.init(lane);
	const int n_clusters = kDevCount ? min(*n_clusters_p, n_clusters_cap) : n_clusters_cap;
	for (int task = blockIdx.x; task < n_tasks; task += gridDim.x) {
	const int cidx = task / max_obj;
	if (cidx >= n_clusters) { if (threadIdx.x == 0) { found[task] = 0; n_tests[task] = 0; } continue; }
	const lmx::Cluster c = cluster_view(cluster_offsets, cidx, xy, xyz, world, cauchy, image, cams, alpha);
	const int32_t *ctie = tie ? tie + cluster_offsets[cidx] : nullptr;
	const uint64_t task_seed = seed + 0x9E3779B97F4A7C15ULL * (uint64_t)(task + 1);
	__syncthreads();                                   // the previous task's s_first / s_pose have been read
	if (threadIdx.x == 0) { s_first = kNoSuccess; s_fail = 0; }
	__syncthreads();
	int tests = 0;
	for (int base = 0; base < max_ransac; base += kDepthWarps) {
		const int h = base + w;
		if (h < max_ransac) {
			int pos[kMaxAlign]; float quat[4];
#pragma unroll
			for (int j = 0; j < kMaxAlign; j++) pos[j] = 0;
			if (draw_sample<32>(task_seed, h, c.n, n_align, c.xy, c.image, ctie, 0xffffffffu, lane, pos, quat)) {
				float pose_lm[7], pose_refit[7], err2[2];
				const int cnt = lmx::hypothesis<V, 32>(team, c, pos, n_align, quat, max_lm, thr, min_npts, my, my_mask, finite_check != 0, pose_lm,
				                                       pose_refit, err2);
				if (cnt > min_npts) {
					atomicMin(&s_first, h);                          // every lane of the warp; idempotent
					if (lane == 0) for (int j = 0; j < 7; j++) s_pose[w][j] = pose_refit[j];
				}
			} else if (lane == 0) s_fail = 1;                        // randSample fails for every test of the task alike -> RANSAC returns false
		}
		__syncthreads();
		tests = min(base + kDepthWarps, max_ransac);
		if (s_first != kNoSuccess) { tests = s_first + 1; break; }
		if (s_fail) { tests = 0; break; }
		__syncthreads();
	}
	const int first = s_first;
	const bool ok = first != kNoSuccess;
	if (ok && w == first % kDepthWarps && lane == 0)
		for (int j = 0; j < 7; j++) pose_out[7 * task + j] = s_pose[w][j];
	if (threadIdx.x == 0) { found[task] = ok ? 1 : 0; n_tests[task] = tests; }
	}
}

// ---- device entries ----
static mc_status depth_scratch(mc_ctx *ctx, size_t warps, size_t slice, float **out) {
	const size_t bytes = warps * slice * sizeof(float);
	if (bytes > (size_t)8 << 30) { ctx->err = "pose (depth): cluster too large for the per-warp LM scratch"; return MC_ERR_ARG; }
	MC_TRY(reserve(ctx, ctx->scratch[kScrDepthLm], bytes));
	*out = (float *)ctx->scratch[kScrDepthLm].p;
	return MC_OK;
}

mc_status pose_depth_hypotheses_device(mc_ctx *ctx, int variant, const int32_t *d_cluster_offsets, const float *d_xy, const float *d_xyz,
                                       const float *d_world, const float *d_cauchy, const int32_t *d_image, const int32_t *d_hyp_cluster,
                                       const int32_t *d_sample_pos, const float *d_init_quat, int n_hyp, int n_max, const mc_pose_params *pp,
                                       float alpha, const int64_t *d_mask_offsets, int32_t *d_n_inliers, float *d_pose_lm, float *d_pose_refit,
                                       float *d_lm_err, uint8_t *d_mask) {
	if (!ctx->d_cams) { ctx->err = "pose (depth): cameras not set (mc_set_cameras)"; return MC_ERR_STATE; }
	if (variant < 0 || variant > 2) { ctx->err = "pose (exact order): variant must be 0 (back-projection + depth), 1 (reprojection + depth) or 2 (moped2 reprojection)"; return MC_ERR_ARG; }
	if (variant != 2 && (!d_world || !d_cauchy)) { ctx->err = "pose (depth): world3D and Cauchy weights are required"; return MC_ERR_ARG; }
	if (pp->n_pts_align < 1 || pp->n_pts_align > kMaxAlign) { ctx->err = "pose (depth): n_pts_align must be in 1..8"; return MC_ERR_ARG; }
	if (n_hyp <= 0) return MC_OK;
	const int R = variant == 1 ? 3 : 2;
	const size_t slice = depth_slice_floats(n_max, R);
	// persistent grid: exactly the CTAs that are resident at once (a CTA that had to wait for a slot would start its strided share late)
	const int W = ctx->depth_team_lanes == 8 ? 8 : 32, teams_per_cta = kDepthWarps * (32 / W);
	int grid = (n_hyp + teams_per_cta - 1) / teams_per_cta;
	int per_sm = 0;
	const void *fn = W == 32 ? (variant == 0 ? (const void *)k_depth_hypotheses<0, 32> : variant == 1 ? (const void *)k_depth_hypotheses<1, 32> : (const void *)k_depth_hypotheses<2, 32>)
	                         : (variant == 0 ? (const void *)k_depth_hypotheses<0, 8> : variant == 1 ? (const void *)k_depth_hypotheses<1, 8> : (const void *)k_depth_hypotheses<2, 8>);
	MC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, 32 * kDepthWarps, 0));
	const int cap = ctx->num_sms * (per_sm > 0 ? per_sm : 1);
	if (grid > cap) grid = cap;
	while (grid > 1 && (size_t)grid * teams_per_cta * slice * sizeof(float) > ((size_t)1 << 30)) grid = (grid + 1) / 2;
	float *scratch = nullptr;
	MC_TRY(depth_scratch(ctx, (size_t)grid * teams_per_cta, slice, &scratch));
#define MC_DEPTH_HYP(V, TW)                                                                                                                     \
	k_depth_hypotheses<V, TW><<<grid, 32 * kDepthWarps, 0, ctx->stream>>>(d_cluster_offsets, d_xy, d_xyz, d_world, d_cauchy, d_image, ctx->d_cams, alpha, \
	                                                                 d_hyp_cluster, d_sample_pos, d_init_quat, n_hyp, pp->n_pts_align,         \
	                                                                 pp->max_lm_tests, pp->error_threshold, pp->min_npts_object,               \
	                                                                 ctx->lm_finite_check ? 1 : 0, scratch, slice, n_max, d_mask_offsets,      \
	                                                                 d_n_inliers, d_pose_lm, d_pose_refit, d_lm_err, d_mask)
	if (W == 32) { if (variant == 0) MC_DEPTH_HYP(0, 32); else if (variant == 1) MC_DEPTH_HYP(1, 32); else MC_DEPTH_HYP(2, 32); }
	else { if (variant == 0) MC_DEPTH_HYP(0, 8); else if (variant == 1) MC_DEPTH_HYP(1, 8); else MC_DEPTH_HYP(2, 8); }
#undef MC_DEPTH_HYP
	MC_LAUNCH_CHECK();
	return MC_OK;
}

// d_n_clusters (nullable): the cluster count on the device (the moped3d frame chain); n_clusters and n_max are then upper bounds
// that size the grid and the LM scratch
mc_status pose_depth_ransac_device(mc_ctx *ctx, int variant, const int32_t *d_cluster_offsets, int n_clusters, int n_max, const float *d_xy,
                                   const float *d_xyz, const float *d_world, const float *d_cauchy, const int32_t *d_image, const int32_t *d_tie,
                                   const mc_pose_params *pp, float alpha, uint8_t *d_found, float *d_pose, int32_t *d_n_tests,
                                   const int32_t *d_n_clusters) {
	if (!ctx->d_cams) { ctx->err = "pose (depth): cameras not set (mc_set_cameras)"; return MC_ERR_STATE; }
	if (variant < 0 || variant > 2) { ctx->err = "pose (exact order): variant must be 0 (back-projection + depth), 1 (reprojection + depth) or 2 (moped2 reprojection)"; return MC_ERR_ARG; }
	if (variant != 2 && (!d_world || !d_cauchy)) { ctx->err = "pose (depth): world3D and Cauchy weights are required"; return MC_ERR_ARG; }
	if (pp->n_pts_align < 1 || pp->n_pts_align > kMaxAlign) { ctx->err = "pose (depth): n_pts_align must be in 1..8"; return MC_ERR_ARG; }
	const int n_tasks = n_clusters * pp->max_objects_per_cluster;
	if (n_tasks <= 0) return MC_OK;
	const int R = variant == 1 ? 3 : 2;
	const size_t slice = depth_slice_floats(n_max, R);
	int per_sm = 0;
	if (d_n_clusters && variant == 2) { ctx->err = "pose (exact order): no device cluster count for variant 2"; return MC_ERR_ARG; }
	const void *fn = d_n_clusters ? (variant == 0 ? (const void *)k_depth_ransac<0, true> : (const void *)k_depth_ransac<1, true>)
	                              : (variant == 0 ? (const void *)k_depth_ransac<0, false> : variant == 1 ? (const void *)k_depth_ransac<1, false>
	                                                                                                   : (const void *)k_depth_ransac<2, false>);
	MC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, 32 * kDepthWarps, 0));
	int grid = ctx->num_sms * (per_sm > 0 ? per_sm : 1);
	if (grid > n_tasks) grid = n_tasks;
	while (grid > 1 && (size_t)grid * kDepthWarps * slice * sizeof(float) > ((size_t)1 << 30)) grid = (grid + 1) / 2;
	float *scratch = nullptr;
	MC_TRY(depth_scratch(ctx, (size_t)grid * kDepthWarps, slice, &scratch));
#define MC_DEPTH_RANSAC(V, DC)                                                                                                                  \
	k_depth_ransac<V, DC><<<grid, 32 * kDepthWarps, 0, ctx->stream>>>(d_cluster_offsets, n_clusters, d_n_clusters, d_xy, d_xyz, d_world, d_cauchy, d_image, d_tie, \
	                                                                ctx->d_cams, alpha, pp->max_objects_per_cluster, pp->max_ransac_tests,     \
	                                                                pp->max_lm_tests, pp->n_pts_align, pp->min_npts_object, pp->error_threshold, \
	                                                                pp->seed, ctx->lm_finite_check ? 1 : 0, scratch, slice, n_max, n_tasks,    \
	                                                                d_found, d_pose, d_n_tests)
	if (d_n_clusters) { if (variant == 0) MC_DEPTH_RANSAC(0, true); else MC_DEPTH_RANSAC(1, true); }
	else if (variant == 0) MC_DEPTH_RANSAC(0, false); else if (variant == 1) MC_DEPTH_RANSAC(1, false); else MC_DEPTH_RANSAC(2, false);
#undef MC_DEPTH_RANSAC
	MC_LAUNCH_CHECK();
	return MC_OK;
}

} // namespace mc
