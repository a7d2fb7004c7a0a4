// pose_staged.cuh — the staged RANSAC driver of the POSE / POSE2 steps (RANSAC(), POSE_RANSAC_LM_DIFF_REPROJECTION_CPU.hpp:188-211),
// templated on a FIT POLICY so that two translation units instantiate the same kernels with different arithmetic:
//   pose.cu        DefaultFit — lane-group LM with butterfly sums and fused multiply-add (meets the oracle statistically)
//   pose_exact.cu  ExactFit   — the order-preserving LM of lm_exact.cuh, compiled with -fmad=false: the strict-IEEE build of the
//                               reference bit for bit (same winning test, same refitted pose)
// A policy provides
//   kFitSmemFloats        shared-memory floats an 8-lane group needs for a sample fit (0 = none)
//   kRefitListInts        shared-memory ints a warp needs for its refit (inlier list; 1 = none)
//   kRefitFloatsPerPoint, kRefitFloatsPerTask   global scratch of a task's refit = PerPoint * cluster size + PerTask (0 = none)
//   fit(...)              sample fit + inlier count of one hypothesis by the calling lane's 8-lane group -> count or -1
//   refit(...)            refit of a successful hypothesis on its inliers by the calling warp
#pragma once
#include "common.cuh"
#include "ransac_sample.cuh"

namespace mc {

constexpr int kPoseThreads = 256;

// ---- staged RANSAC ----
// Same result as k_pose_ransac (the first successful hypothesis in hypothesis order, refitted), organised for lane
// utilisation and occupancy instead of one CTA per task:
//   k_ransac_init   per-task state
//   k_ransac_first  hypotheses 0..HA-1 of EVERY task, one per 8-lane group, groups of different tasks packed four to a
//                   warp (on real clusters hypothesis 0 succeeds, and one-hypothesis-per-warp left 3/4 of the lanes idle:
//                   ncu showed 9.2 active threads per instruction over 76 % of the old kernel's instructions)
//   k_ransac_level  tasks with no success yet (queue built by k_ransac_first) test further hypotheses in escalating
//                   levels, each one launch of a persistent grid over (task, chunk) work items:
//                     level 1: the next 4 hypotheses, one warp per task (a fit succeeds with probability ~1/2 on a real
//                              cluster, so almost every task ends here);
//                     level 2: the next 32, one CTA of 8 warps per task;
//                     (default since round 2, "ransac_merge_levels": levels 1 and 2 as ONE launch over the next 36 — the batch of a
//                      step always holds some task that escalates, and every escalation step is one LM chain latency for the batch)
//                     level 3: ALL remaining ones at once, 32 per item, chunk-major. A cluster that fails all
//                              MaxRANSACTests tests occupies the machine for about one LM latency instead of one SM for
//                              MaxRANSACTests/32 of them. (Running level 3 straight after the first kernel was measured:
//                              the speculative chunks cost more than the tasks they saved, 15.8 vs 8.8 ms per 64 frames.)
//                   An item above an already successful index is skipped, a running fit above one aborts.
//   k_ransac_refit  one warp per successful task: inlier refit (optimizeCamera on `consistent`, :204-208), outputs
constexpr int kNone = 0x7f7f7f7f;      // "no successful hypothesis"
constexpr int kLevels = 3;

struct RansacLevels {                  // hypothesis ranges of the levels after the first kernel
	int h_begin[kLevels + 1];          // level l tests [h_begin[l], h_begin[l+1])
	int hpi[kLevels];                  // hypotheses per work item (4 x warps of the CTA)
	int slot_base[kLevels];            // first chunk_pose slot of the level
	int slots;                         // chunk_pose slots per queued task
};

struct RansacState {
	int32_t *first;       // [tasks] lowest successful hypothesis index or kNone
	int32_t *done;        // [tasks] finished first-round hypotheses
	int32_t *qpos;        // [tasks] position in the queue or -1
	int32_t *queue;       // [tasks]
	int32_t *counters;    // [0] queue length
	uint8_t *fail;        // [tasks] randSample failed (fewer than NPtsAlign distinct points)
	float *fit_pose;      // [tasks][HA][7] sample-fit pose of successful first-round hypotheses
	float *chunk_pose;    // [queue pos][slots][7] sample-fit pose of each work item's lowest success
	float *refit_scratch; // policy-defined global scratch of the refit kernel (nullptr = none), carved per task
	int shard_rank, shard_world;   // RANSAC tasks partitioned by cluster (north_star: "RANSAC work is distributed by cluster"): this call runs the
	                               // tasks of clusters c with c % shard_world == shard_rank and reports found = 0 for the others
};

__device__ __forceinline__ bool ransac_owns(const RansacState &S, int c) { return S.shard_world <= 1 || c % S.shard_world == S.shard_rank; }

// offset of task t's slice inside RansacState::refit_scratch: tasks of cluster c (points [lo, lo + n)) lie back to back
template <class P>
__device__ __forceinline__ size_t refit_slice_offset(int task, int c, int lo, int n, int max_obj) {
	return ((size_t)P::kRefitFloatsPerPoint * lo + (size_t)P::kRefitFloatsPerTask * c) * max_obj +
	       (size_t)(task - c * max_obj) * ((size_t)P::kRefitFloatsPerPoint * n + P::kRefitFloatsPerTask);
}

static __global__ void k_ransac_init(RansacState S, int n_tasks) {
	const int t = blockIdx.x * blockDim.x + threadIdx.x;
	if (t == 0) S.counters[0] = 0;
	if (t >= n_tasks) return;
	S.first[t] = kNone; S.done[t] = 0; S.qpos[t] = -1; S.fail[t] = 0;
}

template <class P>
__global__ void __launch_bounds__(128)
k_ransac_first(const int32_t *__restrict__ cluster_offsets, const int32_t *__restrict__ n_clusters_p, int n_clusters_cap,
               const float *__restrict__ xy, const float *__restrict__ xyz, const int32_t *__restrict__ image,
               const int32_t *__restrict__ tie, const Camera *__restrict__ cams, int max_obj, int max_ransac, int max_lm, int n_align,
               int min_npts, float thr, uint64_t seed, int HA, RansacState S) {
	__shared__ float s_fit[P::kFitSmemFloats > 0 ? 16 * P::kFitSmemFloats : 1];
	const int lane = threadIdx.x & 31, lig = lane & 7, grp = lane >> 3;
	const unsigned mask = 0xFFu << (8 * grp);
	const int n_clusters = n_clusters_p ? min(*n_clusters_p, n_clusters_cap) : n_clusters_cap;
	// the grid may be smaller than the task bound (a lane of a frame batch: the clusters that exist are the first few tasks): groups
	// are walked with the grid's stride, the ones beyond the clusters that exist cost one comparison
	const int64_t n_groups = (int64_t)n_clusters * max_obj * HA;
	for (int64_t g64 = (int64_t)(blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * 4 + grp; g64 < n_groups; g64 += (int64_t)gridDim.x * (blockDim.x >> 5) * 4) {
	const int g = (int)g64;
	const int task = g / HA, h = g - task * HA;
	const int c = task / max_obj;
	if (c >= n_clusters || h >= max_ransac || !ransac_owns(S, c)) continue;
	const int lo = cluster_offsets[c], n = cluster_offsets[c + 1] - lo;
	const float *cxy = xy + 2 * lo, *cxyz = xyz + 3 * lo;
	const int32_t *cim = image + lo, *ctie = tie ? tie + lo : nullptr;
	const uint64_t task_seed = seed + 0x9E3779B97F4A7C15ULL * (uint64_t)(task + 1);
	int cnt = -1;
	float pose[7] = { 0, 0, 0, 1, 0, 0, 0 }, err;
	int pos[kMaxAlign]; float quat[4];
#pragma unroll
	for (int j = 0; j < kMaxAlign; j++) pos[j] = 0;
	bool sample_ok = draw_sample<8>(task_seed, h, n, n_align, cxy, cim, ctie, mask, lig, pos, quat);
	if (sample_ok)
		cnt = P::fit(pos, n_align, quat, n, cxy, cxyz, cim, cams, max_lm, thr, mask, lig, pose, err,
		             HA > 1 ? (const volatile int *)&S.first[task] : nullptr, h, s_fit + (threadIdx.x >> 3) * P::kFitSmemFloats);
	if (lig == 0) {
		if (!sample_ok) S.fail[task] = 1;          // fails for every hypothesis of the task alike -> RANSAC returns false
		if (cnt > min_npts) {
			float *dst = S.fit_pose + ((size_t)task * HA + h) * 7;
#pragma unroll
			for (int j = 0; j < 7; j++) dst[j] = pose[j];
			__threadfence();
			atomicMin(&S.first[task], h);
		}
		__threadfence();
		const int n_first = HA < max_ransac ? HA : max_ransac;
		if (atomicAdd(&S.done[task], 1) + 1 == n_first) {
			// last first-round hypothesis of the task: queue it for the remaining tests if nothing succeeded
			const int f = atomicMin(&S.first[task], kNone);
			if (f == kNone && sample_ok && max_ransac > HA) {
				const int q = atomicAdd(&S.counters[0], 1);
				S.queue[q] = task; S.qpos[task] = q;
			}
		}
	}
	}
}

template <class P>
__global__ void __launch_bounds__(kPoseThreads)
k_ransac_level(const int32_t *__restrict__ cluster_offsets, const float *__restrict__ xy, const float *__restrict__ xyz,
               const int32_t *__restrict__ image, const int32_t *__restrict__ tie, const Camera *__restrict__ cams, int max_obj,
               int max_ransac, int max_lm, int n_align, int min_npts, float thr, uint64_t seed, int h_begin, int h_end, int slot_base,
               int slots, RansacState S) {
	__shared__ float s_pose[kPoseThreads / 8][7];
	__shared__ float s_fit[P::kFitSmemFloats > 0 ? (kPoseThreads / 8) * P::kFitSmemFloats : 1];
	__shared__ int s_first, s_skip;
	const int hpi = (blockDim.x >> 5) * 4;                                  // hypotheses per item
	const int n_chunks = (h_end - h_begin + hpi - 1) / hpi;
	const int nq = S.counters[0];
	const int64_t items = (int64_t)nq * n_chunks;
	const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, lig = lane & 7, grp = lane >> 3;
	const unsigned mask = 0xFFu << (8 * grp);
	for (int64_t item = blockIdx.x; item < items; item += gridDim.x) {
		const int chunk = (int)(item / nq), qi = (int)(item - (int64_t)chunk * nq);
		const int task = S.queue[qi];
		const int h0 = h_begin + chunk * hpi;
		if (threadIdx.x == 0) {
			s_first = kNone;
			s_skip = *(const volatile int *)&S.first[task] < h0;      // a lower index already succeeded: nothing here can win
		}
		__syncthreads();
		if (!s_skip) {
			const int c = task / max_obj;
			const int lo = cluster_offsets[c], n = cluster_offsets[c + 1] - lo;
			const float *cxy = xy + 2 * lo, *cxyz = xyz + 3 * lo;
			const int32_t *cim = image + lo, *ctie = tie ? tie + lo : nullptr;
			const uint64_t task_seed = seed + 0x9E3779B97F4A7C15ULL * (uint64_t)(task + 1);
			const int slot = w * 4 + grp, h = h0 + slot;
			if (h < h_end) {
				int cnt = -1;
				float pose[7] = { 0, 0, 0, 1, 0, 0, 0 }, err;
				int pos[kMaxAlign]; float quat[4];
#pragma unroll
				for (int j = 0; j < kMaxAlign; j++) pos[j] = 0;
				if (draw_sample<8>(task_seed, h, n, n_align, cxy, cim, ctie, mask, lig, pos, quat))
					cnt = P::fit(pos, n_align, quat, n, cxy, cxyz, cim, cams, max_lm, thr, mask, lig, pose, err,
					             (const volatile int *)&S.first[task], h, s_fit + (threadIdx.x >> 3) * P::kFitSmemFloats);
				if (lig == 0 && cnt > min_npts) {
#pragma unroll
					for (int j = 0; j < 7; j++) s_pose[slot][j] = pose[j];
					atomicMin(&s_first, h);
					atomicMin(&S.first[task], h);          // lets higher indices everywhere abort
				}
			}
		}
		__syncthreads();
		if (!s_skip && s_first != kNone && threadIdx.x < 7)
			S.chunk_pose[((size_t)qi * slots + slot_base + chunk) * 7 + threadIdx.x] = s_pose[s_first - h0][threadIdx.x];
		__syncthreads();
	}
}

template <class P>
__global__ void __launch_bounds__(128)
k_ransac_refit(const int32_t *__restrict__ cluster_offsets, const int32_t *__restrict__ n_clusters_p, int n_clusters_cap,
               const float *__restrict__ xy, const float *__restrict__ xyz, const int32_t *__restrict__ image,
               const Camera *__restrict__ cams, int max_obj, int max_ransac, int max_lm, float thr, int HA, RansacLevels L, RansacState S,
               int n_tasks, uint8_t *__restrict__ found, float *__restrict__ pose_out, int32_t *__restrict__ n_tests) {
	__shared__ int s_list[4][P::kRefitListInts];
	const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
	const int n_clusters = n_clusters_p ? min(*n_clusters_p, n_clusters_cap) : n_clusters_cap;
	for (int task = blockIdx.x * 4 + w; task < n_tasks; task += gridDim.x * 4) {       // (bounded grid on the lanes of a frame batch)
	const int c = task / max_obj;
	if (c >= n_clusters || !ransac_owns(S, c)) { if (lane == 0) { found[task] = 0; n_tests[task] = 0; } continue; }
	const int f = S.first[task];
	if (f == kNone) {
		if (lane == 0) { found[task] = 0; n_tests[task] = S.fail[task] ? 0 : max_ransac; }
		continue;
	}
	const float *src = S.fit_pose + ((size_t)task * HA + f) * 7;
	if (f >= HA) {
		int l = 0;
#pragma unroll
		for (int k = 1; k < kLevels; k++) if (f >= L.h_begin[k]) l = k;
		src = S.chunk_pose + ((size_t)S.qpos[task] * L.slots + L.slot_base[l] + (f - L.h_begin[l]) / L.hpi[l]) * 7;
	}
	float pose[7], err;
#pragma unroll
	for (int j = 0; j < 7; j++) pose[j] = src[j];
	const int lo = cluster_offsets[c], n = cluster_offsets[c + 1] - lo;
	P::refit(pose, n, xy + 2 * lo, xyz + 3 * lo, image + lo, cams, thr, max_lm, lane, s_list[w],
	         S.refit_scratch ? S.refit_scratch + refit_slice_offset<P>(task, c, lo, n, max_obj) : nullptr, err);
	if (lane == 0) {
#pragma unroll
		for (int j = 0; j < 7; j++) pose_out[7 * task + j] = pose[j];
		found[task] = 1; n_tests[task] = f + 1;
	}
	__syncwarp();
	}
}

// Host side: plan the levels, carve the state, launch init / first / levels / refit on ctx->stream.
// HA = hypotheses of every task tested by the first kernel (mc_set_tuning's pose_warps_per_task: 1 packs four tasks into a warp
// and wastes nothing when hypothesis 0 succeeds; more trade work for the latency of tasks whose first hypothesis fails).
// n_points_cap = upper bound of the number of cluster points (sizes the policy's refit scratch).
template <class P>
mc_status ransac_staged_launch(mc_ctx *ctx, const int32_t *d_cluster_offsets, const int32_t *d_n_clusters, int n_clusters_cap, int n_points_cap,
                               const float *d_xy, const float *d_xyz, const int32_t *d_image, const int32_t *d_tie, const mc_pose_params *pp,
                               uint8_t *d_found, float *d_pose, int32_t *d_n_tests) {
	const int n_tasks = n_clusters_cap * pp->max_objects_per_cluster;
	const int warps = ctx->pose_warps < 1 ? 1 : (ctx->pose_warps > kPoseThreads / 32 ? kPoseThreads / 32 : ctx->pose_warps);
	const int R = pp->max_ransac_tests;
	const int HA = warps < R ? warps : (R > 0 ? R : 1);
	RansacLevels L;
	// mc_set_option "ransac_merge_levels": levels 1 and 2 as ONE launch of 8-warp CTAs over the next 36 hypotheses (a task whose first
	// hypotheses fail then costs one more LM chain latency instead of two; more speculative work)
	const int level_warps[kLevels] = { ctx->ransac_merge_levels ? 8 : 1, 8, 8 };
	const int level_span[kLevels] = { ctx->ransac_merge_levels ? 36 : 4, ctx->ransac_merge_levels ? 0 : 32, 1 << 30 };
	L.h_begin[0] = HA < R ? HA : R;
	L.slots = 0;
	for (int l = 0; l < kLevels; l++) {
		L.hpi[l] = 4 * level_warps[l];
		const int64_t e = (int64_t)L.h_begin[l] + level_span[l];
		L.h_begin[l + 1] = (int)(e < R ? e : R);
		L.slot_base[l] = L.slots;
		L.slots += (L.h_begin[l + 1] - L.h_begin[l] + L.hpi[l] - 1) / L.hpi[l];
	}
	const size_t refit_floats = ((size_t)P::kRefitFloatsPerPoint * n_points_cap + (size_t)P::kRefitFloatsPerTask * n_clusters_cap) * pp->max_objects_per_cluster;
	const size_t nt = (size_t)n_tasks;
	RansacState S;
	MC_TRY(carve_scratch(ctx, ctx->scratch[kScrRansac], [&](Carve &c) {
		c.take(S.first, nt); c.take(S.done, nt); c.take(S.qpos, nt); c.take(S.queue, nt); c.take(S.counters, 16); c.take(S.fail, nt);
		c.take(S.fit_pose, 7 * nt * HA); c.take(S.chunk_pose, 7 * nt * (L.slots > 0 ? L.slots : 1)); c.take(S.refit_scratch, refit_floats);
	}));
	if (!refit_floats) S.refit_scratch = nullptr;
	S.shard_rank = ctx->ransac_shard_rank; S.shard_world = ctx->ransac_shard_world;
	k_ransac_init<<<(n_tasks + 255) / 256, 256, 0, ctx->stream>>>(S, n_tasks);
	MC_LAUNCH_CHECK();
	const int64_t groups = (int64_t)n_tasks * HA;
	// lanes of a frame batch: at most half an SM count of CTAs per launch (1184 groups / 296 refits at a time; the rest by the grid stride) —
	// the bounds cl_cap x max_obj are hundreds of times the clusters a frame has, and 64 frames' worth of such grids queue behind each other
	const int64_t first_ctas = (groups + 15) / 16, refit_ctas = ((int64_t)n_tasks + 3) / 4, lane_cap = ctx->num_sms / 2;
	k_ransac_first<P><<<(unsigned)(ctx->parent && first_ctas > lane_cap ? lane_cap : first_ctas), 128, 0, ctx->stream>>>(d_cluster_offsets, d_n_clusters, n_clusters_cap, d_xy, d_xyz, d_image, d_tie,
	                                                                          ctx->d_cams, pp->max_objects_per_cluster, R, pp->max_lm_tests,
	                                                                          pp->n_pts_align, pp->min_npts_object, pp->error_threshold, pp->seed, HA, S);
	MC_LAUNCH_CHECK();
	for (int l = 0; l < kLevels; l++) {
		if (L.h_begin[l + 1] <= L.h_begin[l]) continue;
		// persistent grids: queue length and success state are only known on the device; CTAs without items exit at once
		// a lane of a frame batch (ctx->parent) shares the GPU with up to 63 other frames: small grids there (a frame queues a handful of
		// tasks; the CTAs loop over the items whatever their number) — the thousands of CTAs that found an empty queue were a third of
		// all CTA launches of a batch
		const int grid = ctx->parent ? (level_warps[l] == 1 ? 64 : 37) : (level_warps[l] == 1 ? ctx->num_sms * 8 : ctx->num_sms);
		k_ransac_level<P><<<grid, 32 * level_warps[l], 0, ctx->stream>>>(d_cluster_offsets, d_xy, d_xyz, d_image, d_tie, ctx->d_cams, pp->max_objects_per_cluster,
		                                                                R, pp->max_lm_tests, pp->n_pts_align, pp->min_npts_object, pp->error_threshold, pp->seed,
		                                                                L.h_begin[l], L.h_begin[l + 1], L.slot_base[l], L.slots, S);
		MC_LAUNCH_CHECK();
	}
	k_ransac_refit<P><<<(unsigned)(ctx->parent && refit_ctas > lane_cap ? lane_cap : refit_ctas), 128, 0, ctx->stream>>>(d_cluster_offsets, d_n_clusters, n_clusters_cap, d_xy, d_xyz, d_image, ctx->d_cams,
	                                                             pp->max_objects_per_cluster, R, pp->max_lm_tests, pp->error_threshold, HA,
	                                                             L, S, n_tasks, d_found, d_pose, d_n_tests);
	MC_LAUNCH_CHECK();
	return MC_OK;
}

} // namespace mc
