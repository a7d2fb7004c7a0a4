// filter.cu — FILTER / FILTER2 steps: projection scoring, feature ownership, pruning, cluster rebuild.
//
// Replaces FILTER_PROJECTION_CPU::process (moped2/libmoped/src/filter/FILTER_PROJECTION_CPU.hpp:80-162).
//   k_filter_score   one thread per object: reproject every match of its model (project(), moped.hpp:330-354),
//                    in-cluster flag per (object, match), score = sum 1/(err+1) in match order (:95-115)
//   k_filter_own     one thread per match: best (score, visit order) over the objects whose cluster holds a
//                    match with the same (coord2D, image) key — `bestPoints` (:117-129)
//   k_filter_compact one CTA: owned matches of every object's own model, keep/prune (:135-160), then the survivors' clusters in
//                    reference order (model-major, list order)
// moped3d's FILTER_PROJECTION_DEPTH_CPU (moped3d/libmoped/src/filter/FILTER_PROJECTION_DEPTH_CPU.hpp:145-329) is the same filter with a
// penalty from the depth map subtracted from the score before pruning (k_filter_depth_adjust); ownership keeps the unpenalised score.
#include "common.cuh"

#include <math_constants.h>
#include <float.h>

namespace mc {

// TransformMatrix::init (moped.hpp:175-182), each term rounded on its own in source order
__device__ __forceinline__ float tm_diag(float a, float b) {      // 1 - 2 a a - 2 b b
	return __fsub_rn(__fsub_rn(1.f, __fmul_rn(__fmul_rn(2.f, a), a)), __fmul_rn(__fmul_rn(2.f, b), b));
}
__device__ __forceinline__ float tm_off(float a, float b, float c, float d, float sign) {      // 2 a b +- 2 c d
	const float l = __fmul_rn(__fmul_rn(2.f, a), b), r = __fmul_rn(__fmul_rn(2.f, c), d);
	return sign > 0.f ? __fadd_rn(l, r) : __fsub_rn(l, r);
}
__device__ __forceinline__ void pose_matrix(const float *q, const float *t, float *T) {
	T[0] = tm_diag(q[1], q[2]); T[1] = tm_off(q[0], q[1], q[3], q[2], -1.f); T[2] = tm_off(q[0], q[2], q[3], q[1], 1.f); T[3] = t[0];
	T[4] = tm_off(q[0], q[1], q[3], q[2], 1.f); T[5] = tm_diag(q[0], q[2]); T[6] = tm_off(q[1], q[2], q[3], q[0], -1.f); T[7] = t[1];
	T[8] = tm_off(q[0], q[2], q[3], q[1], -1.f); T[9] = tm_off(q[1], q[2], q[3], q[0], 1.f); T[10] = tm_diag(q[0], q[1]); T[11] = t[2];
}

// squared reprojection error of model point X under pose matrix T into camera cam vs observed (u0, v0). Every product and sum is
// rounded on its own, left to right (explicit _rn intrinsics: no fused multiply-add whatever the compiler flags), the order of
// TransformMatrix::transform / inverseTransform and project() (moped.hpp:183-200,330-354) as the oracle restates them.
__device__ __forceinline__ float dot3_rn(float a0, float b0, float a1, float b1, float a2, float b2) {
	return __fadd_rn(__fadd_rn(__fmul_rn(a0, b0), __fmul_rn(a1, b1)), __fmul_rn(a2, b2));
}
__device__ __forceinline__ float reproj_err(const float *T, const Camera &cam, const float *X, float u0, float v0) {
	const float x = __fadd_rn(dot3_rn(X[0], T[0], X[1], T[1], X[2], T[2]), T[3]);
	const float y = __fadd_rn(dot3_rn(X[0], T[4], X[1], T[5], X[2], T[6]), T[7]);
	const float z = __fadd_rn(dot3_rn(X[0], T[8], X[1], T[9], X[2], T[10]), T[11]);
	const float a = __fsub_rn(x, cam.TM[3]), b = __fsub_rn(y, cam.TM[7]), c = __fsub_rn(z, cam.TM[11]);
	const float cx = dot3_rn(a, cam.TM[0], b, cam.TM[4], c, cam.TM[8]);
	const float cy = dot3_rn(a, cam.TM[1], b, cam.TM[5], c, cam.TM[9]);
	const float cz = dot3_rn(a, cam.TM[2], b, cam.TM[6], c, cam.TM[10]);
	float u = FLT_MAX, v = FLT_MAX;
	if (!((double)cz < 0.001)) {
		u = __fadd_rn(__fmul_rn(__fdiv_rn(cx, cz), cam.K[0]), cam.K[2]);
		v = __fadd_rn(__fmul_rn(__fdiv_rn(cy, cz), cam.K[1]), cam.K[3]);
	}
	const float du = __fsub_rn(u, u0), dv = __fsub_rn(v, v0);
	return __fadd_rn(__fmul_rn(du, du), __fmul_rn(dv, dv));
}

// in_cluster: n_objects x max_per_model bytes, row o covers the matches of model(o) (index j - lo).
// One WARP per object: the reprojections run 32 at a time, then lane 0 adds the terms in match order
// (`score += 1./(err+1.)` is a sequential fp32 <- double accumulation in the reference, :106).
__global__ void k_filter_score(const int32_t *__restrict__ match_offsets, const int32_t *__restrict__ match_image,
                               const float *__restrict__ match_xy, const float *__restrict__ match_xyz, const Camera *__restrict__ cams,
                               const int32_t *__restrict__ obj_model, const float *__restrict__ obj_pose, const int32_t *__restrict__ n_obj_p,
                               int n_obj_cap, float feat_dist, int stride, uint8_t *__restrict__ in_cluster, float *__restrict__ score) {
	const int lane = threadIdx.x & 31;
	const int n_obj = n_obj_p ? min(*n_obj_p, n_obj_cap) : n_obj_cap;
	for (int o = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; o < n_obj; o += (gridDim.x * blockDim.x) >> 5) {      // bounded grid, see k_filter_own
	const int m = obj_model[o];
	const int lo = match_offsets[m], hi = match_offsets[m + 1];
	float T[12];
	pose_matrix(obj_pose + 7 * o, obj_pose + 7 * o + 4, T);
	float s = 0.f;
	for (int j0 = lo; j0 < hi; j0 += 32) {
		const int j = j0 + lane;
		float err = CUDART_INF_F;
		if (j < hi) err = reproj_err(T, cams[match_image[j]], match_xyz + 3 * j, match_xy[2 * j], match_xy[2 * j + 1]);
		const bool in = j < hi && err < feat_dist;
		if (j < hi) in_cluster[(size_t)o * stride + (j - lo)] = in ? 1 : 0;
		unsigned msk = __ballot_sync(0xffffffffu, in);
		while (msk) {                                       // in-cluster terms in ascending match order
			const int l = __ffs(msk) - 1;
			msk &= msk - 1;
			const float e = __shfl_sync(0xffffffffu, err, l);
			s = __double2float_rn(__dadd_rn((double)s, __ddiv_rn(1., __dadd_rn((double)e, 1.))));
		}
	}
	if (lane == 0) score[o] = s;
	}
}

// model whose match range holds match j (match_offsets ascending, empty models allowed): the last m with match_offsets[m] <= j
__device__ __forceinline__ int model_of_match(const int32_t *__restrict__ match_offsets, int n_models, int j) {
	int lo = 0, hi = n_models - 1;
	while (lo < hi) {
		const int mid = (lo + hi + 1) >> 1;
		if (match_offsets[mid] <= j) lo = mid; else hi = mid - 1;
	}
	return lo;
}

__device__ __forceinline__ bool better(float s, int m, int o, float bs, int bm, int bo) {
	// strictly higher score wins; on equal score the object visited first (model-major, then list order)
	if (s != bs) return s > bs;
	if (m != bm) return m < bm;
	return o < bo;
}

// owner[j] = object owning match j's (coord2D, image) key, or -1. One CTA per match: the threads scan all
// matches for the same key (usually only j itself), candidates are reduced by (score desc, visit order asc).
__global__ void k_filter_own(const int32_t *__restrict__ match_offsets, int n_models, const int32_t *__restrict__ match_image,
                             const float *__restrict__ match_xy,
                             const int32_t *__restrict__ obj_model, const int32_t *__restrict__ n_obj_p, int n_obj_cap, int stride,
                             const uint8_t *__restrict__ in_cluster, const float *__restrict__ score, int32_t *__restrict__ owner) {
	__shared__ float s_bs[4]; __shared__ int s_bm[4], s_bo[4];
	const int M = match_offsets[n_models];
	const int n_obj = n_obj_p ? min(*n_obj_p, n_obj_cap) : n_obj_cap;
	// a bounded grid walks the matches: a frame has a few hundred of them while the launch bound is the feature count, and a batch of
	// 64 frames would otherwise start 260 000 CTAs that exit at once (CTA launch rate, not work, bounded the stages of a batch)
	for (int j = blockIdx.x; j < M; j += gridDim.x) {
	const float x = match_xy[2 * j], y = match_xy[2 * j + 1];
	const int im = match_image[j];
	float bs = 0.f; int bm = 0x7fffffff, bo = -1;
	for (int j2 = threadIdx.x; j2 < M; j2 += blockDim.x) {
		if (match_image[j2] != im || match_xy[2 * j2] != x || match_xy[2 * j2 + 1] != y) continue;
		const int m2 = model_of_match(match_offsets, n_models, j2);
		const int lo2 = match_offsets[m2];
		for (int o = 0; o < n_obj; o++) {
			if (obj_model[o] != m2 || !in_cluster[(size_t)o * stride + (j2 - lo2)]) continue;
			const float s = score[o];
			if (!(0.f < s)) continue;                  // `point.first < score` with point.first initially 0
			if (bo < 0 || better(s, m2, o, bs, bm, bo)) { bs = s; bm = m2; bo = o; }
		}
	}
	for (int off = 16; off; off >>= 1) {
		const float os = __shfl_xor_sync(0xffffffffu, bs, off);
		const int om = __shfl_xor_sync(0xffffffffu, bm, off), oo = __shfl_xor_sync(0xffffffffu, bo, off);
		if (oo >= 0 && (bo < 0 || better(os, om, oo, bs, bm, bo))) { bs = os; bm = om; bo = oo; }
	}
	const int w = threadIdx.x >> 5;
	if ((threadIdx.x & 31) == 0) { s_bs[w] = bs; s_bm[w] = bm; s_bo[w] = bo; }
	__syncthreads();
	if (threadIdx.x == 0) {
		for (int k = 1; k < (int)(blockDim.x >> 5); k++)
			if (s_bo[k] >= 0 && (bo < 0 || better(s_bs[k], s_bm[k], s_bo[k], bs, bm, bo))) { bs = s_bs[k]; bm = s_bm[k]; bo = s_bo[k]; }
		owner[j] = bo;
	}
	__syncthreads();
	}
}

// one CTA: survivors in (model, list order) -> cluster CSR; also the surviving object list in list order.
// out_n = {#survivors, #members}
__global__ void k_filter_compact(const int32_t *__restrict__ match_offsets, int n_models, const int32_t *__restrict__ obj_model,
                                 const float *__restrict__ obj_pose, const int32_t *__restrict__ n_obj_p, int n_obj_cap,
                                 const int32_t *__restrict__ owner, int32_t *__restrict__ owned, uint8_t *__restrict__ keep,
                                 const float *__restrict__ score, int min_points, float min_score,
                                 int32_t *__restrict__ out_n, int32_t *__restrict__ cluster_model, int32_t *__restrict__ cluster_offsets,
                                 int32_t *__restrict__ members, int32_t *__restrict__ surv_model, float *__restrict__ surv_pose,
                                 float *__restrict__ surv_score) {
	__shared__ int s_rank[1024];
	__shared__ int s_tot[2];
	const int n_obj = n_obj_p ? min(*n_obj_p, n_obj_cap) : n_obj_cap;
	const int tid = threadIdx.x;
	if (tid == 0) { s_tot[0] = 0; s_tot[1] = 0; }
	// per object: number of owned matches of its own model, keep flag (:135-160)
	for (int o = tid; o < n_obj; o += blockDim.x) {
		const int m = obj_model[o];
		int c = 0;
		for (int j = match_offsets[m]; j < match_offsets[m + 1]; j++) c += owner[j] == o;
		owned[o] = c;
		keep[o] = (c < min_points || score[o] < min_score) ? 0 : 1;
	}
	__syncthreads();
	// rank of every survivor in (model, list index) order and start of its members: O(n_obj^2), n_obj is small
	for (int o = tid; o < n_obj; o += blockDim.x) {
		if (!keep[o]) continue;
		int rank = 0, start = 0, list_rank = 0;
		for (int p = 0; p < n_obj; p++) {
			if (!keep[p]) continue;
			const bool before = obj_model[p] < obj_model[o] || (obj_model[p] == obj_model[o] && p < o);
			if (before) { rank++; start += owned[p]; }
			if (p < o) list_rank++;
		}
		cluster_model[rank] = obj_model[o];
		cluster_offsets[rank] = start;
		const int m = obj_model[o], lo = match_offsets[m];
		int t = start;
		for (int j = lo; j < match_offsets[m + 1]; j++)
			if (owner[j] == o) members[t++] = j - lo;
		surv_model[list_rank] = m;
		for (int k = 0; k < 7; k++) surv_pose[7 * list_rank + k] = obj_pose[7 * o + k];
		surv_score[list_rank] = score[o];
		atomicAdd(&s_tot[0], 1);
		atomicAdd(&s_tot[1], owned[o]);
	}
	__syncthreads();
	if (tid == 0) { cluster_offsets[s_tot[0]] = s_tot[1]; out_n[0] = s_tot[0]; out_n[1] = s_tot[1]; }
	(void)s_rank;
}

// ---- moped3d: the depth-map penalty of FILTER_PROJECTION_DEPTH_CPU (:197-270) ----
// One warp per object. (1) clusterSize = matches of its model within PlausibleSqDistance (:201-203). (2) the "incorrect score": every test
// point of the model is moved by the object's pose into the depth camera and projected (:222-231); points off the image or on a pixel
// whose depth was filled in (fill distance > 0) are skipped, the others count as usable; a usable point the depth map does not
// occlude adds 1 - 1/(1 + ((z - d) / (DepthFraction d))^2), accumulated in test-point order as float <- double like the reference
// (:259-263). (3) IS = 0 unless more than MinKeypointFraction of the points were usable, else IS *= clusterSize / usable; final score
// = score - IS (:268-280). The float -> int conversions of a NaN / out-of-range coordinate follow x86 (0x80000000: off the image).
struct DepthFilterArgs {
	const int32_t *test_offsets;      // [n_models + 1]
	const float *test_xyz;            // test points of all models, model-major
	Camera depth_cam;
	int width, height;
	const float *depth, *fill;        // height x width planes: Image::getDepth / the ".distance" map's getProb
	float plausible_dist, depth_fraction, min_keypoint_fraction;
};

__global__ void k_filter_depth_adjust(const int32_t *__restrict__ match_offsets, const int32_t *__restrict__ match_image,
                                      const float *__restrict__ match_xy, const float *__restrict__ match_xyz, const Camera *__restrict__ cams,
                                      const int32_t *__restrict__ obj_model, const float *__restrict__ obj_pose, const int32_t *__restrict__ n_obj_p,
                                      int n_obj_cap, DepthFilterArgs D, const float *__restrict__ raw_score, float *__restrict__ final_score) {
	const int o = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
	const int n_obj = n_obj_p ? min(*n_obj_p, n_obj_cap) : n_obj_cap;
	if (o >= n_obj) return;
	const int m = obj_model[o];
	float T[12];
	pose_matrix(obj_pose + 7 * o, obj_pose + 7 * o + 4, T);
	int cluster_size = 0;
	for (int j = match_offsets[m] + lane; j < match_offsets[m + 1]; j += 32)
		cluster_size += reproj_err(T, cams[match_image[j]], match_xyz + 3 * j, match_xy[2 * j], match_xy[2 * j + 1]) < D.plausible_dist;
	for (int off = 16; off; off >>= 1) cluster_size += __shfl_xor_sync(0xffffffffu, cluster_size, off);
	const int t0 = D.test_offsets[m], n_test = D.test_offsets[m + 1] - t0;
	const Camera &dc = D.depth_cam;
	float IS = 0.f;
	int used = 0;
	for (int k0 = 0; k0 < n_test; k0 += 32) {
		const int k = k0 + lane;
		bool usable = false, adds = false;
		float term = 0.f;
		if (k < n_test) {
			const float *X = D.test_xyz + 3 * (size_t)(t0 + k);
			const float x = __fadd_rn(dot3_rn(X[0], T[0], X[1], T[1], X[2], T[2]), T[3]);
			const float y = __fadd_rn(dot3_rn(X[0], T[4], X[1], T[5], X[2], T[6]), T[7]);
			const float z = __fadd_rn(dot3_rn(X[0], T[8], X[1], T[9], X[2], T[10]), T[11]);
			const float a = __fsub_rn(x, dc.TM[3]), b = __fsub_rn(y, dc.TM[7]), c = __fsub_rn(z, dc.TM[11]);
			const float cx = dot3_rn(a, dc.TM[0], b, dc.TM[4], c, dc.TM[8]);
			const float cy = dot3_rn(a, dc.TM[1], b, dc.TM[5], c, dc.TM[9]);
			const float cz = dot3_rn(a, dc.TM[2], b, dc.TM[6], c, dc.TM[10]);
			const float u = __fadd_rn(__fmul_rn(__fdiv_rn(cx, cz), dc.K[0]), dc.K[2]);
			const float v = __fadd_rn(__fmul_rn(__fdiv_rn(cy, cz), dc.K[1]), dc.K[3]);
			if (u > -2147483648.f && u < 2147483648.f && v > -2147483648.f && v < 2147483648.f) {
				const int ix = (int)u, iy = (int)v;                       // truncation, like the reference's casts
				if (ix >= 0 && ix < D.width && iy >= 0 && iy < D.height && !(D.fill[(size_t)iy * D.width + ix] > 0.f)) {
					usable = true;
					const float kinect = D.depth[(size_t)iy * D.width + ix];
					if (!(kinect < cz)) {
						adds = true;
						term = __fdiv_rn(__fsub_rn(cz, kinect), __fmul_rn(D.depth_fraction, kinect));
						term = __fmul_rn(term, term);
					}
				}
			}
		}
		used += __popc(__ballot_sync(0xffffffffu, usable));
		unsigned msk = __ballot_sync(0xffffffffu, adds);
		while (msk) {                                       // terms in test-point order
			const int l = __ffs(msk) - 1;
			msk &= msk - 1;
			const float t = __shfl_sync(0xffffffffu, term, l);
			IS = __double2float_rn(__dadd_rn((double)IS, __dsub_rn(1.0, __ddiv_rn(1.0, __dadd_rn(1.0, (double)t)))));
		}
	}
	if (lane == 0) {
		if (used <= __float2int_rz(__fmul_rn(D.min_keypoint_fraction, (float)n_test))) IS = 0.f;
		else IS = __fmul_rn(IS, __fdiv_rn((float)cluster_size, (float)used));
		final_score[o] = __fsub_rn(raw_score[o], IS);
	}
}

static mc_status filter_device_impl(mc_ctx *ctx, const int32_t *d_match_offsets, const int32_t *d_match_image, const float *d_match_xy,
                        const float *d_match_xyz, int n_models, int max_matches, const int32_t *d_obj_model, const float *d_obj_pose,
                        const int32_t *d_n_obj, int n_obj_cap, int min_points, float feat_dist, float min_score, const DepthFilterArgs *D,
                        uint8_t *d_keep, float *d_score, int32_t *d_out_n, int32_t *d_cluster_model, int32_t *d_cluster_offsets,
                        int32_t *d_members, int32_t *d_surv_model, float *d_surv_pose, float *d_surv_score);

// device entry. n_obj_dev (nullable) = device-side object count (<= n_obj_cap).
// Outputs: keep/score per input object; out_n = {#survivors, #members}; survivors' clusters (model-major) and
// the surviving objects in list order (surv_*), which is what the next POSE step appends to.
mc_status filter_device(mc_ctx *ctx, const int32_t *d_match_offsets, const int32_t *d_match_image, const float *d_match_xy,
                        const float *d_match_xyz, int n_models, int max_matches, const int32_t *d_obj_model, const float *d_obj_pose,
                        const int32_t *d_n_obj, int n_obj_cap, int min_points, float feat_dist, float min_score,
                        uint8_t *d_keep, float *d_score, int32_t *d_out_n, int32_t *d_cluster_model, int32_t *d_cluster_offsets,
                        int32_t *d_members, int32_t *d_surv_model, float *d_surv_pose, float *d_surv_score) {
	return filter_device_impl(ctx, d_match_offsets, d_match_image, d_match_xy, d_match_xyz, n_models, max_matches, d_obj_model, d_obj_pose, d_n_obj,
	                          n_obj_cap, min_points, feat_dist, min_score, nullptr, d_keep, d_score, d_out_n, d_cluster_model, d_cluster_offsets,
	                          d_members, d_surv_model, d_surv_pose, d_surv_score);
}

// moped3d's FILTER_PROJECTION_DEPTH: D.* are device pointers / host values
mc_status filter_depth_device(mc_ctx *ctx, const int32_t *d_match_offsets, const int32_t *d_match_image, const float *d_match_xy,
                              const float *d_match_xyz, int n_models, int max_matches, const int32_t *d_obj_model, const float *d_obj_pose,
                              const int32_t *d_n_obj, int n_obj_cap, int min_points, float feat_dist, float min_score,
                              const int32_t *d_test_offsets, const float *d_test_xyz, const float *depth_K4, const float *depth_TM12, int width,
                              int height, const float *d_depth, const float *d_fill, float plausible_dist, float depth_fraction,
                              float min_keypoint_fraction, uint8_t *d_keep, float *d_score, int32_t *d_out_n, int32_t *d_cluster_model,
                              int32_t *d_cluster_offsets, int32_t *d_members, int32_t *d_surv_model, float *d_surv_pose, float *d_surv_score) {
	DepthFilterArgs D;
	D.test_offsets = d_test_offsets; D.test_xyz = d_test_xyz;
	for (int i = 0; i < 4; i++) D.depth_cam.K[i] = depth_K4[i];
	for (int i = 0; i < 12; i++) D.depth_cam.TM[i] = depth_TM12[i];
	D.width = width; D.height = height; D.depth = d_depth; D.fill = d_fill;
	D.plausible_dist = plausible_dist; D.depth_fraction = depth_fraction; D.min_keypoint_fraction = min_keypoint_fraction;
	return filter_device_impl(ctx, d_match_offsets, d_match_image, d_match_xy, d_match_xyz, n_models, max_matches, d_obj_model, d_obj_pose, d_n_obj,
	                          n_obj_cap, min_points, feat_dist, min_score, &D, d_keep, d_score, d_out_n, d_cluster_model, d_cluster_offsets,
	                          d_members, d_surv_model, d_surv_pose, d_surv_score);
}

static mc_status filter_device_impl(mc_ctx *ctx, const int32_t *d_match_offsets, const int32_t *d_match_image, const float *d_match_xy,
                        const float *d_match_xyz, int n_models, int max_matches, const int32_t *d_obj_model, const float *d_obj_pose,
                        const int32_t *d_n_obj, int n_obj_cap, int min_points, float feat_dist, float min_score, const DepthFilterArgs *D,
                        uint8_t *d_keep, float *d_score, int32_t *d_out_n, int32_t *d_cluster_model, int32_t *d_cluster_offsets,
                        int32_t *d_members, int32_t *d_surv_model, float *d_surv_pose, float *d_surv_score) {
	if (!ctx->d_cams) { ctx->err = "filter: cameras not set (mc_set_cameras)"; return MC_ERR_STATE; }
	DevBuf &b_in = ctx->scratch[kScrFilterIn], &b_owner = ctx->scratch[kScrFilterOwner], &b_owned = ctx->scratch[kScrFilterOwned];
	const int stride = max_matches > 0 ? max_matches : 1;
	const int cap = n_obj_cap > 0 ? n_obj_cap : 1;
	MC_TRY(reserve(ctx, b_in, (size_t)cap * stride));
	MC_TRY(reserve(ctx, b_owner, sizeof(int32_t) * (size_t)(max_matches + 1)));
	MC_TRY(reserve(ctx, b_owned, sizeof(int32_t) * (size_t)(cap + 1)));
	// depth variant: ownership is decided by the projection score (d_raw), pruning and output use the penalised one (d_score)
	float *d_raw = d_score;
	if (D) { MC_TRY(reserve(ctx, ctx->scratch[kScrFilterRaw], sizeof(float) * (size_t)(cap + 1))); d_raw = (float *)ctx->scratch[kScrFilterRaw].p; }
	if (n_obj_cap > 0) {
		const int score_grid = (n_obj_cap * 32 + 127) / 128 < ctx->num_sms ? (n_obj_cap * 32 + 127) / 128 : ctx->num_sms;
		k_filter_score<<<score_grid, 128, 0, ctx->stream>>>(d_match_offsets, d_match_image, d_match_xy, d_match_xyz, ctx->d_cams, d_obj_model,
		                                                          d_obj_pose, d_n_obj, n_obj_cap, feat_dist, stride, (uint8_t *)b_in.p, d_raw);
		MC_LAUNCH_CHECK();
		if (D) {
			k_filter_depth_adjust<<<(n_obj_cap * 32 + 127) / 128, 128, 0, ctx->stream>>>(d_match_offsets, d_match_image, d_match_xy, d_match_xyz, ctx->d_cams,
			                                                                          d_obj_model, d_obj_pose, d_n_obj, n_obj_cap, *D, d_raw, d_score);
			MC_LAUNCH_CHECK();
		}
	}
	if (max_matches > 0) {
		k_filter_own<<<max_matches < 2 * ctx->num_sms ? max_matches : 2 * ctx->num_sms, 128, 0, ctx->stream>>>(d_match_offsets, n_models, d_match_image, d_match_xy,
		                                                            d_obj_model, d_n_obj, n_obj_cap, stride, (const uint8_t *)b_in.p, d_raw,
		                                                            (int32_t *)b_owner.p);
		MC_LAUNCH_CHECK();
	}
	k_filter_compact<<<1, 256, 0, ctx->stream>>>(d_match_offsets, n_models, d_obj_model, d_obj_pose, d_n_obj, n_obj_cap, (const int32_t *)b_owner.p,
	                                            (int32_t *)b_owned.p, d_keep, d_score, min_points, min_score, d_out_n, d_cluster_model, d_cluster_offsets, d_members,
	                                            d_surv_model, d_surv_pose, d_surv_score);
	MC_LAUNCH_CHECK();
	return MC_OK;
}

} // namespace mc
