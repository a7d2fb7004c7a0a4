// pipeline.cu — device-resident chaining of the stages (SURVEY.md §8f row 1): the FrameData fields that
// the reference keeps in STL containers between `process()` calls (matches, clusters, objects;
// moped2/libmoped/src/util.hpp:68-110) live here as flat device arrays, so that a frame goes
// MATCH -> CLUSTER -> POSE -> FILTER -> POSE2 -> FILTER2 (moped2/libmoped/src/config.hpp:83-120) with one
// host->device copy of the queries and one device->host copy of the objects.
#include "common.cuh"

#include <cstdio>
#include <cstdlib>

namespace mc {

mc_status cluster_device(mc_ctx *ctx, const int32_t *d_match_offsets, const int32_t *d_match_image, const float *d_match_xy,
                         int n_models, int n_images, int max_matches, float radius, float merge, int min_pts, int max_iter,
                         int32_t *d_out_n, int32_t *d_cluster_model, int32_t *d_cluster_offsets, int32_t *d_members);
mc_status pose_ransac_device(mc_ctx *ctx, const int32_t *d_cluster_offsets, const int32_t *d_n_clusters, int n_clusters_cap, int n_points_cap,
                             const float *d_xy, const float *d_xyz, const int32_t *d_image, const int32_t *d_tie,
                             const mc_pose_params *pp, uint8_t *d_found, float *d_pose, int32_t *d_n_tests);
mc_status pose_append_device(mc_ctx *ctx, const int32_t *d_cluster_model, const int32_t *d_n_clusters, int n_clusters_cap, int max_obj,
                             const uint8_t *d_found, const float *d_pose, int32_t *d_n_obj, int obj_cap, int32_t *d_obj_model, float *d_obj_pose);
mc_status filter_device(mc_ctx *ctx, const int32_t *d_match_offsets, const int32_t *d_match_image, const float *d_match_xy,
                        const float *d_match_xyz, int n_models, int max_matches, const int32_t *d_obj_model, const float *d_obj_pose,
                        const int32_t *d_n_obj, int n_obj_cap, int min_points, float feat_dist, float min_score,
                        uint8_t *d_keep, float *d_score, int32_t *d_out_n, int32_t *d_cluster_model, int32_t *d_cluster_offsets,
                        int32_t *d_members, int32_t *d_surv_model, float *d_surv_pose, float *d_surv_score);

// Accepted queries -> matches bucketed by model, query order preserved inside a model
// (`matches[correspModel[nx[0]]].push_back(...)` in query order, MATCH_ANN_CPU.hpp:165-176; the order matters:
// mean-shift is order dependent). One CTA per frame: stable compaction of the accepted queries, then a bitonic sort
// of (model << 13 | rank) keys in shared memory.
// Frame f = blockIdx.x reads fd[f]. out_base (nullable = every frame at 0) places its matches: the per-match arrays and
// acc_list from element out_base[f] on, match_query = out_base[f] + query index in the frame (with out_base = the frames'
// first query ids: the batch-global query id); match_offsets row f (n_models + 1 entries, frame-local: 0 .. matches),
// status[f] and n_obj[f]. A frame cannot write past its own queries' range (matches <= queries), so a batch needs no packing.
// kDepthData (moped3d, mc_process_depth_queries*): DEPTHPROP's per-feature depthData.coord3D (q_world, 3 floats) and .fillDistance
// (q_fill) are gathered into match_world / match_fill in the same pass; they are indexed by batch-global feature id, so out_base
// must then hold the frames' first feature ids. The default instance has no such reads and is the one every other caller launches.
__global__ void k_set_desc(FrameDesc *dst, FrameDesc v) { *dst = v; }

template <bool kDepthData = false>
__global__ void __launch_bounds__(1024)
k_match_compact(const FrameDesc *__restrict__ fd, const int32_t *__restrict__ out_base, int64_t row_base,
                const int32_t *__restrict__ model_of_row, const float *__restrict__ db_xyz, int n_models, int32_t *__restrict__ acc_list,
                int32_t *__restrict__ match_offsets, int32_t *__restrict__ match_query, int32_t *__restrict__ match_row,
                int32_t *__restrict__ match_image, float *__restrict__ match_xy, float *__restrict__ match_xyz,
                int32_t *__restrict__ status, int32_t *__restrict__ n_obj, const float *__restrict__ q_world = nullptr,
                const float *__restrict__ q_fill = nullptr, float *__restrict__ match_world = nullptr, float *__restrict__ match_fill = nullptr) {
	const int f = blockIdx.x;
	fd += f;
	const int base = out_base ? out_base[f] : 0;
	acc_list += base; match_query += base; match_row += base; match_image += base; match_xy += 2 * (size_t)base; match_xyz += 3 * (size_t)base;
	if (kDepthData) { match_world += 3 * (size_t)base; match_fill += base; }
	match_offsets += (size_t)f * (n_models + 1);
	status += f; n_obj += f;
	const int32_t *__restrict__ nn_row = fd->nn_row;
	const uint8_t *__restrict__ accepted = fd->accepted;
	const float *__restrict__ q_xy = fd->q_xy;
	const int32_t *__restrict__ q_image = fd->q_image;     // nullable: every query from image 0
	const int Q = fd->Q;
	__shared__ uint32_t keys[kCompactCap];
	__shared__ int s_warp[32];
	__shared__ int s_base;
	const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
	if (tid == 0) { s_base = 0; status[0] = 0; n_obj[0] = 0; }      // (two memset nodes of the frame chain less)
	__syncthreads();
	for (int q0 = 0; q0 < Q; q0 += 1024) {
		const int q = q0 + tid;
		const bool acc = q < Q && accepted[q];
		const unsigned bal = __ballot_sync(0xffffffffu, acc);
		if (lane == 0) s_warp[w] = __popc(bal);
		__syncthreads();
		int off = s_base;
		for (int i = 0; i < w; i++) off += s_warp[i];
		const int rank = off + __popc(bal & ((1u << lane) - 1));
		if (acc && rank < kCompactCap) {
			acc_list[rank] = q;
			keys[rank] = ((uint32_t)model_of_row[nn_row[2 * q] - row_base] << 13) | (uint32_t)rank;
		}
		__syncthreads();
		if (tid == 0) { int t = 0; for (int i = 0; i < 32; i++) t += s_warp[i]; s_base += t; }
		__syncthreads();
	}
	int M = s_base;
	if (M > kCompactCap) { if (tid == 0) status[0] = 1; M = kCompactCap; }
	int P = 1;
	while (P < M) P <<= 1;
	for (int i = M + tid; i < P; i += 1024) keys[i] = 0xFFFFFFFFu;
	__syncthreads();
	for (int k = 2; k <= P; k <<= 1)
		for (int j = k >> 1; j > 0; j >>= 1) {
			for (int i = tid; i < P; i += 1024) {
				const int ixj = i ^ j;
				if (ixj > i) {
					const uint32_t a = keys[i], b = keys[ixj];
					const bool up = (i & k) == 0;
					if ((a > b) == up) { keys[i] = b; keys[ixj] = a; }
				}
			}
			__syncthreads();
		}
	for (int i = tid; i < M; i += 1024) {
		const uint32_t key = keys[i];
		const int m = (int)(key >> 13), q = acc_list[key & 8191u];
		const int row = nn_row[2 * q];
		match_query[i] = base + q; match_row[i] = row;
		match_image[i] = q_image ? q_image[q] : 0;
		match_xy[2 * i] = q_xy[2 * q]; match_xy[2 * i + 1] = q_xy[2 * q + 1];
		const int64_t lr = (int64_t)row - row_base;
		match_xyz[3 * i] = db_xyz[3 * lr]; match_xyz[3 * i + 1] = db_xyz[3 * lr + 1]; match_xyz[3 * i + 2] = db_xyz[3 * lr + 2];
		if (kDepthData) {
			const size_t g = (size_t)base + q;
			match_world[3 * i] = q_world[3 * g]; match_world[3 * i + 1] = q_world[3 * g + 1]; match_world[3 * i + 2] = q_world[3 * g + 2];
			match_fill[i] = q_fill[g];
		}
		const int mprev = i > 0 ? (int)(keys[i - 1] >> 13) : -1;
		for (int mm = mprev + 1; mm <= m; mm++) match_offsets[mm] = i;
	}
	const int mlast = M > 0 ? (int)(keys[M - 1] >> 13) : -1;
	for (int mm = mlast + 1 + tid; mm <= n_models; mm += 1024) match_offsets[mm] = M;
}

// cluster members -> contiguous per-cluster point arrays (what preprocessAllMatches + `cl` build,
// POSE_..._CPU.hpp:213-237,288-290). tie = match index inside the model (the reference's pointer order).
// moped3d's depth pose stages also take depthData.coord3D (pt_world, nullable) and the Cauchy weight of depthData.fillDistance
// (pt_cauchy, nullable): getCauchyWeight, (float)(1.0 / (1 + f*f)) with f = fill / scale, every operation rounded on its own.
__global__ void k_gather_points(const int32_t *__restrict__ n_p /* {#clusters, #members} */, const int32_t *__restrict__ cluster_model,
                                const int32_t *__restrict__ cluster_offsets, const int32_t *__restrict__ members,
                                const int32_t *__restrict__ match_offsets, const int32_t *__restrict__ match_image,
                                const float *__restrict__ match_xy, const float *__restrict__ match_xyz,
                                float *__restrict__ pt_xy, float *__restrict__ pt_xyz, int32_t *__restrict__ pt_image, int32_t *__restrict__ pt_tie,
                                const float *__restrict__ match_world = nullptr, const float *__restrict__ match_fill = nullptr,
                                float cauchy_scale = 1.f, float *__restrict__ pt_world = nullptr, float *__restrict__ pt_cauchy = nullptr) {
	const int n_clusters = n_p[0];
	for (int c = blockIdx.x; c < n_clusters; c += gridDim.x) {
		const int lo = match_offsets[cluster_model[c]];
		for (int t = cluster_offsets[c] + threadIdx.x; t < cluster_offsets[c + 1]; t += blockDim.x) {
			const int mi = members[t], j = lo + mi;
			pt_xy[2 * t] = match_xy[2 * j]; pt_xy[2 * t + 1] = match_xy[2 * j + 1];
			pt_xyz[3 * t] = match_xyz[3 * j]; pt_xyz[3 * t + 1] = match_xyz[3 * j + 1]; pt_xyz[3 * t + 2] = match_xyz[3 * j + 2];
			pt_image[t] = match_image[j];
			pt_tie[t] = mi;
			if (pt_world) { pt_world[3 * t] = match_world[3 * j]; pt_world[3 * t + 1] = match_world[3 * j + 1]; pt_world[3 * t + 2] = match_world[3 * j + 2]; }
			if (pt_cauchy) {
				const float f = __fdiv_rn(match_fill[j], cauchy_scale);
				pt_cauchy[t] = __double2float_rn(__ddiv_rn(1.0, (double)__fadd_rn(1.f, __fmul_rn(f, f))));
			}
		}
	}
}

__global__ void k_copy_objects(const int32_t *__restrict__ n_p, const int32_t *__restrict__ src_model, const float *__restrict__ src_pose,
                               int32_t *__restrict__ dst_n, int32_t *__restrict__ dst_model, float *__restrict__ dst_pose) {
	const int n = n_p[0];
	for (int i = threadIdx.x; i < n; i += blockDim.x) {
		dst_model[i] = src_model[i];
		for (int j = 0; j < 7; j++) dst_pose[7 * i + j] = src_pose[7 * i + j];
	}
	if (threadIdx.x == 0) *dst_n = n;
}

__global__ void k_export_objects(const FrameDesc *__restrict__ fd, const int32_t *__restrict__ f_n, const int32_t *__restrict__ status,
                                 const int32_t *__restrict__ match_offsets, int n_models, const int32_t *__restrict__ cl_n,
                                 const int32_t *__restrict__ surv_model, const float *__restrict__ surv_pose, const float *__restrict__ surv_score) {
	const int max_objects = fd->max_objects;
	int32_t *out_info = fd->out_info, *out_model = fd->out_model;
	float *out_pose = fd->out_pose, *out_score = fd->out_score;
	const int n = f_n[0];
	const int m = n < max_objects ? n : max_objects;
	for (int i = threadIdx.x; i < m; i += blockDim.x) { out_model[i] = surv_model[i]; out_score[i] = surv_score[i]; }
	for (int i = threadIdx.x; i < 7 * m; i += blockDim.x) out_pose[i] = surv_pose[i];
	if (threadIdx.x == 0) { out_info[0] = n; out_info[1] = status[0]; out_info[2] = match_offsets[n_models]; out_info[3] = cl_n[0]; }
}

__global__ void k_export_empty(int32_t *__restrict__ out_info) {
	if (threadIdx.x < 4) out_info[threadIdx.x] = 0;
}

struct FrameBufs {
	int32_t *nn_row; float *nn_dist; uint8_t *accepted;
	int32_t *acc_list, *match_offsets, *match_query, *match_row, *match_image; float *match_xy, *match_xyz;
	int32_t *status, *cl_n, *cl_model, *cl_offsets, *cl_members;
	float *pt_xy, *pt_xyz; int32_t *pt_image, *pt_tie;
	uint8_t *found; float *task_pose; int32_t *n_tests;
	int32_t *n_obj, *obj_model; float *obj_pose, *obj_score; uint8_t *keep;
	int32_t *f_n, *f_model, *f_offsets, *f_members, *surv_model; float *surv_pose, *surv_score;
};

static mc_status carve(mc_ctx *ctx, FrameBufs &B, int Q, int n_models, int cl_cap, int task_cap, int obj_cap) {
	const size_t q = (size_t)Q, q2 = q + 2, o2 = (size_t)obj_cap + 2;
	return carve_scratch(ctx, ctx->scratch[kScrFrame], [&](Carve &c) {
		c.take(B.nn_row, 2 * q); c.take(B.nn_dist, 2 * q); c.take(B.accepted, q);
		c.take(B.acc_list, q); c.take(B.match_offsets, (size_t)n_models + 2); c.take(B.match_query, q); c.take(B.match_row, q);
		c.take(B.match_image, q); c.take(B.match_xy, 2 * q); c.take(B.match_xyz, 3 * q);
		c.take(B.status, 16); c.take(B.cl_n, 16); c.take(B.cl_model, q2); c.take(B.cl_offsets, q2); c.take(B.cl_members, q2);
		c.take(B.pt_xy, 2 * q); c.take(B.pt_xyz, 3 * q); c.take(B.pt_image, q); c.take(B.pt_tie, q);
		c.take(B.found, task_cap); c.take(B.task_pose, 7 * (size_t)task_cap); c.take(B.n_tests, task_cap);
		c.take(B.n_obj, 16); c.take(B.obj_model, obj_cap); c.take(B.obj_pose, 7 * (size_t)obj_cap); c.take(B.obj_score, obj_cap); c.take(B.keep, obj_cap);
		c.take(B.f_n, 16); c.take(B.f_model, o2); c.take(B.f_offsets, o2); c.take(B.f_members, q2);
		c.take(B.surv_model, obj_cap); c.take(B.surv_pose, 7 * (size_t)obj_cap); c.take(B.surv_score, obj_cap);
	});
}

struct FrameCaps { int cl_cap, obj_cap, task_cap; };

static FrameCaps frame_caps(int Q, const mc_pipeline_params *P) {
	FrameCaps c;
	const int min_pts = P->cluster_min_pts > 0 ? P->cluster_min_pts : 1;
	c.cl_cap = Q / min_pts + 1;
	const int max_obj_per = P->pose.max_objects_per_cluster > P->pose2.max_objects_per_cluster ? P->pose.max_objects_per_cluster : P->pose2.max_objects_per_cluster;
	c.obj_cap = 2 * c.cl_cap * max_obj_per + 8;
	c.task_cap = c.obj_cap * max_obj_per + 8;
	return c;
}

// Enqueue one frame on ctx->stream (ctx may be a lane of a batch): MATCH (only when d_q is given; otherwise the
// descriptor already points at nearest neighbours: object-sharded databases, frame batches) -> CLUSTER -> POSE ->
// FILTER -> POSE2 -> FILTER2 (-> export into the descriptor's output slots when `do_export`). No host
// synchronisation: cluster and object counts stay on the device, grids are sized by upper bounds derived from Q (an
// upper bound of the frame's feature count; the true count is read from the descriptor). Everything that differs
// between frames is read through ctx->frame_desc, so the enqueued chain can be captured once and replayed.
// The surviving objects end in B.f_n / B.surv_*; `ev` (nullable, 7 events) brackets the six stages.
static mc_status frame_enqueue(mc_ctx *ctx, const float *d_q, int Q, const mc_pipeline_params *P,
                               FrameBufs &B, const FrameCaps &caps, cudaEvent_t *ev, bool do_export) {
	const FrameDesc *fd = (const FrameDesc *)ctx->frame_desc.p;
	const int cl_cap = caps.cl_cap, obj_cap = caps.obj_cap;
	auto mark = [&](int i) { if (ev) cudaEventRecord(ev[i], ctx->stream); };
	mark(0);                                             // (B.status / B.n_obj are zeroed by k_match_compact)
	if (d_q) MC_TRY(match_device(ctx, d_q, Q, P->match_ratio, P->match_mode, B.nn_row, B.nn_dist, B.accepted));
	k_match_compact<<<1, 1024, 0, ctx->stream>>>(fd, nullptr, ctx->table_base, ctx->d_model_of_row, ctx->d_xyz, ctx->n_models,
	                                            B.acc_list, B.match_offsets, B.match_query, B.match_row, B.match_image, B.match_xy, B.match_xyz, B.status, B.n_obj);
	MC_LAUNCH_CHECK();
	mark(1);
	// CLUSTER
	MC_TRY(cluster_device(ctx, B.match_offsets, B.match_image, B.match_xy, ctx->n_models, ctx->n_images, Q, P->cluster_radius, P->cluster_merge,
	                      P->cluster_min_pts, P->cluster_max_iterations, B.cl_n, B.cl_model, B.cl_offsets, B.cl_members));
	mark(2);
	// POSE
	k_gather_points<<<ctx->num_sms, 128, 0, ctx->stream>>>(B.cl_n, B.cl_model, B.cl_offsets, B.cl_members, B.match_offsets, B.match_image, B.match_xy,
	                                                     B.match_xyz, B.pt_xy, B.pt_xyz, B.pt_image, B.pt_tie);
	MC_LAUNCH_CHECK();
	MC_TRY(pose_ransac_device(ctx, B.cl_offsets, B.cl_n, cl_cap, Q, B.pt_xy, B.pt_xyz, B.pt_image, B.pt_tie, &P->pose, B.found, B.task_pose, B.n_tests));
	MC_TRY(pose_append_device(ctx, B.cl_model, B.cl_n, cl_cap, P->pose.max_objects_per_cluster, B.found, B.task_pose, B.n_obj, obj_cap, B.obj_model, B.obj_pose));
	mark(3);
	// FILTER
	MC_TRY(filter_device(ctx, B.match_offsets, B.match_image, B.match_xy, B.match_xyz, ctx->n_models, Q, B.obj_model, B.obj_pose, B.n_obj, obj_cap,
	                     P->filter_min_points, P->filter_feature_distance, P->filter_min_score, B.keep, B.obj_score, B.f_n, B.f_model, B.f_offsets,
	                     B.f_members, B.surv_model, B.surv_pose, B.surv_score));
	mark(4);
	// POSE2: the surviving objects stay in the list, new hypotheses from the rebuilt clusters are appended (:295-303)
	k_copy_objects<<<1, 256, 0, ctx->stream>>>(B.f_n, B.surv_model, B.surv_pose, B.n_obj, B.obj_model, B.obj_pose);
	MC_LAUNCH_CHECK();
	k_gather_points<<<ctx->num_sms, 128, 0, ctx->stream>>>(B.f_n, B.f_model, B.f_offsets, B.f_members, B.match_offsets, B.match_image, B.match_xy,
	                                                     B.match_xyz, B.pt_xy, B.pt_xyz, B.pt_image, B.pt_tie);
	MC_LAUNCH_CHECK();
	const int cl2_cap = obj_cap / 2;
	MC_TRY(pose_ransac_device(ctx, B.f_offsets, B.f_n, cl2_cap, Q, B.pt_xy, B.pt_xyz, B.pt_image, B.pt_tie, &P->pose2, B.found, B.task_pose, B.n_tests));
	MC_TRY(pose_append_device(ctx, B.f_model, B.f_n, cl2_cap, P->pose2.max_objects_per_cluster, B.found, B.task_pose, B.n_obj, obj_cap, B.obj_model, B.obj_pose));
	mark(5);
	// FILTER2
	MC_TRY(filter_device(ctx, B.match_offsets, B.match_image, B.match_xy, B.match_xyz, ctx->n_models, Q, B.obj_model, B.obj_pose, B.n_obj, obj_cap,
	                     P->filter2_min_points, P->filter2_feature_distance, P->filter2_min_score, B.keep, B.obj_score, B.f_n, B.f_model, B.f_offsets,
	                     B.f_members, B.surv_model, B.surv_pose, B.surv_score));
	mark(6);
	if (do_export) {
		k_export_objects<<<1, 128, 0, ctx->stream>>>(fd, B.f_n, B.status, B.match_offsets, ctx->n_models, B.cl_n, B.surv_model, B.surv_pose, B.surv_score);
		MC_LAUNCH_CHECK();
	}
	return MC_OK;
}

// for the moped3d frame chain (depth_frames.cu)
mc_status gather_depth_points_device(mc_ctx *ctx, const int32_t *d_n, const int32_t *d_cluster_model, const int32_t *d_cluster_offsets,
                                     const int32_t *d_members, const int32_t *d_match_offsets, const int32_t *d_match_image, const float *d_match_xy,
                                     const float *d_match_xyz, const float *d_match_world, const float *d_match_fill, float cauchy_scale, float *d_pt_xy,
                                     float *d_pt_xyz, float *d_pt_world, float *d_pt_cauchy, int32_t *d_pt_image, int32_t *d_pt_tie) {
	k_gather_points<<<ctx->num_sms, 128, 0, ctx->stream>>>(d_n, d_cluster_model, d_cluster_offsets, d_members, d_match_offsets, d_match_image, d_match_xy,
	                                                     d_match_xyz, d_pt_xy, d_pt_xyz, d_pt_image, d_pt_tie, d_match_world, d_match_fill, cauchy_scale,
	                                                     d_pt_world, d_pt_cauchy);
	MC_LAUNCH_CHECK();
	return MC_OK;
}

// for moped3d's batched MATCH (adaptive.cu): the compaction of n_frames frames in one launch; with d_q_world given (then also d_q_fill,
// d_match_world, d_match_fill, and d_out_base = the frames' first feature ids) it also gathers DEPTHPROP's per-feature depth data
mc_status match_compact_frames_device(mc_ctx *ctx, const FrameDesc *d_fd, const int32_t *d_out_base, int n_frames, int n_models, int32_t *d_acc_list,
                                      int32_t *d_match_offsets, int32_t *d_match_query, int32_t *d_match_row, int32_t *d_match_image,
                                      float *d_match_xy, float *d_match_xyz, int32_t *d_status, int32_t *d_n_obj, const float *d_q_world,
                                      const float *d_q_fill, float *d_match_world, float *d_match_fill) {
	if (d_q_world)
		k_match_compact<true><<<n_frames, 1024, 0, ctx->stream>>>(d_fd, d_out_base, ctx->table_base, ctx->d_model_of_row, ctx->d_xyz, n_models, d_acc_list,
		                                                         d_match_offsets, d_match_query, d_match_row, d_match_image, d_match_xy, d_match_xyz,
		                                                         d_status, d_n_obj, d_q_world, d_q_fill, d_match_world, d_match_fill);
	else
		k_match_compact<<<n_frames, 1024, 0, ctx->stream>>>(d_fd, d_out_base, ctx->table_base, ctx->d_model_of_row, ctx->d_xyz, n_models, d_acc_list,
		                                                   d_match_offsets, d_match_query, d_match_row, d_match_image, d_match_xy, d_match_xyz, d_status,
		                                                   d_n_obj);
	MC_LAUNCH_CHECK();
	return MC_OK;
}

mc_status copy_objects_device(mc_ctx *ctx, const int32_t *d_n, const int32_t *d_src_model, const float *d_src_pose, int32_t *d_dst_n,
                              int32_t *d_dst_model, float *d_dst_pose) {
	k_copy_objects<<<1, 256, 0, ctx->stream>>>(d_n, d_src_model, d_src_pose, d_dst_n, d_dst_model, d_dst_pose);
	MC_LAUNCH_CHECK();
	return MC_OK;
}

static mc_status set_frame_desc(mc_ctx *ctx, const FrameDesc &d) {
	MC_TRY(reserve(ctx, ctx->frame_desc, 256));
	k_set_desc<<<1, 1, 0, ctx->stream>>>((FrameDesc *)ctx->frame_desc.p, d);
	MC_LAUNCH_CHECK();
	return MC_OK;
}

static uint64_t fnv(uint64_t h, const void *p, size_t n) {
	const unsigned char *b = (const unsigned char *)p;
	for (size_t i = 0; i < n; i++) { h ^= b[i]; h *= 1099511628211ULL; }
	return h;
}

// The stage chain of one frame of a batch on a lane (the descriptor is already set): compaction, CLUSTER .. FILTER2,
// export. Replayed from a CUDA graph of the lane when one exists for this configuration (feature-count bucket, stage
// parameters, database) and the lane's scratch buffers have not moved since it was captured; otherwise the chain is
// captured, instantiated and launched. If the capture finds that a scratch buffer has to grow (reserve() refuses to
// allocate while capturing) the frame runs eagerly instead — that run makes the reservations and the next frame captures.
// ~40 kernel launches per frame become one graph launch: with 64 frames per batch the host was the bottleneck of the
// stages after MATCH (2000 launches x ~3.3 us against ~3 ms of device work).
static mc_status frame_chain(mc_ctx *lane, int Q, const mc_pipeline_params *P, cudaEvent_t *ev) {
	mc_ctx *ctx = lane;
	const int q_cap = (Q + 511) & ~511;                  // grids and buffers are sized by upper bounds: a few sizes serve all frames
	const FrameCaps caps = frame_caps(q_cap, P);
	FrameBufs B;
	if (!lane->frame_graphs || ev) {
		MC_TRY(carve(lane, B, q_cap, lane->n_models, caps.cl_cap, caps.task_cap, caps.obj_cap));
		return frame_enqueue(lane, nullptr, q_cap, P, B, caps, ev, true);
	}
	uint64_t cfg = fnv(1469598103934665603ULL, &q_cap, sizeof q_cap);
	cfg = fnv(cfg, P, sizeof *P);
	const int64_t ints[] = { lane->n_models, lane->n_images, lane->table_base, lane->pose_warps, lane->ransac_fused, (int64_t)lane->num_sms, lane->pose_exact_order, lane->ransac_merge_levels };
	cfg = fnv(cfg, ints, sizeof ints);
	const void *ptrs[] = { lane->d_cams, lane->d_xyz, lane->d_model_of_row };
	cfg = fnv(cfg, ptrs, sizeof ptrs);
	auto ptr_key = [&]() {
		uint64_t k = 1469598103934665603ULL;
		for (const DevBuf &b : lane->scratch) k = fnv(k, &b.p, sizeof b.p);
		return fnv(k, &lane->frame_desc.p, sizeof lane->frame_desc.p);
	};
	for (size_t i = 0; i < lane->fgraphs.size(); i++) {
		mc_ctx::FrameGraph &g = lane->fgraphs[i];
		if (g.cfg != cfg) continue;
		if (g.ptr_key == ptr_key()) {
			MC_CUDA(cudaGraphLaunch(g.exec, lane->stream));
			lane->launches += g.nodes;
			return MC_OK;
		}
		cudaGraphExecDestroy(g.exec);                    // a scratch buffer moved: the captured addresses are stale
		lane->fgraphs.erase(lane->fgraphs.begin() + (long)i);
		break;
	}
	const int64_t l0 = lane->launches;
	MC_CUDA(cudaStreamBeginCapture(lane->stream, cudaStreamCaptureModeRelaxed));
	lane->capturing = true;
	mc_status st = carve(lane, B, q_cap, lane->n_models, caps.cl_cap, caps.task_cap, caps.obj_cap);
	if (st == MC_OK) st = frame_enqueue(lane, nullptr, q_cap, P, B, caps, nullptr, true);
	lane->capturing = false;
	cudaGraph_t graph = nullptr;
	const cudaError_t e_end = cudaStreamEndCapture(lane->stream, &graph);
	const int nodes = (int)(lane->launches - l0);
	lane->launches = l0;
	if (st == MC_ERR_STATE) {                            // a reservation is missing: run this frame eagerly (it allocates)
		if (graph) cudaGraphDestroy(graph);
		cudaGetLastError();
		MC_TRY(carve(lane, B, q_cap, lane->n_models, caps.cl_cap, caps.task_cap, caps.obj_cap));
		return frame_enqueue(lane, nullptr, q_cap, P, B, caps, nullptr, true);
	}
	if (st != MC_OK || e_end != cudaSuccess || !graph) {
		if (graph) cudaGraphDestroy(graph);
		cudaGetLastError();
		if (st == MC_OK) { lane->err = std::string("graph capture: ") + cudaGetErrorString(e_end); st = MC_ERR_CUDA; }
		return st;
	}
	mc_ctx::FrameGraph g;
	g.cfg = cfg; g.ptr_key = ptr_key(); g.nodes = nodes; g.exec = nullptr;
	const cudaError_t e_inst = cudaGraphInstantiate(&g.exec, graph, 0);
	cudaGraphDestroy(graph);
	if (e_inst != cudaSuccess) { lane->err = std::string("cudaGraphInstantiate: ") + cudaGetErrorString(e_inst); return MC_ERR_CUDA; }
	if (lane->fgraphs.size() >= 8) { cudaGraphExecDestroy(lane->fgraphs.front().exec); lane->fgraphs.erase(lane->fgraphs.begin()); }
	lane->fgraphs.push_back(g);
	MC_CUDA(cudaGraphLaunch(g.exec, lane->stream));
	lane->launches += g.nodes;
	return MC_OK;
}

// One frame, queries resident on the device. Results are copied to the host at the end (one sync).
mc_status process_frame_device(mc_ctx *ctx, const float *d_q, const float *d_qxy, const int32_t *d_qimg, int Q, const mc_pipeline_params *P,
                               int max_objects, int32_t *n_objects, int32_t *obj_model, float *obj_pose, float *obj_score, float *stage_ms,
                               const int32_t *d_nn_row_in, const uint8_t *d_accepted_in) {
	if (!ctx->d_db) { ctx->err = "process_frame: no database uploaded"; return MC_ERR_STATE; }
	if (!ctx->d_cams) { ctx->err = "process_frame: cameras not set"; return MC_ERR_STATE; }
	if (Q <= 0) { *n_objects = 0; return MC_OK; }
	const FrameCaps caps = frame_caps(Q, P);
	const int obj_cap = caps.obj_cap;
	FrameBufs B;
	MC_TRY(carve(ctx, B, Q, ctx->n_models, caps.cl_cap, caps.task_cap, caps.obj_cap));
	cudaEvent_t ev[7];
	if (stage_ms) for (int i = 0; i < 7; i++) MC_CUDA(cudaEventCreate(&ev[i]));
	FrameDesc d;
	d.nn_row = d_nn_row_in ? d_nn_row_in : B.nn_row; d.accepted = d_accepted_in ? d_accepted_in : B.accepted;
	d.q_xy = d_qxy; d.q_image = d_qimg; d.Q = Q; d.max_objects = max_objects;
	d.out_info = nullptr; d.out_model = nullptr; d.out_pose = nullptr; d.out_score = nullptr;
	MC_TRY(set_frame_desc(ctx, d));
	MC_TRY(frame_enqueue(ctx, d_nn_row_in ? nullptr : d_q, Q, P, B, caps, stage_ms ? ev : nullptr, false));
	// results -> host
	const size_t bytes = 64 + (size_t)max_objects * (4 + 28 + 4);
	MC_TRY(pinned(ctx, bytes + 64));
	char *hp = (char *)ctx->h_pinned;
	int32_t *h_n = (int32_t *)hp; int32_t *h_status = (int32_t *)(hp + 32);
	int32_t *h_model = (int32_t *)(hp + 64); float *h_pose = (float *)(hp + 64 + 4ull * max_objects); float *h_score = (float *)(hp + 64 + 32ull * max_objects);
	const int ncopy = max_objects < obj_cap ? max_objects : obj_cap;
	MC_CUDA(cudaMemcpyAsync(h_n, B.f_n, 8, cudaMemcpyDeviceToHost, ctx->stream));
	MC_CUDA(cudaMemcpyAsync(h_status, B.status, 4, cudaMemcpyDeviceToHost, ctx->stream));
	MC_CUDA(cudaMemcpyAsync(h_model, B.surv_model, 4ull * ncopy, cudaMemcpyDeviceToHost, ctx->stream));
	MC_CUDA(cudaMemcpyAsync(h_pose, B.surv_pose, 28ull * ncopy, cudaMemcpyDeviceToHost, ctx->stream));
	MC_CUDA(cudaMemcpyAsync(h_score, B.surv_score, 4ull * ncopy, cudaMemcpyDeviceToHost, ctx->stream));
	MC_CUDA(cudaStreamSynchronize(ctx->stream));
	if (stage_ms) {
		for (int i = 0; i < 6; i++) { cudaEventElapsedTime(&stage_ms[i], ev[i], ev[i + 1]); }
		for (int i = 0; i < 7; i++) cudaEventDestroy(ev[i]);
	}
	if (*h_status) { ctx->err = "process_frame: more than 8192 accepted matches in one frame"; return MC_ERR_CAPACITY; }
	int n = h_n[0];
	if (n > ncopy) { ctx->err = "process_frame: object buffer too small"; *n_objects = n; return MC_ERR_CAPACITY; }
	*n_objects = n;
	memcpy(obj_model, h_model, 4ull * n);
	memcpy(obj_pose, h_pose, 28ull * n);
	memcpy(obj_score, h_score, 4ull * n);
	return MC_OK;
}

// =============================================================================================
// one frame, RANSAC partitioned by cluster across ranks (north_star: "RANSAC work is distributed by cluster";
// the reference's task list: POSE_RANSAC_LM_DIFF_REPROJECTION_CPU.hpp:275-282 hands (cluster, try) tasks to its worker threads)
// =============================================================================================
// Every rank holds the frame's merged nearest neighbours and runs the cheap stages redundantly (compaction, CLUSTER, FILTER:
// identical on all ranks by construction); the (cluster, try) tasks of POSE and POSE2 are dealt round-robin by cluster, rank r
// running the clusters c with c % world == r. A task's random stream depends on its index alone, so the union of the ranks'
// results is the single-GPU result bit for bit. The two exchange points are the caller's (an NCCL all-gather of one small
// record per rank, in place in `exchange`), which is why the frame is three calls:
//   phase 0  compaction, CLUSTER, POSE tasks of this rank        -> record in slot `rank` of `exchange`
//   phase 1  (gathered records) objects, FILTER, POSE2 tasks     -> record in slot `rank`
//   phase 2  (gathered records) objects, FILTER2, export
// Record of a phase: found[task_cap] (bytes) | pose[task_cap][7] | n_tests[task_cap], each part 256-byte aligned.
struct ShardSlot { uint8_t *found; float *pose; int32_t *n_tests; size_t bytes; };

// record `slot` of `exchange`; exchange == nullptr: the record's size only
static ShardSlot shard_slot(void *exchange, int slot, int task_cap) {
	ShardSlot s;
	auto layout = [&](Carve &c) { c.take(s.found, task_cap); c.take(s.pose, 7 * (size_t)task_cap); c.take(s.n_tests, task_cap); };
	Carve c;
	layout(c);
	s.bytes = c.off;
	if (exchange) { c = Carve{(char *)exchange + (size_t)slot * s.bytes}; layout(c); }
	return s;
}

// task t belongs to the rank that owns its cluster: take its result from that rank's record
__global__ void k_shard_select(const uint8_t *__restrict__ exchange, size_t slot_bytes, size_t o_pose, size_t o_tests, int world, int n_tasks, int max_obj,
                               uint8_t *__restrict__ found, float *__restrict__ pose, int32_t *__restrict__ n_tests) {
	const int t = blockIdx.x * blockDim.x + threadIdx.x;
	if (t >= n_tasks) return;
	const uint8_t *b = exchange + (size_t)((t / max_obj) % world) * slot_bytes;
	found[t] = b[t];
	const float *sp = (const float *)(b + o_pose) + 7 * (size_t)t;
#pragma unroll
	for (int j = 0; j < 7; j++) pose[7 * (size_t)t + j] = sp[j];
	n_tests[t] = ((const int32_t *)(b + o_tests))[t];
}

size_t frame_shard_slot_bytes(int Q, const mc_pipeline_params *P) { return shard_slot(nullptr, 0, frame_caps(Q, P).task_cap).bytes; }

mc_status process_frame_sharded_device(mc_ctx *ctx, int phase, const int32_t *d_nn_row, const uint8_t *d_accepted, const float *d_qxy,
                                       const int32_t *d_qimg, int Q, const mc_pipeline_params *P, int shard_rank, int shard_world, void *d_exchange,
                                       int max_objects, int32_t *d_out_info, int32_t *d_out_model, float *d_out_pose, float *d_out_score) {
	if (!ctx->d_cams) { ctx->err = "process_frame_sharded: cameras not set"; return MC_ERR_STATE; }
	if (!ctx->d_xyz || !ctx->d_model_of_row) { ctx->err = "process_frame_sharded: no database tables (mc_db_upload / mc_db_set_global_tables)"; return MC_ERR_STATE; }
	const FrameCaps caps = frame_caps(Q, P);
	const int cl_cap = caps.cl_cap, obj_cap = caps.obj_cap, cl2_cap = obj_cap / 2;
	FrameBufs B;
	MC_TRY(carve(ctx, B, Q, ctx->n_models, caps.cl_cap, caps.task_cap, caps.obj_cap));
	const FrameDesc *fd = (const FrameDesc *)ctx->frame_desc.p;
	const ShardSlot mine = shard_slot(d_exchange, shard_rank, caps.task_cap), base = shard_slot(d_exchange, 0, caps.task_cap);
	const size_t o_pose = (size_t)((char *)base.pose - (char *)base.found), o_tests = (size_t)((char *)base.n_tests - (char *)base.found);
	auto select = [&](int n_tasks, int max_obj) -> mc_status {
		k_shard_select<<<(n_tasks + 255) / 256, 256, 0, ctx->stream>>>((const uint8_t *)d_exchange, base.bytes, o_pose, o_tests, shard_world, n_tasks, max_obj,
		                                                              B.found, B.task_pose, B.n_tests);
		MC_LAUNCH_CHECK();
		return MC_OK;
	};
	struct ShardScope {                    // the RANSAC launches inside read the partition from the context
		mc_ctx *c;
		ShardScope(mc_ctx *c_, int r, int w) : c(c_) { c->ransac_shard_rank = r; c->ransac_shard_world = w; }
		~ShardScope() { c->ransac_shard_rank = 0; c->ransac_shard_world = 1; }
	} scope(ctx, shard_rank, shard_world);
	if (phase == 0) {
		FrameDesc d;
		d.nn_row = d_nn_row; d.accepted = d_accepted; d.q_xy = d_qxy; d.q_image = d_qimg; d.Q = Q; d.max_objects = max_objects;
		d.out_info = d_out_info; d.out_model = d_out_model; d.out_pose = d_out_pose; d.out_score = d_out_score;
		MC_TRY(set_frame_desc(ctx, d));
		fd = (const FrameDesc *)ctx->frame_desc.p;
		k_match_compact<<<1, 1024, 0, ctx->stream>>>(fd, nullptr, ctx->table_base, ctx->d_model_of_row, ctx->d_xyz, ctx->n_models,
		                                            B.acc_list, B.match_offsets, B.match_query, B.match_row, B.match_image, B.match_xy, B.match_xyz, B.status, B.n_obj);
		MC_LAUNCH_CHECK();
		MC_TRY(cluster_device(ctx, B.match_offsets, B.match_image, B.match_xy, ctx->n_models, ctx->n_images, Q, P->cluster_radius, P->cluster_merge,
		                      P->cluster_min_pts, P->cluster_max_iterations, B.cl_n, B.cl_model, B.cl_offsets, B.cl_members));
		k_gather_points<<<ctx->num_sms, 128, 0, ctx->stream>>>(B.cl_n, B.cl_model, B.cl_offsets, B.cl_members, B.match_offsets, B.match_image, B.match_xy,
		                                                     B.match_xyz, B.pt_xy, B.pt_xyz, B.pt_image, B.pt_tie);
		MC_LAUNCH_CHECK();
		return pose_ransac_device(ctx, B.cl_offsets, B.cl_n, cl_cap, Q, B.pt_xy, B.pt_xyz, B.pt_image, B.pt_tie, &P->pose, mine.found, mine.pose, mine.n_tests);
	}
	if (phase == 1) {
		MC_TRY(select(cl_cap * P->pose.max_objects_per_cluster, P->pose.max_objects_per_cluster));
		MC_TRY(pose_append_device(ctx, B.cl_model, B.cl_n, cl_cap, P->pose.max_objects_per_cluster, B.found, B.task_pose, B.n_obj, obj_cap, B.obj_model, B.obj_pose));
		MC_TRY(filter_device(ctx, B.match_offsets, B.match_image, B.match_xy, B.match_xyz, ctx->n_models, Q, B.obj_model, B.obj_pose, B.n_obj, obj_cap,
		                     P->filter_min_points, P->filter_feature_distance, P->filter_min_score, B.keep, B.obj_score, B.f_n, B.f_model, B.f_offsets,
		                     B.f_members, B.surv_model, B.surv_pose, B.surv_score));
		k_copy_objects<<<1, 256, 0, ctx->stream>>>(B.f_n, B.surv_model, B.surv_pose, B.n_obj, B.obj_model, B.obj_pose);
		MC_LAUNCH_CHECK();
		k_gather_points<<<ctx->num_sms, 128, 0, ctx->stream>>>(B.f_n, B.f_model, B.f_offsets, B.f_members, B.match_offsets, B.match_image, B.match_xy,
		                                                     B.match_xyz, B.pt_xy, B.pt_xyz, B.pt_image, B.pt_tie);
		MC_LAUNCH_CHECK();
		return pose_ransac_device(ctx, B.f_offsets, B.f_n, cl2_cap, Q, B.pt_xy, B.pt_xyz, B.pt_image, B.pt_tie, &P->pose2, mine.found, mine.pose, mine.n_tests);
	}
	if (phase == 2) {
		MC_TRY(select(cl2_cap * P->pose2.max_objects_per_cluster, P->pose2.max_objects_per_cluster));
		MC_TRY(pose_append_device(ctx, B.f_model, B.f_n, cl2_cap, P->pose2.max_objects_per_cluster, B.found, B.task_pose, B.n_obj, obj_cap, B.obj_model, B.obj_pose));
		MC_TRY(filter_device(ctx, B.match_offsets, B.match_image, B.match_xy, B.match_xyz, ctx->n_models, Q, B.obj_model, B.obj_pose, B.n_obj, obj_cap,
		                     P->filter2_min_points, P->filter2_feature_distance, P->filter2_min_score, B.keep, B.obj_score, B.f_n, B.f_model, B.f_offsets,
		                     B.f_members, B.surv_model, B.surv_pose, B.surv_score));
		k_export_objects<<<1, 128, 0, ctx->stream>>>(fd, B.f_n, B.status, B.match_offsets, ctx->n_models, B.cl_n, B.surv_model, B.surv_pose, B.surv_score);
		MC_LAUNCH_CHECK();
		return MC_OK;
	}
	ctx->err = "process_frame_sharded: phase must be 0, 1 or 2";
	return MC_ERR_ARG;
}

// =============================================================================================
// frame batches (BASELINE.json configs[4], SURVEY.md §8f row 1)
// =============================================================================================
// A batch is a list of independent frames (each its own FrameData in the reference: moped.cpp:166-194 runs
// them one after the other). MATCH runs once for the queries of all frames — one pass over the database tile
// images, query tiles of 256 may straddle frames — and the stages after it, which are latency-bound chains of
// small kernels, run per frame on concurrent lanes. Every frame gives exactly the result of mc_process_frame.

// frame result -> its slot of the batch output. info = {objects, status, accepted matches, clusters after CLUSTER}
static void lane_borrow(mc_ctx *ctx, mc_ctx *lane) {
	lane->device = ctx->device; lane->num_sms = ctx->num_sms;
	lane->n_rows = ctx->n_rows; lane->row_base = ctx->row_base; lane->n_tiles = ctx->n_tiles; lane->D = ctx->D; lane->n_models = ctx->n_models;
	lane->d_db = ctx->d_db; lane->d_db_img = ctx->d_db_img; lane->d_xyz = ctx->d_xyz; lane->d_model_of_row = ctx->d_model_of_row;
	lane->table_base = ctx->table_base; lane->table_rows = ctx->table_rows;
	lane->db_norm2_min = ctx->db_norm2_min; lane->db_norm2_max = ctx->db_norm2_max;
	lane->d_cams = ctx->d_cams; lane->n_images = ctx->n_images;
	lane->pose_warps = ctx->pose_warps;
	lane->fit_thread_min = ctx->fit_thread_min; lane->fit_stream = ctx->fit_stream; lane->ransac_merge_levels = ctx->ransac_merge_levels; lane->ransac_fused = ctx->ransac_fused; lane->frame_graphs = ctx->frame_graphs;
	lane->pose_exact_order = ctx->pose_exact_order;
}

mc_status ensure_lanes(mc_ctx *ctx, int n) {
	if (!ctx->ev_fork) MC_CUDA(cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
	while ((int)ctx->lanes.size() < n) {
		mc_ctx *lane = new mc_ctx;
		lane->parent = ctx;
		// highest priority: when MATCH of a later chunk (or of the next step) is queued on the context's stream, the small
		// latency-bound stage kernels of the lanes get the SM slots that free up first
		int prio_least = 0, prio_greatest = 0;
		cudaDeviceGetStreamPriorityRange(&prio_least, &prio_greatest);
		bool ok;
		if (ctx->green_stage) ok = sm_partition_stage_stream(ctx, &lane->stream, prio_greatest) == MC_OK;   // confined to the stage partition's SMs
		else ok = cudaStreamCreateWithPriority(&lane->stream, cudaStreamNonBlocking, prio_greatest) == cudaSuccess;
		if (!ok || cudaEventCreateWithFlags(&lane->ev_done, cudaEventDisableTiming) != cudaSuccess) {
			delete lane;
			ctx->err = "process_frames: cannot create a lane stream";
			return MC_ERR_CUDA;
		}
		lane->own_stream = true;
		ctx->lanes.push_back(lane);
	}
	for (mc_ctx *lane : ctx->lanes) lane_borrow(ctx, lane);
	return MC_OK;
}

// order ctx->stream after everything the lanes have been given since the last join
mc_status join_lanes(mc_ctx *ctx) {
	for (int l = 0; l < ctx->lanes_pending && l < (int)ctx->lanes.size(); l++) {
		mc_ctx *lane = ctx->lanes[l];
		MC_CUDA(cudaEventRecord(lane->ev_done, lane->stream));
		MC_CUDA(cudaStreamWaitEvent(ctx->stream, lane->ev_done, 0));
		ctx->launches += lane->launches; lane->launches = 0;
	}
	ctx->lanes_pending = 0;
	return MC_OK;
}

// Frames [f_begin, f_end) of a batch whose queries (all frames, concatenated) are resident on the device.
// d_nn_row_in / d_accepted_in (nullable, all frames): merged nearest neighbours of an object-sharded database;
// otherwise MATCH runs here for the queries of frames [f_begin, f_end). Outputs are DEVICE arrays with one slot
// per processed frame: out_info 4 ints, out_model max_objects, out_pose 7*max_objects, out_score max_objects.
// Asynchronous: returns with the work enqueued and ctx->stream ordered after all lanes.
mc_status process_frames_device(mc_ctx *ctx, const float *d_q, const float *d_qxy, const int32_t *d_qimg, const int32_t *frame_offsets,
                                int f_begin, int f_end, const mc_pipeline_params *P, int max_objects, const int32_t *d_nn_row_in,
                                const uint8_t *d_accepted_in, int32_t *d_out_info, int32_t *d_out_model, float *d_out_pose, float *d_out_score,
                                cudaEvent_t *ev3) {
	if (!ctx->d_db) { ctx->err = "process_frames: no database uploaded"; return MC_ERR_STATE; }
	if (!ctx->d_cams) { ctx->err = "process_frames: cameras not set"; return MC_ERR_STATE; }
	const int nf = f_end - f_begin;
	if (nf <= 0) return MC_OK;
	const int q_lo = frame_offsets[f_begin], q_hi = frame_offsets[f_end];
	const int Qb = q_hi - q_lo;
	if (ev3) MC_CUDA(cudaEventRecord(ev3[0], ctx->stream));
	const int32_t *nn_row = d_nn_row_in;
	const uint8_t *accepted = d_accepted_in;
	const bool do_match = !d_nn_row_in && Qb > 0;
	if (do_match) {
		MC_TRY(reserve(ctx, ctx->nn_row, sizeof(int32_t) * 2 * (size_t)Qb));
		MC_TRY(reserve(ctx, ctx->nn_dist, sizeof(float) * 2 * (size_t)Qb));
		MC_TRY(reserve(ctx, ctx->accepted, (size_t)Qb));
		// the batch-local arrays are indexed by global query id below
		nn_row = (const int32_t *)ctx->nn_row.p - 2 * (size_t)q_lo;
		accepted = (const uint8_t *)ctx->accepted.p - (size_t)q_lo;
	}
	int n_lanes = ctx->n_lanes_wanted < nf ? ctx->n_lanes_wanted : nf;
	if (n_lanes < 1) n_lanes = 1;
	MC_TRY(ensure_lanes(ctx, n_lanes));
	// Chunks: MATCH of chunk c+1 (ctx->stream, tensor-bound, one CTA per SM) overlaps the latency-bound stages
	// of chunk c (lanes), whose small CTAs fit beside a matching CTA on the same SM.
	int n_chunks = do_match ? ctx->match_chunks : 1;
	if (n_chunks > nf) n_chunks = nf;
	if (n_chunks < 1) n_chunks = 1;
	while ((int)ctx->ev_chunk.size() < n_chunks) {
		cudaEvent_t e;
		MC_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
		ctx->ev_chunk.push_back(e);
	}
	static const bool trace = getenv("MOPED_CUDA_TRACE") != nullptr;     // debugging aid: per-frame stage timeline on stderr
	std::vector<cudaEvent_t> tev;
	cudaEvent_t t0 = nullptr;
	if (trace) {
		tev.resize(7 * (size_t)nf);
		for (auto &e : tev) cudaEventCreate(&e);
		cudaEventCreate(&t0);
		cudaEventRecord(t0, ctx->stream);
	}
	// ---- one CUDA graph for the stage chains of ALL frames of the call ("batch graph") ----
	// Lane streams are host-visible queues and the hardware has 32 of them: 64 frames on 64 lane streams run as two rounds of 32
	// (traced), which is why a 64-frame batch spent two chain latencies after MATCH. The branches of ONE graph are not bound by
	// that: a graph of 128 independent 10-kernel chains runs in 1.3 chain latencies on a B200 (scripts/probe/graph_branches.cu,
	// profiles/graph_branches_r2b.jsonl). So the fork to the lanes, every frame's descriptor + chain and the join are captured once
	// into a single graph (keyed by everything the chains read: descriptors, sizes, parameters, scratch addresses) and replayed
	// with one launch per batch. Not used with a deferred lane join / an SM partition (there the lanes must stay separate streams
	// that run beside the next MATCH), with several MATCH chunks, or while a lane still has to grow its scratch (that call runs
	// the per-lane path below, which allocates; the next one captures).
	const bool own_stream = ctx->stream != nullptr && ctx->stream != cudaStreamLegacy && ctx->stream != cudaStreamPerThread;
	if (ctx->batch_graph && ctx->frame_graphs && !ctx->defer_lane_join && !ctx->green_stage && n_chunks == 1 && !trace && own_stream && nf > 1) {
		const int cq_lo = frame_offsets[f_begin], cq = frame_offsets[f_end] - cq_lo;
		if (do_match && cq > 0)
			MC_TRY(match_device(ctx, d_q + (size_t)cq_lo * ctx->D, cq, P->match_ratio, P->match_mode, (int32_t *)nn_row + 2 * (size_t)cq_lo,
			                    (float *)ctx->nn_dist.p + 2 * (size_t)(cq_lo - q_lo), (uint8_t *)accepted + cq_lo));
		if (ev3) MC_CUDA(cudaEventRecord(ev3[1], ctx->stream));
		std::vector<FrameDesc> descs((size_t)nf);
		std::vector<int> Qs((size_t)nf);
		for (int s = 0; s < nf; s++) {
			const int f = f_begin + s;
			const int q0 = frame_offsets[f], Q = frame_offsets[f + 1] - q0;
			FrameDesc &d = descs[(size_t)s];
			memset(&d, 0, sizeof d);
			d.nn_row = nn_row + 2 * (size_t)q0; d.accepted = accepted + q0; d.q_xy = d_qxy + 2 * (size_t)q0; d.q_image = d_qimg + q0;
			d.Q = Q; d.max_objects = max_objects;
			d.out_info = d_out_info + 4 * (size_t)s; d.out_model = d_out_model + (size_t)s * max_objects;
			d.out_pose = d_out_pose + 7 * (size_t)s * max_objects; d.out_score = d_out_score + (size_t)s * max_objects;
			Qs[(size_t)s] = Q;
		}
		auto batch_key = [&]() {
			uint64_t k = fnv(1469598103934665603ULL, descs.data(), sizeof(FrameDesc) * descs.size());
			k = fnv(k, P, sizeof *P);
			const int64_t ints[] = { nf, n_lanes, ctx->n_models, ctx->n_images, ctx->table_base, ctx->pose_warps, ctx->ransac_fused, (int64_t)ctx->num_sms,
			                         ctx->pose_exact_order, max_objects, ctx->ransac_merge_levels };
			k = fnv(k, ints, sizeof ints);
			const void *ptrs[] = { ctx->d_cams, ctx->d_xyz, ctx->d_model_of_row };
			k = fnv(k, ptrs, sizeof ptrs);
			for (int l = 0; l < n_lanes; l++) {
				for (const DevBuf &b : ctx->lanes[(size_t)l]->scratch) k = fnv(k, &b.p, sizeof b.p);
				k = fnv(k, &ctx->lanes[(size_t)l]->frame_desc.p, sizeof(void *));
			}
			return k;
		};
		uint64_t key = batch_key();
		bool launched = false;
		for (size_t i = 0; i < ctx->bgraphs.size() && !launched; i++)
			if (ctx->bgraphs[i].key == key) {
				MC_CUDA(cudaGraphLaunch(ctx->bgraphs[i].exec, ctx->stream));
				ctx->launches += ctx->bgraphs[i].nodes;
				launched = true;
			}
		if (!launched) {
			mc_status st = MC_OK;
			for (int l = 0; l < n_lanes; l++) ctx->lanes[(size_t)l]->launches = 0;
			MC_CUDA(cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeRelaxed));
			cudaError_t e = cudaEventRecord(ctx->ev_fork, ctx->stream);
			for (int l = 0; l < n_lanes && e == cudaSuccess; l++) { ctx->lanes[(size_t)l]->capturing = true; e = cudaStreamWaitEvent(ctx->lanes[(size_t)l]->stream, ctx->ev_fork, 0); }
			for (int s = 0; s < nf && st == MC_OK && e == cudaSuccess; s++) {
				mc_ctx *lane = ctx->lanes[(size_t)(s % n_lanes)];
				if (Qs[(size_t)s] <= 0) {
					k_export_empty<<<1, 32, 0, lane->stream>>>(descs[(size_t)s].out_info);
					lane->launches++;
					continue;
				}
				st = set_frame_desc(lane, descs[(size_t)s]);
				if (st != MC_OK) break;
				const int q_cap = (Qs[(size_t)s] + 511) & ~511;
				const FrameCaps caps = frame_caps(q_cap, P);
				FrameBufs B;
				st = carve(lane, B, q_cap, lane->n_models, caps.cl_cap, caps.task_cap, caps.obj_cap);
				if (st == MC_OK) st = frame_enqueue(lane, nullptr, q_cap, P, B, caps, nullptr, true);
			}
			int nodes = 0;
			for (int l = 0; l < n_lanes; l++) {
				mc_ctx *lane = ctx->lanes[(size_t)l];
				lane->capturing = false;
				if (e == cudaSuccess) e = cudaEventRecord(lane->ev_done, lane->stream);
				if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->stream, lane->ev_done, 0);
				nodes += (int)lane->launches; lane->launches = 0;
			}
			cudaGraph_t graph = nullptr;
			const cudaError_t e_end = cudaStreamEndCapture(ctx->stream, &graph);
			if (st == MC_OK && e == cudaSuccess && e_end == cudaSuccess && graph) {
				mc_ctx::BatchGraph g;
				g.key = batch_key();                 // (set_frame_desc may have made a lane's first descriptor buffer: addresses are final now)
				g.nodes = nodes; g.exec = nullptr;
				const cudaError_t e_inst = cudaGraphInstantiate(&g.exec, graph, 0);
				cudaGraphDestroy(graph);
				if (e_inst != cudaSuccess) { ctx->err = std::string("cudaGraphInstantiate (batch graph): ") + cudaGetErrorString(e_inst); return MC_ERR_CUDA; }
				if (ctx->bgraphs.size() >= 6) { cudaGraphExecDestroy(ctx->bgraphs.front().exec); ctx->bgraphs.erase(ctx->bgraphs.begin()); }
				ctx->bgraphs.push_back(g);
				MC_CUDA(cudaGraphLaunch(g.exec, ctx->stream));
				ctx->launches += nodes;
				launched = true;
			} else {
				if (graph) cudaGraphDestroy(graph);
				cudaGetLastError();
				if (st != MC_OK && st != MC_ERR_STATE) { ctx->err = ctx->lanes[0]->err; for (mc_ctx *lane : ctx->lanes) if (!lane->err.empty()) ctx->err = lane->err; return st; }
				if (st == MC_OK) { ctx->err = std::string("batch graph capture: ") + cudaGetErrorString(e != cudaSuccess ? e : e_end); return MC_ERR_CUDA; }
				// a lane has to grow a scratch buffer: this call takes the per-lane path (which allocates)
			}
		}
		if (launched) {
			if (ev3) MC_CUDA(cudaEventRecord(ev3[2], ctx->stream));
			ctx->batch_stats[0] = nf; ctx->batch_stats[3] = n_lanes;
			return MC_OK;
		}
		// fall through to the per-lane path WITHOUT matching again
		for (int s = 0; s < nf; s++) {
			mc_ctx *lane = ctx->lanes[(size_t)(s % n_lanes)];
			if (s < n_lanes) {
				MC_CUDA(cudaEventRecord(ctx->ev_fork, ctx->stream));
				MC_CUDA(cudaStreamWaitEvent(lane->stream, ctx->ev_fork, 0));
			}
			mc_status st = MC_OK;
			if (Qs[(size_t)s] <= 0) { k_export_empty<<<1, 32, 0, lane->stream>>>(descs[(size_t)s].out_info); lane->launches++; }
			else {
				st = set_frame_desc(lane, descs[(size_t)s]);
				if (st == MC_OK) st = frame_chain(lane, Qs[(size_t)s], P, nullptr);
			}
			if (st != MC_OK) { ctx->err = lane->err; return st; }
		}
		if (n_lanes > ctx->lanes_pending) ctx->lanes_pending = n_lanes;
		MC_TRY(join_lanes(ctx));
		if (ev3) MC_CUDA(cudaEventRecord(ev3[2], ctx->stream));
		ctx->batch_stats[0] = nf; ctx->batch_stats[3] = n_lanes;
		return MC_OK;
	}
	for (int c = 0; c < n_chunks; c++) {
		const int fb = f_begin + (int)((int64_t)nf * c / n_chunks), fe = f_begin + (int)((int64_t)nf * (c + 1) / n_chunks);
		const int cq_lo = frame_offsets[fb], cq = frame_offsets[fe] - cq_lo;
		if (do_match && cq > 0)
			MC_TRY(match_device(ctx, d_q + (size_t)cq_lo * ctx->D, cq, P->match_ratio, P->match_mode, (int32_t *)nn_row + 2 * (size_t)cq_lo,
			                    (float *)ctx->nn_dist.p + 2 * (size_t)(cq_lo - q_lo), (uint8_t *)accepted + cq_lo));
		if (ev3 && c == n_chunks - 1) MC_CUDA(cudaEventRecord(ev3[1], ctx->stream));
		MC_CUDA(cudaEventRecord(ctx->ev_chunk[c], ctx->stream));
		const int used = (fe - fb) < n_lanes ? (fe - fb) : n_lanes;
		for (int l = 0; l < used; l++) MC_CUDA(cudaStreamWaitEvent(ctx->lanes[(fb - f_begin + l) % n_lanes]->stream, ctx->ev_chunk[c], 0));
		for (int f = fb; f < fe; f++) {
			const int s = f - f_begin;
			mc_ctx *lane = ctx->lanes[s % n_lanes];
			const int q0 = frame_offsets[f], Q = frame_offsets[f + 1] - q0;
			int32_t *o_info = d_out_info + 4 * (size_t)s;
			mc_status st = MC_OK;
			if (Q <= 0) {
				k_export_empty<<<1, 32, 0, lane->stream>>>(o_info);
				lane->launches++;
			} else {
				FrameDesc d;
				d.nn_row = nn_row + 2 * (size_t)q0; d.accepted = accepted + q0; d.q_xy = d_qxy + 2 * (size_t)q0; d.q_image = d_qimg + q0;
				d.Q = Q; d.max_objects = max_objects;
				d.out_info = o_info; d.out_model = d_out_model + (size_t)s * max_objects;
				d.out_pose = d_out_pose + 7 * (size_t)s * max_objects; d.out_score = d_out_score + (size_t)s * max_objects;
				st = set_frame_desc(lane, d);
				if (st == MC_OK) st = frame_chain(lane, Q, P, trace ? &tev[7 * (size_t)s] : nullptr);
			}
			if (st != MC_OK) { ctx->err = lane->err; return st; }
		}
	}
	if (n_lanes > ctx->lanes_pending) ctx->lanes_pending = n_lanes;
	if (!ctx->defer_lane_join) MC_TRY(join_lanes(ctx));
	if (ev3) MC_CUDA(cudaEventRecord(ev3[2], ctx->stream));
	if (trace) {
		cudaStreamSynchronize(ctx->stream);
		for (int s = 0; s < nf; s++) {
			if (frame_offsets[f_begin + s + 1] - frame_offsets[f_begin + s] <= 0) continue;
			fprintf(stderr, "[trace] frame %3d:", f_begin + s);
			for (int i = 0; i < 7; i++) { float ms = 0.f; cudaEventElapsedTime(&ms, t0, tev[7 * (size_t)s + i]); fprintf(stderr, " %7.3f", ms); }
			fprintf(stderr, "  (ms since batch start: begin, compact, cluster, pose, filter, pose2, filter2)\n");
		}
		for (auto &e : tev) cudaEventDestroy(e);
		cudaEventDestroy(t0);
	}
	ctx->batch_stats[0] = nf; ctx->batch_stats[3] = n_lanes;
	return MC_OK;
}

// Host-facing tail: batch outputs -> host arrays (one copy, one synchronisation).
mc_status process_frames_host(mc_ctx *ctx, const float *d_q, const float *d_qxy, const int32_t *d_qimg, const int32_t *frame_offsets, int n_frames,
                              const mc_pipeline_params *P, int max_objects, int32_t *n_objects, int32_t *obj_model, float *obj_pose, float *obj_score,
                              int32_t *frame_info, float *stage_ms) {
	const size_t bytes = batch_slots_bytes(n_frames, max_objects);
	MC_TRY(reserve(ctx, ctx->batch_out, bytes + 256));
	MC_TRY(pinned(ctx, bytes + 256));
	const BatchSlots d = batch_slots(ctx->batch_out.p, n_frames, max_objects);
	cudaEvent_t ev[3];
	if (stage_ms) for (int i = 0; i < 3; i++) MC_CUDA(cudaEventCreate(&ev[i]));
	MC_TRY(process_frames_device(ctx, d_q, d_qxy, d_qimg, frame_offsets, 0, n_frames, P, max_objects, nullptr, nullptr, d.info, d.model, d.pose, d.score,
	                             stage_ms ? ev : nullptr));
	MC_CUDA(cudaMemcpyAsync(ctx->h_pinned, ctx->batch_out.p, bytes, cudaMemcpyDeviceToHost, ctx->stream));
	MC_CUDA(cudaStreamSynchronize(ctx->stream));
	if (stage_ms) {
		cudaEventElapsedTime(&stage_ms[0], ev[0], ev[1]);
		cudaEventElapsedTime(&stage_ms[1], ev[1], ev[2]);
		for (int i = 0; i < 3; i++) cudaEventDestroy(ev[i]);
	}
	const BatchSlots h = batch_slots(ctx->h_pinned, n_frames, max_objects);
	int tot_m = 0, tot_o = 0;
	for (int f = 0; f < n_frames; f++) { tot_m += h.info[4 * f + 2]; tot_o += h.info[4 * f]; }
	ctx->batch_stats[1] = tot_m; ctx->batch_stats[2] = tot_o;
	int first_bad, first_over;
	unpack_batch(h, n_frames, max_objects, n_objects, obj_model, obj_pose, obj_score, frame_info, first_bad, first_over);
	if (first_bad >= 0) { ctx->err = "process_frames: more than 8192 accepted matches in one frame"; return MC_ERR_CAPACITY; }
	if (first_over >= 0) { ctx->err = "process_frames: object buffer too small"; return MC_ERR_CAPACITY; }
	return MC_OK;
}

void unpack_batch(const BatchSlots &h, int n_frames, int max_objects, int32_t *n_objects, int32_t *obj_model, float *obj_pose, float *obj_score,
                  int32_t *frame_info, int &first_bad, int &first_over) {
	first_bad = first_over = -1;
	for (int f = 0; f < n_frames; f++) {
		const int n = h.info[4 * f];
		if (frame_info) memcpy(frame_info + 4 * f, h.info + 4 * f, 16);
		n_objects[f] = n;
		if (h.info[4 * f + 1]) { if (first_bad < 0) first_bad = f; continue; }
		if (n > max_objects) { if (first_over < 0) first_over = f; continue; }
		const size_t at = (size_t)f * max_objects;
		memcpy(obj_model + at, h.model + at, 4ull * n);
		memcpy(obj_pose + 7 * at, h.pose + 7 * at, 28ull * n);
		memcpy(obj_score + at, h.score + at, 4ull * n);
	}
}

} // namespace mc
