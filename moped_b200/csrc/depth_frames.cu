// depth_frames.cu — moped3d's recognition steps chained on the device (mc_process_depth_frames*): the FrameData of a frame after
// DEPTHPROP goes CLUSTER (CLUSTER_LINKAGE) -> POSE -> FILTER -> POSE2 -> FILTER2 (moped3d/libmoped/src/config.hpp:45-49) with the
// per-match arrays and depth maps copied to the device once and the objects copied back once.
//
// Every step is the kernel of its stage-by-stage entry, so a frame gives exactly what mc_cluster_linkage (per model),
// mc_pose_depth_ransac (tie = match index inside the model, as pose_depth_cuda_base.hpp passes it) and mc_filter_projection give:
//   CLUSTER  the linkage kernels of linkage.cu over all models of the frame at once (one launch per kernel, one agglomeration CTA
//            per model), then the clusters model-major (k_link_compact)
//   POSE     k_gather_points with depthData.coord3D and the Cauchy weight of depthData.fillDistance, k_depth_ransac reading the
//            cluster count from the device (grid and LM scratch sized by host upper bounds), k_pose_append
//   FILTER   filter_device (moped3d's FILTER_PROJECTION_CPU is moped2's), or filter_depth_device (FILTER_PROJECTION_DEPTH) with the
//            calling context's test points (mc_set_depth_filter) and the frame's own depth and ".distance" planes
//   POSE2    the survivors stay in the object list (k_copy_objects), new objects from their rebuilt clusters are appended
// No host synchronisation between the steps: counts stay on the device. The frames of a batch are dealt to the context's frame
// lanes (pipeline.cu), each of which owns its buffers.
#include "common.cuh"

#include <algorithm>
#include <cstring>

namespace mc {

mc_status pose_depth_ransac_device(mc_ctx *ctx, int variant, const int32_t *d_cluster_offsets, int n_clusters, int n_max, const float *d_xy,
                                   const float *d_xyz, const float *d_world, const float *d_cauchy, const int32_t *d_image, const int32_t *d_tie,
                                   const mc_pose_params *pp, float alpha, uint8_t *d_found, float *d_pose, int32_t *d_n_tests,
                                   const int32_t *d_n_clusters);
mc_status pose_append_device(mc_ctx *ctx, const int32_t *d_cluster_model, const int32_t *d_n_clusters, int n_clusters_cap, int max_obj,
                             const uint8_t *d_found, const float *d_pose, int32_t *d_n_obj, int obj_cap, int32_t *d_obj_model, float *d_obj_pose);
mc_status filter_device(mc_ctx *ctx, const int32_t *d_match_offsets, const int32_t *d_match_image, const float *d_match_xy,
                        const float *d_match_xyz, int n_models, int max_matches, const int32_t *d_obj_model, const float *d_obj_pose,
                        const int32_t *d_n_obj, int n_obj_cap, int min_points, float feat_dist, float min_score,
                        uint8_t *d_keep, float *d_score, int32_t *d_out_n, int32_t *d_cluster_model, int32_t *d_cluster_offsets,
                        int32_t *d_members, int32_t *d_surv_model, float *d_surv_pose, float *d_surv_score);
mc_status filter_depth_device(mc_ctx *ctx, const int32_t *d_match_offsets, const int32_t *d_match_image, const float *d_match_xy,
                              const float *d_match_xyz, int n_models, int max_matches, const int32_t *d_obj_model, const float *d_obj_pose,
                              const int32_t *d_n_obj, int n_obj_cap, int min_points, float feat_dist, float min_score,
                              const int32_t *d_test_offsets, const float *d_test_xyz, const float *depth_K4, const float *depth_TM12, int width,
                              int height, const float *d_depth, const float *d_fill, float plausible_dist, float depth_fraction,
                              float min_keypoint_fraction, uint8_t *d_keep, float *d_score, int32_t *d_out_n, int32_t *d_cluster_model,
                              int32_t *d_cluster_offsets, int32_t *d_members, int32_t *d_surv_model, float *d_surv_pose, float *d_surv_score);

// sum over a frame's models of n^2: the five similarity matrices and the merge lists of the linkage take 24 bytes per element,
// so 2^24 elements are ~400 MB per lane (several models of the 2048-match limit of mc_cluster_linkage)
constexpr int64_t kLinkArenaMax = (int64_t)1 << 24;
constexpr int kMaxModelMatches = 2048;

__global__ void k_depth_export(const int32_t *__restrict__ st /* {status, n_obj, cl_n[2], f_n[2]} */, int n_matches,
                               const int32_t *__restrict__ surv_model, const float *__restrict__ surv_pose, const float *__restrict__ surv_score,
                               int max_objects, int32_t *__restrict__ out_info, int32_t *__restrict__ out_model, float *__restrict__ out_pose,
                               float *__restrict__ out_score) {
	const int n = st[4];
	const int m = n < max_objects ? n : max_objects;
	for (int i = threadIdx.x; i < m; i += blockDim.x) { out_model[i] = surv_model[i]; out_score[i] = surv_score[i]; }
	for (int i = threadIdx.x; i < 7 * m; i += blockDim.x) out_pose[i] = surv_pose[i];
	if (threadIdx.x == 0) { out_info[0] = n; out_info[1] = st[0]; out_info[2] = n_matches; out_info[3] = st[2]; }
}

// host view of one frame of a batch
struct DepthPlan {
	int base, M;                 // global index of the frame's first match, its match count
	int n_slices, n_max;         // models with matches, the largest
	int64_t sq;                  // sum of n^2 over its models
	int cl_cap;                  // clusters <= sum over models of n / (min_pts + 1)
	size_t meta;                 // offset of its local offsets (n_models + 1) and LinkSlices in the metadata buffer
};

struct DepthInputs { const int32_t *image; const float *xy, *xyz, *world, *fill, *depth, *distance; };     // device, whole batch

struct DepthCaps { int cl_cap, cl2_cap, obj_cap, task_cap; };

static DepthCaps depth_caps(const DepthPlan &p, const mc_depth_pipeline_params *P) {
	const int mo1 = std::max(P->pose.max_objects_per_cluster, 0), mo2 = std::max(P->pose2.max_objects_per_cluster, 0);
	DepthCaps c;
	c.cl_cap = p.cl_cap;
	c.cl2_cap = p.cl_cap * mo1;                      // FILTER keeps at most the objects of POSE, one cluster each
	c.obj_cap = c.cl2_cap + c.cl2_cap * mo2;         // POSE2 appends to the survivors
	c.task_cap = std::max(c.cl_cap * mo1, c.cl2_cap * mo2);
	return c;
}

struct DepthBufs {
	int32_t *st;                 // {status, n_obj, cl_n[2], f_n[2]}
	int32_t *cl_model, *cl_offsets, *cl_members;
	float *pt_xy, *pt_xyz, *pt_world, *pt_cauchy; int32_t *pt_image, *pt_tie;
	uint8_t *found; float *task_pose; int32_t *n_tests;
	int32_t *obj_model; float *obj_pose, *obj_score; uint8_t *keep;
	int32_t *f_model, *f_offsets, *f_members, *surv_model; float *surv_pose, *surv_score;
};

static mc_status depth_carve(mc_ctx *lane, int M, const DepthCaps &caps, DepthBufs &B) {
	const size_t m1 = (size_t)M + 2, c2 = (size_t)caps.cl_cap + 2, o2 = (size_t)caps.obj_cap + 2, t1 = (size_t)caps.task_cap + 1;
	return carve_scratch(lane, lane->scratch[kScrDepthFrame], [&](Carve &c) {
		c.take(B.st, 16); c.take(B.cl_model, c2); c.take(B.cl_offsets, c2); c.take(B.cl_members, m1);
		c.take(B.pt_xy, 2 * m1); c.take(B.pt_xyz, 3 * m1); c.take(B.pt_world, 3 * m1); c.take(B.pt_cauchy, m1); c.take(B.pt_image, m1); c.take(B.pt_tie, m1);
		c.take(B.found, t1); c.take(B.task_pose, 7 * t1); c.take(B.n_tests, t1);
		c.take(B.obj_model, o2); c.take(B.obj_pose, 7 * o2); c.take(B.obj_score, o2); c.take(B.keep, o2);
		c.take(B.f_model, o2); c.take(B.f_offsets, o2); c.take(B.f_members, m1); c.take(B.surv_model, o2); c.take(B.surv_pose, 7 * o2); c.take(B.surv_score, o2);
	});
}

// Enqueue one frame on lane->stream; its objects go to the frame's output slots. `ev` (nullable, 6 events) brackets the five steps.
// `df`: the FILTER / FILTER2 settings of the calling context (a lane is a context of its own and holds none).
static mc_status depth_frame_enqueue(mc_ctx *lane, const DepthPlan &p, const char *d_meta, const DepthInputs &in, int f, int n_models, int W, int H,
                                     const mc_depth_pipeline_params *P, const DepthFilterTable *df, int max_objects, const BatchSlots &out,
                                     cudaEvent_t *ev) {
	mc_ctx *ctx = lane;
	cudaStream_t s = lane->stream;
	int32_t *o_info = out.info + 4 * (size_t)f;
	if (p.M == 0) {                                     // nothing to cluster: no objects
		MC_CUDA(cudaMemsetAsync(o_info, 0, 16, s));
		if (ev) for (int i = 0; i < 6; i++) MC_CUDA(cudaEventRecord(ev[i], s));
		return MC_OK;
	}
	const DepthCaps c = depth_caps(p, P);
	DepthBufs B;
	MC_TRY(depth_carve(lane, p.M, c, B));
	MC_TRY(reserve(lane, lane->link_buf, link_arena_bytes(p.sq, p.M, p.n_slices)));
	const int32_t *d_off = (const int32_t *)(d_meta + p.meta);                 // the frame's model CSR, from 0
	const size_t slice_at = (((size_t)n_models + 1) * 4 + 15) & ~(size_t)15;
	const int32_t *image = in.image + p.base;
	const float *xy = in.xy + 2 * (size_t)p.base, *xyz = in.xyz + 3 * (size_t)p.base, *world = in.world + 3 * (size_t)p.base, *fill = in.fill + p.base;
	const size_t px = (size_t)W * H;
	LinkFrame F;
	F.slices = (const LinkSlice *)(d_meta + p.meta + slice_at); F.n_slices = p.n_slices; F.n_max = p.n_max;
	F.xy = xy; F.xyz = xyz; F.world = world; F.depth = in.depth + (size_t)f * px; F.distance = in.distance + (size_t)f * px; F.W = W; F.H = H;
	F.status = B.st;
	link_carve(lane->link_buf.p, p.sq, p.M, p.n_slices, F);
	const float scale = P->variant == 1 ? (float)25.0 : (float)0.100;
	auto mark = [&](int i) { if (ev) cudaEventRecord(ev[i], s); };
	// the FILTER step: FILTER_PROJECTION, or FILTER_PROJECTION_DEPTH with the step's test points and the frame's planes (the penalty kernel
	// runs inside the step, so stage_ms counts it there)
	auto filter = [&](const DepthFilterTable &t, int min_points, float feat_dist, float min_score) {
		if (!t.d_offsets)
			return filter_device(lane, d_off, image, xy, xyz, n_models, p.M, B.obj_model, B.obj_pose, B.st + 1, c.obj_cap, min_points, feat_dist,
			                     min_score, B.keep, B.obj_score, B.st + 4, B.f_model, B.f_offsets, B.f_members, B.surv_model, B.surv_pose,
			                     B.surv_score);
		return filter_depth_device(lane, d_off, image, xy, xyz, n_models, p.M, B.obj_model, B.obj_pose, B.st + 1, c.obj_cap, min_points, feat_dist,
		                           min_score, t.d_offsets, t.d_xyz, t.K, t.TM, W, H, F.depth, F.distance, t.plausible_sq_distance, t.depth_fraction,
		                           t.min_keypoint_fraction, B.keep, B.obj_score, B.st + 4, B.f_model, B.f_offsets, B.f_members, B.surv_model,
		                           B.surv_pose, B.surv_score);
	};
	MC_CUDA(cudaMemsetAsync(B.st, 0, 64, s));
	mark(0);
	// CLUSTER
	MC_TRY(link_frame_device(lane, F, P->cluster_cutoff, P->cluster_min_pts, P->cluster_use_3d_filter, P->cluster_linkage_type, P->cluster_sigma_2d,
	                         P->cluster_sigma_3d));
	MC_TRY(link_compact_device(lane, F, B.st + 2, B.cl_model, B.cl_offsets, B.cl_members, B.st + 1));
	mark(1);
	// POSE
	MC_TRY(gather_depth_points_device(lane, B.st + 2, B.cl_model, B.cl_offsets, B.cl_members, d_off, image, xy, xyz, world, fill, scale, B.pt_xy,
	                                  B.pt_xyz, B.pt_world, B.pt_cauchy, B.pt_image, B.pt_tie));
	MC_TRY(pose_depth_ransac_device(lane, P->variant, B.cl_offsets, c.cl_cap, p.n_max, B.pt_xy, B.pt_xyz, B.pt_world, B.pt_cauchy, B.pt_image, B.pt_tie,
	                                &P->pose, P->pose_alpha, B.found, B.task_pose, B.n_tests, B.st + 2));
	MC_TRY(pose_append_device(lane, B.cl_model, B.st + 2, c.cl_cap, P->pose.max_objects_per_cluster, B.found, B.task_pose, B.st + 1, c.obj_cap,
	                          B.obj_model, B.obj_pose));
	mark(2);
	// FILTER
	MC_TRY(filter(df[0], P->filter_min_points, P->filter_feature_distance, P->filter_min_score));
	mark(3);
	// POSE2: the surviving objects stay in the list, the objects found on their rebuilt clusters are appended
	MC_TRY(copy_objects_device(lane, B.st + 4, B.surv_model, B.surv_pose, B.st + 1, B.obj_model, B.obj_pose));
	MC_TRY(gather_depth_points_device(lane, B.st + 4, B.f_model, B.f_offsets, B.f_members, d_off, image, xy, xyz, world, fill, scale, B.pt_xy,
	                                  B.pt_xyz, B.pt_world, B.pt_cauchy, B.pt_image, B.pt_tie));
	MC_TRY(pose_depth_ransac_device(lane, P->variant, B.f_offsets, c.cl2_cap, p.n_max, B.pt_xy, B.pt_xyz, B.pt_world, B.pt_cauchy, B.pt_image, B.pt_tie,
	                                &P->pose2, P->pose2_alpha, B.found, B.task_pose, B.n_tests, B.st + 4));
	MC_TRY(pose_append_device(lane, B.f_model, B.st + 4, c.cl2_cap, P->pose2.max_objects_per_cluster, B.found, B.task_pose, B.st + 1, c.obj_cap,
	                          B.obj_model, B.obj_pose));
	mark(4);
	// FILTER2
	MC_TRY(filter(df[1], P->filter2_min_points, P->filter2_feature_distance, P->filter2_min_score));
	mark(5);
	k_depth_export<<<1, 128, 0, s>>>(B.st, p.M, B.surv_model, B.surv_pose, B.surv_score, max_objects, o_info, out.model + (size_t)f * max_objects,
	                                 out.pose + 7 * (size_t)f * max_objects, out.score + (size_t)f * max_objects);
	MC_LAUNCH_CHECK();
	return MC_OK;
}

static mc_status depth_params_check(mc_ctx *ctx, const char *who, const mc_depth_pipeline_params *P, int n_models) {
	auto fail = [&](mc_status st, const std::string &msg) { ctx->err = std::string(who) + ": " + msg; return st; };
	if (P->variant < 0 || P->variant > 1) return fail(MC_ERR_ARG, "variant must be 0 (back-projection) or 1 (reprojection)");
	// with cutoff <= -1 the merge loop has no stopping point once a single cluster is left (the reference then spins on the host)
	if (!(P->cluster_cutoff > -1.f)) return fail(MC_ERR_ARG, "cluster_cutoff must be > -1");
	if (P->pose.n_pts_align < 1 || P->pose.n_pts_align > 8 || P->pose2.n_pts_align < 1 || P->pose2.n_pts_align > 8)
		return fail(MC_ERR_ARG, "n_pts_align must be in 1..8");
	for (int s = 0; s < 2; s++) {
		const DepthFilterTable &t = ctx->depth_filter[s];
		if (t.d_offsets && t.n_models != n_models)
			return fail(MC_ERR_ARG, std::string(s ? "FILTER2" : "FILTER") + "'s depth-filter test points cover " + std::to_string(t.n_models) +
			                            " models, the call has " + std::to_string(n_models) + " (mc_set_depth_filter)");
	}
	return MC_OK;
}

// Checks on the host, then plans every frame and lays out the metadata (per frame: local CSR, LinkSlices). Returns the number of
// matches the per-match arrays must hold. frame_status (nullable): a frame over the chain's limits (a model with more than 2048
// matches, or more than 2^24 similarity entries) gets status 4 and an empty plan instead of failing the call.
static mc_status depth_plan(mc_ctx *ctx, const char *who, const int32_t *match_offsets, int n_frames, int n_models, int width, int height,
                            const mc_depth_pipeline_params *P, int max_objects, std::vector<DepthPlan> &plans, std::vector<char> &meta, int *m_total,
                            int32_t *frame_status = nullptr) {
	auto fail = [&](mc_status st, const std::string &msg) { ctx->err = std::string(who) + ": " + msg; return st; };
	if (!match_offsets || n_frames < 1 || n_models < 1 || width < 1 || height < 1 || max_objects <= 0) return fail(MC_ERR_ARG, "bad argument");
	MC_TRY(depth_params_check(ctx, who, P, n_models));
	const int per_cl = P->cluster_min_pts + 1 > 1 ? P->cluster_min_pts + 1 : 1;     // a cluster has more than min_pts members
	plans.assign((size_t)n_frames, DepthPlan());
	meta.clear();
	int mt = 0;
	for (int f = 0; f < n_frames; f++) {
		const int32_t *row = match_offsets + (size_t)f * (n_models + 1);
		DepthPlan &p = plans[(size_t)f];
		if (row[0] < 0) return fail(MC_ERR_ARG, "match_offsets must be >= 0 (frame " + std::to_string(f) + ")");
		p.base = row[0]; p.M = 0; p.n_slices = 0; p.n_max = 0; p.sq = 0; p.cl_cap = 0;
		std::vector<LinkSlice> sl;
		bool over = false;
		for (int m = 0; m < n_models; m++) {
			const int n = row[m + 1] - row[m];
			if (n < 0) return fail(MC_ERR_ARG, "match_offsets must ascend (frame " + std::to_string(f) + ")");
			if (n > kMaxModelMatches) {
				if (!frame_status) return fail(MC_ERR_ARG, "a model has more than 2048 matches (frame " + std::to_string(f) + ")");
				over = true;
			}
			if (n == 0) continue;
			sl.push_back(LinkSlice{ p.sq, row[m] - row[0], n, m, 0 });
			p.sq += (int64_t)n * n;
			p.n_max = std::max(p.n_max, n);
			p.cl_cap += n / per_cl;
		}
		if (p.sq > kLinkArenaMax) {
			if (!frame_status) return fail(MC_ERR_CAPACITY, "the models of frame " + std::to_string(f) + " need more than 2^24 similarity entries");
			over = true;
		}
		p.M = row[n_models] - row[0];
		if (over) {                                       // nothing of this frame runs
			frame_status[f] = 4;
			sl.clear();
			p.M = 0; p.n_max = 0; p.sq = 0; p.cl_cap = 0;
		}
		p.n_slices = (int)sl.size();
		mt = std::max(mt, (int)row[n_models]);
		p.meta = meta.size();
		const size_t slice_at = (((size_t)n_models + 1) * 4 + 15) & ~(size_t)15;
		meta.resize(p.meta + ((slice_at + sizeof(LinkSlice) * sl.size() + 255) & ~(size_t)255));
		int32_t *loc = (int32_t *)(meta.data() + p.meta);
		for (int m = 0; m <= n_models; m++) loc[m] = over ? 0 : row[m] - row[0];
		if (!sl.empty()) memcpy(meta.data() + p.meta + slice_at, sl.data(), sizeof(LinkSlice) * sl.size());
	}
	if (!ctx->d_cams) return fail(MC_ERR_STATE, "cameras not set (mc_set_cameras)");
	*m_total = mt;
	return MC_OK;
}

// span (nullable, 2 events): recorded on ctx->stream at the fork to the lanes and after their join; unlike stage_ms, it leaves the
// frames dealt to the lanes
static mc_status depth_frames_run(mc_ctx *ctx, const char *who, const std::vector<DepthPlan> &plans, const std::vector<char> &meta,
                                  const DepthInputs &in, int n_models, int W, int H, const mc_depth_pipeline_params *P, int max_objects,
                                  int32_t *n_objects, int32_t *obj_model, float *obj_pose, float *obj_score, int32_t *frame_info, float *stage_ms,
                                  cudaEvent_t *span = nullptr) {
	const int nf = (int)plans.size();
	MC_TRY(reserve(ctx, ctx->scratch[kScrDepthMeta], meta.size() + 256));
	char *d_meta = (char *)ctx->scratch[kScrDepthMeta].p;
	MC_CUDA(cudaMemcpyAsync(d_meta, meta.data(), meta.size(), cudaMemcpyHostToDevice, ctx->stream));
	const size_t bytes = batch_slots_bytes(nf, max_objects);
	MC_TRY(reserve(ctx, ctx->batch_out, bytes + 256));
	MC_TRY(pinned(ctx, bytes + 256));
	const BatchSlots d = batch_slots(ctx->batch_out.p, nf, max_objects);
	int n_lanes = stage_ms ? 1 : std::min(std::max(ctx->n_lanes_wanted, 1), nf);
	MC_TRY(ensure_lanes(ctx, n_lanes));
	for (int l = 0; l < n_lanes; l++) { ctx->lanes[(size_t)l]->linkage_cached = ctx->linkage_cached; ctx->lanes[(size_t)l]->lm_finite_check = ctx->lm_finite_check; }
	std::vector<cudaEvent_t> ev;
	if (stage_ms) {
		ev.resize(6 * (size_t)nf);
		for (auto &e : ev) MC_CUDA(cudaEventCreate(&e));
	}
	if (span) MC_CUDA(cudaEventRecord(span[0], ctx->stream));
	MC_CUDA(cudaEventRecord(ctx->ev_fork, ctx->stream));
	for (int l = 0; l < n_lanes; l++) MC_CUDA(cudaStreamWaitEvent(ctx->lanes[(size_t)l]->stream, ctx->ev_fork, 0));
	if (n_lanes > ctx->lanes_pending) ctx->lanes_pending = n_lanes;
	mc_status st = MC_OK;
	for (int f = 0; f < nf && st == MC_OK; f++) {
		mc_ctx *lane = ctx->lanes[(size_t)(f % n_lanes)];
		st = depth_frame_enqueue(lane, plans[(size_t)f], d_meta, in, f, n_models, W, H, P, ctx->depth_filter, max_objects, d,
		                         stage_ms ? &ev[6 * (size_t)f] : nullptr);
		if (st != MC_OK) ctx->err = lane->err;
	}
	const mc_status sj = join_lanes(ctx);
	if (st == MC_OK) st = sj;
	if (st == MC_OK && span) MC_CUDA(cudaEventRecord(span[1], ctx->stream));
	if (st == MC_OK) {
		MC_CUDA(cudaMemcpyAsync(ctx->h_pinned, ctx->batch_out.p, bytes, cudaMemcpyDeviceToHost, ctx->stream));
		MC_CUDA(cudaStreamSynchronize(ctx->stream));
	}
	if (stage_ms) {
		if (st == MC_OK) {
			for (int i = 0; i < 5; i++) stage_ms[i] = 0.f;
			for (int f = 0; f < nf; f++)
				for (int i = 0; i < 5; i++) { float ms = 0.f; cudaEventElapsedTime(&ms, ev[6 * (size_t)f + i], ev[6 * (size_t)f + i + 1]); stage_ms[i] += ms; }
		}
		for (auto &e : ev) cudaEventDestroy(e);
	}
	if (st != MC_OK) return st;
	int bad_frame, over_frame;
	unpack_batch(batch_slots(ctx->h_pinned, nf, max_objects), nf, max_objects, n_objects, obj_model, obj_pose, obj_score, frame_info, bad_frame,
	             over_frame);
	if (bad_frame >= 0) { ctx->err = std::string(who) + ": a match of frame " + std::to_string(bad_frame) + " lies outside the depth map"; return MC_ERR_ARG; }
	if (over_frame >= 0) { ctx->err = std::string(who) + ": frame " + std::to_string(over_frame) + " has more than max_objects objects"; return MC_ERR_CAPACITY; }
	return MC_OK;
}

// ---- moped3d from features to objects (mc_process_depth_queries*) ----------------------------------------------------------------
// MATCH (adaptive.cu) for frames [frame_begin, frame_end), its compaction also gathering DEPTHPROP's per-feature depth data per match,
// into context scratch (global feature ids, as MATCH writes them); the one synchronisation of MATCH brings the offsets and the frame
// flags to the host for the chain's plan; then the chain on the frame lanes. `dev` = false: the host inputs are uploaded first (the
// range is then the whole batch). frame_info status: 1 a match outside the depth map, 2 a row outside the tables, 3 more than 8192
// accepted matches, 4 over the chain's per-frame limits; such a frame gets no objects (with 2, 3 or 4 the chain does not run for it).
static mc_status depth_queries(mc_ctx *ctx, bool dev, const char *who, const RowSource &src, const float *q_xy, const int32_t *q_image,
                               const float *q_world, const float *q_fill, const int32_t *frame_offsets, int n_frames, int frame_begin,
                               int frame_end, const float *depth, const float *fill_distance, int width, int height,
                               const mc_adaptive_model *models, int n_models, float maximum_depth, float default_depth, float cauchy_scale,
                               const mc_depth_pipeline_params *P, int max_objects, int32_t *n_objects, int32_t *obj_model, float *obj_pose,
                               float *obj_score, int32_t *frame_info, float *stage_ms) {
	if (!ctx) return MC_ERR_ARG;
	auto fail = [&](mc_status st, const std::string &msg) { ctx->err = std::string(who) + ": " + msg; return st; };
	if (!P || !n_objects || !obj_model || !obj_pose || !obj_score || max_objects <= 0 || !frame_offsets || n_frames < 1 || n_models < 1 ||
	    width < 1 || height < 1 || !depth || !fill_distance)
		return fail(MC_ERR_ARG, "bad argument");
	if (frame_begin < 0 || frame_begin > frame_end || frame_end > n_frames) return fail(MC_ERR_ARG, "frame range outside 0..n_frames");
	if (frame_offsets[0] != 0) return fail(MC_ERR_ARG, "frame_offsets[0] must be 0");
	for (int f = 0; f < n_frames; f++)
		if (frame_offsets[f + 1] < frame_offsets[f]) return fail(MC_ERR_ARG, "frame_offsets do not ascend");
	const int Q = frame_offsets[n_frames], n_range = frame_end - frame_begin;
	const bool any = frame_offsets[frame_end] > frame_offsets[frame_begin];
	if (any && (!q_xy || !q_world || !q_fill || (!dev && !src.q_desc))) return fail(MC_ERR_ARG, "bad argument");
	MC_TRY(depth_params_check(ctx, who, P, n_models));
	if (!ctx->d_cams) return fail(MC_ERR_STATE, "cameras not set (mc_set_cameras)");
	MC_CUDA(cudaSetDevice(ctx->device));
	// per match (capacity Q, global ids): feature, image, xy, xyz, world, fill; the host entry's inputs behind them
	const size_t planes = (size_t)width * height * n_range, q = (size_t)Q;
	int32_t *m_feat, *m_img; float *m_xy, *m_xyz, *m_world, *m_fill, *up_qw = nullptr, *up_qf = nullptr, *up_depth = nullptr, *up_fill = nullptr;
	MC_TRY(carve_scratch(ctx, ctx->scratch[kScrDepthQueries], [&](Carve &c) {
		c.take(m_feat, q); c.take(m_img, q); c.take(m_xy, 2 * q); c.take(m_xyz, 3 * q); c.take(m_world, 3 * q); c.take(m_fill, q);
		if (!dev) { c.take(up_qw, 3 * q); c.take(up_qf, q); c.take(up_depth, planes); c.take(up_fill, planes); }
	}));
	RowSource rs = src;
	const float *d_xy = q_xy, *d_qw = q_world, *d_qf = q_fill, *d_depth = depth, *d_fill = fill_distance;
	const int32_t *d_img = q_image;
	if (!dev) {
		cudaStream_t s = ctx->stream;
		if (Q > 0) {
			MC_TRY(reserve(ctx, ctx->q_desc, sizeof(float) * (size_t)Q * ctx->D));
			MC_TRY(reserve(ctx, ctx->q_xy, 8ull * Q));
			MC_CUDA(cudaMemcpyAsync(ctx->q_desc.p, src.q_desc, sizeof(float) * (size_t)Q * ctx->D, cudaMemcpyHostToDevice, s));
			MC_CUDA(cudaMemcpyAsync(ctx->q_xy.p, q_xy, 8ull * Q, cudaMemcpyHostToDevice, s));
			MC_CUDA(cudaMemcpyAsync(up_qw, q_world, 12ull * Q, cudaMemcpyHostToDevice, s));
			MC_CUDA(cudaMemcpyAsync(up_qf, q_fill, 4ull * Q, cudaMemcpyHostToDevice, s));
			if (q_image) {
				MC_TRY(reserve(ctx, ctx->q_image, 4ull * Q));
				MC_CUDA(cudaMemcpyAsync(ctx->q_image.p, q_image, 4ull * Q, cudaMemcpyHostToDevice, s));
				d_img = (const int32_t *)ctx->q_image.p;
			}
		}
		MC_CUDA(cudaMemcpyAsync(up_depth, depth, 4 * planes, cudaMemcpyHostToDevice, s));
		MC_CUDA(cudaMemcpyAsync(up_fill, fill_distance, 4 * planes, cudaMemcpyHostToDevice, s));
		rs.q_desc = (const float *)ctx->q_desc.p; d_xy = (const float *)ctx->q_xy.p;
		d_qw = up_qw; d_qf = up_qf; d_depth = up_depth; d_fill = up_fill;
	}
	DepthInputs in;
	in.image = m_img; in.xy = m_xy; in.xyz = m_xyz; in.world = m_world; in.fill = m_fill; in.depth = d_depth; in.distance = d_fill;
	struct Events {                                     // MATCH start / end, chain fork / join (stage_ms)
		cudaEvent_t e[4] = {nullptr, nullptr, nullptr, nullptr};
		~Events() { for (cudaEvent_t x : e) if (x) cudaEventDestroy(x); }
	} ev;
	if (stage_ms) for (cudaEvent_t &x : ev.e) MC_CUDA(cudaEventCreate(&x));
	const size_t stride = (size_t)n_models + 1;
	// (at least one row each: MATCH takes a NULL array as an argument error, also for an empty range)
	const size_t rows = n_range > 0 ? (size_t)n_range : 1;
	std::vector<int32_t> moff(stride * rows), minfo(3 * rows, 0), status(rows, 0);
	const mc_status sm = match_adaptive_frames(ctx, true, who, rs, d_xy, d_img, frame_offsets, n_frames, frame_begin, frame_end, d_depth, d_fill, width,
	                                           height, models, n_models, maximum_depth, default_depth, cauchy_scale, moff.data(), m_feat, m_img, m_xy,
	                                           m_xyz, nullptr, nullptr, nullptr, minfo.data(), d_qw, d_qf, m_world, m_fill, stage_ms ? ev.e : nullptr);
	bool match_failed = false;                          // frames MATCH left empty (its status 2, or 1 = over its cap)
	for (int f = 0; f < n_range; f++)
		if (minfo[3 * (size_t)f + 2]) { status[(size_t)f] = minfo[3 * (size_t)f + 2] == 2 ? 2 : 3; match_failed = true; }
	if (sm != MC_OK && !match_failed) return sm;
	if (n_range == 0) return MC_OK;
	std::vector<DepthPlan> plans;
	std::vector<char> meta;
	std::vector<int32_t> plan_status((size_t)n_range, 0);
	int M = 0;
	MC_TRY(depth_plan(ctx, who, moff.data(), n_range, n_models, width, height, P, max_objects, plans, meta, &M, plan_status.data()));
	std::vector<int32_t> info(4 * (size_t)n_range);
	const mc_status sc = depth_frames_run(ctx, who, plans, meta, in, n_models, width, height, P, max_objects, n_objects, obj_model, obj_pose, obj_score,
	                                      info.data(), nullptr, stage_ms ? ev.e + 2 : nullptr);
	if (sc != MC_OK && sc != MC_ERR_ARG && sc != MC_ERR_CAPACITY) return sc;
	int first_arg = -1, first_cap = -1;
	for (int f = 0; f < n_range; f++) {
		int32_t *fi = info.data() + 4 * (size_t)f;
		if (plan_status[(size_t)f]) status[(size_t)f] = 4;
		if (status[(size_t)f]) {                         // nothing ran after MATCH: no objects, no clusters
			const int32_t *row = moff.data() + (size_t)f * stride;
			fi[0] = 0; fi[1] = status[(size_t)f]; fi[2] = row[n_models] - row[0]; fi[3] = 0;
		}
		const int s = fi[1];
		if ((s == 1 || s == 2) && first_arg < 0) first_arg = f;
		if ((s == 3 || s == 4 || (s == 0 && fi[0] > max_objects)) && first_cap < 0) first_cap = f;
	}
	if (frame_info) memcpy(frame_info, info.data(), 16 * (size_t)n_range);
	if (stage_ms) {
		stage_ms[0] = stage_ms[1] = 0.f;
		if (any) MC_CUDA(cudaEventElapsedTime(&stage_ms[0], ev.e[0], ev.e[1]));
		if (sc == MC_OK || first_arg >= 0 || first_cap >= 0) MC_CUDA(cudaEventElapsedTime(&stage_ms[1], ev.e[2], ev.e[3]));
	}
	const std::string frame = "frame " + std::to_string(frame_begin + (first_arg >= 0 ? first_arg : first_cap));
	if (first_arg >= 0)
		return fail(MC_ERR_ARG, info[4 * (size_t)first_arg + 1] == 1 ? "a match of " + frame + " lies outside the depth map"
		                                                             : frame + " has a nearest row outside the database tables");
	if (first_cap >= 0) {
		const int s = info[4 * (size_t)first_cap + 1];
		return fail(MC_ERR_CAPACITY, frame + (s == 3   ? " has more than " + std::to_string(kCompactCap) + " accepted matches"
		                                      : s == 4 ? " has a model with more than 2048 matches or needs more than 2^24 similarity entries"
		                                               : " has more than max_objects objects"));
	}
	return sc;
}

} // namespace mc

using namespace mc;

extern "C" {

void mc_depth_pipeline_default_params(mc_depth_pipeline_params *p) {
	if (!p) return;
	memset(p, 0, sizeof *p);
	p->variant = 0;
	p->cluster_cutoff = 0.1f; p->cluster_min_pts = 7; p->cluster_use_3d_filter = 2; p->cluster_linkage_type = 1;   // CLUSTER_LINKAGE(0.1, 7, 2, 1, 0.0, 1, -1, -1)
	p->cluster_sigma_2d = -1.f; p->cluster_sigma_3d = -1.f;
	p->pose = mc_pose_params{ 192, 100, 4, 5, 6, 8.f, 1 }; p->pose_alpha = 0.5f;          // POSE(192, 100, 4, 5, 6, 8, 0.5)
	p->filter_min_points = 6; p->filter_feature_distance = 4096.f; p->filter_min_score = 2.f;     // FILTER(6, 4096, 2)
	p->pose2 = mc_pose_params{ 64, 250, 4, 6, 8, 5.f, 2 }; p->pose2_alpha = 0.5f;          // POSE2(64, 250, 4, 6, 8, 5, 0.5)
	p->filter2_min_points = 8; p->filter2_feature_distance = 8192.f; p->filter2_min_score = 1e-4f;  // FILTER2(8, 8192, 1e-4)
}

mc_status mc_set_depth_filter(mc_ctx *ctx, int step, const mc_depth_filter_params *p, const int32_t *test_offsets, const float *test_xyz,
                              int n_models) {
	if (!ctx) return MC_ERR_ARG;
	auto fail = [&](const std::string &msg) { ctx->err = "mc_set_depth_filter: " + msg; return MC_ERR_ARG; };
	if (step < 0 || step > 1) return fail("step must be 0 (FILTER) or 1 (FILTER2)");
	if (p) {                                            // everything is checked before the current setting is touched
		if (n_models < 1 || !test_offsets) return fail("bad argument");
		if (test_offsets[0] != 0) return fail("test_offsets must start at 0");
		for (int m = 0; m < n_models; m++)
			if (test_offsets[m + 1] < test_offsets[m]) return fail("test_offsets must ascend");
		if (test_offsets[n_models] > 0 && !test_xyz) return fail("test_xyz is NULL");
	}
	MC_CUDA(cudaSetDevice(ctx->device));
	MC_CUDA(cudaStreamSynchronize(ctx->stream));       // the chain's last frames may still read the current table
	DepthFilterTable t;
	if (p) {                                            // copied once, into memory of its own (12 bytes per test point)
		const size_t n_pts = (size_t)test_offsets[n_models];
		cudaError_t e = cudaMalloc(&t.d_offsets, 4 * ((size_t)n_models + 1));
		if (e == cudaSuccess) e = cudaMalloc(&t.d_xyz, 12 * std::max(n_pts, (size_t)1));
		if (e == cudaSuccess) e = cudaMemcpyAsync(t.d_offsets, test_offsets, 4 * ((size_t)n_models + 1), cudaMemcpyHostToDevice, ctx->stream);
		if (e == cudaSuccess && n_pts) e = cudaMemcpyAsync(t.d_xyz, test_xyz, 12 * n_pts, cudaMemcpyHostToDevice, ctx->stream);
		if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
		if (e != cudaSuccess) {
			cudaFree(t.d_offsets); cudaFree(t.d_xyz);
			ctx->err = std::string("mc_set_depth_filter: ") + cudaGetErrorString(e);
			return MC_ERR_CUDA;
		}
		t.n_models = n_models;
		t.plausible_sq_distance = p->plausible_sq_distance; t.depth_fraction = p->depth_fraction; t.min_keypoint_fraction = p->min_keypoint_fraction;
		for (int i = 0; i < 4; i++) t.K[i] = p->depth_K[i];
		pose_tm(p->depth_pose, t.TM);                   // as mc_filter_projection_depth: the same bits
	}
	DepthFilterTable &cur = ctx->depth_filter[step];
	cudaFree(cur.d_offsets); cudaFree(cur.d_xyz);
	cur = t;
	return MC_OK;
}

mc_status mc_process_depth_frames(mc_ctx *ctx, const int32_t *match_offsets, int n_frames, int n_models, const int32_t *match_image,
                                  const float *match_xy, const float *match_xyz, const float *match_world, const float *match_fill,
                                  const float *depth, const float *fill_distance, int width, int height, const mc_depth_pipeline_params *params,
                                  int max_objects, int32_t *n_objects, int32_t *obj_model, float *obj_pose, float *obj_score, int32_t *frame_info,
                                  float *stage_ms) {
	const char *who = "mc_process_depth_frames";
	if (!ctx) return MC_ERR_ARG;
	if (!params || !n_objects || !obj_model || !obj_pose || !obj_score || !depth || !fill_distance) { ctx->err = std::string(who) + ": bad argument"; return MC_ERR_ARG; }
	std::vector<DepthPlan> plans;
	std::vector<char> meta;
	int M = 0;
	MC_TRY(depth_plan(ctx, who, match_offsets, n_frames, n_models, width, height, params, max_objects, plans, meta, &M));
	if (M > 0 && (!match_image || !match_xy || !match_xyz || !match_world || !match_fill)) { ctx->err = std::string(who) + ": null match array"; return MC_ERR_ARG; }
	// the blend kernel reads the fill-distance map at every match's pixel unchecked (like the reference, CLUSTER_LINKAGE_CPU.hpp:324-365):
	// a coordinate outside the map is an argument error, found before anything is copied
	for (int f = 0; f < n_frames; f++) {
		const DepthPlan &p = plans[(size_t)f];
		for (int i = p.base; i < p.base + p.M; i++) {
			const float x = match_xy[2 * (size_t)i], y = match_xy[2 * (size_t)i + 1];
			if (!(x >= 0.f && y >= 0.f && (int)x < width && (int)y < height)) {
				ctx->err = std::string(who) + ": a match of frame " + std::to_string(f) + " lies outside the depth map";
				return MC_ERR_ARG;
			}
		}
	}
	MC_CUDA(cudaSetDevice(ctx->device));
	const size_t px = (size_t)width * height, Ms = (size_t)M + 1;
	int32_t *d_im; float *d_xy, *d_xyz, *d_w, *d_f, *d_d, *d_fd;
	MC_TRY(carve_scratch(ctx, ctx->scratch[kScrDepthFramesIn], [&](Carve &c) {
		c.take(d_im, Ms); c.take(d_xy, 2 * Ms); c.take(d_xyz, 3 * Ms); c.take(d_w, 3 * Ms); c.take(d_f, Ms);
		c.take(d_d, px * n_frames); c.take(d_fd, px * n_frames);
	}));
	cudaStream_t s = ctx->stream;
	if (M > 0) {
		MC_CUDA(cudaMemcpyAsync(d_im, match_image, 4ull * M, cudaMemcpyHostToDevice, s));
		MC_CUDA(cudaMemcpyAsync(d_xy, match_xy, 8ull * M, cudaMemcpyHostToDevice, s));
		MC_CUDA(cudaMemcpyAsync(d_xyz, match_xyz, 12ull * M, cudaMemcpyHostToDevice, s));
		MC_CUDA(cudaMemcpyAsync(d_w, match_world, 12ull * M, cudaMemcpyHostToDevice, s));
		MC_CUDA(cudaMemcpyAsync(d_f, match_fill, 4ull * M, cudaMemcpyHostToDevice, s));
	}
	MC_CUDA(cudaMemcpyAsync(d_d, depth, 4 * px * n_frames, cudaMemcpyHostToDevice, s));
	MC_CUDA(cudaMemcpyAsync(d_fd, fill_distance, 4 * px * n_frames, cudaMemcpyHostToDevice, s));
	const DepthInputs in = { d_im, d_xy, d_xyz, d_w, d_f, d_d, d_fd };
	return depth_frames_run(ctx, who, plans, meta, in, n_models, width, height, params, max_objects, n_objects, obj_model, obj_pose, obj_score,
	                        frame_info, stage_ms);
}

mc_status mc_process_depth_frames_dev(mc_ctx *ctx, const int32_t *match_offsets, int n_frames, int n_models, const int32_t *match_image_dev,
                                      const float *match_xy_dev, const float *match_xyz_dev, const float *match_world_dev, const float *match_fill_dev,
                                      const float *depth_dev, const float *fill_distance_dev, int width, int height,
                                      const mc_depth_pipeline_params *params, int max_objects, int32_t *n_objects, int32_t *obj_model, float *obj_pose,
                                      float *obj_score, int32_t *frame_info, float *stage_ms) {
	const char *who = "mc_process_depth_frames_dev";
	if (!ctx) return MC_ERR_ARG;
	if (!params || !n_objects || !obj_model || !obj_pose || !obj_score || !depth_dev || !fill_distance_dev) { ctx->err = std::string(who) + ": bad argument"; return MC_ERR_ARG; }
	std::vector<DepthPlan> plans;
	std::vector<char> meta;
	int M = 0;
	MC_TRY(depth_plan(ctx, who, match_offsets, n_frames, n_models, width, height, params, max_objects, plans, meta, &M));
	if (M > 0 && (!match_image_dev || !match_xy_dev || !match_xyz_dev || !match_world_dev || !match_fill_dev)) {
		ctx->err = std::string(who) + ": null match array";
		return MC_ERR_ARG;
	}
	MC_CUDA(cudaSetDevice(ctx->device));
	DepthInputs in;
	in.image = match_image_dev; in.xy = match_xy_dev; in.xyz = match_xyz_dev; in.world = match_world_dev; in.fill = match_fill_dev;
	in.depth = depth_dev; in.distance = fill_distance_dev;
	return depth_frames_run(ctx, who, plans, meta, in, n_models, width, height, params, max_objects, n_objects, obj_model, obj_pose, obj_score,
	                        frame_info, stage_ms);
}

mc_status mc_process_depth_queries(mc_ctx *ctx, const float *q_desc, const float *q_xy, const int32_t *q_image, const float *q_world, const float *q_fill,
                                   const int32_t *frame_offsets, int n_frames, const float *depth, const float *fill_distance, int width, int height,
                                   const mc_adaptive_model *models, int n_models, float maximum_depth, float default_depth, float cauchy_scale,
                                   const mc_depth_pipeline_params *params, int max_objects, int32_t *n_objects, int32_t *obj_model, float *obj_pose,
                                   float *obj_score, int32_t *frame_info, float *stage_ms) {
	const RowSource src = {q_desc, nullptr, 0};
	return depth_queries(ctx, false, "mc_process_depth_queries", src, q_xy, q_image, q_world, q_fill, frame_offsets, n_frames, 0, n_frames, depth,
	                     fill_distance, width, height, models, n_models, maximum_depth, default_depth, cauchy_scale, params, max_objects, n_objects,
	                     obj_model, obj_pose, obj_score, frame_info, stage_ms);
}

mc_status mc_process_depth_queries_dev(mc_ctx *ctx, const float *q_desc_dev, const float *q_xy_dev, const int32_t *q_image_dev,
                                       const float *q_world_dev, const float *q_fill_dev, const int32_t *frame_offsets, int n_frames,
                                       const float *depth_dev, const float *fill_distance_dev, int width, int height, const mc_adaptive_model *models,
                                       int n_models, float maximum_depth, float default_depth, float cauchy_scale,
                                       const mc_depth_pipeline_params *params, int max_objects, int32_t *n_objects, int32_t *obj_model,
                                       float *obj_pose, float *obj_score, int32_t *frame_info, float *stage_ms) {
	const RowSource src = {q_desc_dev, nullptr, 0};
	return depth_queries(ctx, true, "mc_process_depth_queries_dev", src, q_xy_dev, q_image_dev, q_world_dev, q_fill_dev, frame_offsets, n_frames, 0,
	                     n_frames, depth_dev, fill_distance_dev, width, height, models, n_models, maximum_depth, default_depth, cauchy_scale, params,
	                     max_objects, n_objects, obj_model, obj_pose, obj_score, frame_info, stage_ms);
}

mc_status mc_process_depth_queries_merged_dev(mc_ctx *ctx, const void *packed_all_dev, int n_shards, const float *q_xy_dev, const int32_t *q_image_dev,
                                              const float *q_world_dev, const float *q_fill_dev, const int32_t *frame_offsets, int n_frames,
                                              int frame_begin, int frame_end, const float *depth_dev, const float *fill_distance_dev, int width,
                                              int height, const mc_adaptive_model *models, int n_models, float maximum_depth, float default_depth,
                                              float cauchy_scale, const mc_depth_pipeline_params *params, int max_objects, int32_t *n_objects,
                                              int32_t *obj_model, float *obj_pose, float *obj_score, int32_t *frame_info, float *stage_ms) {
	if (ctx && (!packed_all_dev || n_shards < 1)) { ctx->err = "mc_process_depth_queries_merged_dev: bad argument"; return MC_ERR_ARG; }
	const RowSource src = {nullptr, (const int32_t *)packed_all_dev, n_shards};
	return depth_queries(ctx, true, "mc_process_depth_queries_merged_dev", src, q_xy_dev, q_image_dev, q_world_dev, q_fill_dev, frame_offsets, n_frames,
	                     frame_begin, frame_end, depth_dev, fill_distance_dev, width, height, models, n_models, maximum_depth, default_depth,
	                     cauchy_scale, params, max_objects, n_objects, obj_model, obj_pose, obj_score, frame_info, stage_ms);
}

} // extern "C"
