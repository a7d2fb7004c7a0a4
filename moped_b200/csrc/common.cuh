// common.cuh — shared declarations of libmoped_cuda (B200 / sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <string>
#include <vector>

#include "../../include/moped_cuda.h"

namespace mc {

// ---- sizes fixed by the tensor-core matcher -------------------------------------------------
constexpr int kD = 128;                 // descriptor length of the tcgen05 path (SIFT)
constexpr int kTileRows = 128;          // DB rows / query rows per operand tile image
constexpr int kTileBytes = kTileRows * kD * 2;   // 32 KiB: fp16, two 128B-swizzle K atoms of 64 elements
constexpr int kMTile = 256;             // queries per CTA (two 128-row halves)
#ifndef MC_TOPK
#define MC_TOPK 4
#endif
constexpr int kTopK = MC_TOPK;          // coarse candidates kept per (query, DB split) by the fp16 pass
#ifndef MC_TOPK8
#define MC_TOPK8 8
#endif
constexpr int kTopK8 = MC_TOPK8;               // ... by the 8-bit pass (its certificate charges a ~12x larger score error)
constexpr int kMaxSplits = 64;

struct Camera {            // FrameData::images[i]: K=(fx,fy,cx,cy), TM = 3x4 of cameraPose (moped.hpp:226-241)
	float K[4];
	float TM[12];
};

struct FrameDesc {         // what differs between the frames of a stream: read by the stage chain through ONE indirection,
	const int32_t *nn_row;      // so that the chain itself (a CUDA graph per lane) never changes
	const uint8_t *accepted;
	const float *q_xy;
	const int32_t *q_image;
	int32_t *out_info, *out_model;
	float *out_pose, *out_score;
	int Q, max_objects;
};

struct DevBuf {            // grow-only device scratch
	void *p = nullptr;
	size_t cap = 0;
};

// mc_ctx::scratch: one grow-only buffer per owner. The frame graphs (pipeline.cu) key on the address of every slot.
enum ScratchSlot : int {
	kScrClusterCount,         // cluster_device: per-model cluster counts
	kScrClusterSizes,         // cluster_device: cluster sizes
	kScrClusterMembers,       // cluster_device: cluster members
	kScrClusterF,             // cluster_device: per-match float state
	kScrClusterI,             // cluster_device: per-match int state
	kScrClusterList,          // cluster_device: the models to cluster and their count
	kScrFilterIn,             // filter_device: object x match inlier flags
	kScrFilterOwner,          // filter_device: owner of each match
	kScrFilterOwned,          // filter_device: matches owned per object
	kScrFilterRaw,            // filter_device, depth variant: scores before the depth penalty
	kScrFitStream,            // pose_hypotheses_device: counters of the persistent fit kernel
	kScrRefitLists,           // pose_hypotheses_device: refit buckets
	kScrRansac,               // ransac_staged_launch: RansacState
	kScrDepthLm,              // pose_depth.cu: per-warp LM work arrays
	kScrAdaptive,             // adaptive.cu: uploads and per-frame state of mc_match_adaptive and match_adaptive_frames
	kScrFrame,                // pipeline.cu carve: a frame's chain (FrameBufs)
	kScrDepthFrame,           // depth_frames.cu depth_carve: a frame's chain (DepthBufs)
	kScrDepthMeta,            // depth_frames_run: per-frame model CSR and LinkSlices
	kScrDepthFramesIn,        // mc_process_depth_frames: uploaded per-match arrays and depth maps
	kScrDepthQueries,         // depth_queries: per-match arrays of mc_process_depth_queries*
	kScrHostCluster,          // mc_cluster_meanshift
	kScrHostPose,             // mc_pose_hypotheses
	kScrHostRansac,           // mc_pose_ransac
	// the two entries of each pair below share one buffer: they never run at the same time on a context, and a caller that
	// alternates them reuses the larger allocation
	kScrHostPoseDepth,        // mc_pose_depth_hypotheses, mc_pose_depth_ransac
	kScrHostFilter,           // mc_filter_projection, mc_filter_projection_depth
	kScrUndistort,            // mc_undistort: the uploaded images and their undistorted copies
	kScratchSlots
};

// Consecutive arrays in one buffer, each on a 256-byte boundary. A layout is a callable that takes every array once, in order:
// run with base == nullptr it only sizes the buffer (the pointers it sets are null), run with a base it points each array into it.
struct Carve {
	char *base = nullptr;
	size_t off = 0;
	template <class T> void take(T *&p, size_t n) {
		p = base ? (T *)(base + off) : nullptr;
		off += (n * sizeof(T) + 255) & ~(size_t)255;
	}
};

// TransformMatrix::init(cameraPose) on the host (moped.hpp:175-182): the 3x4 matrix of a pose (quaternion x y z w, translation).
// One expression for every caller (mc_set_cameras, mc_filter_projection_depth, mc_set_depth_filter), so their bits agree.
inline void pose_tm(const float *pose, float *T) {
	const float *q = pose, *t = pose + 4;
	T[0] = 1 - 2 * q[1] * q[1] - 2 * q[2] * q[2]; T[1] = 2 * q[0] * q[1] - 2 * q[3] * q[2]; T[2] = 2 * q[0] * q[2] + 2 * q[3] * q[1]; T[3] = t[0];
	T[4] = 2 * q[0] * q[1] + 2 * q[3] * q[2]; T[5] = 1 - 2 * q[0] * q[0] - 2 * q[2] * q[2]; T[6] = 2 * q[1] * q[2] - 2 * q[3] * q[0]; T[7] = t[1];
	T[8] = 2 * q[0] * q[2] - 2 * q[3] * q[1]; T[9] = 2 * q[1] * q[2] + 2 * q[3] * q[0]; T[10] = 1 - 2 * q[0] * q[0] - 2 * q[1] * q[1]; T[11] = t[2];
}

// FILTER_PROJECTION_DEPTH for one filter step of the moped3d chain (mc_set_depth_filter): the test points on the device, owned by the
// context, and the step's parameters. d_offsets == nullptr: the step runs FILTER_PROJECTION.
struct DepthFilterTable {
	int32_t *d_offsets = nullptr;     // [n_models + 1], from 0
	float *d_xyz = nullptr;           // test points, model-major (at least one point's room)
	int n_models = 0;
	float plausible_sq_distance = 0.f, depth_fraction = 0.f, min_keypoint_fraction = 0.f;
	float K[4] = {0.f, 0.f, 0.f, 0.f}, TM[12] = {0.f};
};

// UNDISTORTED_IMAGE of one camera (mc_set_undistortion): a RemapEntry per pixel, then the 32 x 32 RemapWeights (undistort.cuh), in
// one device allocation the context owns. d_map == nullptr: no table.
constexpr int kUndistortCameras = 16;
struct UndistortTable {
	void *d_map = nullptr;
	int height = 0, width = 0;
};

} // namespace mc

struct mc_ctx {
	int device = 0;
	int num_sms = 148;
	cudaStream_t stream = nullptr;
	bool own_stream = false;
	std::string err;
	int64_t launches = 0;

	// model database (device resident)
	int64_t n_rows = 0, row_base = 0, n_tiles = 0;
	int D = 0, n_models = 0;
	float *d_db = nullptr;            // n_rows x D fp32, row-major (exact re-rank / exact scan)
	__half *d_db_img = nullptr;       // n_tiles x 32 KiB pre-swizzled fp16 operand tiles (tcgen05 B operand)
	uint8_t *d_db_img8 = nullptr;     // n_tiles x 16 KiB pre-swizzled u8 / s8 operand tiles, one scale for all rows
	float db_scale = 0.f;             // 8-bit image: q8 = round(db_scale * x); 0 = no usable image (empty / non-finite database)
	bool db_signed = false;           // 8-bit image holds s8 (some element is negative) instead of u8
	float db_err_max = 0.f;           // max over rows of |x - q8 / db_scale|_2
	float *d_xyz = nullptr;           // table_rows x 3 (coord3D of rows table_base .. table_base+table_rows)
	int32_t *d_model_of_row = nullptr;
	int64_t table_base = 0, table_rows = 0;   // = this shard's rows unless mc_db_set_global_tables was called
	float db_norm2_min = 1.f, db_norm2_max = 1.f;

	// cameras
	mc::Camera *d_cams = nullptr;
	int n_images = 0;

	// scratch
	mc::DevBuf q_desc, q_img, q_norm2, tau, cand_score, cand_row, flag_list, flag_count, nn_key;
	mc::DevBuf q_img8, q_signed, q_scale, q_err, flag_list2, tau2, cand_score2, cand_row2;   // 8-bit pass + fp16 second-chance pass
	int coarse_kind = 1;              // mc_set_option "match_coarse_kind": 1 = 8-bit pass first (default), 0 = fp16 pass only
	// spatial partition (sm_partition.cu, mc_set_option "stage_sm_partition"): green contexts, the stream the coarse kernel runs on
	void *green_match = nullptr, *green_stage = nullptr;
	cudaStream_t match_green_stream = nullptr;
	cudaEvent_t ev_green[2] = {nullptr, nullptr};
	int match_sms = 0, stage_sms = 0; // SMs of the two partitions (0 = no partition)
	int match_splits = 0;             // mc_set_option "match_splits": database splits per query tile in the coarse pass (0 = chosen from the grid)
	int match_stagger = 1;            // mc_set_option "match_stagger": CTAs of one DB split start at different tiles
	int match_reserve_sms = 0;        // mc_set_option "match_reserve_sms": SMs the persistent matching kernel leaves to concurrent work
	mc::DevBuf nn_row, nn_dist, accepted, q_xy, q_image;
	mc::DevBuf scratch[mc::kScratchSlots];
	void *h_pinned = nullptr; size_t h_pinned_cap = 0;
	int last_stats[4] = {0, 0, 0, 0};
	int last_match_q = 0, last_match_tensor = 0;   // queries / mode of the last match_device pass (mc_match_last_stats)
	bool profile = false;             // record CUDA events around the dominant kernel (k_match_coarse)
	cudaEvent_t ev_coarse[2] = {nullptr, nullptr};
	bool ev_valid = false;

	// frame batches (mc_process_frames*): the stages after MATCH of different frames run concurrently on
	// "lanes" — child contexts with their own stream and scratch that borrow this context's database tables
	// and cameras. A lane never owns the database.
	mc_ctx *parent = nullptr;
	std::vector<mc_ctx *> lanes;
	int n_lanes_wanted = 8;           // mc_set_tuning
	int pose_warps = 8;               // warps per RANSAC task CTA (mc_set_tuning); results do not depend on it
	int64_t fit_thread_min = 16384;   // mc_set_option: explicit-hypothesis calls with at least this many use one thread per hypothesis
	bool fit_stream = true;           // mc_set_option "pose_fit_stream": the persistent phase-synchronous one-thread-per-hypothesis kernel (0: k_pose_fit_thread)
	int ransac_shard_rank = 0, ransac_shard_world = 1;   // set around the RANSAC calls of mc_process_frame_sharded_dev (pose_staged.cuh)
	bool ransac_merge_levels = true;  // mc_set_option "ransac_merge_levels" (pose_staged.cuh)
	bool ransac_fused = false;        // mc_set_option: the one-CTA-per-task RANSAC kernel instead of the staged kernels (A/B aid)
	int depth_team_lanes = 32;        // mc_set_option: lanes per explicit hypothesis in k_depth_hypotheses (32 or 8)
	bool linkage_cached = true;       // mc_set_option: cached-row-maximum agglomeration (linkage_cached.cuh) for average linkage (0: the O(n^2)-scan kernel)
	bool pose_exact_order = false;    // mc_set_option: mc_pose_hypotheses / mc_pose_ransac run the order-preserving LM (pose_depth.cu, variant 2)
	bool lm_finite_check = false;     // mc_set_option: depth pose stages keep levmar's stop on a non-finite ||e||^2 (a strict-IEEE build of the reference)
	int match_chunks = 1;             // MATCH launches per batch (mc_set_tuning): chunk c+1 matches while chunk c runs its lanes
	cudaEvent_t ev_fork = nullptr, ev_done = nullptr;
	std::vector<cudaEvent_t> ev_chunk;
	mc::DevBuf batch_out;             // per-frame result slots of the running batch
	// per-lane CUDA graph of the stage chain CLUSTER..FILTER2 (+ compaction and export): replayed once per frame
	mc::DevBuf frame_desc;            // device copy of the current frame's FrameDesc
	struct FrameGraph { uint64_t cfg, ptr_key; cudaGraphExec_t exec; int nodes; };
	std::vector<FrameGraph> fgraphs;  // one per configuration seen on this lane (sizes, parameters), most recent last
	struct BatchGraph { uint64_t key; cudaGraphExec_t exec; int nodes; };
	std::vector<BatchGraph> bgraphs;  // one graph per batch configuration: the stage chains of all frames of a call as parallel branches (pipeline.cu)
	bool batch_graph = true;          // mc_set_option "batch_graph"
	bool capturing = false;           // reserve() must not allocate while the lane's stream is being captured
	bool frame_graphs = true;         // mc_set_option "frame_graphs"
	bool defer_lane_join = false;     // mc_set_option "defer_lane_join": mc_process_frames_matched_dev returns without ordering the context's
	                                  // stream after the lanes; mc_join_lanes does that later (MATCH of the next chunk overlaps this chunk's stages)
	int lanes_pending = 0;            // lanes used since the last join
	int batch_stats[4] = {0, 0, 0, 0};   // {frames, accepted matches, objects, lanes used} of the last batch
	mc::DevBuf link_buf;                 // linkage clustering (linkage.cu): inputs, similarity matrices, agglomeration state
	mc::DepthFilterTable depth_filter[2];   // FILTER / FILTER2 of mc_process_depth_frames* / _queries* (mc_set_depth_filter)
	void *sift_state = nullptr;          // feature extraction (sift.cu): scale-space plan and buffers, created on first use
	mc::UndistortTable undistort[mc::kUndistortCameras];   // per camera (mc_set_undistortion); camera c serves image c of a rig frame
};

namespace mc {

#define MC_CUDA(call)                                                                         \
	do {                                                                                      \
		cudaError_t e__ = (call);                                                             \
		if (e__ != cudaSuccess) {                                                             \
			ctx->err = std::string(#call) + ": " + cudaGetErrorString(e__);                   \
			return MC_ERR_CUDA;                                                               \
		}                                                                                     \
	} while (0)

#define MC_LAUNCH_CHECK()                                                                     \
	do {                                                                                      \
		ctx->launches++;                                                                      \
		cudaError_t e__ = cudaGetLastError();                                                 \
		if (e__ != cudaSuccess) {                                                             \
			ctx->err = std::string("kernel launch: ") + cudaGetErrorString(e__);              \
			return MC_ERR_CUDA;                                                               \
		}                                                                                     \
	} while (0)

#define MC_TRY(expr)                                                                          \
	do {                                                                                      \
		mc_status s__ = (expr);                                                               \
		if (s__ != MC_OK) return s__;                                                         \
	} while (0)

inline mc_status reserve(mc_ctx *ctx, DevBuf &b, size_t bytes) {
	if (bytes <= b.cap && b.p) return MC_OK;
	if (ctx->capturing) { ctx->err = "scratch allocation requested during graph capture"; return MC_ERR_STATE; }
	if (b.p) { MC_CUDA(cudaFree(b.p)); b.p = nullptr; b.cap = 0; }
	size_t cap = bytes < 256 ? 256 : bytes + bytes / 4;
	MC_CUDA(cudaMalloc(&b.p, cap));
	b.cap = cap;
	return MC_OK;
}

// Sizes `layout` (a Carve layout), grows b to fit it and points its arrays into b. Inside a graph capture a buffer that has to
// grow fails with MC_ERR_STATE (reserve) and no pointer is set.
template <class Layout> inline mc_status carve_scratch(mc_ctx *ctx, DevBuf &b, Layout &&layout) {
	Carve c;
	layout(c);
	MC_TRY(reserve(ctx, b, c.off));
	c = Carve{(char *)b.p};
	layout(c);
	return MC_OK;
}

inline mc_status pinned(mc_ctx *ctx, size_t bytes) {
	if (bytes <= ctx->h_pinned_cap) return MC_OK;
	if (ctx->h_pinned) { MC_CUDA(cudaFreeHost(ctx->h_pinned)); ctx->h_pinned = nullptr; ctx->h_pinned_cap = 0; }
	size_t cap = bytes + bytes / 4 + 4096;
	MC_CUDA(cudaMallocHost(&ctx->h_pinned, cap));
	ctx->h_pinned_cap = cap;
	return MC_OK;
}

// ---- stage entry points implemented in the .cu files (device pointers, async on ctx->stream) ----
mc_status db_build_images(mc_ctx *ctx);
mc_status match_configure_device(mc_ctx *ctx);
mc_status cluster_configure_device(mc_ctx *ctx);
mc_status sm_partition_create(mc_ctx *ctx, int stage_sms);
void sm_partition_destroy(mc_ctx *ctx);
mc_status sm_partition_stage_stream(mc_ctx *ctx, cudaStream_t *out, int priority);
void sift_free(mc_ctx *ctx);
mc_status sift_set_two_pass(mc_ctx *ctx, int on);
mc_status sift_set_gather(mc_ctx *ctx, int on);
mc_status sift_extract_device(mc_ctx *ctx, const uint8_t *d_gray, int B, int H, int W, int dbl, int max_kp,
                              float *d_xy, float *d_so, float *d_desc, int32_t *d_counts, int32_t *d_offsets, int match_normalise);
mc_status process_frames_host(mc_ctx *ctx, const float *d_q, const float *d_qxy, const int32_t *d_qimg, const int32_t *frame_offsets, int n_frames,
                              const mc_pipeline_params *P, int max_objects, int32_t *n_objects, int32_t *obj_model, float *obj_pose, float *obj_score,
                              int32_t *frame_info, float *stage_ms);
size_t frame_shard_slot_bytes(int Q, const mc_pipeline_params *P);
mc_status process_frame_sharded_device(mc_ctx *ctx, int phase, const int32_t *d_nn_row, const uint8_t *d_accepted, const float *d_qxy,
                                       const int32_t *d_qimg, int Q, const mc_pipeline_params *P, int shard_rank, int shard_world, void *d_exchange,
                                       int max_objects, int32_t *d_out_info, int32_t *d_out_model, float *d_out_pose, float *d_out_score);
// Camera rigs (undistort.cu). undistort_check_rig: has[c] = camera c has a table; MC_ERR_ARG when that table is not H[c] x W[c].
// undistort_rig_device: one launch for a batch of H x W images whose image b belongs to camera cameras[b % n_cameras] (at least one
// of them with a table).
mc_status undistort_check_rig(mc_ctx *ctx, const char *who, int n_cameras, const int *H, const int *W, bool *has);
mc_status undistort_rig_device(mc_ctx *ctx, const int *cameras, int n_cameras, const uint8_t *d_in, int B, int H, int W, uint8_t *d_out);
mc_status match_device(mc_ctx *ctx, const float *d_q, int Q, float ratio, int mode,
                       int32_t *d_nn_row, float *d_nn_dist, uint8_t *d_accepted);

// ---- frame lanes and chain pieces shared by the moped2 and moped3d frame chains (pipeline.cu) ----
mc_status ensure_lanes(mc_ctx *ctx, int n);
mc_status join_lanes(mc_ctx *ctx);
mc_status gather_depth_points_device(mc_ctx *ctx, const int32_t *d_n, const int32_t *d_cluster_model, const int32_t *d_cluster_offsets,
                                     const int32_t *d_members, const int32_t *d_match_offsets, const int32_t *d_match_image, const float *d_match_xy,
                                     const float *d_match_xyz, const float *d_match_world, const float *d_match_fill, float cauchy_scale, float *d_pt_xy,
                                     float *d_pt_xyz, float *d_pt_world, float *d_pt_cauchy, int32_t *d_pt_image, int32_t *d_pt_tie);
mc_status copy_objects_device(mc_ctx *ctx, const int32_t *d_n, const int32_t *d_src_model, const float *d_src_pose, int32_t *d_dst_n,
                              int32_t *d_dst_model, float *d_dst_pose);
mc_status match_compact_frames_device(mc_ctx *ctx, const FrameDesc *d_fd, const int32_t *d_out_base, int n_frames, int n_models, int32_t *d_acc_list,
                                      int32_t *d_match_offsets, int32_t *d_match_query, int32_t *d_match_row, int32_t *d_match_image,
                                      float *d_match_xy, float *d_match_xyz, int32_t *d_status, int32_t *d_n_obj,
                                      const float *d_q_world = nullptr, const float *d_q_fill = nullptr, float *d_match_world = nullptr,
                                      float *d_match_fill = nullptr);
constexpr int kCompactCap = 8192;    // accepted matches per frame handled by the compaction (k_match_compact)

// The result slots of a frame batch, on the device (ctx->batch_out) and in its pinned host copy: per frame info[4] = {objects,
// status, accepted matches, clusters}, model[max_objects], pose[7 * max_objects] and score[max_objects], each field frame-major.
struct BatchSlots { int32_t *info, *model; float *pose, *score; };
inline size_t batch_slots_bytes(int n_frames, int max_objects) { return (16 + 36 * (size_t)max_objects) * (size_t)n_frames; }
inline BatchSlots batch_slots(void *base, int n_frames, int max_objects) {
	char *b = (char *)base;
	const size_t nf = (size_t)n_frames, mo = (size_t)max_objects;
	return { (int32_t *)b, (int32_t *)(b + 16 * nf), (float *)(b + (16 + 4 * mo) * nf), (float *)(b + (16 + 32 * mo) * nf) };
}
// Host copy of the slots -> the caller's arrays: frame_info (nullable) and n_objects of every frame, the objects of a frame whose
// status is 0 and whose objects fit. first_bad / first_over: the first frame with a non-zero status / more than max_objects objects, or -1.
void unpack_batch(const BatchSlots &h, int n_frames, int max_objects, int32_t *n_objects, int32_t *obj_model, float *obj_pose, float *obj_score,
                  int32_t *frame_info, int &first_bad, int &first_over);

// ---- moped3d's batched MATCH (adaptive.cu), shared by mc_match_adaptive_frames* and mc_process_depth_queries* ----
// Where the nearest rows come from: one cascade pass over q_desc against the context's database (n_shards = 0), or the merge of
// n_shards gathered packed blocks (device) against the context's tables.
struct RowSource {
	const float *q_desc;
	const int32_t *packed_all;
	int n_shards;
};
mc_status match_adaptive_frames(mc_ctx *ctx, bool dev, const char *who, const RowSource &src, const float *q_xy, const int32_t *q_image,
                                const int32_t *frame_offsets, int n_frames, int frame_begin, int frame_end, const float *depth,
                                const float *fill_distance, int width, int height, const mc_adaptive_model *models, int n_models,
                                float maximum_depth, float default_depth, float cauchy_scale, int32_t *match_offsets, int32_t *match_feature,
                                int32_t *match_image, float *match_xy, float *match_xyz, int32_t *nn_row, float *nn_dist, uint8_t *accepted,
                                int32_t *frame_info, const float *q_world, const float *q_fill, float *match_world, float *match_fill,
                                cudaEvent_t *ev);

// ---- moped3d linkage clustering of all models of a frame at once (linkage.cu) ----
struct LinkSlice {         // one model of a frame: matches lo .. lo+n of the frame, n x n matrix block at element sq of the arena
	int64_t sq;
	int32_t lo, n, model, pad;
};
struct LinkFrame {         // device pointers unless noted
	const LinkSlice *slices; int n_slices, n_max;      // models with matches, ascending; n_slices / n_max (largest n) on the host
	const float *xy, *xyz, *world;                     // the frame's per-match arrays
	const float *depth, *distance; int W, H;           // depth map and its fill-distance map
	int32_t *status;                                   // nullable: set to 1 when a match lies outside the maps (the frame is then skipped)
	float *K2D, *K3D, *K3F, *K, *D, *tmp, *scal;       // arena (link_carve)
	int32_t *valid, *lists, *sz, *ints3, *out_count, *out_offsets, *out_members, *compact;
};
size_t link_arena_bytes(int64_t sq_total, int M, int S);
void link_carve(void *arena, int64_t sq_total, int M, int S, LinkFrame &F);
mc_status link_frame_device(mc_ctx *ctx, const LinkFrame &F, float cutoff, int min_pts, int use3DFilter, int linkage, float sigma2D, float sigma3D);
mc_status link_compact_device(mc_ctx *ctx, const LinkFrame &F, int32_t *d_out_n, int32_t *d_cluster_model, int32_t *d_cluster_offsets,
                              int32_t *d_members, int32_t *d_n_obj);
mc_status match_merge_device(mc_ctx *ctx, const int32_t *rows_all, const float *dist_all, size_t stride, int n_shards, int Q, float ratio,
                             int32_t *d_nn_row, float *d_nn_dist, uint8_t *d_accepted);

} // namespace mc
