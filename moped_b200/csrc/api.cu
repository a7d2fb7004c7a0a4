// api.cu — the C ABI of libmoped_cuda.so (include/moped_cuda.h): context, database upload, and the
// host-buffer wrappers around the device stage entry points. No CPU fallback anywhere: every path ends in
// a kernel launch on the context's device or returns an error.
#include "common.cuh"

#include <cstring>
#include <cmath>
#include <algorithm>

namespace mc {
mc_status filter_depth_device(mc_ctx *ctx, const int32_t *d_match_offsets, const int32_t *d_match_image, const float *d_match_xy,
                              const float *d_match_xyz, int n_models, int max_matches, const int32_t *d_obj_model, const float *d_obj_pose,
                              const int32_t *d_n_obj, int n_obj_cap, int min_points, float feat_dist, float min_score,
                              const int32_t *d_test_offsets, const float *d_test_xyz, const float *depth_K4, const float *depth_TM12, int width,
                              int height, const float *d_depth, const float *d_fill, float plausible_dist, float depth_fraction,
                              float min_keypoint_fraction, uint8_t *d_keep, float *d_score, int32_t *d_out_n, int32_t *d_cluster_model,
                              int32_t *d_cluster_offsets, int32_t *d_members, int32_t *d_surv_model, float *d_surv_pose, float *d_surv_score);
}
namespace mc {
mc_status cluster_device(mc_ctx *ctx, const int32_t *d_match_offsets, const int32_t *d_match_image, const float *d_match_xy,
                         int n_models, int n_images, int max_matches, float radius, float merge, int min_pts, int max_iter,
                         int32_t *d_out_n, int32_t *d_cluster_model, int32_t *d_cluster_offsets, int32_t *d_members);
mc_status pose_hypotheses_device(mc_ctx *ctx, const int32_t *d_cluster_offsets, const float *d_xy, const float *d_xyz, const int32_t *d_image,
                                 const int32_t *d_hyp_cluster, const int32_t *d_sample_pos, const float *d_init_quat, int n_hyp,
                                 const mc_pose_params *pp, const int64_t *d_mask_offsets, int32_t *d_n_inliers, float *d_pose_lm,
                                 float *d_pose_refit, float *d_lm_err, uint8_t *d_mask);
mc_status pose_ransac_device(mc_ctx *ctx, const int32_t *d_cluster_offsets, const int32_t *d_n_clusters, int n_clusters_cap, int n_points_cap,
                             const float *d_xy, const float *d_xyz, const int32_t *d_image, const int32_t *d_tie,
                             const mc_pose_params *pp, uint8_t *d_found, float *d_pose, int32_t *d_n_tests);
mc_status pose_depth_hypotheses_device(mc_ctx *ctx, int variant, const int32_t *d_cluster_offsets, const float *d_xy, const float *d_xyz,
                                       const float *d_world, const float *d_cauchy, const int32_t *d_image, const int32_t *d_hyp_cluster,
                                       const int32_t *d_sample_pos, const float *d_init_quat, int n_hyp, int n_max, const mc_pose_params *pp,
                                       float alpha, const int64_t *d_mask_offsets, int32_t *d_n_inliers, float *d_pose_lm, float *d_pose_refit,
                                       float *d_lm_err, uint8_t *d_mask);
mc_status pose_depth_ransac_device(mc_ctx *ctx, int variant, const int32_t *d_cluster_offsets, int n_clusters, int n_max, const float *d_xy,
                                   const float *d_xyz, const float *d_world, const float *d_cauchy, const int32_t *d_image, const int32_t *d_tie,
                                   const mc_pose_params *pp, float alpha, uint8_t *d_found, float *d_pose, int32_t *d_n_tests,
                                   const int32_t *d_n_clusters);
mc_status filter_device(mc_ctx *ctx, const int32_t *d_match_offsets, const int32_t *d_match_image, const float *d_match_xy,
                        const float *d_match_xyz, int n_models, int max_matches, const int32_t *d_obj_model, const float *d_obj_pose,
                        const int32_t *d_n_obj, int n_obj_cap, int min_points, float feat_dist, float min_score,
                        uint8_t *d_keep, float *d_score, int32_t *d_out_n, int32_t *d_cluster_model, int32_t *d_cluster_offsets,
                        int32_t *d_members, int32_t *d_surv_model, float *d_surv_pose, float *d_surv_score);
mc_status process_frame_device(mc_ctx *ctx, const float *d_q, const float *d_qxy, const int32_t *d_qimg, int Q, const mc_pipeline_params *P,
                               int max_objects, int32_t *n_objects, int32_t *obj_model, float *obj_pose, float *obj_score, float *stage_ms,
                               const int32_t *d_nn_row_in = nullptr, const uint8_t *d_accepted_in = nullptr);
mc_status process_frames_device(mc_ctx *ctx, const float *d_q, const float *d_qxy, const int32_t *d_qimg, const int32_t *frame_offsets,
                                int f_begin, int f_end, const mc_pipeline_params *P, int max_objects, const int32_t *d_nn_row_in,
                                const uint8_t *d_accepted_in, int32_t *d_out_info, int32_t *d_out_model, float *d_out_pose, float *d_out_score,
                                cudaEvent_t *ev3);
mc_status join_lanes(mc_ctx *ctx);
mc_status process_frames_host(mc_ctx *ctx, const float *d_q, const float *d_qxy, const int32_t *d_qimg, const int32_t *frame_offsets, int n_frames,
                              const mc_pipeline_params *P, int max_objects, int32_t *n_objects, int32_t *obj_model, float *obj_pose, float *obj_score,
                              int32_t *frame_info, float *stage_ms);

template <typename T> static mc_status h2d(mc_ctx *ctx, T *dst, const T *src, size_t n) {
	if (n == 0) return MC_OK;
	MC_CUDA(cudaMemcpyAsync(dst, src, n * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
	return MC_OK;
}
template <typename T> static mc_status d2h(mc_ctx *ctx, T *dst, const T *src, size_t n) {
	if (n == 0) return MC_OK;
	MC_CUDA(cudaMemcpyAsync(dst, src, n * sizeof(T), cudaMemcpyDeviceToHost, ctx->stream));
	return MC_OK;
}
} // namespace mc

using namespace mc;

static thread_local std::string g_create_err;

extern "C" {

const char *mc_version(void) { return "libmoped_cuda 0.1 (sm_100a)"; }

mc_status mc_create(mc_ctx **out, int device) {
	if (!out) return MC_ERR_ARG;
	*out = nullptr;
	int n = 0;
	cudaError_t e = cudaGetDeviceCount(&n);
	if (e != cudaSuccess || n <= 0 || device < 0 || device >= n) {
		g_create_err = std::string("mc_create: no usable CUDA device (") + (e != cudaSuccess ? cudaGetErrorString(e) : "bad index") + ")";
		return MC_ERR_CUDA;
	}
	cudaDeviceProp prop;
	if (cudaGetDeviceProperties(&prop, device) != cudaSuccess || prop.major != 10) {
		g_create_err = "mc_create: libmoped_cuda is built for sm_100a (B200) only";
		return MC_ERR_CUDA;
	}
	if (cudaSetDevice(device) != cudaSuccess) { g_create_err = "mc_create: cudaSetDevice failed"; return MC_ERR_CUDA; }
	mc_ctx *ctx = new mc_ctx;
	ctx->device = device;
	ctx->num_sms = prop.multiProcessorCount;
	if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) { delete ctx; g_create_err = "mc_create: stream"; return MC_ERR_CUDA; }
	ctx->own_stream = true;
	// opt-in shared-memory sizes are per-device function attributes: set them for THIS context's device
	if (match_configure_device(ctx) != MC_OK || cluster_configure_device(ctx) != MC_OK) {
		g_create_err = "mc_create: " + ctx->err;
		cudaStreamDestroy(ctx->stream);
		delete ctx;
		return MC_ERR_CUDA;
	}
	*out = ctx;
	return MC_OK;
}

static void free_db(mc_ctx *ctx) {
	cudaFree(ctx->d_db); cudaFree(ctx->d_db_img); cudaFree(ctx->d_db_img8); cudaFree(ctx->d_xyz); cudaFree(ctx->d_model_of_row);
	ctx->d_db = nullptr; ctx->d_db_img = nullptr; ctx->d_db_img8 = nullptr; ctx->d_xyz = nullptr; ctx->d_model_of_row = nullptr;
	ctx->n_rows = 0; ctx->n_tiles = 0;
}

static void free_scratch(mc_ctx *ctx);

static void destroy_lanes(mc_ctx *ctx) {
	for (mc_ctx *lane : ctx->lanes) {          // lanes borrow the database and cameras: free only what they own
		cudaStreamSynchronize(lane->stream);
		free_scratch(lane);
		if (lane->ev_done) cudaEventDestroy(lane->ev_done);
		cudaStreamDestroy(lane->stream);
		delete lane;
	}
	ctx->lanes.clear();
	ctx->lanes_pending = 0;
}

void mc_destroy(mc_ctx *ctx) {
	if (!ctx) return;
	cudaSetDevice(ctx->device);
	cudaStreamSynchronize(ctx->stream);
	destroy_lanes(ctx);
	sm_partition_destroy(ctx);
	if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
	for (cudaEvent_t e : ctx->ev_chunk) cudaEventDestroy(e);
	if (ctx->ev_coarse[0]) { cudaEventDestroy(ctx->ev_coarse[0]); cudaEventDestroy(ctx->ev_coarse[1]); }
	free_db(ctx);
	sift_free(ctx);
	cudaFree(ctx->d_cams);
	for (DepthFilterTable &t : ctx->depth_filter) { cudaFree(t.d_offsets); cudaFree(t.d_xyz); }
	for (UndistortTable &t : ctx->undistort) cudaFree(t.d_map);
	free_scratch(ctx);
	if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
	delete ctx;
}

static void free_scratch(mc_ctx *ctx) {
	DevBuf *named[] = { &ctx->q_desc, &ctx->q_img, &ctx->q_norm2, &ctx->tau, &ctx->cand_score, &ctx->cand_row, &ctx->flag_list, &ctx->flag_count,
	                    &ctx->nn_key, &ctx->nn_row, &ctx->nn_dist, &ctx->accepted, &ctx->q_xy, &ctx->q_image,
	                    &ctx->q_img8, &ctx->q_signed, &ctx->q_scale, &ctx->q_err, &ctx->flag_list2, &ctx->tau2, &ctx->cand_score2, &ctx->cand_row2 };
	for (DevBuf *b : named) cudaFree(b->p);
	for (DevBuf &b : ctx->scratch) cudaFree(b.p);
	cudaFree(ctx->batch_out.p);
	cudaFree(ctx->link_buf.p);
	cudaFree(ctx->frame_desc.p);
	for (auto &g : ctx->fgraphs) cudaGraphExecDestroy(g.exec);
	ctx->fgraphs.clear();
	for (auto &g : ctx->bgraphs) cudaGraphExecDestroy(g.exec);
	ctx->bgraphs.clear();
	if (ctx->h_pinned) cudaFreeHost(ctx->h_pinned);
}

const char *mc_last_error(const mc_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_err.c_str(); }

mc_status mc_set_stream(mc_ctx *ctx, void *cuda_stream) {
	if (!ctx) return MC_ERR_ARG;
	MC_CUDA(cudaSetDevice(ctx->device));
	MC_CUDA(cudaStreamSynchronize(ctx->stream));
	if (ctx->own_stream) { cudaStreamDestroy(ctx->stream); ctx->own_stream = false; }
	if (cuda_stream) ctx->stream = (cudaStream_t)cuda_stream;
	else { MC_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)); ctx->own_stream = true; }
	return MC_OK;
}

mc_status mc_synchronize(mc_ctx *ctx) {
	if (!ctx) return MC_ERR_ARG;
	MC_CUDA(cudaStreamSynchronize(ctx->stream));
	return MC_OK;
}

int64_t mc_kernel_launches(const mc_ctx *ctx) { return ctx ? ctx->launches : 0; }

mc_status mc_set_tuning(mc_ctx *ctx, int frame_lanes, int pose_warps_per_task, int match_chunks) {
	if (!ctx) return MC_ERR_ARG;
	if (frame_lanes > 64 || pose_warps_per_task > 8 || match_chunks > 16) { ctx->err = "mc_set_tuning: at most 64 lanes, 8 warps per task, 16 chunks"; return MC_ERR_ARG; }
	if (frame_lanes > 0) ctx->n_lanes_wanted = frame_lanes;
	if (pose_warps_per_task > 0) ctx->pose_warps = pose_warps_per_task;
	if (match_chunks > 0) ctx->match_chunks = match_chunks;
	return MC_OK;
}

mc_status mc_set_option(mc_ctx *ctx, const char *key, int64_t value) {
	if (!ctx || !key) return MC_ERR_ARG;
	const std::string k(key);
	if (k == "pose_fit_thread_min") ctx->fit_thread_min = value < 1 ? 1 : value;
	else if (k == "pose_fit_stream") ctx->fit_stream = value != 0;
	else if (k == "ransac_fused") ctx->ransac_fused = value != 0;
	else if (k == "ransac_merge_levels") ctx->ransac_merge_levels = value != 0;
	else if (k == "frame_graphs") ctx->frame_graphs = value != 0;
	else if (k == "batch_graph") ctx->batch_graph = value != 0;
	else if (k == "defer_lane_join") ctx->defer_lane_join = value != 0;
	else if (k == "match_coarse_kind") { if (value != 0 && value != 1) { ctx->err = "mc_set_option: match_coarse_kind must be 0 (fp16) or 1 (8-bit first)"; return MC_ERR_ARG; } ctx->coarse_kind = (int)value; }
	else if (k == "match_stagger") ctx->match_stagger = value != 0;
	else if (k == "match_splits") { if (value < 0 || value > 64) { ctx->err = "mc_set_option: match_splits must be in 0..64"; return MC_ERR_ARG; } ctx->match_splits = (int)value; }
	else if (k == "stage_sm_partition") {
		if (value < 0 || value > 96 || value % 8) { ctx->err = "mc_set_option: stage_sm_partition must be 0 or a multiple of 8 up to 96"; return MC_ERR_ARG; }
		MC_CUDA(cudaSetDevice(ctx->device));
		MC_CUDA(cudaStreamSynchronize(ctx->stream));
		destroy_lanes(ctx);                        // their streams belong to the old partition
		return sm_partition_create(ctx, (int)value);
	}
	else if (k == "match_reserve_sms") { if (value < 0 || value > 64) { ctx->err = "mc_set_option: match_reserve_sms must be in 0..64"; return MC_ERR_ARG; } ctx->match_reserve_sms = (int)value; }
	else if (k == "lm_finite_check") ctx->lm_finite_check = value != 0;
	else if (k == "pose_exact_order") ctx->pose_exact_order = value != 0;
	else if (k == "linkage_cached") ctx->linkage_cached = value != 0;
	else if (k == "depth_team_lanes") { if (value != 8 && value != 32) { ctx->err = "mc_set_option: depth_team_lanes must be 8 or 32"; return MC_ERR_ARG; } ctx->depth_team_lanes = (int)value; }
	else if (k == "sift_two_pass") return sift_set_two_pass(ctx, (int)value);
	else if (k == "sift_describe_gather") return sift_set_gather(ctx, (int)value);
	else { ctx->err = "mc_set_option: unknown key '" + k + "'"; return MC_ERR_ARG; }
	for (mc_ctx *lane : ctx->lanes) { lane->fit_thread_min = ctx->fit_thread_min; lane->fit_stream = ctx->fit_stream; lane->ransac_merge_levels = ctx->ransac_merge_levels; lane->ransac_fused = ctx->ransac_fused; lane->frame_graphs = ctx->frame_graphs; }
	return MC_OK;
}

mc_status mc_set_profiling(mc_ctx *ctx, int on) {
	if (!ctx) return MC_ERR_ARG;
	MC_CUDA(cudaSetDevice(ctx->device));
	if (on && !ctx->ev_coarse[0]) { MC_CUDA(cudaEventCreate(&ctx->ev_coarse[0])); MC_CUDA(cudaEventCreate(&ctx->ev_coarse[1])); }
	ctx->profile = on != 0; ctx->ev_valid = false;
	return MC_OK;
}

mc_status mc_profile_read(mc_ctx *ctx, float *coarse_ms) {
	if (!ctx || !coarse_ms) return MC_ERR_ARG;
	*coarse_ms = 0.f;
	if (!ctx->profile || !ctx->ev_valid) { ctx->err = "mc_profile_read: no profiled launch"; return MC_ERR_STATE; }
	MC_CUDA(cudaEventSynchronize(ctx->ev_coarse[1]));
	MC_CUDA(cudaEventElapsedTime(coarse_ms, ctx->ev_coarse[0], ctx->ev_coarse[1]));
	return MC_OK;
}
mc_status mc_match_last_stats(mc_ctx *ctx, int32_t *stats) {
	if (!ctx || !stats) return MC_ERR_ARG;
	MC_CUDA(cudaSetDevice(ctx->device));
	int32_t n_flag = 0;
	if (ctx->last_match_tensor && ctx->flag_count.p) {
		MC_CUDA(cudaMemcpyAsync(&n_flag, (const int32_t *)ctx->flag_count.p + 1, sizeof n_flag, cudaMemcpyDeviceToHost, ctx->stream));
		MC_CUDA(cudaStreamSynchronize(ctx->stream));
	}
	if (ctx->last_match_tensor) { stats[0] = ctx->last_match_q - n_flag; stats[1] = n_flag; stats[2] = ctx->last_stats[2]; stats[3] = ctx->last_stats[3]; }
	else { stats[0] = 0; stats[1] = ctx->last_match_q; stats[2] = 0; stats[3] = 0; }
	return MC_OK;
}
mc_status mc_match_tier_stats(mc_ctx *ctx, int32_t *tiers) {
	if (!ctx || !tiers) return MC_ERR_ARG;
	MC_CUDA(cudaSetDevice(ctx->device));
	int32_t n[2] = { 0, 0 };
	if (ctx->last_match_tensor && ctx->flag_count.p) {
		MC_CUDA(cudaMemcpyAsync(n, ctx->flag_count.p, sizeof n, cudaMemcpyDeviceToHost, ctx->stream));
		MC_CUDA(cudaStreamSynchronize(ctx->stream));
	}
	const bool i8 = ctx->last_match_tensor && ctx->coarse_kind == 1 && ctx->db_scale > 0.f;
	tiers[0] = ctx->last_match_q;
	tiers[1] = !ctx->last_match_tensor ? 0 : i8 ? ctx->last_match_q - n[0] : 0;         // certified by the 8-bit pass
	tiers[3] = ctx->last_match_tensor ? n[1] : ctx->last_match_q;                          // exhaustive exact scan
	tiers[2] = ctx->last_match_q - tiers[1] - tiers[3];                                    // certified by the fp16 pass
	if (i8 && tiers[1] < 0) tiers[1] = 0;
	return MC_OK;
}
mc_status mc_sm_partition(mc_ctx *ctx, int32_t *sms) {
	if (!ctx || !sms) return MC_ERR_ARG;
	sms[0] = ctx->match_sms ? ctx->match_sms : ctx->num_sms - ctx->match_reserve_sms;
	sms[1] = ctx->stage_sms;
	return MC_OK;
}
int64_t mc_db_rows(const mc_ctx *ctx) { return ctx ? ctx->n_rows : 0; }

mc_status mc_db_upload(mc_ctx *ctx, const float *desc, const float *xyz, const int32_t *model_of_row, int64_t n_rows, int desc_dim,
                       int n_models, int64_t row_base) {
	if (!ctx || !desc || !xyz || !model_of_row || n_rows <= 0 || n_models <= 0) { if (ctx) ctx->err = "mc_db_upload: bad argument"; return MC_ERR_ARG; }
	if (desc_dim < 1 || desc_dim > 4096) { ctx->err = "mc_db_upload: descriptor length must be in 1..4096"; return MC_ERR_ARG; }
	if (n_rows + row_base > 0x7fffffffLL) { ctx->err = "mc_db_upload: row ids must fit in int32"; return MC_ERR_ARG; }
	MC_CUDA(cudaSetDevice(ctx->device));
	MC_CUDA(cudaStreamSynchronize(ctx->stream));
	free_db(ctx);
	ctx->n_rows = n_rows; ctx->row_base = row_base; ctx->D = desc_dim; ctx->n_models = n_models;
	ctx->table_base = row_base; ctx->table_rows = n_rows;
	MC_CUDA(cudaMalloc(&ctx->d_db, sizeof(float) * (size_t)n_rows * desc_dim));
	MC_CUDA(cudaMalloc(&ctx->d_xyz, sizeof(float) * 3 * (size_t)n_rows));
	MC_CUDA(cudaMalloc(&ctx->d_model_of_row, sizeof(int32_t) * (size_t)n_rows));
	MC_CUDA(cudaMemcpyAsync(ctx->d_db, desc, sizeof(float) * (size_t)n_rows * desc_dim, cudaMemcpyHostToDevice, ctx->stream));
	MC_CUDA(cudaMemcpyAsync(ctx->d_xyz, xyz, sizeof(float) * 3 * (size_t)n_rows, cudaMemcpyHostToDevice, ctx->stream));
	MC_CUDA(cudaMemcpyAsync(ctx->d_model_of_row, model_of_row, sizeof(int32_t) * (size_t)n_rows, cudaMemcpyHostToDevice, ctx->stream));
	MC_TRY(db_build_images(ctx));
	MC_CUDA(cudaStreamSynchronize(ctx->stream));
	return MC_OK;
}

mc_status mc_db_set_global_tables(mc_ctx *ctx, const float *xyz_all, const int32_t *model_of_row_all, int64_t n_rows_all, int n_models_all) {
	if (!ctx || !xyz_all || !model_of_row_all || n_rows_all <= 0 || n_models_all <= 0) { if (ctx) ctx->err = "mc_db_set_global_tables: bad argument"; return MC_ERR_ARG; }
	if (!ctx->d_db) { ctx->err = "mc_db_set_global_tables: upload the shard first"; return MC_ERR_STATE; }
	MC_CUDA(cudaSetDevice(ctx->device));
	MC_CUDA(cudaStreamSynchronize(ctx->stream));
	cudaFree(ctx->d_xyz); cudaFree(ctx->d_model_of_row);
	ctx->d_xyz = nullptr; ctx->d_model_of_row = nullptr;
	MC_CUDA(cudaMalloc(&ctx->d_xyz, sizeof(float) * 3 * (size_t)n_rows_all));
	MC_CUDA(cudaMalloc(&ctx->d_model_of_row, sizeof(int32_t) * (size_t)n_rows_all));
	MC_CUDA(cudaMemcpy(ctx->d_xyz, xyz_all, sizeof(float) * 3 * (size_t)n_rows_all, cudaMemcpyHostToDevice));
	MC_CUDA(cudaMemcpy(ctx->d_model_of_row, model_of_row_all, sizeof(int32_t) * (size_t)n_rows_all, cudaMemcpyHostToDevice));
	ctx->table_base = 0; ctx->table_rows = n_rows_all; ctx->n_models = n_models_all;
	return MC_OK;
}

mc_status mc_set_cameras(mc_ctx *ctx, const float *K, const float *cam_pose, int n_images) {
	if (!ctx || !K || !cam_pose || n_images <= 0) { if (ctx) ctx->err = "mc_set_cameras: bad argument"; return MC_ERR_ARG; }
	MC_CUDA(cudaSetDevice(ctx->device));
	std::vector<Camera> cams(n_images);
	for (int i = 0; i < n_images; i++) {
		for (int j = 0; j < 4; j++) cams[i].K[j] = K[4 * i + j];
		pose_tm(cam_pose + 7 * i, cams[i].TM);               // image->TM.init(cameraPose), moped.cpp:168-169
	}
	MC_CUDA(cudaStreamSynchronize(ctx->stream));
	if (ctx->d_cams) { MC_CUDA(cudaFree(ctx->d_cams)); ctx->d_cams = nullptr; }
	MC_CUDA(cudaMalloc(&ctx->d_cams, sizeof(Camera) * n_images));
	MC_CUDA(cudaMemcpy(ctx->d_cams, cams.data(), sizeof(Camera) * n_images, cudaMemcpyHostToDevice));
	ctx->n_images = n_images;
	return MC_OK;
}

// ---- MATCH -----------------------------------------------------------------------------------
mc_status mc_match_dev(mc_ctx *ctx, const float *q_desc_dev, int n_queries, float ratio, int mode, int32_t *nn_row_dev, float *nn_dist_dev,
                       uint8_t *accepted_dev) {
	if (!ctx || !q_desc_dev || !nn_row_dev || !nn_dist_dev || !accepted_dev || n_queries < 0) { if (ctx) ctx->err = "mc_match_dev: bad argument"; return MC_ERR_ARG; }
	MC_CUDA(cudaSetDevice(ctx->device));
	return match_device(ctx, q_desc_dev, n_queries, ratio, mode, nn_row_dev, nn_dist_dev, accepted_dev);
}

mc_status mc_match(mc_ctx *ctx, const float *q_desc, int Q, float ratio, int mode, int32_t *nn_row, float *nn_dist, uint8_t *accepted, int32_t *stats) {
	if (!ctx || !q_desc || !nn_row || !nn_dist || !accepted || Q < 0) { if (ctx) ctx->err = "mc_match: bad argument"; return MC_ERR_ARG; }
	if (!ctx->d_db) { ctx->err = "mc_match: no database uploaded"; return MC_ERR_STATE; }
	if (Q == 0) return MC_OK;
	MC_CUDA(cudaSetDevice(ctx->device));
	MC_TRY(reserve(ctx, ctx->q_desc, sizeof(float) * (size_t)Q * ctx->D));
	MC_TRY(reserve(ctx, ctx->nn_row, sizeof(int32_t) * 2 * (size_t)Q));
	MC_TRY(reserve(ctx, ctx->nn_dist, sizeof(float) * 2 * (size_t)Q));
	MC_TRY(reserve(ctx, ctx->accepted, (size_t)Q));
	MC_TRY(h2d(ctx, (float *)ctx->q_desc.p, q_desc, (size_t)Q * ctx->D));
	MC_TRY(match_device(ctx, (const float *)ctx->q_desc.p, Q, ratio, mode, (int32_t *)ctx->nn_row.p, (float *)ctx->nn_dist.p, (uint8_t *)ctx->accepted.p));
	MC_TRY(d2h(ctx, nn_row, (const int32_t *)ctx->nn_row.p, 2 * (size_t)Q));
	MC_TRY(d2h(ctx, nn_dist, (const float *)ctx->nn_dist.p, 2 * (size_t)Q));
	MC_TRY(d2h(ctx, accepted, (const uint8_t *)ctx->accepted.p, (size_t)Q));
	int32_t n_flag = 0;
	const bool tensor = ctx->last_match_tensor != 0;         // descriptor lengths other than 128 take the exact scan whatever `mode` says
	if (stats && tensor) MC_TRY(d2h(ctx, &n_flag, (const int32_t *)ctx->flag_count.p + 1, 1));
	MC_CUDA(cudaStreamSynchronize(ctx->stream));
	if (stats) {
		if (tensor) { stats[0] = Q - n_flag; stats[1] = n_flag; stats[2] = ctx->last_stats[2]; stats[3] = ctx->last_stats[3]; }
		else { stats[0] = 0; stats[1] = Q; stats[2] = 0; stats[3] = 0; }
	}
	return MC_OK;
}

mc_status mc_match_merge_dev(mc_ctx *ctx, const int32_t *rows_all, const float *dist_all, int n_shards, int Q, float ratio,
                             int32_t *nn_row_dev, float *nn_dist_dev, uint8_t *accepted_dev) {
	if (!ctx || !rows_all || !dist_all || n_shards <= 0 || Q < 0) { if (ctx) ctx->err = "mc_match_merge_dev: bad argument"; return MC_ERR_ARG; }
	MC_CUDA(cudaSetDevice(ctx->device));
	return match_merge_device(ctx, rows_all, dist_all, 2 * (size_t)Q, n_shards, Q, ratio, nn_row_dev, nn_dist_dev, accepted_dev);
}

mc_status mc_match_merge_packed_dev(mc_ctx *ctx, const void *packed_all, int n_shards, int Q, float ratio, int32_t *nn_row_dev, float *nn_dist_dev,
                                    uint8_t *accepted_dev) {
	if (!ctx || !packed_all || n_shards <= 0 || Q < 0) { if (ctx) ctx->err = "mc_match_merge_packed_dev: bad argument"; return MC_ERR_ARG; }
	MC_CUDA(cudaSetDevice(ctx->device));
	const int32_t *rows = (const int32_t *)packed_all;
	return match_merge_device(ctx, rows, (const float *)(rows + 2 * (size_t)Q), 4 * (size_t)Q, n_shards, Q, ratio, nn_row_dev, nn_dist_dev, accepted_dev);
}

// ---- CLUSTER ---------------------------------------------------------------------------------
mc_status mc_cluster_meanshift(mc_ctx *ctx, const int32_t *match_offsets, const int32_t *match_image, const float *match_xy, int n_models,
                               int n_images, float radius, float merge, int min_pts, int max_iterations, int32_t *n_clusters,
                               int32_t *cluster_model, int32_t *cluster_offsets, int32_t *members) {
	if (!ctx || !match_offsets || !n_clusters || !cluster_model || !cluster_offsets || !members || n_models <= 0 || n_images <= 0) {
		if (ctx) ctx->err = "mc_cluster_meanshift: bad argument";
		return MC_ERR_ARG;
	}
	MC_CUDA(cudaSetDevice(ctx->device));
	const int M = match_offsets[n_models];
	const size_t m = (size_t)M;
	int32_t *d_off, *d_img, *d_n, *d_cm, *d_co, *d_mem; float *d_xy;
	MC_TRY(carve_scratch(ctx, ctx->scratch[kScrHostCluster], [&](Carve &c) {
		c.take(d_off, (size_t)n_models + 1); c.take(d_img, m + 1); c.take(d_xy, 2 * (m + 1));
		c.take(d_n, 16); c.take(d_cm, m + 2); c.take(d_co, m + 2); c.take(d_mem, m + 2);
	}));
	MC_TRY(h2d(ctx, d_off, match_offsets, (size_t)n_models + 1));
	MC_TRY(h2d(ctx, d_img, match_image, m));
	MC_TRY(h2d(ctx, d_xy, match_xy, 2 * m));
	MC_TRY(cluster_device(ctx, d_off, d_img, d_xy, n_models, n_images, M, radius, merge, min_pts, max_iterations, d_n, d_cm, d_co, d_mem));
	int32_t hn[2] = { 0, 0 };
	MC_TRY(d2h(ctx, hn, d_n, 2));
	MC_CUDA(cudaStreamSynchronize(ctx->stream));
	*n_clusters = hn[0];
	MC_TRY(d2h(ctx, cluster_model, d_cm, (size_t)hn[0]));
	MC_TRY(d2h(ctx, cluster_offsets, d_co, (size_t)hn[0] + 1));
	MC_TRY(d2h(ctx, members, d_mem, (size_t)hn[1]));
	MC_CUDA(cudaStreamSynchronize(ctx->stream));
	return MC_OK;
}

// ---- POSE ------------------------------------------------------------------------------------
mc_status mc_pose_hypotheses(mc_ctx *ctx, const int32_t *cluster_offsets, int n_clusters, const float *pt_xy, const float *pt_xyz,
                             const int32_t *pt_image, const int32_t *hyp_cluster, const int32_t *sample_pos, const float *init_quat, int n_hyp,
                             const mc_pose_params *params, int32_t *n_inliers, float *pose_lm, float *pose_refit, float *lm_err,
                             uint8_t *inlier_mask) {
	if (!ctx || !cluster_offsets || !pt_xy || !pt_xyz || !pt_image || !hyp_cluster || !sample_pos || !init_quat || !params || !n_inliers ||
	    !pose_lm || !pose_refit || !lm_err || n_clusters <= 0 || n_hyp < 0) {
		if (ctx) ctx->err = "mc_pose_hypotheses: bad argument";
		return MC_ERR_ARG;
	}
	if (n_hyp == 0) return MC_OK;
	MC_CUDA(cudaSetDevice(ctx->device));
	const int M = cluster_offsets[n_clusters];
	const int na = params->n_pts_align;
	if (na < 1 || na > 8) { ctx->err = "pose: n_pts_align must be in 1..8"; return MC_ERR_ARG; }
	std::vector<int64_t> mask_off(n_hyp + 1, 0);
	for (int h = 0; h < n_hyp; h++) {
		const int c = hyp_cluster[h];
		if (c < 0 || c >= n_clusters) { ctx->err = "mc_pose_hypotheses: hyp_cluster out of range"; return MC_ERR_ARG; }
		const int n = cluster_offsets[c + 1] - cluster_offsets[c];
		for (int j = 0; j < na; j++) {                       // before anything is uploaded, in both LM modes
			const int sp = sample_pos[(size_t)h * na + j];
			if (sp < 0 || sp >= n) { ctx->err = "mc_pose_hypotheses: sample_pos out of range"; return MC_ERR_ARG; }
		}
		mask_off[h + 1] = mask_off[h] + n;
	}
	const size_t m = (size_t)M, nh = (size_t)n_hyp;
	int32_t *d_co, *d_im, *d_hc, *d_sp, *d_ni; float *d_xy, *d_xyz, *d_iq, *d_pl, *d_pr, *d_le; int64_t *d_mo; uint8_t *d_mask;
	MC_TRY(carve_scratch(ctx, ctx->scratch[kScrHostPose], [&](Carve &c) {
		c.take(d_co, (size_t)n_clusters + 1); c.take(d_xy, 2 * m); c.take(d_xyz, 3 * m); c.take(d_im, m);
		c.take(d_hc, nh); c.take(d_sp, nh * na); c.take(d_iq, 4 * nh); c.take(d_mo, nh + 1);
		c.take(d_ni, nh); c.take(d_pl, 7 * nh); c.take(d_pr, 7 * nh); c.take(d_le, 2 * nh);
		c.take(d_mask, inlier_mask ? (size_t)mask_off[n_hyp] + 1 : 1);
	}));
	if (!inlier_mask) d_mask = nullptr;
	MC_TRY(h2d(ctx, d_co, cluster_offsets, (size_t)n_clusters + 1));
	MC_TRY(h2d(ctx, d_xy, pt_xy, 2 * m));
	MC_TRY(h2d(ctx, d_xyz, pt_xyz, 3 * m));
	MC_TRY(h2d(ctx, d_im, pt_image, m));
	MC_TRY(h2d(ctx, d_hc, hyp_cluster, nh));
	MC_TRY(h2d(ctx, d_sp, sample_pos, nh * na));
	MC_TRY(h2d(ctx, d_iq, init_quat, 4 * nh));
	MC_TRY(h2d(ctx, d_mo, mask_off.data(), nh + 1));
	if (ctx->pose_exact_order) {
		int n_max = 0;
		for (int c = 0; c < n_clusters; c++) n_max = std::max(n_max, cluster_offsets[c + 1] - cluster_offsets[c]);
		MC_TRY(pose_depth_hypotheses_device(ctx, 2, d_co, d_xy, d_xyz, nullptr, nullptr, d_im, d_hc, d_sp, d_iq, n_hyp, n_max, params, 0.f, d_mo, d_ni,
		                                    d_pl, d_pr, d_le, d_mask));
	} else
	MC_TRY(pose_hypotheses_device(ctx, d_co, d_xy, d_xyz, d_im, d_hc, d_sp, d_iq, n_hyp, params, d_mo, d_ni, d_pl, d_pr, d_le, d_mask));
	MC_TRY(d2h(ctx, n_inliers, d_ni, nh));
	MC_TRY(d2h(ctx, pose_lm, d_pl, 7 * nh));
	MC_TRY(d2h(ctx, pose_refit, d_pr, 7 * nh));
	MC_TRY(d2h(ctx, lm_err, d_le, 2 * nh));
	if (inlier_mask) MC_TRY(d2h(ctx, inlier_mask, d_mask, (size_t)mask_off[n_hyp]));
	MC_CUDA(cudaStreamSynchronize(ctx->stream));
	return MC_OK;
}

mc_status mc_pose_hypotheses_dev(mc_ctx *ctx, const int32_t *cluster_offsets_dev, const float *pt_xy_dev, const float *pt_xyz_dev,
                                 const int32_t *pt_image_dev, const int32_t *hyp_cluster_dev, const int32_t *sample_pos_dev,
                                 const float *init_quat_dev, int n_hyp, const mc_pose_params *params, int32_t *n_inliers_dev,
                                 float *pose_lm_dev, float *pose_refit_dev, float *lm_err_dev) {
	if (!ctx || !cluster_offsets_dev || !pt_xy_dev || !pt_xyz_dev || !pt_image_dev || !hyp_cluster_dev || !sample_pos_dev || !init_quat_dev ||
	    !params || !n_inliers_dev || !pose_lm_dev || !pose_refit_dev || !lm_err_dev || n_hyp < 0) {
		if (ctx) ctx->err = "mc_pose_hypotheses_dev: bad argument";
		return MC_ERR_ARG;
	}
	if (n_hyp == 0) return MC_OK;
	MC_CUDA(cudaSetDevice(ctx->device));
	return pose_hypotheses_device(ctx, cluster_offsets_dev, pt_xy_dev, pt_xyz_dev, pt_image_dev, hyp_cluster_dev, sample_pos_dev, init_quat_dev,
	                              n_hyp, params, nullptr, n_inliers_dev, pose_lm_dev, pose_refit_dev, lm_err_dev, nullptr);
}

mc_status mc_pose_ransac(mc_ctx *ctx, const int32_t *cluster_offsets, int n_clusters, const float *pt_xy, const float *pt_xyz,
                         const int32_t *pt_image, const mc_pose_params *params, uint8_t *found, float *pose, int32_t *n_tests) {
	if (!ctx || !cluster_offsets || !pt_xy || !pt_xyz || !pt_image || !params || !found || !pose || !n_tests || n_clusters <= 0) {
		if (ctx) ctx->err = "mc_pose_ransac: bad argument";
		return MC_ERR_ARG;
	}
	MC_CUDA(cudaSetDevice(ctx->device));
	const int M = cluster_offsets[n_clusters];
	const int n_tasks = n_clusters * params->max_objects_per_cluster;
	const size_t m = (size_t)M, nt = (size_t)n_tasks;
	int32_t *d_co, *d_im, *d_nt; float *d_xy, *d_xyz, *d_p; uint8_t *d_f;
	MC_TRY(carve_scratch(ctx, ctx->scratch[kScrHostRansac], [&](Carve &c) {
		c.take(d_co, (size_t)n_clusters + 1); c.take(d_xy, 2 * m); c.take(d_xyz, 3 * m); c.take(d_im, m);
		c.take(d_f, nt); c.take(d_p, 7 * nt); c.take(d_nt, nt);
	}));
	MC_TRY(h2d(ctx, d_co, cluster_offsets, (size_t)n_clusters + 1));
	MC_TRY(h2d(ctx, d_xy, pt_xy, 2 * m));
	MC_TRY(h2d(ctx, d_xyz, pt_xyz, 3 * m));
	MC_TRY(h2d(ctx, d_im, pt_image, m));
	MC_CUDA(cudaMemsetAsync(d_p, 0, 28 * nt, ctx->stream));
	// exact-order mode (mc_set_option "pose_exact_order") is handled inside: the same staged driver with the order-preserving LM
	MC_TRY(pose_ransac_device(ctx, d_co, nullptr, n_clusters, M, d_xy, d_xyz, d_im, nullptr, params, d_f, d_p, d_nt));
	MC_TRY(d2h(ctx, found, d_f, nt));
	MC_TRY(d2h(ctx, pose, d_p, 7 * nt));
	MC_TRY(d2h(ctx, n_tests, d_nt, nt));
	MC_CUDA(cudaStreamSynchronize(ctx->stream));
	return MC_OK;
}

// ---- POSE, moped3d depth-aware variants (pose_depth.cu) ----------------------------------------
static int largest_cluster(const int32_t *cluster_offsets, int n_clusters) {
	int m = 0;
	for (int c = 0; c < n_clusters; c++) m = std::max(m, cluster_offsets[c + 1] - cluster_offsets[c]);
	return m;
}

mc_status mc_pose_depth_hypotheses(mc_ctx *ctx, int variant, const int32_t *cluster_offsets, int n_clusters, const float *pt_xy,
                                   const float *pt_xyz, const float *pt_world, const float *pt_cauchy, const int32_t *pt_image,
                                   const int32_t *hyp_cluster, const int32_t *sample_pos, const float *init_quat, int n_hyp,
                                   const mc_pose_params *params, float alpha, int32_t *n_inliers, float *pose_lm, float *pose_refit,
                                   float *lm_err, uint8_t *inlier_mask) {
	if (!ctx || !cluster_offsets || !pt_xy || !pt_xyz || !pt_world || !pt_cauchy || !pt_image || !hyp_cluster || !sample_pos || !init_quat ||
	    !params || !n_inliers || !pose_lm || !pose_refit || !lm_err || n_clusters <= 0 || n_hyp < 0) {
		if (ctx) ctx->err = "mc_pose_depth_hypotheses: bad argument";
		return MC_ERR_ARG;
	}
	if (n_hyp == 0) return MC_OK;
	MC_CUDA(cudaSetDevice(ctx->device));
	const int M = cluster_offsets[n_clusters];
	const int na = params->n_pts_align;
	std::vector<int64_t> mask_off(n_hyp + 1, 0);
	for (int h = 0; h < n_hyp; h++) {
		const int c = hyp_cluster[h];
		if (c < 0 || c >= n_clusters) { ctx->err = "mc_pose_depth_hypotheses: hyp_cluster out of range"; return MC_ERR_ARG; }
		const int n = cluster_offsets[c + 1] - cluster_offsets[c];
		for (int j = 0; j < na; j++) {
			const int s = sample_pos[(size_t)h * na + j];
			if (s < 0 || s >= n) { ctx->err = "mc_pose_depth_hypotheses: sample_pos out of range"; return MC_ERR_ARG; }
		}
		mask_off[h + 1] = mask_off[h] + n;
	}
	const size_t m = (size_t)M, nh = (size_t)n_hyp;
	int32_t *d_co, *d_im, *d_hc, *d_sp, *d_ni; float *d_xy, *d_xyz, *d_w, *d_cw, *d_iq, *d_pl, *d_pr, *d_le; int64_t *d_mo; uint8_t *d_mask;
	MC_TRY(carve_scratch(ctx, ctx->scratch[kScrHostPoseDepth], [&](Carve &c) {
		c.take(d_co, (size_t)n_clusters + 1); c.take(d_xy, 2 * m); c.take(d_xyz, 3 * m); c.take(d_w, 3 * m); c.take(d_cw, m); c.take(d_im, m);
		c.take(d_hc, nh); c.take(d_sp, nh * na); c.take(d_iq, 4 * nh); c.take(d_mo, nh + 1);
		c.take(d_ni, nh); c.take(d_pl, 7 * nh); c.take(d_pr, 7 * nh); c.take(d_le, 2 * nh);
		c.take(d_mask, inlier_mask ? (size_t)mask_off[n_hyp] + 1 : 1);
	}));
	if (!inlier_mask) d_mask = nullptr;
	MC_TRY(h2d(ctx, d_co, cluster_offsets, (size_t)n_clusters + 1));
	MC_TRY(h2d(ctx, d_xy, pt_xy, 2 * m));
	MC_TRY(h2d(ctx, d_xyz, pt_xyz, 3 * m));
	MC_TRY(h2d(ctx, d_w, pt_world, 3 * m));
	MC_TRY(h2d(ctx, d_cw, pt_cauchy, m));
	MC_TRY(h2d(ctx, d_im, pt_image, m));
	MC_TRY(h2d(ctx, d_hc, hyp_cluster, nh));
	MC_TRY(h2d(ctx, d_sp, sample_pos, nh * na));
	MC_TRY(h2d(ctx, d_iq, init_quat, 4 * nh));
	MC_TRY(h2d(ctx, d_mo, mask_off.data(), nh + 1));
	MC_TRY(pose_depth_hypotheses_device(ctx, variant, d_co, d_xy, d_xyz, d_w, d_cw, d_im, d_hc, d_sp, d_iq, n_hyp, largest_cluster(cluster_offsets, n_clusters),
	                                    params, alpha, d_mo, d_ni, d_pl, d_pr, d_le, d_mask));
	MC_TRY(d2h(ctx, n_inliers, d_ni, nh));
	MC_TRY(d2h(ctx, pose_lm, d_pl, 7 * nh));
	MC_TRY(d2h(ctx, pose_refit, d_pr, 7 * nh));
	MC_TRY(d2h(ctx, lm_err, d_le, 2 * nh));
	if (inlier_mask) MC_TRY(d2h(ctx, inlier_mask, d_mask, (size_t)mask_off[n_hyp]));
	MC_CUDA(cudaStreamSynchronize(ctx->stream));
	return MC_OK;
}

mc_status mc_pose_depth_hypotheses_dev(mc_ctx *ctx, int variant, const int32_t *cluster_offsets_dev, int max_cluster_size, const float *pt_xy_dev,
                                       const float *pt_xyz_dev, const float *pt_world_dev, const float *pt_cauchy_dev, const int32_t *pt_image_dev,
                                       const int32_t *hyp_cluster_dev, const int32_t *sample_pos_dev, const float *init_quat_dev, int n_hyp,
                                       const mc_pose_params *params, float alpha, int32_t *n_inliers_dev, float *pose_lm_dev,
                                       float *pose_refit_dev, float *lm_err_dev) {
	if (!ctx || !cluster_offsets_dev || !pt_xy_dev || !pt_xyz_dev || !pt_image_dev || !hyp_cluster_dev || !sample_pos_dev || !init_quat_dev ||
	    !params || !n_inliers_dev || !pose_lm_dev || !pose_refit_dev || !lm_err_dev || n_hyp < 0 || max_cluster_size < 1) {
		if (ctx) ctx->err = "mc_pose_depth_hypotheses_dev: bad argument";
		return MC_ERR_ARG;
	}
	if (n_hyp == 0) return MC_OK;
	MC_CUDA(cudaSetDevice(ctx->device));
	return pose_depth_hypotheses_device(ctx, variant, cluster_offsets_dev, pt_xy_dev, pt_xyz_dev, pt_world_dev, pt_cauchy_dev, pt_image_dev,
	                                    hyp_cluster_dev, sample_pos_dev, init_quat_dev, n_hyp, max_cluster_size, params, alpha, nullptr,
	                                    n_inliers_dev, pose_lm_dev, pose_refit_dev, lm_err_dev, nullptr);
}

mc_status mc_pose_depth_ransac(mc_ctx *ctx, int variant, const int32_t *cluster_offsets, int n_clusters, const float *pt_xy, const float *pt_xyz,
                               const float *pt_world, const float *pt_cauchy, const int32_t *pt_image, const int32_t *pt_tie,
                               const mc_pose_params *params, float alpha, uint8_t *found, float *pose, int32_t *n_tests) {
	if (!ctx || !cluster_offsets || !pt_xy || !pt_xyz || !pt_world || !pt_cauchy || !pt_image || !params || !found || !pose || !n_tests ||
	    n_clusters <= 0) {
		if (ctx) ctx->err = "mc_pose_depth_ransac: bad argument";
		return MC_ERR_ARG;
	}
	MC_CUDA(cudaSetDevice(ctx->device));
	const int M = cluster_offsets[n_clusters];
	const int n_tasks = n_clusters * params->max_objects_per_cluster;
	if (n_tasks <= 0) return MC_OK;
	const size_t m = (size_t)M, nt = (size_t)n_tasks;
	int32_t *d_co, *d_im, *d_tie, *d_nt; float *d_xy, *d_xyz, *d_w, *d_cw, *d_p; uint8_t *d_f;
	MC_TRY(carve_scratch(ctx, ctx->scratch[kScrHostPoseDepth], [&](Carve &c) {
		c.take(d_co, (size_t)n_clusters + 1); c.take(d_xy, 2 * m); c.take(d_xyz, 3 * m); c.take(d_w, 3 * m); c.take(d_cw, m); c.take(d_im, m); c.take(d_tie, m);
		c.take(d_f, nt); c.take(d_p, 7 * nt); c.take(d_nt, nt);
	}));
	if (!pt_tie) d_tie = nullptr;
	MC_TRY(h2d(ctx, d_co, cluster_offsets, (size_t)n_clusters + 1));
	MC_TRY(h2d(ctx, d_xy, pt_xy, 2 * m));
	MC_TRY(h2d(ctx, d_xyz, pt_xyz, 3 * m));
	MC_TRY(h2d(ctx, d_w, pt_world, 3 * m));
	MC_TRY(h2d(ctx, d_cw, pt_cauchy, m));
	MC_TRY(h2d(ctx, d_im, pt_image, m));
	if (pt_tie) MC_TRY(h2d(ctx, d_tie, pt_tie, m));
	MC_CUDA(cudaMemsetAsync(d_p, 0, 28 * nt, ctx->stream));
	MC_TRY(pose_depth_ransac_device(ctx, variant, d_co, n_clusters, largest_cluster(cluster_offsets, n_clusters), d_xy, d_xyz, d_w, d_cw, d_im, d_tie,
	                                params, alpha, d_f, d_p, d_nt, nullptr));
	MC_TRY(d2h(ctx, found, d_f, nt));
	MC_TRY(d2h(ctx, pose, d_p, 7 * nt));
	MC_TRY(d2h(ctx, n_tests, d_nt, nt));
	MC_CUDA(cudaStreamSynchronize(ctx->stream));
	return MC_OK;
}

// ---- FILTER ----------------------------------------------------------------------------------
mc_status mc_filter_projection(mc_ctx *ctx, const int32_t *match_offsets, const int32_t *match_image, const float *match_xy,
                               const float *match_xyz, int n_models, const int32_t *obj_model, const float *obj_pose, int n_objects,
                               int min_points, float feature_distance, float min_score, uint8_t *keep, float *score, int32_t *n_survivors,
                               int32_t *cluster_offsets, int32_t *members) {
	if (!ctx || !match_offsets || !n_survivors || !cluster_offsets || !members || n_models <= 0 || n_objects < 0) {
		if (ctx) ctx->err = "mc_filter_projection: bad argument";
		return MC_ERR_ARG;
	}
	MC_CUDA(cudaSetDevice(ctx->device));
	const int M = match_offsets[n_models];
	const size_t m = (size_t)M, no = n_objects > 0 ? (size_t)n_objects : 1;
	int32_t *d_off, *d_img, *d_om, *d_n, *d_cm, *d_co, *d_mem, *d_sm; float *d_xy, *d_xyz, *d_op, *d_sc, *d_sp, *d_ss; uint8_t *d_keep;
	MC_TRY(carve_scratch(ctx, ctx->scratch[kScrHostFilter], [&](Carve &c) {
		c.take(d_off, (size_t)n_models + 1); c.take(d_img, m + 1); c.take(d_xy, 2 * (m + 1)); c.take(d_xyz, 3 * (m + 1));
		c.take(d_om, no); c.take(d_op, 7 * no); c.take(d_keep, no); c.take(d_sc, no); c.take(d_n, 16);
		c.take(d_cm, no + 2); c.take(d_co, no + 2); c.take(d_mem, m + 2);
		c.take(d_sm, no); c.take(d_sp, 7 * no); c.take(d_ss, no);
	}));
	MC_TRY(h2d(ctx, d_off, match_offsets, (size_t)n_models + 1));
	MC_TRY(h2d(ctx, d_img, match_image, m));
	MC_TRY(h2d(ctx, d_xy, match_xy, 2 * m));
	MC_TRY(h2d(ctx, d_xyz, match_xyz, 3 * m));
	MC_TRY(h2d(ctx, d_om, obj_model, (size_t)n_objects));
	MC_TRY(h2d(ctx, d_op, obj_pose, 7 * (size_t)n_objects));
	MC_TRY(filter_device(ctx, d_off, d_img, d_xy, d_xyz, n_models, M, d_om, d_op, nullptr, n_objects, min_points, feature_distance, min_score, d_keep,
	                     d_sc, d_n, d_cm, d_co, d_mem, d_sm, d_sp, d_ss));
	int32_t hn[2] = { 0, 0 };
	MC_TRY(d2h(ctx, hn, d_n, 2));
	MC_TRY(d2h(ctx, keep, d_keep, (size_t)n_objects));
	MC_TRY(d2h(ctx, score, d_sc, (size_t)n_objects));
	MC_CUDA(cudaStreamSynchronize(ctx->stream));
	*n_survivors = hn[0];
	MC_TRY(d2h(ctx, cluster_offsets, d_co, (size_t)hn[0] + 1));
	MC_TRY(d2h(ctx, members, d_mem, (size_t)hn[1]));
	MC_CUDA(cudaStreamSynchronize(ctx->stream));
	return MC_OK;
}

mc_status mc_filter_projection_depth(mc_ctx *ctx, const int32_t *match_offsets, const int32_t *match_image, const float *match_xy,
                                     const float *match_xyz, int n_models, const int32_t *obj_model, const float *obj_pose, int n_objects,
                                     int min_points, float feature_distance, float plausible_sq_distance, float min_score, float depth_fraction,
                                     float min_keypoint_fraction, const int32_t *test_offsets, const float *test_xyz, const float *depth_K,
                                     const float *depth_pose, int width, int height, const float *depth, const float *fill_distance,
                                     uint8_t *keep, float *score, int32_t *n_survivors, int32_t *cluster_offsets, int32_t *members) {
	if (!ctx || !match_offsets || !n_survivors || !cluster_offsets || !members || !test_offsets || !depth_K || !depth_pose || !depth || !fill_distance ||
	    n_models <= 0 || n_objects < 0 || width <= 0 || height <= 0) {
		if (ctx) ctx->err = "mc_filter_projection_depth: bad argument";
		return MC_ERR_ARG;
	}
	for (int m = 0; m < n_models; m++)
		if (test_offsets[m + 1] < test_offsets[m] || test_offsets[0] != 0) { ctx->err = "mc_filter_projection_depth: test_offsets must start at 0 and ascend"; return MC_ERR_ARG; }
	if (test_offsets[n_models] > 0 && !test_xyz) { ctx->err = "mc_filter_projection_depth: bad argument"; return MC_ERR_ARG; }
	MC_CUDA(cudaSetDevice(ctx->device));
	const int M = match_offsets[n_models];
	const int NT = test_offsets[n_models];
	const size_t px = (size_t)width * height;
	const size_t m = (size_t)M, no = n_objects > 0 ? (size_t)n_objects : 1;
	int32_t *d_off, *d_img, *d_om, *d_n, *d_cm, *d_co, *d_mem, *d_sm, *d_to; float *d_xy, *d_xyz, *d_op, *d_sc, *d_sp, *d_ss, *d_tx, *d_d, *d_f;
	uint8_t *d_keep;
	MC_TRY(carve_scratch(ctx, ctx->scratch[kScrHostFilter], [&](Carve &c) {
		c.take(d_off, (size_t)n_models + 1); c.take(d_img, m + 1); c.take(d_xy, 2 * (m + 1)); c.take(d_xyz, 3 * (m + 1));
		c.take(d_om, no); c.take(d_op, 7 * no); c.take(d_keep, no); c.take(d_sc, no); c.take(d_n, 16);
		c.take(d_cm, no + 2); c.take(d_co, no + 2); c.take(d_mem, m + 2);
		c.take(d_sm, no); c.take(d_sp, 7 * no); c.take(d_ss, no);
		c.take(d_to, (size_t)n_models + 1); c.take(d_tx, 3 * ((size_t)NT + 1)); c.take(d_d, px); c.take(d_f, px);
	}));
	MC_TRY(h2d(ctx, d_off, match_offsets, (size_t)n_models + 1));
	MC_TRY(h2d(ctx, d_img, match_image, m));
	MC_TRY(h2d(ctx, d_xy, match_xy, 2 * m));
	MC_TRY(h2d(ctx, d_xyz, match_xyz, 3 * m));
	MC_TRY(h2d(ctx, d_om, obj_model, (size_t)n_objects));
	MC_TRY(h2d(ctx, d_op, obj_pose, 7 * (size_t)n_objects));
	MC_TRY(h2d(ctx, d_to, test_offsets, (size_t)n_models + 1));
	MC_TRY(h2d(ctx, d_tx, test_xyz, 3 * (size_t)NT));
	MC_TRY(h2d(ctx, d_d, depth, px));
	MC_TRY(h2d(ctx, d_f, fill_distance, px));
	float TM[12];
	pose_tm(depth_pose, TM);                                 // depthmap->TM.init(cameraPose)
	MC_TRY(filter_depth_device(ctx, d_off, d_img, d_xy, d_xyz, n_models, M, d_om, d_op, nullptr, n_objects, min_points, feature_distance, min_score, d_to,
	                           d_tx, depth_K, TM, width, height, d_d, d_f, plausible_sq_distance, depth_fraction, min_keypoint_fraction, d_keep, d_sc,
	                           d_n, d_cm, d_co, d_mem, d_sm, d_sp, d_ss));
	int32_t hn[2] = { 0, 0 };
	MC_TRY(d2h(ctx, hn, d_n, 2));
	MC_TRY(d2h(ctx, keep, d_keep, (size_t)n_objects));
	MC_TRY(d2h(ctx, score, d_sc, (size_t)n_objects));
	MC_CUDA(cudaStreamSynchronize(ctx->stream));
	*n_survivors = hn[0];
	MC_TRY(d2h(ctx, cluster_offsets, d_co, (size_t)hn[0] + 1));
	MC_TRY(d2h(ctx, members, d_mem, (size_t)hn[1]));
	MC_CUDA(cudaStreamSynchronize(ctx->stream));
	return MC_OK;
}

// ---- whole frame ------------------------------------------------------------------------------
void mc_pipeline_default_params(mc_pipeline_params *p) {
	if (!p) return;
	memset(p, 0, sizeof *p);
	p->match_ratio = 0.8f; p->match_mode = MC_MATCH_TENSOR;                                   // config.hpp:83
	p->cluster_radius = 200.f; p->cluster_merge = 20.f; p->cluster_min_pts = 7; p->cluster_max_iterations = 100;   // :101
	p->pose = mc_pose_params{ 600, 200, 4, 5, 6, 10.f, 1 };                                    // :110
	p->filter_min_points = 5; p->filter_feature_distance = 4096.f; p->filter_min_score = 2.f;  // :115
	p->pose2 = mc_pose_params{ 100, 500, 4, 6, 8, 5.f, 2 };                                    // :118
	p->filter2_min_points = 7; p->filter2_feature_distance = 4096.f; p->filter2_min_score = 3.f;   // :120
}

mc_status mc_process_frame_dev(mc_ctx *ctx, const float *q_desc_dev, const float *q_xy_dev, const int32_t *q_image_dev, int n_queries,
                               const mc_pipeline_params *params, int max_objects, int32_t *n_objects, int32_t *obj_model, float *obj_pose,
                               float *obj_score, float *stage_ms) {
	if (!ctx || !q_desc_dev || !q_xy_dev || !q_image_dev || !params || !n_objects || !obj_model || !obj_pose || !obj_score || max_objects <= 0) {
		if (ctx) ctx->err = "mc_process_frame_dev: bad argument";
		return MC_ERR_ARG;
	}
	MC_CUDA(cudaSetDevice(ctx->device));
	return process_frame_device(ctx, q_desc_dev, q_xy_dev, q_image_dev, n_queries, params, max_objects, n_objects, obj_model, obj_pose, obj_score, stage_ms);
}

mc_status mc_process_matched_dev(mc_ctx *ctx, const int32_t *nn_row_dev, const uint8_t *accepted_dev, const float *q_xy_dev,
                                 const int32_t *q_image_dev, int n_queries, const mc_pipeline_params *params, int max_objects,
                                 int32_t *n_objects, int32_t *obj_model, float *obj_pose, float *obj_score, float *stage_ms) {
	if (!ctx || !nn_row_dev || !accepted_dev || !q_xy_dev || !q_image_dev || !params || !n_objects || !obj_model || !obj_pose || !obj_score || max_objects <= 0) {
		if (ctx) ctx->err = "mc_process_matched_dev: bad argument";
		return MC_ERR_ARG;
	}
	MC_CUDA(cudaSetDevice(ctx->device));
	return process_frame_device(ctx, nullptr, q_xy_dev, q_image_dev, n_queries, params, max_objects, n_objects, obj_model, obj_pose, obj_score, stage_ms,
	                            nn_row_dev, accepted_dev);
}

mc_status mc_process_frame(mc_ctx *ctx, const float *q_desc, const float *q_xy, const int32_t *q_image, int Q, const mc_pipeline_params *params,
                           int max_objects, int32_t *n_objects, int32_t *obj_model, float *obj_pose, float *obj_score, float *stage_ms) {
	if (!ctx || !q_desc || !q_xy || !q_image || !params || !n_objects || Q < 0) { if (ctx) ctx->err = "mc_process_frame: bad argument"; return MC_ERR_ARG; }
	if (!ctx->d_db) { ctx->err = "mc_process_frame: no database uploaded"; return MC_ERR_STATE; }
	if (Q == 0) { *n_objects = 0; return MC_OK; }
	MC_CUDA(cudaSetDevice(ctx->device));
	MC_TRY(reserve(ctx, ctx->q_desc, sizeof(float) * (size_t)Q * ctx->D));
	MC_TRY(reserve(ctx, ctx->q_xy, sizeof(float) * 2 * (size_t)Q));
	MC_TRY(reserve(ctx, ctx->q_image, sizeof(int32_t) * (size_t)Q));
	MC_TRY(h2d(ctx, (float *)ctx->q_desc.p, q_desc, (size_t)Q * ctx->D));
	MC_TRY(h2d(ctx, (float *)ctx->q_xy.p, q_xy, 2 * (size_t)Q));
	MC_TRY(h2d(ctx, (int32_t *)ctx->q_image.p, q_image, (size_t)Q));
	return process_frame_device(ctx, (const float *)ctx->q_desc.p, (const float *)ctx->q_xy.p, (const int32_t *)ctx->q_image.p, Q, params, max_objects,
	                            n_objects, obj_model, obj_pose, obj_score, stage_ms);
}

// ---- frame batches ------------------------------------------------------------------------------
static mc_status check_frames(mc_ctx *ctx, const int32_t *frame_offsets, int n_frames, const char *who) {
	if (!frame_offsets || n_frames <= 0 || frame_offsets[0] != 0) { ctx->err = std::string(who) + ": bad frame_offsets"; return MC_ERR_ARG; }
	for (int f = 0; f < n_frames; f++)
		if (frame_offsets[f + 1] < frame_offsets[f]) { ctx->err = std::string(who) + ": frame_offsets must ascend"; return MC_ERR_ARG; }
	return MC_OK;
}

mc_status mc_process_frames_dev(mc_ctx *ctx, const float *q_desc_dev, const float *q_xy_dev, const int32_t *q_image_dev, const int32_t *frame_offsets,
                                int n_frames, const mc_pipeline_params *params, int max_objects, int32_t *n_objects, int32_t *obj_model,
                                float *obj_pose, float *obj_score, int32_t *frame_info, float *stage_ms) {
	if (!ctx || !params || !n_objects || !obj_model || !obj_pose || !obj_score || max_objects <= 0) { if (ctx) ctx->err = "mc_process_frames_dev: bad argument"; return MC_ERR_ARG; }
	MC_TRY(check_frames(ctx, frame_offsets, n_frames, "mc_process_frames_dev"));
	if (frame_offsets[n_frames] > 0 && (!q_desc_dev || !q_xy_dev || !q_image_dev)) { ctx->err = "mc_process_frames_dev: null query pointer"; return MC_ERR_ARG; }
	MC_CUDA(cudaSetDevice(ctx->device));
	return process_frames_host(ctx, q_desc_dev, q_xy_dev, q_image_dev, frame_offsets, n_frames, params, max_objects, n_objects, obj_model, obj_pose, obj_score,
	                           frame_info, stage_ms);
}

mc_status mc_process_frames(mc_ctx *ctx, const float *q_desc, const float *q_xy, const int32_t *q_image, const int32_t *frame_offsets, int n_frames,
                            const mc_pipeline_params *params, int max_objects, int32_t *n_objects, int32_t *obj_model, float *obj_pose,
                            float *obj_score, int32_t *frame_info, float *stage_ms) {
	if (!ctx || !params || !n_objects || !obj_model || !obj_pose || !obj_score || max_objects <= 0) { if (ctx) ctx->err = "mc_process_frames: bad argument"; return MC_ERR_ARG; }
	MC_TRY(check_frames(ctx, frame_offsets, n_frames, "mc_process_frames"));
	if (!ctx->d_db) { ctx->err = "mc_process_frames: no database uploaded"; return MC_ERR_STATE; }
	const size_t Q = (size_t)frame_offsets[n_frames];
	if (Q > 0 && (!q_desc || !q_xy || !q_image)) { ctx->err = "mc_process_frames: null query pointer"; return MC_ERR_ARG; }
	MC_CUDA(cudaSetDevice(ctx->device));
	MC_TRY(reserve(ctx, ctx->q_desc, sizeof(float) * (Q + 1) * ctx->D));
	MC_TRY(reserve(ctx, ctx->q_xy, sizeof(float) * 2 * (Q + 1)));
	MC_TRY(reserve(ctx, ctx->q_image, sizeof(int32_t) * (Q + 1)));
	MC_TRY(h2d(ctx, (float *)ctx->q_desc.p, q_desc, Q * ctx->D));
	MC_TRY(h2d(ctx, (float *)ctx->q_xy.p, q_xy, 2 * Q));
	MC_TRY(h2d(ctx, (int32_t *)ctx->q_image.p, q_image, Q));
	return process_frames_host(ctx, (const float *)ctx->q_desc.p, (const float *)ctx->q_xy.p, (const int32_t *)ctx->q_image.p, frame_offsets, n_frames,
	                           params, max_objects, n_objects, obj_model, obj_pose, obj_score, frame_info, stage_ms);
}

mc_status mc_process_frames_matched_dev(mc_ctx *ctx, const int32_t *nn_row_dev, const uint8_t *accepted_dev, const float *q_xy_dev,
                                        const int32_t *q_image_dev, const int32_t *frame_offsets, int n_frames, int frame_begin, int frame_end,
                                        const mc_pipeline_params *params, int max_objects, int32_t *frame_info_dev, int32_t *obj_model_dev,
                                        float *obj_pose_dev, float *obj_score_dev) {
	if (!ctx || !nn_row_dev || !accepted_dev || !q_xy_dev || !q_image_dev || !params || !frame_info_dev || !obj_model_dev || !obj_pose_dev ||
	    !obj_score_dev || max_objects <= 0) {
		if (ctx) ctx->err = "mc_process_frames_matched_dev: bad argument";
		return MC_ERR_ARG;
	}
	MC_TRY(check_frames(ctx, frame_offsets, n_frames, "mc_process_frames_matched_dev"));
	if (frame_begin < 0 || frame_end > n_frames || frame_begin > frame_end) { ctx->err = "mc_process_frames_matched_dev: bad frame range"; return MC_ERR_ARG; }
	MC_CUDA(cudaSetDevice(ctx->device));
	return process_frames_device(ctx, nullptr, q_xy_dev, q_image_dev, frame_offsets, frame_begin, frame_end, params, max_objects, nn_row_dev, accepted_dev,
	                             frame_info_dev, obj_model_dev, obj_pose_dev, obj_score_dev, nullptr);
}

size_t mc_frame_shard_slot_bytes(int n_features, const mc_pipeline_params *params) {
	if (!params || n_features <= 0) return 0;
	return frame_shard_slot_bytes(n_features, params);
}

mc_status mc_process_frame_sharded_dev(mc_ctx *ctx, int phase, const int32_t *nn_row_dev, const uint8_t *accepted_dev, const float *q_xy_dev,
                                       const int32_t *q_image_dev, int n_features, const mc_pipeline_params *params, int shard_rank, int shard_world,
                                       void *exchange_dev, int max_objects, int32_t *frame_info_dev, int32_t *obj_model_dev, float *obj_pose_dev,
                                       float *obj_score_dev) {
	if (!ctx || !nn_row_dev || !accepted_dev || !q_xy_dev || !q_image_dev || !params || !exchange_dev || !frame_info_dev || !obj_model_dev ||
	    !obj_pose_dev || !obj_score_dev || max_objects <= 0 || n_features <= 0) {
		if (ctx) ctx->err = "mc_process_frame_sharded_dev: bad argument";
		return MC_ERR_ARG;
	}
	if (shard_world < 1 || shard_rank < 0 || shard_rank >= shard_world) { ctx->err = "mc_process_frame_sharded_dev: bad shard rank / world"; return MC_ERR_ARG; }
	if (phase < 0 || phase > 2) { ctx->err = "mc_process_frame_sharded_dev: phase must be 0, 1 or 2"; return MC_ERR_ARG; }
	MC_CUDA(cudaSetDevice(ctx->device));
	return process_frame_sharded_device(ctx, phase, nn_row_dev, accepted_dev, q_xy_dev, q_image_dev, n_features, params, shard_rank, shard_world, exchange_dev,
	                                    max_objects, frame_info_dev, obj_model_dev, obj_pose_dev, obj_score_dev);
}

mc_status mc_join_lanes(mc_ctx *ctx) {
	if (!ctx) return MC_ERR_ARG;
	MC_CUDA(cudaSetDevice(ctx->device));
	return join_lanes(ctx);
}

} // extern "C"
