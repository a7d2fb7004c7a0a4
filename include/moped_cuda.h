/*
 * moped_cuda.h — C ABI of libmoped_cuda.so, the B200 (sm_100a) implementation of MOPED's
 * data-parallel recognition core. Plain pointers and sizes only; no C++/torch types.
 *
 * One entry point per reference stage `process()` (the drop-in boundary is
 * `virtual void MopedAlg::process(FrameData&)`, moped2/libmoped/src/util.hpp:147); the header-only
 * stage classes in moped_b200/stages/ (MATCH_CUDA, CLUSTER_MEAN_SHIFT_CUDA, POSE_RANSAC_LM_CUDA,
 * FILTER_PROJECTION_CUDA) flatten FrameData into these calls. All citations are relative to
 * /root/reference/.
 *
 * Conventions
 *  - every function returns MC_OK (0) or a negative mc_status; mc_last_error() gives the text.
 *    There is NO CPU fallback: without a usable CUDA device every call fails with MC_ERR_CUDA.
 *  - "host" pointers are ordinary host memory (pinned memory makes the copies asynchronous);
 *    "dev" pointers are device memory of the context's GPU. Ownership always stays with the caller.
 *  - all work is enqueued on the context's stream (mc_set_stream; default = a private stream).
 *    Host-buffer calls synchronise that stream before returning; *_dev calls do not.
 *  - squared distances everywhere; quaternions are (x, y, z, w); poses are quat + translation
 *    (7 floats, Pose::operator[] order, moped2/libmoped/include/moped.hpp:136-164).
 *  - CSR layout: `offsets[n+1]` ascending, group g owns [offsets[g], offsets[g+1]).
 */
#ifndef MOPED_CUDA_H
#define MOPED_CUDA_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct mc_ctx mc_ctx;
typedef int mc_status;

enum {
	MC_OK = 0,
	MC_ERR_CUDA = -1,        /* CUDA runtime/driver error, or no sm_100 device */
	MC_ERR_ARG = -2,         /* bad argument (null pointer, size, unsupported descriptor length) */
	MC_ERR_STATE = -3,       /* call order (e.g. match before db upload) */
	MC_ERR_CAPACITY = -4     /* an output buffer given by the caller is too small */
};

/* match modes */
enum {
	MC_MATCH_TENSOR = 0,     /* fp16 tcgen05 coarse top-k + exact fp32 re-rank + certificate, exact fallback scan */
	MC_MATCH_EXACT = 1       /* exhaustive exact fp32 scan (the reference's Quality=0 arithmetic for every row) */
};

/* ---- context ------------------------------------------------------------------------------ */
mc_status mc_create(mc_ctx **ctx, int device);
void mc_destroy(mc_ctx *ctx);
const char *mc_last_error(const mc_ctx *ctx);
const char *mc_version(void);
/* Use an existing cudaStream_t (e.g. the caller framework's current stream). NULL = private stream. */
mc_status mc_set_stream(mc_ctx *ctx, void *cuda_stream);
mc_status mc_synchronize(mc_ctx *ctx);

/* ---- model database: replaces MATCH_ANN_CPU::Update (kd-tree build),
 *      moped2/libmoped/src/match/MATCH_ANN_CPU.hpp:72-109 ------------------------------------ */
/* desc: N x D row-major fp32, ALREADY L2-normalised by the host stage (MATCH_ANN_CPU.hpp:94);
 * desc_dim = the stage's DescriptorSize (MATCH_ANN_CPU.hpp:113), any length in 1..4096: 128 (SIFT) gets the
 * tensor-core path, every other length is matched by the exhaustive exact scan (same results by definition);
 * xyz: N x 3 (Model::IP::coord3D); model_of_row: N (correspModel); rows are in model order.
 * row_base = global id of row 0 (non-zero when this context holds one shard of an object-sharded DB). */
mc_status mc_db_upload(mc_ctx *ctx, const float *desc, const float *xyz, const int32_t *model_of_row,
                       int64_t n_rows, int desc_dim, int n_models, int64_t row_base);
int64_t mc_db_rows(const mc_ctx *ctx);
/* Object-sharded databases: descriptors stay sharded (mc_db_upload with row_base), but the stages after
 * MATCH need coord3D and the model id of ANY global row, so every rank also holds these two small tables
 * for the whole database (16 B per row). Call after mc_db_upload. */
mc_status mc_db_set_global_tables(mc_ctx *ctx, const float *xyz_all, const int32_t *model_of_row_all, int64_t n_rows_all, int n_models_all);

/* ---- cameras: FrameData::images[i]->{intrinsicLinearCalibration, cameraPose},
 *      moped2/libmoped/include/moped.hpp:226-241 --------------------------------------------- */
mc_status mc_set_cameras(mc_ctx *ctx, const float *K /* n x (fx,fy,cx,cy) */, const float *cam_pose /* n x 7 */, int n_images);

/* ---- MATCH: replaces MATCH_ANN_CPU::process, MATCH_ANN_CPU.hpp:136-178 ---------------------- */
/* q_desc: Q x D normalised queries (host). Outputs (host, query order): nn_row Q x 2 global row ids of the
 * two nearest DB rows, nn_dist Q x 2 their squared distances (reference summation order), accepted Q =
 * (nn_dist[0]/nn_dist[1] < ratio). stats (optional, 4 ints): {#queries certified by the coarse pass,
 * #queries sent to the exact fallback scan, #candidates per query, #DB splits}. */
mc_status mc_match(mc_ctx *ctx, const float *q_desc, int n_queries, float ratio, int mode,
                   int32_t *nn_row, float *nn_dist, uint8_t *accepted, int32_t *stats);
/* Same with device pointers, asynchronous on the context stream. */
mc_status mc_match_dev(mc_ctx *ctx, const float *q_desc_dev, int n_queries, float ratio, int mode,
                       int32_t *nn_row_dev, float *nn_dist_dev, uint8_t *accepted_dev);
/* Object-sharded databases: after all-gathering every shard's (nn_row, nn_dist) — n_shards x Q x 2 each —
 * pick the global two nearest per query (smaller distance, then smaller global row id) and redo the ratio test. */
mc_status mc_match_merge_dev(mc_ctx *ctx, const int32_t *nn_row_all_dev, const float *nn_dist_all_dev, int n_shards,
                             int n_queries, float ratio, int32_t *nn_row_dev, float *nn_dist_dev, uint8_t *accepted_dev);

/* ---- MATCH, moped3d's depth-adaptive variant (SURVEY.md 8f row 4): replaces MATCH_ADAPTIVE_FLANN_CPU::Update / process,
 *      moped3d/libmoped/src/match/MATCH_ADAPTIVE_FLANN_CPU.hpp:101-174,419-490 ---------------------------------------- */
/* Ratio curve of one model over depth: the acceptance threshold rises linearly from ratio_low (depth 0) to ratio_high
 * (depth_peak), stays there up to depth_fade and falls linearly to zero at 2 * depth_fade. */
typedef struct {
	float depth_peak, depth_fade;    /* metres */
	float ratio_low, ratio_high;
} mc_adaptive_model;
/* Host helper, once per model change (what Update() derives per model, :146-169): depth_peak / depth_fade = the depths at which
 * the largest face of the bounding box projects to dimension_peak / dimension_fade pixels under intrinsics K = (fx, fy, cx, cy);
 * ratio_low / ratio_high = points inside [min_ratio_min, min_ratio_max] / [max_ratio_min, max_ratio_max] chosen by the model's
 * feature count (sparse models get the permissive end). The six trailing arguments are the stage's constructor parameters. */
void mc_adaptive_model_init(mc_adaptive_model *out, const float *bbox_min, const float *bbox_max, const float *K, int n_features,
                            float min_ratio_min, float min_ratio_max, float max_ratio_min, float max_ratio_max, float dimension_peak,
                            float dimension_fade);
/* q_desc Q x D normalised queries, q_xy Q x 2 their coord2D (host); depth / fill_distance: height x width planes (host) — the depth
 * component of the IMAGE_TYPE_DEPTH_MAP image and its "<name>.distance" probability map (moped3d/libmoped/include/moped.hpp:261-284);
 * models: one curve per database model. maximum_depth / default_depth / cauchy_scale: 4.0 / 1.0 / 0.1 in the reference (:106-108).
 * Outputs (host, query order): the two nearest rows and squared distances as mc_match returns them, and accepted[i] = the feature lies
 * within maximum_depth and nn_dist[0]/nn_dist[1] is below the blend of its model's curve at the feature's depth and at default_depth
 * (Cauchy weight of the fill distance). The threshold is evaluated on the device, one thread per feature. */
mc_status mc_match_adaptive(mc_ctx *ctx, const float *q_desc, const float *q_xy, int n_queries, const float *depth, const float *fill_distance,
                            int width, int height, const mc_adaptive_model *models, int n_models, float maximum_depth, float default_depth,
                            float cauchy_scale, int32_t *nn_row, float *nn_dist, uint8_t *accepted);
/* moped3d's MATCH step for a batch of n_frames independent frames: what MATCH_ADAPTIVE_CUDA::process does per frame, with ONE
 * matching pass over the queries of all frames.
 *   q_desc Q x D normalised, q_xy Q x 2 (coord2D), q_image Q (imageIdx; NULL = 0), Q = frame_offsets[n_frames]
 *   frame_offsets  host, n_frames + 1 ascending ints from 0: frame f owns features [frame_offsets[f], frame_offsets[f+1])
 *   depth / fill_distance  n_frames x height x width: each frame's depth map and its ".distance" map (one map per frame applies
 *                  to all of its features, as in the single-frame entry)
 *   models / n_models / maximum_depth / default_depth / cauchy_scale  as mc_match_adaptive (models stays a host array)
 * Outputs:
 *   match_offsets  host, n_frames x (n_models + 1): row f = frame f's model-major CSR, GLOBAL indices into the per-match arrays.
 *                  Frame f's matches start at frame_offsets[f], so frames leave gaps (allowed by mc_process_depth_frames*); what the
 *                  per-match arrays hold inside a gap is unspecified.
 *   per match (capacity Q): match_feature (global feature index), match_image, match_xy, match_xyz (coord3D of the nearest row).
 *                  Accepted features of a model appear in feature order (FrameData::matches after MATCH).
 *   optional, per feature: nn_row Q x 2, nn_dist Q x 2, accepted Q (exactly what mc_match_adaptive returns for that frame)
 *   optional frame_info n_frames x 3: {features, accepted matches, status (1 = more than 8192 accepted matches)}
 * Every frame's results are bit for bit those of mc_match_adaptive on that frame's features followed by MATCH_ADAPTIVE_CUDA::emit,
 * whatever the batch. Kernel launches per call do not depend on n_frames.
 * Errors (the context stays usable): MC_ERR_STATE without a database or with an object-sharded one (row_base != 0, or global tables
 * larger than the shard); MC_ERR_ARG for a NULL required pointer, n_frames outside 1..65535, frame_offsets that do not start at 0 or do
 * not ascend, width / height < 1, fewer curves than database models; MC_ERR_CAPACITY when a frame has more than 8192 accepted matches:
 * that frame's row is empty and its frame_info status is 1, every other frame's results are complete. */
mc_status mc_match_adaptive_frames(mc_ctx *ctx, const float *q_desc, const float *q_xy, const int32_t *q_image,
                                   const int32_t *frame_offsets, int n_frames, const float *depth, const float *fill_distance,
                                   int width, int height, const mc_adaptive_model *models, int n_models,
                                   float maximum_depth, float default_depth, float cauchy_scale,
                                   int32_t *match_offsets, int32_t *match_feature, int32_t *match_image, float *match_xy, float *match_xyz,
                                   int32_t *nn_row, float *nn_dist, uint8_t *accepted, int32_t *frame_info);
/* The same with the queries, the planes and the per-match / per-feature outputs on the device. frame_offsets, models, match_offsets
 * and frame_info stay on the host: the call synchronises once, to return the offsets mc_process_depth_frames_dev takes. */
mc_status mc_match_adaptive_frames_dev(mc_ctx *ctx, const float *q_desc_dev, const float *q_xy_dev, const int32_t *q_image_dev,
                                       const int32_t *frame_offsets, int n_frames, const float *depth_dev, const float *fill_distance_dev,
                                       int width, int height, const mc_adaptive_model *models, int n_models,
                                       float maximum_depth, float default_depth, float cauchy_scale,
                                       int32_t *match_offsets, int32_t *match_feature_dev, int32_t *match_image_dev, float *match_xy_dev,
                                       float *match_xyz_dev, int32_t *nn_row_dev, float *nn_dist_dev, uint8_t *accepted_dev,
                                       int32_t *frame_info);
/* moped3d's MATCH step on an object-sharded database, for the frames [frame_begin, frame_end) of a batch of n_frames frames.
 *   packed_all_dev  n_shards blocks back to back in the layout of mc_match_merge_packed_dev: [nn_row Q x 2 int32 | nn_dist Q x 2 fp32]
 *                  per shard, Q = frame_offsets[n_frames]; each block is what mc_match_dev(ratio 1.0, MC_MATCH_TENSOR) writes for the whole
 *                  batch on a context holding one shard (the all-gathered blocks of the ranks)
 * The features of the range get the global two nearest rows (smaller distance, then smaller global row id, as mc_match_merge_dev), then
 * the depth-adaptive test and the model-major lists of mc_match_adaptive_frames_dev. Index conventions:
 *   q_xy_dev, q_image_dev (NULL = image 0), the per-feature and the per-match outputs: GLOBAL feature indices, capacity Q; only the
 *                  slots of the range's features are written (frame f's matches from frame_offsets[f] on)
 *   depth_dev / fill_distance_dev  (frame_end - frame_begin) x height x width: the planes of the range's frames only, starting with frame
 *                  frame_begin (the same planes mc_process_depth_frames_dev takes for these frames)
 *   match_offsets  host, (frame_end - frame_begin) x (n_models + 1): one row per frame of the range, global indices
 *   frame_info     optional host, (frame_end - frame_begin) x 3: {features, accepted matches, status}; status 1 = more than 8192 accepted
 *                  matches, 2 = a row id in the blocks that is neither -1 nor inside the context's tables
 * The context needs coord3D and model tables covering every row id of the blocks: mc_db_set_global_tables on a shard context, or a context
 * holding the whole database (then n_shards = 1 with that context's own mc_match_dev block reproduces mc_match_adaptive_frames_dev).
 * Its descriptors are not read. Every frame of the range equals, bit for bit, what mc_match_adaptive_frames_dev returns for it on one
 * context holding the whole database. Kernel launches per call depend neither on n_frames, nor on the range, nor on n_shards.
 * Errors (the context stays usable): MC_ERR_STATE without tables; MC_ERR_ARG for a NULL required pointer, n_shards < 1, a range outside
 * 0 <= frame_begin <= frame_end <= n_frames (an empty range returns MC_OK and writes nothing), and the cases of mc_match_adaptive_frames;
 * MC_ERR_CAPACITY as mc_match_adaptive_frames (status 1). A row outside the tables is never used as an index: its feature is not accepted,
 * its frame's status is 2 and its row is empty, every other frame is complete, and the call returns MC_ERR_ARG naming the first such
 * frame (before a capacity error). */
mc_status mc_match_adaptive_frames_merged_dev(mc_ctx *ctx, const void *packed_all_dev, int n_shards, const float *q_xy_dev,
                                              const int32_t *q_image_dev, const int32_t *frame_offsets, int n_frames, int frame_begin,
                                              int frame_end, const float *depth_dev, const float *fill_distance_dev, int width, int height,
                                              const mc_adaptive_model *models, int n_models, float maximum_depth, float default_depth,
                                              float cauchy_scale, int32_t *match_offsets, int32_t *match_feature_dev, int32_t *match_image_dev,
                                              float *match_xy_dev, float *match_xyz_dev, int32_t *nn_row_dev, float *nn_dist_dev,
                                              uint8_t *accepted_dev, int32_t *frame_info);

/* The same for shards gathered as ONE packed block each — [nn_row Q x 2 int32 | nn_dist Q x 2 fp32], 16 Q bytes per shard, n_shards
 * blocks back to back: mc_match_dev can write both halves of a rank's block directly (nn_row_dev = block, nn_dist_dev = block + 8 Q
 * bytes), so one all-gather moves everything the merge needs. */
mc_status mc_match_merge_packed_dev(mc_ctx *ctx, const void *packed_all_dev, int n_shards, int n_queries, float ratio,
                                    int32_t *nn_row_dev, float *nn_dist_dev, uint8_t *accepted_dev);

/* ---- CLUSTER: replaces CLUSTER_MEAN_SHIFT_CPU::process,
 *      moped2/libmoped/src/cluster/CLUSTER_MEAN_SHIFT_CPU.hpp:182-199 ------------------------- */
/* matches as CSR over models (match_offsets[n_models+1]); match_image / match_xy per match (host).
 * Output clusters in reference order (model-major, image, surviving-canopy order): cluster_model[c],
 * cluster_offsets[c+1], members (indices into the model's match list, splice order).
 * Capacities: cluster_model/cluster_offsets >= n_matches+1, members >= n_matches. */
mc_status mc_cluster_meanshift(mc_ctx *ctx, const int32_t *match_offsets, const int32_t *match_image, const float *match_xy,
                               int n_models, int n_images, float radius, float merge, int min_pts, int max_iterations,
                               int32_t *n_clusters, int32_t *cluster_model, int32_t *cluster_offsets, int32_t *members);

/* ---- POSE: replaces POSE_RANSAC_LM_DIFF_REPROJECTION_CPU::process,
 *      moped2/libmoped/src/pose/POSE_RANSAC_LM_DIFF_REPROJECTION_CPU.hpp:264-307 -------------- */
typedef struct {
	int32_t max_ransac_tests;        /* MaxRANSACTests */
	int32_t max_lm_tests;            /* MaxLMTests (LM itmax) */
	int32_t max_objects_per_cluster; /* MaxObjectsPerCluster */
	int32_t n_pts_align;             /* NPtsAlign (<= 8) */
	int32_t min_npts_object;         /* MinNPtsObject (strict >) */
	float error_threshold;           /* ErrorThreshold, px^2 */
	uint64_t seed;                   /* RNG stream of this call */
} mc_pose_params;

/* Per-hypothesis evaluation on EXPLICIT (sample positions, initial quaternion) sets — the parity entry
 * point: hypothesis h belongs to cluster hyp_cluster[h]; sample_pos[h*n_pts_align + j] = position inside
 * that cluster. clusters given as CSR over points: pt_xy, pt_xyz, pt_image (host).
 * Outputs per hypothesis (host): n_inliers (-1 = LM failed on the samples), pose_lm (after the sample
 * fit), pose_refit (after the inlier refit, = pose_lm when not refitted), lm_err (2: ||e||^2 of both fits,
 * -2 = no refit), inlier_mask (CSR-aligned: hyp h writes at mask_offsets = h-th prefix of its cluster size;
 * pass NULL to skip). */
mc_status mc_pose_hypotheses(mc_ctx *ctx, const int32_t *cluster_offsets, int n_clusters,
                             const float *pt_xy, const float *pt_xyz, const int32_t *pt_image,
                             const int32_t *hyp_cluster, const int32_t *sample_pos, const float *init_quat, int n_hyp,
                             const mc_pose_params *params,
                             int32_t *n_inliers, float *pose_lm, float *pose_refit, float *lm_err, uint8_t *inlier_mask);

/* The same with every array resident on the device (no inlier masks); asynchronous on the context's stream.
 * The entry BASELINE.json configs[3] (64 clusters x 2048 hypotheses) is measured through. */
mc_status mc_pose_hypotheses_dev(mc_ctx *ctx, const int32_t *cluster_offsets_dev, const float *pt_xy_dev, const float *pt_xyz_dev,
                                 const int32_t *pt_image_dev, const int32_t *hyp_cluster_dev, const int32_t *sample_pos_dev,
                                 const float *init_quat_dev, int n_hyp, const mc_pose_params *params,
                                 int32_t *n_inliers_dev, float *pose_lm_dev, float *pose_refit_dev, float *lm_err_dev);

/* Full RANSAC per (cluster, try): tasks = clusters x max_objects_per_cluster; each task tests up to
 * max_ransac_tests hypotheses (own counter-based RNG) and returns the FIRST successful one in hypothesis
 * order, refitted on its inliers. Outputs (host): found[t], pose[t*7], n_tests[t] (hypotheses consumed). */
mc_status mc_pose_ransac(mc_ctx *ctx, const int32_t *cluster_offsets, int n_clusters,
                         const float *pt_xy, const float *pt_xyz, const int32_t *pt_image,
                         const mc_pose_params *params, uint8_t *found, float *pose, int32_t *n_tests);

/* ---- POSE, moped3d's depth-aware variants (SURVEY.md 8f row 4). variant 0 replaces
 *      POSE_RANSAC_LM_DIFF_BACKPROJECTION_DEPTH_CPU::process (moped3d/libmoped/src/pose/POSE_RANSAC_LM_DIFF_BACKPROJECTION_DEPTH_CPU.hpp:391-470,
 *      the stage of moped3d's shipped pipeline, moped3d/libmoped/src/config.hpp:46); variant 1 replaces
 *      POSE_RANSAC_LM_DIFF_REPROJECTION_DEPTH_CPU::process (…/POSE_RANSAC_LM_DIFF_REPROJECTION_DEPTH_CPU.hpp:357-435).
 * Every correspondence additionally carries pt_world (Match::depthData.coord3D, the back-projected depth-filled point, 3 floats) and
 * pt_cauchy (getCauchyWeight(depthData.fillDistance), computed by the caller with the stage's scale: 0.100 / 25); alpha = the stage's Alpha.
 * The LM takes every sum in levmar's order with unfused multiply-add: results equal the strict-IEEE build of the reference bit for bit.
 * Outputs as for mc_pose_hypotheses / mc_pose_ransac. pt_tie (nullable): each point's index in its model's match list (randSample breaks
 * key ties by it); NULL = position in the cluster. ---- */
mc_status mc_pose_depth_hypotheses(mc_ctx *ctx, int variant, const int32_t *cluster_offsets, int n_clusters,
                                   const float *pt_xy, const float *pt_xyz, const float *pt_world, const float *pt_cauchy, const int32_t *pt_image,
                                   const int32_t *hyp_cluster, const int32_t *sample_pos, const float *init_quat, int n_hyp,
                                   const mc_pose_params *params, float alpha,
                                   int32_t *n_inliers, float *pose_lm, float *pose_refit, float *lm_err, uint8_t *inlier_mask);
/* The explicit-hypothesis entry with every array resident on the device (no inlier masks); asynchronous on the context's stream.
 * max_cluster_size = the largest cluster (sizes the per-warp LM scratch). variant 2 = the moped2 residual in exact-order mode
 * (pt_world_dev / pt_cauchy_dev may be NULL): the configs[3] workload of bench.py --pose-mode exact. */
mc_status mc_pose_depth_hypotheses_dev(mc_ctx *ctx, int variant, const int32_t *cluster_offsets_dev, int max_cluster_size,
                                       const float *pt_xy_dev, const float *pt_xyz_dev, const float *pt_world_dev, const float *pt_cauchy_dev,
                                       const int32_t *pt_image_dev, const int32_t *hyp_cluster_dev, const int32_t *sample_pos_dev,
                                       const float *init_quat_dev, int n_hyp, const mc_pose_params *params, float alpha,
                                       int32_t *n_inliers_dev, float *pose_lm_dev, float *pose_refit_dev, float *lm_err_dev);
mc_status mc_pose_depth_ransac(mc_ctx *ctx, int variant, const int32_t *cluster_offsets, int n_clusters,
                               const float *pt_xy, const float *pt_xyz, const float *pt_world, const float *pt_cauchy, const int32_t *pt_image,
                               const int32_t *pt_tie, const mc_pose_params *params, float alpha,
                               uint8_t *found, float *pose, int32_t *n_tests);

/* ---- FILTER: replaces FILTER_PROJECTION_CPU::process,
 *      moped2/libmoped/src/filter/FILTER_PROJECTION_CPU.hpp:80-162 ---------------------------- */
/* matches as CSR over models (+ image, xy, xyz per match); objects in list order (obj_model, obj_pose).
 * Outputs (host): keep[o], score[o]; clusters of the survivors ordered model-major then list order:
 * cluster_offsets[n_survivors+1], members (indices into the model's match list, ascending).
 * Capacities: cluster_offsets >= n_objects+1, members >= n_matches. */
mc_status mc_filter_projection(mc_ctx *ctx, const int32_t *match_offsets, const int32_t *match_image, const float *match_xy,
                               const float *match_xyz, int n_models, const int32_t *obj_model, const float *obj_pose, int n_objects,
                               int min_points, float feature_distance, float min_score,
                               uint8_t *keep, float *score, int32_t *n_survivors, int32_t *cluster_offsets, int32_t *members);

/* moped3d's FILTER_PROJECTION_DEPTH_CPU::process (moped3d/libmoped/src/filter/FILTER_PROJECTION_DEPTH_CPU.hpp:145-329): the projection
 * filter with a penalty from the depth map. test_offsets / test_xyz: the test points of every model (all its keypoints, or the
 * TestSampleSize the class draws once, :94-118 — the caller's choice, e.g. the stage class FILTER_PROJECTION_DEPTH_CUDA). depth /
 * fill_distance: height x width planes (Image::getDepth of the depth map, getProb of its ".distance" map), depth_K / depth_pose: the
 * depth camera's intrinsics (fx, fy, cx, cy) and pose (quaternion x y z w, translation). An object's score is its projection score
 * minus the penalty (:276); features are owned by the best PROJECTION score (:283), pruning uses the penalised one (:314).
 * Outputs as mc_filter_projection. */
mc_status mc_filter_projection_depth(mc_ctx *ctx, const int32_t *match_offsets, const int32_t *match_image, const float *match_xy,
                                     const float *match_xyz, int n_models, const int32_t *obj_model, const float *obj_pose, int n_objects,
                                     int min_points, float feature_distance, float plausible_sq_distance, float min_score, float depth_fraction,
                                     float min_keypoint_fraction, const int32_t *test_offsets, const float *test_xyz, const float *depth_K,
                                     const float *depth_pose, int width, int height, const float *depth, const float *fill_distance,
                                     uint8_t *keep, float *score, int32_t *n_survivors, int32_t *cluster_offsets, int32_t *members);

/* ---- whole frame on the device (SURVEY.md §8f row 1): MATCH..FILTER2 chained without leaving HBM ---- */
typedef struct {
	float match_ratio; int32_t match_mode;
	float cluster_radius, cluster_merge; int32_t cluster_min_pts, cluster_max_iterations;
	mc_pose_params pose; int32_t filter_min_points; float filter_feature_distance, filter_min_score;
	mc_pose_params pose2; int32_t filter2_min_points; float filter2_feature_distance, filter2_min_score;
} mc_pipeline_params;
void mc_pipeline_default_params(mc_pipeline_params *p);   /* moped2/libmoped/src/config.hpp:83-120 */

/* Queries on the host: q_desc Q x D (normalised), q_xy Q x 2, q_image Q. Results: up to max_objects
 * objects (model id, pose, score) in reference order. stage_ms (optional, 6 floats): device time per stage. */
mc_status mc_process_frame(mc_ctx *ctx, const float *q_desc, const float *q_xy, const int32_t *q_image, int n_queries,
                           const mc_pipeline_params *params, int max_objects,
                           int32_t *n_objects, int32_t *obj_model, float *obj_pose, float *obj_score, float *stage_ms);
/* Same with the queries already resident in HBM (bench `value` leg). Results still land on the host. */
mc_status mc_process_frame_dev(mc_ctx *ctx, const float *q_desc_dev, const float *q_xy_dev, const int32_t *q_image_dev, int n_queries,
                               const mc_pipeline_params *params, int max_objects,
                               int32_t *n_objects, int32_t *obj_model, float *obj_pose, float *obj_score, float *stage_ms);

/* Stages after MATCH only (CLUSTER..FILTER2), from merged nearest neighbours already on the device: the
 * multi-GPU path runs mc_match_dev per shard, all-gathers, mc_match_merge_dev, then this. */
mc_status mc_process_matched_dev(mc_ctx *ctx, const int32_t *nn_row_dev, const uint8_t *accepted_dev, const float *q_xy_dev,
                                 const int32_t *q_image_dev, int n_queries, const mc_pipeline_params *params, int max_objects,
                                 int32_t *n_objects, int32_t *obj_model, float *obj_pose, float *obj_score, float *stage_ms);

/* ---- frame batches (BASELINE.json configs[4]: batched multi-camera stream; SURVEY.md §8f row 1) ----
 * A batch is n_frames INDEPENDENT frames — what the reference does by calling Moped::processImages once per
 * frame (moped2/libmoped/src/moped.cpp:166-194) — given as concatenated query arrays and frame_offsets
 * (n_frames+1 ascending ints on the host, frame f owns queries [frame_offsets[f], frame_offsets[f+1])).
 * MATCH runs once for all queries (one pass over the database); the stages after it run per frame on
 * concurrent lanes (mc_set_tuning). Frame f's objects are exactly those mc_process_frame returns for it.
 * Outputs: n_objects[f]; obj_model / obj_score [f*max_objects + i]; obj_pose [(f*max_objects + i)*7].
 * frame_info (optional, n_frames x 4): {objects, status, accepted matches, clusters after CLUSTER}.
 * stage_ms (optional, 2 floats): device time of MATCH and of CLUSTER..FILTER2 for the whole batch. */
mc_status mc_process_frames(mc_ctx *ctx, const float *q_desc, const float *q_xy, const int32_t *q_image, const int32_t *frame_offsets,
                            int n_frames, const mc_pipeline_params *params, int max_objects,
                            int32_t *n_objects, int32_t *obj_model, float *obj_pose, float *obj_score, int32_t *frame_info, float *stage_ms);
/* Same with the queries already resident in HBM. Results land on the host. */
mc_status mc_process_frames_dev(mc_ctx *ctx, const float *q_desc_dev, const float *q_xy_dev, const int32_t *q_image_dev,
                                const int32_t *frame_offsets, int n_frames, const mc_pipeline_params *params, int max_objects,
                                int32_t *n_objects, int32_t *obj_model, float *obj_pose, float *obj_score, int32_t *frame_info, float *stage_ms);
/* Stages after MATCH for frames [frame_begin, frame_end) of a batch whose merged nearest neighbours (all
 * frames) are on the device — the multi-GPU path: every rank matches all queries against its shard, the
 * (row, distance) pairs are all-gathered and merged (mc_match_merge_dev), then rank r runs its share of the
 * frames here and the per-frame results are all-gathered. Asynchronous; outputs are DEVICE arrays with one
 * slot per processed frame (slot = f - frame_begin): frame_info_dev 4 ints, obj_model_dev max_objects,
 * obj_pose_dev 7*max_objects, obj_score_dev max_objects. */
mc_status mc_process_frames_matched_dev(mc_ctx *ctx, const int32_t *nn_row_dev, const uint8_t *accepted_dev, const float *q_xy_dev,
                                        const int32_t *q_image_dev, const int32_t *frame_offsets, int n_frames, int frame_begin, int frame_end,
                                        const mc_pipeline_params *params, int max_objects, int32_t *frame_info_dev, int32_t *obj_model_dev,
                                        float *obj_pose_dev, float *obj_score_dev);
/* ONE frame with the RANSAC work distributed by cluster over shard_world ranks (north_star; the reference hands its (cluster, try)
 * task list to worker threads, POSE_RANSAC_LM_DIFF_REPROJECTION_CPU.hpp:275-282): every rank holds the merged nearest neighbours of
 * the frame, runs compaction / CLUSTER / FILTER redundantly (identical on all ranks) and the POSE / POSE2 tasks of the clusters c
 * with c % shard_world == shard_rank. A task's random stream depends on its index alone, so the result equals mc_process_matched_dev
 * bit for bit for any shard_world. Three asynchronous calls per frame with the caller's exchange between them:
 *   phase 0 -> all-gather `exchange_dev` in place (slot r = rank r's record) -> phase 1 -> all-gather again -> phase 2.
 * exchange_dev: shard_world x mc_frame_shard_slot_bytes(n_features, params) bytes; this rank writes slot shard_rank only.
 * The same arguments must be passed to all three phases, and no other frame / stage call may run on this context between phase 0 and
 * phase 2 (the frame's intermediate state lives in the context's scratch buffers). Outputs (phase 2, device): frame_info 4 ints {objects, status, accepted
 * matches, clusters after CLUSTER}, obj_model max_objects, obj_pose 7*max_objects, obj_score max_objects — identical on every rank. */
size_t mc_frame_shard_slot_bytes(int n_features, const mc_pipeline_params *params);
mc_status mc_process_frame_sharded_dev(mc_ctx *ctx, int phase, const int32_t *nn_row_dev, const uint8_t *accepted_dev, const float *q_xy_dev,
                                       const int32_t *q_image_dev, int n_features, const mc_pipeline_params *params, int shard_rank, int shard_world,
                                       void *exchange_dev, int max_objects, int32_t *frame_info_dev, int32_t *obj_model_dev, float *obj_pose_dev,
                                       float *obj_score_dev);
/* With mc_set_option("defer_lane_join", 1) mc_process_frames_matched_dev returns WITHOUT ordering the context's stream after the frame
 * lanes, so that work enqueued next on that stream (MATCH and the exchange of the batch's next chunk) overlaps the stages just started;
 * mc_join_lanes orders the context's stream after everything the lanes were given since the last join. */
mc_status mc_join_lanes(mc_ctx *ctx);
/* Scheduling knobs that never change results: frame_lanes = concurrent frames after MATCH in a batch (1..64,
 * default 8); pose_warps_per_task = hypotheses of EVERY RANSAC task tested by the first RANSAC kernel (1..8, default
 * 8: lowest single-frame latency when a task's first hypotheses fail; 1 packs the first hypothesis of four tasks into
 * one warp and wastes nothing when it succeeds — the setting for frame batches); match_chunks = MATCH launches per batch
 * (1..16, default 1): with c > 1 the matching of chunk i+1 overlaps the latency-bound stages of chunk i.
 * 0 keeps the current value. */
mc_status mc_set_tuning(mc_ctx *ctx, int frame_lanes, int pose_warps_per_task, int match_chunks);

/* ---- model-database loader (SURVEY.md 8f row 2): replaces sXML + Moped::addModel,
 *      moped2/libmoped/include/sXML.hpp:55-127, moped2/libmoped/src/moped.cpp:100-158 ---------- */
typedef struct mc_model_db mc_model_db;
mc_status mc_model_db_create(mc_model_db **db);
void mc_model_db_destroy(mc_model_db *db);
const char *mc_model_db_last_error(const mc_model_db *db);
/* Parse `.moped.xml` model files (the format MopedModeling.py / sfm_export_xml.m write) and add them in list order;
 * a model whose name already exists replaces it in place and — as in the reference, whose `found` flag only remembers
 * the last list entry — is also appended unless it was the last model (moped.cpp:138-149). Files are parsed by n_threads host
 * threads (0 = all cores); if any file fails nothing is added. */
mc_status mc_model_db_add_xml_file(mc_model_db *db, const char *path);
mc_status mc_model_db_add_xml_files(mc_model_db *db, const char *const *paths, int n_files, int n_threads);
mc_status mc_model_db_add_xml_buffer(mc_model_db *db, const char *data, int64_t len);
mc_status mc_model_db_remove(mc_model_db *db, const char *name);           /* Moped::removeModel */
int mc_model_db_n_models(const mc_model_db *db);
const char *mc_model_db_model_name(const mc_model_db *db, int i);
mc_status mc_model_db_model_bbox(const mc_model_db *db, int i, float *bbox6 /* min xyz, max xyz */);
/* Rows of one descriptor type in the matcher's numbering (models in order, points in file order,
 * MATCH_ANN_CPU.hpp:85-100); the first desc_size values of each descriptor, L2-normalised over the whole stored
 * descriptor when normalise != 0 (:54-57,94). The returned arrays belong to the database object and stay valid
 * until it changes. */
mc_status mc_model_db_pack(mc_model_db *db, const char *desc_type, int desc_size, int normalise, int64_t *n_rows, const float **desc,
                           const float **xyz, const int32_t **model_of_row, const int32_t **n_pts_per_model);
/* pack (normalised) + mc_db_upload: what modelsUpdated() -> MATCH::Update() amounts to on this path */
mc_status mc_model_db_upload(mc_model_db *db, mc_ctx *ctx, const char *desc_type, int desc_size);
/* binary cache of the parsed models (all descriptor types, unnormalised): parse the XML text once */
mc_status mc_model_db_save(const mc_model_db *db, const char *path);
mc_status mc_model_db_load(mc_model_db *db, const char *path);

/* ---- feature extraction (SURVEY.md 8f row 3): replaces FEAT_SIFT_CPU::process,
 *      moped2/libmoped/src/feat/FEAT_SIFT_CPU.hpp:78-112, i.e. GetKeypoints of the vendored libsiftfast 1.1
 *      (moped2/libmoped/libs/libs.tgz!libsiftfast-1.1-src/libsiftfast.cpp:301-361) ------------------------------ */
/* gray: n_images images of height x width bytes each (Image::data of a 1-channel image, FEAT_SIFT_CPU.hpp:88), all the
 * same size — a camera rig or a stream batch; one set of kernel launches serves the whole batch.
 * double_size != 0 is ScaleOrigin "-1" (DoubleImSize=1, FEAT_SIFT_CPU.hpp:69-76).
 * Outputs, one block of max_keypoints slots per image (image f, keypoint i at slot f*max_keypoints + i), in the order
 * FEAT_SIFT_CPU appends detectedFeatures: counts[f] = keypoints FOUND in image f; xy = coord2D = (col, row) in input
 * pixels; scale_ori (optional) = (scale, orientation); desc = 128 floats (unit length, clamped at 0.2 like the
 * reference's). If an image has more than max_keypoints keypoints the call returns MC_ERR_CAPACITY: counts[f] still holds
 * the number found, the slots hold max_keypoints of them (an unspecified subset). */
mc_status mc_sift_extract(mc_ctx *ctx, const uint8_t *gray, int n_images, int height, int width, int double_size,
                          int max_keypoints, int32_t *counts, float *xy, float *scale_ori, float *desc);
/* Same with every array on the device, asynchronous on the context's stream: desc_dev blocks feed mc_match_dev /
 * mc_process_frames_dev without leaving HBM. counts_dev may exceed max_keypoints (see above). */
mc_status mc_sift_extract_dev(mc_ctx *ctx, const uint8_t *gray_dev, int n_images, int height, int width, int double_size,
                              int max_keypoints, float *xy_dev, float *scale_ori_dev, float *desc_dev, int32_t *counts_dev);
/* ---- UNDISTORTED_IMAGE (UTIL_UNDISTORT), the step both pipelines register before SIFT (pipeline3d_cuda.hpp:2) ---------------- */
/* UNDISTORTED_IMAGE (UTIL_UNDISTORT: cvInitUndistortMap + cvRemap, bilinear, constant border 0) for images of camera `camera`:
 * K = (fx, fy, cx, cy) as given to mc_set_cameras, kc = OpenCV's (k1, k2, p1, p2[, k3]), n_kc 4 or 5; kc == NULL clears.
 * The remap table of a height x width image is built on the host once per call, in double precision in the order of OpenCV's
 * scalar loop, and kept in device memory the context owns (8 bytes per pixel: 2.4 MB for 640x480) until the camera is set again,
 * cleared, or mc_destroy. Images undistorted with it equal cv2.initUndistortRectifyMap(K, kc, None, K, (width, height), CV_32FC1)
 * followed by cv2.remap(INTER_LINEAR, BORDER_CONSTANT, 0) bit for bit (K and kc rounded to float as here).
 * Errors (the previous table stays): MC_ERR_ARG for camera outside 0..15, n_kc other than 4 or 5, a non-finite K or kc, fx or fy
 * equal to 0, height or width outside 8..32767. */
mc_status mc_set_undistortion(mc_ctx *ctx, int camera, const float *K, const float *kc, int n_kc, int height, int width);
/* n_images images of camera `camera` (height x width bytes each) -> out, same layout; one kernel launch for the batch.
 * Errors: MC_ERR_STATE when the camera has no table; MC_ERR_ARG for a NULL pointer, n_images outside 1..65535, a camera outside
 * 0..15 or a size other than the table's. */
mc_status mc_undistort(mc_ctx *ctx, int camera, const uint8_t *gray, int n_images, int height, int width, uint8_t *out);
/* Same with device pointers, asynchronous on the context's stream (gray_dev and out_dev must not overlap): composes with
 * mc_sift_extract_dev for camera rigs. */
mc_status mc_undistort_dev(mc_ctx *ctx, int camera, const uint8_t *gray_dev, int n_images, int height, int width, uint8_t *out_dev);

/* Images in, objects out: FEAT chained to MATCH..FILTER2 for a batch of n_frames single-camera frames of one size (each
 * frame is what Moped::processImages gets with one image, moped2/libmoped/src/moped.cpp:166-194; camera 0 of
 * mc_set_cameras applies to every frame). When camera 0 has an undistortion table (mc_set_undistortion), the uploaded batch is
 * undistorted on the device first (one more launch), as UNDISTORTED_IMAGE runs before SIFT in the reference's pipeline; a size
 * other than the table's returns MC_ERR_ARG before any launch. Without a table the images go to SIFT as given.
 * Descriptors stay in HBM between the steps, normalised on the device with the
 * MATCH stage's expression. Outputs like mc_process_frames; n_features (optional) = keypoints per frame;
 * stage_ms (optional, 3 floats) = device time of FEAT (incl. the image upload and undistortion), MATCH, CLUSTER..FILTER2. */
mc_status mc_process_images(mc_ctx *ctx, const uint8_t *gray, int n_frames, int height, int width, int double_size, int max_keypoints,
                            const mc_pipeline_params *params, int max_objects, int32_t *n_objects, int32_t *obj_model, float *obj_pose,
                            float *obj_score, int32_t *n_features, int32_t *frame_info, float *stage_ms);
/* Images in, objects out for camera rigs: n_frames frames of n_cameras images each, gray = [n_frames][n_cameras][height][width]
 * bytes, all of one size. Frame f is what Moped::processImages gets with n_cameras images: image c of every frame belongs to camera c,
 * whose intrinsics and pose are entry c of mc_set_cameras and whose undistortion table, if it has one, is camera c's of
 * mc_set_undistortion (an image of a camera without a table goes to SIFT as given; one remap launch serves the whole batch, none
 * when no camera of the rig has a table). The frame's query list is the keypoints of camera 0, then camera 1, ..., each in
 * FEAT_SIFT_CPU's order with imageIdx = camera, as FEAT_SIFT_CUDA::process appends them; MATCH..FILTER2 run as in
 * mc_process_frames. Outputs as mc_process_images, except n_features (optional) = n_frames x n_cameras keypoint counts, one per
 * image, in input order. n_cameras = 1 is mc_process_images (same outputs, same launches) with the camera check below.
 * Errors, all before any launch: MC_ERR_ARG for n_cameras outside 1..16, n_frames x n_cameras above 65535, or a camera of the rig
 * whose table is not height x width; MC_ERR_STATE when mc_set_cameras set fewer than n_cameras cameras, and as mc_process_images.
 * An image with more than max_keypoints keypoints returns MC_ERR_CAPACITY; n_features still holds the numbers found. */
mc_status mc_process_rig_images(mc_ctx *ctx, const uint8_t *gray, int n_frames, int n_cameras, int height, int width,
                                int double_size, int max_keypoints, const mc_pipeline_params *params, int max_objects,
                                int32_t *n_objects, int32_t *obj_model, float *obj_pose, float *obj_score,
                                int32_t *n_features, int32_t *frame_info, float *stage_ms);
/* One camera of a rig as mc_process_rig_cameras reads it: the camera's image of frame f is height x width bytes at
 * gray + f * frame_stride. Per-camera buffers [n_frames][height][width] have frame_stride = height * width; camera c of one
 * [n_frames][C][H][W] buffer is gray = base + c * H * W with frame_stride = C * H * W. */
typedef struct {
	const uint8_t *gray;      /* camera c's image of frame 0 */
	int64_t frame_stride;     /* bytes between frames, >= height * width */
	int32_t height, width;    /* this camera's image size, 8..32767 each */
} mc_rig_camera;
/* mc_process_rig_images for rigs whose cameras may differ in image size and whose images may sit in separate buffers: camera c's
 * images are described by cameras[c]. Its intrinsics and pose are entry c of mc_set_cameras; its undistortion table, if it has one,
 * is camera c's of mc_set_undistortion and must be that camera's own size. Cameras of one size form a group and share one SIFT batch
 * (and one remap launch when a camera of the group has a table); the groups' keypoints are then merged on the device so that frame f's
 * query list is camera 0's keypoints, then camera 1's, ..., each in FEAT_SIFT_CPU's order with imageIdx = camera, exactly as
 * mc_process_rig_images orders them. When every camera has one size the call issues mc_process_rig_images' launches. Outputs as
 * mc_process_rig_images: n_features (optional) = n_frames x n_cameras counts, frame-major; stage_ms (optional, 3 floats) with FEAT
 * including the merge. Errors, all before any copy or launch: MC_ERR_ARG for n_cameras outside 1..16, a NULL pointer, n_frames,
 * max_keypoints or max_objects below 1, a size outside 8..32767, frame_stride < height * width, a table whose size is not its
 * camera's, more than 65535 images, or more than 7281 images of one size (SIFT's batch limit); MC_ERR_STATE when mc_set_cameras set
 * fewer than n_cameras cameras, no database is uploaded or its descriptors are not 128-d. An image with more than max_keypoints
 * keypoints returns MC_ERR_CAPACITY; n_features still holds the numbers found. */
mc_status mc_process_rig_cameras(mc_ctx *ctx, const mc_rig_camera *cameras, int n_cameras, int n_frames, int double_size,
                                 int max_keypoints, const mc_pipeline_params *params, int max_objects, int32_t *n_objects,
                                 int32_t *obj_model, float *obj_pose, float *obj_score, int32_t *n_features, int32_t *frame_info,
                                 float *stage_ms);
/* The same with every cameras[c].gray a device pointer (the array `cameras` itself on the host); results on the host, like
 * mc_process_frames_dev. A group whose cameras already lie [frame][camera-in-group] in one buffer is read in place; other
 * groups are gathered with device-to-device copies. The images are not modified. */
mc_status mc_process_rig_cameras_dev(mc_ctx *ctx, const mc_rig_camera *cameras, int n_cameras, int n_frames, int double_size,
                                     int max_keypoints, const mc_pipeline_params *params, int max_objects, int32_t *n_objects,
                                     int32_t *obj_model, float *obj_pose, float *obj_score, int32_t *n_features,
                                     int32_t *frame_info, float *stage_ms);
/* FEAT alone for the frames mc_process_rig_cameras takes: the front half of that call (the upload or in-place read, the remap of each
 * size group with a table, SIFT per size group and the merge into frame-major order), with the query arrays left in the caller's device
 * buffers instead of going on to MATCH. No database is needed. For hosts that run MATCH themselves (an object-sharded database, see
 * INTEGRATION.md §4c) or a step of their own between FEAT and MATCH (moped3d's DEPTHPROP before mc_process_depth_queries_dev).
 *   q_desc_dev   n_frames x n_cameras x max_keypoints rows of 128 floats, 16-byte aligned: the descriptors, normalised with MATCH's
 *                expression (the kernels store them as float4)
 *   q_xy_dev     the same number of rows of 2 floats, 8-byte aligned (coord2D); q_image_dev the same number of ints (imageIdx = camera)
 *                The call cannot see the buffers' sizes: each must hold all those rows, since SIFT writes up to max_keypoints per image
 *                before the counts are known.
 *   frame_offsets  host, n_frames + 1 ints: frame f owns rows [frame_offsets[f], frame_offsets[f+1]); rows from frame_offsets[n_frames]
 *                on are unspecified
 *   n_features   optional host, n_frames x n_cameras keypoint counts, frame-major; feat_ms optional host, 1 float: device time of FEAT
 * The arrays are exactly what mc_process_rig_cameras hands to MATCH: mc_process_frames_dev on them returns what mc_process_rig_cameras
 * returns, and the call issues that call's launches and copies before MATCH. The call synchronises the context's stream once, to read
 * the offsets. Errors, all before any copy or launch: those of mc_process_rig_cameras except the database's and max_objects, plus
 * MC_ERR_ARG for a NULL or misaligned q_desc_dev, q_xy_dev or q_image_dev and a NULL frame_offsets. An image with more than max_keypoints
 * keypoints returns
 * MC_ERR_CAPACITY; n_features still holds the numbers found. */
mc_status mc_extract_rig_cameras(mc_ctx *ctx, const mc_rig_camera *cameras, int n_cameras, int n_frames, int double_size, int max_keypoints,
                                 float *q_desc_dev, float *q_xy_dev, int32_t *q_image_dev, int32_t *frame_offsets, int32_t *n_features,
                                 float *feat_ms);
/* The same with every cameras[c].gray a device pointer, as mc_process_rig_cameras_dev reads them. */
mc_status mc_extract_rig_cameras_dev(mc_ctx *ctx, const mc_rig_camera *cameras, int n_cameras, int n_frames, int double_size, int max_keypoints,
                                     float *q_desc_dev, float *q_xy_dev, int32_t *q_image_dev, int32_t *frame_offsets, int32_t *n_features,
                                     float *feat_ms);
/* test/bench introspection: one plane of the scale-space left by the last extraction (stack 0 Gaussian 0..5, 1 DoG 0..4,
 * 2 gradient magnitude 0..2, 3 orientation 0..2); out may be NULL to query the octave's size. After a mc_process_rig_cameras*
 * call with cameras of several sizes it is the scale-space of the last size group's batch. */
mc_status mc_sift_read_plane(mc_ctx *ctx, int frame, int octave, int stack, int index, float *out, int32_t *rows, int32_t *cols);

/* ---- moped3d clustering (SURVEY.md 8f row 4): replaces CLUSTER_LINKAGE_CPU::process for the matches of ONE model,
 *      moped3d/libmoped/src/cluster/CLUSTER_LINKAGE_CPU.hpp:577-704 ------------------------------------------------------- */
/* match_xy n x 2 (coord2D), match_xyz n x 3 (model coord3D), match_world n x 3 (depthData.coord3D, the back-projected point);
 * depth / fill_distance: height x width row-major maps (Image::getDepth / the ".distance" probability map, moped.hpp:262-300).
 * Parameters as the constructor's: cutoff (Cutoff), min_pts (MinPts, strict >), use_3d_filter (0 none, 1 sum, 2 product),
 * linkage_type (0 minimum, 1 average, 2 maximum), sigma_2d / sigma_3d (-1 = average nearest-neighbour distance). Outputs
 * (host): clusters in the reference's order, members in its list order; capacities n+1 / n. similarity_out (optional,
 * n x n): the blended similarity matrix the agglomeration ran on. n_matches <= 2048. */
mc_status mc_cluster_linkage(mc_ctx *ctx, const float *match_xy, const float *match_xyz, const float *match_world, int n_matches,
                             const float *depth, const float *fill_distance, int width, int height,
                             float cutoff, int min_pts, int use_3d_filter, int linkage_type, float sigma_2d, float sigma_3d,
                             int32_t *n_clusters, int32_t *cluster_offsets, int32_t *members, float *similarity_out);
/* hierarchicalCluster (:414-531) alone, on a caller-supplied n x n similarity matrix (host) */
mc_status mc_linkage_agglomerate(mc_ctx *ctx, const float *similarity, int n, float cutoff, int min_pts, int linkage_type,
                                 int32_t *n_clusters, int32_t *cluster_offsets, int32_t *members);

/* ---- moped3d frames on the device: CLUSTER -> POSE -> FILTER -> POSE2 -> FILTER2 of moped3d's shipped pipeline
 *      (moped3d/libmoped/src/config.hpp:45-49) in one call, from FrameData as DEPTHPROP leaves it ------------------------------- */
typedef struct {
	int32_t variant;              /* 0 = POSE_RANSAC_LM_DIFF_BACKPROJECTION_DEPTH (shipped), 1 = ..._REPROJECTION_DEPTH; the Cauchy
	                               * scale of the fill distance follows (0.100 / 25.0) */
	float cluster_cutoff; int32_t cluster_min_pts, cluster_use_3d_filter, cluster_linkage_type;   /* CLUSTER_LINKAGE, as mc_cluster_linkage */
	float cluster_sigma_2d, cluster_sigma_3d;
	mc_pose_params pose;  float pose_alpha;                                                      /* POSE (+ Alpha) */
	int32_t filter_min_points;  float filter_feature_distance,  filter_min_score;                /* FILTER (FILTER_PROJECTION) */
	mc_pose_params pose2; float pose2_alpha;                                                     /* POSE2 */
	int32_t filter2_min_points; float filter2_feature_distance, filter2_min_score;               /* FILTER2 */
} mc_depth_pipeline_params;

/* the parameters addCudaRecognition3d registers (stages/pipeline3d_cuda.hpp; moped3d config.hpp:45-49); RANSAC seeds 1 and 2 */
void mc_depth_pipeline_default_params(mc_depth_pipeline_params *p);

/* A batch of n_frames frames (n_frames = 1: one frame). Per frame, the matches of every model as DEPTHPROP leaves them:
 *   match_offsets  host, n_frames x (n_models + 1): row f is frame f's model-major CSR, global indices into the per-match arrays
 *                  (ascending within a row; rows need not be contiguous)
 *   per match      match_image (imageIdx), match_xy (coord2D, 2), match_xyz (coord3D, 3), match_world (depthData.coord3D, 3),
 *                  match_fill (depthData.fillDistance), in FrameData::matches[model] order
 *   depth / fill_distance  n_frames x height x width: the depth map and its ".distance" map of each frame
 * Cameras come from mc_set_cameras (MC_ERR_STATE without them); no database is needed.
 * Outputs as mc_process_frames: n_objects[f], obj_model / obj_score [f * max_objects + i], obj_pose [(f * max_objects + i) * 7],
 * frame_info (optional) [4f..4f+3] = {objects, status (1 = a match outside the depth map), matches, clusters after CLUSTER}.
 * stage_ms (optional, 5 floats): device time of CLUSTER, POSE, FILTER, POSE2, FILTER2 summed over the frames; with it the
 * frames run one after another on one lane, without it they are dealt to the frame lanes (mc_set_tuning).
 * Every frame gives exactly the result of the stage-by-stage calls (mc_cluster_linkage per model, mc_pose_depth_ransac with the
 * match index as tie id, mc_filter_projection, ...). The models of a frame are clustered together: one launch per linkage kernel.
 * Errors: MC_ERR_ARG for a model with more than 2048 matches in a frame, cluster_cutoff <= -1, n_pts_align outside 1..8,
 * variant outside 0..1, offsets that do not ascend, or a match outside its frame's depth map (checked before any launch);
 * MC_ERR_CAPACITY when a frame has more than max_objects objects (n_objects[f] holds the true count) or when the sum over a
 * frame's models of n^2 exceeds 2^24 (the similarity matrices and merge lists would take more than 400 MB per lane). */
mc_status mc_process_depth_frames(mc_ctx *ctx, const int32_t *match_offsets, int n_frames, int n_models,
                                  const int32_t *match_image, const float *match_xy, const float *match_xyz, const float *match_world,
                                  const float *match_fill, const float *depth, const float *fill_distance, int width, int height,
                                  const mc_depth_pipeline_params *params, int max_objects,
                                  int32_t *n_objects, int32_t *obj_model, float *obj_pose, float *obj_score, int32_t *frame_info, float *stage_ms);
/* The same with the per-match arrays and the maps resident on the device (match_offsets and the outputs stay on the host).
 * A match outside the depth map is found on the device: its frame reads nothing out of range, reports status 1 and no
 * objects, and the call returns MC_ERR_ARG naming the first such frame. */
mc_status mc_process_depth_frames_dev(mc_ctx *ctx, const int32_t *match_offsets, int n_frames, int n_models,
                                      const int32_t *match_image_dev, const float *match_xy_dev, const float *match_xyz_dev,
                                      const float *match_world_dev, const float *match_fill_dev, const float *depth_dev,
                                      const float *fill_distance_dev, int width, int height, const mc_depth_pipeline_params *params,
                                      int max_objects, int32_t *n_objects, int32_t *obj_model, float *obj_pose, float *obj_score,
                                      int32_t *frame_info, float *stage_ms);

/* moped3d's MATCH -> (DEPTHPROP's per-feature depth data, gathered per match) -> CLUSTER -> POSE -> FILTER -> POSE2 -> FILTER2 for a
 * batch of n_frames independent frames, in one call: features in, objects out.
 *   q_desc, q_xy, q_image, frame_offsets, depth / fill_distance, models .. cauchy_scale  as mc_match_adaptive_frames
 *   q_world Q x 3, q_fill Q  DEPTHPROP's depthData.coord3D and depthData.fillDistance of every feature (required when Q > 0)
 *   params, max_objects, outputs  as mc_process_depth_frames: n_objects[f], obj_model / obj_score [f * max_objects + i],
 *                  obj_pose [(f * max_objects + i) * 7]
 *   frame_info     optional, n_frames x 4: {objects, status, accepted matches, clusters after CLUSTER}
 *   stage_ms       optional, 2 floats: device time of MATCH (cascade, finalize, compaction), then of CLUSTER..FILTER2 (events on the
 *                  context's stream around the fork to the frame lanes and their join: the frames stay dealt to the lanes)
 * Every frame's objects and frame_info equal mc_match_adaptive_frames_dev, a gather of q_world / q_fill through match_feature and
 * mc_process_depth_frames_dev on the same batch, bit for bit. The per-match arrays stay in the context's memory; the call synchronises
 * once between MATCH and CLUSTER (the chain's plan needs the per-model counts) and once for the objects. Kernel launches per call are
 * those of mc_match_adaptive_frames_dev plus those of mc_process_depth_frames_dev on the same batch.
 * A frame that fails gets status != 0 and no objects; every other frame is complete and the context stays usable:
 *   1  an accepted match outside the frame's depth map (MATCH clamps pixels into the map, so a feature at x == width or x < 0 can be
 *      accepted; nothing is read out of range)                                                         MC_ERR_ARG
 *   2  a row id in the gathered blocks outside the tables (mc_process_depth_queries_merged_dev)        MC_ERR_ARG
 *   3  more than 8192 accepted matches (accepted matches reported as 0: the lists are empty)          MC_ERR_CAPACITY
 *   4  a model with more than 2048 matches, or more than 2^24 similarity entries over the frame's models MC_ERR_CAPACITY
 *   0  with more than max_objects objects (n_objects[f] holds the true count)                          MC_ERR_CAPACITY
 * The call returns the code of the first failed frame, MC_ERR_ARG before MC_ERR_CAPACITY.
 * Other errors: MC_ERR_STATE without a database, with an object-sharded one, or without cameras; MC_ERR_ARG for a NULL required pointer
 * (q_world / q_fill included) and the argument errors of mc_match_adaptive_frames and mc_process_depth_frames. */
mc_status mc_process_depth_queries(mc_ctx *ctx, const float *q_desc, const float *q_xy, const int32_t *q_image, const float *q_world,
                                   const float *q_fill, const int32_t *frame_offsets, int n_frames, const float *depth, const float *fill_distance,
                                   int width, int height, const mc_adaptive_model *models, int n_models, float maximum_depth, float default_depth,
                                   float cauchy_scale, const mc_depth_pipeline_params *params, int max_objects, int32_t *n_objects,
                                   int32_t *obj_model, float *obj_pose, float *obj_score, int32_t *frame_info, float *stage_ms);
/* The same with q_* and the planes on the device; frame_offsets, models and the outputs stay on the host. */
mc_status mc_process_depth_queries_dev(mc_ctx *ctx, const float *q_desc_dev, const float *q_xy_dev, const int32_t *q_image_dev,
                                       const float *q_world_dev, const float *q_fill_dev, const int32_t *frame_offsets, int n_frames,
                                       const float *depth_dev, const float *fill_distance_dev, int width, int height,
                                       const mc_adaptive_model *models, int n_models, float maximum_depth, float default_depth,
                                       float cauchy_scale, const mc_depth_pipeline_params *params, int max_objects, int32_t *n_objects,
                                       int32_t *obj_model, float *obj_pose, float *obj_score, int32_t *frame_info, float *stage_ms);
/* One rank of an object-sharded database: the all-gathered mc_match_dev blocks take the place of the matching pass, for frames
 * [frame_begin, frame_end) of the batch, with the conventions of mc_match_adaptive_frames_merged_dev: q_xy_dev, q_image_dev, q_world_dev,
 * q_fill_dev hold the whole batch (global feature ids); depth_dev / fill_distance_dev hold the range's planes only; n_objects,
 * frame_info and the obj_* rows are one per frame of the range. Every frame equals mc_process_depth_queries_dev on one context holding
 * the whole database. An empty range returns MC_OK and writes nothing. */
mc_status mc_process_depth_queries_merged_dev(mc_ctx *ctx, const void *packed_all_dev, int n_shards, const float *q_xy_dev,
                                              const int32_t *q_image_dev, const float *q_world_dev, const float *q_fill_dev,
                                              const int32_t *frame_offsets, int n_frames, int frame_begin, int frame_end, const float *depth_dev,
                                              const float *fill_distance_dev, int width, int height, const mc_adaptive_model *models,
                                              int n_models, float maximum_depth, float default_depth, float cauchy_scale,
                                              const mc_depth_pipeline_params *params, int max_objects, int32_t *n_objects, int32_t *obj_model,
                                              float *obj_pose, float *obj_score, int32_t *frame_info, float *stage_ms);

/* moped3d's FILTER_PROJECTION_DEPTH_CPU as FILTER and / or FILTER2 of the chain above (all five entries: mc_process_depth_frames*,
 * mc_process_depth_queries*), for a pipeline that registers FILTER_PROJECTION_DEPTH_CUDA in place of FILTER_PROJECTION_CUDA. */
typedef struct {
	float plausible_sq_distance, depth_fraction, min_keypoint_fraction;  /* PlausibleSqDistance, DepthFraction, MinKeypointFraction */
	float depth_K[4];                                                    /* the depth map's intrinsics (fx, fy, cx, cy) */
	float depth_pose[7];                                                 /* the depth map's cameraPose (quat x y z w, t) */
} mc_depth_filter_params;
/* step 0 = FILTER, 1 = FILTER2 of the mc_process_depth_frames* / mc_process_depth_queries* chain. p != NULL: that step runs
 * FILTER_PROJECTION_DEPTH with these parameters and these test points (test_offsets[n_models + 1] from 0, test_xyz model-major,
 * copied to the device now). MinPoints / FeatureDistance / MinScore still come from mc_depth_pipeline_params. p == NULL: the step
 * goes back to FILTER_PROJECTION (the default).
 * Each step keeps its own table (each FILTER_PROJECTION_DEPTH_CPU instance draws its own TestSampleSize points), in device memory the
 * context owns until the step is set again or mc_destroy: 12 bytes per test point, uploaded once and not per batch. A frame's depth
 * and ".distance" planes are the ones the chain call takes; the depth camera's matrix is computed from depth_pose as
 * mc_filter_projection_depth computes it, so every frame equals the stage-by-stage calls with mc_filter_projection_depth bit for bit.
 * The penalty kernel adds one launch per depth-filtered step and frame; stage_ms counts it in FILTER / FILTER2.
 * Errors (the previous setting stays): MC_ERR_ARG for a NULL ctx, a step outside 0..1, n_models < 1, test_offsets that do not start at 0
 * or do not ascend, or a NULL test_xyz with points. A chain call whose n_models differs from a set table's returns MC_ERR_ARG before any
 * launch; an object-sharded context (mc_process_depth_queries_merged_dev) takes global model ids, so every rank holds the whole table. */
mc_status mc_set_depth_filter(mc_ctx *ctx, int step, const mc_depth_filter_params *p, const int32_t *test_offsets, const float *test_xyz,
                              int n_models);

/* Named integer options (scheduling / kernel-shape choices; unknown keys are an error):
 *   "pose_fit_thread_min"  mc_pose_hypotheses* calls with at least this many hypotheses and no inlier masks run one
 *                          THREAD per hypothesis instead of one 8-lane group (default 16384; 1 = always)
 *   "pose_fit_stream"      != 0 (default): those thread-per-hypothesis calls run the persistent phase-synchronous kernel (a finished
 *                          lane fetches the next hypothesis at once; one residual evaluation per warp trip serves the start point,
 *                          a Jacobian column or an LM trial point) followed by a scoring kernel; 0: the one-launch kernel (A/B aid).
 *                          Same arithmetic per hypothesis.
 *   "depth_team_lanes"     32 (default) or 8: lanes that share one explicit hypothesis in mc_pose_depth_hypotheses* (8 = four hypotheses
 *                          per warp). Results do not depend on it (the LM keeps levmar's summation order for any team width).
 *   "linkage_cached"       != 0: mc_cluster_linkage / mc_linkage_agglomerate / mc_process_depth_frames* with average linkage keep a cached maximum per row
 *                          (same merge sequence and clusters; O(n) per merge instead of an O(n^2) scan). Default 1 (2.7x at 600 matches
 *                          on B200); 0 = the O(n^2)-scan kernel.
 *   "pose_exact_order"     != 0: mc_pose_hypotheses / mc_pose_ransac (host entries) run the order-preserving LM of the depth stages
 *                          (pose_depth.cu, lm_exact.cuh) with the moped2 residual: every sum in levmar's order, unfused multiply-add —
 *                          poses, inlier masks and ||e||^2 equal the strict-IEEE build of POSE_RANSAC_LM_DIFF_REPROJECTION_CPU bit for
 *                          bit (slower than the default kernels, which re-associate; the frame pipeline keeps the default).
 *   "lm_finite_check"      != 0: the depth pose stages stop an LM whose ||e||^2 became non-finite with LM_ERROR, like a strict-IEEE
 *                          build of levmar (lm_core.c:551,732); 0 (default): the test is folded away as in the reference's
 *                          -ffast-math build.
 *   "ransac_fused"         != 0: mc_pose_ransac / the frame pipeline use the single one-CTA-per-task RANSAC kernel
 *                          instead of the staged kernels (same results; kept for A/B measurements)
 *   "defer_lane_join"      != 0: see mc_join_lanes (default 0)
 *   "match_coarse_kind"    1 (default): MC_MATCH_TENSOR runs the 8-bit integer coarse pass (tcgen05 kind::i8, twice the fp16 MMA
 *                          rate) first and the fp16 pass only for the queries whose certificate it fails; 0: fp16 pass for all
 *                          queries. Same results bit for bit (both end in the exact re-rank and, failing the certificate, in the
 *                          exhaustive scan).
 *   "match_splits"         database splits per query tile in the tensor-core coarse pass (every split of a query keeps its own candidate
 *                          lists); 0 (default) = chosen from the grid and the shard size. A tuning knob: the cascade certifies or
 *                          re-does every query, so results never depend on it.
 *   "match_stagger"        != 0 (default): the CTAs that scan the same database split at the same time start at different tiles
 *                          (kept as a switch for A/B measurements; results do not depend on it)
 *   "stage_sm_partition"   0 (default) or a multiple of 8 up to 96: partition the GPU with CUDA green contexts — this many SMs for the
 *                          streams of the frame lanes (the stages after MATCH), the rest for the stream the persistent coarse matching
 *                          kernel runs on — so that MATCH of one batch or chunk really runs beside the stages of the previous one
 *                          (without it a stage CTA on an SM keeps a whole matching CTA out). Existing lanes are recreated.
 *                          mc_sm_partition reports the SM counts the driver granted.
 *   "match_reserve_sms"    0..64 (default 0): the persistent coarse matching kernel runs on (SMs - this many) CTAs, so that
 *                          concurrent work (the frame lanes' stage kernels of an earlier chunk or step) finds free SMs
 *   "frame_graphs"         != 0 (default): mc_process_frames* replay one CUDA graph per frame for the stages after
 *                          MATCH instead of ~40 kernel launches (same kernels, same results)
 *   "ransac_merge_levels"  != 0 (default): the staged RANSAC tests the 36 hypotheses after the first round in one launch (8-warp CTAs)
 *                          instead of 4 and then 32 in two: a task whose first hypotheses fail costs one more LM chain latency instead
 *                          of two, at the price of more speculative fits (CLUSTER..FILTER2 of a 64-frame batch 3.2 -> 2.7 ms with 4
 *                          first-round hypotheses per task). Same winner (the lowest successful hypothesis index).
 *   "batch_graph"          != 0 (default): the stage chains of ALL frames of an mc_process_frames* call are captured into ONE CUDA graph
 *                          (a branch per lane) and replayed with one launch per batch: graph branches are not bound by the 32
 *                          hardware stream connections, so 64 frames on 64 lanes run together instead of in two rounds. Not used
 *                          with "defer_lane_join" / an SM partition or several MATCH chunks. Same kernels, same results.
 *   "sift_two_pass"        != 0: mc_sift_extract* blur with the separate row / column kernels instead of the fused
 *                          shared-memory kernel (same bits; kept for A/B measurements)
 *   "sift_describe_gather" != 0: descriptors by the cell-gather kernel (one CTA per keypoint) instead of the default
 *                          warp-per-keypoint kernel with private accumulators (same terms, other summation order) */
mc_status mc_set_option(mc_ctx *ctx, const char *key, int64_t value);

/* ---- introspection for tests and bench ------------------------------------------------------ */
/* number of kernels launched by this context since creation (bench.py's gpu_launches) */
int64_t mc_kernel_launches(const mc_ctx *ctx);
/* when on, CUDA events are recorded on the context stream around the dominant kernel (the tcgen05 coarse
 * matching kernel); mc_profile_read waits for the last such launch and returns its device time (ms) */
mc_status mc_set_profiling(mc_ctx *ctx, int on);
mc_status mc_profile_read(mc_ctx *ctx, float *coarse_kernel_ms);
/* MATCH bookkeeping of the LAST mc_match_dev / mc_process_frame* / mc_process_frames* matching pass on this context (waits for the
 * stream): stats = {#queries certified by the coarse pass, #queries sent to the exhaustive fallback scan, #coarse candidates
 * per query, #DB splits}; certified + fallback == the queries of that pass. Exact-mode passes report {0, Q, 0, 0}. */
mc_status mc_match_last_stats(mc_ctx *ctx, int32_t *stats);
/* The same pass by tier of the matching cascade: tiers = {#queries, #certified by the 8-bit integer coarse pass, #certified by
 * the fp16 coarse pass, #sent to the exhaustive exact scan}; the last three add up to the first. Every tier returns the exact
 * scan's bits. */
mc_status mc_match_tier_stats(mc_ctx *ctx, int32_t *tiers);
/* sms = {SMs (persistent CTAs) of the coarse matching kernel, SMs of the stage partition (0 = the GPU is not partitioned)} */
mc_status mc_sm_partition(mc_ctx *ctx, int32_t *sms);
/* same for feature extraction: summed device time of the five octave-0 Gaussian+DoG launches (the dominant kernel of
 * mc_sift_extract*) of the last extraction, and their algorithmic bytes (1 plane read + 2 planes written per launch) */
mc_status mc_sift_profile_read(mc_ctx *ctx, float *blur_ms, double *algorithmic_bytes);

#ifdef __cplusplus
}
#endif
#endif /* MOPED_CUDA_H */
