// adaptive.cu — moped3d's MATCH step on the device: the exact two nearest rows of every feature (match.cu) followed by the
// depth-adaptive ratio test as a finalize kernel, plus the host-side derivation of a model's ratio curve.
//
// Replaces MATCH_ADAPTIVE_FLANN_CPU::Update / process (moped3d/libmoped/src/match/MATCH_ADAPTIVE_FLANN_CPU.hpp:101-174,419-490).
// The reference looks a depth up per feature, evaluates a per-model piecewise-linear threshold on the host and then tests
// dx[0]/dx[1] against it; here the curves of all models are a small table in device memory (16 bytes per model), the depth and
// fill-distance planes are uploaded once per frame, and one thread per feature reads its pixel, its nearest row's model and that
// model's curve (adaptive_threshold.cuh) — the decision leaves the device as one byte per feature.
//
// Frame batches (mc_match_adaptive_frames*): ONE matching pass over the queries of all frames (query tiles of 256 straddle
// frames; every query's rows are certified exact, so nothing depends on the batching), the same finalize kernel with a frame
// dimension (each frame reads its own planes), and the compaction of the moped2 frame chain (k_match_compact, one CTA per frame)
// writing every frame's model-major match lists from the frame's first query id on — the layout mc_process_depth_frames_dev takes.
//
// Object-sharded databases (mc_match_adaptive_frames_merged_dev): every rank matches the whole batch against its shard (mc_match_dev)
// and the packed blocks are all-gathered; one kernel merges the blocks' top-2 pairs for the features of a frame range and takes the
// adaptive decision, then the same compaction runs over the range's frames.
#include "common.cuh"
#include "adaptive_threshold.cuh"
#include "top2.cuh"

#include <cmath>
#include <cstring>

namespace mc {

// frame f = blockIdx.y owns queries [frame_offsets[f], frame_offsets[f+1]) and the planes at f * width * height;
// frame_offsets = nullptr: one frame of Q queries
__global__ void k_match_finalize_adaptive(const int32_t *__restrict__ nn_row, const float *__restrict__ nn_dist, int Q, const int32_t *__restrict__ frame_offsets,
                                          const float *__restrict__ q_xy, const float *__restrict__ depth, const float *__restrict__ fill, int width, int height,
                                          const int32_t *__restrict__ model_of_row, int64_t table_base, const mc_adaptive_model *__restrict__ curves,
                                          int n_models, AdaptiveParams P, uint8_t *__restrict__ accepted) {
	const int f = blockIdx.y;
	const int lo = frame_offsets ? frame_offsets[f] : 0, hi = frame_offsets ? frame_offsets[f + 1] : Q;
	const int i = lo + blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= hi) return;
	bool ok = false;
	const int r0 = nn_row[2 * i], r1 = nn_row[2 * i + 1];
	if (r0 >= 0 && r1 >= 0) {
		const int px = adaptive_pixel(q_xy[2 * i], q_xy[2 * i + 1], width, height);
		const int m = model_of_row[r0 - table_base];
		const float *dp = depth + (size_t)f * width * height, *fp = fill + (size_t)f * width * height;   // (offset here, not before the branch: the single-frame register count)
		if (m >= 0 && m < n_models) ok = adaptive_accept(curves[m], dp[px], fp[px], nn_dist[2 * i], nn_dist[2 * i + 1], P);
	}
	accepted[i] = ok ? 1 : 0;
}

// The same decision on the global top-2 of gathered shard blocks: packed_all = n_shards blocks [nn_row Q x 2 | nn_dist Q x 2], merged by
// k_match_merge's rule (top2.cuh). frame f = blockIdx.y owns features [frame_offsets[f], frame_offsets[f+1]) (global ids) and the
// planes at f * width * height. The blocks come from other processes: a row id that is neither -1 nor inside the tables
// [table_base, table_base + table_rows) is never used as an index — the feature is rejected and bad[f] set.
__global__ void k_match_merge_adaptive(const int32_t *__restrict__ packed_all, int n_shards, int Q, const int32_t *__restrict__ frame_offsets,
                                       const float *__restrict__ q_xy, const float *__restrict__ depth, const float *__restrict__ fill, int width,
                                       int height, const int32_t *__restrict__ model_of_row, int64_t table_base, int64_t table_rows,
                                       const mc_adaptive_model *__restrict__ curves, int n_models, AdaptiveParams P, int32_t *__restrict__ nn_row,
                                       float *__restrict__ nn_dist, uint8_t *__restrict__ accepted, int32_t *__restrict__ bad) {
	const int f = blockIdx.y;
	const int i = frame_offsets[f] + blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= frame_offsets[f + 1]) return;
	Top2 t = top2_empty();
	bool outside = false;
	for (int s = 0; s < n_shards; s++) {
		const int32_t *rows = packed_all + (size_t)s * 4 * Q + 2 * (size_t)i;
		const float *dist = (const float *)(rows + 2 * (size_t)Q);
		for (int k = 0; k < 2; k++) {
			outside |= rows[k] != -1 && (uint64_t)(rows[k] - table_base) >= (uint64_t)table_rows;
			top2_push(t, dist[k], rows[k]);
		}
	}
	nn_row[2 * i] = t.i0; nn_row[2 * i + 1] = t.i1;
	nn_dist[2 * i] = t.d0; nn_dist[2 * i + 1] = t.d1;
	bool ok = false;
	if (outside) bad[f] = 1;
	else if (t.i0 >= 0 && t.i1 >= 0) {
		const int px = adaptive_pixel(q_xy[2 * i], q_xy[2 * i + 1], width, height);
		const int m = model_of_row[t.i0 - table_base];
		const size_t plane = (size_t)f * width * height;
		if (m >= 0 && m < n_models) ok = adaptive_accept(curves[m], depth[plane + px], fill[plane + px], t.d0, t.d1, P);
	}
	accepted[i] = ok ? 1 : 0;
}

// ---- ratio curve of one model (host, once per model change) ---------------------------------------------------------------------
// The reference asks: at which depth does the largest face of the model's bounding box, centred on the optical axis and parallel
// to the image plane, project to a square of `target` pixels a side? It answers by doubling an upper bound from 2 m and bisecting
// (at most 100 evaluations in total, stop within 1 %). The projected side is evaluated like the reference does — pinhole
// projection of the face's corners, extent of the projections, square root of the area — but only for the two distinct values each
// image coordinate takes (the four corners share them pairwise), which yields the same floats.
namespace {

struct Face { float half_a, half_b; };      // half extents of the largest face, a along image x, b along image y

Face largest_face(const float *lo, const float *hi) {
	const float ex = hi[0] - lo[0], ey = hi[1] - lo[1], ez = hi[2] - lo[2];
	// centred coordinates: +-e/2; the face areas are products of full extents rebuilt from the halves, as the reference forms them
	const float hx = ex / 2, hy = ey / 2, hz = ez / 2;
	const float fx = hx - (-hx), fy = hy - (-hy), fz = hz - (-hz);
	const float area_xy = fx * fy, area_xz = fx * fz, area_yz = fy * fz;
	Face f;
	if (area_xy >= area_yz && area_xy >= area_xz) { f.half_a = hx; f.half_b = hy; }
	else if (area_xz >= area_yz && area_xz >= area_xy) { f.half_a = hx; f.half_b = hz; }
	else { f.half_a = hy; f.half_b = hz; }
	return f;
}

float projected_side(const Face &f, const float *K, float z) {
	const float u_lo = (K[0] * -f.half_a + K[2] * z) / z, u_hi = (K[0] * f.half_a + K[2] * z) / z;
	const float v_lo = (K[1] * -f.half_b + K[3] * z) / z, v_hi = (K[1] * f.half_b + K[3] * z) / z;
	const float du = std::fmax(u_lo, u_hi) - std::fmin(u_lo, u_hi), dv = std::fmax(v_lo, v_hi) - std::fmin(v_lo, v_hi);
	return std::sqrt(du * dv);
}

float depth_for_side(const Face &f, const float *K, float target) {
	const int budget = 100;
	const float tolerance = 0.01;                     // a double literal narrowed to float, as the reference's parameter is
	int used = 0;
	float near = 0.f, far = 2.f;
	while (used < budget) {                           // push the far bound out until the face looks smaller than the target
		used++;
		if (projected_side(f, K, far) > target) far *= 2;
		else break;
	}
	const float slack = target * tolerance;
	while (used < budget) {
		used++;
		const float mid = (near + far) / 2;
		const float side = projected_side(f, K, mid);
		if (std::fabs(side - target) < slack) return mid;
		if (side > target) near = mid;
		else far = mid;
	}
	return (near + far) / 2;
}

} // namespace

// ---- frame batches (mc_match_adaptive_frames / _dev / _merged_dev, and MATCH of mc_process_depth_queries*) ------------------------
// Frames [frame_begin, frame_end) of the batch are processed (the cascade always takes the whole batch). `dev`: queries, planes and
// the per-match / per-feature outputs are device pointers; otherwise host arrays, staged through the context's buffers. The planes
// start with frame frame_begin; per-feature and per-match arrays use global feature ids; match_offsets and frame_info have one row per
// frame of the range. frame_offsets, match_offsets and frame_info are host arrays either way. One synchronisation per call.
// q_world / q_fill (device, `dev` only, nullable): DEPTHPROP's per-feature depth data, gathered into match_world / match_fill by the
// compaction. ev (nullable, 2 events): recorded on ctx->stream around the device work of MATCH (cascade or merge, finalize, compaction).
mc_status match_adaptive_frames(mc_ctx *ctx, bool dev, const char *who, const RowSource &src, const float *q_xy, const int32_t *q_image,
                                const int32_t *frame_offsets, int n_frames, int frame_begin, int frame_end, const float *depth,
                                const float *fill_distance, int width, int height, const mc_adaptive_model *models, int n_models,
                                float maximum_depth, float default_depth, float cauchy_scale, int32_t *match_offsets, int32_t *match_feature,
                                int32_t *match_image, float *match_xy, float *match_xyz, int32_t *nn_row, float *nn_dist, uint8_t *accepted,
                                int32_t *frame_info, const float *q_world, const float *q_fill, float *match_world, float *match_fill,
                                cudaEvent_t *ev) {
	if (!ctx) return MC_ERR_ARG;
	auto fail = [&](mc_status st, const std::string &what) { ctx->err = std::string(who) + ": " + what; return st; };
	const bool merge = src.n_shards > 0;
	if (!frame_offsets || n_frames < 1 || !depth || !fill_distance || !models || !match_offsets || width < 1 || height < 1 || n_models < 1)
		return fail(MC_ERR_ARG, "bad argument");
	if (n_frames > 65535) return fail(MC_ERR_ARG, "more than 65535 frames in one call");       // the finalize grid's y extent
	if (frame_begin < 0 || frame_begin > frame_end || frame_end > n_frames) return fail(MC_ERR_ARG, "frame range outside 0..n_frames");
	if (frame_offsets[0] != 0) return fail(MC_ERR_ARG, "frame_offsets[0] must be 0");
	int q_max = 0;
	for (int f = 0; f < n_frames; f++) {
		const int n = frame_offsets[f + 1] - frame_offsets[f];
		if (n < 0) return fail(MC_ERR_ARG, "frame_offsets do not ascend");
		if (f >= frame_begin && f < frame_end) q_max = n > q_max ? n : q_max;
	}
	const int Q = frame_offsets[n_frames], n_range = frame_end - frame_begin;
	const int32_t *range_offsets = frame_offsets + frame_begin;
	const bool any = range_offsets[n_range] > range_offsets[0];
	if (any && ((!merge && !src.q_desc) || !q_xy || !match_feature || !match_image || !match_xy || !match_xyz)) return fail(MC_ERR_ARG, "bad argument");
	if (merge) {
		if (!ctx->d_model_of_row) return fail(MC_ERR_STATE, "no database tables (mc_db_upload, and mc_db_set_global_tables on a shard)");
	} else {
		if (!ctx->d_db) return fail(MC_ERR_STATE, "no database uploaded");
		if (ctx->row_base != 0 || ctx->table_base != 0 || ctx->table_rows != ctx->n_rows)
			return fail(MC_ERR_STATE, "object-sharded database (rows from a base other than 0, or global tables) is not supported");
	}
	if (n_models < ctx->n_models) return fail(MC_ERR_ARG, "fewer ratio curves than models in the database");
	const int stride = n_models + 1;
	if (!any) {                                        // nothing to match: every frame of the range empty
		for (int f = 0; f < n_range; f++) {
			for (int m = 0; m < stride; m++) match_offsets[(size_t)f * stride + m] = range_offsets[f];
			if (frame_info) frame_info[3 * f] = frame_info[3 * f + 1] = frame_info[3 * f + 2] = 0;
		}
		return MC_OK;
	}
	MC_CUDA(cudaSetDevice(ctx->device));
	const size_t planes = (size_t)width * height * n_range, q = (size_t)Q, nr = (size_t)n_range;
	mc_adaptive_model *d_curves; FrameDesc *d_fd;
	int32_t *d_fo, *d_moff, *d_status, *d_nobj, *d_acc_list, *d_mrow, *up_feat = nullptr, *up_mimg = nullptr;
	float *up_depth = nullptr, *up_fill = nullptr, *up_mxy = nullptr, *up_mxyz = nullptr;
	MC_TRY(carve_scratch(ctx, ctx->scratch[kScrAdaptive], [&](Carve &c) {
		if (!dev) { c.take(up_depth, planes); c.take(up_fill, planes); }
		c.take(d_curves, n_models); c.take(d_fo, nr + 1); c.take(d_fd, nr); c.take(d_moff, (size_t)stride * nr);
		// the compaction's overflow flags, then (merge) the flags of frames with a row outside the tables: one copy to the host
		c.take(d_status, 2 * nr); c.take(d_nobj, nr);
		c.take(d_acc_list, q); c.take(d_mrow, q);
		if (!dev) { c.take(up_feat, q); c.take(up_mimg, q); c.take(up_mxy, 2 * q); c.take(up_mxyz, 3 * q); }
	}));
	const float *d_q = src.q_desc, *d_xy = q_xy, *d_depth = depth, *d_fill = fill_distance;
	const int32_t *d_img = q_image;
	int32_t *d_feat = match_feature, *d_mimg = match_image;
	float *d_mxy = match_xy, *d_mxyz = match_xyz;
	if (!dev) {
		MC_TRY(reserve(ctx, ctx->q_desc, sizeof(float) * (size_t)Q * ctx->D));
		MC_TRY(reserve(ctx, ctx->q_xy, sizeof(float) * 2 * (size_t)Q));
		MC_CUDA(cudaMemcpyAsync(ctx->q_desc.p, src.q_desc, sizeof(float) * (size_t)Q * ctx->D, cudaMemcpyHostToDevice, ctx->stream));
		MC_CUDA(cudaMemcpyAsync(ctx->q_xy.p, q_xy, sizeof(float) * 2 * (size_t)Q, cudaMemcpyHostToDevice, ctx->stream));
		if (q_image) {
			MC_TRY(reserve(ctx, ctx->q_image, sizeof(int32_t) * (size_t)Q));
			MC_CUDA(cudaMemcpyAsync(ctx->q_image.p, q_image, sizeof(int32_t) * (size_t)Q, cudaMemcpyHostToDevice, ctx->stream));
			d_img = (const int32_t *)ctx->q_image.p;
		}
		MC_CUDA(cudaMemcpyAsync(up_depth, depth, sizeof(float) * planes, cudaMemcpyHostToDevice, ctx->stream));
		MC_CUDA(cudaMemcpyAsync(up_fill, fill_distance, sizeof(float) * planes, cudaMemcpyHostToDevice, ctx->stream));
		d_q = (const float *)ctx->q_desc.p; d_xy = (const float *)ctx->q_xy.p;
		d_depth = up_depth; d_fill = up_fill;
		d_feat = up_feat; d_mimg = up_mimg; d_mxy = up_mxy; d_mxyz = up_mxyz;
	}
	// per-feature results: the caller's device arrays when given, the context's otherwise
	int32_t *d_nn_row = dev ? nn_row : nullptr;
	float *d_nn_dist = dev ? nn_dist : nullptr;
	uint8_t *d_acc = dev ? accepted : nullptr;
	if (!d_nn_row) { MC_TRY(reserve(ctx, ctx->nn_row, sizeof(int32_t) * 2 * (size_t)Q)); d_nn_row = (int32_t *)ctx->nn_row.p; }
	if (!d_nn_dist) { MC_TRY(reserve(ctx, ctx->nn_dist, sizeof(float) * 2 * (size_t)Q)); d_nn_dist = (float *)ctx->nn_dist.p; }
	if (!d_acc) { MC_TRY(reserve(ctx, ctx->accepted, (size_t)Q)); d_acc = (uint8_t *)ctx->accepted.p; }
	std::vector<FrameDesc> descs((size_t)n_range);
	for (int f = 0; f < n_range; f++) {
		FrameDesc &d = descs[(size_t)f];
		memset(&d, 0, sizeof d);
		const int q0 = range_offsets[f];
		d.nn_row = d_nn_row + 2 * (size_t)q0; d.accepted = d_acc + q0; d.q_xy = d_xy + 2 * (size_t)q0; d.q_image = d_img ? d_img + q0 : nullptr;
		d.Q = range_offsets[f + 1] - q0;
	}
	MC_CUDA(cudaMemcpyAsync(d_curves, models, sizeof(mc_adaptive_model) * (size_t)n_models, cudaMemcpyHostToDevice, ctx->stream));
	MC_CUDA(cudaMemcpyAsync(d_fo, range_offsets, sizeof(int32_t) * (n_range + 1ull), cudaMemcpyHostToDevice, ctx->stream));
	MC_CUDA(cudaMemcpyAsync(d_fd, descs.data(), sizeof(FrameDesc) * (size_t)n_range, cudaMemcpyHostToDevice, ctx->stream));
	AdaptiveParams P;
	P.maximum_depth = maximum_depth; P.default_depth = default_depth; P.cauchy_scale = cauchy_scale;
	const dim3 grid((unsigned)((q_max + 255) / 256), (unsigned)n_range);
	int32_t *d_bad = d_status + n_range;
	if (ev) MC_CUDA(cudaEventRecord(ev[0], ctx->stream));
	if (merge) {
		MC_CUDA(cudaMemsetAsync(d_bad, 0, sizeof(int32_t) * (size_t)n_range, ctx->stream));
		k_match_merge_adaptive<<<grid, 256, 0, ctx->stream>>>(src.packed_all, src.n_shards, Q, d_fo, d_xy, d_depth, d_fill, width, height,
		                                                    ctx->d_model_of_row, ctx->table_base, ctx->table_rows, d_curves, n_models, P, d_nn_row,
		                                                    d_nn_dist, d_acc, d_bad);
	} else {
		// one cascade pass over all queries (its fixed-ratio flags are overwritten by the adaptive kernel)
		MC_TRY(match_device(ctx, d_q, Q, 1.0f, MC_MATCH_TENSOR, d_nn_row, d_nn_dist, d_acc));
		k_match_finalize_adaptive<<<grid, 256, 0, ctx->stream>>>(d_nn_row, d_nn_dist, Q, d_fo, d_xy, d_depth, d_fill, width, height, ctx->d_model_of_row,
		                                                       ctx->table_base, d_curves, n_models, P, d_acc);
	}
	MC_LAUNCH_CHECK();
	MC_TRY(match_compact_frames_device(ctx, d_fd, d_fo, n_range, n_models, d_acc_list, d_moff, d_feat, d_mrow, d_mimg, d_mxy, d_mxyz, d_status, d_nobj,
	                                   q_world, q_fill, match_world, match_fill));
	if (ev) MC_CUDA(cudaEventRecord(ev[1], ctx->stream));
	// frame-local offsets and frame flags -> host; the host entry also takes the per-match and per-feature arrays
	const size_t h_moff_bytes = sizeof(int32_t) * (size_t)stride * n_range, h_flag_bytes = sizeof(int32_t) * (merge ? 2 : 1) * (size_t)n_range;
	MC_TRY(pinned(ctx, h_moff_bytes + h_flag_bytes));
	int32_t *h_moff = (int32_t *)ctx->h_pinned, *h_status = h_moff + (size_t)stride * n_range, *h_bad = h_status + n_range;
	MC_CUDA(cudaMemcpyAsync(h_moff, d_moff, h_moff_bytes, cudaMemcpyDeviceToHost, ctx->stream));
	MC_CUDA(cudaMemcpyAsync(h_status, d_status, h_flag_bytes, cudaMemcpyDeviceToHost, ctx->stream));
	if (!dev) {
		MC_CUDA(cudaMemcpyAsync(match_feature, d_feat, sizeof(int32_t) * (size_t)Q, cudaMemcpyDeviceToHost, ctx->stream));
		MC_CUDA(cudaMemcpyAsync(match_image, d_mimg, sizeof(int32_t) * (size_t)Q, cudaMemcpyDeviceToHost, ctx->stream));
		MC_CUDA(cudaMemcpyAsync(match_xy, d_mxy, sizeof(float) * 2 * (size_t)Q, cudaMemcpyDeviceToHost, ctx->stream));
		MC_CUDA(cudaMemcpyAsync(match_xyz, d_mxyz, sizeof(float) * 3 * (size_t)Q, cudaMemcpyDeviceToHost, ctx->stream));
		if (nn_row) MC_CUDA(cudaMemcpyAsync(nn_row, d_nn_row, sizeof(int32_t) * 2 * (size_t)Q, cudaMemcpyDeviceToHost, ctx->stream));
		if (nn_dist) MC_CUDA(cudaMemcpyAsync(nn_dist, d_nn_dist, sizeof(float) * 2 * (size_t)Q, cudaMemcpyDeviceToHost, ctx->stream));
		if (accepted) MC_CUDA(cudaMemcpyAsync(accepted, d_acc, (size_t)Q, cudaMemcpyDeviceToHost, ctx->stream));
	}
	MC_CUDA(cudaStreamSynchronize(ctx->stream));
	// local offsets -> global; a frame over the compaction's cap (status 1: its per-feature results are complete) or with a row outside
	// the tables (status 2: that feature is rejected) keeps an empty row
	mc_status st = MC_OK;
	int first_over = -1, first_bad = -1;
	for (int f = 0; f < n_range; f++) {
		const int base = range_offsets[f];
		const int status = merge && h_bad[f] ? 2 : h_status[f] != 0 ? 1 : 0;
		const int32_t *loc = h_moff + (size_t)f * stride;
		int32_t *row = match_offsets + (size_t)f * stride;
		for (int m = 0; m < stride; m++) row[m] = base + (status ? 0 : loc[m]);
		if (frame_info) {
			frame_info[3 * f] = range_offsets[f + 1] - base; frame_info[3 * f + 1] = status ? 0 : loc[n_models]; frame_info[3 * f + 2] = status;
		}
		if (status == 1 && first_over < 0) first_over = frame_begin + f;
		if (status == 2 && first_bad < 0) first_bad = frame_begin + f;
	}
	if (first_bad >= 0) st = fail(MC_ERR_ARG, "frame " + std::to_string(first_bad) + " has a nearest row outside the database tables");
	else if (first_over >= 0)
		st = fail(MC_ERR_CAPACITY, "frame " + std::to_string(first_over) + " has more than " + std::to_string(kCompactCap) + " accepted matches");
	return st;
}

} // namespace mc

using namespace mc;

extern "C" {

void mc_adaptive_model_init(mc_adaptive_model *out, const float *bbox_min, const float *bbox_max, const float *K, int n_features,
                            float min_ratio_min, float min_ratio_max, float max_ratio_min, float max_ratio_max, float dimension_peak,
                            float dimension_fade) {
	if (!out || !bbox_min || !bbox_max || !K) return;
	const Face f = largest_face(bbox_min, bbox_max);
	out->depth_peak = depth_for_side(f, K, dimension_peak);
	out->depth_fade = depth_for_side(f, K, dimension_fade);
	// sparse models (few features) get the permissive ends of both ratio ranges, dense ones the strict ends: a logistic in the
	// feature count centred on 1750 features with scale 250 (MATCH_ADAPTIVE_FLANN_CPU.hpp:103-104,160-166), evaluated in double
	const float centre = 1750, scale = 250;
	const float count = (float)n_features;
	const float x = (centre - count) / scale;
	const float density = (float)(1.0 / (1.0 + std::exp(-1.0 * (double)x)));
	out->ratio_low = min_ratio_min + density * (min_ratio_max - min_ratio_min);
	out->ratio_high = max_ratio_min + density * (max_ratio_max - max_ratio_min);
}

mc_status mc_match_adaptive(mc_ctx *ctx, const float *q_desc, const float *q_xy, int Q, const float *depth, const float *fill_distance, int width,
                            int height, const mc_adaptive_model *models, int n_models, float maximum_depth, float default_depth, float cauchy_scale,
                            int32_t *nn_row, float *nn_dist, uint8_t *accepted) {
	if (!ctx || !q_desc || !q_xy || !depth || !fill_distance || !models || !nn_row || !nn_dist || !accepted || Q < 0 || width < 1 || height < 1 ||
	    n_models < 1) {
		if (ctx) ctx->err = "mc_match_adaptive: bad argument";
		return MC_ERR_ARG;
	}
	if (!ctx->d_db) { ctx->err = "mc_match_adaptive: no database uploaded"; return MC_ERR_STATE; }
	if (n_models < ctx->n_models) { ctx->err = "mc_match_adaptive: fewer ratio curves than models in the database"; return MC_ERR_ARG; }
	if (Q == 0) return MC_OK;
	MC_CUDA(cudaSetDevice(ctx->device));
	const size_t px = (size_t)width * height;
	MC_TRY(reserve(ctx, ctx->q_desc, sizeof(float) * (size_t)Q * ctx->D));
	MC_TRY(reserve(ctx, ctx->nn_row, sizeof(int32_t) * 2 * (size_t)Q));
	MC_TRY(reserve(ctx, ctx->nn_dist, sizeof(float) * 2 * (size_t)Q));
	MC_TRY(reserve(ctx, ctx->accepted, (size_t)Q));
	MC_TRY(reserve(ctx, ctx->q_xy, sizeof(float) * 2 * (size_t)Q));
	float *d_depth, *d_fill; mc_adaptive_model *d_curves;
	MC_TRY(carve_scratch(ctx, ctx->scratch[kScrAdaptive], [&](Carve &c) { c.take(d_depth, px); c.take(d_fill, px); c.take(d_curves, n_models); }));
	MC_CUDA(cudaMemcpyAsync(ctx->q_desc.p, q_desc, sizeof(float) * (size_t)Q * ctx->D, cudaMemcpyHostToDevice, ctx->stream));
	MC_CUDA(cudaMemcpyAsync(ctx->q_xy.p, q_xy, sizeof(float) * 2 * (size_t)Q, cudaMemcpyHostToDevice, ctx->stream));
	MC_CUDA(cudaMemcpyAsync(d_depth, depth, sizeof(float) * px, cudaMemcpyHostToDevice, ctx->stream));
	MC_CUDA(cudaMemcpyAsync(d_fill, fill_distance, sizeof(float) * px, cudaMemcpyHostToDevice, ctx->stream));
	MC_CUDA(cudaMemcpyAsync(d_curves, models, sizeof(mc_adaptive_model) * (size_t)n_models, cudaMemcpyHostToDevice, ctx->stream));
	// the fixed-ratio flags of the plain matcher are overwritten by the adaptive kernel
	MC_TRY(match_device(ctx, (const float *)ctx->q_desc.p, Q, 1.0f, MC_MATCH_TENSOR, (int32_t *)ctx->nn_row.p, (float *)ctx->nn_dist.p, (uint8_t *)ctx->accepted.p));
	AdaptiveParams P;
	P.maximum_depth = maximum_depth; P.default_depth = default_depth; P.cauchy_scale = cauchy_scale;
	k_match_finalize_adaptive<<<(Q + 255) / 256, 256, 0, ctx->stream>>>((const int32_t *)ctx->nn_row.p, (const float *)ctx->nn_dist.p, Q, nullptr, (const float *)ctx->q_xy.p,
	                                                                  d_depth, d_fill, width, height, ctx->d_model_of_row, ctx->table_base, d_curves, n_models, P,
	                                                                  (uint8_t *)ctx->accepted.p);
	MC_LAUNCH_CHECK();
	MC_CUDA(cudaMemcpyAsync(nn_row, ctx->nn_row.p, sizeof(int32_t) * 2 * (size_t)Q, cudaMemcpyDeviceToHost, ctx->stream));
	MC_CUDA(cudaMemcpyAsync(nn_dist, ctx->nn_dist.p, sizeof(float) * 2 * (size_t)Q, cudaMemcpyDeviceToHost, ctx->stream));
	MC_CUDA(cudaMemcpyAsync(accepted, ctx->accepted.p, (size_t)Q, cudaMemcpyDeviceToHost, ctx->stream));
	MC_CUDA(cudaStreamSynchronize(ctx->stream));
	return MC_OK;
}

mc_status mc_match_adaptive_frames(mc_ctx *ctx, const float *q_desc, const float *q_xy, const int32_t *q_image, const int32_t *frame_offsets, int n_frames,
                                   const float *depth, const float *fill_distance, int width, int height, const mc_adaptive_model *models, int n_models,
                                   float maximum_depth, float default_depth, float cauchy_scale, int32_t *match_offsets, int32_t *match_feature,
                                   int32_t *match_image, float *match_xy, float *match_xyz, int32_t *nn_row, float *nn_dist, uint8_t *accepted,
                                   int32_t *frame_info) {
	const RowSource src = {q_desc, nullptr, 0};
	return match_adaptive_frames(ctx, false, "mc_match_adaptive_frames", src, q_xy, q_image, frame_offsets, n_frames, 0, n_frames, depth, fill_distance,
	                             width, height, models, n_models, maximum_depth, default_depth, cauchy_scale, match_offsets, match_feature, match_image, match_xy,
	                             match_xyz, nn_row, nn_dist, accepted, frame_info, nullptr, nullptr, nullptr, nullptr, nullptr);
}

mc_status mc_match_adaptive_frames_dev(mc_ctx *ctx, const float *q_desc_dev, const float *q_xy_dev, const int32_t *q_image_dev, const int32_t *frame_offsets,
                                       int n_frames, const float *depth_dev, const float *fill_distance_dev, int width, int height,
                                       const mc_adaptive_model *models, int n_models, float maximum_depth, float default_depth, float cauchy_scale,
                                       int32_t *match_offsets, int32_t *match_feature_dev, int32_t *match_image_dev, float *match_xy_dev,
                                       float *match_xyz_dev, int32_t *nn_row_dev, float *nn_dist_dev, uint8_t *accepted_dev, int32_t *frame_info) {
	const RowSource src = {q_desc_dev, nullptr, 0};
	return match_adaptive_frames(ctx, true, "mc_match_adaptive_frames_dev", src, q_xy_dev, q_image_dev, frame_offsets, n_frames, 0, n_frames, depth_dev,
	                             fill_distance_dev, width, height, models, n_models, maximum_depth, default_depth, cauchy_scale, match_offsets,
	                             match_feature_dev, match_image_dev, match_xy_dev, match_xyz_dev, nn_row_dev, nn_dist_dev, accepted_dev, frame_info, nullptr,
	                             nullptr, nullptr, nullptr, nullptr);
}

mc_status mc_match_adaptive_frames_merged_dev(mc_ctx *ctx, const void *packed_all_dev, int n_shards, const float *q_xy_dev, const int32_t *q_image_dev,
                                              const int32_t *frame_offsets, int n_frames, int frame_begin, int frame_end, const float *depth_dev,
                                              const float *fill_distance_dev, int width, int height, const mc_adaptive_model *models, int n_models,
                                              float maximum_depth, float default_depth, float cauchy_scale, int32_t *match_offsets,
                                              int32_t *match_feature_dev, int32_t *match_image_dev, float *match_xy_dev, float *match_xyz_dev,
                                              int32_t *nn_row_dev, float *nn_dist_dev, uint8_t *accepted_dev, int32_t *frame_info) {
	if (ctx && (!packed_all_dev || n_shards < 1)) { ctx->err = "mc_match_adaptive_frames_merged_dev: bad argument"; return MC_ERR_ARG; }
	const RowSource src = {nullptr, (const int32_t *)packed_all_dev, n_shards};
	return match_adaptive_frames(ctx, true, "mc_match_adaptive_frames_merged_dev", src, q_xy_dev, q_image_dev, frame_offsets, n_frames, frame_begin,
	                             frame_end, depth_dev, fill_distance_dev, width, height, models, n_models, maximum_depth, default_depth, cauchy_scale,
	                             match_offsets, match_feature_dev, match_image_dev, match_xy_dev, match_xyz_dev, nn_row_dev, nn_dist_dev, accepted_dev,
	                             frame_info, nullptr, nullptr, nullptr, nullptr, nullptr);
}

} // extern "C"
