// cluster.cu — CLUSTER step: canopy mean-shift over matched image coordinates, per (model, image).
//
// Replaces CLUSTER_MEAN_SHIFT_CPU::process / MeanShift
// (moped2/libmoped/src/cluster/CLUSTER_MEAN_SHIFT_CPU.hpp:80-158,182-199).
// The reference algorithm is order-dependent (canopies are merged by pointer chasing in list order), so
// the kernel keeps the list order and the floating-point summation order of the reference:
//   (i)   aggregate of every live canopy: all threads, each walking the live list in order (O(n^2/threads));
//   (ii)  merge redirection in list order: the "aggregates closer than Merge" predicate of every (canopy, earlier canopy)
//         pair does not depend on the redirections, so all warps evaluate it 64 list rows at a time into a bit matrix
//         in shared memory (one ballot = one word) and one thread then applies the set bits in ascending (row, column)
//         order — the order of the reference's double loop;
//   (iii) folding of redirected canopies into their targets in list order: one thread (O(n)).
// One CTA per model, images in sequence; working set staged in shared memory (<= kCap points per group,
// larger groups use the same code on a global-memory scratch area).
#include "common.cuh"

namespace mc {

constexpr int kClusterThreads = 256;
constexpr int kCap = 1024;       // points per (model, image) group held in shared memory
constexpr int kBitRows = 64;     // list rows of the merge predicate evaluated per round
constexpr int kBitWords = kCap / 32;
constexpr size_t kClusterSmem = sizeof(float) * 4 * kCap + sizeof(int) * 7 * kCap + sizeof(unsigned) * kBitRows * kBitWords;

struct MsArrays {
	float *cx, *cy, *ax, *ay;
	int *size, *target, *alive, *head, *tail, *next;
};

__device__ void meanshift_group(const MsArrays &A, int n, float sq_radius, float sq_merge, int min_pts, int max_iter,
                                const int *pid, int *out_count, int *out_sizes, int *out_members, int &n_clusters, int &n_members,
                                int *sh_n_alive, int *sh_done, unsigned *bits) {
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, n_warps = blockDim.x >> 5;
	for (int i = tid; i < n; i += blockDim.x) {
		A.size[i] = 1; A.target[i] = i; A.alive[i] = i; A.head[i] = i; A.tail[i] = i; A.next[i] = -1;
	}
	if (tid == 0) { *sh_n_alive = n; *sh_done = 0; }
	__syncthreads();
	for (int it = 0; it < max_iter; it++) {
		const int n_alive = *sh_n_alive;
		if (*sh_done) break;
		__syncthreads();
		// (i) size-weighted mean of the live centres within Radius, summed in list order (:102-120)
		for (int a = tid; a < n_alive; a += blockDim.x) {
			const int c = A.alive[a];
			const float ccx = A.cx[c], ccy = A.cy[c];
			float sx = __fmul_rn(ccx, (float)A.size[c]), sy = __fmul_rn(ccy, (float)A.size[c]);
			int touch = A.size[c];
			for (int b = 0; b < n_alive; b++) {
				const int o = A.alive[b];
				if (o == c) continue;
				const float ox = A.cx[o], oy = A.cy[o];
				const float dx = __fsub_rn(ox, ccx), dy = __fsub_rn(oy, ccy);
				const float dist = __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
				if (dist < sq_radius) {
					const float s = (float)A.size[o];
					touch += A.size[o];
					sx = __fadd_rn(sx, __fmul_rn(ox, s));
					sy = __fadd_rn(sy, __fmul_rn(oy, s));
				}
			}
			A.ax[c] = __fdiv_rn(sx, (float)touch);
			A.ay[c] = __fdiv_rn(sy, (float)touch);
		}
		__syncthreads();
		// (ii) redirections, in list order (:122-132)
		if (n_alive <= kCap) {
			for (int a0 = 1; a0 < n_alive; a0 += kBitRows) {
				const int a1 = a0 + kBitRows < n_alive ? a0 + kBitRows : n_alive;
				for (int a = a0 + warp; a < a1; a += n_warps) {           // predicate bits of rows [a0, a1): one warp per row
					const int c = A.alive[a];
					const float acx = A.ax[c], acy = A.ay[c];
					const int nw = (a + 31) >> 5;
					for (int w = 0; w < nw; w++) {
						const int b = (w << 5) + lane;
						bool close = false;
						if (b < a) {
							const int o = A.alive[b];
							const float dx = __fsub_rn(A.ax[o], acx), dy = __fsub_rn(A.ay[o], acy);
							close = __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)) < sq_merge;
						}
						const unsigned m = __ballot_sync(0xffffffffu, close);
						if (lane == 0) bits[(a - a0) * kBitWords + w] = m;
					}
				}
				__syncthreads();
				if (tid == 0) {                                           // apply in ascending (row, column) order
					for (int a = a0; a < a1; a++) {
						const int c = A.alive[a];
						const int nw = (a + 31) >> 5;
						for (int w = 0; w < nw; w++) {
							unsigned m = bits[(a - a0) * kBitWords + w];
							while (m) {
								const int o = A.alive[(w << 5) + __ffs(m) - 1];
								m &= m - 1;
								A.target[A.target[o]] = c;
								A.target[o] = c;
							}
						}
					}
				}
				__syncthreads();
			}
		} else if (tid < 32) {                                            // groups beyond the shared-memory capacity: one warp, 32 at a time
			for (int a = 1; a < n_alive; a++) {
				const int c = A.alive[a];
				const float acx = A.ax[c], acy = A.ay[c];
				for (int b0 = 0; b0 < a; b0 += 32) {
					const int b = b0 + lane;
					bool close = false;
					if (b < a) {
						const int o = A.alive[b];
						const float dx = __fsub_rn(A.ax[o], acx), dy = __fsub_rn(A.ay[o], acy);
						close = __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)) < sq_merge;
					}
					unsigned m = __ballot_sync(0xffffffffu, close);
					if (lane == 0) {
						while (m) {
							const int o = A.alive[b0 + __ffs(m) - 1];
							m &= m - 1;
							A.target[A.target[o]] = c;
							A.target[o] = c;
						}
					}
					__syncwarp();
				}
			}
		}
		__syncthreads();
		// (iii) fold redirected canopies into their targets, in list order (:134-148); one thread
		if (tid == 0) {
			int w = 0, done = 1;
			for (int a = 0; a < n_alive; a++) {
				const int c = A.alive[a];
				const int t = A.target[c];
				if (t != c) {
					const float st = (float)A.size[t], sc = (float)A.size[c];
					float nx = __fadd_rn(__fmul_rn(A.cx[t], st), __fmul_rn(A.cx[c], sc));
					float ny = __fadd_rn(__fmul_rn(A.cy[t], st), __fmul_rn(A.cy[c], sc));
					A.next[A.tail[t]] = A.head[c];
					A.tail[t] = A.tail[c];
					A.size[t] += A.size[c];
					const float ns = (float)A.size[t];
					A.cx[t] = __fdiv_rn(nx, ns);
					A.cy[t] = __fdiv_rn(ny, ns);
					done = 0;
				} else A.alive[w++] = c;
			}
			*sh_n_alive = w;
			*sh_done = done;
		}
		__syncthreads();
	}
	__syncthreads();
	// emit canopies with >= MinPts points in surviving order, members in splice order (:151-157)
	if (tid == 0) {
		const int n_alive = *sh_n_alive;
		for (int a = 0; a < n_alive; a++) {
			const int c = A.alive[a];
			if (A.size[c] < min_pts) continue;
			out_sizes[n_clusters++] = A.size[c];
			for (int p = A.head[c]; p >= 0; p = A.next[p]) out_members[n_members++] = pid[p];
		}
		*out_count = n_clusters;
	}
	__syncthreads();
}

// The models that can have a cluster at all (>= min_pts matches), and model_count = 0 for everybody. One CTA. A frame matches a
// handful of the database's models: k_meanshift then starts a CTA per listed model instead of one per model — 1000 CTAs of 70 KB of
// shared memory each, all but ~8 of which only found out that they had nothing to do (and, 64 frames at a time, kept each other's
// working CTAs waiting for shared memory).
__global__ void k_cluster_nonempty(const int32_t *__restrict__ match_offsets, int n_models, int min_pts, int32_t *__restrict__ model_count,
                                   int32_t *__restrict__ list, int32_t *__restrict__ n_list) {
	__shared__ int s_n;
	if (threadIdx.x == 0) s_n = 0;
	__syncthreads();
	for (int m = threadIdx.x; m < n_models; m += blockDim.x) {
		model_count[m] = 0;
		const int cnt = match_offsets[m + 1] - match_offsets[m];
		if (cnt >= min_pts && cnt > 0) list[atomicAdd(&s_n, 1)] = m;        // any order: the models are independent
	}
	__syncthreads();
	if (threadIdx.x == 0) *n_list = s_n;
}

// One CTA per LISTED model (grid-stride if there are more than CTAs). Output per model m (region = the model's match range [lo, hi)):
//   model_count[m] = #clusters, sizes[lo + k] = size of its k-th cluster, members[lo ...] = concatenated members
__global__ void __launch_bounds__(kClusterThreads)
k_meanshift(const int32_t *__restrict__ match_offsets, const int32_t *__restrict__ match_image, const float *__restrict__ match_xy,
            int n_models, int n_images, float radius, float merge, int min_pts, int max_iter,
            const int32_t *__restrict__ list, const int32_t *__restrict__ n_list,
            int32_t *__restrict__ model_count, int32_t *__restrict__ sizes, int32_t *__restrict__ members,
            float *__restrict__ gscratch_f, int32_t *__restrict__ gscratch_i) {
	extern __shared__ __align__(16) unsigned char s_dyn[];
	float *s_f = reinterpret_cast<float *>(s_dyn);
	int *s_i = reinterpret_cast<int *>(s_f + 4 * kCap);
	unsigned *s_bits = reinterpret_cast<unsigned *>(s_i + 7 * kCap);
	__shared__ int sh_n, sh_n_alive, sh_done;
	const int tid = threadIdx.x;
	const int n_listed = *n_list;
	for (int li = blockIdx.x; li < n_listed; li += gridDim.x) {
	__syncthreads();
	const int m = list[li];
	const int lo = match_offsets[m], hi = match_offsets[m + 1], cnt = hi - lo;
	MsArrays A;
	int *pid;
	if (cnt <= kCap) {
		A.cx = s_f; A.cy = s_f + kCap; A.ax = s_f + 2 * kCap; A.ay = s_f + 3 * kCap;
		A.size = s_i; A.target = s_i + kCap; A.alive = s_i + 2 * kCap; A.head = s_i + 3 * kCap; A.tail = s_i + 4 * kCap; A.next = s_i + 5 * kCap;
		pid = s_i + 6 * kCap;
	} else {
		const int tot = match_offsets[n_models];
		A.cx = gscratch_f + lo; A.cy = gscratch_f + tot + lo; A.ax = gscratch_f + 2 * tot + lo; A.ay = gscratch_f + 3 * tot + lo;
		A.size = gscratch_i + lo; A.target = gscratch_i + tot + lo; A.alive = gscratch_i + 2 * tot + lo; A.head = gscratch_i + 3 * tot + lo;
		A.tail = gscratch_i + 4 * tot + lo; A.next = gscratch_i + 5 * tot + lo;
		pid = gscratch_i + 6 * tot + lo;
	}
	const float sq_radius = __fmul_rn(radius, radius), sq_merge = __fmul_rn(merge, merge);
	int n_clusters = 0, n_members = 0;
	for (int im = 0; im < n_images; im++) {
		// points of this image, in match order (:189-192)
		__syncthreads();
		if (tid < 32) {
			int k = 0;
			for (int j0 = lo; j0 < hi; j0 += 32) {
				const int j = j0 + tid;
				const bool sel = j < hi && match_image[j] == im;
				const unsigned msk = __ballot_sync(0xffffffffu, sel);
				if (sel) {
					const int pos = k + __popc(msk & ((1u << tid) - 1));
					A.cx[pos] = match_xy[2 * j]; A.cy[pos] = match_xy[2 * j + 1]; pid[pos] = j - lo;
				}
				k += __popc(msk);
			}
			if (tid == 0) sh_n = k;
		}
		__syncthreads();
		const int n = sh_n;
		if (n == 0) continue;
		meanshift_group(A, n, sq_radius, sq_merge, min_pts, max_iter, pid, &model_count[m], sizes + lo, members + lo, n_clusters, n_members,
		                &sh_n_alive, &sh_done, s_bits);
	}
	}
}

// Single-CTA compaction of the per-model outputs into the reference's cluster order:
// cluster_model[c], cluster_offsets[c+1], members. out_n = {#clusters, #members}.
__global__ void k_cluster_compact(const int32_t *__restrict__ match_offsets, int n_models, const int32_t *__restrict__ model_count,
                                  const int32_t *__restrict__ sizes, const int32_t *__restrict__ members_in,
                                  int32_t *__restrict__ out_n, int32_t *__restrict__ cluster_model, int32_t *__restrict__ cluster_offsets,
                                  int32_t *__restrict__ members_out) {
	__shared__ int s_c[1024], s_m[1024];
	__shared__ int base_c, base_m;
	const int tid = threadIdx.x;
	if (tid == 0) { base_c = 0; base_m = 0; }
	__syncthreads();
	for (int m0 = 0; m0 < n_models; m0 += blockDim.x) {
		const int m = m0 + tid;
		int nc = 0, nm = 0, lo = 0;
		if (m < n_models) {
			nc = model_count[m]; lo = match_offsets[m];
			for (int k = 0; k < nc; k++) nm += sizes[lo + k];
		}
		s_c[tid] = nc; s_m[tid] = nm;
		__syncthreads();
		// inclusive scan (Hillis-Steele)
		for (int o = 1; o < blockDim.x; o <<= 1) {
			int vc = tid >= o ? s_c[tid - o] : 0, vm = tid >= o ? s_m[tid - o] : 0;
			__syncthreads();
			s_c[tid] += vc; s_m[tid] += vm;
			__syncthreads();
		}
		int c0 = base_c + s_c[tid] - nc, t0 = base_m + s_m[tid] - nm;
		if (m < n_models) {
			int src = lo;
			for (int k = 0; k < nc; k++) {
				const int sz = sizes[lo + k];
				cluster_model[c0 + k] = m;
				cluster_offsets[c0 + k] = t0;
				for (int j = 0; j < sz; j++) members_out[t0 + j] = members_in[src + j];
				t0 += sz; src += sz;
			}
		}
		__syncthreads();
		if (tid == blockDim.x - 1) { base_c += s_c[tid]; base_m += s_m[tid]; }
		__syncthreads();
	}
	if (tid == 0) { cluster_offsets[base_c] = base_m; out_n[0] = base_c; out_n[1] = base_m; }
}

// per-device function attribute, set by mc_create for the context's device
mc_status cluster_configure_device(mc_ctx *ctx) {
	MC_CUDA(cudaFuncSetAttribute(k_meanshift, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kClusterSmem));
	return MC_OK;
}

// device entry: matches (CSR over models) -> clusters; all pointers device, async on ctx->stream
mc_status cluster_device(mc_ctx *ctx, const int32_t *d_match_offsets, const int32_t *d_match_image, const float *d_match_xy,
                         int n_models, int n_images, int max_matches, float radius, float merge, int min_pts, int max_iter,
                         int32_t *d_out_n, int32_t *d_cluster_model, int32_t *d_cluster_offsets, int32_t *d_members) {
	if (n_models <= 0) return MC_OK;
	DevBuf &b_count = ctx->scratch[kScrClusterCount], &b_sizes = ctx->scratch[kScrClusterSizes], &b_members = ctx->scratch[kScrClusterMembers],
	       &b_f = ctx->scratch[kScrClusterF], &b_i = ctx->scratch[kScrClusterI], &b_list = ctx->scratch[kScrClusterList];
	MC_TRY(reserve(ctx, b_count, sizeof(int32_t) * (n_models + 1)));
	MC_TRY(reserve(ctx, b_sizes, sizeof(int32_t) * (max_matches + 1)));
	MC_TRY(reserve(ctx, b_members, sizeof(int32_t) * (max_matches + 1)));
	MC_TRY(reserve(ctx, b_f, sizeof(float) * 4 * (size_t)(max_matches + 1)));
	MC_TRY(reserve(ctx, b_i, sizeof(int32_t) * 7 * (size_t)(max_matches + 1)));
	MC_TRY(reserve(ctx, b_list, sizeof(int32_t) * (size_t)(n_models + 16)));
	int32_t *d_list = (int32_t *)b_list.p + 16, *d_n_list = (int32_t *)b_list.p;
	k_cluster_nonempty<<<1, 1024, 0, ctx->stream>>>(d_match_offsets, n_models, min_pts, (int32_t *)b_count.p, d_list, d_n_list);
	MC_LAUNCH_CHECK();
	k_meanshift<<<n_models < 64 ? n_models : 64, kClusterThreads, kClusterSmem, ctx->stream>>>(d_match_offsets, d_match_image, d_match_xy, n_models, n_images,
	                                                         radius, merge, min_pts, max_iter, d_list, d_n_list,
	                                                         (int32_t *)b_count.p, (int32_t *)b_sizes.p, (int32_t *)b_members.p,
	                                                         (float *)b_f.p, (int32_t *)b_i.p);
	MC_LAUNCH_CHECK();
	k_cluster_compact<<<1, 1024, 0, ctx->stream>>>(d_match_offsets, n_models, (const int32_t *)b_count.p, (const int32_t *)b_sizes.p,
	                                              (const int32_t *)b_members.p, d_out_n, d_cluster_model, d_cluster_offsets, d_members);
	MC_LAUNCH_CHECK();
	return MC_OK;
}

} // namespace mc
