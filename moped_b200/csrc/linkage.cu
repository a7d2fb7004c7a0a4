// linkage.cu — moped3d's clustering stage on the device (SURVEY.md §8f row 4, first CUDA component of that row).
// Replaces CLUSTER_LINKAGE_CPU::process for the matches of one model (moped3d/libmoped/src/cluster/CLUSTER_LINKAGE_CPU.hpp:577-704):
// pairwise similarity matrices over the model's matches, then agglomerative clustering down to a similarity cutoff.
//
// Shape of the work (n = matches of one model, tens to a few hundred): the similarity matrix is n^2 independent entries, each a
// handful of expf/atan2f plus — for the depth-discontinuity kernel — a walk along the Bresenham path between two features in
// the depth map: one thread per pair. The agglomeration is a sequential chain of merges, each needing an argmax over the
// live pairs: one CTA, the argmax and the row update parallel over the CTA, the chain itself serial (latency-bound, like
// mean-shift in cluster.cu).
//
// mc_process_depth_frames* runs the same kernels over all models of a frame at once (a model dimension in every grid, one
// agglomeration CTA per model: the serial merge chains of different models run side by side); mc_cluster_linkage is the case of one model.
//
// Arithmetic: compiled with -fmad=false; every expression in the reference's order and types (the stage is built without
// -fsingle-precision-constant: literals are double where the reference's are). expf/atan2f/sqrtf: CUDA's vs glibc's differ by
// an ulp, so similarity values agree with the oracle to ~1e-6 and the agglomeration — which only compares them — is checked
// bit-exactly on the oracle's own matrix (mc_linkage_agglomerate) and as partitions end to end.
//
// Quirks of the reference that decide the output and are therefore kept (see oracle/moped_linkage_oracle.c): the merged-away
// index stays in the candidate list until the scan reaches it, and the scan skips the element that follows it; pairs are
// compared with strict >, so the FIRST maximum in (list position, list position) order wins; adaptiveWeightSum runs with
// alpha = 0.5, gamma = 25 whatever the constructor got.
#include "common.cuh"
#include "linkage_cached.cuh"

#include <float.h>
#include <math.h>

namespace mc {

constexpr int kLinkThreads = 256;

__device__ __forceinline__ float sq_dist2(const float *a, const float *b) {      // Pt<2>::sqEuclDist (moped.hpp:125)
	float d, r = 0;
	d = b[0] - a[0]; r += d * d;
	d = b[1] - a[1]; r += d * d;
	return r;
}
__device__ __forceinline__ float sq_dist3(const float *a, const float *b) {
	float d, r = 0;
	d = b[0] - a[0]; r += d * d;
	d = b[1] - a[1]; r += d * d;
	d = b[2] - a[2]; r += d * d;
	return r;
}

// Every kernel below works on the models of one frame at once (LinkSlice, common.cuh): model a of the launch owns matches
// lo .. lo+n of the frame's per-match arrays, n x n floats at element sq of each matrix arena, and n-element slices at lo of the
// per-match state (3n at 3 lo for the triples). Scalars: scal[4a .. 4a+3] = sigma2D, sigma3D, first and second maximum.
// mc_cluster_linkage runs them with one model at 0.

// getAverageNNDistances (:98-123): nearest-neighbour distance of every match in the image and in model space; the two averages
// are summed by one thread in match order (float sums are order-dependent). One CTA per model. With `status` given, a match
// outside the W x H maps sets it to 1 (the blend and agglomeration kernels then skip the frame).
__global__ void __launch_bounds__(kLinkThreads, 1) k_link_sigma(const LinkSlice *__restrict__ slices, const float *__restrict__ xy_all,
                                                            const float *__restrict__ xyz_all, float sigma2D, float sigma3D, float *__restrict__ tmp,
                                                            float *__restrict__ scal, int W, int H, int32_t *__restrict__ status) {
	const int n = slices[blockIdx.x].n, lo = slices[blockIdx.x].lo;
	const float *xy = xy_all + 2 * (size_t)lo, *xyz = xyz_all + 3 * (size_t)lo;
	float *nn_scratch = tmp + 3 * (size_t)lo, *sigmas = scal + 4 * (size_t)blockIdx.x;
	if (status) {
		int bad = 0;
		for (int i = threadIdx.x; i < n; i += blockDim.x) {
			const float x = xy[2 * i], y = xy[2 * i + 1];
			bad |= !(x >= 0.f && y >= 0.f && x < (float)W && y < (float)H);
		}
		if (__syncthreads_or(bad) && threadIdx.x == 0) atomicOr(status, 1);
	}
	if (sigma2D == -1 || sigma3D == -1) {
		for (int i = threadIdx.x; i < n; i += blockDim.x) {
			float b2 = (float)DBL_MAX, b3 = (float)DBL_MAX;
			for (int j = 0; j < n; j++) {
				if (i == j) continue;
				float d2 = sqrtf(sq_dist2(xy + 2 * j, xy + 2 * i)), d3 = sqrtf(sq_dist3(xyz + 3 * j, xyz + 3 * i));
				if (b2 > d2) b2 = d2;
				if (b3 > d3) b3 = d3;
			}
			nn_scratch[i] = b2; nn_scratch[n + i] = b3;
		}
		__syncthreads();
		if (threadIdx.x == 0) {
			float s2 = 0, s3 = 0;
			for (int i = 0; i < n; i++) { s2 += nn_scratch[i]; s3 += nn_scratch[n + i]; }
			float k2 = s2 / n, k3 = s3 / n;
			if (sigma2D != -1) k2 = sigma2D;
			if (sigma3D != -1) k3 = sigma3D;
			sigmas[0] = k2; sigmas[1] = k3;
		}
	} else if (threadIdx.x == 0) { sigmas[0] = sigma2D; sigmas[1] = sigma3D; }
}

__device__ __forceinline__ int sat(int v, int hi) { v = v < 0 ? 0 : v; return v >= hi ? hi - 1 : v; }

// getDiscontinuityMatrix entry (:233-285) with bresenhamIterate (:175-223) walked on the fly: the largest change of slope
// between the straight depth ramp from feature i to feature j and the ~20 sampled segments of the path between them
__device__ float discontinuity(const float *xy_i, const float *xy_j, int W, int H, const float *__restrict__ depth) {
	const int lix = sat((int)xy_i[0], W), liy = sat((int)xy_i[1], H), ljx = sat((int)xy_j[0], W), ljy = sat((int)xy_j[1], H);
	const float dStart = depth[(size_t)liy * W + lix], dEnd = depth[(size_t)ljy * W + ljx];
	const int xd = lix - ljx, yd = liy - ljy;
	const float planeDist = sqrtf((float)(xd * xd + yd * yd));
	const float direct = atan2f(dEnd - dStart, planeDist);
	int x0 = lix, y0 = liy, x1 = ljx, y1 = ljy, t;
	const bool steep = abs(y1 - y0) > abs(x1 - x0);
	if (steep) { t = x0; x0 = y0; y0 = t; t = x1; x1 = y1; y1 = t; }
	if (x0 > x1) { t = x0; x0 = x1; x1 = t; t = y0; y0 = y1; y1 = t; }
	const float deltaX = (float)x1 - x0, deltaY = fabsf((float)y1 - y0);
	const int yStep = (y0 < y1) ? 1 : -1;
	int perStep = (int)(x1 - x0) / 20;
	if (perStep < 1) perStep = 1;
	float error = 0.0f;
	const float deltaError = deltaY / deltaX;
	int y = y0;
	float maxDiff = -1;
	int px = 0, py = 0;
	bool have_prev = false;
	for (int x = x0; x <= x1;) {
		const int cx = steep ? y : x, cy = steep ? x : y;
		if (have_prev) {
			const float d1 = depth[(size_t)py * W + px], d2 = depth[(size_t)cy * W + cx];
			const float dx = px - cx, dy = py - cy;
			const float pixDist = sqrtf(dx * dx + dy * dy);
			const float pixAngle = atan2f(d2 - d1, pixDist);
			const float diff = fabsf(direct - pixAngle);
			if (diff > maxDiff) maxDiff = diff;
		}
		px = cx; py = cy; have_prev = true;
		x += perStep;
		if (x > x1) break;
		error += deltaError * perStep * yStep;
		float intPart;
		error = modff(error, &intPart);
		y += intPart;
	}
	const float div = (float)(-2 * (M_PI / 128) * (M_PI / 128));
	return expf(maxDiff * maxDiff / div);
}

// One thread per pair (i <= j): K2D, K3D + BK (getGaussK :133-150, getSum :295-301) and K3F (get3DFilterK :152-172)
// grid (columns / kLinkThreads, rows, models)
__global__ void __launch_bounds__(kLinkThreads) k_link_pairs(const LinkSlice *__restrict__ slices, int n_slices, const float *__restrict__ xy_all,
                                                            const float *__restrict__ xyz_all, const float *__restrict__ world_all, int W, int H,
                                                            const float *__restrict__ depth, const float *__restrict__ scal, int use3DFilter,
                                                            float *__restrict__ K2D_all, float *__restrict__ K3D_all, float *__restrict__ K3F_all) {
	for (int m = blockIdx.z; m < n_slices; m += gridDim.z) {
	const LinkSlice sl = slices[m];
	const int n = sl.n;
	const int j = blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y;
	if (j >= n || j < i) continue;
	const float *xy = xy_all + 2 * (size_t)sl.lo, *xyz = xyz_all + 3 * (size_t)sl.lo, *world = world_all + 3 * (size_t)sl.lo;
	float *K2D = K2D_all + sl.sq, *K3D = K3D_all + sl.sq, *K3F = K3F_all + sl.sq;
	const float s2 = scal[4 * (size_t)m], s3 = scal[4 * (size_t)m + 1];
	const float two2 = 2 * s2 * s2, two3 = 2 * s3 * s3;
	const float k2 = expf(-1 * sq_dist2(xy + 2 * i, xy + 2 * j) / two2);
	float k3 = expf(-1 * sq_dist3(world + 3 * i, world + 3 * j) / two3);
	k3 = k3 + discontinuity(xy + 2 * i, xy + 2 * j, W, H, depth);
	const size_t a = (size_t)j * n + i, b = (size_t)i * n + j;
	K2D[a] = k2; K2D[b] = k2;
	K3D[a] = k3; K3D[b] = k3;
	if (use3DFilter) {
		float f;
		if (i == j) f = (float)1.0;
		else {
			const float sigma = (float)0.1;
			const float two = 2 * sigma * sigma;
			const float dm = sqrtf(sq_dist3(xyz + 3 * j, xyz + 3 * i)), dw = sqrtf(sq_dist3(world + 3 * j, world + 3 * i));
			const float e = fabsf(dm - dw) / dm;
			f = expf((-1 * e * e) / two);
		}
		K3F[a] = f; K3F[b] = f;
	}
	}
}

// normalizeSimilarityMatrix (:303-322) in two kernels: the maximum (order-independent), then the division. `combine`: 0 = plain,
// 1 = K += F first, 2 = K *= F first (getSum / getProduct before the second normalisation, :636-642)
// grid (blocks per model, models); `slot` = 2 (first maximum) or 3 (second)
__global__ void __launch_bounds__(kLinkThreads) k_link_max(const LinkSlice *__restrict__ slices, float *__restrict__ K_all, const float *__restrict__ F_all,
                                                          int combine, float *__restrict__ scal, int slot) {
	__shared__ float s_m[kLinkThreads / 32];
	const LinkSlice sl = slices[blockIdx.y];
	const size_t nn = (size_t)sl.n * sl.n;
	float *K = K_all + sl.sq;
	const float *F = F_all + sl.sq;
	float *out_max = scal + 4 * (size_t)blockIdx.y + slot;
	float m = -1;
	for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < nn; k += (size_t)gridDim.x * blockDim.x) {
		float v = K[k];
		if (combine == 1) { v = v + F[k]; K[k] = v; }
		else if (combine == 2) { v = v * F[k]; K[k] = v; }
		if (v > m) m = v;
	}
#pragma unroll
	for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
	if ((threadIdx.x & 31) == 0) s_m[threadIdx.x >> 5] = m;
	__syncthreads();
	if (threadIdx.x == 0) {
		for (int w = 1; w < kLinkThreads / 32; w++) m = fmaxf(m, s_m[w]);
		// m is never NaN: `v > m` and fmaxf skip the NaN of duplicate matches (get3DFilterK's 0/0). It is -1 (a negative int, which
		// loses to the zeroed slot) or a sum / product of exponentials >= 0, whose int bit patterns order like the floats
		atomicMax((int *)out_max, __float_as_int(m));
	}
}
__global__ void __launch_bounds__(kLinkThreads) k_link_scale(const LinkSlice *__restrict__ slices, float *__restrict__ K_all, const float *__restrict__ scal,
                                                            int slot) {
	const LinkSlice sl = slices[blockIdx.y];
	const size_t nn = (size_t)sl.n * sl.n;
	float *K = K_all + sl.sq;
	const float m = scal[4 * (size_t)blockIdx.y + slot];
	for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < nn; k += (size_t)gridDim.x * blockDim.x) K[k] = K[k] / m;
}

// adaptiveWeightSum (:324-365) with alpha = 0.5, gamma = 25 (:651)
// grid as k_link_pairs. Reads the fill-distance map at every match's pixel unclamped, like the reference: a frame whose `status`
// was set by k_link_sigma is skipped
__global__ void __launch_bounds__(kLinkThreads) k_link_blend(const LinkSlice *__restrict__ slices, int n_slices, const float *__restrict__ xy_all, int W,
                                                            const float *__restrict__ distance, const float *__restrict__ K2D_all,
                                                            const float *__restrict__ K3D_all, float *__restrict__ K_all, const int32_t *__restrict__ status) {
	if (status && *status) return;
	for (int m = blockIdx.z; m < n_slices; m += gridDim.z) {
	const LinkSlice sl = slices[m];
	const int n = sl.n;
	const int j = blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y;
	if (j >= n || j < i) continue;
	const float *xy = xy_all + 2 * (size_t)sl.lo;
	const float *K2D = K2D_all + sl.sq, *K3D = K3D_all + sl.sq;
	float *K = K_all + sl.sq;
	const float alpha = (float)0.5, gamma = 25;
	const float gammaSq = gamma * gamma;
	const float di = distance[(size_t)((int)xy[2 * i + 1]) * W + (int)xy[2 * i]], dj = distance[(size_t)((int)xy[2 * j + 1]) * W + (int)xy[2 * j]];
	const float wi = (float)(1.0 / (1 + (di * di / gammaSq))), wj = (float)(1.0 / (1 + (dj * dj / gammaSq)));
	const float alphaBar = (float)(1.0 - alpha);
	const float k2 = K2D[(size_t)j * n + i], k3 = K3D[(size_t)j * n + i];
	const float joint = wi * wj;
	const float w2D = (float)(alpha + alphaBar * (1.0 - joint)), w3D = alphaBar * joint;
	const float val = w2D * k2 + w3D * k3;
	K[(size_t)j * n + i] = val; K[(size_t)i * n + j] = val;
	}
}

// hierarchicalCluster (:414-531): one CTA. D = working similarity matrix (n x n, global), members = n lists in a pool of n*n
// ints is avoided: cluster c's members live in `pool` as a linked structure would cost pointer chasing, so each cluster owns a
// slice of `lists` that is rebuilt on merge by thread 0 (total copies are O(n^2) in the worst case, n is a few hundred).
// One CTA per model (the merge chains of a frame's models run side by side). Model a's result: out_count[a] clusters, their
// offsets at out_offsets[lo + a ..], members (match indices inside the model) at out_members[lo ..].
__global__ void __launch_bounds__(kLinkThreads, 1) k_link_agglomerate(const LinkSlice *__restrict__ slices, const float *__restrict__ K_all, float *__restrict__ D_all,
                                                                  float cutoff, int min_pts, int linkage, int *__restrict__ valid_all, int *__restrict__ lists_all,
                                                                  int *__restrict__ sz_all, float *__restrict__ tmp_all, int *__restrict__ out_count_all,
                                                                  int *__restrict__ out_offsets_all, int *__restrict__ out_members_all,
                                                                  const int32_t *__restrict__ status) {
	__shared__ float s_val[kLinkThreads];
	__shared__ int s_a[kLinkThreads], s_b[kLinkThreads];
	__shared__ int s_nv, s_r, s_p1, s_p2, s_stop, s_sU, s_sR;
	const int tid = threadIdx.x;
	const int n = slices[blockIdx.x].n, lo = slices[blockIdx.x].lo;
	const int64_t sq = slices[blockIdx.x].sq;
	int *out_count = out_count_all + blockIdx.x, *out_offsets = out_offsets_all + lo + blockIdx.x, *out_members = out_members_all + lo;
	if (status && *status) { if (tid == 0) { *out_count = 0; out_offsets[0] = 0; } return; }
	const float *K = K_all + sq;
	float *D = D_all + sq, *tmp = tmp_all + 3 * (size_t)lo;
	int *valid = valid_all + lo, *lists = lists_all + sq, *sz = sz_all + lo;
	for (size_t k = tid; k < (size_t)n * n; k += blockDim.x) D[k] = K[k];       // distances[i][j] = K->getProb(i, j) (:434-439)
	for (int i = tid; i < n; i += blockDim.x) { valid[i] = i; lists[(size_t)i * n] = i; sz[i] = 1; }
	if (tid == 0) { s_nv = n; s_r = -1; s_stop = 0; }
	__syncthreads();
	for (;;) {
		const int nv = s_nv, r = s_r;      // r = position of the merged-away index in the list, or -1
		// argmax over the pairs the reference's double loop visits: position a (not r, not r+1: erase-then-++ skips it) with every later
		// position b; strict > keeps the first maximum in (a, b) order and, like the reference's, never picks a NaN (duplicate matches)
		float best = -1;
		int ba = 0x7fffffff, bb = 0x7fffffff;
		for (int a = tid; a < nv; a += blockDim.x) {
			if (r >= 0 && (a == r || a == r + 1)) continue;
			const float *row = D + (size_t)valid[a] * n;
			for (int b = a + 1; b < nv; b++) {
				const float v = row[valid[b]];
				if (v > best) { best = v; ba = a; bb = b; }        // a ascends within a thread: ties keep the earlier pair
			}
		}
		s_val[tid] = best; s_a[tid] = ba; s_b[tid] = bb;
		__syncthreads();
		for (int o = kLinkThreads / 2; o > 0; o >>= 1) {
			if (tid < o) {
				const float v2 = s_val[tid + o];
				const int a2 = s_a[tid + o], b2 = s_b[tid + o];
				if (v2 > s_val[tid] || (v2 == s_val[tid] && (a2 < s_a[tid] || (a2 == s_a[tid] && b2 < s_b[tid])))) { s_val[tid] = v2; s_a[tid] = a2; s_b[tid] = b2; }
			}
			__syncthreads();
		}
		if (tid == 0) {
			const float maxSim = s_val[0];
			const int p1 = s_a[0] < nv ? valid[s_a[0]] : 0, p2 = s_b[0] < nv ? valid[s_b[0]] : 0;      // maxPair stays (0,0)-like if nothing was found
			int nvn = nv;
			if (r >= 0) {                                   // validIndices.erase(position r)
				for (int k = r; k < nv - 1; k++) valid[k] = valid[k + 1];
				nvn = nv - 1;
			}
			s_nv = nvn;
			if (maxSim < cutoff) s_stop = 1;
			else {
				s_p1 = p1; s_p2 = p2; s_sU = sz[p1]; s_sR = sz[p2];
				// merge: the second cluster is appended back to front (:480-483)
				int *l1 = lists + (size_t)p1 * n, *l2 = lists + (size_t)p2 * n;
				while (sz[p2] != 0) l1[sz[p1]++] = l2[--sz[p2]];
				int pos = -1;                                // removeValue = p2: its position in the (already erased) list
				for (int k = 0; k < nvn; k++) if (valid[k] == p2) { pos = k; break; }
				s_r = pos;
			}
		}
		__syncthreads();
		if (s_stop) break;
		const int tU = s_p1, rV = s_p2, sU = s_sU, sR = s_sR;
		// row/column update of the merged cluster (:489-512). Every i reads the OLD (toUpdate, i) and (removeValue, i): new values go
		// to tmp first (the sequential loop reads entries before it overwrites them because toUpdate < removeValue)
		for (int i = tid; i < n; i += blockDim.x) {
			float v;
			if (linkage == 1) v = (float)((1.0 / (sU + sR)) * (sU * D[(size_t)tU * n + i] + sR * D[(size_t)rV * n + i]));
			else {
				v = linkage == 0 ? (float)1e20 : -1;
				const int *li = lists + (size_t)i * n, *lu = lists + (size_t)tU * n;
				const int si = sz[i], su = sz[tU];
				for (int a = 0; a < si; a++)
					for (int b = 0; b < su; b++) {
						const float k = K[(size_t)lu[b] * n + li[a]];
						if (linkage == 0 ? (k < v) : (k > v)) v = k;
					}
			}
			tmp[i] = v;
		}
		__syncthreads();
		for (int i = tid; i < n; i += blockDim.x) { D[(size_t)tU * n + i] = tmp[i]; D[(size_t)i * n + tU] = tmp[i]; }
		__syncthreads();
	}
	if (tid == 0) {                                       // clusters with more than MinPts members, in index order (:519-529)
		int nc = 0, k = 0;
		out_offsets[0] = 0;
		for (int i = 0; i < n; i++)
			if (sz[i] > min_pts) {
				const int *l = lists + (size_t)i * n;
				for (int a = 0; a < sz[i]; a++) out_members[k++] = l[a];
				out_offsets[++nc] = k;
			}
		*out_count = nc;
	}
}

// The same agglomeration with a cached maximum per row (linkage_cached.cuh; average linkage only): O(n) per merge plus repairs
// instead of an O(n^2) scan. mc_set_option("linkage_cached", 1).
__global__ void __launch_bounds__(kLinkThreads) k_link_agglomerate_cached(const LinkSlice *__restrict__ slices, const float *__restrict__ K_all,
                                                                         float *__restrict__ D_all, float cutoff, int min_pts, int *__restrict__ L_all,
                                                                         int *__restrict__ lists_all, int *__restrict__ sz_all, float *__restrict__ tmp3_all,
                                                                         int *__restrict__ ints3_all, int *__restrict__ out_count_all,
                                                                         int *__restrict__ out_offsets_all, int *__restrict__ out_members_all,
                                                                         const int32_t *__restrict__ status) {
	__shared__ float s_val[kLinkThreads];
	__shared__ int s_idx[kLinkThreads], s_ctl[16];
	const LinkSlice sl = slices[blockIdx.x];
	const int n = sl.n;
	int *out_count = out_count_all + blockIdx.x, *out_offsets = out_offsets_all + sl.lo + blockIdx.x, *out_members = out_members_all + sl.lo;
	if (status && *status) { if (threadIdx.x == 0) { *out_count = 0; out_offsets[0] = 0; } return; }
	float *tmp3 = tmp3_all + 3 * (size_t)sl.lo;
	int *ints3 = ints3_all + 3 * (size_t)sl.lo;
	lkx::State s;
	s.n = n; s.D = D_all + sl.sq; s.L = L_all + sl.lo; s.lists = lists_all + sl.sq; s.sz = sz_all + sl.lo;
	s.tmp = tmp3; s.oldcol = tmp3 + n; s.best = tmp3 + 2 * (size_t)n;
	s.posOf = ints3; s.arg = ints3 + n; s.tmpi = ints3 + 2 * (size_t)n;
	s.s_val = s_val; s.s_idx = s_idx; s.ctl = s_ctl;
	lkx::Block<kLinkThreads> blk;
	blk.tid = threadIdx.x;
	lkx::agglomerate_average(blk, s, K_all + sl.sq, cutoff, min_pts, out_count, out_offsets, out_members);
}

// The clusters of every model of a frame, model-major (what CLUSTER_LINKAGE leaves in frameData.clusters[model]): cluster_model,
// cluster_offsets (into members), members = match indices inside the model in the agglomeration's list order. One CTA.
// out_n = {clusters, members}. Also zeroes the frame's object count for the POSE step that follows.
__global__ void __launch_bounds__(kLinkThreads) k_link_compact(const LinkSlice *__restrict__ slices, int n_slices, const int *__restrict__ out_count,
                                                              const int *__restrict__ out_offsets, const int *__restrict__ out_members,
                                                              int *__restrict__ base, int32_t *__restrict__ out_n, int32_t *__restrict__ cluster_model,
                                                              int32_t *__restrict__ cluster_offsets, int32_t *__restrict__ members,
                                                              int32_t *__restrict__ n_obj) {
	if (threadIdx.x == 0) {                     // cluster and member base of every model
		int c = 0, k = 0;
		for (int a = 0; a < n_slices; a++) {
			base[2 * a] = c; base[2 * a + 1] = k;
			const int nc = out_count[a];
			c += nc; k += out_offsets[slices[a].lo + a + nc];
		}
		out_n[0] = c; out_n[1] = k;
		cluster_offsets[c] = k;
		*n_obj = 0;
	}
	__syncthreads();
	for (int a = 0; a < n_slices; a++) {
		const LinkSlice sl = slices[a];
		const int nc = out_count[a], c0 = base[2 * a], k0 = base[2 * a + 1];
		const int *off = out_offsets + sl.lo + a, *mem = out_members + sl.lo;
		for (int c = threadIdx.x; c < nc; c += blockDim.x) { cluster_model[c0 + c] = sl.model; cluster_offsets[c0 + c] = k0 + off[c]; }
		for (int t = threadIdx.x; t < off[nc]; t += blockDim.x) members[k0 + t] = mem[t];
	}
}

// ---- host side -------------------------------------------------------------------------------------------------------------

// Arena of one frame's linkage (sq_total = sum of n^2 over its models, M = its matches, S = its models): five n x n matrices and the
// merge lists per model, per-match state, and the per-model outputs. Laid out by link_carve.
size_t link_arena_bytes(int64_t sq_total, int M, int S) {
	const size_t floats = 5 * (size_t)sq_total + 3 * (size_t)M + 4 * (size_t)S;
	const size_t ints = (size_t)sq_total + 5 * (size_t)M + (size_t)S + ((size_t)M + S + 1) + (size_t)M + 2 * (size_t)S + 2;
	return (floats + ints) * 4 + 64;
}

void link_carve(void *arena, int64_t sq_total, int M, int S, LinkFrame &F) {
	const size_t sq = (size_t)sq_total;
	float *f = (float *)arena;
	F.K2D = f; f += sq; F.K3D = f; f += sq; F.K3F = f; f += sq; F.K = f; f += sq; F.D = f; f += sq;
	F.tmp = f; f += 3 * (size_t)M; F.scal = f; f += 4 * (size_t)S;
	int *i = (int *)f;
	F.valid = i; i += M; F.lists = i; i += sq; F.sz = i; i += M; F.ints3 = i; i += 3 * (size_t)M;
	F.out_count = i; i += S; F.out_offsets = i; i += (size_t)M + S + 1; F.out_members = i; i += M; F.compact = i;
}

static mc_status link_agglomerate_only(mc_ctx *ctx, const LinkFrame &F, float cutoff, int min_pts, int linkage);

// sigma -> pairs -> max/scale (x2 with the 3-D filter) -> blend -> agglomeration for every model of F, one launch each
mc_status link_frame_device(mc_ctx *ctx, const LinkFrame &F, float cutoff, int min_pts, int use3DFilter, int linkage, float sigma2D, float sigma3D) {
	cudaStream_t st = ctx->stream;
	const int S = F.n_slices, nmax = F.n_max;
	if (S <= 0) return MC_OK;
	MC_CUDA(cudaMemsetAsync(F.scal, 0, 4 * (size_t)S * sizeof(float), st));
	k_link_sigma<<<S, kLinkThreads, 0, st>>>(F.slices, F.xy, F.xyz, sigma2D, sigma3D, F.tmp, F.scal, F.W, F.H, F.status);
	MC_LAUNCH_CHECK();
	const dim3 g((nmax + kLinkThreads - 1) / kLinkThreads, nmax, S < 65535 ? S : 65535);
	k_link_pairs<<<g, kLinkThreads, 0, st>>>(F.slices, S, F.xy, F.xyz, F.world, F.W, F.H, F.depth, F.scal, use3DFilter, F.K2D, F.K3D, F.K3F);
	MC_LAUNCH_CHECK();
	// the maximum is order-independent and the scaling elementwise: any number of blocks per model gives the same bits
	const int64_t want = ((int64_t)nmax * nmax + kLinkThreads - 1) / kLinkThreads, per = (4 * ctx->num_sms + S - 1) / S;
	const dim3 gr((unsigned)(want < per ? want : per), S);
	k_link_max<<<gr, kLinkThreads, 0, st>>>(F.slices, F.K3D, nullptr, 0, F.scal, 2);
	MC_LAUNCH_CHECK();
	k_link_scale<<<gr, kLinkThreads, 0, st>>>(F.slices, F.K3D, F.scal, 2);
	MC_LAUNCH_CHECK();
	if (use3DFilter) {
		k_link_max<<<gr, kLinkThreads, 0, st>>>(F.slices, F.K3D, F.K3F, use3DFilter == 1 ? 1 : 2, F.scal, 3);
		MC_LAUNCH_CHECK();
		k_link_scale<<<gr, kLinkThreads, 0, st>>>(F.slices, F.K3D, F.scal, 3);
		MC_LAUNCH_CHECK();
	}
	k_link_blend<<<g, kLinkThreads, 0, st>>>(F.slices, S, F.xy, F.W, F.distance, F.K2D, F.K3D, F.K, F.status);
	MC_LAUNCH_CHECK();
	return link_agglomerate_only(ctx, F, cutoff, min_pts, linkage);
}

static mc_status link_agglomerate_only(mc_ctx *ctx, const LinkFrame &F, float cutoff, int min_pts, int linkage) {
	cudaStream_t st = ctx->stream;
	const int S = F.n_slices;
	if (ctx->linkage_cached && linkage == 1)
		k_link_agglomerate_cached<<<S, kLinkThreads, 0, st>>>(F.slices, F.K, F.D, cutoff, min_pts, F.valid, F.lists, F.sz, F.tmp, F.ints3, F.out_count,
		                                                      F.out_offsets, F.out_members, F.status);
	else
		k_link_agglomerate<<<S, kLinkThreads, 0, st>>>(F.slices, F.K, F.D, cutoff, min_pts, linkage, F.valid, F.lists, F.sz, F.tmp, F.out_count,
		                                               F.out_offsets, F.out_members, F.status);
	MC_LAUNCH_CHECK();
	return MC_OK;
}

mc_status link_compact_device(mc_ctx *ctx, const LinkFrame &F, int32_t *d_out_n, int32_t *d_cluster_model, int32_t *d_cluster_offsets,
                              int32_t *d_members, int32_t *d_n_obj) {
	k_link_compact<<<1, kLinkThreads, 0, ctx->stream>>>(F.slices, F.n_slices, F.out_count, F.out_offsets, F.out_members, F.compact, d_out_n,
	                                                    d_cluster_model, d_cluster_offsets, d_members, d_n_obj);
	MC_LAUNCH_CHECK();
	return MC_OK;
}

// One model on ctx->stream (mc_cluster_linkage, mc_linkage_agglomerate): its inputs and slice descriptor ahead of the arena in
// ctx->link_buf
struct LinkOne { float *xy, *xyz, *world, *depth, *distance; LinkFrame F; };

static mc_status link_one_alloc(mc_ctx *ctx, int n, size_t px, LinkOne &B) {
	const size_t nn = (size_t)n * n;
	const size_t in_floats = 8 * (size_t)n + 2 * px + 8;
	MC_TRY(reserve(ctx, ctx->link_buf, in_floats * sizeof(float) + sizeof(LinkSlice) + link_arena_bytes((int64_t)nn, n, 1) + 256));
	float *f = (float *)ctx->link_buf.p;
	B.xy = f; f += 2 * (size_t)n; B.xyz = f; f += 3 * (size_t)n; B.world = f; f += 3 * (size_t)n;
	B.depth = f; f += px; B.distance = f; f += px;
	LinkSlice *slice = (LinkSlice *)(((uintptr_t)f + 63) & ~(uintptr_t)63);
	const LinkSlice one = { 0, 0, n, 0, 0 };
	MC_CUDA(cudaMemcpyAsync(slice, &one, sizeof one, cudaMemcpyHostToDevice, ctx->stream));
	LinkFrame &F = B.F;
	F.slices = slice; F.n_slices = 1; F.n_max = n;
	F.xy = B.xy; F.xyz = B.xyz; F.world = B.world; F.depth = B.depth; F.distance = B.distance; F.W = 0; F.H = 0;
	F.status = nullptr;
	link_carve(slice + 1, (int64_t)nn, n, 1, F);
	return MC_OK;
}

// the model's clusters -> host (CSR as mc_cluster_linkage returns it)
static mc_status link_one_download(mc_ctx *ctx, const LinkOne &B, int n, int32_t *n_clusters, int32_t *cluster_offsets, int32_t *members) {
	cudaStream_t st = ctx->stream;
	// out_count, out_offsets (n + 2) and out_members are contiguous in the arena
	const size_t words = 1 + (size_t)(n + 2) + (size_t)n;
	MC_TRY(pinned(ctx, words * sizeof(int)));
	int *h = (int *)ctx->h_pinned;
	MC_CUDA(cudaMemcpyAsync(h, B.F.out_count, words * sizeof(int), cudaMemcpyDeviceToHost, st));
	MC_CUDA(cudaStreamSynchronize(st));
	const int nc = h[0];
	*n_clusters = nc;
	for (int c = 0; c <= nc; c++) cluster_offsets[c] = h[1 + c];
	for (int k = 0; k < h[1 + nc]; k++) members[k] = h[1 + (n + 2) + k];
	return MC_OK;
}

} // namespace mc

using namespace mc;

static mc_status link_check(mc_ctx *ctx, int n, const char *who) {
	if (n < 1 || n > 2048) { ctx->err = std::string(who) + ": n_matches must be in 1..2048"; return MC_ERR_ARG; }
	return MC_OK;
}

extern "C" mc_status mc_cluster_linkage(mc_ctx *ctx, const float *match_xy, const float *match_xyz, const float *match_world, int n_matches,
                                        const float *depth, const float *fill_distance, int width, int height,
                                        float cutoff, int min_pts, int use_3d_filter, int linkage_type, float sigma_2d, float sigma_3d,
                                        int32_t *n_clusters, int32_t *cluster_offsets, int32_t *members, float *similarity_out) {
	if (!ctx) return MC_ERR_ARG;
	if (!match_xy || !match_xyz || !match_world || !depth || !fill_distance || !n_clusters || !cluster_offsets || !members || width < 1 || height < 1) {
		ctx->err = "mc_cluster_linkage: bad argument"; return MC_ERR_ARG;
	}
	if (n_matches == 0) { *n_clusters = 0; cluster_offsets[0] = 0; return MC_OK; }
	MC_TRY(link_check(ctx, n_matches, "mc_cluster_linkage"));
	// the blend kernel reads the fill-distance map at every match's pixel (the reference indexes its map unchecked,
	// CLUSTER_LINKAGE_CPU.hpp:324-365): a coordinate outside the map is an argument error here, not an illegal address
	for (int i = 0; i < n_matches; i++) {
		const float x = match_xy[2 * i], y = match_xy[2 * i + 1];
		if (!(x >= 0.f && y >= 0.f && (int)x < width && (int)y < height)) { ctx->err = "mc_cluster_linkage: match coordinate outside the depth map"; return MC_ERR_ARG; }
	}
	// with cutoff <= -1 the merge loop has no stopping point once a single cluster is left (the reference then spins on the host)
	if (!(cutoff > -1.f)) { ctx->err = "mc_cluster_linkage: cutoff must be > -1"; return MC_ERR_ARG; }
	MC_CUDA(cudaSetDevice(ctx->device));
	const int n = n_matches;
	const size_t px = (size_t)width * height;
	LinkOne B;
	MC_TRY(link_one_alloc(ctx, n, px, B));
	cudaStream_t st = ctx->stream;
	MC_CUDA(cudaMemcpyAsync(B.xy, match_xy, sizeof(float) * 2 * n, cudaMemcpyHostToDevice, st));
	MC_CUDA(cudaMemcpyAsync(B.xyz, match_xyz, sizeof(float) * 3 * n, cudaMemcpyHostToDevice, st));
	MC_CUDA(cudaMemcpyAsync(B.world, match_world, sizeof(float) * 3 * n, cudaMemcpyHostToDevice, st));
	MC_CUDA(cudaMemcpyAsync(B.depth, depth, sizeof(float) * px, cudaMemcpyHostToDevice, st));
	MC_CUDA(cudaMemcpyAsync(B.distance, fill_distance, sizeof(float) * px, cudaMemcpyHostToDevice, st));
	B.F.W = width; B.F.H = height;
	MC_TRY(link_frame_device(ctx, B.F, cutoff, min_pts, use_3d_filter, linkage_type, sigma_2d, sigma_3d));
	if (similarity_out) MC_CUDA(cudaMemcpyAsync(similarity_out, B.F.K, sizeof(float) * (size_t)n * n, cudaMemcpyDeviceToHost, st));
	return link_one_download(ctx, B, n, n_clusters, cluster_offsets, members);
}

extern "C" mc_status mc_linkage_agglomerate(mc_ctx *ctx, const float *similarity, int n, float cutoff, int min_pts, int linkage_type,
                                            int32_t *n_clusters, int32_t *cluster_offsets, int32_t *members) {
	if (!ctx) return MC_ERR_ARG;
	if (!similarity || !n_clusters || !cluster_offsets || !members) { ctx->err = "mc_linkage_agglomerate: null pointer"; return MC_ERR_ARG; }
	if (n == 0) { *n_clusters = 0; cluster_offsets[0] = 0; return MC_OK; }
	MC_TRY(link_check(ctx, n, "mc_linkage_agglomerate"));
	if (!(cutoff > -1.f)) { ctx->err = "mc_linkage_agglomerate: cutoff must be > -1"; return MC_ERR_ARG; }
	MC_CUDA(cudaSetDevice(ctx->device));
	LinkOne B;
	MC_TRY(link_one_alloc(ctx, n, 1, B));
	MC_CUDA(cudaMemcpyAsync(B.F.K, similarity, sizeof(float) * (size_t)n * n, cudaMemcpyHostToDevice, ctx->stream));
	MC_TRY(link_agglomerate_only(ctx, B.F, cutoff, min_pts, linkage_type));
	return link_one_download(ctx, B, n, n_clusters, cluster_offsets, members);
}
