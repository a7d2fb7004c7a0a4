// sift.cu — step 1 of MOPED's pipeline (feature extraction) on the device: the producer on the input side of MATCH
// (SURVEY.md §8f row 3). Replaces FEAT_SIFT_CPU::process (moped2/libmoped/src/feat/FEAT_SIFT_CPU.hpp:78-112) over the
// vendored libsiftfast 1.1 (libs.tgz!libsiftfast-1.1-src/libsiftfast.cpp; the vendored copy #undef's __SSE*__ at :40-42,
// so the reference runs its scalar branches — those are the ones followed here).
//
// Design (B200): a BATCH of equally sized images per call; every kernel has the frame as a grid dimension, so one
// set of ~100 launches serves all frames of a camera rig / stream batch. The scale-space of a 640x480 frame
// (1278x958 after doubling, 7 octaves) is ~110 MB and stays L2/HBM resident; the pyramid kernels are HBM/L2-bound
// streaming kernels, the keypoint kernels (one warp / one CTA per keypoint) are latency-bound and small.
//
// Arithmetic: sums are in the reference's source order; the convolution taps accumulate with explicit fused
// multiply-add in tap order (one of the roundings -ffast-math leaves to the reference's compiler, see the oracle's
// header), everything else is compiled with -fmad=false (separate multiply and add); '/' and sqrtf are IEEE. So the
// pyramid, the DoG extrema, the sub-pixel fit and hence the keypoint SET are bit-identical to the C restatement
// (oracle/moped_sift_oracle.c). Only expf/atan2f/sinf/cosf/powf differ from
// glibc's by an ulp or two. Orientation-histogram and descriptor bins are gathered into per-thread PRIVATE accumulators
// (no two threads ever add to the same word) and combined in a fixed order: deterministic run to run and independent
// of the batch, within float rounding of the reference's sequential chain.
//
// Output order = the order FEAT_SIFT_CPU emits with one OpenMP thread: the reverse of creation order
// (libsiftfast.cpp:941-951,1423), i.e. octave descending, then DoG index / row / column descending, then
// orientation peak descending.
#include "common.cuh"

#include <algorithm>
#include <math.h>
#include <string.h>

namespace mc {

constexpr int kSiftScales = 3;
constexpr int kSiftMaxOct = 16;
constexpr float kSiftInitSigma = 1.6f;
#define SIFT_PI 3.141592654f
#define SIFT_SQRT2 1.4142136f

struct GaussK { float k[64]; int ksize; };

struct SiftOct {
	int rows, cols;
	size_t plane;                 // rows*cols
	float *gauss, *dog, *grad, *ori;   // [frame][6|5|3|3][plane]
	int32_t *claim;               // [frame][plane]: smallest scan id that reached this pixel (duplicate suppression)
};

struct SiftCand { int frame, oct, index, row, col, scan_id; float X[3]; };
struct SiftKp { int frame, oct, index; float frow, fcol, fsize, ori; unsigned long long key; int slot; };

struct SiftState {
	int B = 0, H = 0, W = 0, dbl = -1, n_oct = 0, max_kp = 0, cap_cand = 0;
	SiftOct oct[kSiftMaxOct];
	DevBuf pyr, tmp, tmp2, gray, cand, kp, counters, lut, offs;
	GaussK k_init, k_oct[kSiftScales + 2];
	bool has_init = false;
	cudaEvent_t ev[2 * (kSiftScales + 2)] = {};   // mc_set_profiling: around the five octave-0 Gaussian+DoG launches
	bool ev_valid = false;
	double ev_bytes = 0;
	unsigned smem_configured = 0;  // bit per kernel instance whose dynamic shared-memory limit was raised on this context's device
	bool two_pass = false;
	bool gather = false;          // mc_set_option("sift_describe_gather"): the cell-gather descriptor kernel (A/B aid)        // mc_set_option("sift_two_pass"): the unfused blur kernels (A/B aid, same bits)
};

// GaussianBlur's kernel (libsiftfast.cpp:470-508): ksize+1 weights enter the sum, ksize are normalised (host, glibc expf)
static void make_kernel(float fblur, GaussK &g) {
	const float GaussTruncate = 4.0f;
	int ksize = (int)(2.0f * GaussTruncate * fblur + 1.0f);
	if (ksize < 3) ksize = 3;
	ksize += !(ksize & 1);
	double faccum = 0;
	int width = ksize >> 1;
	memset(g.k, 0, sizeof(g.k));
	for (int i = 0; i <= ksize; ++i) {
		float fweight = expf(-(float)(i - width) * (i - width) / (2.0f * fblur * fblur));
		faccum += (double)fweight;
		g.k[i] = fweight;
	}
	for (int i = 0; i < ksize; ++i) g.k[i] /= (float)faccum;
	g.k[ksize] = 0.f;
	g.ksize = ksize;
}

// ---- pyramid kernels -------------------------------------------------------------------------------------------

// FEAT_SIFT_CPU.hpp:86-90 (pixel = (float)(g * 1./255.), a 256-entry table computed on the host in double) followed by
// SiftDoubleSize (libsiftfast.cpp:363-380) or SiftCopyImage (:382-388)
__global__ void k_sift_base(const uint8_t *__restrict__ gray, const float *__restrict__ lut, int H, int W, int dbl,
                            float *__restrict__ dst, int rows, int cols) {
	int c = blockIdx.x * blockDim.x + threadIdx.x, r = blockIdx.y, f = blockIdx.z;
	if (c >= cols) return;
	const uint8_t *g = gray + (size_t)f * H * W;
	float v;
	if (!dbl) v = lut[g[(size_t)r * W + c]];
	else {
		int i = r >> 1, j = c >> 1;
		float p00 = lut[g[(size_t)i * W + j]], p01 = lut[g[(size_t)i * W + j + 1]];
		float p10 = lut[g[(size_t)(i + 1) * W + j]], p11 = lut[g[(size_t)(i + 1) * W + j + 1]];
		if (!(r & 1)) v = (c & 1) ? 0.5f * (p00 + p01) : p00;
		else v = (c & 1) ? 0.25f * (p00 + p01 + p10 + p11) : 0.5f * (p00 + p10);
	}
	dst[(size_t)f * rows * cols + (size_t)r * cols + c] = v;
}

// ConvHorizontal + ConvBuffer (libsiftfast.cpp:523-546,573-581): replicate padding, taps summed in order j = 0..ksize-1.
// src/dst frames are fstride_src / fstride_dst floats apart.
__global__ void k_sift_blur_h(const float *__restrict__ src, size_t fstride_src, float *__restrict__ dst, size_t fstride_dst,
                              int rows, int cols, const __grid_constant__ GaussK gk) {
	int c = blockIdx.x * blockDim.x + threadIdx.x, r = blockIdx.y, f = blockIdx.z;
	if (c >= cols) return;
	const float *p = src + (size_t)f * fstride_src + (size_t)r * cols;
	const int ksize = gk.ksize, width = ksize >> 1;
	float acc = 0.f;
	for (int j = 0; j < ksize; ++j) {
		int x = c + j - width;
		x = x < 0 ? 0 : (x >= cols ? cols - 1 : x);
		acc = __fmaf_rn(__ldg(p + x), gk.k[j], acc);
	}
	dst[(size_t)f * fstride_dst + (size_t)r * cols + c] = acc;
}

// ConvVertical (:548-571) fused with SubtractImage (:460-464): dst = blur_v(src); if dog: dog = prev - dst
// (prev = the image being blurred; every stack has its own frame stride)
__global__ void k_sift_blur_v(const float *__restrict__ src, size_t fstride_src, float *__restrict__ dst, size_t fstride_dst,
                              const float *__restrict__ prev, size_t fstride_prev, float *__restrict__ dog, size_t fstride_dog, int rows, int cols,
                              const __grid_constant__ GaussK gk) {
	int c = blockIdx.x * blockDim.x + threadIdx.x, r = blockIdx.y, f = blockIdx.z;
	if (c >= cols) return;
	const float *p = src + (size_t)f * fstride_src + c;
	const int ksize = gk.ksize, width = ksize >> 1;
	float acc = 0.f;
	for (int j = 0; j < ksize; ++j) {
		int y = r + j - width;
		y = y < 0 ? 0 : (y >= rows ? rows - 1 : y);
		acc = __fmaf_rn(__ldg(p + (size_t)y * cols), gk.k[j], acc);
	}
	size_t o = (size_t)r * cols + c;
	dst[(size_t)f * fstride_dst + o] = acc;
	if (dog) dog[(size_t)f * fstride_dog + o] = prev[(size_t)f * fstride_prev + o] - acc;
}

// GaussianBlur (:470-521) as ONE persistent kernel: a CTA takes 64x64 output tiles in turn; it loads a tile plus its halo (replicate-clamped at the image
// border like ConvHorizontal/ConvVertical's padded line buffers), runs the horizontal pass into shared memory (also for
// the halo rows the vertical pass needs), then the vertical pass, and writes the Gaussian image and — SubtractImage
// (:460-464) fused — the DoG image = (centre of the input tile) - result. Per output pixel the taps are summed in the
// reference's order j = 0..ksize-1 exactly as in the two-pass kernels above, so the result is bit-identical to them.
// Register blocking: a thread produces 8 consecutive outputs from one sliding window of ksize+7 shared-memory loads;
// in the horizontal pass the lanes of a warp span ROWS (odd pitches -> conflict-free), in the vertical pass columns.
// HBM traffic per blur: 1 plane read (+halo from L2), 2 planes written, instead of 6 plane passes unfused.
// The tile loads are cp.async requests into a second buffer issued BEFORE the current tile is convolved (ncu on the
// load -> barrier -> compute version: 57 % of the stall samples on the shared-memory store waiting for the global loads).
// cp.async of one 4-byte word (global -> shared, bypassing registers): lets a CTA request its NEXT tile while it
// convolves the current one
__device__ __forceinline__ void cp_async4(float *smem_dst, const float *gmem_src) {
	asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }

template <int KS>
__global__ void __launch_bounds__(256) k_sift_blur(const float *__restrict__ src, size_t fstride_src, float *__restrict__ dst, size_t fstride_dst,
                                                   float *__restrict__ dog, size_t fstride_dog, int rows, int cols, int ntx, int nty, int n_tiles,
                                                   const __grid_constant__ GaussK gk) {
	constexpr int W = KS / 2, TW = 64, TH = 64, IH = TH + 2 * W, IW = TW + 2 * W, PIN = IW + 1, PMID = TW + 1, G = 8;
	extern __shared__ float sm[];
	float *s_mid = sm + 2 * IH * PIN;                  // sm[0 .. 2*IH*PIN): input tile + halo, double buffered
	const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;

	// requests tile t into buffer b: a warp per tile row (row clamp and row pointer once per row), lanes along the row;
	// replicate-clamped at the image border like ConvHorizontal/ConvVertical's padded line buffers
	auto prefetch = [&](int t, int b) {
		const int f = t / (ntx * nty), rem = t - f * (ntx * nty), by = rem / ntx, bx = rem - by * ntx;
		const int c0 = bx * TW, r0 = by * TH;
		const float *p = src + (size_t)f * fstride_src;
		const bool interior = r0 >= W && r0 + TH + W <= rows && c0 >= W && c0 + TW + W <= cols;      // block-uniform
		for (int i = wid; i < IH; i += 8) {
			int y = r0 - W + i;
			y = y < 0 ? 0 : (y >= rows ? rows - 1 : y);
			const float *prow = p + (size_t)y * cols + (c0 - W);
			float *srow = sm + b * (IH * PIN) + i * PIN;
			if (interior) {
#pragma unroll
				for (int j = lane; j < IW; j += 32) cp_async4(srow + j, prow + j);
			} else {
#pragma unroll
				for (int j = lane; j < IW; j += 32) {
					int x = c0 - W + j;
					x = x < 0 ? 0 : (x >= cols ? cols - 1 : x);
					cp_async4(srow + j, prow + (x - (c0 - W)));
				}
			}
		}
		cp_async_commit();
	};

	int t = blockIdx.x, cur = 0;
	if (t < n_tiles) prefetch(t, 0);
	for (; t < n_tiles; t += gridDim.x, cur ^= 1) {
		const int tn = t + gridDim.x;
		if (tn < n_tiles) { prefetch(tn, cur ^ 1); cp_async_wait<1>(); } else cp_async_wait<0>();
		__syncthreads();                                // tile t is in s_buf[cur] for every thread
		const float *s_in = sm + cur * (IH * PIN);
		const int f = t / (ntx * nty), rem = t - f * (ntx * nty), by = rem / ntx, bx = rem - by * ntx;
		const int c0 = bx * TW, r0 = by * TH;
		for (int item = threadIdx.x; item < IH * (TW / G); item += 256) {
			int row = item % IH, g = item / IH;
			const float *in = s_in + row * PIN + g * G;
			float v[KS + G - 1], acc[G];
#pragma unroll
			for (int q = 0; q < KS + G - 1; ++q) v[q] = in[q];
#pragma unroll
			for (int k = 0; k < G; ++k) acc[k] = 0.f;
#pragma unroll
			for (int j = 0; j < KS; ++j)
#pragma unroll
				for (int k = 0; k < G; ++k) acc[k] = __fmaf_rn(v[k + j], gk.k[j], acc[k]);
#pragma unroll
			for (int k = 0; k < G; ++k) s_mid[row * PMID + g * G + k] = acc[k];
		}
		__syncthreads();
		for (int item = threadIdx.x; item < TW * (TH / G); item += 256) {
			int col = item % TW, h = item / TW;
			const float *in = s_mid + (h * G) * PMID + col;
			float v[KS + G - 1], acc[G];
#pragma unroll
			for (int q = 0; q < KS + G - 1; ++q) v[q] = in[q * PMID];
#pragma unroll
			for (int k = 0; k < G; ++k) acc[k] = 0.f;
#pragma unroll
			for (int j = 0; j < KS; ++j)
#pragma unroll
				for (int k = 0; k < G; ++k) acc[k] = __fmaf_rn(v[k + j], gk.k[j], acc[k]);
			const int x = c0 + col, nrow = rows - (r0 + h * G);        // nrow = rows of this strip inside the image
			if (x < cols && nrow > 0) {
				const size_t o = (size_t)(r0 + h * G) * cols + x;        // one address per strip, rows advance by `cols`
				float *dp = dst + (size_t)f * fstride_dst + o;
				const float *cin = s_in + (h * G + W) * PIN + col + W;
				if (dog) {
					float *gp = dog + (size_t)f * fstride_dog + o;
#pragma unroll
					for (int k = 0; k < G; ++k)
						if (k < nrow) { dp[(size_t)k * cols] = acc[k]; gp[(size_t)k * cols] = cin[k * PIN] - acc[k]; }
				} else {
#pragma unroll
					for (int k = 0; k < G; ++k)
						if (k < nrow) dp[(size_t)k * cols] = acc[k];
				}
			}
		}
		__syncthreads();                                // s_buf[cur] and s_mid are free again: the next iteration prefetches into s_buf[cur]
	}
}

template <int KS>
static mc_status launch_blur_t(mc_ctx *ctx, unsigned &configured, const float *src, size_t fs_src, float *dst, size_t fs_dst, float *dog, size_t fs_dog,
                               int rows, int cols, int B, const GaussK &gk) {
	constexpr int W = KS / 2, IH = 64 + 2 * W, IW = 64 + 2 * W;
	constexpr size_t smem = (2 * (size_t)IH * (IW + 1) + (size_t)IH * 65) * sizeof(float);
	if (!(configured & (1u << W))) {        // the attribute belongs to the device of this context, not to the process
		MC_CUDA(cudaFuncSetAttribute(k_sift_blur<KS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
		configured |= 1u << W;
	}
	const int ntx = (cols + 63) / 64, nty = (rows + 63) / 64, n_tiles = ntx * nty * B;
	const int per_sm = (int)((227 * 1024) / (smem + 1024));                  // resident CTAs per SM by shared memory
	const int grid = n_tiles < ctx->num_sms * per_sm ? n_tiles : ctx->num_sms * per_sm;
	k_sift_blur<KS><<<grid, 256, smem, ctx->stream>>>(src, fs_src, dst, fs_dst, dog, fs_dog, rows, cols, ntx, nty, n_tiles, gk);
	MC_LAUNCH_CHECK();
	return MC_OK;
}

// HalfImageSize (:390-408)
__global__ void k_sift_half(const float *__restrict__ src, size_t fstride_src, int cols, float *__restrict__ dst, size_t fstride_dst,
                            int nrows, int ncols) {
	int c = blockIdx.x * blockDim.x + threadIdx.x, r = blockIdx.y, f = blockIdx.z;
	if (c >= ncols) return;
	dst[(size_t)f * fstride_dst + (size_t)r * ncols + c] = src[(size_t)f * fstride_src + (size_t)(2 * r) * cols + 2 * c];
}

// GradOriImages (:959-992) of the Gaussian images 1..3 (blockIdx.z = frame*3 + (index-1)); a block covers 128 columns x 8 rows
constexpr int kRowsPerBlock = 8;
__global__ void __launch_bounds__(128) k_sift_gradori(const float *__restrict__ gauss, float *__restrict__ grad, float *__restrict__ ori, int rows, int cols) {
	const int j = blockIdx.x * blockDim.x + threadIdx.x, f = blockIdx.z / kSiftScales, s = blockIdx.z % kSiftScales;
	if (j >= cols) return;
	const size_t plane = (size_t)rows * cols;
	const float *img = gauss + ((size_t)f * (kSiftScales + 3) + s + 1) * plane;
	const int i0 = blockIdx.y * kRowsPerBlock;
	// all loads of the thread's 8-row column strip first (rows i0-1 .. i0+8 of columns j-1, j, j+1; clamped rows are
	// loaded but not used), then the arithmetic: the loads overlap instead of each row waiting for its own
	const int jl = j == 0 ? 0 : j - 1, jr = j == cols - 1 ? j : j + 1;
	float c[kRowsPerBlock + 2], l[kRowsPerBlock], r[kRowsPerBlock];
#pragma unroll
	for (int k = 0; k < kRowsPerBlock + 2; ++k) {
		int i = i0 + k - 1;
		i = i < 0 ? 0 : (i >= rows ? rows - 1 : i);
		c[k] = __ldg(img + (size_t)i * cols + j);
	}
#pragma unroll
	for (int k = 0; k < kRowsPerBlock; ++k) {
		int i = i0 + k;
		i = i >= rows ? rows - 1 : i;
		l[k] = __ldg(img + (size_t)i * cols + jl);
		r[k] = __ldg(img + (size_t)i * cols + jr);
	}
#pragma unroll
	for (int k = 0; k < kRowsPerBlock; ++k) {
		const int i = i0 + k;
		if (i < rows) {
			// the reference's expressions (:974-989) on p[j-1], p[j], p[j+1], p[j-cols], p[j+cols]
			float fdiffc, fdiffr;
			if (j == 0) fdiffc = 2.0f * (r[k] - c[k + 1]);
			else if (j == cols - 1) fdiffc = 2.0f * (c[k + 1] - l[k]);
			else fdiffc = r[k] - l[k];
			if (i == 0) fdiffr = 2.0f * (c[k + 1] - c[k + 2]);
			else if (i == rows - 1) fdiffr = 2.0f * (c[k] - c[k + 1]);
			else fdiffr = c[k] - c[k + 2];
			const size_t o = ((size_t)f * kSiftScales + s) * plane + (size_t)i * cols + j;
			grad[o] = sqrtf(fdiffc * fdiffc + fdiffr * fdiffr);
			ori[o] = atan2f(fdiffr, fdiffc);
		}
	}
}

// ---- extrema ---------------------------------------------------------------------------------------------------

// LocalMaxMin (:1126-1147)
__device__ __forceinline__ bool local_max_min(float fval, const float *d, int cols, int r, int c) {
	for (int row = r - 1; row <= r + 1; ++row) {
		const float *pf = d + (size_t)row * cols + c - 1;
		if (fval > 0) { if (pf[0] > fval || pf[1] > fval || pf[2] > fval) return false; }
		else { if (fval > pf[0] || fval > pf[1] || fval > pf[2]) return false; }
	}
	return true;
}

// NotOnEdge (:1149-1162)
__device__ __forceinline__ bool not_on_edge(const float *d, int s, int row, int col) {
	const float *p = d + (size_t)row * s;
	float f1 = p[-s + col] - p[col] * 2 + p[s + col];
	float f2 = p[col - 1] - p[col] * 2 + p[col + 1];
	float f3 = p[s + col + 1] - p[s + col - 1];
	float f4 = p[-s + col + 1] - p[-s + col - 1];
	float f5 = (f3 - f4) * 0.25f;
	float f6 = f1 * f2 - f5 * f5;
	float f8 = f1 + f2;
	return f6 * 11 * 11 > f8 * f8 * 10;
}

// SolveLinearSystem (:1235-1274) for dim 3
__device__ void solve3(float *Y, float *H) {
	const int dim = 3;
	int bestj = 0;
	for (int i = 0; i < dim - 1; ++i) {
		float fmax = -1;
		for (int j = i; j < dim; ++j) {
			float f = H[j * dim + i];
			if (f < 0) f = -f;
			if (f > fmax) { fmax = f; bestj = j; }
		}
		if (bestj != i) {
			for (int j = 0; j < dim; ++j) { float t = H[bestj * dim + j]; H[bestj * dim + j] = H[i * dim + j]; H[i * dim + j] = t; }
			float t = Y[bestj]; Y[bestj] = Y[i]; Y[i] = t;
		}
		for (int j = i + 1; j < dim; ++j) {
			float f = H[j * dim + i] / H[i * dim + i];
			for (int k = i; k < dim; ++k) H[j * dim + k] -= f * H[i * dim + k];
			Y[j] -= Y[i] * f;
		}
	}
	for (int i = dim - 1; i >= 0; --i) {
		for (int j = dim - 1; j > i; --j) Y[i] -= Y[j] * H[i * dim + j];
		Y[i] /= H[i * dim + i];
	}
}

// FitQuadratic (:1208-1231)
__device__ float fit_quadratic(float *X, const float *d0, const float *d1, const float *d2, int s, int r, int c) {
	float H[9], Y[3];
	const float *p0 = d0 + (size_t)r * s, *p1 = d1 + (size_t)r * s, *p2 = d2 + (size_t)r * s;
	Y[0] = 0.5f * (p2[c] - p0[c]);
	Y[1] = 0.5f * (p1[s + c] - p1[-s + c]);
	Y[2] = 0.5f * (p1[c + 1] - p1[c - 1]);
	H[0] = p0[c] - 2.0f * p1[c] + p2[c];
	H[4] = p1[-s + c] - 2.0f * p1[c] + p1[s + c];
	H[8] = p1[c - 1] - 2.0f * p1[c] + p1[c + 1];
	H[3] = H[1] = 0.25f * ((p2[s + c] - p2[-s + c]) - (p0[s + c] - p0[-s + c]));
	H[6] = H[2] = 0.25f * ((p2[c + 1] - p2[c - 1]) - (p0[c + 1] - p0[c - 1]));
	H[7] = H[5] = 0.25f * ((p1[s + c + 1] - p1[s + c - 1]) - (p1[-s + c + 1] - p1[-s + c - 1]));
	X[0] = -Y[0]; X[1] = -Y[1]; X[2] = -Y[2];
	solve3(X, H);
	return p1[c] + 0.5f * (X[0] * Y[0] + X[1] * Y[1] + X[2] * Y[2]);
}

// FindMaxMin's scan (:898-939) + InterpKeyPoint (:1164-1205) up to the duplicate test. The reference marks
// s_MaxMinArray[row, col] when the FIRST extremum in scan order arrives there; here every extremum that passes the
// tests bids its scan id with atomicMin and k_sift_orient keeps the winner — the same survivor.
__global__ void k_sift_detect(const float *__restrict__ dog, int32_t *__restrict__ claim, int rows, int cols, int oct, float peak_thresh,
                              SiftCand *__restrict__ cand, int *__restrict__ n_cand, int cap_cand) {
	const int cx = blockIdx.x * blockDim.x + threadIdx.x + 5;
	const int f = blockIdx.z / kSiftScales, index = blockIdx.z % kSiftScales + 1;
	const bool valid = cx < cols - 5;                  // no early exit: every lane takes part in the shuffles below
	const int c0 = valid ? cx : cols - 6;
	const size_t plane = (size_t)rows * cols;
	const float *d1 = dog + ((size_t)f * (kSiftScales + 2) + index) * plane;
	const float *d0 = d1 - plane, *d2 = d1 + plane;
	// the thread walks down its column keeping (up, centre, down) in registers and gets (left, right) from its warp
	// neighbours: four of the 26 neighbour comparisons cost no extra load and reject most threshold passers before
	// the full test (which repeats them, so the outcome is exactly LocalMaxMin x3 + NotOnEdge)
	const int rbeg = blockIdx.y * kRowsPerBlock + 5, rend = min(rbeg + kRowsPerBlock, rows - 5);
	const int lane = threadIdx.x & 31;
	// (up, centre, down) roll through registers; rows are requested two iterations before they are needed
	float up = __ldg(d1 + (size_t)(rbeg - 1) * cols + c0), cur = __ldg(d1 + (size_t)rbeg * cols + c0);
	float dn = __ldg(d1 + (size_t)min(rbeg + 1, rows - 1) * cols + c0), ahead = __ldg(d1 + (size_t)min(rbeg + 2, rows - 1) * cols + c0), ahead2 = 0.f;
#pragma unroll 1
	for (int r0 = rbeg; r0 < rend; ++r0, up = cur, cur = dn, dn = ahead, ahead = ahead2) {
	ahead2 = __ldg(d1 + (size_t)min(r0 + 3, rows - 1) * cols + c0);
	const float left = __shfl_up_sync(0xffffffffu, cur, 1), right = __shfl_down_sync(0xffffffffu, cur, 1);
	bool go = valid && fabsf(cur) > peak_thresh * 0.8f;
	if (go) {
		if (cur > 0) go = !(up > cur || dn > cur || (lane > 0 && left > cur) || (lane < 31 && c0 + 1 < cols - 5 && right > cur));
		else go = !(cur > up || cur > dn || (lane > 0 && cur > left) || (lane < 31 && c0 + 1 < cols - 5 && cur > right));
	}
	if (!go) continue;
	{ const float fval = cur;
	if (!(local_max_min(fval, d1, cols, r0, c0) && local_max_min(fval, d0, cols, r0, c0) && local_max_min(fval, d2, cols, r0, c0) &&
	      not_on_edge(d1, cols, r0, c0)))
		continue;
	}
	int rowstart = r0, colstart = c0, steps = 5;
	float X[3], fquad;
	for (;;) {
		fquad = fit_quadratic(X, d0, d1, d2, cols, rowstart, colstart);
		int newrow = rowstart, newcol = colstart;
		if (X[1] > 0.6f && rowstart < rows - 3) newrow++;
		if (X[1] < -0.6f && rowstart > 3) newrow--;
		if (X[2] > 0.6f && colstart < cols - 3) newcol++;
		if (X[2] < -0.6f && colstart > 3) newcol--;
		if (steps > 0 && (newrow != rowstart || newcol != colstart)) { rowstart = newrow; colstart = newcol; steps--; continue; }
		break;
	}
	if (fabsf(X[0]) <= 1.5f && fabsf(X[1]) <= 1.5f && fabsf(X[2]) <= 1.5f && fabsf(fquad) >= peak_thresh) {
		int scan_id = ((index - 1) * rows + r0) * cols + c0;
		atomicMin(&claim[(size_t)f * plane + (size_t)rowstart * cols + colstart], scan_id);
		int slot = atomicAdd(n_cand, 1);
		if (slot < cap_cand) {
			SiftCand k;
			k.frame = f; k.oct = oct; k.index = index; k.row = rowstart; k.col = colstart; k.scan_id = scan_id;
			k.X[0] = X[0]; k.X[1] = X[1]; k.X[2] = X[2];
			cand[slot] = k;
		}
	}
	}
}

// ---- orientation: AssignOriHist (:1276-1382), one warp per surviving extremum ---------------------------------

struct SiftOctView { int rows, cols; const float *grad, *ori; const int32_t *claim; };
struct SiftOctViews { SiftOctView o[kSiftMaxOct]; float fscale0; };


// 64-bit fixed-point accumulator (2^-40 units) in shared memory as (lo, hi) 32-bit words: a 64-bit or a float atomicAdd on
// shared memory compiles to a compare-and-swap spin loop (ATOMS.CAST.SPIN), two native 32-bit ATOMS.ADD do not, and — unlike
// a plain load/add/store — they carry no dependency from one sample to the next. The carry out of the low word is
// recovered from the value the first atomic returns. Integer addition commutes: the sum does not depend on the order.
constexpr float kFix = 1099511627776.f;        // 2^40
constexpr float kFixInv = 1.f / 1099511627776.f;
struct Fix64 { unsigned int lo, hi; };
__device__ __forceinline__ void fix_add(Fix64 *a, float v) {
	unsigned long long q = (unsigned long long)__float2ll_rn(v * kFix);
	unsigned int lo = (unsigned int)q, hi = (unsigned int)(q >> 32);
	unsigned int old = atomicAdd(&a->lo, lo);
	hi += (old + lo) < old;
	if (hi) atomicAdd(&a->hi, hi);
}

__global__ void __launch_bounds__(128) k_sift_orient(const SiftCand *__restrict__ cand, const int *__restrict__ n_cand, int cap_cand,
                                                     const __grid_constant__ SiftOctViews views, SiftKp *__restrict__ kp,
                                                     int *__restrict__ kp_count, int max_kp) {
	__shared__ Fix64 s_hist[4][36][32];   // [warp][bin][lane]: one private histogram per lane (bank pair = lane): no conflicts
	__shared__ float s_h[4][2][36];       // smoothing ping-pong
	const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
	const int n = min(*n_cand, cap_cand);
	for (int i = blockIdx.x * 4 + w; i < n; i += gridDim.x * 4) {
	SiftCand k = cand[i];
	const SiftOctView v = views.o[k.oct];
	const int rows = v.rows, cols = v.cols;
	const size_t plane = (size_t)rows * cols;
	if (v.claim[(size_t)k.frame * plane + (size_t)k.row * cols + k.col] != k.scan_id) continue;     // a duplicate (warp-uniform)
	const float *grad = v.grad + ((size_t)k.frame * kSiftScales + (k.index - 1)) * plane;
	const float *orim = v.ori + ((size_t)k.frame * kSiftScales + (k.index - 1)) * plane;
	const float fSize = kSiftInitSigma * powf(2.0f, ((float)k.index + k.X[0]) / (float)kSiftScales);
	const float frowstart = (float)k.row + k.X[1], fcolstart = (float)k.col + k.X[2];
	const int rowstart = (int)(frowstart + 0.5f), colstart = (int)(fcolstart + 0.5f);
	const float fexpmult = -1.0f / (2.0f * 1.5f * 1.5f * fSize * fSize);
	const float fbinmult = 36.0f / (2 * SIFT_PI);
	const float fbinadd = (float)(SIFT_PI + 0.001f) * fbinmult;
	const int windowsize = (int)(fSize * 1.5f * 3.0f);
#pragma unroll
	for (int b = 0; b < 36; ++b) s_hist[w][b][lane] = Fix64{0u, 0u};
	// the window clipped to the rows/columns the reference visits (:1294-1300): 32 consecutive pixels per step
	const int r_lo = max(rowstart - windowsize, 0), r_hi = min(rowstart + windowsize, rows - 3);
	const int c_lo = max(colstart - windowsize, 0), c_hi = min(colstart + windowsize, cols - 3);
	const int bw = c_hi - c_lo + 1;
	if (bw > 0 && r_hi >= r_lo) {
		int rowcur = r_lo + lane / bw, colcur = c_lo + lane % bw;
		const float wlimit = (float)(windowsize * windowsize) + 0.5f;
		constexpr int U = 4;                             // loads of four steps in flight (see k_sift_describe_warp)
		while (rowcur <= r_hi) {
			int rr[U], cc[U];
			float gg[U], oo[U];
#pragma unroll
			for (int u = 0; u < U; ++u) {
				rr[u] = rowcur; cc[u] = colcur;
				if (rowcur <= r_hi) { const size_t px = (size_t)rowcur * cols + colcur; gg[u] = __ldg(grad + px); oo[u] = __ldg(orim + px); }
				colcur += 32;
				while (colcur > c_hi) { colcur -= bw; ++rowcur; }
			}
#pragma unroll
			for (int u = 0; u < U; ++u) {
				if (rr[u] > r_hi) continue;
				const float fdx = gg[u];
				if (fdx > 0) {
					float fdrow = (float)rr[u] - frowstart, fdcol = (float)cc[u] - fcolstart;
					float fradius2 = fdrow * fdrow + fdcol * fdcol;
					if (wlimit > fradius2) {
						float fweight = expf(fradius2 * fexpmult);
						int binindex = (int)(oo[u] * fbinmult + fbinadd);
						if (binindex > 36) binindex = 0;
						if (binindex == 36) binindex = 35;
						if (binindex < 0) binindex = 0;
						fix_add(&s_hist[w][binindex][lane], fdx * fweight);
					}
				}
			}
		}
	}
	__syncwarp();
	for (int b = lane; b < 36; b += 32) {          // bin = exact integer sum of the 32 private copies (rotated: conflict-free)
		unsigned long long sum = 0ull;
		for (int t = 0; t < 32; ++t) { const Fix64 c = s_hist[w][b][(t + lane) & 31]; sum += ((unsigned long long)c.hi << 32) | c.lo; }
		s_h[w][0][b] = __ll2float_rn((long long)sum) * kFixInv;
	}
	// SmoothHistogram x6 (:1329-1330,1395-1407), all bins in parallel: its in-place loop only ever reads ORIGINAL values
	// (fprev/forg are saved originals, phist[i+1] and ffirst are not yet overwritten), so a pass is a circular 3-tap
	// filter new[i] = ((old[i-1] + old[i]) + old[i+1]) * c with c = 0.33333333f, and 0.3333333f for the last bin
	int cur = 0;
	for (int it = 0; it < 6; ++it, cur ^= 1) {
		__syncwarp();
		const float *h = s_h[w][cur];
		float *hn = s_h[w][cur ^ 1];
		hn[lane] = (h[(lane + 35) % 36] + h[lane] + h[lane + 1]) * 0.33333333f;
		if (lane < 4) { const int b = 32 + lane; hn[b] = (h[b - 1] + h[b] + h[(b + 1) % 36]) * (b == 35 ? 0.3333333f : 0.33333333f); }
	}
	__syncwarp();
	const float *hists = s_h[w][cur];
	float fmaxval = fmaxf(0.f, fmaxf(hists[lane], lane < 4 ? hists[32 + lane] : 0.f));      // scalar maximum from 0 (:1352-1356)
#pragma unroll
	for (int o = 16; o > 0; o >>= 1) fmaxval = fmaxf(fmaxval, __shfl_xor_sync(0xffffffffu, fmaxval, o));
	fmaxval *= 0.8f;
	const float foriadd = 0.5f * 2 * SIFT_PI / 36.0f - SIFT_PI, forimult = 2 * SIFT_PI / 36.0f;
	for (int index = lane; index < 36; index += 32) {       // every peak makes a keypoint (:1362-1379); its rank comes from the key
		const int previndex = index == 0 ? 35 : index - 1, nextindex = index == 35 ? 0 : index + 1;
		if (hists[index] <= hists[previndex] || hists[index] <= hists[nextindex] || hists[index] < fmaxval) continue;
		float f0 = hists[previndex], f1 = hists[index], f2 = hists[nextindex];
		if (f1 < 0) { f0 = -f0; f1 = -f1; f2 = -f2; }
		float fpeak = 0.5f * (f0 - f2) / (f0 - 2.0f * f1 + f2);
		float forient = (index + fpeak) * forimult + foriadd;
		int slot = atomicAdd(&kp_count[k.frame], 1);
		if (slot < max_kp) {
			SiftKp q;
			q.frame = k.frame; q.oct = k.oct; q.index = k.index; q.frow = frowstart; q.fcol = fcolstart; q.fsize = fSize; q.ori = forient;
			q.key = ((unsigned long long)k.oct << 40) | ((unsigned long long)(unsigned)k.scan_id << 6) | (unsigned long long)index;
			q.slot = -1;
			kp[(size_t)k.frame * max_kp + slot] = q;
		}
	}
	__syncwarp();
	}
}

// output slot of every keypoint = number of keypoints of its frame with a larger key (reverse creation order)
__global__ void k_sift_rank(SiftKp *__restrict__ kp, const int *__restrict__ kp_count, int max_kp, int32_t *__restrict__ offsets, int n_frames) {
	int f = blockIdx.y, i = blockIdx.x * blockDim.x + threadIdx.x;
	if (offsets && f == 0 && i == 0) {            // compact output: frame f's keypoints start at offsets[f]
		int acc = 0;
		for (int k = 0; k < n_frames; ++k) { offsets[k] = acc; acc += min(kp_count[k], max_kp); }
		offsets[n_frames] = acc;
	}
	int n = min(kp_count[f], max_kp);
	if (i >= n) return;
	SiftKp *base = kp + (size_t)f * max_kp;
	unsigned long long key = base[i].key;
	int rank = 0;
	for (int j = 0; j < n; ++j) rank += base[j].key > key;
	base[i].slot = rank;
}

// ---- descriptor: MakeKeypoint / KeySample / AddSample / PlaceInIndex (:1409-1668), one CTA per keypoint -----------
__global__ void __launch_bounds__(128) k_sift_describe(const SiftKp *__restrict__ kp, const int *__restrict__ kp_count, int max_kp, int n_frames,
                                                       const int32_t *__restrict__ offsets, int match_normalise,
                                                       const __grid_constant__ SiftOctViews views,
                                                       float *__restrict__ out_xy, float *__restrict__ out_so, float *__restrict__ out_desc) {
	__shared__ float s_acc[8][128];        // [orientation bin][thread]: private accumulators, bank = thread % 32
	__shared__ float s_d[128];
	__shared__ float s_scale;
	__shared__ int s_clamped;
	// Gather formulation, no atomics: the 128 threads are 16 groups of 8 lanes, group g owns descriptor cell
	// (ci, cj) = (g / 4, g % 4) and scans the bounding box of that cell's support (the samples whose trilinear footprint
	// touches the cell: |rx - ci| < 1, |cx - cj| < 1) in the image, 8 consecutive pixels per step. Every pixel is put
	// through the reference's own expressions (KeySample / AddSample / PlaceInIndex), so a sample adds to this cell
	// exactly the terms the reference adds to it; only the ORDER of the float additions differs (fixed, so results are
	// deterministic). Same-address shared-memory atomics of the scatter formulation ran at ~1 lane per clock per SM.
	const int g = threadIdx.x >> 3, l8 = threadIdx.x & 7, ci = g >> 2, cj = g & 3;
	for (int item = blockIdx.x; item < n_frames * max_kp; item += gridDim.x) {
	const int f = item / max_kp, i = item % max_kp;
	if (i >= min(kp_count[f], max_kp)) continue;      // empty slot (block-uniform)
	const SiftKp q = kp[(size_t)f * max_kp + i];
	__syncthreads();
	const SiftOctView v = views.o[q.oct];
	const int rows = v.rows, cols = v.cols;
	const size_t plane = (size_t)rows * cols;
	const float *grad = v.grad + ((size_t)f * kSiftScales + (q.index - 1)) * plane;
	const float *orim = v.ori + ((size_t)f * kSiftScales + (q.index - 1)) * plane;
#pragma unroll
	for (int b8 = 0; b8 < 8; ++b8) s_acc[b8][threadIdx.x] = 0.f;
	const float fSize = q.fsize, frowstart = q.frow, fcolstart = q.fcol, keyori = q.ori;
	const int rowstart = (int)(frowstart + 0.5f), colstart = (int)(fcolstart + 0.5f);
	const float sinang = sinf(keyori), cosang = cosf(keyori);
	const float fdrow = frowstart - (float)rowstart, fdcol = fcolstart - (float)colstart;
	const float frealsize = 3.0f * fSize;
	const float firealsize = 1.0f / (3.0f * fSize);
	const int windowsize = (int)(frealsize * SIFT_SQRT2 * 5.0f * 0.5f + 0.5f);
	const float fsr = sinang * firealsize, fcr = cosang * firealsize, fdrr = -fdrow * firealsize, fdcr = -fdcol * firealsize;
	// image-space bounding box of the cell's support: (rpos, cpos) = R(row, col) / (3 fSize) + (fdrr, fdcr) inverted at the
	// cell centre (rpos, cpos) = (ci - 1.5, cj - 1.5), half extent (|cos| + |sin|) * 3 fSize, one pixel of slack for rounding;
	// clipped to the reference's window and to the image
	const float rp = (float)ci - 1.5f - fdrr, cp = (float)cj - 1.5f - fdcr;
	const float rowc = frealsize * (cosang * rp - sinang * cp), colc = frealsize * (sinang * rp + cosang * cp);
	const float half = frealsize * (fabsf(cosang) + fabsf(sinang)) + 1.0f;
	// NOTE (nvcc/ptxas 12.9, sm_100a): max(max(x, -w), -r) was compiled to a three-input VIMNMX3 that dropped the
	// negation of w (lower bounds came out as +windowsize); written as max(x, -min(w, r)) the code is correct.
	const int r_lo = max((int)floorf(rowc - half), -min(windowsize, rowstart)), r_hi = min((int)ceilf(rowc + half), min(windowsize, rows - 1 - rowstart));
	const int c_lo = max((int)floorf(colc - half), -min(windowsize, colstart)), c_hi = min((int)ceilf(colc + half), min(windowsize, cols - 1 - colstart));
	const int bw = c_hi - c_lo + 1;
	if (bw > 0 && r_hi >= r_lo) {
		int row = r_lo + l8 / bw, col = c_lo + l8 % bw;
		for (; row <= r_hi;) {
			float frow = (float)row, fcol = (float)col;     // the reference's running fcol takes exactly these integer values
			float rpos = fsr * fcol + fcr * frow + fdrr;
			float cpos = fcr * fcol - fsr * frow + fdcr;
			float rx = rpos + (2.0f - 0.5f);
			float cx = cpos + (2.0f - 0.5f);
			if (rx > -0.9999f && rx < 3.9999f && cx > -0.9999f && cx < 3.9999f) {
				// PlaceInIndex: which of the (up to) 2 x 2 cells this sample feeds, and with which weights
				int newrow = rx < 0 ? (int)(rx - 1) : (int)rx;
				int newcol = cx < 0 ? (int)(cx - 1) : (int)cx;
				const int a = ci - newrow, b = cj - newcol;
				if ((unsigned)a < 2u && (unsigned)b < 2u) {
					const int r = rowstart + row, c = colstart + col;
					float mag = grad[(size_t)r * cols + c] * expf(-0.125f * (rpos * rpos + cpos * cpos));
					float fo = orim[(size_t)r * cols + c] - keyori;
					while (fo > 2 * SIFT_PI) fo -= 2 * SIFT_PI;
					while (fo < 0) fo += 2 * SIFT_PI;
					float oribin = fo * (8.0f / (2 * (float)SIFT_PI));
					float rfrac = rx - (float)newrow;
					float cfrac = cx - (float)newcol;
					int neworient = oribin < 0 ? (int)(oribin - 1) : (int)oribin;
					float ofrac = oribin - (float)neworient;
					float frowgrad = a == 0 ? mag * (1 - rfrac) : mag * rfrac;
					float fcolgrad = b == 0 ? frowgrad * (1 - cfrac) : frowgrad * cfrac;
					s_acc[neworient & 7][threadIdx.x] += fcolgrad * (1 - ofrac);
					s_acc[(neworient + 1) & 7][threadIdx.x] += fcolgrad * ofrac;
				}
			}
			col += 8;
			while (col > c_hi) { col -= bw; ++row; }
		}
	}
	__syncthreads();
	{   // bin (g, l8) = sum over the group's 8 lanes, in a fixed rotated order (rotation keeps the reads conflict-free)
		float sum = 0.f;
#pragma unroll
		for (int k = 0; k < 8; ++k) sum += s_acc[l8][g * 8 + ((k + l8) & 7)];
		s_d[threadIdx.x] = sum;
	}
	__syncthreads();
	// scalar normalisation branch (:1503-1516): NormalizeVec, clamp at 0.2, NormalizeVec again if anything was clamped
	if (threadIdx.x == 0) {
		float faccum = 0;
		for (int j = 0; j < 128; ++j) faccum += s_d[j] * s_d[j];
		s_scale = 1 / sqrtf(faccum);
		s_clamped = 0;
	}
	__syncthreads();
	float d = s_d[threadIdx.x] * s_scale;
	if (d > 0.2f) { d = 0.2f; s_clamped = 1; }
	s_d[threadIdx.x] = d;
	__syncthreads();
	if (s_clamped) {
		if (threadIdx.x == 0) {
			float faccum = 0;
			for (int j = 0; j < 128; ++j) faccum += s_d[j] * s_d[j];
			s_scale = 1 / sqrtf(faccum);
		}
		__syncthreads();
		d = d * s_scale;
	}
	if (match_normalise) {
		// what the MATCH stage does to every query first (MATCH_ANN_CPU.hpp:54-57,157; the expression of
		// MATCH_CUDA::normalise): sequential sum of squares, inv = (float)(1. / sqrtf(ss)), scale — done here so
		// that the descriptors can go to the matcher without leaving HBM
		__syncthreads();
		s_d[threadIdx.x] = d;
		__syncthreads();
		if (threadIdx.x == 0) {
			float ss = 0;
			for (int j = 0; j < 128; ++j) ss += s_d[j] * s_d[j];
			s_scale = (float)(1. / (double)sqrtf(ss));
		}
		__syncthreads();
		d = d * s_scale;
	}
	size_t o = offsets ? (size_t)offsets[f] + q.slot : (size_t)f * max_kp + q.slot;
	out_desc[o * 128 + threadIdx.x] = d;
	if (threadIdx.x == 0) {
		float fscale = views.fscale0;
		for (int k = 0; k < q.oct; ++k) fscale += fscale;
		out_xy[2 * o] = fscale * fcolstart; out_xy[2 * o + 1] = fscale * frowstart;      // coord2D = (col, row), FEAT_SIFT_CPU.hpp:102-103
		if (out_so) { out_so[2 * o] = fscale * fSize; out_so[2 * o + 1] = keyori; }
	}
	}
}

// The same step, scatter formulation with PRIVATE accumulators (the default): one warp per keypoint, every lane owns a full
// 128-bin copy of the descriptor in shared memory ([bin][lane], bank = lane), walks the reference's window (KeySample's
// double loop, clipped to the image) 32 consecutive pixels per step, evaluates each sample ONCE with the reference's
// expressions and adds its up to 8 terms to its own copy — no atomics, no two lanes ever touch the same word. The 32
// copies are then summed in a fixed rotated order (conflict-free) and re-zeroed in the same pass. Against the gather
// kernel above (every sample evaluated by up to four cell groups plus bounding-box waste) this executes ~6x fewer
// instructions; the price is 16 KB of shared memory per warp.
__global__ void __launch_bounds__(128) k_sift_describe_warp(const SiftKp *__restrict__ kp, int max_kp, int n_frames,
                                                            const int32_t *__restrict__ offs, int compact, int match_normalise,
                                                            const __grid_constant__ SiftOctViews views,
                                                            float *__restrict__ out_xy, float *__restrict__ out_so, float *__restrict__ out_desc) {
	extern __shared__ float sm_desc[];
	const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
	float (*acc)[32] = (float (*)[32])(sm_desc + (size_t)w * 128 * 32);
	float *sd = sm_desc + 4 * 128 * 32 + w * 128;
#pragma unroll 8
	for (int b = 0; b < 128; ++b) acc[b][lane] = 0.f;
	const int total = offs[n_frames];
	for (int idx = blockIdx.x * 4 + w; idx < total; idx += gridDim.x * 4) {
		int f = 0, hi = n_frames;                         // frame of the idx-th keypoint of the batch: offs[f] <= idx < offs[f+1]
		while (hi - f > 1) { const int mid = (f + hi) >> 1; if (offs[mid] <= idx) f = mid; else hi = mid; }
		const SiftKp q = kp[(size_t)f * max_kp + (idx - offs[f])];
		const SiftOctView v = views.o[q.oct];
		const int rows = v.rows, cols = v.cols;
		const size_t plane = (size_t)rows * cols;
		const float *grad = v.grad + ((size_t)f * kSiftScales + (q.index - 1)) * plane;
		const float *orim = v.ori + ((size_t)f * kSiftScales + (q.index - 1)) * plane;
		const float fSize = q.fsize, frowstart = q.frow, fcolstart = q.fcol, keyori = q.ori;
		const int rowstart = (int)(frowstart + 0.5f), colstart = (int)(fcolstart + 0.5f);
		const float sinang = sinf(keyori), cosang = cosf(keyori);
		const float fdrow = frowstart - (float)rowstart, fdcol = fcolstart - (float)colstart;
		const float frealsize = 3.0f * fSize;
		const float firealsize = 1.0f / (3.0f * fSize);
		const int windowsize = (int)(frealsize * SIFT_SQRT2 * 5.0f * 0.5f + 0.5f);
		const float fsr = sinang * firealsize, fcr = cosang * firealsize, fdrr = -fdrow * firealsize, fdcr = -fdcol * firealsize;
		// KeySample's window (:1544-1566) clipped to the image (AddSample's bounds test, :1593-1594)
		const int r_lo = -min(windowsize, rowstart), r_hi = min(windowsize, rows - 1 - rowstart);
		const int c_lo = -min(windowsize, colstart), c_hi = min(windowsize, cols - 1 - colstart);
		const int bw = c_hi - c_lo + 1;
		if (bw > 0 && r_hi >= r_lo) {
			// ncu: a third of all stall samples sat on the first use of the gradient/orientation loads (scattered windows: L1 hit
			// 17 %, ~11 warps per SM). So the loads of EIGHT steps are issued unconditionally up front (the addresses only depend on
			// the walk, not on the acceptance test), then the eight samples are processed: 16 loads in flight per lane.
			constexpr int U = 8;
			int row = r_lo + lane / bw, col = c_lo + lane % bw;
			while (row <= r_hi) {
				int rr[U], cc[U];
				float gg[U], oo[U];
#pragma unroll
				for (int u = 0; u < U; ++u) {
					rr[u] = row; cc[u] = col;
					if (row <= r_hi) {
						const size_t px = (size_t)(rowstart + row) * cols + (colstart + col);
						gg[u] = __ldg(grad + px); oo[u] = __ldg(orim + px);
					}
					col += 32;
					while (col > c_hi) { col -= bw; ++row; }
				}
#pragma unroll
				for (int u = 0; u < U; ++u) {
					if (rr[u] > r_hi) continue;
					const float frow = (float)rr[u], fcol = (float)cc[u];     // the reference's running fcol takes exactly these integer values
					const float rpos = fsr * fcol + fcr * frow + fdrr;
					const float cpos = fcr * fcol - fsr * frow + fdcr;
					const float rx = rpos + (2.0f - 0.5f);
					const float cx = cpos + (2.0f - 0.5f);
					if (!(rx > -0.9999f && rx < 3.9999f && cx > -0.9999f && cx < 3.9999f)) continue;
					const float mag = gg[u] * expf(-0.125f * (rpos * rpos + cpos * cpos));
					float fo = oo[u] - keyori;
					while (fo > 2 * SIFT_PI) fo -= 2 * SIFT_PI;
					while (fo < 0) fo += 2 * SIFT_PI;
					// PlaceInIndex (:1609-1668)
					const float oribin = fo * (8.0f / (2 * (float)SIFT_PI));
					const int newrow = rx < 0 ? (int)(rx - 1) : (int)rx;
					const float rfrac = rx - (float)newrow;
					const int newcol = cx < 0 ? (int)(cx - 1) : (int)cx;
					const float cfrac = cx - (float)newcol;
					const int neworient = oribin < 0 ? (int)(oribin - 1) : (int)oribin;
					const float ofrac = oribin - (float)neworient;
					const int o0 = neworient & 7, o1 = (neworient + 1) & 7;
#pragma unroll
					for (int a = 0; a < 2; ++a) {
						if ((unsigned)(a + newrow) >= 4) continue;
						const float frowgrad = a == 0 ? mag * (1 - rfrac) : mag * rfrac;
#pragma unroll
						for (int b = 0; b < 2; ++b) {
							if ((unsigned)(b + newcol) >= 4) continue;
							const float fcolgrad = b == 0 ? frowgrad * (1 - cfrac) : frowgrad * cfrac;
							const int basebin = 8 * (4 * (a + newrow) + b + newcol);
							acc[basebin + o0][lane] += fcolgrad * (1 - ofrac);
							acc[basebin + o1][lane] += fcolgrad * ofrac;
						}
					}
				}
			}
		}
		__syncwarp();
#pragma unroll
		for (int j = 0; j < 4; ++j) {        // bin = sum of the 32 private copies, fixed rotated order; copies re-zeroed on the way
			const int b = lane + 32 * j;
			float sum = 0.f;
#pragma unroll 8
			for (int t = 0; t < 32; ++t) { const int c = (t + lane) & 31; sum += acc[b][c]; acc[b][c] = 0.f; }
			sd[b] = sum;
		}
		__syncwarp();
		// scalar normalisation branch (:1503-1516): NormalizeVec (sequential sum), clamp at 0.2, NormalizeVec again if clamped
		float scale = 0.f;
		if (lane == 0) { float faccum = 0; for (int j = 0; j < 128; ++j) faccum += sd[j] * sd[j]; scale = 1 / sqrtf(faccum); }
		scale = __shfl_sync(0xffffffffu, scale, 0);
		float d[4];
		bool clamped = false;
#pragma unroll
		for (int j = 0; j < 4; ++j) { d[j] = sd[lane + 32 * j] * scale; if (d[j] > 0.2f) { d[j] = 0.2f; clamped = true; } }
		if (__any_sync(0xffffffffu, clamped)) {
#pragma unroll
			for (int j = 0; j < 4; ++j) sd[lane + 32 * j] = d[j];
			__syncwarp();
			if (lane == 0) { float faccum = 0; for (int j = 0; j < 128; ++j) faccum += sd[j] * sd[j]; scale = 1 / sqrtf(faccum); }
			scale = __shfl_sync(0xffffffffu, scale, 0);
#pragma unroll
			for (int j = 0; j < 4; ++j) d[j] = d[j] * scale;
			__syncwarp();
		}
		if (match_normalise) {               // the MATCH stage's query normalisation (see k_sift_describe)
#pragma unroll
			for (int j = 0; j < 4; ++j) sd[lane + 32 * j] = d[j];
			__syncwarp();
			if (lane == 0) { float ss = 0; for (int j = 0; j < 128; ++j) ss += sd[j] * sd[j]; scale = (float)(1. / (double)sqrtf(ss)); }
			scale = __shfl_sync(0xffffffffu, scale, 0);
#pragma unroll
			for (int j = 0; j < 4; ++j) d[j] = d[j] * scale;
		}
		__syncwarp();
		const size_t o = compact ? (size_t)offs[f] + q.slot : (size_t)f * max_kp + q.slot;
#pragma unroll
		for (int j = 0; j < 4; ++j) out_desc[o * 128 + lane + 32 * j] = d[j];
		if (lane == 0) {
			float fscale = views.fscale0;
			for (int k = 0; k < q.oct; ++k) fscale += fscale;
			out_xy[2 * o] = fscale * fcolstart; out_xy[2 * o + 1] = fscale * frowstart;      // coord2D = (col, row), FEAT_SIFT_CPU.hpp:102-103
			if (out_so) { out_so[2 * o] = fscale * fSize; out_so[2 * o + 1] = keyori; }
		}
	}
}


// ---- host side -------------------------------------------------------------------------------------------------

static SiftState *state(mc_ctx *ctx) {
	if (!ctx->sift_state) ctx->sift_state = new SiftState();
	return (SiftState *)ctx->sift_state;
}

void sift_free(mc_ctx *ctx) {
	SiftState *s = (SiftState *)ctx->sift_state;
	if (!s) return;
	for (cudaEvent_t e : s->ev) if (e) cudaEventDestroy(e);
	DevBuf *bufs[] = { &s->pyr, &s->tmp, &s->tmp2, &s->gray, &s->cand, &s->kp, &s->counters, &s->lut, &s->offs };
	for (DevBuf *b : bufs) cudaFree(b->p);
	delete s;
	ctx->sift_state = nullptr;
}

// Device bytes of sift_plan's buffers for a batch shape
struct SiftBytes {
	size_t pyr, tmp, cand, kp, counters;
	int cap_cand;
};

static SiftBytes sift_bytes(int B, int H, int W, int dbl, int max_kp) {
	const int rows = dbl ? 2 * H - 2 : H, cols = dbl ? 2 * W - 2 : W;
	const int per_px = (kSiftScales + 3) + (kSiftScales + 2) + 2 * kSiftScales + 1;   // gauss, dog, grad, ori, claim
	size_t total = 0;
	for (int r = rows, c = cols, n = 0; r > 12 && c > 12 && n < kSiftMaxOct; r >>= 1, c >>= 1, n++) total += (size_t)r * c * per_px * B;
	SiftBytes b;
	b.pyr = total * sizeof(float) + 256;
	b.tmp = (size_t)rows * cols * B * sizeof(float) + 256;
	b.cap_cand = B * (max_kp > 8192 ? max_kp : 8192) * 2;
	b.cand = (size_t)b.cap_cand * sizeof(SiftCand);
	b.kp = (size_t)B * max_kp * sizeof(SiftKp);
	b.counters = (size_t)(B + 1) * sizeof(int);
	return b;
}

static mc_status sift_reserve(mc_ctx *ctx, SiftState *s, const SiftBytes &b) {
	if (!s->pyr.p || b.pyr > s->pyr.cap) s->B = 0;     // the pyramid moves: the plan's octave pointers go stale, the next sift_plan replans
	MC_TRY(reserve(ctx, s->pyr, b.pyr));
	MC_TRY(reserve(ctx, s->tmp, b.tmp));
	MC_TRY(reserve(ctx, s->tmp2, b.tmp));
	MC_TRY(reserve(ctx, s->cand, b.cand));
	MC_TRY(reserve(ctx, s->kp, b.kp));
	MC_TRY(reserve(ctx, s->counters, b.counters));
	MC_TRY(reserve(ctx, s->offs, b.counters));
	return MC_OK;
}

// (re)plans the scale-space for a batch shape: octave sizes like GetKeypoints' loop (libsiftfast.cpp:344-348)
static mc_status sift_plan(mc_ctx *ctx, SiftState *s, int B, int H, int W, int dbl, int max_kp) {
	if (s->B == B && s->H == H && s->W == W && s->dbl == dbl && s->max_kp == max_kp) return MC_OK;
	const int rows = dbl ? 2 * H - 2 : H, cols = dbl ? 2 * W - 2 : W;
	int n = 0;
	int r = rows, c = cols;
	while (r > 12 && c > 12 && n < kSiftMaxOct) {
		s->oct[n].rows = r; s->oct[n].cols = c; s->oct[n].plane = (size_t)r * c;
		r >>= 1; c >>= 1; n++;
	}
	s->n_oct = n;
	const SiftBytes bytes = sift_bytes(B, H, W, dbl, max_kp);
	MC_TRY(sift_reserve(ctx, s, bytes));
	float *p = (float *)s->pyr.p;
	for (int o = 0; o < n; ++o) {
		SiftOct &q = s->oct[o];
		size_t pl = q.plane * B;
		q.gauss = p; p += pl * (kSiftScales + 3);
		q.dog = p; p += pl * (kSiftScales + 2);
		q.grad = p; p += pl * kSiftScales;
		q.ori = p; p += pl * kSiftScales;
		q.claim = (int32_t *)p; p += pl;
	}
	s->cap_cand = bytes.cap_cand;
	if (!s->lut.p) {
		MC_TRY(reserve(ctx, s->lut, 256 * sizeof(float)));
		float lut[256];
		for (int g = 0; g < 256; ++g) lut[g] = (float)(((float)g) * 1. / 255.);
		MC_CUDA(cudaMemcpyAsync(s->lut.p, lut, sizeof(lut), cudaMemcpyHostToDevice, ctx->stream));
		MC_CUDA(cudaStreamSynchronize(ctx->stream));
	}
	// GetKeypoints (:326-332) and OctaveKeypoints (:414-430)
	float fnewscale = dbl ? 1.0f : 0.5f;
	s->has_init = kSiftInitSigma > fnewscale;
	if (s->has_init) make_kernel(sqrtf(kSiftInitSigma * kSiftInitSigma - fnewscale * fnewscale), s->k_init);
	float fwidth = powf(2.0f, 1.0f / (float)kSiftScales);
	float fincsigma = sqrtf(fwidth * fwidth - 1.0f);
	float sigma = kSiftInitSigma;
	for (int i = 1; i < kSiftScales + 3; ++i) { make_kernel(fincsigma * sigma, s->k_oct[i - 1]); sigma *= fwidth; }
	s->B = B; s->H = H; s->W = W; s->dbl = dbl; s->max_kp = max_kp;
	return MC_OK;
}

// dst = GaussianBlur(src) (+ dog = src - dst): the fused kernel for the tap counts the reference's sigmas produce
// (11, 13, 17, 21, 25), the two-pass kernels through `tmp` for anything else. src and dst must be different buffers.
static mc_status blur(mc_ctx *ctx, SiftState *s, const float *src, size_t fs_src, float *dst, size_t fs_dst, float *dog, size_t fs_dog,
                      int rows, int cols, size_t plane, int B, const GaussK &gk) {
	if (!s->two_pass) {
		switch (gk.ksize) {
		case 11: return launch_blur_t<11>(ctx, s->smem_configured, src, fs_src, dst, fs_dst, dog, fs_dog, rows, cols, B, gk);
		case 13: return launch_blur_t<13>(ctx, s->smem_configured, src, fs_src, dst, fs_dst, dog, fs_dog, rows, cols, B, gk);
		case 17: return launch_blur_t<17>(ctx, s->smem_configured, src, fs_src, dst, fs_dst, dog, fs_dog, rows, cols, B, gk);
		case 21: return launch_blur_t<21>(ctx, s->smem_configured, src, fs_src, dst, fs_dst, dog, fs_dog, rows, cols, B, gk);
		case 25: return launch_blur_t<25>(ctx, s->smem_configured, src, fs_src, dst, fs_dst, dog, fs_dog, rows, cols, B, gk);
		default: break;
		}
	}
	const int TB = 128;
	dim3 g((cols + TB - 1) / TB, rows, B);
	k_sift_blur_h<<<g, TB, 0, ctx->stream>>>(src, fs_src, (float *)s->tmp2.p, plane, rows, cols, gk);
	MC_LAUNCH_CHECK();
	k_sift_blur_v<<<g, TB, 0, ctx->stream>>>((const float *)s->tmp2.p, plane, dst, fs_dst, src, fs_src, dog, fs_dog, rows, cols, gk);
	MC_LAUNCH_CHECK();
	return MC_OK;
}

static inline dim3 grid2(int cols, int rows, int z, int bx) { return dim3((cols + bx - 1) / bx, rows, z); }

mc_status sift_extract_device(mc_ctx *ctx, const uint8_t *d_gray, int B, int H, int W, int dbl, int max_kp,
                              float *d_xy, float *d_so, float *d_desc, int32_t *d_counts, int32_t *d_offsets, int match_normalise) {
	if (B < 1 || H < 8 || W < 8 || max_kp < 1 || (size_t)B * 3 * kSiftScales > 65535) { ctx->err = "mc_sift: bad batch shape"; return MC_ERR_ARG; }
	SiftState *s = state(ctx);
	MC_TRY(sift_plan(ctx, s, B, H, W, dbl ? 1 : 0, max_kp));
	cudaStream_t st = ctx->stream;
	const int TB = 128;
	const float peak_thresh = 0.04f / (float)kSiftScales;
	int *n_cand = (int *)s->counters.p, *kp_count = n_cand + 1;
	MC_CUDA(cudaMemsetAsync(s->counters.p, 0, (size_t)(B + 1) * sizeof(int), st));
	for (int o = 0; o < s->n_oct; ++o) MC_CUDA(cudaMemsetAsync(s->oct[o].claim, 0x7f, s->oct[o].plane * B * sizeof(int32_t), st));

	SiftOct &o0 = s->oct[0];
	const size_t gstride0 = o0.plane * (kSiftScales + 3);
	if (s->n_oct > 0) {
		float *base = s->has_init ? (float *)s->tmp.p : o0.gauss;
		size_t bstride = s->has_init ? o0.plane : gstride0;
		k_sift_base<<<grid2(o0.cols, o0.rows, B, TB), TB, 0, st>>>(d_gray, (const float *)s->lut.p, H, W, dbl ? 1 : 0, base, o0.rows, o0.cols);
		MC_LAUNCH_CHECK();
		if (s->has_init)       // the reference blurs in place; here: base image in `tmp` -> gauss[0]
			MC_TRY(blur(ctx, s, base, bstride, o0.gauss, gstride0, nullptr, 0, o0.rows, o0.cols, o0.plane, B, s->k_init));
	}
	SiftOctViews views;
	memset(&views, 0, sizeof(views));
	views.fscale0 = dbl ? 0.5f : 1.0f;
	for (int o = 0; o < s->n_oct; ++o) {
		SiftOct &q = s->oct[o];
		const size_t gstride = q.plane * (kSiftScales + 3), dstride = q.plane * (kSiftScales + 2);
		const bool prof = ctx->profile && o == 0;      // bench.py's roofline: the dominant kernel timed on its own stream
		for (int i = 1; i < kSiftScales + 3; ++i) {    // gauss[i] = blur(gauss[i-1]); dog[i-1] = gauss[i-1] - gauss[i]
			if (prof) {
				if (!s->ev[2 * i - 2]) { MC_CUDA(cudaEventCreate(&s->ev[2 * i - 2])); MC_CUDA(cudaEventCreate(&s->ev[2 * i - 1])); }
				MC_CUDA(cudaEventRecord(s->ev[2 * i - 2], st));
			}
			MC_TRY(blur(ctx, s, q.gauss + (size_t)(i - 1) * q.plane, gstride, q.gauss + (size_t)i * q.plane, gstride,
			            q.dog + (size_t)(i - 1) * q.plane, dstride, q.rows, q.cols, q.plane, B, s->k_oct[i - 1]));
			if (prof) MC_CUDA(cudaEventRecord(s->ev[2 * i - 1], st));
		}
		if (prof) { s->ev_valid = true; s->ev_bytes = 3.0 * sizeof(float) * (double)q.plane * B * (kSiftScales + 2); }
		k_sift_gradori<<<grid2(q.cols, (q.rows + kRowsPerBlock - 1) / kRowsPerBlock, B * kSiftScales, TB), TB, 0, st>>>(q.gauss, q.grad, q.ori, q.rows, q.cols);
		MC_LAUNCH_CHECK();
		if (q.rows > 10 && q.cols > 10) {
			k_sift_detect<<<grid2(q.cols - 10, (q.rows - 10 + kRowsPerBlock - 1) / kRowsPerBlock, B * kSiftScales, TB), TB, 0, st>>>(q.dog, q.claim, q.rows, q.cols, o, peak_thresh,
			                                                                                 (SiftCand *)s->cand.p, n_cand, s->cap_cand);
			MC_LAUNCH_CHECK();
		}
		if (o + 1 < s->n_oct) {
			SiftOct &nx = s->oct[o + 1];
			k_sift_half<<<grid2(nx.cols, nx.rows, B, TB), TB, 0, st>>>(q.gauss + (size_t)kSiftScales * q.plane, gstride, q.cols, nx.gauss,
			                                                           nx.plane * (kSiftScales + 3), nx.rows, nx.cols);
			MC_LAUNCH_CHECK();
		}
		views.o[o].rows = q.rows; views.o[o].cols = q.cols; views.o[o].grad = q.grad; views.o[o].ori = q.ori; views.o[o].claim = q.claim;
	}
	// the numbers of extrema / keypoints are only known on the device: persistent grids loop over what is there
	const int pgrid = ctx->num_sms * 8;
	k_sift_orient<<<pgrid, 128, 0, st>>>((const SiftCand *)s->cand.p, n_cand, s->cap_cand, views, (SiftKp *)s->kp.p, kp_count, max_kp);
	MC_LAUNCH_CHECK();
	int32_t *offs = d_offsets ? d_offsets : (int32_t *)s->offs.p;     // keypoints of frame f = entries [offs[f], offs[f+1]) of the batch
	k_sift_rank<<<dim3((max_kp + 127) / 128, B), 128, 0, st>>>((SiftKp *)s->kp.p, kp_count, max_kp, offs, B);
	MC_LAUNCH_CHECK();
	if (s->gather) {
		k_sift_describe<<<pgrid, 128, 0, st>>>((const SiftKp *)s->kp.p, kp_count, max_kp, B, d_offsets, match_normalise, views, d_xy, d_so, d_desc);
	} else {
		constexpr size_t smem = (4 * 128 * 32 + 4 * 128) * sizeof(float);
		if (!(s->smem_configured & 1u)) { MC_CUDA(cudaFuncSetAttribute(k_sift_describe_warp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); s->smem_configured |= 1u; }
		k_sift_describe_warp<<<ctx->num_sms * 3, 128, smem, st>>>((const SiftKp *)s->kp.p, max_kp, B, offs, d_offsets ? 1 : 0, match_normalise, views,
		                                                         d_xy, d_so, d_desc);
	}
	MC_LAUNCH_CHECK();
	MC_CUDA(cudaMemcpyAsync(d_counts, kp_count, (size_t)B * sizeof(int), cudaMemcpyDeviceToDevice, st));
	return MC_OK;
}

} // namespace mc

using namespace mc;

extern "C" mc_status mc_sift_extract_dev(mc_ctx *ctx, const uint8_t *gray_dev, int n_images, int height, int width, int double_size,
                                         int max_keypoints, float *xy_dev, float *scale_ori_dev, float *desc_dev, int32_t *counts_dev) {
	if (!ctx) return MC_ERR_ARG;
	if (!gray_dev || !xy_dev || !desc_dev || !counts_dev) { ctx->err = "mc_sift_extract_dev: null pointer"; return MC_ERR_ARG; }
	MC_CUDA(cudaSetDevice(ctx->device));
	return sift_extract_device(ctx, gray_dev, n_images, height, width, double_size, max_keypoints, xy_dev, scale_ori_dev, desc_dev, counts_dev, nullptr, 0);
}

extern "C" mc_status mc_sift_extract(mc_ctx *ctx, const uint8_t *gray, int n_images, int height, int width, int double_size,
                                     int max_keypoints, int32_t *counts, float *xy, float *scale_ori, float *desc) {
	if (!ctx) return MC_ERR_ARG;
	if (!gray || !counts || !xy || !desc) { ctx->err = "mc_sift_extract: null pointer"; return MC_ERR_ARG; }
	if (n_images < 1 || max_keypoints < 1) { ctx->err = "mc_sift_extract: bad sizes"; return MC_ERR_ARG; }
	MC_CUDA(cudaSetDevice(ctx->device));
	SiftState *s = state(ctx);
	const size_t npx = (size_t)n_images * height * width, nk = (size_t)n_images * max_keypoints;
	MC_TRY(reserve(ctx, s->gray, npx + nk * (2 + 2 + 128) * sizeof(float) + (size_t)n_images * sizeof(int32_t) + 1024));
	uint8_t *d_gray = (uint8_t *)s->gray.p;
	float *d_xy = (float *)(d_gray + ((npx + 255) & ~(size_t)255));
	float *d_so = d_xy + nk * 2, *d_desc = d_so + nk * 2;
	int32_t *d_counts = (int32_t *)(d_desc + nk * 128);
	MC_CUDA(cudaMemcpyAsync(d_gray, gray, npx, cudaMemcpyHostToDevice, ctx->stream));
	MC_TRY(sift_extract_device(ctx, d_gray, n_images, height, width, double_size, max_keypoints, d_xy, d_so, d_desc, d_counts, nullptr, 0));
	MC_CUDA(cudaMemcpyAsync(counts, d_counts, (size_t)n_images * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
	int n_extrema = 0;
	MC_CUDA(cudaMemcpyAsync(&n_extrema, s->counters.p, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
	MC_CUDA(cudaStreamSynchronize(ctx->stream));
	if (n_extrema > s->cap_cand) { ctx->err = "mc_sift_extract: more scale-space extrema than the candidate list holds; raise max_keypoints"; return MC_ERR_CAPACITY; }
	mc_status rc = MC_OK;
	for (int f = 0; f < n_images; ++f) {
		int n = counts[f];
		if (n > max_keypoints) { n = max_keypoints; ctx->err = "mc_sift_extract: more keypoints than max_keypoints (counts[] holds the number found)"; rc = MC_ERR_CAPACITY; }
		if (!n) continue;
		size_t o = (size_t)f * max_keypoints;
		MC_CUDA(cudaMemcpyAsync(xy + o * 2, d_xy + o * 2, (size_t)n * 2 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
		if (scale_ori) MC_CUDA(cudaMemcpyAsync(scale_ori + o * 2, d_so + o * 2, (size_t)n * 2 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
		MC_CUDA(cudaMemcpyAsync(desc + o * 128, d_desc + o * 128, (size_t)n * 128 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
	}
	MC_CUDA(cudaStreamSynchronize(ctx->stream));
	return rc;
}

namespace mc {

// Rig frames: image b of the batch belongs to camera b % n_cameras, so its keypoints, entries [offs[b], offs[b+1]) of the compacted
// list, get imageIdx = that camera. One CTA per image.
__global__ void k_rig_image_index(const int32_t *__restrict__ offs, int n_cameras, int32_t *__restrict__ q_image) {
	const int b = blockIdx.x, c = b % n_cameras, hi = offs[b + 1];
	for (int i = offs[b] + threadIdx.x; i < hi; i += blockDim.x) q_image[i] = c;
}

// Rigs with cameras of several sizes: each size group ran its own SIFT batch, images [frame][camera-in-group], into its own compacted
// list. Camera c's image of frame f is image f * k[c] of its group's batch: its count found is counts[c][f * k[c]] and its keypoints
// are entries [offs[c][f * k[c]], offs[c][f * k[c] + 1]) of xy[c] / desc[c] (the pointers already advanced to the camera's slot).
struct RigMerge {
	const int32_t *counts[kUndistortCameras], *offs[kUndistortCameras];
	const float *xy[kUndistortCameras], *desc[kUndistortCameras];
	int k[kUndistortCameras];
};

constexpr int kMergeScanThreads = 1024, kMergeThreads = 256, kMergeSplit = 8;

// One CTA: frame-major image i = f * n_cameras + c gets counts[i] = the count found and offs[i] = where its keypoints go in the merged
// list, so offs[f * n_cameras] is frame f's query offset and offs[n_img] the total. The destinations use the numbers SIFT wrote
// (offset differences), which a count found above max_keypoints exceeds.
__global__ void __launch_bounds__(kMergeScanThreads) k_rig_merge_scan(const __grid_constant__ RigMerge m, int n_cameras, int n_img,
                                                                      int32_t *__restrict__ counts, int32_t *__restrict__ offs) {
	__shared__ int warp_sum[kMergeScanThreads / 32];
	const int per = (n_img + kMergeScanThreads - 1) / kMergeScanThreads;
	const int lo = min((int)threadIdx.x * per, n_img), hi = min(lo + per, n_img);
	int sum = 0;
	for (int i = lo; i < hi; ++i) {
		const int c = i % n_cameras;
		const int32_t *o = m.offs[c] + (i / n_cameras) * m.k[c];
		sum += o[1] - o[0];
	}
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	int incl = sum;
#pragma unroll
	for (int d = 1; d < 32; d <<= 1) {
		const int v = __shfl_up_sync(0xffffffffu, incl, d);
		if (lane >= d) incl += v;
	}
	if (lane == 31) warp_sum[warp] = incl;
	__syncthreads();
	if (warp == 0) {
		int w = warp_sum[lane];
#pragma unroll
		for (int d = 1; d < 32; d <<= 1) {
			const int v = __shfl_up_sync(0xffffffffu, w, d);
			if (lane >= d) w += v;
		}
		warp_sum[lane] = w;
	}
	__syncthreads();
	int run = incl - sum + (warp ? warp_sum[warp - 1] : 0);
	for (int i = lo; i < hi; ++i) {
		const int c = i % n_cameras, b = (i / n_cameras) * m.k[c];
		const int32_t *o = m.offs[c] + b;
		counts[i] = m.counts[c][b];
		offs[i] = run;
		run += o[1] - o[0];
	}
	if (threadIdx.x == kMergeScanThreads - 1) offs[n_img] = run;
}

// grid (n_img, kMergeSplit): frame-major image i's descriptors (128 floats, as float4) and xy move from its group's list to offs[i] of
// the merged list, and its keypoints get imageIdx = camera.
__global__ void __launch_bounds__(kMergeThreads) k_rig_merge_interleave(const __grid_constant__ RigMerge m, int n_cameras,
                                                                        const int32_t *__restrict__ offs, float *__restrict__ xy,
                                                                        float *__restrict__ desc, int32_t *__restrict__ q_image) {
	const int i = blockIdx.x, c = i % n_cameras;
	const int32_t *so = m.offs[c] + (i / n_cameras) * m.k[c];
	const int src = so[0], dst = offs[i], n = offs[i + 1] - dst;
	const int t0 = blockIdx.y * kMergeThreads + threadIdx.x, step = gridDim.y * kMergeThreads;
	const float4 *s4 = (const float4 *)(m.desc[c] + (size_t)src * 128);
	float4 *d4 = (float4 *)(desc + (size_t)dst * 128);
#pragma unroll 4
	for (int t = t0; t < n * 32; t += step) d4[t] = __ldg(s4 + t);
	const float2 *s2 = (const float2 *)(m.xy[c] + (size_t)src * 2);
	float2 *d2 = (float2 *)(xy + (size_t)dst * 2);
	for (int t = t0; t < n; t += step) {
		d2[t] = __ldg(s2 + t);
		q_image[dst + t] = c;
	}
}

// Checks of the rig entries before anything is read or queued
static mc_status rig_check(mc_ctx *ctx, const char *who, int n_frames, int n_cameras) {
	const std::string name(who);
	if (n_cameras < 1 || n_cameras > kUndistortCameras) {
		ctx->err = name + ": n_cameras must be in 1.." + std::to_string(kUndistortCameras); return MC_ERR_ARG;
	}
	if ((int64_t)n_frames * n_cameras > 65535) { ctx->err = name + ": more than 65535 images in a batch"; return MC_ERR_ARG; }
	if (ctx->n_images < n_cameras) {
		ctx->err = name + ": " + std::to_string(n_cameras) + " cameras in the rig, " + std::to_string(ctx->n_images) + " set with mc_set_cameras";
		return MC_ERR_STATE;
	}
	return MC_OK;
}

// Cameras of one image size, in camera order. Their images form one SIFT batch laid out [frame][camera-in-group].
struct RigGroup {
	int H = 0, W = 0, k = 0;
	int cams[kUndistortCameras];
	bool table = false;               // a camera of the group has an undistortion table: one remap launch
	bool packed = false;              // the cameras' images already lie in the batch layout, in one buffer
	size_t n = 0, npx = 0;            // images, bytes of the batch
	uint8_t *d_gray = nullptr, *d_undist = nullptr;
	float *d_xy = nullptr, *d_desc = nullptr;
	int32_t *d_counts = nullptr;      // counts[n], then offsets[n + 1]
};

/* FEAT for a batch of n_frames frames of n_cameras images each, camera c's images as cams[c] describes them, in host (dev = false)
 * or device memory: UNDISTORTED_IMAGE and SIFT per size group, then the frame-major query arrays (SURVEY.md 8f row 3). Cameras of one
 * size run as one SIFT batch. The describe kernel writes the descriptors compacted (image-major) and already normalised the way MATCH
 * normalises its queries. With one size group, a frame's images follow each other in camera order already; with several, two merge
 * kernels interleave the groups' lists into that order. d_desc / d_xy / d_qimg are the caller's arrays of n_frames x n_cameras x
 * max_keypoints rows, or NULL for arrays carved from the context's SIFT scratch (returned through the references). Only the per-image
 * keypoint counts and offsets (4 B each) come back to the host, in the call's one synchronisation: frame_offsets[n_frames + 1] is the
 * frame partition of the query list, host-side state of the batch driver. Every check is made before any copy or launch. */
static mc_status extract_rig(mc_ctx *ctx, const char *who, const mc_rig_camera *cams, int n_cameras, int n_frames, bool dev, int double_size,
                             int max_keypoints, float *&d_desc, float *&d_xy, int32_t *&d_qimg, int32_t *frame_offsets, int32_t *n_features,
                             float *feat_ms) {
	const std::string name(who);
	if (!cams || n_frames < 1 || max_keypoints < 1) { ctx->err = name + ": bad argument"; return MC_ERR_ARG; }
	int H[kUndistortCameras], W[kUndistortCameras];
	std::vector<RigGroup> groups;
	for (int c = 0; c < n_cameras; ++c) {
		const mc_rig_camera &cam = cams[c];
		if (!cam.gray) { ctx->err = name + ": camera " + std::to_string(c) + " has no images"; return MC_ERR_ARG; }
		if (cam.height < 8 || cam.height > 32767 || cam.width < 8 || cam.width > 32767) {
			ctx->err = name + ": camera " + std::to_string(c) + "'s images are " + std::to_string(cam.width) + "x" + std::to_string(cam.height) +
			           "; sizes must be in 8..32767";
			return MC_ERR_ARG;
		}
		if (cam.frame_stride < (int64_t)cam.height * cam.width) {
			ctx->err = name + ": camera " + std::to_string(c) + "'s frame_stride is below height x width"; return MC_ERR_ARG;
		}
		H[c] = cam.height; W[c] = cam.width;
		size_t g = 0;
		while (g < groups.size() && (groups[g].H != H[c] || groups[g].W != W[c])) ++g;
		if (g == groups.size()) { groups.emplace_back(); groups[g].H = H[c]; groups[g].W = W[c]; }
		groups[g].cams[groups[g].k++] = c;
	}
	for (const RigGroup &g : groups)
		if ((int64_t)n_frames * g.k * 3 * kSiftScales > 65535) {
			ctx->err = name + ": more than " + std::to_string(65535 / (3 * kSiftScales)) + " images of one size in a batch"; return MC_ERR_ARG;
		}
	// UNDISTORTED_IMAGE before SIFT for the cameras with a table (mc_set_undistortion); their sizes are checked before anything is queued
	bool has_table[kUndistortCameras];
	MC_TRY(undistort_check_rig(ctx, who, n_cameras, H, W, has_table));
	MC_CUDA(cudaSetDevice(ctx->device));
	SiftState *s = state(ctx);
	const bool merge = groups.size() > 1;
	SiftBytes need = {};                  // every group's batch fits the scale-space buffers: nothing is reallocated between groups
	for (RigGroup &g : groups) {
		const size_t plane = (size_t)g.H * g.W;
		g.n = (size_t)n_frames * g.k;
		g.npx = g.n * plane;
		const mc_rig_camera &c0 = cams[g.cams[0]];
		g.packed = c0.frame_stride == (int64_t)(g.k * plane);
		for (int j = 0; j < g.k; ++j) {
			g.table |= has_table[g.cams[j]];
			g.packed &= cams[g.cams[j]].gray == c0.gray + j * plane && cams[g.cams[j]].frame_stride == c0.frame_stride;
		}
		const SiftBytes b = sift_bytes((int)g.n, g.H, g.W, double_size ? 1 : 0, max_keypoints);
		need.pyr = std::max(need.pyr, b.pyr); need.tmp = std::max(need.tmp, b.tmp); need.cand = std::max(need.cand, b.cand);
		need.kp = std::max(need.kp, b.kp); need.counters = std::max(need.counters, b.counters);
	}
	MC_TRY(sift_reserve(ctx, s, need));
	const int n_img = n_frames * n_cameras;
	const size_t nk = (size_t)n_img * max_keypoints;
	const bool own = !d_desc;                           // the query arrays live in the context's scratch
	int32_t *d_counts = nullptr;
	MC_TRY(carve_scratch(ctx, s->gray, [&](Carve &c) {
		for (RigGroup &g : groups) {
			c.take(g.d_gray, dev && g.packed ? 0 : g.npx);     // device images in the batch layout are read where they are
			c.take(g.d_undist, g.table ? g.npx : 0);
		}
		if (own) {
			c.take(d_xy, nk * 2);
			c.take(d_desc, nk * 128);
			c.take(d_qimg, nk);
		}
		c.take(d_counts, (size_t)2 * n_img + 2);          // counts[n_img], then offsets[n_img + 1], frame-major
		for (RigGroup &g : groups) {                      // with several groups each has its own list, merged into the arrays above
			const size_t gk = merge ? g.n * max_keypoints : 0;
			c.take(g.d_xy, gk * 2);
			c.take(g.d_desc, gk * 128);
			c.take(g.d_counts, merge ? 2 * g.n + 2 : 0);
		}
	}));
	int32_t *d_offsets = d_counts + n_img;
	if (!merge) { groups[0].d_xy = d_xy; groups[0].d_desc = d_desc; groups[0].d_counts = d_counts; }
	MC_TRY(pinned(ctx, (size_t)(2 * n_img + 2) * sizeof(int32_t)));
	cudaEvent_t ev[2];
	if (feat_ms) { MC_CUDA(cudaEventCreate(&ev[0])); MC_CUDA(cudaEventCreate(&ev[1])); MC_CUDA(cudaEventRecord(ev[0], ctx->stream)); }
	const cudaMemcpyKind kind = dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
	for (RigGroup &g : groups) {                          // each group's batch: one copy when it is packed, else one per camera
		const size_t plane = (size_t)g.H * g.W;
		if (dev && g.packed) continue;
		if (g.packed) { MC_CUDA(cudaMemcpyAsync(g.d_gray, cams[g.cams[0]].gray, g.npx, kind, ctx->stream)); continue; }
		for (int j = 0; j < g.k; ++j) {
			const mc_rig_camera &cam = cams[g.cams[j]];
			MC_CUDA(cudaMemcpy2DAsync(g.d_gray + j * plane, g.k * plane, cam.gray, (size_t)cam.frame_stride, plane, n_frames, kind, ctx->stream));
		}
	}
	if (n_cameras == 1) MC_CUDA(cudaMemsetAsync(d_qimg, 0, nk * sizeof(int32_t), ctx->stream));     // one camera per frame: imageIdx = 0
	for (RigGroup &g : groups) {
		const uint8_t *d_feat_in = dev && g.packed ? cams[g.cams[0]].gray : g.d_gray;
		if (g.table) {
			MC_TRY(undistort_rig_device(ctx, g.cams, g.k, d_feat_in, (int)g.n, g.H, g.W, g.d_undist));
			d_feat_in = g.d_undist;
		}
		MC_TRY(sift_extract_device(ctx, d_feat_in, (int)g.n, g.H, g.W, double_size, max_keypoints, g.d_xy, nullptr, g.d_desc, g.d_counts,
		                           g.d_counts + g.n, 1));
	}
	if (merge) {
		RigMerge m = {};
		for (const RigGroup &g : groups)
			for (int j = 0; j < g.k; ++j) {
				const int c = g.cams[j];
				m.counts[c] = g.d_counts + j;
				m.offs[c] = g.d_counts + g.n + j;
				m.xy[c] = g.d_xy;
				m.desc[c] = g.d_desc;
				m.k[c] = g.k;
			}
		k_rig_merge_scan<<<1, kMergeScanThreads, 0, ctx->stream>>>(m, n_cameras, n_img, d_counts, d_offsets);
		MC_LAUNCH_CHECK();
		k_rig_merge_interleave<<<dim3(n_img, kMergeSplit), kMergeThreads, 0, ctx->stream>>>(m, n_cameras, d_offsets, d_xy, d_desc, d_qimg);
		MC_LAUNCH_CHECK();
	} else if (n_cameras > 1) {
		k_rig_image_index<<<n_img, 128, 0, ctx->stream>>>(d_offsets, n_cameras, d_qimg);
		MC_LAUNCH_CHECK();
	}
	int32_t *h = (int32_t *)ctx->h_pinned;
	MC_CUDA(cudaMemcpyAsync(h, d_counts, (size_t)(2 * n_img + 1) * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
	if (feat_ms) MC_CUDA(cudaEventRecord(ev[1], ctx->stream));
	MC_CUDA(cudaStreamSynchronize(ctx->stream));
	if (feat_ms) { cudaEventElapsedTime(feat_ms, ev[0], ev[1]); cudaEventDestroy(ev[0]); cudaEventDestroy(ev[1]); }
	for (int f = 0; f <= n_frames; ++f) frame_offsets[f] = h[n_img + f * n_cameras];     // frame f = images [f * n_cameras, (f + 1) * n_cameras)
	bool overflow = false;
	for (int i = 0; i < n_img; ++i) {
		if (n_features) n_features[i] = h[i];
		overflow |= h[i] > max_keypoints;
	}
	if (overflow) { ctx->err = name + ": more keypoints than max_keypoints in a frame (n_features[] holds the numbers found)"; return MC_ERR_CAPACITY; }
	return MC_OK;
}

/* Images in, objects out (SURVEY.md 8f rows 1+3 chained): extract_rig into the context's scratch, then MATCH -> CLUSTER -> POSE ->
 * FILTER -> POSE2 -> FILTER2. The descriptors never leave HBM. */
static mc_status process_images(mc_ctx *ctx, const char *who, const mc_rig_camera *cams, int n_cameras, int n_frames, bool dev,
                                int double_size, int max_keypoints, const mc_pipeline_params *params, int max_objects, int32_t *n_objects,
                                int32_t *obj_model, float *obj_pose, float *obj_score, int32_t *n_features, int32_t *frame_info, float *stage_ms) {
	const std::string name(who);
	if (!cams || !params || !n_objects || !obj_model || !obj_pose || !obj_score || n_frames < 1 || max_keypoints < 1 || max_objects < 1) {
		ctx->err = name + ": bad argument"; return MC_ERR_ARG;
	}
	if (!ctx->d_db) { ctx->err = name + ": no database uploaded"; return MC_ERR_STATE; }
	if (ctx->D != 128) { ctx->err = name + ": the database does not hold 128-d descriptors"; return MC_ERR_STATE; }
	float *d_desc = nullptr, *d_xy = nullptr;
	int32_t *d_qimg = nullptr;
	std::vector<int32_t> offsets(n_frames + 1);
	MC_TRY(extract_rig(ctx, who, cams, n_cameras, n_frames, dev, double_size, max_keypoints, d_desc, d_xy, d_qimg, offsets.data(), n_features,
	                   stage_ms));
	return process_frames_host(ctx, d_desc, d_xy, d_qimg, offsets.data(), n_frames, params, max_objects, n_objects, obj_model, obj_pose, obj_score,
	                           frame_info, stage_ms ? stage_ms + 1 : nullptr);
}

} // namespace mc

extern "C" mc_status mc_process_images(mc_ctx *ctx, const uint8_t *gray, int n_frames, int height, int width, int double_size, int max_keypoints,
                                       const mc_pipeline_params *params, int max_objects, int32_t *n_objects, int32_t *obj_model, float *obj_pose,
                                       float *obj_score, int32_t *n_features, int32_t *frame_info, float *stage_ms) {
	if (!ctx) return MC_ERR_ARG;
	if (!gray) { ctx->err = "mc_process_images: bad argument"; return MC_ERR_ARG; }
	const mc_rig_camera cam = { gray, (int64_t)height * width, height, width };
	return process_images(ctx, "mc_process_images", &cam, 1, n_frames, false, double_size, max_keypoints, params, max_objects, n_objects,
	                      obj_model, obj_pose, obj_score, n_features, frame_info, stage_ms);
}

extern "C" mc_status mc_process_rig_images(mc_ctx *ctx, const uint8_t *gray, int n_frames, int n_cameras, int height, int width, int double_size,
                                           int max_keypoints, const mc_pipeline_params *params, int max_objects, int32_t *n_objects,
                                           int32_t *obj_model, float *obj_pose, float *obj_score, int32_t *n_features, int32_t *frame_info,
                                           float *stage_ms) {
	if (!ctx) return MC_ERR_ARG;
	MC_TRY(rig_check(ctx, "mc_process_rig_images", n_frames, n_cameras));
	if (!gray) { ctx->err = "mc_process_rig_images: bad argument"; return MC_ERR_ARG; }
	mc_rig_camera cams[kUndistortCameras];          // camera c of one [n_frames][n_cameras][height][width] buffer
	const int64_t plane = (int64_t)height * width;
	for (int c = 0; c < n_cameras; ++c) cams[c] = { gray + c * plane, n_cameras * plane, height, width };
	return process_images(ctx, "mc_process_rig_images", cams, n_cameras, n_frames, false, double_size, max_keypoints, params, max_objects,
	                      n_objects, obj_model, obj_pose, obj_score, n_features, frame_info, stage_ms);
}

extern "C" mc_status mc_process_rig_cameras(mc_ctx *ctx, const mc_rig_camera *cameras, int n_cameras, int n_frames, int double_size,
                                            int max_keypoints, const mc_pipeline_params *params, int max_objects, int32_t *n_objects,
                                            int32_t *obj_model, float *obj_pose, float *obj_score, int32_t *n_features, int32_t *frame_info,
                                            float *stage_ms) {
	if (!ctx) return MC_ERR_ARG;
	MC_TRY(rig_check(ctx, "mc_process_rig_cameras", n_frames, n_cameras));
	return process_images(ctx, "mc_process_rig_cameras", cameras, n_cameras, n_frames, false, double_size, max_keypoints, params, max_objects,
	                      n_objects, obj_model, obj_pose, obj_score, n_features, frame_info, stage_ms);
}

extern "C" mc_status mc_process_rig_cameras_dev(mc_ctx *ctx, const mc_rig_camera *cameras, int n_cameras, int n_frames, int double_size,
                                                int max_keypoints, const mc_pipeline_params *params, int max_objects, int32_t *n_objects,
                                                int32_t *obj_model, float *obj_pose, float *obj_score, int32_t *n_features,
                                                int32_t *frame_info, float *stage_ms) {
	if (!ctx) return MC_ERR_ARG;
	MC_TRY(rig_check(ctx, "mc_process_rig_cameras_dev", n_frames, n_cameras));
	return process_images(ctx, "mc_process_rig_cameras_dev", cameras, n_cameras, n_frames, true, double_size, max_keypoints, params, max_objects,
	                      n_objects, obj_model, obj_pose, obj_score, n_features, frame_info, stage_ms);
}

static mc_status extract_rig_cameras(mc_ctx *ctx, const char *who, const mc_rig_camera *cameras, int n_cameras, int n_frames, bool dev,
                                     int double_size, int max_keypoints, float *q_desc_dev, float *q_xy_dev, int32_t *q_image_dev,
                                     int32_t *frame_offsets, int32_t *n_features, float *feat_ms) {
	if (!ctx) return MC_ERR_ARG;
	MC_TRY(rig_check(ctx, who, n_frames, n_cameras));
	if (!q_desc_dev || !q_xy_dev || !q_image_dev || !frame_offsets) { ctx->err = std::string(who) + ": bad argument"; return MC_ERR_ARG; }
	if ((uintptr_t)q_desc_dev % 16 || (uintptr_t)q_xy_dev % 8 || (uintptr_t)q_image_dev % 4) {     // float4 / float2 / int stores
		ctx->err = std::string(who) + ": q_desc_dev must be 16-byte, q_xy_dev 8-byte and q_image_dev 4-byte aligned"; return MC_ERR_ARG;
	}
	return extract_rig(ctx, who, cameras, n_cameras, n_frames, dev, double_size, max_keypoints, q_desc_dev, q_xy_dev, q_image_dev, frame_offsets,
	                   n_features, feat_ms);
}

extern "C" mc_status mc_extract_rig_cameras(mc_ctx *ctx, const mc_rig_camera *cameras, int n_cameras, int n_frames, int double_size,
                                            int max_keypoints, float *q_desc_dev, float *q_xy_dev, int32_t *q_image_dev, int32_t *frame_offsets,
                                            int32_t *n_features, float *feat_ms) {
	return extract_rig_cameras(ctx, "mc_extract_rig_cameras", cameras, n_cameras, n_frames, false, double_size, max_keypoints, q_desc_dev, q_xy_dev,
	                           q_image_dev, frame_offsets, n_features, feat_ms);
}

extern "C" mc_status mc_extract_rig_cameras_dev(mc_ctx *ctx, const mc_rig_camera *cameras, int n_cameras, int n_frames, int double_size,
                                                int max_keypoints, float *q_desc_dev, float *q_xy_dev, int32_t *q_image_dev, int32_t *frame_offsets,
                                                int32_t *n_features, float *feat_ms) {
	return extract_rig_cameras(ctx, "mc_extract_rig_cameras_dev", cameras, n_cameras, n_frames, true, double_size, max_keypoints, q_desc_dev, q_xy_dev,
	                           q_image_dev, frame_offsets, n_features, feat_ms);
}

/* With mc_set_profiling on: device time (ms, summed) of the five octave-0 Gaussian+DoG launches of the last extraction and
 * their algorithmic bytes (per launch: one plane read, the Gaussian and the DoG plane written, for every frame of the batch). */
extern "C" mc_status mc_sift_profile_read(mc_ctx *ctx, float *blur_ms, double *algorithmic_bytes) {
	if (!ctx || !blur_ms) return MC_ERR_ARG;
	SiftState *s = (SiftState *)ctx->sift_state;
	*blur_ms = 0.f;
	if (!s || !ctx->profile || !s->ev_valid) { ctx->err = "mc_sift_profile_read: no profiled extraction"; return MC_ERR_STATE; }
	for (int i = 0; i < kSiftScales + 2; ++i) {
		float ms = 0.f;
		MC_CUDA(cudaEventSynchronize(s->ev[2 * i + 1]));
		MC_CUDA(cudaEventElapsedTime(&ms, s->ev[2 * i], s->ev[2 * i + 1]));
		*blur_ms += ms;
	}
	if (algorithmic_bytes) *algorithmic_bytes = s->ev_bytes;
	return MC_OK;
}

mc_status mc::sift_set_two_pass(mc_ctx *ctx, int on) { state(ctx)->two_pass = on != 0; return MC_OK; }
mc_status mc::sift_set_gather(mc_ctx *ctx, int on) { state(ctx)->gather = on != 0; return MC_OK; }

/* test/bench introspection: one plane of the scale-space of the LAST mc_sift_extract* call.
 * stack: 0 Gaussian (index 0..5), 1 DoG (0..4), 2 gradient magnitude (0..2 = Gaussian 1..3), 3 orientation (0..2) */
extern "C" mc_status mc_sift_read_plane(mc_ctx *ctx, int frame, int octave, int stack, int index, float *out, int32_t *rows, int32_t *cols) {
	if (!ctx) return MC_ERR_ARG;
	SiftState *s = (SiftState *)ctx->sift_state;
	if (!s || s->B == 0) { ctx->err = "mc_sift_read_plane: no extraction has run"; return MC_ERR_STATE; }
	const int depth[4] = { kSiftScales + 3, kSiftScales + 2, kSiftScales, kSiftScales };
	if (frame < 0 || frame >= s->B || octave < 0 || octave >= s->n_oct || stack < 0 || stack > 3 || index < 0 || index >= depth[stack]) {
		ctx->err = "mc_sift_read_plane: bad index"; return MC_ERR_ARG;
	}
	const SiftOct &q = s->oct[octave];
	if (rows) *rows = q.rows;
	if (cols) *cols = q.cols;
	if (!out) return MC_OK;
	const float *base = stack == 0 ? q.gauss : stack == 1 ? q.dog : stack == 2 ? q.grad : q.ori;
	MC_CUDA(cudaSetDevice(ctx->device));
	MC_CUDA(cudaMemcpyAsync(out, base + ((size_t)frame * depth[stack] + index) * q.plane, q.plane * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
	MC_CUDA(cudaStreamSynchronize(ctx->stream));
	return MC_OK;
}
