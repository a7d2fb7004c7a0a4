// match.cu — MATCH step on B200: device-resident model-descriptor database, tcgen05 distance contraction
// (8-bit integer operands first, fp16 for the queries that pass cannot certify) with a fused per-query top-k
// epilogue, exact fp32 re-rank in the reference's summation order, a per-query exactness certificate with an
// exhaustive exact fallback, and the ratio test.
//
// Replaces MATCH_ANN_CPU::Update/process (moped2/libmoped/src/match/MATCH_ANN_CPU.hpp:72-109,136-178)
// and the ANN kd-tree search behind it (libs.tgz!ann_1.1.1/kd_search.cpp:89-210). Parity target: the
// reference matcher in exact mode (Quality=0): same two nearest rows, same squared distances bit for bit.
//
// Kernels
//   k_pack_tiles      fp32 rows -> fp16 operand tile images, pre-swizzled (128B swizzle, K-major) so one
//                     32 KiB cp.async.bulk lands a ready-to-MMA tile in shared memory
//   k_pack_tiles_q8   fp32 rows -> u8 / s8 operand tile images (16 KiB) + the quantisation residual norms
//   k_match_coarse<K> persistent warp-specialised tcgen05 kernel: TMA producer / MMA issuer / 8 epilogue warps;
//                     K = 0 kind::f16 (fp32 accumulators), K = 1 kind::i8 (exact int32 accumulators)
//   k_match_rerank    exact distances of the coarse candidates, top-2, certificate
//   k_match_exact*    exhaustive exact scan (fallback for uncertified queries, and MC_MATCH_EXACT)
//   k_match_finalize  ratio test
#include "common.cuh"
#include "top2.cuh"

#include <math_constants.h>
#include <type_traits>

// MC_COARSE_DBG (experiments only, never in the shipped library): 1 = the epilogue hands the accumulator stage back without
// reading it (MMA + TMA pace alone), 2 = the epilogue reads TMEM but skips the top-k scan (adds the TMEM-read pace),
// 3 = full epilogue without the insertion path (wrong candidates: what the slow path costs),
// 5 = as 1 and no MMAs are issued (TMA streaming pace alone), 6 = as 1 and no DB tiles are copied (MMA + hand-off pace alone)
#ifndef MC_COARSE_DBG
#define MC_COARSE_DBG 0
#endif
#ifndef MC_MMA_THREADS
#define MC_MMA_THREADS 2      // MMA-issuing threads per CTA (1 or 2)
#endif

namespace mc {

// =============================================================================================
// small PTX wrappers (sm_100a)
// =============================================================================================
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
	asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
	asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
	asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// the retry loop branches on the try_wait predicate itself (labels are local to the braces, so every inlined copy has its own)
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
	asm volatile(
	    "{\n\t.reg .pred p;\n"
	    "MC_WAIT:\n\t"
	    "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
	    "@!p bra MC_WAIT;\n\t}"
	    ::"r"(bar), "r"(parity)
	    : "memory");
}
// warpgroup-wide register budget (all 128 threads of the warpgroup execute it, before any divergence): the warpgroup's threads
// give registers back to the CTA's pool / take them from it
template <uint32_t R> __device__ __forceinline__ void regs_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(R)); }
template <uint32_t R> __device__ __forceinline__ void regs_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(R)); }
__device__ __forceinline__ void fence_barrier_init() {
	asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
	asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
// 1-D bulk copy global -> shared (TMA engine, UBLKCP), completion counted on an mbarrier
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
	asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
	             ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst, uint32_t ncols) {
	asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols) : "memory");
	asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
	asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, fp16 inputs, fp32 accumulate; issued by ONE thread
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
	asm volatile(
	    "{\n\t.reg .pred p;\n\t"
	    "setp.ne.b32 p, %4, 0;\n\t"
	    "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
	    ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
	    : "memory");
}
// the same with 8-bit integer inputs (signedness of A and B in the instruction descriptor), int32 accumulate
__device__ __forceinline__ void umma_i8(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
	asm volatile(
	    "{\n\t.reg .pred p;\n\t"
	    "setp.ne.b32 p, %4, 0;\n\t"
	    "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
	    ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
	    : "memory");
}
// mbarrier arrive when all previously issued MMAs of this thread have completed
__device__ __forceinline__ void umma_commit(uint32_t bar) {
	asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// 32 lanes x 32 consecutive 32-bit columns: thread t gets row (lane base + t), u[j] = column (col base + j)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&u)[32]) {
	asm volatile(
	    "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
	    "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
	    "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
	    : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]),
	      "=r"(u[8]), "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15]),
	      "=r"(u[16]), "=r"(u[17]), "=r"(u[18]), "=r"(u[19]), "=r"(u[20]), "=r"(u[21]), "=r"(u[22]), "=r"(u[23]),
	      "=r"(u[24]), "=r"(u[25]), "=r"(u[26]), "=r"(u[27]), "=r"(u[28]), "=r"(u[29]), "=r"(u[30]), "=r"(u[31])
	    : "r"(taddr)
	    : "memory");
}

// order-preserving float <-> uint map, so that atomicMax works on scores of either sign.
// 0 (a cleared buffer) decodes to -inf.
__device__ __forceinline__ uint32_t f2o(float f) {
	uint32_t u = __float_as_uint(f);
	return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float o2f(uint32_t o) {
	if (o <= 0x007FFFFFu) return -CUDART_INF_F;
	return __uint_as_float((o & 0x80000000u) ? (o ^ 0x80000000u) : ~o);
}

// =============================================================================================
// operand tile images
// =============================================================================================
// fp16 tile image of 128 rows x 128 fp16 (K-major): two K atoms of 64 elements; inside an atom row r is a
// 128-byte line at (r/8)*1024 + (r%8)*128 whose 16-byte chunk c sits at chunk position c ^ (r%8)
// (the 128B swizzle tcgen05 smem descriptors expect). One thread writes one 16-byte chunk.
// `list` (nullable): gather — image row i is source row list[i] for i < *list_count, zero beyond (the second-chance pass
// of the cascade packs the queries the 8-bit pass could not certify).
__global__ void k_pack_tiles(const float *__restrict__ src, int64_t n_rows, int64_t n_tiles, __half *__restrict__ img,
                             float *__restrict__ norm2 /* nullable: per-row sum of squares */,
                             const int32_t *__restrict__ list, const int32_t *__restrict__ list_count) {
	int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	int64_t total = n_tiles * 2048;
	if (gid >= total) return;
	int c = (int)(gid & 7);
	int r = (int)((gid >> 3) & 127);
	int a = (int)((gid >> 10) & 1);
	int64_t t = gid >> 11;
	int64_t row = t * kTileRows + r;
	if (list) {
		const int64_t n_list = *list_count < n_rows ? *list_count : n_rows;
		row = row < n_list ? (int64_t)list[row] : n_rows;
	}
	uint4 out = make_uint4(0, 0, 0, 0);
	if (row < n_rows) {
		const float4 *p = reinterpret_cast<const float4 *>(src + row * kD + a * 64 + c * 8);
		float4 v0 = p[0], v1 = p[1];
		__half2 h0 = __floats2half2_rn(v0.x, v0.y), h1 = __floats2half2_rn(v0.z, v0.w);
		__half2 h2 = __floats2half2_rn(v1.x, v1.y), h3 = __floats2half2_rn(v1.z, v1.w);
		out.x = *reinterpret_cast<uint32_t *>(&h0); out.y = *reinterpret_cast<uint32_t *>(&h1);
		out.z = *reinterpret_cast<uint32_t *>(&h2); out.w = *reinterpret_cast<uint32_t *>(&h3);
	}
	size_t off = (size_t)t * kTileBytes + (size_t)a * 16384 + (size_t)(r >> 3) * 1024 + (size_t)(r & 7) * 128 + (size_t)((c ^ (r & 7)) * 16);
	*reinterpret_cast<uint4 *>(reinterpret_cast<char *>(img) + off) = out;
	if (norm2 && a == 0 && c == 0 && row < n_rows) {
		const float *p = src + row * kD;
		float s = 0.f;
		for (int d = 0; d < kD; d++) s = fmaf(p[d], p[d], s);
		norm2[row] = s;
	}
}

// 8-bit tile image of 128 rows x 128 bytes (K-major, ONE 128-byte K atom, the same 128B swizzle): row r = round(S * x) as
// u8 (all values of the tile >= 0: S = 255 / max) or s8 (S = 127 / max|x|). One CTA per tile, a warp per 16 rows, a lane per
// 4 consecutive dimensions.
//   per_row != 0 (queries): every row has its own scale S_r = top / max_d |x_rd| (scores of different queries are never
//     compared with each other), the signedness is per TILE (one tcgen05.mma covers 128 rows of A) -> tile_signed[t];
//   per_row == 0 (database): one scale and one signedness for all rows (scores of different rows ARE compared).
// err[r] = |x_r - q_r / S|_2 (what the certificate charges for the quantisation, clamping included), norm2[r] = |x_r|^2,
// scale[r] = S_r; err_max (nullable): maximum of err over all rows (bits of a non-negative float, atomicMax).
constexpr int kTile8Bytes = kTileRows * kD;      // 16 KiB
__global__ void __launch_bounds__(256)
k_pack_tiles_q8(const float *__restrict__ src, int64_t n_rows, uint8_t *__restrict__ img, int per_row, float fixed_scale, int fixed_signed,
                uint8_t *__restrict__ tile_signed, float *__restrict__ scale, float *__restrict__ err, float *__restrict__ norm2,
                int *__restrict__ err_max_bits) {
	const int64_t t = blockIdx.x;
	const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
	float4 v[16];
	bool neg = false;
#pragma unroll
	for (int i = 0; i < 16; i++) {
		const int64_t row = t * kTileRows + w * 16 + i;
		v[i] = row < n_rows ? __ldg(reinterpret_cast<const float4 *>(src + row * kD) + lane) : make_float4(0.f, 0.f, 0.f, 0.f);
		neg |= v[i].x < 0.f || v[i].y < 0.f || v[i].z < 0.f || v[i].w < 0.f;
	}
	const int sgn = per_row ? __syncthreads_or(neg ? 1 : 0) : fixed_signed;
	if (per_row && threadIdx.x == 0 && tile_signed) tile_signed[t] = sgn ? 1 : 0;
	const float top = sgn ? 127.f : 255.f, bottom = sgn ? -127.f : 0.f;
	float worst = 0.f;
#pragma unroll
	for (int i = 0; i < 16; i++) {
		const int r = w * 16 + i;
		const int64_t row = t * kTileRows + r;
		float S = fixed_scale;
		if (per_row) {
			float m = fmaxf(fmaxf(fabsf(v[i].x), fabsf(v[i].y)), fmaxf(fabsf(v[i].z), fabsf(v[i].w)));
			for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
			S = m > 0.f ? top / m : 0.f;
		}
		const float inv = S > 0.f ? 1.f / S : 0.f;
		const float x[4] = { v[i].x, v[i].y, v[i].z, v[i].w };
		uint32_t packed = 0;
		float e2 = 0.f, n2 = 0.f;
#pragma unroll
		for (int j = 0; j < 4; j++) {
			const float qf = fminf(fmaxf(rintf(x[j] * S), bottom), top);     // NaN -> bottom (fmaxf drops it); the residual then is NaN: uncertified
			const int qi = (int)qf;
			packed |= ((uint32_t)qi & 0xffu) << (8 * j);
			const float d = x[j] - qf * inv;
			e2 = fmaf(d, d, e2);
			n2 = fmaf(x[j], x[j], n2);
		}
		for (int o = 16; o; o >>= 1) { e2 += __shfl_xor_sync(0xffffffffu, e2, o); n2 += __shfl_xor_sync(0xffffffffu, n2, o); }
		const int c = lane >> 2;
		const size_t off = (size_t)t * kTile8Bytes + (size_t)(r >> 3) * 1024 + (size_t)(r & 7) * 128 + (size_t)((c ^ (r & 7)) * 16) + (size_t)(lane & 3) * 4;
		*reinterpret_cast<uint32_t *>(img + off) = packed;
		if (row < n_rows) {
			const float e = sqrtf(e2) * 1.0001f;
			if (lane == 0) {
				if (scale) scale[row] = S;
				if (err) err[row] = e;
				if (norm2) norm2[row] = n2;
			}
			worst = e > worst || e != e ? e : worst;          // keeps a NaN
		}
	}
	if (err_max_bits && lane == 0) {
		if (worst != worst) worst = CUDART_INF_F;
		atomicMax(err_max_bits, __float_as_int(worst));
	}
}

__global__ void k_minmax(const float *__restrict__ v, int64_t n, float *__restrict__ out2) {
	float lo = CUDART_INF_F, hi = -CUDART_INF_F;
	for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
		lo = fminf(lo, v[i]); hi = fmaxf(hi, v[i]);
	}
	for (int o = 16; o; o >>= 1) { lo = fminf(lo, __shfl_xor_sync(0xffffffffu, lo, o)); hi = fmaxf(hi, __shfl_xor_sync(0xffffffffu, hi, o)); }
	if ((threadIdx.x & 31) == 0) {
		atomicMin(reinterpret_cast<int *>(&out2[0]), __float_as_int(lo));   // norms are positive: int order == float order
		atomicMax(reinterpret_cast<int *>(&out2[1]), __float_as_int(hi));
	}
}

// database-wide max |x| (bits of a non-negative float) and "any element negative"
__global__ void k_absmax(const float *__restrict__ v, int64_t n, int *__restrict__ out2) {
	float hi = 0.f;
	int neg = 0;
	for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
		const float x = v[i];
		hi = fmaxf(hi, fabsf(x));
		neg |= x < 0.f;
	}
	for (int o = 16; o; o >>= 1) { hi = fmaxf(hi, __shfl_xor_sync(0xffffffffu, hi, o)); neg |= __shfl_xor_sync(0xffffffffu, neg, o); }
	if ((threadIdx.x & 31) == 0) {
		atomicMax(&out2[0], __float_as_int(hi));
		if (neg) atomicOr(&out2[1], 1);
	}
}

// =============================================================================================
// coarse pass: tcgen05 contraction with fused per-query top-k, persistent over (query tile, DB split) work items
// =============================================================================================
// KIND 0: fp16 operands, fp32 accumulators (kind::f16; 2 K atoms x 4 MMAs of K=16 per 128 x 128 block)
// KIND 1: 8-bit integer operands, exact int32 accumulators (kind::i8; 4 MMAs of K=32), twice the MMA rate and half the
//         operand bytes; its scores carry the quantisation error, which the certificate of k_match_rerank charges in full
#ifndef MC_COARSE_CG
#define MC_COARSE_CG 2
#endif
constexpr int kCG = MC_COARSE_CG;       // column groups: epilogue threads per query (1 or 2)
template <int KIND> struct CoarseKind;
template <> struct CoarseKind<0> {
	typedef float acc_t;
	static constexpr int kTile = kTileBytes, kStages = 4, kABuf = 1, kK = kTopK, kSteps = 8;           // kK candidates per (query, split, column group)
};
template <> struct CoarseKind<1> {
	typedef float acc_t;            // int32 accumulators READ AS FLOAT BIT PATTERNS, see k_match_coarse
	static constexpr int kTile = kTile8Bytes, kStages = 8, kABuf = 2, kK = kTopK8 / kCG, kSteps = 4;
};
constexpr int kCoarseThreads = 128 + 256 * kCG;   // warp 0 TMA, warp 1 MMA, warp 2 TMEM alloc, warp 3 second MMA issuer, then 8 epilogue warps per column group
// Register budgets (setmaxnreg): the CTA is launched with what __launch_bounds__(kCoarseThreads, 1) allows every thread (96 for
// kCG = 2); warpgroup 0 runs single-lane control code and gives half of it back, the epilogue warpgroups take it:
// 128 x 48 + 512 x 104 <= 640 x 96. (At 32 / 40 the MMA issuers spill, and the epilogue cannot use more than 104 either way.)
constexpr uint32_t kRegsLaunch = (65536 / kCoarseThreads) & ~7u;
constexpr uint32_t kRegsControl = 48;
constexpr uint32_t kRegsEpilogue = ((kRegsLaunch * kCoarseThreads - 128 * kRegsControl) / (256 * kCG)) & ~7u;
static_assert(kRegsEpilogue <= 256 && 128 * kRegsControl + 256 * kCG * kRegsEpilogue <= kRegsLaunch * kCoarseThreads, "register pool");
// the CTA-wide barrier before TMEM is freed, reached from both warpgroup branches: barrier.sync without .aligned (code reachable
// from the epilogue that needs a warp-collective call, as the .aligned forms in divergent code do, pins its registers to the
// launch budget)
__device__ __forceinline__ void teardown_sync() { asm volatile("barrier.sync 1, %0;" ::"n"(kCoarseThreads) : "memory"); }
constexpr uint32_t kSmemA = 0;          // A operand: kABuf x (2 halves x kTile) = 64 KiB for both kinds
constexpr uint32_t kSmemB = 65536;      // B ring: kStages x kTile = 128 KiB for both kinds
constexpr uint32_t kSmemBar = kSmemB + 131072;
constexpr uint32_t kCoarseSmemBytes = kSmemBar + 256 + 1024;   // + barriers + alignment slack

// UMMA shared-memory descriptor: K-major, 128B swizzle, 8-row groups 1024 B apart (SBO), version 1
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr) {
	return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) |
	       ((uint64_t)2 << 61);
}
// instruction descriptors, both operands K-major, N=128, M=128. f16: D=f32, A=B=f16. i8: D=s32, A/B signedness at bits 7 / 10.
constexpr uint32_t kIdescF16 = (1u << 4) | ((128u >> 3) << 17) | ((128u >> 4) << 24);
constexpr uint32_t kIdescI8 = (2u << 4) | ((128u >> 3) << 17) | ((128u >> 4) << 24);

// running-threshold encodings for atomicMax; 0 (a cleared buffer) decodes to "none"
template <typename T> struct Score;
template <> struct Score<float> {
	static __device__ __forceinline__ float none() { return -CUDART_INF_F; }
	static __device__ __forceinline__ uint32_t enc(float f) { return f2o(f); }
	static __device__ __forceinline__ float dec(uint32_t o) { return o2f(o); }
	static __device__ __forceinline__ float vmax(float a, float b) { return fmaxf(a, b); }
};
template <typename T, int K>
__device__ __forceinline__ void topk_insert(T (&ts)[K], int (&ti)[K], T v, int row) {
	ts[K - 1] = v; ti[K - 1] = row;
#pragma unroll
	for (int j = K - 1; j > 0; j--) {
		bool sw = ts[j] > ts[j - 1];
		T a = ts[j], b = ts[j - 1];
		int ia = ti[j], ib = ti[j - 1];
		ts[j - 1] = sw ? a : b; ts[j] = sw ? b : a;
		ti[j - 1] = sw ? ia : ib; ti[j] = sw ? ib : ia;
	}
}

// One chunk of 32 accumulator columns of this thread's query. Fast path: 4 group maxima against the
// running threshold; slow path (rare once the threshold has warmed up): insertion of the survivors.
template <typename T, int K>
__device__ __forceinline__ void scan_chunk(const T (&r)[32], int row_base, T &tau, T (&ts)[K], int (&ti)[K]) {
	typedef Score<T> S;
#define MC_MAX8(g) S::vmax(S::vmax(S::vmax(r[8 * g], r[8 * g + 1]), S::vmax(r[8 * g + 2], r[8 * g + 3])), S::vmax(S::vmax(r[8 * g + 4], r[8 * g + 5]), S::vmax(r[8 * g + 6], r[8 * g + 7])))
	const T m0 = MC_MAX8(0), m1 = MC_MAX8(1), m2 = MC_MAX8(2), m3 = MC_MAX8(3);
#undef MC_MAX8
	const T m = S::vmax(S::vmax(m0, m1), S::vmax(m2, m3));
#if MC_COARSE_DBG == 3
	if (m > tau) { tau = m; ts[K - 1] = m; ti[K - 1] = row_base; }      // timing experiment: the fast path alone (wrong candidates)
	return;
#endif
	if (m > tau) {
		// Slow path (a few per cent of the chunks once the threshold has warmed up, and a warp pays it for all 32 queries): only
		// the groups that hold a survivor are visited, every element by its own predicated test — everything stays in
		// registers (an earlier version staged the group through local memory: ~180 instructions per visit, now ~45).
#define MC_VISIT_GROUP(g, mg)                                                   \
		if (mg > tau) {                                                         \
			_Pragma("unroll") for (int j = 0; j < 8; j++)                       \
				if (r[8 * g + j] > tau) {                                       \
					topk_insert<T, K>(ts, ti, r[8 * g + j], row_base + 8 * g + j); \
					tau = S::vmax(tau, ts[K - 1]);                              \
				}                                                               \
		}
		MC_VISIT_GROUP(0, m0) MC_VISIT_GROUP(1, m1) MC_VISIT_GROUP(2, m2) MC_VISIT_GROUP(3, m3)
#undef MC_VISIT_GROUP
	}
}

template <typename T>
__device__ __forceinline__ void mask_tail(T (&r)[32], int64_t row_base, int64_t n_rows) {
#pragma unroll
	for (int j = 0; j < 32; j++)
		if (row_base + j >= n_rows) r[j] = Score<T>::none();
}

struct CoarseArgs {
	const uint8_t *q_img;          // query tile images, 2 x kTile per tile of 256 queries
	const uint8_t *db_img;         // database tile images
	int64_t n_tiles, n_rows;
	int tiles_per_split, n_splits, n_mtiles;
	const int32_t *q_count;        // nullable: number of live queries on the device (second-chance pass) -> live query tiles
	const uint8_t *a_signed;       // KIND 1: signedness of every 128-query half tile (k_pack_tiles_q8)
	uint32_t b_signed;             // KIND 1: signedness of the database image
	int stagger;                   // CTAs of one split start at different tiles (see k_match_coarse)
	uint32_t *item_counter;        // zeroed before the launch: next work item (dynamic assignment)
	uint32_t *g_tau;               // per query: best published k-th score over all work items (encoded, 0 = none)
	uint32_t *cand_score;          // [query][split][column group][k] raw accumulator bits (float / int32)
	int32_t *cand_row;             // [query][split][column group][k] shard-local row, -1 = empty
};

// A CTA is persistent: its TMA thread takes the next work item from a global counter and hands the number to the other warps
// through a two-slot ring in shared memory (item = query tile + live tiles x DB split, handed out in order, so that the CTAs
// running at the same time stream the same DB split out of L2). Dynamic, because the kernel shares the GPU: a CTA that gets its
// SM late — stage kernels of an earlier batch still hold it — simply takes fewer items instead of delaying the whole launch. Per item it keeps the 256 queries'
// image resident in shared memory (A, double-buffered for the 8-bit kind) and streams the split's DB tile images through a
// ring (B) with one elected TMA thread; one elected MMA thread issues the MMAs of a DB tile, 128 queries (a "half") at a
// time, into one of two TMEM accumulator stages; the 8 epilogue warps (4 per half, warp%4 = TMEM lane quarter) read their
// half of the finished stage back with tcgen05.ld, ONE QUERY PER THREAD, and keep that query's top-k (score, row) in
// registers. Every (stage, half) has its own full / empty barrier pair, so the MMA thread refills a half as soon as ITS
// four warps are done with it. The pipeline state (ring and stage phases) runs on across items; TMEM is allocated once.
// `stagger`: CTA b starts its split at tile (ntiles * b / CTAs) and wraps around, so that the CTAs working on the same split
// at the same time pull different tiles out of L2 instead of all asking for the same one.
// 8-bit kind: the epilogue compares the int32 accumulators AS FLOATS (full-rate FMNMX instead of half-rate integer min/max).
// Bit patterns of non-negative int32 below 2^31 order like the integers themselves (zero, denormals, normals; match.cu is
// compiled without flush-to-zero); a negative accumulator is a negative float or a NaN pattern, which `>` and fmaxf drop.
// So only rows with a score > 0 can become candidates, the running threshold starts at 0 instead of -inf, and "every row that
// is not a candidate scored <= T" holds with T >= 0.
template <int KIND>
__global__ void __launch_bounds__(kCoarseThreads, 1)
k_match_coarse(const CoarseArgs a) {
	typedef CoarseKind<KIND> C;
	typedef typename C::acc_t T;
	typedef Score<T> S;
	constexpr int K = C::kK;
	extern __shared__ uint8_t smem_raw[];
	const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
	uint8_t *smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	int n_mt = a.n_mtiles;
	if (a.q_count) { const int live = (*a.q_count + kMTile - 1) / kMTile; n_mt = live < n_mt ? live : n_mt; }
	const int n_items = n_mt * a.n_splits;
	if (n_items <= 0) return;

	// barrier block (8 B each): full[8], empty[8], a_full[2], a_empty[2], tfull[2] (+2 unused), tempty[2][2], then the TMEM base slot
	const uint32_t bar0 = smem_base + kSmemBar;
	auto bar_full = [&](int s) { return bar0 + 8u * s; };
	auto bar_empty = [&](int s) { return bar0 + 8u * (8 + s); };
	auto bar_afull = [&](int s) { return bar0 + 8u * (16 + s); };
	auto bar_aempty = [&](int s) { return bar0 + 8u * (18 + s); };
	auto bar_tfull = [&](int s) { return bar0 + 8u * (20 + s); };
	auto bar_tempty = [&](int s, int h) { return bar0 + 8u * (24 + 2 * s + h); };
	volatile uint32_t *tmem_slot = reinterpret_cast<volatile uint32_t *>(smem_gen + kSmemBar + 8 * 28);
	auto bar_ifull = [&](int s) { return bar0 + 8u * (22 + s); };
	auto bar_iempty = [&](int s) { return bar0 + 8u * (29 + s); };
	volatile int32_t *item_ring = reinterpret_cast<volatile int32_t *>(smem_gen + kSmemBar + 8 * 31);   // two slots

	if (threadIdx.x == 0) {
		for (int s = 0; s < C::kStages; s++) { mbar_init(bar_full(s), 1); mbar_init(bar_empty(s), 1); }
		for (int s = 0; s < 2; s++) { mbar_init(bar_afull(s), 1); mbar_init(bar_aempty(s), MC_MMA_THREADS); }
		for (int s = 0; s < 2; s++) { mbar_init(bar_ifull(s), 1); mbar_init(bar_iempty(s), MC_MMA_THREADS + 8 * kCG); }
		for (int s = 0; s < 2; s++) {
			mbar_init(bar_tfull(s), 1);
			for (int h = 0; h < 2; h++) mbar_init(bar_tempty(s, h), 4 * kCG);
		}
		fence_barrier_init();
	}
	if (warp == 2) tmem_alloc(smem_base + kSmemBar + 8 * 28, 512);
	tc_fence_before();
	__syncthreads();
	tc_fence_after();
	const uint32_t tmem_base = *tmem_slot;

	auto item_range = [&](int item, int &mtile, int &split, int64_t &t0, int &ntiles, int &first) {
		mtile = item % n_mt; split = item / n_mt;
		t0 = (int64_t)split * a.tiles_per_split;
		const int64_t t1 = (t0 + a.tiles_per_split < a.n_tiles) ? t0 + a.tiles_per_split : a.n_tiles;
		ntiles = (int)(t1 > t0 ? t1 - t0 : 0);
		// 32-bit on purpose: a 64-bit division is a called subroutine, and a call in the epilogue pins its registers to the launch
		// budget. The product wraps only beyond 2^32 / gridDim.x tiles in a split, and the quotient stays below ntiles even then.
		first = a.stagger ? (int)((uint32_t)ntiles * blockIdx.x / gridDim.x) : 0;
	};
	auto tile_at = [](int i, int first, int ntiles) { const int t = i + first; return t >= ntiles ? t - ntiles : t; };
	// consumers of the item ring: the it-th item of this CTA, or -1 when the counter has run out
	auto next_item = [&](uint32_t it, bool whole_warp) {      // whole_warp: called by all 32 lanes (epilogue) / by one thread (MMA issuer)
		const uint32_t sl = it & 1;
		mbar_wait(bar_ifull(sl), (it >> 1) & 1);
		const int item = item_ring[sl];
		if (whole_warp) __syncwarp();
		if (lane == 0) mbar_arrive(bar_iempty(sl));
		return item;
	};

	if (warp < 4) {
		// warpgroup 0 (TMA producer, MMA issuers, TMEM allocator) runs single-lane code: it gives registers to the epilogue
		regs_dec<kRegsControl>();
		if (warp == 0) {
			// ===== TMA producer =====
			if (lane == 0) {
				uint32_t tc = 0;
				for (uint32_t it = 0;; it++) {
					const uint32_t sl = it & 1;
					mbar_wait(bar_iempty(sl), ((it >> 1) & 1) ^ 1);
					int item = (int)atomicAdd(a.item_counter, 1u);
					if (item >= n_items) item = -1;
					item_ring[sl] = item;
					mbar_arrive(bar_ifull(sl));            // release: the consumers' wait acquires the slot
					if (item < 0) break;
					int mtile, split, ntiles, first; int64_t t0;
					item_range(item, mtile, split, t0, ntiles, first);
					const uint32_t ab = it % C::kABuf;
					mbar_wait(bar_aempty(ab), ((it / C::kABuf) & 1) ^ 1);
					mbar_expect_tx(bar_afull(ab), 2 * C::kTile);
					bulk_g2s(smem_base + kSmemA + ab * 2 * C::kTile, a.q_img + (size_t)mtile * 2 * C::kTile, 2 * C::kTile, bar_afull(ab));
					for (int i = 0; i < ntiles; i++, tc++) {
						const uint32_t b = tc % C::kStages;
						mbar_wait(bar_empty(b), ((tc / C::kStages) & 1) ^ 1);
#if MC_COARSE_DBG == 6
						mbar_arrive(bar_full(b));
#else
						mbar_expect_tx(bar_full(b), C::kTile);
						bulk_g2s(smem_base + kSmemB + b * C::kTile, a.db_img + (size_t)(t0 + tile_at(i, first, ntiles)) * C::kTile, C::kTile, bar_full(b));
#endif
					}
				}
			}
			__syncwarp();
		} else if (warp == 1 || (warp == 3 && MC_MMA_THREADS == 2)) {
			// ===== MMA issuer(s): one thread, or two that take alternate tiles (thread p owns accumulator stage p) =====
			// ONE tcgen05.commit per DB tile: every commit costs the issuing thread about 190 cycles in which it issues nothing
			// (measured: tile time = MMA floor + 190 x commits), so the shared-memory stage is handed back to the TMA producer by
			// an epilogue thread once it has seen this commit, and a second issuer fills the gap of the first.
			const int p = warp == 3 ? 1 : 0;
			if (lane == 0) {
				uint32_t tc = 0;
				for (uint32_t it = 0;; it++) {
					const int item = next_item(it, false);
					if (item < 0) break;
					int mtile, split, ntiles, first; int64_t t0;
					item_range(item, mtile, split, t0, ntiles, first);
					const uint32_t ab = it % C::kABuf;
					uint32_t idesc[2] = { kIdescF16, kIdescF16 };
					if (KIND == 1)
						for (int h = 0; h < 2; h++) idesc[h] = kIdescI8 | ((uint32_t)a.a_signed[2 * mtile + h] << 7) | (a.b_signed << 10);
					mbar_wait(bar_afull(ab), (it / C::kABuf) & 1);
					for (int i = 0; i < ntiles; i++, tc++) {
						if (MC_MMA_THREADS == 2 && (int)(tc & 1) != p) continue;
						const uint32_t s = tc & 1, b = tc % C::kStages;
						mbar_wait(bar_full(b), (tc / C::kStages) & 1);
#pragma unroll
						for (int h = 0; h < 2; h++) {
							mbar_wait(bar_tempty(s, h), ((tc >> 1) & 1) ^ 1);
							tc_fence_after();
#if MC_COARSE_DBG != 5
							const uint32_t d_tmem = tmem_base + (uint32_t)(s * 256 + h * 128);
#pragma unroll
							for (int k = 0; k < C::kSteps; k++) {
								const uint32_t koff = KIND == 0 ? (uint32_t)((k >> 2) * 16384 + (k & 3) * 32) : (uint32_t)(k * 32);
								const uint64_t a_desc = make_desc(smem_base + kSmemA + (ab * 2 + h) * C::kTile + koff);
								const uint64_t b_desc = make_desc(smem_base + kSmemB + b * C::kTile + koff);
								if (KIND == 0) umma_f16(d_tmem, a_desc, b_desc, idesc[h], k > 0 ? 1u : 0u);
								else umma_i8(d_tmem, a_desc, b_desc, idesc[h], k > 0 ? 1u : 0u);
							}
#endif
						}
#if MC_COARSE_DBG == 5
						(void)idesc;
						mbar_arrive(bar_tfull(s));
#else
						umma_commit(bar_tfull(s));         // both halves of the accumulator stage complete, shared-memory stage b read
#endif
					}
					umma_commit(bar_aempty(ab));           // query image reusable once the item's MMAs (of this issuer) have read it
				}
			}
			__syncwarp();
		}
		tc_fence_before();
		teardown_sync();
		if (warp == 2) { tc_fence_after(); tmem_dealloc(tmem_base, 512); }
	} else {
		regs_inc<kRegsEpilogue>();
		// ===== epilogue: one (query, column group) per thread =====
		// kCG = 2: 16 warps, four per SM sub-partition; a thread scans 64 of the tile's 128 columns for its query and keeps its
		// own top-k — the chain "wait for the stage, tcgen05.ld, max tree, compare" is latency-bound (about 7 cycles per
		// instruction with two warps per sub-partition), four warps hide twice as much of it.
		const int e = __shfl_sync(0xffffffffu, warp, 0) - 4;     // known to be warp-uniform: per-warp values stay in uniform registers
		const int quarter = e & 3, half = (e >> 2) & 1, cg = e >> 3;          // TMEM lane quarter == warp % 4
		constexpr int kCols = 128 / kCG;                   // accumulator columns (DB rows of a tile) per thread
		// accumulator stage s = tc & 1 adds 256 columns to the TMEM address and 8 s / 16 s bytes to its full / empty barrier
		const uint32_t taddr0 = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(half * 128 + cg * kCols);
		const uint32_t tfull0 = bar_tfull(0), tempty0 = bar_tempty(0, half);
		const bool returns_stage = e == 0 && lane == 0;   // hands the shared-memory stage of a tile back to the TMA producer
		uint32_t tc = 0;
		T ra[32], rb[32];
		uint32_t (&ua)[32] = reinterpret_cast<uint32_t (&)[32]>(ra);
		uint32_t (&ub)[32] = reinterpret_cast<uint32_t (&)[32]>(rb);
		for (uint32_t it = 0;; it++) {
			const int item = next_item(it, true);
			if (item < 0) break;
			int mtile, split, ntiles, first; int64_t t0;
			item_range(item, mtile, split, t0, ntiles, first);
			const int qid = mtile * kMTile + half * 128 + quarter * 32 + lane;
			uint32_t *const gtau = a.g_tau + qid;
			T ts[K]; int ti[K];
#pragma unroll
			for (int j = 0; j < K; j++) { ts[j] = S::none(); ti[j] = -1; }
			T tau = KIND == 1 ? (T)0 : S::none(), published = tau;
			uint32_t og = 0;
			// first DB row of this thread's columns: runs through the split from tile `first` and wraps to the split's first tile
			const int row_lo = (int)t0 * kTileRows + cg * kCols, row_end = row_lo + ntiles * kTileRows;
			int row0 = row_lo + first * kTileRows;
			// the tile loop; only the items whose split holds the database's ragged last tile run the instance that masks it
			auto tiles = [&](auto ragged) {
				for (int i0 = 0; i0 < ntiles; i0 += 8) {
					// other items' threshold: fetched once per 8 tiles and consumed 8 tiles later (a load the next tile already waits
					// for would put an L2 round trip into every tile); this thread's k-th best is published at the same pace. Both
					// are no-ops in the first block: og = 0 decodes to -inf and the list is still empty.
					tau = S::vmax(tau, S::dec(og));
					if (ts[K - 1] > published) { published = ts[K - 1]; atomicMax(gtau, S::enc(published)); }
					og = __ldcg(gtau);
					const int n = ntiles - i0 < 8 ? ntiles - i0 : 8;
					for (int j = 0; j < n; j++, tc++) {
						const uint32_t s = tc & 1;
						const uint32_t taddr = taddr0 + (s << 8);
						mbar_wait(tfull0 + 8 * s, (tc >> 1) & 1);
						tc_fence_after();
						if (returns_stage) mbar_arrive(bar_empty(tc % C::kStages));   // the tile's MMAs have read their shared-memory stage
#if MC_COARSE_DBG == 1 || MC_COARSE_DBG == 5 || MC_COARSE_DBG == 6
						tc_fence_before();
						__syncwarp();
						if (lane == 0) mbar_arrive(tempty0 + 16 * s);
						(void)taddr; (void)ua; (void)ub; (void)ragged;
#elif MC_COARSE_DBG == 2
						for (int c = 0; c < kCols; c += 64) {
							tmem_ld32(taddr + c, ua); tmem_ld32(taddr + c + 32, ub); tmem_ld_wait();
							tau = S::vmax(tau, S::vmax(ra[0], rb[31]));
						}
						tc_fence_before();
						__syncwarp();
						if (lane == 0) mbar_arrive(tempty0 + 16 * s);
						(void)ragged;
#else
#pragma unroll
						for (int c = 0; c < kCols; c += 64) {
							tmem_ld32(taddr + c, ua);
							tmem_ld32(taddr + c + 32, ub);
							tmem_ld_wait();
							if (c + 64 == kCols) {
								// all TMEM reads of this thread's part of the half stage are done: hand it back to the MMA thread
								tc_fence_before();
								__syncwarp();
								if (lane == 0) mbar_arrive(tempty0 + 16 * s);
							}
							if constexpr (decltype(ragged)::value) {
								if (row0 + c + 64 > a.n_rows) { mask_tail<T>(ra, row0 + c, a.n_rows); mask_tail<T>(rb, row0 + c + 32, a.n_rows); }
							}
							scan_chunk<T, K>(ra, row0 + c, tau, ts, ti);
							scan_chunk<T, K>(rb, row0 + c + 32, tau, ts, ti);
						}
#endif
						row0 += kTileRows;
						if (row0 == row_end) row0 = row_lo;
					}
				}
			};
			if (a.n_rows % kTileRows != 0 && t0 + ntiles == a.n_tiles) tiles(std::true_type());
			else tiles(std::false_type());
			if (ts[K - 1] > published) atomicMax(&a.g_tau[qid], S::enc(ts[K - 1]));   // what the certificate reads: every list's final k-th best
			const size_t o = (((size_t)qid * a.n_splits + split) * kCG + cg) * K;
#pragma unroll
			for (int j = 0; j < K; j++) {
				a.cand_score[o + j] = __float_as_uint(ts[j]);
				a.cand_row[o + j] = ti[j];
			}
		}
		tc_fence_before();
		teardown_sync();
	}
}

// =============================================================================================
// exact arithmetic of the reference: dist = sum_d (q[d]-p[d])^2, sequential, product and sum each
// rounded to fp32 (VMULSS + VADDSS in the compiled reference, libs.tgz!ann_1.1.1/kd_search.cpp:188-199);
// the two nearest rows are kept by Top2 (top2.cuh)
// =============================================================================================

// Exact re-rank of the coarse candidates; one warp per query.
//
// Scores -> dot products: s' = score (fp16 pass) or score / (S_q S_db) (8-bit pass). Error bound |q.p - s'| <= E:
//   fp16:  E = 1.1e-3 |q| max|p| + 1e-5   (fp16 input rounding 2^-10 |q||p|, fp16 subnormals, fp32 accumulation of the tensor core)
//   8-bit: q = q8/S_q + e_q, p = p8/S_db + e_p, integer accumulation is exact, so q.p - s' = (q8/S_q).e_p + e_q.p and
//          E = (|q| + |e_q|) max|e_p| + |e_q| max|p|  with the residual norms |e_q|, max|e_p| measured when the images were packed.
// Pruning: a candidate whose s' + E is below the second largest s' - E (minus the spread of |p|^2 and a rounding slack) cannot
// be one of the two nearest rows, so its exact distance is never computed — with 8 candidates per DB split that is most of them.
// Certificate: every row that is NOT a candidate scored <= T = final shared threshold of this query in the coarse pass, so
// its true squared distance is >= |q|^2 + min|p|^2 - 2 (T' + E); if that bound exceeds the exact 2nd-best candidate distance
// the two nearest rows are proven to be among the candidates. Uncertified queries go to the next tier: `flag_list` (up to
// flag_cap entries: the fp16 second-chance pass after an 8-bit pass) and beyond that / otherwise `exact_list` (exhaustive scan).
struct RerankArgs {
	const float *q; int Q;
	const int32_t *list; const int32_t *list_count; int list_cap;      // nullable: compact index li -> query list[li]
	const float *q_norm2, *q_scale, *q_err;                             // per QUERY id (q_scale / q_err: 8-bit pass only)
	const float *db;
	const uint32_t *cand_score; const int32_t *cand_row; int n_cand;    // per COMPACT index
	const uint32_t *g_tau;
	int kind; float db_scale, db_err_max, db_n2_min, db_n2_max; int64_t row_base;
	int32_t *nn_row; float *nn_dist;
	int32_t *flag_list, *flag_count; int flag_cap;                      // nullable
	int32_t *exact_list, *exact_count;
	unsigned long long *nn_key;
};
constexpr int kRerankMaxCand = kMaxSplits * (kTopK8 > kTopK * kCG ? kTopK8 : kTopK * kCG);

__global__ void __launch_bounds__(256)
k_match_rerank(const RerankArgs a) {
	__shared__ float qs[8][kD];
	__shared__ int16_t keep[8][kRerankMaxCand];
	const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
	const int li = blockIdx.x * 8 + w;
	int n = a.Q;
	if (a.list) { n = *a.list_count; n = n < a.list_cap ? n : a.list_cap; }
	if (li >= n) return;
	const int qi = a.list ? a.list[li] : li;
	for (int d = lane; d < kD; d += 32) qs[w][d] = a.q[(size_t)qi * kD + d];
	const float qn2 = a.q_norm2[qi];
	float unit = 1.f, E;
	if (a.kind == 1) {
		const float eq = a.q_err[qi];
		unit = 1.f / (a.q_scale[qi] * a.db_scale);
		E = ((sqrtf(qn2) + eq) * a.db_err_max + eq * sqrtf(a.db_n2_max)) * 1.001f + 1e-5f;
	} else {
		E = 1.1e-3f * sqrtf(qn2 * a.db_n2_max) + 1e-5f;
	}
	auto dot_of = [&](uint32_t bits) { return a.kind == 1 ? (float)(int32_t)bits * unit : __uint_as_float(bits); };   // 8-bit pass: the bits ARE the int32 score
	const uint32_t *cs = a.cand_score + (size_t)li * a.n_cand;
	const int32_t *cr = a.cand_row + (size_t)li * a.n_cand;
	// second largest score among the candidates
	float b0 = -CUDART_INF_F, b1 = -CUDART_INF_F;
	for (int c = lane; c < a.n_cand; c += 32)
		if (cr[c] >= 0) {
			const float s = dot_of(cs[c]);
			if (s > b0) { b1 = b0; b0 = s; } else if (s > b1) b1 = s;
		}
	for (int o = 16; o; o >>= 1) {
		const float o0 = __shfl_xor_sync(0xffffffffu, b0, o), o1 = __shfl_xor_sync(0xffffffffu, b1, o);
		if (o0 > b0) { b1 = fmaxf(b0, o1); b0 = o0; } else b1 = fmaxf(b1, o0);
	}
	// NaN scores / bounds keep everything (comparisons with NaN are false)
	const float cut = b1 - 2.f * E - 0.5f * (a.db_n2_max - a.db_n2_min) - 1e-4f;
	int n_keep = 0;
	for (int base = 0; base < a.n_cand; base += 32) {
		const int c = base + lane;
		const bool k = c < a.n_cand && cr[c] >= 0 && !(dot_of(cs[c]) < cut);
		const unsigned bal = __ballot_sync(0xffffffffu, k);
		if (k) keep[w][n_keep + __popc(bal & ((1u << lane) - 1))] = (int16_t)c;
		n_keep += __popc(bal);
	}
	__syncwarp();
	Top2 t = top2_empty();
	for (int j = lane; j < n_keep; j += 32) {
		const int32_t row = cr[keep[w][j]];
		const float4 *p = reinterpret_cast<const float4 *>(a.db + (size_t)row * kD);
		float dist = 0.f;
#pragma unroll 4
		for (int d4 = 0; d4 < kD / 4; d4++) {
			float4 v = __ldg(&p[d4]);
			float t0 = __fsub_rn(qs[w][4 * d4 + 0], v.x); dist = __fadd_rn(dist, __fmul_rn(t0, t0));
			float t1 = __fsub_rn(qs[w][4 * d4 + 1], v.y); dist = __fadd_rn(dist, __fmul_rn(t1, t1));
			float t2 = __fsub_rn(qs[w][4 * d4 + 2], v.z); dist = __fadd_rn(dist, __fmul_rn(t2, t2));
			float t3 = __fsub_rn(qs[w][4 * d4 + 3], v.w); dist = __fadd_rn(dist, __fmul_rn(t3, t3));
		}
		top2_push(t, dist, row);
	}
	top2_warp_reduce(t);
	if (lane == 0) {
		const uint32_t og = a.g_tau[li];
		// fp16 pass: no threshold ever published = every row is a candidate. 8-bit pass: the threshold starts at score 0 (rows
		// scoring <= 0 are never candidates), a published one is the int32 score in float bits (f2o of a non-negative float)
		const bool no_T = a.kind == 0 && og == 0;
		const float T = a.kind == 1 ? (float)(int32_t)(og & 0x7fffffffu) * unit : o2f(og);
		const float bound = qn2 + a.db_n2_min - 2.f * (T + E) - 1e-4f;
		const bool certified = (t.i1 >= 0) && (no_T || t.d1 < bound);
		a.nn_row[2 * qi] = t.i0 >= 0 ? (int32_t)(t.i0 + a.row_base) : -1;
		a.nn_row[2 * qi + 1] = t.i1 >= 0 ? (int32_t)(t.i1 + a.row_base) : -1;
		a.nn_dist[2 * qi] = t.d0; a.nn_dist[2 * qi + 1] = t.d1;
		if (!certified) {
			int slot = a.flag_list ? atomicAdd(a.flag_count, 1) : a.flag_cap;
			if (slot < a.flag_cap) a.flag_list[slot] = qi;
			else {
				a.exact_list[atomicAdd(a.exact_count, 1)] = qi;
				a.nn_key[2 * (size_t)qi] = ~0ull; a.nn_key[2 * (size_t)qi + 1] = ~0ull;
			}
		}
	}
}

// Two-smallest accumulator over 64-bit keys (distance bits << 32 | row): slot 0 takes every key by
// atomicMin; whichever of (old slot 0, key) loses goes to slot 1 by atomicMin. Keys are unique, the
// global minimum is never a loser and the global second minimum always is, so slot 1 ends as the 2nd.
__device__ __forceinline__ void key2_push(unsigned long long *slot, float d, int32_t row) {
	if (row < 0) return;
	unsigned long long key = ((unsigned long long)__float_as_uint(d) << 32) | (uint32_t)row;
	unsigned long long old = atomicMin(&slot[0], key);
	unsigned long long loser = old < key ? key : old;
	if (loser != ~0ull) atomicMin(&slot[1], loser);
}

// Exhaustive exact scan. Work item = (group of 8 listed queries, row chunk); persistent grid.
// Each thread walks rows (stride blockDim) of the chunk and carries the 8 queries' running sums through
// the descriptor in order, 16 dimensions at a time; a block-reduced top-2 per query is merged into the
// query's global two-smallest slots.
constexpr int kExactQ = 8;
constexpr int kExactThreads = 256;
constexpr int kMaxAnyD = 4096;          // longest descriptor the generic exact scan stages in shared memory (8 x 4096 floats = 128 KiB)
__global__ void __launch_bounds__(kExactThreads)
k_match_exact(const float *__restrict__ q, const int32_t *__restrict__ list, const int32_t *__restrict__ list_count, int list_all,
              const float *__restrict__ db, int64_t n_rows, int n_chunks, int chunk_rows,
              unsigned long long *__restrict__ nn_key) {
	__shared__ __align__(16) float qs[kExactQ][kD];
	__shared__ Top2 red[kExactQ][kExactThreads / 32];
	const int n_list = list ? *list_count : list_all;
	const int n_groups = (n_list + kExactQ - 1) / kExactQ;
	const int64_t n_items = (int64_t)n_groups * n_chunks;
	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	for (int64_t item = blockIdx.x; item < n_items; item += gridDim.x) {
		const int g = (int)(item / n_chunks), ch = (int)(item % n_chunks);
		__syncthreads();
		for (int x = threadIdx.x; x < kExactQ * kD; x += blockDim.x) {
			int k = x / kD, li = g * kExactQ + k;
			int qi = li < n_list ? (list ? list[li] : li) : -1;
			qs[k][x % kD] = qi >= 0 ? q[(size_t)qi * kD + (x % kD)] : 0.f;
		}
		__syncthreads();
		Top2 t[kExactQ];
#pragma unroll
		for (int k = 0; k < kExactQ; k++) t[k] = top2_empty();
		const int64_t r_lo = (int64_t)ch * chunk_rows;
		const int64_t r_hi = r_lo + chunk_rows < n_rows ? r_lo + chunk_rows : n_rows;
		for (int64_t row = r_lo + threadIdx.x; row < r_hi; row += blockDim.x) {
			const float4 *p = reinterpret_cast<const float4 *>(db + (size_t)row * kD);
			float dist[kExactQ];
#pragma unroll
			for (int k = 0; k < kExactQ; k++) dist[k] = 0.f;
#pragma unroll 2
			for (int b = 0; b < kD / 16; b++) {
				float4 v0 = __ldg(&p[4 * b]), v1 = __ldg(&p[4 * b + 1]), v2 = __ldg(&p[4 * b + 2]), v3 = __ldg(&p[4 * b + 3]);
				const float pv[16] = { v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w, v2.x, v2.y, v2.z, v2.w, v3.x, v3.y, v3.z, v3.w };
#pragma unroll
				for (int k = 0; k < kExactQ; k++) {
					const float4 *qq = reinterpret_cast<const float4 *>(&qs[k][16 * b]);
					float4 a0 = qq[0], a1 = qq[1], a2 = qq[2], a3 = qq[3];
					const float qv[16] = { a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w, a2.x, a2.y, a2.z, a2.w, a3.x, a3.y, a3.z, a3.w };
					float d = dist[k];
#pragma unroll
					for (int j = 0; j < 16; j++) { float tt = __fsub_rn(qv[j], pv[j]); d = __fadd_rn(d, __fmul_rn(tt, tt)); }
					dist[k] = d;
				}
			}
#pragma unroll
			for (int k = 0; k < kExactQ; k++) top2_push(t[k], dist[k], (int32_t)row);
		}
#pragma unroll
		for (int k = 0; k < kExactQ; k++) {
			top2_warp_reduce(t[k]);
			if (lane == 0) red[k][warp] = t[k];
		}
		__syncthreads();
		if (threadIdx.x < kExactQ) {
			const int k = threadIdx.x, li = g * kExactQ + k;
			if (li < n_list) {
				Top2 r = red[k][0];
				for (int ww = 1; ww < kExactThreads / 32; ww++) { top2_push(r, red[k][ww].d0, red[k][ww].i0); top2_push(r, red[k][ww].d1, red[k][ww].i1); }
				const int qi = list ? list[li] : li;
				key2_push(nn_key + 2 * (size_t)qi, r.d0, r.i0);
				key2_push(nn_key + 2 * (size_t)qi, r.d1, r.i1);
			}
		}
	}
}

// The same exhaustive scan for ANY descriptor length (MATCH_ANN_CPU's constructor takes DescriptorSize, e.g. SURF-64,
// moped2/libmoped/src/match/MATCH_ANN_CPU.hpp:113): runtime D, the group's queries staged in dynamic shared memory
// (kExactQ x D floats), every distance summed over d = 0..D-1 in order with unfused multiply and add like the 128-d kernel.
__global__ void __launch_bounds__(kExactThreads)
k_match_exact_any(const float *__restrict__ q, int D, const int32_t *__restrict__ list, const int32_t *__restrict__ list_count, int list_all,
                  const float *__restrict__ db, int64_t n_rows, int n_chunks, int chunk_rows, unsigned long long *__restrict__ nn_key) {
	extern __shared__ __align__(16) float qs_any[];            // [kExactQ][D]
	__shared__ Top2 red[kExactQ][kExactThreads / 32];
	const int n_list = list ? *list_count : list_all;
	const int n_groups = (n_list + kExactQ - 1) / kExactQ;
	const int64_t n_items = (int64_t)n_groups * n_chunks;
	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	const bool vec4 = (D & 3) == 0;
	for (int64_t item = blockIdx.x; item < n_items; item += gridDim.x) {
		const int g = (int)(item / n_chunks), ch = (int)(item % n_chunks);
		__syncthreads();
		for (int x = threadIdx.x; x < kExactQ * D; x += blockDim.x) {
			const int k = x / D, d = x - k * D, li = g * kExactQ + k;
			const int qi = li < n_list ? (list ? list[li] : li) : -1;
			qs_any[x] = qi >= 0 ? q[(size_t)qi * D + d] : 0.f;
		}
		__syncthreads();
		Top2 t[kExactQ];
#pragma unroll
		for (int k = 0; k < kExactQ; k++) t[k] = top2_empty();
		const int64_t r_lo = (int64_t)ch * chunk_rows;
		const int64_t r_hi = r_lo + chunk_rows < n_rows ? r_lo + chunk_rows : n_rows;
		for (int64_t row = r_lo + threadIdx.x; row < r_hi; row += blockDim.x) {
			const float *p = db + (size_t)row * D;
			float dist[kExactQ];
#pragma unroll
			for (int k = 0; k < kExactQ; k++) dist[k] = 0.f;
			if (vec4) {
				for (int d = 0; d < D; d += 4) {
					const float4 v = __ldg(reinterpret_cast<const float4 *>(p + d));
#pragma unroll
					for (int k = 0; k < kExactQ; k++) {
						const float4 a = *reinterpret_cast<const float4 *>(&qs_any[k * D + d]);
						float dd = dist[k], tt;
						tt = __fsub_rn(a.x, v.x); dd = __fadd_rn(dd, __fmul_rn(tt, tt));
						tt = __fsub_rn(a.y, v.y); dd = __fadd_rn(dd, __fmul_rn(tt, tt));
						tt = __fsub_rn(a.z, v.z); dd = __fadd_rn(dd, __fmul_rn(tt, tt));
						tt = __fsub_rn(a.w, v.w); dd = __fadd_rn(dd, __fmul_rn(tt, tt));
						dist[k] = dd;
					}
				}
			} else {
				for (int d = 0; d < D; d++) {
					const float v = __ldg(p + d);
#pragma unroll
					for (int k = 0; k < kExactQ; k++) { const float tt = __fsub_rn(qs_any[k * D + d], v); dist[k] = __fadd_rn(dist[k], __fmul_rn(tt, tt)); }
				}
			}
#pragma unroll
			for (int k = 0; k < kExactQ; k++) top2_push(t[k], dist[k], (int32_t)row);
		}
#pragma unroll
		for (int k = 0; k < kExactQ; k++) {
			top2_warp_reduce(t[k]);
			if (lane == 0) red[k][warp] = t[k];
		}
		__syncthreads();
		if (threadIdx.x < kExactQ) {
			const int k = threadIdx.x, li = g * kExactQ + k;
			if (li < n_list) {
				Top2 r = red[k][0];
				for (int ww = 1; ww < kExactThreads / 32; ww++) { top2_push(r, red[k][ww].d0, red[k][ww].i0); top2_push(r, red[k][ww].d1, red[k][ww].i1); }
				const int qi = list ? list[li] : li;
				key2_push(nn_key + 2 * (size_t)qi, r.d0, r.i0);
				key2_push(nn_key + 2 * (size_t)qi, r.d1, r.i1);
			}
		}
	}
}

// decode the two-smallest slots of every listed query into (global row id, distance)
__global__ void k_match_exact_decode(const int32_t *__restrict__ list, const int32_t *__restrict__ list_count, int list_all,
                                     const unsigned long long *__restrict__ nn_key, int64_t row_base,
                                     int32_t *__restrict__ nn_row, float *__restrict__ nn_dist) {
	const int n_list = list ? *list_count : list_all;
	for (int li = blockIdx.x * blockDim.x + threadIdx.x; li < n_list; li += gridDim.x * blockDim.x) {
		const int qi = list ? list[li] : li;
#pragma unroll
		for (int j = 0; j < 2; j++) {
			unsigned long long k = nn_key[2 * (size_t)qi + j];
			bool ok = k != ~0ull;
			nn_row[2 * qi + j] = ok ? (int32_t)((int64_t)(uint32_t)(k & 0xffffffffull) + row_base) : -1;
			nn_dist[2 * qi + j] = ok ? __uint_as_float((uint32_t)(k >> 32)) : 3.402823466e+38f;
		}
	}
}

// ratio test on squared distances, fp32 division like `ds[0]/ds[1] < Ratio` (MATCH_ANN_CPU.hpp:165)
__global__ void k_match_finalize(const int32_t *__restrict__ nn_row, const float *__restrict__ nn_dist, int Q, float ratio,
                                 uint8_t *__restrict__ accepted) {
	int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= Q) return;
	bool ok = nn_row[2 * i] >= 0 && nn_row[2 * i + 1] >= 0 && __fdiv_rn(nn_dist[2 * i], nn_dist[2 * i + 1]) < ratio;
	accepted[i] = ok ? 1 : 0;
}

// global top-2 over object shards: (smaller distance, then smaller global row id)
// shard s's rows / distances start `stride` elements after shard s-1's (2 Q for two separate arrays, 4 Q for packed blocks)
__global__ void k_match_merge(const int32_t *__restrict__ rows_all, const float *__restrict__ dist_all, size_t stride, int n_shards, int Q, float ratio,
                              int32_t *__restrict__ nn_row, float *__restrict__ nn_dist, uint8_t *__restrict__ accepted) {
	int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= Q) return;
	Top2 t = top2_empty();
	for (int s = 0; s < n_shards; s++) {
		size_t o = (size_t)s * stride + (size_t)i * 2;
		top2_push(t, dist_all[o], rows_all[o]);
		top2_push(t, dist_all[o + 1], rows_all[o + 1]);
	}
	nn_row[2 * i] = t.i0; nn_row[2 * i + 1] = t.i1;
	nn_dist[2 * i] = t.d0; nn_dist[2 * i + 1] = t.d1;
	accepted[i] = (t.i0 >= 0 && t.i1 >= 0 && __fdiv_rn(t.d0, t.d1) < ratio) ? 1 : 0;
}

__global__ void k_row_norm2(const float *__restrict__ src, int n, float *__restrict__ norm2) {
	int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	const float *p = src + (size_t)i * kD;
	float s = 0.f;
	for (int d = 0; d < kD; d++) s = fmaf(p[d], p[d], s);
	norm2[i] = s;
}

// =============================================================================================
// host side
// =============================================================================================
// Function attributes are PER DEVICE: called by mc_create for the context's device (a process may hold contexts on
// several GPUs), never behind a process-wide flag.
mc_status match_configure_device(mc_ctx *ctx) {
	MC_CUDA(cudaFuncSetAttribute(k_match_coarse<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kCoarseSmemBytes));
	MC_CUDA(cudaFuncSetAttribute(k_match_coarse<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kCoarseSmemBytes));
	MC_CUDA(cudaFuncSetAttribute(k_match_exact_any, cudaFuncAttributeMaxDynamicSharedMemorySize, kExactQ * kMaxAnyD * (int)sizeof(float)));
	return MC_OK;
}

// Both operand images of the database: fp16 (second-chance pass / fp16-only mode) and 8-bit with ONE scale for all rows
// (u8 when no element is negative — SIFT —, s8 otherwise), plus what the certificates need: min / max |p|^2, max |e_p|.
mc_status db_build_images(mc_ctx *ctx) {
	if (ctx->D != kD) return MC_OK;     // tensor path needs D == 128; other lengths use the exact scan
	ctx->n_tiles = (ctx->n_rows + kTileRows - 1) / kTileRows;
	MC_CUDA(cudaMalloc(&ctx->d_db_img, (size_t)ctx->n_tiles * kTileBytes));
	MC_CUDA(cudaMalloc(&ctx->d_db_img8, (size_t)ctx->n_tiles * kTile8Bytes));
	float *d_norm2 = nullptr, *d_mm = nullptr;
	int *d_am = nullptr;
	MC_CUDA(cudaMalloc(&d_norm2, sizeof(float) * (size_t)(ctx->n_rows + 1)));
	MC_CUDA(cudaMalloc(&d_mm, 2 * sizeof(float)));
	MC_CUDA(cudaMalloc(&d_am, 4 * sizeof(int)));
	const float init[2] = { 3.0e38f, 0.f };
	MC_CUDA(cudaMemcpyAsync(d_mm, init, sizeof init, cudaMemcpyHostToDevice, ctx->stream));
	MC_CUDA(cudaMemsetAsync(d_am, 0, 4 * sizeof(int), ctx->stream));
	int64_t total = ctx->n_tiles * 2048;
	k_pack_tiles<<<(unsigned)((total + 255) / 256), 256, 0, ctx->stream>>>(ctx->d_db, ctx->n_rows, ctx->n_tiles, ctx->d_db_img, d_norm2, nullptr, nullptr);
	MC_LAUNCH_CHECK();
	k_minmax<<<296, 256, 0, ctx->stream>>>(d_norm2, ctx->n_rows, d_mm);
	MC_LAUNCH_CHECK();
	k_absmax<<<592, 256, 0, ctx->stream>>>(ctx->d_db, ctx->n_rows * kD, d_am);
	MC_LAUNCH_CHECK();
	float mm[2];
	int am[4];
	MC_CUDA(cudaMemcpyAsync(mm, d_mm, sizeof mm, cudaMemcpyDeviceToHost, ctx->stream));
	MC_CUDA(cudaMemcpyAsync(am, d_am, sizeof am, cudaMemcpyDeviceToHost, ctx->stream));
	MC_CUDA(cudaStreamSynchronize(ctx->stream));
	ctx->db_norm2_min = mm[0]; ctx->db_norm2_max = mm[1];
	float absmax;
	memcpy(&absmax, &am[0], sizeof absmax);
	ctx->db_signed = am[1] != 0;
	ctx->db_scale = absmax > 0.f && absmax < 3.0e38f ? (ctx->db_signed ? 127.f : 255.f) / absmax : 0.f;
	k_pack_tiles_q8<<<(unsigned)ctx->n_tiles, 256, 0, ctx->stream>>>(ctx->d_db, ctx->n_rows, ctx->d_db_img8, 0, ctx->db_scale, ctx->db_signed ? 1 : 0,
	                                                              nullptr, nullptr, nullptr, nullptr, d_am + 2);
	MC_LAUNCH_CHECK();
	MC_CUDA(cudaMemcpyAsync(am, d_am, sizeof am, cudaMemcpyDeviceToHost, ctx->stream));
	MC_CUDA(cudaStreamSynchronize(ctx->stream));
	memcpy(&ctx->db_err_max, &am[2], sizeof(float));
	MC_CUDA(cudaFree(d_norm2));
	MC_CUDA(cudaFree(d_mm));
	MC_CUDA(cudaFree(d_am));
	return MC_OK;
}

static mc_status exact_scan(mc_ctx *ctx, const float *d_q, int Q, const int32_t *d_list, const int32_t *d_count, int32_t *d_nn_row, float *d_nn_dist) {
	// chunks: enough items to fill the machine even for a single group of queries
	int n_chunks = ctx->num_sms * 2;
	int chunk_rows = (int)((ctx->n_rows + n_chunks - 1) / n_chunks);
	if (chunk_rows < kExactThreads) chunk_rows = kExactThreads;
	n_chunks = (int)((ctx->n_rows + chunk_rows - 1) / chunk_rows);
	if (!d_list) MC_CUDA(cudaMemsetAsync(ctx->nn_key.p, 0xFF, sizeof(unsigned long long) * 2 * (size_t)Q, ctx->stream));
	if (ctx->D == kD)
		k_match_exact<<<ctx->num_sms * 4, kExactThreads, 0, ctx->stream>>>(d_q, d_list, d_count, Q, ctx->d_db, ctx->n_rows, n_chunks, chunk_rows,
		                                                                 (unsigned long long *)ctx->nn_key.p);
	else
		k_match_exact_any<<<ctx->num_sms * 4, kExactThreads, sizeof(float) * kExactQ * (size_t)ctx->D, ctx->stream>>>(
		    d_q, ctx->D, d_list, d_count, Q, ctx->d_db, ctx->n_rows, n_chunks, chunk_rows, (unsigned long long *)ctx->nn_key.p);
	MC_LAUNCH_CHECK();
	k_match_exact_decode<<<ctx->num_sms, 256, 0, ctx->stream>>>(d_list, d_count, Q, (const unsigned long long *)ctx->nn_key.p, ctx->row_base,
	                                                          d_nn_row, d_nn_dist);
	MC_LAUNCH_CHECK();
	return MC_OK;
}

// DB splits for n_mtiles query tiles on `ctas` persistent CTAs. Work item = (query tile, DB split), all items equally long,
// handed out dynamically. Few query tiles (one frame): one item per CTA, floor(ctas / tiles) splits. Many query tiles (frame
// batches): keep at least 8 splits so that every query has enough candidate lists for the certificate, and take the SMALLEST
// count in 8..16 whose last round is at least 97 % full (every split of a query starts one more list, i.e. costs insertions
// and candidates; a search for the best-filled last round up to 64 splits once picked 31 splits for 124 CTAs and made the
// pass 50 % slower).
static void choose_splits(const mc_ctx *ctx, int n_mtiles, int ctas, int &n_splits, int &tiles_per_split) {
	n_splits = ctas / n_mtiles;
	if (ctx->match_splits > 0) n_splits = ctx->match_splits;      // mc_set_option "match_splits": tuning override (the cascade stays exact)
	else if (n_splits < 8 && ctx->n_tiles <= 4800) {
		// shards up to ~600 k rows (the ranks of a 2..8-GPU job): 4 splits. Work items are handed out dynamically, so a ragged last round
		// costs little, while every split of a query starts two more cold candidate lists (insertions) and adds 16 candidates to the
		// re-rank; fewer than 4 sends too many queries to the fp16 second-chance pass. Whole MATCH pass, 128 000 queries, B200
		// (profiles/coarse_splits_r2b.md): 125 k rows 4.01 -> 3.42 ms, 500 k rows 9.42 -> 9.08 ms; at 1 M rows 4 / 6 / 9 splits are equal.
		n_splits = 4;
	} else if (n_splits < 8) {
		double best = -1.0;
		for (int sp = 8; sp <= 16; sp++) {
			const int64_t items = (int64_t)n_mtiles * sp;
			const int64_t rounds = (items + ctas - 1) / ctas;
			const double eff = (double)items / (double)(rounds * ctas);
			if (eff > best) { best = eff; n_splits = sp; }
			if (eff >= 0.97) { n_splits = sp; break; }
		}
	}
	if (n_splits < 1) n_splits = 1;
	if (n_splits > kMaxSplits) n_splits = kMaxSplits;
	if ((int64_t)n_splits > ctx->n_tiles) n_splits = (int)ctx->n_tiles;
	tiles_per_split = (int)((ctx->n_tiles + n_splits - 1) / n_splits);
	n_splits = (int)((ctx->n_tiles + tiles_per_split - 1) / tiles_per_split);
}

constexpr int kSecondChanceCap = 16384;     // queries the fp16 second-chance pass of the cascade takes (64 query tiles); more go to the exact scan

mc_status match_device(mc_ctx *ctx, const float *d_q, int Q, float ratio, int mode, int32_t *d_nn_row, float *d_nn_dist, uint8_t *d_accepted) {
	if (!ctx->d_db) { ctx->err = "mc_match: no database uploaded"; return MC_ERR_STATE; }
	if (Q <= 0) return MC_OK;
	MC_TRY(reserve(ctx, ctx->nn_key, sizeof(unsigned long long) * 2 * (size_t)Q));
	// the tensor-core path is built for 128-d descriptors (SIFT); any other DescriptorSize takes the exhaustive exact scan —
	// the same result by definition (MC_MATCH_TENSOR only ever promises the exact scan's bits)
	ctx->last_match_q = Q;
	ctx->last_match_tensor = !(mode == MC_MATCH_EXACT || ctx->D != kD);
	if (mode == MC_MATCH_EXACT || ctx->D != kD) {
		MC_TRY(exact_scan(ctx, d_q, Q, nullptr, nullptr, d_nn_row, d_nn_dist));
	} else {
		// Cascade: [8-bit coarse pass -> re-rank + certificate ->] fp16 coarse pass (of everything, or of the queries the 8-bit
		// certificate refused) -> re-rank + certificate -> exhaustive exact scan of what is still uncertified. Every tier
		// returns the exact scan's bits for the queries it certifies; nothing comes back to the host in between.
		const bool i8 = ctx->coarse_kind == 1 && ctx->db_scale > 0.f;
		const int n_mtiles = (Q + kMTile - 1) / kMTile;
		const int q_pad = n_mtiles * kMTile;
		// persistent CTAs: the SMs of the MATCH partition when the GPU is partitioned (the coarse kernel is then launched on that
		// partition's stream), otherwise all SMs minus match_reserve_sms
		int ctas = ctx->match_green_stream ? ctx->match_sms : ctx->num_sms - ctx->match_reserve_sms;
		if (ctas < 8) ctas = 8;
		cudaStream_t cs = ctx->match_green_stream ? ctx->match_green_stream : ctx->stream;
		auto fork = [&]() -> cudaError_t {
			if (!ctx->match_green_stream) return cudaSuccess;
			cudaError_t e = cudaEventRecord(ctx->ev_green[0], ctx->stream);
			return e != cudaSuccess ? e : cudaStreamWaitEvent(cs, ctx->ev_green[0], 0);
		};
		auto join = [&]() -> cudaError_t {
			if (!ctx->match_green_stream) return cudaSuccess;
			cudaError_t e = cudaEventRecord(ctx->ev_green[1], cs);
			return e != cudaSuccess ? e : cudaStreamWaitEvent(ctx->stream, ctx->ev_green[1], 0);
		};
		int n_splits, tiles_per_split;
		choose_splits(ctx, n_mtiles, ctas, n_splits, tiles_per_split);
		const int k1 = (i8 ? CoarseKind<1>::kK : CoarseKind<0>::kK) * kCG;     // candidates per (query, split)
		const int n_cand = n_splits * k1;
		MC_TRY(reserve(ctx, ctx->q_norm2, sizeof(float) * q_pad));
		MC_TRY(reserve(ctx, ctx->tau, sizeof(uint32_t) * q_pad));
		MC_TRY(reserve(ctx, ctx->cand_score, sizeof(uint32_t) * (size_t)q_pad * n_cand));
		MC_TRY(reserve(ctx, ctx->cand_row, sizeof(int32_t) * (size_t)q_pad * n_cand));
		MC_TRY(reserve(ctx, ctx->flag_list, sizeof(int32_t) * q_pad));          // exact-scan list
		MC_TRY(reserve(ctx, ctx->flag_count, 256));                             // [0] uncertified by the 8-bit pass, [1] exact-scan list length
		MC_CUDA(cudaMemsetAsync(ctx->tau.p, 0, sizeof(uint32_t) * q_pad, ctx->stream));
		MC_CUDA(cudaMemsetAsync(ctx->flag_count.p, 0, 4 * sizeof(int32_t), ctx->stream));   // + [2], [3]: work-item counters of the two coarse launches
		int32_t *d_counts = (int32_t *)ctx->flag_count.p;
		RerankArgs r;
		r.q = d_q; r.Q = Q; r.list = nullptr; r.list_count = nullptr; r.list_cap = 0;
		r.q_norm2 = (const float *)ctx->q_norm2.p; r.q_scale = nullptr; r.q_err = nullptr;
		r.db = ctx->d_db; r.db_scale = ctx->db_scale; r.db_err_max = ctx->db_err_max; r.db_n2_min = ctx->db_norm2_min; r.db_n2_max = ctx->db_norm2_max;
		r.row_base = ctx->row_base; r.nn_row = d_nn_row; r.nn_dist = d_nn_dist;
		r.exact_list = (int32_t *)ctx->flag_list.p; r.exact_count = d_counts + 1; r.nn_key = (unsigned long long *)ctx->nn_key.p;
		CoarseArgs c;
		c.n_tiles = ctx->n_tiles; c.n_rows = ctx->n_rows; c.b_signed = ctx->db_signed ? 1u : 0u;
		int cap2 = 0;
		if (i8) {
			cap2 = q_pad < kSecondChanceCap ? q_pad : kSecondChanceCap;
			MC_TRY(reserve(ctx, ctx->q_img8, (size_t)n_mtiles * 2 * kTile8Bytes));
			MC_TRY(reserve(ctx, ctx->q_signed, (size_t)n_mtiles * 2));
			MC_TRY(reserve(ctx, ctx->q_scale, sizeof(float) * q_pad));
			MC_TRY(reserve(ctx, ctx->q_err, sizeof(float) * q_pad));
			MC_TRY(reserve(ctx, ctx->flag_list2, sizeof(int32_t) * cap2));      // second-chance list
			k_pack_tiles_q8<<<n_mtiles * 2, 256, 0, ctx->stream>>>(d_q, Q, (uint8_t *)ctx->q_img8.p, 1, 0.f, 0, (uint8_t *)ctx->q_signed.p,
			                                                    (float *)ctx->q_scale.p, (float *)ctx->q_err.p, (float *)ctx->q_norm2.p, nullptr);
			MC_LAUNCH_CHECK();
			c.q_img = (const uint8_t *)ctx->q_img8.p; c.db_img = ctx->d_db_img8;
			c.tiles_per_split = tiles_per_split; c.n_splits = n_splits; c.n_mtiles = n_mtiles; c.q_count = nullptr;
			c.a_signed = (const uint8_t *)ctx->q_signed.p; c.stagger = ctx->match_stagger; c.item_counter = (uint32_t *)d_counts + 2;
			c.g_tau = (uint32_t *)ctx->tau.p; c.cand_score = (uint32_t *)ctx->cand_score.p; c.cand_row = (int32_t *)ctx->cand_row.p;
			const int grid = (int64_t)n_mtiles * n_splits < ctas ? n_mtiles * n_splits : ctas;
			MC_CUDA(fork());
			if (ctx->profile) MC_CUDA(cudaEventRecord(ctx->ev_coarse[0], cs));
			k_match_coarse<1><<<grid, kCoarseThreads, kCoarseSmemBytes, cs>>>(c);
			MC_LAUNCH_CHECK();
			if (ctx->profile) { MC_CUDA(cudaEventRecord(ctx->ev_coarse[1], cs)); ctx->ev_valid = true; }
			MC_CUDA(join());
			r.kind = 1; r.q_scale = (const float *)ctx->q_scale.p; r.q_err = (const float *)ctx->q_err.p;
			r.cand_score = (const uint32_t *)ctx->cand_score.p; r.cand_row = (const int32_t *)ctx->cand_row.p; r.n_cand = n_cand;
			r.g_tau = (const uint32_t *)ctx->tau.p;
			r.flag_list = (int32_t *)ctx->flag_list2.p; r.flag_count = d_counts; r.flag_cap = cap2;
			k_match_rerank<<<(Q + 7) / 8, 256, 0, ctx->stream>>>(r);
			MC_LAUNCH_CHECK();
		}
		// fp16 pass: all queries (fp16-only mode) or the second-chance list
		{
			const int m2 = i8 ? cap2 / kMTile : n_mtiles;
			int sp2 = n_splits, tps2 = tiles_per_split;
			if (i8) { sp2 = kMaxSplits; if ((int64_t)sp2 > ctx->n_tiles) sp2 = (int)ctx->n_tiles; tps2 = (int)((ctx->n_tiles + sp2 - 1) / sp2); sp2 = (int)((ctx->n_tiles + tps2 - 1) / tps2); }
			const int n_cand2 = sp2 * CoarseKind<0>::kK * kCG;
			DevBuf &tau2 = i8 ? ctx->tau2 : ctx->tau, &cs2 = i8 ? ctx->cand_score2 : ctx->cand_score, &cr2 = i8 ? ctx->cand_row2 : ctx->cand_row;
			if (i8) {
				MC_TRY(reserve(ctx, tau2, sizeof(uint32_t) * (size_t)m2 * kMTile));
				MC_TRY(reserve(ctx, cs2, sizeof(uint32_t) * (size_t)m2 * kMTile * n_cand2));
				MC_TRY(reserve(ctx, cr2, sizeof(int32_t) * (size_t)m2 * kMTile * n_cand2));
				MC_CUDA(cudaMemsetAsync(tau2.p, 0, sizeof(uint32_t) * (size_t)m2 * kMTile, ctx->stream));
			}
			MC_TRY(reserve(ctx, ctx->q_img, (size_t)m2 * 2 * kTileBytes));
			const int64_t total = (int64_t)m2 * 2 * 2048;
			k_pack_tiles<<<(unsigned)((total + 255) / 256), 256, 0, ctx->stream>>>(d_q, Q, (int64_t)m2 * 2, (__half *)ctx->q_img.p,
			                                                                      i8 ? nullptr : (float *)ctx->q_norm2.p,
			                                                                      i8 ? (const int32_t *)ctx->flag_list2.p : nullptr, i8 ? d_counts : nullptr);
			MC_LAUNCH_CHECK();
			c.q_img = (const uint8_t *)ctx->q_img.p; c.db_img = (const uint8_t *)ctx->d_db_img;
			c.tiles_per_split = tps2; c.n_splits = sp2; c.n_mtiles = m2; c.q_count = i8 ? d_counts : nullptr; c.a_signed = nullptr; c.stagger = ctx->match_stagger; c.item_counter = (uint32_t *)d_counts + 3;
			c.g_tau = (uint32_t *)tau2.p; c.cand_score = (uint32_t *)cs2.p; c.cand_row = (int32_t *)cr2.p;
			const int grid = (int64_t)m2 * sp2 < ctas ? m2 * sp2 : ctas;
			MC_CUDA(fork());
			if (!i8 && ctx->profile) MC_CUDA(cudaEventRecord(ctx->ev_coarse[0], cs));
			k_match_coarse<0><<<grid, kCoarseThreads, kCoarseSmemBytes, cs>>>(c);
			MC_LAUNCH_CHECK();
			if (!i8 && ctx->profile) { MC_CUDA(cudaEventRecord(ctx->ev_coarse[1], cs)); ctx->ev_valid = true; }
			MC_CUDA(join());
			r.kind = 0; r.q_scale = nullptr; r.q_err = nullptr;
			r.list = i8 ? (const int32_t *)ctx->flag_list2.p : nullptr; r.list_count = i8 ? d_counts : nullptr; r.list_cap = cap2;
			r.cand_score = (const uint32_t *)cs2.p; r.cand_row = (const int32_t *)cr2.p; r.n_cand = n_cand2; r.g_tau = (const uint32_t *)tau2.p;
			r.flag_list = nullptr; r.flag_count = nullptr; r.flag_cap = 0;
			k_match_rerank<<<((i8 ? cap2 : Q) + 7) / 8, 256, 0, ctx->stream>>>(r);
			MC_LAUNCH_CHECK();
		}
		MC_TRY(exact_scan(ctx, d_q, Q, (const int32_t *)ctx->flag_list.p, d_counts + 1, d_nn_row, d_nn_dist));
		ctx->last_stats[2] = n_cand; ctx->last_stats[3] = n_splits;
	}
	k_match_finalize<<<(Q + 255) / 256, 256, 0, ctx->stream>>>(d_nn_row, d_nn_dist, Q, ratio, d_accepted);
	MC_LAUNCH_CHECK();
	return MC_OK;
}

mc_status match_merge_device(mc_ctx *ctx, const int32_t *rows_all, const float *dist_all, size_t stride, int n_shards, int Q, float ratio,
                             int32_t *d_nn_row, float *d_nn_dist, uint8_t *d_accepted) {
	if (Q <= 0) return MC_OK;
	k_match_merge<<<(Q + 255) / 256, 256, 0, ctx->stream>>>(rows_all, dist_all, stride, n_shards, Q, ratio, d_nn_row, d_nn_dist, d_accepted);
	MC_LAUNCH_CHECK();
	return MC_OK;
}

} // namespace mc
