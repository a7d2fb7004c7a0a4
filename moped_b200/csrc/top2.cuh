// top2.cuh — the two nearest rows of a query as the reference keeps them (smaller squared distance first, then smaller global row
// id), shared by the exact re-rank and scan (match.cu), the merge of object shards (match.cu) and moped3d's merged MATCH (adaptive.cu).
#pragma once
#include <stdint.h>

namespace mc {

struct Top2 {
	float d0, d1;
	int32_t i0, i1;
};
__device__ __forceinline__ bool closer(float d, int32_t i, float e, int32_t j) { return d < e || (d == e && (uint32_t)i < (uint32_t)j); }
__device__ __forceinline__ void top2_push(Top2 &t, float d, int32_t i) {
	if (i < 0) return;
	if (closer(d, i, t.d0, t.i0)) { t.d1 = t.d0; t.i1 = t.i0; t.d0 = d; t.i0 = i; }
	else if (closer(d, i, t.d1, t.i1)) { t.d1 = d; t.i1 = i; }
}
__device__ __forceinline__ void top2_warp_reduce(Top2 &t) {
#pragma unroll
	for (int o = 16; o; o >>= 1) {
		float d0 = __shfl_xor_sync(0xffffffffu, t.d0, o), d1 = __shfl_xor_sync(0xffffffffu, t.d1, o);
		int32_t i0 = __shfl_xor_sync(0xffffffffu, t.i0, o), i1 = __shfl_xor_sync(0xffffffffu, t.i1, o);
		top2_push(t, d0, i0);
		top2_push(t, d1, i1);
	}
}
__device__ __forceinline__ Top2 top2_empty() {
	Top2 t; t.d0 = t.d1 = 3.402823466e+38f /* PQ_NULL_KEY = ANN_DIST_INF: a missing neighbour */; t.i0 = t.i1 = -1; return t;
}

} // namespace mc
