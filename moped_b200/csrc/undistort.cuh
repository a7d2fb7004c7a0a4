// undistort.cuh — UNDISTORTED_IMAGE (moped's UTIL_UNDISTORT: cvInitUndistortMap + cvRemap with CV_INTER_LINEAR +
// CV_WARP_FILL_OUTLIERS, fill value 0) for 8-bit gray images. The host builds one remap table per camera (double precision, in
// the order of OpenCV's scalar loop); the device only does integer arithmetic on it. Included by undistort.cu and, compiled by g++
// with -ffp-contract=off, by tests/cpp/undistort_host.cpp.
#pragma once

#include <stdint.h>
#include <math.h>
#include <limits.h>

#if defined(__CUDACC__)
#define MC_UND_HD __host__ __device__ __forceinline__
#else
#define MC_UND_HD inline
#endif

namespace mc {

constexpr int kInterBits = 5;                      // OpenCV's INTER_BITS: 1/32-pixel fractions
constexpr int kInterTab = 1 << kInterBits;
constexpr int kRemapCoefBits = 15;                 // INTER_REMAP_COEF_BITS: weights sum to 2^15
constexpr int kUndistortMaxSize = 32767;           // source coordinates are int16 (cvRemap's fixed-point map)

// One output pixel: the top-left source neighbour (saturated to int16) and the fraction index (fy * 32 + fx).
struct alignas(8) RemapEntry {
	int16_t sx, sy;
	uint16_t frac, pad;
};
// Bilinear weights of one fraction, for the neighbours (x, y), (x+1, y), (x, y+1), (x+1, y+1). At most 2^15, so unsigned.
struct alignas(8) RemapWeights {
	uint16_t w[4];
};

// cvInitUndistortMap(K, kc, mapx, mapy) with newCameraMatrix = K and R = I (initUndistortRectifyMap's scalar loop). K = (fx, fy,
// cx, cy) and kc = (k1, k2, p1, p2[, k3]) widened from float; every step in double, multiply and add kept separate.
inline void undistort_maps(const float *K4, const float *kc, int n_kc, int H, int W, float *mx, float *my) {
	const double fx = K4[0], fy = K4[1], u0 = K4[2], v0 = K4[3];
	const double k1 = kc[0], k2 = kc[1], p1 = kc[2], p2 = kc[3], k3 = n_kc > 4 ? kc[4] : 0.0;
	// iR = K^-1 as Matx33d::inv(DECOMP_LU) computes a 3x3 inverse: cofactors times 1 / det
	const double a[3][3] = {{fx, 0.0, u0}, {0.0, fy, v0}, {0.0, 0.0, 1.0}};
	const double det = a[0][0] * (a[1][1] * a[2][2] - a[2][1] * a[1][2]) - a[0][1] * (a[1][0] * a[2][2] - a[2][0] * a[1][2]) +
	                   a[0][2] * (a[1][0] * a[2][1] - a[2][0] * a[1][1]);
	const double d = 1.0 / det;
	double ir[9];
	ir[0] = (a[1][1] * a[2][2] - a[1][2] * a[2][1]) * d;
	ir[1] = (a[0][2] * a[2][1] - a[0][1] * a[2][2]) * d;
	ir[2] = (a[0][1] * a[1][2] - a[0][2] * a[1][1]) * d;
	ir[3] = (a[1][2] * a[2][0] - a[1][0] * a[2][2]) * d;
	ir[4] = (a[0][0] * a[2][2] - a[0][2] * a[2][0]) * d;
	ir[5] = (a[0][2] * a[1][0] - a[0][0] * a[1][2]) * d;
	ir[6] = (a[1][0] * a[2][1] - a[1][1] * a[2][0]) * d;
	ir[7] = (a[0][1] * a[2][0] - a[0][0] * a[2][1]) * d;
	ir[8] = (a[0][0] * a[1][1] - a[0][1] * a[1][0]) * d;
	for (int i = 0; i < H; i++) {
		double _x = i * ir[1] + ir[2], _y = i * ir[4] + ir[5], _w = i * ir[7] + ir[8];
		for (int j = 0; j < W; j++, _x += ir[0], _y += ir[3], _w += ir[6]) {     // a running sum, as OpenCV's loop
			const double w = 1.0 / _w, x = _x * w, y = _y * w;
			const double x2 = x * x, y2 = y * y, r2 = x2 + y2, _2xy = 2 * x * y;
			const double kr = (1 + ((k3 * r2 + k2) * r2 + k1) * r2) / (1 + ((0 * r2 + 0) * r2 + 0) * r2);
			const double u = fx * (x * kr + p1 * _2xy + p2 * (r2 + 2 * x2)) + u0;
			const double v = fy * (y * kr + p1 * (r2 + 2 * y2) + p2 * _2xy) + v0;
			mx[(size_t)i * W + j] = (float)u;
			my[(size_t)i * W + j] = (float)v;
		}
	}
}

// cvRound(32 * m) saturated to int: half to even (the default rounding mode); NaN maps to INT_MIN, which lies outside any image.
inline int remap_fixed(float m) {
	const double v = (double)m * kInterTab;
	if (!(v == v)) return INT_MIN;
	const double r = nearbyint(v);
	return r >= 2147483647.0 ? INT_MAX : r <= -2147483648.0 ? INT_MIN : (int)r;
}

inline int16_t sat_i16(int v) { return (int16_t)(v > 32767 ? 32767 : v < -32768 ? -32768 : v); }

// cvRemap's conversion of a float map entry (u, v) to its fixed-point form
inline RemapEntry remap_entry(float u, float v) {
	const int X = remap_fixed(u), Y = remap_fixed(v);
	RemapEntry e;
	e.sx = sat_i16(X >> kInterBits);
	e.sy = sat_i16(Y >> kInterBits);
	e.frac = (uint16_t)((Y & (kInterTab - 1)) * kInterTab + (X & (kInterTab - 1)));
	e.pad = 0;
	return e;
}

// OpenCV's initInterTab2D(INTER_LINEAR, fixed point): float products of (1 - b, b) x (1 - a, a), each rounded to 2^15; a set that
// does not sum to 2^15 gives the difference back through its largest entry (sum short) or its smallest (sum over).
inline void remap_weights(RemapWeights *tab) {
	for (int i = 0; i < kInterTab; i++) {
		for (int j = 0; j < kInterTab; j++) {
			const float b = i * (1.f / kInterTab), a = j * (1.f / kInterTab);
			const float cy[2] = {1.f - b, b}, cx[2] = {1.f - a, a};
			int t[4], sum = 0;
			for (int k1 = 0; k1 < 2; k1++)
				for (int k2 = 0; k2 < 2; k2++) {
					const float p = cy[k1] * cx[k2];
					t[k1 * 2 + k2] = (int)nearbyint((double)(p * (float)(1 << kRemapCoefBits)));
					sum += t[k1 * 2 + k2];
				}
			const int diff = sum - (1 << kRemapCoefBits);
			if (diff) {
				int lo = 0, hi = 0;
				for (int k = 1; k < 4; k++) {
					if (t[k] < t[lo]) lo = k;
					if (t[k] > t[hi]) hi = k;
				}
				t[diff < 0 ? hi : lo] -= diff;
			}
			for (int k = 0; k < 4; k++) tab[i * kInterTab + j].w[k] = (uint16_t)t[k];
		}
	}
}

template <class T> MC_UND_HD T und_load(const T *p) {
#if defined(__CUDA_ARCH__)
	return __ldg(p);
#else
	return *p;
#endif
}

// One output pixel of cvRemap (bilinear, constant border 0): a neighbour outside the H x W source reads 0.
MC_UND_HD uint8_t remap_pixel(const uint8_t *src, int H, int W, RemapEntry e, const RemapWeights &wt) {
	const int x0 = e.sx, y0 = e.sy;
	const bool cx0 = (unsigned)x0 < (unsigned)W, cx1 = (unsigned)(x0 + 1) < (unsigned)W;
	const bool cy0 = (unsigned)y0 < (unsigned)H, cy1 = (unsigned)(y0 + 1) < (unsigned)H;
	const int64_t i0 = (int64_t)y0 * W + x0, i1 = i0 + W;          // indices, dereferenced only when inside
	const int p00 = cy0 && cx0 ? und_load(src + i0) : 0, p01 = cy0 && cx1 ? und_load(src + i0 + 1) : 0;
	const int p10 = cy1 && cx0 ? und_load(src + i1) : 0, p11 = cy1 && cx1 ? und_load(src + i1 + 1) : 0;
	const int s = wt.w[0] * p00 + wt.w[1] * p01 + wt.w[2] * p10 + wt.w[3] * p11;
	const int r = (s + (1 << (kRemapCoefBits - 1))) >> kRemapCoefBits;
	return (uint8_t)(r > 255 ? 255 : r);
}

} // namespace mc
