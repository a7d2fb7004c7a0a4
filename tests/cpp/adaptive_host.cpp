// adaptive_host.cpp — moped_b200/csrc/adaptive_threshold.cuh (the acceptance rule of moped3d's depth-adaptive MATCH step, as the
// device kernel k_match_finalize_adaptive evaluates it) compiled by g++ -ffp-contract=off for tests/test_match_adaptive_frames_host.py.
#include <cstddef>     // size_t for include/moped_cuda.h
#include "../../moped_b200/csrc/adaptive_threshold.cuh"

extern "C" {

// per feature i: model[i] selects the curve; outputs the curve value at depth[i], the blended threshold and the accept decision
void ah_eval(int n, const mc_adaptive_model *curves, const int32_t *model, const float *depth, const float *fill, const float *d0, const float *d1,
             float maximum_depth, float default_depth, float cauchy_scale, float *curve, float *threshold, uint8_t *accept) {
	mc::AdaptiveParams P;
	P.maximum_depth = maximum_depth; P.default_depth = default_depth; P.cauchy_scale = cauchy_scale;
	for (int i = 0; i < n; i++) {
		const mc_adaptive_model &c = curves[model[i]];
		curve[i] = mc::ratio_curve(c, depth[i], maximum_depth);
		threshold[i] = mc::adaptive_threshold(c, depth[i], fill[i], P);
		accept[i] = mc::adaptive_accept(c, depth[i], fill[i], d0[i], d1[i], P) ? 1 : 0;
	}
}

void ah_pixel(int n, const float *xy, int width, int height, int32_t *px) {
	for (int i = 0; i < n; i++) px[i] = mc::adaptive_pixel(xy[2 * i], xy[2 * i + 1], width, height);
}

} // extern "C"
