// undistort_host.cpp — moped_b200/csrc/undistort.cuh (the remap table builder of mc_set_undistortion and the per-pixel function of
// k_undistort) compiled by g++ -ffp-contract=off for tests/test_undistort_host.py.
#include <cstddef>
#include "../../moped_b200/csrc/undistort.cuh"

extern "C" {

void uh_maps(const float *K, const float *kc, int n_kc, int H, int W, float *mx, float *my) { mc::undistort_maps(K, kc, n_kc, H, W, mx, my); }

void uh_entries(int n, const float *mx, const float *my, int16_t *sx, int16_t *sy, uint16_t *frac) {
	for (int i = 0; i < n; i++) {
		const mc::RemapEntry e = mc::remap_entry(mx[i], my[i]);
		sx[i] = e.sx; sy[i] = e.sy; frac[i] = e.frac;
	}
}

void uh_weights(uint16_t *w) { mc::remap_weights((mc::RemapWeights *)w); }

// the table of mc_set_undistortion applied to B images with remap_pixel, as k_undistort applies it
void uh_undistort(const float *K, const float *kc, int n_kc, const uint8_t *src, int B, int H, int W, uint8_t *out) {
	const size_t npx = (size_t)H * W;
	float *mx = new float[npx], *my = new float[npx];
	mc::undistort_maps(K, kc, n_kc, H, W, mx, my);
	mc::RemapWeights tab[mc::kInterTab * mc::kInterTab];
	mc::remap_weights(tab);
	for (size_t i = 0; i < npx; i++) {
		const mc::RemapEntry e = mc::remap_entry(mx[i], my[i]);
		for (int b = 0; b < B; b++) out[b * npx + i] = mc::remap_pixel(src + b * npx, H, W, e, tab[e.frac]);
	}
	delete[] mx;
	delete[] my;
}

} // extern "C"
