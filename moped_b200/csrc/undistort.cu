// undistort.cu — UNDISTORTED_IMAGE on the device (moped's UTIL_UNDISTORT: cvInitUndistortMap + cvRemap, bilinear, constant
// border 0), registered before SIFT in both moped2 and moped3d pipelines. Per camera the host builds the remap table once
// (undistort.cuh, compiled with -ffp-contract=off so that its doubles round like OpenCV's scalar loop) and the kernel only does
// integer arithmetic: one table entry and four source bytes per output pixel.
#include "common.cuh"
#include "undistort.cuh"

#include <cmath>
#include <vector>

namespace mc {

constexpr int kUndBlockX = 32, kUndBlockY = 8, kUndPix = 4;     // a thread writes 4 consecutive pixels of one row

// Image z of a batch belongs to camera z % n_cameras; a camera without a table (null map) has its images copied through.
struct UndistortMaps {
	const RemapEntry *map[kUndistortCameras];
};

// grid (columns / 128, rows / 8, images); the weight table (the same for every camera) is copied to shared memory by every block
__global__ void __launch_bounds__(kUndBlockX * kUndBlockY) k_undistort(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst,
                                                                       const __grid_constant__ UndistortMaps maps, int n_cameras,
                                                                       const RemapWeights *__restrict__ wtab, int H, int W, int vec4) {
	__shared__ RemapWeights w[kInterTab * kInterTab];
	const int tid = threadIdx.y * kUndBlockX + threadIdx.x;
	for (int i = tid; i < kInterTab * kInterTab; i += kUndBlockX * kUndBlockY) w[i] = wtab[i];
	__syncthreads();
	const int y = blockIdx.y * kUndBlockY + threadIdx.y, x0 = (blockIdx.x * kUndBlockX + threadIdx.x) * kUndPix;
	if (y >= H || x0 >= W) return;
	const size_t plane = (size_t)H * W;
	const uint8_t *img = src + blockIdx.z * plane;
	uint8_t *out = dst + blockIdx.z * plane + (size_t)y * W + x0;
	const RemapEntry *map = maps.map[blockIdx.z % n_cameras];
	const int n = min(kUndPix, W - x0);
	uint8_t px[kUndPix];
	if (map) {
		const RemapEntry *m = map + (size_t)y * W + x0;
#pragma unroll
		for (int k = 0; k < kUndPix; k++) {
			if (k < n) {
				const RemapEntry e = m[k];
				px[k] = remap_pixel(img, H, W, e, w[e.frac]);
			}
		}
	} else {
		const uint8_t *in = img + (size_t)y * W + x0;
#pragma unroll
		for (int k = 0; k < kUndPix; k++)
			if (k < n) px[k] = und_load(in + k);
	}
	if (vec4 && n == kUndPix) {
		*(uint32_t *)out = (uint32_t)px[0] | (uint32_t)px[1] << 8 | (uint32_t)px[2] << 16 | (uint32_t)px[3] << 24;
	} else {
		for (int k = 0; k < n; k++) out[k] = px[k];
	}
}

static bool finite_all(const float *v, int n) {
	for (int i = 0; i < n; i++)
		if (!std::isfinite(v[i])) return false;
	return true;
}

// The camera's table, or an error: MC_ERR_ARG for a bad camera or a size other than the table's, MC_ERR_STATE without a table.
static mc_status camera_table(mc_ctx *ctx, const char *who, int camera, int H, int W, const UndistortTable **out) {
	if (camera < 0 || camera >= kUndistortCameras) {
		ctx->err = std::string(who) + ": camera must be in 0.." + std::to_string(kUndistortCameras - 1);
		return MC_ERR_ARG;
	}
	const UndistortTable &t = ctx->undistort[camera];
	if (!t.d_map) { ctx->err = std::string(who) + ": no undistortion set for camera " + std::to_string(camera) + " (mc_set_undistortion)"; return MC_ERR_STATE; }
	if (H != t.height || W != t.width) {
		ctx->err = std::string(who) + ": images are " + std::to_string(W) + "x" + std::to_string(H) + ", camera " + std::to_string(camera) +
		           "'s table is " + std::to_string(t.width) + "x" + std::to_string(t.height);
		return MC_ERR_ARG;
	}
	*out = &t;
	return MC_OK;
}

// One launch for a batch of n_cameras-camera frames; wtab is the weight table of any camera's allocation.
static mc_status launch_undistort(mc_ctx *ctx, const UndistortMaps &maps, int n_cameras, const RemapWeights *wtab, const uint8_t *d_in, int B,
                                  int H, int W, uint8_t *d_out) {
	const dim3 block(kUndBlockX, kUndBlockY);
	const dim3 grid((W + kUndBlockX * kUndPix - 1) / (kUndBlockX * kUndPix), (H + kUndBlockY - 1) / kUndBlockY, B);
	const int vec4 = W % 4 == 0 && (uintptr_t)d_out % 4 == 0;
	k_undistort<<<grid, block, 0, ctx->stream>>>(d_in, d_out, maps, n_cameras, wtab, H, W, vec4);
	MC_LAUNCH_CHECK();
	return MC_OK;
}

static const RemapEntry *table_map(const UndistortTable &t) { return (const RemapEntry *)t.d_map; }
static const RemapWeights *table_weights(const UndistortTable &t) { return (const RemapWeights *)(table_map(t) + (size_t)t.height * t.width); }

static mc_status launch_camera(mc_ctx *ctx, const UndistortTable &t, const uint8_t *d_in, int B, uint8_t *d_out) {
	UndistortMaps maps = {};
	maps.map[0] = table_map(t);
	return launch_undistort(ctx, maps, 1, table_weights(t), d_in, B, t.height, t.width, d_out);
}

mc_status undistort_check_rig(mc_ctx *ctx, const char *who, int n_cameras, const int *H, const int *W, bool *has) {
	for (int c = 0; c < n_cameras; c++) {
		const UndistortTable &t = ctx->undistort[c];
		has[c] = t.d_map != nullptr;
		if (!has[c]) continue;
		if (t.height != H[c] || t.width != W[c]) {
			ctx->err = std::string(who) + ": images are " + std::to_string(W[c]) + "x" + std::to_string(H[c]) + ", camera " + std::to_string(c) +
			           "'s undistortion table is " + std::to_string(t.width) + "x" + std::to_string(t.height);
			return MC_ERR_ARG;
		}
	}
	return MC_OK;
}

mc_status undistort_rig_device(mc_ctx *ctx, const int *cameras, int n_cameras, const uint8_t *d_in, int B, int H, int W, uint8_t *d_out) {
	UndistortMaps maps = {};
	const RemapWeights *wtab = nullptr;
	for (int j = 0; j < n_cameras; j++) {
		const UndistortTable &t = ctx->undistort[cameras[j]];
		if (!t.d_map) continue;
		maps.map[j] = table_map(t);
		wtab = table_weights(t);
	}
	if (!wtab) { ctx->err = "undistort: no camera of the rig has an undistortion table"; return MC_ERR_STATE; }
	return launch_undistort(ctx, maps, n_cameras, wtab, d_in, B, H, W, d_out);
}

} // namespace mc

using namespace mc;

extern "C" mc_status mc_set_undistortion(mc_ctx *ctx, int camera, const float *K, const float *kc, int n_kc, int height, int width) {
	if (!ctx) return MC_ERR_ARG;
	auto fail = [&](const std::string &msg) { ctx->err = "mc_set_undistortion: " + msg; return MC_ERR_ARG; };
	if (camera < 0 || camera >= kUndistortCameras) return fail("camera must be in 0.." + std::to_string(kUndistortCameras - 1));
	UndistortTable &t = ctx->undistort[camera];
	if (!kc) {                    // clear
		MC_CUDA(cudaSetDevice(ctx->device));
		MC_CUDA(cudaStreamSynchronize(ctx->stream));
		MC_CUDA(cudaFree(t.d_map));
		t = UndistortTable{};
		return MC_OK;
	}
	if (!K) return fail("K is NULL");
	if (n_kc != 4 && n_kc != 5) return fail("n_kc must be 4 or 5");
	if (!finite_all(K, 4) || !finite_all(kc, n_kc) || K[0] == 0.f || K[1] == 0.f) return fail("K and kc must be finite, fx and fy non-zero");
	if (height < 8 || width < 8 || height > kUndistortMaxSize || width > kUndistortMaxSize)
		return fail("height and width must be in 8.." + std::to_string(kUndistortMaxSize));
	const size_t npx = (size_t)height * width;
	std::vector<float> mx(npx), my(npx);
	undistort_maps(K, kc, n_kc, height, width, mx.data(), my.data());
	std::vector<RemapEntry> h((npx * sizeof(RemapEntry) + sizeof(RemapWeights) * kInterTab * kInterTab) / sizeof(RemapEntry));
	for (size_t i = 0; i < npx; i++) h[i] = remap_entry(mx[i], my[i]);
	remap_weights((RemapWeights *)(h.data() + npx));     // the weight table follows the map in the same allocation
	MC_CUDA(cudaSetDevice(ctx->device));
	void *d = nullptr;
	MC_CUDA(cudaMalloc(&d, h.size() * sizeof(RemapEntry)));
	cudaError_t e = cudaMemcpy(d, h.data(), h.size() * sizeof(RemapEntry), cudaMemcpyHostToDevice);
	if (e != cudaSuccess) { cudaFree(d); ctx->err = std::string("mc_set_undistortion: ") + cudaGetErrorString(e); return MC_ERR_CUDA; }
	MC_CUDA(cudaStreamSynchronize(ctx->stream));       // work queued with the old table finishes before it goes
	MC_CUDA(cudaFree(t.d_map));
	t.d_map = d; t.height = height; t.width = width;
	return MC_OK;
}

extern "C" mc_status mc_undistort_dev(mc_ctx *ctx, int camera, const uint8_t *gray_dev, int n_images, int height, int width, uint8_t *out_dev) {
	if (!ctx) return MC_ERR_ARG;
	if (!gray_dev || !out_dev || n_images < 1 || n_images > 65535) { ctx->err = "mc_undistort_dev: bad argument"; return MC_ERR_ARG; }
	MC_CUDA(cudaSetDevice(ctx->device));
	const UndistortTable *t = nullptr;
	MC_TRY(camera_table(ctx, "mc_undistort_dev", camera, height, width, &t));
	return launch_camera(ctx, *t, gray_dev, n_images, out_dev);
}

extern "C" mc_status mc_undistort(mc_ctx *ctx, int camera, const uint8_t *gray, int n_images, int height, int width, uint8_t *out) {
	if (!ctx) return MC_ERR_ARG;
	if (!gray || !out || n_images < 1 || n_images > 65535) { ctx->err = "mc_undistort: bad argument"; return MC_ERR_ARG; }
	MC_CUDA(cudaSetDevice(ctx->device));
	const UndistortTable *t = nullptr;
	MC_TRY(camera_table(ctx, "mc_undistort", camera, height, width, &t));
	const size_t n = (size_t)n_images * height * width;
	uint8_t *d_in = nullptr, *d_out = nullptr;
	MC_TRY(carve_scratch(ctx, ctx->scratch[kScrUndistort], [&](Carve &c) { c.take(d_in, n); c.take(d_out, n); }));
	MC_CUDA(cudaMemcpyAsync(d_in, gray, n, cudaMemcpyHostToDevice, ctx->stream));
	MC_TRY(launch_camera(ctx, *t, d_in, n_images, d_out));
	MC_CUDA(cudaMemcpyAsync(out, d_out, n, cudaMemcpyDeviceToHost, ctx->stream));
	MC_CUDA(cudaStreamSynchronize(ctx->stream));
	return MC_OK;
}
