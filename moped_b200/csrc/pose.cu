// pose.cu — POSE / POSE2 steps: RANSAC hypotheses with Levenberg–Marquardt pose refinement on
// reprojection error, inlier scoring, refit on inliers.
//
// Replaces POSE_RANSAC_LM_DIFF_REPROJECTION_CPU (moped2/libmoped/src/pose/POSE_RANSAC_LM_DIFF_REPROJECTION_CPU.hpp:66-307)
// and the slevmar_dif it calls (libs.tgz!levmar-2.4/lm_core.c:427-836, misc_core.c:135-168, Axb_core.c:888-1035).
//
// Mapping: a hypothesis is owned by a GROUP of G lanes of one warp — G=8 for the 5/6-point sample fit
// (4 hypotheses per warp, one correspondence per lane), G=32 for the refit on the inliers (one warp,
// correspondences strided over the lanes). Residuals, the finite-difference Jacobian and the Broyden
// update are computed per lane for the lane's own correspondences; ||e||^2, J^T J and J^T e are
// warp-shuffle (butterfly) reductions inside the group; the 7x7 damped normal equations are solved
// redundantly by every lane (no communication). Inlier scoring is a ballot over the cluster's points.
// Compiled with -ftz=true: the reference process runs with FTZ/DAZ and its dominant LM exit is an
// underflow of ||Dp||^2 (SURVEY.md Appendix C).
//
// Provenance: lm_dif and lu_solve7 are DERIVED FROM levmar 2.4 (Manolis Lourakis; GPL; vendored by the reference as
// libs.tgz!levmar-2.4): the control flow of slevmar_dif (lm_core.c:427-836: damping, Broyden updates, the stop tests and their order),
// the forward-difference Jacobian (misc_core.c:135-168) and the Crout LU with implicit scaling (Axb_core.c:888-1035) follow that
// code step for step, with its variable names, because the result has to follow its arithmetic. The parallel decomposition (lane
// groups, butterfly sums, the persistent state machine, LDL^T in front of the LU) is this repository's.
#include "common.cuh"
#include "ransac_sample.cuh"
#include "pose_staged.cuh"

#include <math_constants.h>
#include <float.h>
#include <cstdlib>

namespace mc {

constexpr int kRefitCap = 512;      // inliers used by the refit (16 per lane)

struct LmPoint {                    // one 2D-3D correspondence of a lane
	float u, v, X, Y, Z;
	int cam;
};

template <int G> __device__ __forceinline__ float grp_sum(float v, unsigned mask) {
#pragma unroll
	for (int o = G / 2; o; o >>= 1) v += __shfl_xor_sync(mask, v, o);
	return v;
}
template <int G> __device__ __forceinline__ int grp_sum_i(int v, unsigned mask) {
#pragma unroll
	for (int o = G / 2; o; o >>= 1) v += __shfl_xor_sync(mask, v, o);
	return v;
}

// residual pair of one correspondence under the 3x4 pose matrix T (already built from the normalised
// quaternion): (du^2, dv^2), or (-z+10, -z+10) behind the camera. lmFuncQuat, POSE_..._CPU.hpp:116-136.
__device__ __forceinline__ void residual(const float *T, const Camera &cam, const LmPoint &pt, float &r0, float &r1) {
	const float x = pt.X * T[0] + pt.Y * T[1] + pt.Z * T[2] + T[3];
	const float y = pt.X * T[4] + pt.Y * T[5] + pt.Z * T[6] + T[7];
	const float z = pt.X * T[8] + pt.Y * T[9] + pt.Z * T[10] + T[11];
	const float a = x - cam.TM[3], b = y - cam.TM[7], c = z - cam.TM[11];
	const float cx = a * cam.TM[0] + b * cam.TM[4] + c * cam.TM[8];
	const float cy = a * cam.TM[1] + b * cam.TM[5] + c * cam.TM[9];
	const float cz = a * cam.TM[2] + b * cam.TM[6] + c * cam.TM[10];
	if (cz < 0.f) {
		r0 = -cz + 10.f; r1 = -cz + 10.f;
	} else {
		const float du = cx / cz * cam.K[0] + cam.K[2] - pt.u;
		const float dv = cy / cz * cam.K[1] + cam.K[3] - pt.v;
		r0 = du * du; r1 = dv * dv;
	}
}

// pose.rotation.norm() + TransformMatrix::init (moped.hpp:122,175-182)
__device__ __forceinline__ void pose_to_T(const float *p, float *T) {
	float d = p[0] * p[0] + p[1] * p[1] + p[2] * p[2] + p[3] * p[3];
	d = 1.0f / sqrtf(d);
	const float q0 = p[0] * d, q1 = p[1] * d, q2 = p[2] * d, q3 = p[3] * d;
	T[0] = 1 - 2 * q1 * q1 - 2 * q2 * q2; T[1] = 2 * q0 * q1 - 2 * q3 * q2; T[2] = 2 * q0 * q2 + 2 * q3 * q1; T[3] = p[4];
	T[4] = 2 * q0 * q1 + 2 * q3 * q2; T[5] = 1 - 2 * q0 * q0 - 2 * q2 * q2; T[6] = 2 * q1 * q2 - 2 * q3 * q0; T[7] = p[5];
	T[8] = 2 * q0 * q2 - 2 * q3 * q1; T[9] = 2 * q1 * q2 + 2 * q3 * q0; T[10] = 1 - 2 * q0 * q0 - 2 * q1 * q1; T[11] = p[6];
}

template <int S>
__device__ __forceinline__ void eval_residuals(const float *p, const LmPoint (&pts)[S], int n_own, const Camera *cams, float (&out)[S][2]) {
	float T[12];
	pose_to_T(p, T);
#pragma unroll
	for (int s = 0; s < S; s++) {
		if (s < n_own) residual(T, cams[pts[s].cam], pts[s], out[s][0], out[s][1]);
		else { out[s][0] = 0.f; out[s][1] = 0.f; }
	}
}

// Solve (A + mu I) x = b for symmetric 7x7 A (lower triangle packed, tri(i,j) = i(i+1)/2 + j), by Crout LU
// with implicit row scaling and partial pivoting — sAx_eq_b_LU_noLapack, Axb_core.c:888-1035.
// Every lane of the group runs it on identical data. Returns false if singular.
__device__ __forceinline__ int tri(int i, int j) { return i * (i + 1) / 2 + j; }

__device__ __forceinline__ bool lu_solve7_inline(const float (&A)[28], float mu, const float (&b)[7], float (&x)[7]) {
	float a[7][7], work[7];
#pragma unroll
	for (int i = 0; i < 7; i++)
#pragma unroll
		for (int j = 0; j < 7; j++) a[i][j] = (i >= j) ? A[tri(i, j)] : A[tri(j, i)];
#pragma unroll
	for (int i = 0; i < 7; i++) { a[i][i] += mu; x[i] = b[i]; }
	bool singular = false;
#pragma unroll
	for (int i = 0; i < 7; i++) {
		float mx = 0.f;
#pragma unroll
		for (int j = 0; j < 7; j++) mx = fmaxf(mx, fabsf(a[i][j]));
		if (mx == 0.f) singular = true;
		work[i] = 1.0f / mx;
	}
	if (singular) return false;
#pragma unroll
	for (int j = 0; j < 7; j++) {
#pragma unroll
		for (int i = 0; i < j; i++) {
			float sum = a[i][j];
#pragma unroll
			for (int k = 0; k < i; k++) sum -= a[i][k] * a[k][j];
			a[i][j] = sum;
		}
		float mx = 0.f;
		int maxi = j;
#pragma unroll
		for (int i = j; i < 7; i++) {
			float sum = a[i][j];
#pragma unroll
			for (int k = 0; k < j; k++) sum -= a[i][k] * a[k][j];
			a[i][j] = sum;
			const float t = work[i] * fabsf(sum);
			if (t >= mx) { mx = t; maxi = i; }
		}
		if (maxi != j) {
#pragma unroll
			for (int i = j + 1; i < 7; i++) {
				const bool sw = (maxi == i);
#pragma unroll
				for (int k = 0; k < 7; k++) {
					const float u = a[i][k], w = a[j][k];
					a[i][k] = sw ? w : u; a[j][k] = sw ? u : w;
				}
				const float xu = x[i], xw = x[j];
				x[i] = sw ? xw : xu; x[j] = sw ? xu : xw;
				work[i] = sw ? work[j] : work[i];
			}
		}
		if (a[j][j] == 0.f) a[j][j] = FLT_EPSILON;
		if (j != 6) {
			const float t = 1.0f / a[j][j];
#pragma unroll
			for (int i = j + 1; i < 7; i++) a[i][j] *= t;
		}
	}
#pragma unroll
	for (int i = 0; i < 7; i++) {
		float sum = x[i];
#pragma unroll
		for (int j = 0; j < i; j++) sum -= a[i][j] * x[j];
		x[i] = sum;
	}
#pragma unroll
	for (int i = 6; i >= 0; i--) {
		float sum = x[i];
#pragma unroll
		for (int j = i + 1; j < 7; j++) sum -= a[i][j] * x[j];
		x[i] = sum / a[i][i];
	}
	return true;
}

// out of line: the cold path of solve7 below
__device__ __noinline__ bool lu_solve7(const float (&A)[28], float mu, const float (&b)[7], float (&x)[7]) { return lu_solve7_inline(A, mu, b, x); }

// The damped normal equations (J^T J + mu I) Dp = J^T e of the DEFAULT kernels. levmar solves them with the pivoting LU above; the
// matrix is symmetric positive definite for mu > 0, so an unpivoted LDL^T factorisation gives the same solution to within the
// rounding both methods carry (measured on the oracle: 99.2 % of the systems of an LM run keep every pivot above 1e-3 of its
// diagonal entry; with LDL^T there and the LU elsewhere, accept decisions of 1792 hypotheses are identical and refitted poses
// differ by 1.3e-5 m at the median / 2.6e-4 m at the 90th percentile — the spread between the reference's own two builds,
// profiles/lm_parity_r2.md) at a quarter of the instructions: ~210 against ~890 executed SASS instructions per solve, and the
// solve was 35 % of the instructions of the thread-per-hypothesis kernel (ncu) and the longest stretch of the lane-group kernels'
// dependent chain. A system that loses three digits in a pivot (mu underflowed, J^T J rank-deficient along the quaternion's scale),
// or holds a NaN, takes levmar's LU with its singularity rules. The exact-order mode (lm_exact.cuh) always runs the LU.
__device__ __forceinline__ float rcp_approx(float v) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v)); return r; }
__device__ __forceinline__ int ltri(int i, int j) { return i * (i - 1) / 2 + j; }       // strict lower triangle, j < i

__device__ __forceinline__ bool ldl_solve7(const float (&A)[28], float mu, const float (&b)[7], float (&x)[7]) {
	float L[21], d[7], r[7], z[7];
	bool ok = true;
#pragma unroll
	for (int j = 0; j < 7; j++) {
		const float ajj = A[tri(j, j)] + mu;
		float v[7];
		float s = ajj;
#pragma unroll
		for (int k = 0; k < j; k++) { v[k] = L[ltri(j, k)] * d[k]; s -= L[ltri(j, k)] * v[k]; }
		ok = ok && (s > 1E-03f * ajj);                    // false for a NaN as well
		d[j] = s;
		r[j] = rcp_approx(s);                            // MUFU.RCP, 1 ulp: the pivoting LU this replaces differs from it by far more (cond * eps)
#pragma unroll
		for (int i = j + 1; i < 7; i++) {
			float t = A[tri(i, j)];
#pragma unroll
			for (int k = 0; k < j; k++) t -= L[ltri(i, k)] * v[k];
			L[ltri(i, j)] = t * r[j];
		}
	}
	if (!ok) return false;
#pragma unroll
	for (int i = 0; i < 7; i++) {
		float t = b[i];
#pragma unroll
		for (int k = 0; k < i; k++) t -= L[ltri(i, k)] * z[k];
		z[i] = t;
	}
#pragma unroll
	for (int i = 6; i >= 0; i--) {
		float t = z[i] * r[i];
#pragma unroll
		for (int k = i + 1; k < 7; k++) t -= L[ltri(k, i)] * x[k];
		x[i] = t;
	}
	return true;
}

__device__ __forceinline__ bool solve7(const float (&A)[28], float mu, const float (&b)[7], float (&x)[7]) {
	if (ldl_solve7(A, mu, b, x)) return true;
	return lu_solve7(A, mu, b, x);
}

// slevmar_dif restated for a lane group: m = 7, target 0, default options (lm.h:83-85), forward-difference
// Jacobian (misc_core.c:135-168), Broyden rank-1 updates, K = 10 (lm_core.c:484-836). `pts` holds this
// lane's correspondences (n_own of them). On return p is the solution (if >= 0 is returned) and err = ||e||^2.
// Returns the iteration count or -1 (LM_ERROR, stop = 4).
// `abort_if_below` (nullable): shared word holding the lowest hypothesis index that already succeeded; a group
// working on a higher index gives up (its result could not be chosen any more).
template <int G, int S>
__device__ int lm_dif(float (&p)[7], int itmax, const LmPoint (&pts)[S], int n_own, const Camera *cams, unsigned mask, float &err,
                      const volatile int *abort_if_below = nullptr, int my_index = 0) {
	const float tau = 1E-03f, eps1 = 1E-17f, eps2 = 1E-17f, eps2_sq = 1E-17f * 1E-17f, eps3 = 1E-17f, delta = 1E-06f;
	float J[S][2][7], hx[S][2], wrk[S][2];
	float jtj[28], jte[7], diag[7], Dp[7], pDp[7];
	float mu = 0.f, jte_inf = 0.f, p_L2 = 0.f, p_eL2, pDp_eL2;
	int nu = 20, stop = 0, updjac = 0, updp = 1, newjac = 0, k;
	const int K = 10;

	eval_residuals<S>(p, pts, n_own, cams, hx);
	{
		float s = 0.f;
#pragma unroll
		for (int i = 0; i < S; i++) s += hx[i][0] * hx[i][0] + hx[i][1] * hx[i][1];
		p_eL2 = grp_sum<G>(s, mask);
	}
#pragma unroll
	for (int i = 0; i < S; i++)
#pragma unroll
		for (int r = 0; r < 2; r++)
#pragma unroll
			for (int j = 0; j < 7; j++) J[i][r][j] = 0.f;

	for (k = 0; k < itmax && !stop; ++k) {
		if (abort_if_below && *abort_if_below < my_index) { stop = 4; break; }
		if (p_eL2 <= eps3) { stop = 6; break; }

		if ((updp && nu > 16) || updjac == K) {
#pragma unroll
			for (int j = 0; j < 7; j++) {
				float d = fabsf(1E-04f * p[j]);
				if (d < delta) d = delta;
				const float save = p[j];
				p[j] += d;
				eval_residuals<S>(p, pts, n_own, cams, wrk);
				p[j] = save;
				d = 1.0f / d;
#pragma unroll
				for (int i = 0; i < S; i++) { J[i][0][j] = (wrk[i][0] - hx[i][0]) * d; J[i][1][j] = (wrk[i][1] - hx[i][1]) * d; }
			}
			nu = 2; updjac = 0; updp = 0; newjac = 1;
		}

		if (newjac) {
			newjac = 0;
#pragma unroll
			for (int i = 0; i < 28; i++) jtj[i] = 0.f;
#pragma unroll
			for (int i = 0; i < 7; i++) jte[i] = 0.f;
#pragma unroll
			for (int s = 0; s < S; s++)
#pragma unroll
				for (int r = 0; r < 2; r++) {
					const float e = -hx[s][r];                     // e = x - hx with x = 0
#pragma unroll
					for (int i = 0; i < 7; i++) {
						const float alpha = J[s][r][i];
#pragma unroll
						for (int j = 0; j <= i; j++) jtj[tri(i, j)] += J[s][r][j] * alpha;
						jte[i] += alpha * e;
					}
				}
#pragma unroll
			for (int i = 0; i < 28; i++) jtj[i] = grp_sum<G>(jtj[i], mask);
#pragma unroll
			for (int i = 0; i < 7; i++) jte[i] = grp_sum<G>(jte[i], mask);
			p_L2 = 0.f; jte_inf = 0.f;
#pragma unroll
			for (int i = 0; i < 7; i++) {
				jte_inf = fmaxf(jte_inf, fabsf(jte[i]));
				diag[i] = jtj[tri(i, i)];
				p_L2 += p[i] * p[i];
			}
		}

		if (jte_inf <= eps1) { stop = 1; break; }

		if (k == 0) {
			float t = -FLT_MAX;
#pragma unroll
			for (int i = 0; i < 7; i++) t = fmaxf(t, diag[i]);
			mu = tau * t;
		}

		const bool solved = solve7(jtj, mu, jte, Dp);
		if (solved) {
			float Dp_L2 = 0.f;
#pragma unroll
			for (int i = 0; i < 7; i++) { pDp[i] = p[i] + Dp[i]; Dp_L2 += Dp[i] * Dp[i]; }
			if (Dp_L2 <= eps2_sq * p_L2) { stop = 2; break; }
			if (Dp_L2 >= (p_L2 + eps2) / (1E-12f * 1E-12f)) { stop = 4; break; }

			eval_residuals<S>(pDp, pts, n_own, cams, wrk);
			{
				float s = 0.f;
#pragma unroll
				for (int i = 0; i < S; i++) s += wrk[i][0] * wrk[i][0] + wrk[i][1] * wrk[i][1];
				pDp_eL2 = grp_sum<G>(s, mask);
			}
			const float dF = p_eL2 - pDp_eL2;
			if (updp || dF > 0.f) {
				const float inv = 1.0f / Dp_L2;
#pragma unroll
				for (int s = 0; s < S; s++)
#pragma unroll
					for (int r = 0; r < 2; r++) {
						float t = 0.f;
#pragma unroll
						for (int l = 0; l < 7; l++) t += J[s][r][l] * Dp[l];
						t = (wrk[s][r] - hx[s][r] - t) * inv;
#pragma unroll
						for (int j = 0; j < 7; j++) J[s][r][j] += t * Dp[j];
					}
				++updjac; newjac = 1;
			}
			float dL = 0.f;
#pragma unroll
			for (int i = 0; i < 7; i++) dL += Dp[i] * (mu * Dp[i] + jte[i]);
			if (dL > 0.f && dF > 0.f) {
				float t = 2.0f * dF / dL - 1.0f;
				t = 1.0f - t * t * t;
				mu = mu * ((t >= 0.3333333334f) ? t : 0.3333333334f);
				nu = 2;
#pragma unroll
				for (int i = 0; i < 7; i++) p[i] = pDp[i];
#pragma unroll
				for (int s = 0; s < S; s++) { hx[s][0] = wrk[s][0]; hx[s][1] = wrk[s][1]; }
				p_eL2 = pDp_eL2;
				updp = 1;
				continue;
			}
		}
		mu *= nu;
		const int nu2 = nu << 1;
		if (nu2 <= nu) { stop = 5; break; }
		nu = nu2;
	}
	err = p_eL2;
	return (stop != 4) ? k : -1;
}

// optimizeCamera (POSE_..._CPU.hpp:140-164): LM, then re-normalise the quaternion. Returns false on LM_ERROR
// (pose untouched).
template <int G, int S>
__device__ bool optimize_camera(float (&pose)[7], int itmax, const LmPoint (&pts)[S], int n_own, const Camera *cams, unsigned mask, float &err,
                                const volatile int *abort_if_below = nullptr, int my_index = 0) {
	float p[7];
#pragma unroll
	for (int i = 0; i < 7; i++) p[i] = pose[i];
	const int r = lm_dif<G, S>(p, itmax, pts, n_own, cams, mask, err, abort_if_below, my_index);
	if (r < 0) { err = -1.f; return false; }
	float d = p[0] * p[0] + p[1] * p[1] + p[2] * p[2] + p[3] * p[3];
	d = 1.0f / sqrtf(d);
	pose[0] = p[0] * d; pose[1] = p[1] * d; pose[2] = p[2] * d; pose[3] = p[3] * d;
	pose[4] = p[4]; pose[5] = p[5]; pose[6] = p[6];
	return true;
}

// squared reprojection error used by testAllPoints / project() (POSE_..._CPU.hpp:166-180, moped.hpp:330-354)
__device__ __forceinline__ float proj_err(const float *T, const Camera &cam, float X, float Y, float Z, float u0, float v0) {
	const float x = X * T[0] + Y * T[1] + Z * T[2] + T[3];
	const float y = X * T[4] + Y * T[5] + Z * T[6] + T[7];
	const float z = X * T[8] + Y * T[9] + Z * T[10] + T[11];
	const float a = x - cam.TM[3], b = y - cam.TM[7], c = z - cam.TM[11];
	const float cx = a * cam.TM[0] + b * cam.TM[4] + c * cam.TM[8];
	const float cy = a * cam.TM[1] + b * cam.TM[5] + c * cam.TM[9];
	const float cz = a * cam.TM[2] + b * cam.TM[6] + c * cam.TM[10];
	float u = FLT_MAX, v = FLT_MAX;
	if (!((double)cz < 0.001)) { u = cx / cz * cam.K[0] + cam.K[2]; v = cy / cz * cam.K[1] + cam.K[3]; }
	const float du = u - u0, dv = v - v0;
	return du * du + dv * dv;
}

__device__ __forceinline__ void pose7_to_T(const float *pose, float *T) {   // pose already normalised: TransformMatrix::init
	const float q0 = pose[0], q1 = pose[1], q2 = pose[2], q3 = pose[3];
	T[0] = 1 - 2 * q1 * q1 - 2 * q2 * q2; T[1] = 2 * q0 * q1 - 2 * q3 * q2; T[2] = 2 * q0 * q2 + 2 * q3 * q1; T[3] = pose[4];
	T[4] = 2 * q0 * q1 + 2 * q3 * q2; T[5] = 1 - 2 * q0 * q0 - 2 * q2 * q2; T[6] = 2 * q1 * q2 - 2 * q3 * q0; T[7] = pose[5];
	T[8] = 2 * q0 * q2 - 2 * q3 * q1; T[9] = 2 * q1 * q2 + 2 * q3 * q0; T[10] = 1 - 2 * q0 * q0 - 2 * q1 * q1; T[11] = pose[6];
}

// inlier count of `pose` over a cluster's points by a lane group; optionally writes the mask
template <int G>
__device__ int count_inliers(const float *pose, int n, const float *xy, const float *xyz, const int32_t *image, const Camera *cams,
                             float thr, unsigned mask, int lig, uint8_t *out_mask) {
	float T[12];
	pose7_to_T(pose, T);
	int c = 0;
	for (int i = lig; i < n; i += G) {
		const float e = proj_err(T, cams[image[i]], xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2], xy[2 * i], xy[2 * i + 1]);
		const int in = e < thr;
		if (out_mask) out_mask[i] = (uint8_t)in;
		c += in;
	}
	return grp_sum_i<G>(c, mask);
}

// sample fit + inlier count of one hypothesis by an 8-lane group. Returns #inliers or -1.
__device__ int fit_and_score(const int (&pos)[kMaxAlign], int n_align, const float (&quat)[4], int n, const float *xy, const float *xyz,
                             const int32_t *image, const Camera *cams, int max_lm, float thr, unsigned mask, int lig,
                             float (&pose)[7], float &err, uint8_t *out_mask, const volatile int *abort_if_below = nullptr, int my_index = 0) {
	LmPoint pts[1];
	int mine = 0;
#pragma unroll
	for (int j = 0; j < kMaxAlign; j++) if (j == lig) mine = pos[j];
	const int n_own = lig < n_align ? 1 : 0;
	if (n_own) {
		pts[0].u = xy[2 * mine]; pts[0].v = xy[2 * mine + 1];
		pts[0].X = xyz[3 * mine]; pts[0].Y = xyz[3 * mine + 1]; pts[0].Z = xyz[3 * mine + 2];
		pts[0].cam = image[mine];
	} else { pts[0].u = pts[0].v = pts[0].X = pts[0].Y = pts[0].Z = 0.f; pts[0].cam = 0; }
	pose[0] = quat[0]; pose[1] = quat[1]; pose[2] = quat[2]; pose[3] = quat[3];
	pose[4] = 0.f; pose[5] = 0.f; pose[6] = 0.5f;
	if (!optimize_camera<8, 1>(pose, max_lm, pts, n_own, cams, mask, err, abort_if_below, my_index)) return -1;
	return count_inliers<8>(pose, n, xy, xyz, image, cams, thr, mask, lig, out_mask);
}

// refit of `pose` on its inliers by a full warp (optimizeCamera(pose, consistent), :204-208).
// list = per-warp shared scratch of kRefitCap ints. Returns false if LM failed (pose unchanged).
template <int S>
__device__ bool refit_S(float (&pose)[7], int n_inl, const int *list, const float *xy, const float *xyz, const int32_t *image,
                        const Camera *cams, int max_lm, int lane, float &err) {
	LmPoint pts[S];
	int n_own = 0;
#pragma unroll
	for (int s = 0; s < S; s++) {
		const int k = lane + 32 * s;
		if (k < n_inl) {
			const int i = list[k];
			pts[s].u = xy[2 * i]; pts[s].v = xy[2 * i + 1];
			pts[s].X = xyz[3 * i]; pts[s].Y = xyz[3 * i + 1]; pts[s].Z = xyz[3 * i + 2];
			pts[s].cam = image[i];
			n_own = s + 1;
		} else { pts[s].u = pts[s].v = pts[s].X = pts[s].Y = pts[s].Z = 0.f; pts[s].cam = 0; }
	}
	return optimize_camera<32, S>(pose, max_lm, pts, n_own, cams, 0xffffffffu, err);
}

__device__ bool refit_warp(float (&pose)[7], int n, const float *xy, const float *xyz, const int32_t *image, const Camera *cams,
                           float thr, int max_lm, int lane, int *list, float &err) {
	// inliers of `pose` in cluster order -> list (the reference refits on `consistent` in cluster order)
	float T[12];
	pose7_to_T(pose, T);
	int n_inl = 0;
	for (int i0 = 0; i0 < n; i0 += 32) {
		const int i = i0 + lane;
		bool in = false;
		if (i < n) in = proj_err(T, cams[image[i]], xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2], xy[2 * i], xy[2 * i + 1]) < thr;
		const unsigned m = __ballot_sync(0xffffffffu, in);
		if (in) {
			const int k = n_inl + __popc(m & ((1u << lane) - 1));
			if (k < kRefitCap) list[k] = i;
		}
		n_inl += __popc(m);
	}
	__syncwarp();
	if (n_inl > kRefitCap) n_inl = kRefitCap;
	if (n_inl <= 32) return refit_S<1>(pose, n_inl, list, xy, xyz, image, cams, max_lm, lane, err);
	if (n_inl <= 64) return refit_S<2>(pose, n_inl, list, xy, xyz, image, cams, max_lm, lane, err);
	if (n_inl <= 128) return refit_S<4>(pose, n_inl, list, xy, xyz, image, cams, max_lm, lane, err);
	if (n_inl <= 256) return refit_S<8>(pose, n_inl, list, xy, xyz, image, cams, max_lm, lane, err);
	return refit_S<16>(pose, n_inl, list, xy, xyz, image, cams, max_lm, lane, err);
}

// ---- kernel A: explicit hypotheses, sample fit + inlier scoring; 4 hypotheses per warp ----
__global__ void __launch_bounds__(kPoseThreads)
k_pose_fit(const int32_t *__restrict__ cluster_offsets, const float *__restrict__ xy, const float *__restrict__ xyz,
           const int32_t *__restrict__ image, const Camera *__restrict__ cams, const int32_t *__restrict__ hyp_cluster,
           const int32_t *__restrict__ sample_pos, const float *__restrict__ init_quat, int n_hyp, int n_align, int max_lm, float thr,
           const int64_t *__restrict__ mask_offsets, int32_t *__restrict__ n_inliers, float *__restrict__ pose_lm,
           float *__restrict__ lm_err, uint8_t *__restrict__ inlier_mask) {
	const int lane = threadIdx.x & 31, lig = lane & 7, grp = lane >> 3;
	const unsigned mask = 0xFFu << (8 * grp);
	const int h = (blockIdx.x * (kPoseThreads / 32) + (threadIdx.x >> 5)) * 4 + grp;
	if (h >= n_hyp) return;
	const int c = hyp_cluster[h];
	const int lo = cluster_offsets[c], n = cluster_offsets[c + 1] - lo;
	int pos[kMaxAlign];
#pragma unroll
	for (int j = 0; j < kMaxAlign; j++) pos[j] = j < n_align ? sample_pos[(size_t)h * n_align + j] : 0;
	float quat[4] = { init_quat[4 * h], init_quat[4 * h + 1], init_quat[4 * h + 2], init_quat[4 * h + 3] };
	float pose[7], err;
	uint8_t *om = inlier_mask ? inlier_mask + mask_offsets[h] : nullptr;
	if (om) for (int i = lig; i < n; i += 8) om[i] = 0;
	const int cnt = fit_and_score(pos, n_align, quat, n, xy + 2 * lo, xyz + 3 * lo, image + lo, cams, max_lm, thr, mask, lig, pose, err, om);
	if (lig == 0) {
		n_inliers[h] = cnt;
		lm_err[2 * h] = err; lm_err[2 * h + 1] = -2.f;
		for (int j = 0; j < 7; j++) pose_lm[7 * h + j] = cnt >= 0 ? pose[j] : 0.f;
	}
}

// ---- kernel A': the same per-hypothesis work with ONE THREAD per hypothesis (throughput shape) ----
// The lane-group kernel spends most of its instructions on work every lane repeats (the 7x7 solve) or on moving
// partial sums between lanes; with thousands of independent hypotheses (BASELINE configs[3]) a thread can own a whole
// hypothesis instead: its NPtsAlign correspondences, Jacobian and normal equations live in its registers, sums run
// sequentially over the residuals (levmar's own order), and a warp advances 32 hypotheses per instruction.
template <int S>
__global__ void __launch_bounds__(128)
k_pose_fit_thread(const int32_t *__restrict__ cluster_offsets, const float *__restrict__ xy, const float *__restrict__ xyz,
                  const int32_t *__restrict__ image, const Camera *__restrict__ cams, const int32_t *__restrict__ hyp_cluster,
                  const int32_t *__restrict__ sample_pos, const float *__restrict__ init_quat, int n_hyp, int n_align, int max_lm, float thr,
                  int32_t *__restrict__ n_inliers, float *__restrict__ pose_lm, float *__restrict__ lm_err) {
	const int h = blockIdx.x * blockDim.x + threadIdx.x;
	if (h >= n_hyp) return;
	const int c = hyp_cluster[h];
	const int lo = cluster_offsets[c], n = cluster_offsets[c + 1] - lo;
	const float *cxy = xy + 2 * lo, *cxyz = xyz + 3 * lo;
	const int32_t *cim = image + lo;
	LmPoint pts[S];
#pragma unroll
	for (int j = 0; j < S; j++) {
		if (j < n_align) {
			const int i = sample_pos[(size_t)h * n_align + j];
			pts[j].u = cxy[2 * i]; pts[j].v = cxy[2 * i + 1];
			pts[j].X = cxyz[3 * i]; pts[j].Y = cxyz[3 * i + 1]; pts[j].Z = cxyz[3 * i + 2];
			pts[j].cam = cim[i];
		} else { pts[j].u = pts[j].v = pts[j].X = pts[j].Y = pts[j].Z = 0.f; pts[j].cam = 0; }
	}
	float pose[7] = { init_quat[4 * h], init_quat[4 * h + 1], init_quat[4 * h + 2], init_quat[4 * h + 3], 0.f, 0.f, 0.5f };
	float err;
	int cnt = -1;
	if (optimize_camera<1, S>(pose, max_lm, pts, n_align, cams, 0u, err))
		cnt = count_inliers<1>(pose, n, cxy, cxyz, cim, cams, thr, 0u, 0, nullptr);
	n_inliers[h] = cnt;
	lm_err[2 * h] = err; lm_err[2 * h + 1] = -2.f;
#pragma unroll
	for (int j = 0; j < 7; j++) pose_lm[7 * h + j] = cnt >= 0 ? pose[j] : 0.f;
}

// ---- kernel A'': one thread per hypothesis, PERSISTENT and PHASE-SYNCHRONOUS (the default throughput shape) ----
// k_pose_fit_thread keeps 9.9 of 32 lanes busy (ncu, profiles/ncu_stage_kernels_r1i.md): hypotheses leave the LM loop after different
// iteration counts and the finite-difference Jacobian (7 residual evaluations, more instructions than the rest of an iteration) is
// due at different iterations in different lanes, so a warp pays for it on almost every trip. Here a thread is a small state machine
// and a warp trip has ONE residual evaluation that every lane uses for whatever it needs next:
//   INIT   the residuals at the start pose of a freshly fetched hypothesis (a finished lane takes the next hypothesis from a global
//          counter at once instead of idling until the slowest lane of its warp is done),
//   JAC    column jc of the forward-difference Jacobian (a lane that needs a new Jacobian spends 7 trips here),
//   SOLVE  the trial point p + Dp of an LM iteration (normal equations, the 7x7 solve before it; Broyden update, gain ratio after).
// Per hypothesis the arithmetic and its order are those of lm_dif<1, S> (one lane, sequential sums). The Jacobian and the sample
// points live in shared memory, element-major ([e][thread]: conflict-free), which brings the kernel from 254 to <= 168 registers.
// Inlier scoring moved to k_pose_score (one 8-lane group per hypothesis): inside the state machine it would run with one or two
// active lanes.
// Measured variants of this kernel (B200, 131072 hypotheses, profiles/fit_stream_experiments_r2b.md): this one 4.04 ms (ncu: 13.6 active
// lanes, 49 % issue utilisation, top stall `no_instruction` — twelve warps spread over the branches of a 3.5 k-instruction body);
// LDL^T first + out-of-line LU fallback (solve7): 14 % fewer executed instructions but 4.24 ms (a warp pays the fallback whenever one
// of its lanes needs it, at 2.3 active lanes; instruction-cache hit rate 74 -> 64 %); the same with the row loops rolled and hx / trial
// residuals in shared memory (2.5 k -> 1.2 k hot instructions): 5.08 ms (loop overhead and dynamic addressing cost more than the
// fetch stalls they remove); 4 CTAs per SM at 128 registers: no change. The lane-group kernels do use solve7 (their solve is redundant
// per lane and on the critical path of a single LM chain: k_pose_refit_lists 0.86 -> 0.49 ms, frame batch 5.5 -> 4.0 ms).
constexpr int kStreamThreads = 128;
constexpr int kStreamFloats = 20;                                       // shared-memory floats per thread and sample point: J 14, point 6
enum { kModeIdle = 0, kModeInit = 1, kModeSolve = 2, kModeJac = 3 };

template <int S, int MINB>
__global__ void __launch_bounds__(kStreamThreads, MINB)
k_pose_fit_stream(const int32_t *__restrict__ cluster_offsets, const float *__restrict__ xy, const float *__restrict__ xyz,
                  const int32_t *__restrict__ image, const Camera *__restrict__ cams, const int32_t *__restrict__ hyp_cluster,
                  const int32_t *__restrict__ sample_pos, const float *__restrict__ init_quat, int n_hyp, int n_align, int itmax,
                  uint32_t *__restrict__ next_hyp, int32_t *__restrict__ n_inliers, float *__restrict__ pose_lm, float *__restrict__ lm_err) {
	extern __shared__ float s_stream[];
	const int nt = kStreamThreads;
	float *Js = s_stream + threadIdx.x;                                  // J[s][r][j] at Js[((s * 2 + r) * 7 + j) * nt]
	float *Ps = s_stream + (size_t)S * 14 * nt + threadIdx.x;            // point s, component c (u v X Y Z cam) at Ps[(s * 6 + c) * nt]
	const float tau = 1E-03f, eps1 = 1E-17f, eps2 = 1E-17f, eps2_sq = 1E-17f * 1E-17f, eps3 = 1E-17f, delta = 1E-06f;
	const int K = 10;
	float p[7], hx[S][2], jtj[28], jte[7];
	float mu = 0.f, jte_inf = 0.f, p_L2 = 0.f, p_eL2 = 0.f, dcur = 0.f;
	int nu = 20, updjac = 0, updp = 1, newjac = 0, k = 0, jc = 0, h = -1, mode = kModeIdle;
	bool more = true;
#pragma unroll
	for (int i = 0; i < 28; i++) jtj[i] = 0.f;
#pragma unroll
	for (int i = 0; i < 7; i++) { jte[i] = 0.f; p[i] = 0.f; }
#pragma unroll
	for (int i = 0; i < S; i++) { hx[i][0] = 0.f; hx[i][1] = 0.f; }

	auto load_pts = [&](LmPoint (&pts)[S]) {
#pragma unroll
		for (int s = 0; s < S; s++) {
			pts[s].u = Ps[(s * 6 + 0) * nt]; pts[s].v = Ps[(s * 6 + 1) * nt];
			pts[s].X = Ps[(s * 6 + 2) * nt]; pts[s].Y = Ps[(s * 6 + 3) * nt]; pts[s].Z = Ps[(s * 6 + 4) * nt];
			pts[s].cam = __float_as_int(Ps[(s * 6 + 5) * nt]);
		}
	};
	// the hypothesis leaves the LM: optimizeCamera's epilogue (quaternion re-normalised; LM_ERROR leaves no pose)
	auto finish = [&](int stop) {
		if (stop == 4) {
			n_inliers[h] = -1;
			lm_err[2 * h] = -1.f; lm_err[2 * h + 1] = -2.f;
#pragma unroll
			for (int j = 0; j < 7; j++) pose_lm[7 * h + j] = 0.f;
		} else {
			float d = p[0] * p[0] + p[1] * p[1] + p[2] * p[2] + p[3] * p[3];
			d = 1.0f / sqrtf(d);
			n_inliers[h] = 0;                                              // k_pose_score counts
			lm_err[2 * h] = p_eL2; lm_err[2 * h + 1] = -2.f;
#pragma unroll
			for (int j = 0; j < 4; j++) pose_lm[7 * h + j] = p[j] * d;
#pragma unroll
			for (int j = 4; j < 7; j++) pose_lm[7 * h + j] = p[j];
		}
		mode = kModeIdle;
	};

	for (;;) {
		if (mode == kModeIdle && more) {
			h = (int)atomicAdd(next_hyp, 1u);
			if (h >= n_hyp) more = false;
			else {
				const int c = hyp_cluster[h];
				const int lo = cluster_offsets[c];
#pragma unroll
				for (int s = 0; s < S; s++) {
					float u = 0.f, v = 0.f, X = 0.f, Y = 0.f, Z = 0.f; int cam = 0;
					if (s < n_align) {
						const int i = lo + sample_pos[(size_t)h * n_align + s];
						u = xy[2 * i]; v = xy[2 * i + 1]; X = xyz[3 * i]; Y = xyz[3 * i + 1]; Z = xyz[3 * i + 2]; cam = image[i];
					}
					Ps[(s * 6 + 0) * nt] = u; Ps[(s * 6 + 1) * nt] = v; Ps[(s * 6 + 2) * nt] = X; Ps[(s * 6 + 3) * nt] = Y; Ps[(s * 6 + 4) * nt] = Z;
					Ps[(s * 6 + 5) * nt] = __int_as_float(cam);
				}
				p[0] = init_quat[4 * h]; p[1] = init_quat[4 * h + 1]; p[2] = init_quat[4 * h + 2]; p[3] = init_quat[4 * h + 3];
				p[4] = 0.f; p[5] = 0.f; p[6] = 0.5f;
				mode = kModeInit;
			}
		}
		if (!__any_sync(0xffffffffu, mode != kModeIdle)) break;

		float x[7], Dp[7], Dp_L2 = 0.f;
		bool ev = false;
		// ---- top of an LM iteration (lm_core.c:484-520): stop tests, is a new Jacobian due? ----
		if (mode == kModeSolve) {
			if (k >= itmax) finish(3);
			else if (p_eL2 <= eps3) finish(6);
			else if ((updp && nu > 16) || updjac == K) { mode = kModeJac; jc = 0; }
		}
		// ---- normal equations and the damped solve ----
		if (mode == kModeSolve) {
			if (newjac) {
				newjac = 0;
#pragma unroll
				for (int i = 0; i < 28; i++) jtj[i] = 0.f;
#pragma unroll
				for (int i = 0; i < 7; i++) jte[i] = 0.f;
#pragma unroll
				for (int s = 0; s < S; s++)
#pragma unroll
					for (int r = 0; r < 2; r++) {
						float Jr[7];
#pragma unroll
						for (int j = 0; j < 7; j++) Jr[j] = Js[((s * 2 + r) * 7 + j) * nt];
						const float e = -hx[s][r];
#pragma unroll
						for (int i = 0; i < 7; i++) {
							const float alpha = Jr[i];
#pragma unroll
							for (int j = 0; j <= i; j++) jtj[tri(i, j)] += Jr[j] * alpha;
							jte[i] += alpha * e;
						}
					}
				p_L2 = 0.f; jte_inf = 0.f;
#pragma unroll
				for (int i = 0; i < 7; i++) {
					jte_inf = fmaxf(jte_inf, fabsf(jte[i]));
					p_L2 += p[i] * p[i];
				}
			}
			if (jte_inf <= eps1) finish(1);
			else {
				if (k == 0) {
					float t = -FLT_MAX;
#pragma unroll
					for (int i = 0; i < 7; i++) t = fmaxf(t, jtj[tri(i, i)]);
					mu = tau * t;
				}
				if (lu_solve7_inline(jtj, mu, jte, Dp)) {        // (LDL^T + out-of-line LU measured here: 14 % fewer instructions, 5 % slower — see below)
#pragma unroll
					for (int i = 0; i < 7; i++) { x[i] = p[i] + Dp[i]; Dp_L2 += Dp[i] * Dp[i]; }
					if (Dp_L2 <= eps2_sq * p_L2) finish(2);
					else if (Dp_L2 >= (p_L2 + eps2) / (1E-12f * 1E-12f)) finish(4);
					else ev = true;
				} else {
					mu *= nu;
					const int nu2 = nu << 1;
					if (nu2 <= nu) finish(5);
					else { nu = nu2; ++k; }
				}
			}
		} else if (mode == kModeJac) {
#pragma unroll
			for (int j = 0; j < 7; j++) {
				x[j] = p[j];
				if (j == jc) {
					float d = fabsf(1E-04f * p[j]);
					if (d < delta) d = delta;
					dcur = d;
					x[j] = p[j] + d;
				}
			}
			ev = true;
		} else if (mode == kModeInit) {
#pragma unroll
			for (int j = 0; j < 7; j++) x[j] = p[j];
			ev = true;
		}

		// ---- the trip's residual evaluation ----
		if (ev) {
			float wrk[S][2];
			{
				LmPoint pts[S];
				load_pts(pts);
				eval_residuals<S>(x, pts, n_align, cams, wrk);
			}
			if (mode == kModeInit) {
				float s2 = 0.f;
#pragma unroll
				for (int i = 0; i < S; i++) { hx[i][0] = wrk[i][0]; hx[i][1] = wrk[i][1]; s2 += wrk[i][0] * wrk[i][0] + wrk[i][1] * wrk[i][1]; }
				p_eL2 = s2;
				mu = 0.f; jte_inf = 0.f; p_L2 = 0.f;
				nu = 20; updjac = 0; updp = 1; newjac = 0; k = 0;
				mode = kModeSolve;
			} else if (mode == kModeJac) {
				const float dinv = 1.0f / dcur;
#pragma unroll
				for (int i = 0; i < S; i++) {
					Js[((i * 2 + 0) * 7 + jc) * nt] = (wrk[i][0] - hx[i][0]) * dinv;
					Js[((i * 2 + 1) * 7 + jc) * nt] = (wrk[i][1] - hx[i][1]) * dinv;
				}
				if (++jc == 7) { nu = 2; updjac = 0; updp = 0; newjac = 1; mode = kModeSolve; }
			} else {
				float s2 = 0.f;
#pragma unroll
				for (int i = 0; i < S; i++) s2 += wrk[i][0] * wrk[i][0] + wrk[i][1] * wrk[i][1];
				const float pDp_eL2 = s2;
				const float dF = p_eL2 - pDp_eL2;
				if (updp || dF > 0.f) {
					const float inv = 1.0f / Dp_L2;
#pragma unroll
					for (int s = 0; s < S; s++)
#pragma unroll
						for (int r = 0; r < 2; r++) {
							float Jr[7];
#pragma unroll
							for (int j = 0; j < 7; j++) Jr[j] = Js[((s * 2 + r) * 7 + j) * nt];
							float t = 0.f;
#pragma unroll
							for (int l = 0; l < 7; l++) t += Jr[l] * Dp[l];
							t = (wrk[s][r] - hx[s][r] - t) * inv;
#pragma unroll
							for (int j = 0; j < 7; j++) Js[((s * 2 + r) * 7 + j) * nt] = Jr[j] + t * Dp[j];
						}
					++updjac; newjac = 1;
				}
				float dL = 0.f;
#pragma unroll
				for (int i = 0; i < 7; i++) dL += Dp[i] * (mu * Dp[i] + jte[i]);
				if (dL > 0.f && dF > 0.f) {
					float t = 2.0f * dF / dL - 1.0f;
					t = 1.0f - t * t * t;
					mu = mu * ((t >= 0.3333333334f) ? t : 0.3333333334f);
					nu = 2;
#pragma unroll
					for (int i = 0; i < 7; i++) p[i] = x[i];
#pragma unroll
					for (int s = 0; s < S; s++) { hx[s][0] = wrk[s][0]; hx[s][1] = wrk[s][1]; }
					p_eL2 = pDp_eL2;
					updp = 1;
					++k;
				} else {
					mu *= nu;
					const int nu2 = nu << 1;
					if (nu2 <= nu) finish(5);
					else { nu = nu2; ++k; }
				}
			}
		}
	}
}

// inlier count of every sample-fit pose k_pose_fit_stream left (testAllPoints, POSE_..._CPU.hpp:166-180): one 8-lane group per hypothesis
__global__ void __launch_bounds__(256)
k_pose_score(const int32_t *__restrict__ cluster_offsets, const float *__restrict__ xy, const float *__restrict__ xyz,
             const int32_t *__restrict__ image, const Camera *__restrict__ cams, const int32_t *__restrict__ hyp_cluster, int n_hyp, float thr,
             int32_t *__restrict__ n_inliers, const float *__restrict__ pose_lm) {
	const int lane = threadIdx.x & 31, lig = lane & 7, grp = lane >> 3;
	const unsigned mask = 0xFFu << (8 * grp);
	const int h = (blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * 4 + grp;
	if (h >= n_hyp || n_inliers[h] < 0) return;
	const int c = hyp_cluster[h];
	const int lo = cluster_offsets[c], n = cluster_offsets[c + 1] - lo;
	float pose[7];
#pragma unroll
	for (int j = 0; j < 7; j++) pose[j] = pose_lm[7 * h + j];
	const int cnt = count_inliers<8>(pose, n, xy + 2 * lo, xyz + 3 * lo, image + lo, cams, thr, mask, lig, nullptr);
	if (lig == 0) n_inliers[h] = cnt;
}

// ---- kernel B: refit of every hypothesis with more than min_npts inliers; one warp per hypothesis ----
__global__ void __launch_bounds__(kPoseThreads)
k_pose_refit(const int32_t *__restrict__ cluster_offsets, const float *__restrict__ xy, const float *__restrict__ xyz,
             const int32_t *__restrict__ image, const Camera *__restrict__ cams, const int32_t *__restrict__ hyp_cluster, int n_hyp,
             int max_lm, float thr, int min_npts, const int32_t *__restrict__ n_inliers, const float *__restrict__ pose_lm,
             float *__restrict__ pose_refit, float *__restrict__ lm_err) {
	__shared__ int s_list[kPoseThreads / 32][kRefitCap];
	const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
	const int h = blockIdx.x * (kPoseThreads / 32) + w;
	if (h >= n_hyp) return;
	float pose[7];
#pragma unroll
	for (int j = 0; j < 7; j++) pose[j] = pose_lm[7 * h + j];
	if (n_inliers[h] > min_npts) {
		const int c = hyp_cluster[h];
		const int lo = cluster_offsets[c], n = cluster_offsets[c + 1] - lo;
		float err;
		refit_warp(pose, n, xy + 2 * lo, xyz + 3 * lo, image + lo, cams, thr, max_lm, lane, s_list[w], err);
		if (lane == 0) lm_err[2 * h + 1] = err;
	}
	if (lane == 0)
		for (int j = 0; j < 7; j++) pose_refit[7 * h + j] = pose[j];
}

// ---- kernel B': the same refit for MANY hypotheses of which few are accepted (the thread-per-hypothesis path) ----
// k_pose_refit gives every hypothesis a warp and compiles for the largest refit (16 correspondences per lane: 255 registers, 8 warps
// per SM). With 131072 hypotheses of which 2 % are accepted (BASELINE configs[3]) that is 128 k idle warps and a latency-bound LM at
// two warps per scheduler. Here k_refit_buckets copies the sample-fit pose of every hypothesis and appends the accepted ones to one of
// five lists by inlier count (<= 32, 64, 128, 256, more); k_pose_refit_list<S> / k_pose_refit_lists<1, 2> then run a persistent grid of warps over a list with S
// correspondences per lane in registers, compiled for that S alone (S = 1, 2: 3 CTAs of 4 warps per SM). Same arithmetic as refit_warp.
constexpr int kRefitBuckets = 5;

__global__ void k_refit_buckets(int n_hyp, int min_npts, const int32_t *__restrict__ n_inliers, const float *__restrict__ pose_lm,
                                float *__restrict__ pose_refit, int32_t *__restrict__ counts, int32_t *__restrict__ lists) {
	const int h = blockIdx.x * blockDim.x + threadIdx.x;
	if (h >= n_hyp) return;
#pragma unroll
	for (int j = 0; j < 7; j++) pose_refit[7 * (size_t)h + j] = pose_lm[7 * (size_t)h + j];
	const int n = n_inliers[h];
	if (n > min_npts) {
		const int b = n <= 32 ? 0 : n <= 64 ? 1 : n <= 128 ? 2 : n <= 256 ? 3 : 4;
		lists[(size_t)b * n_hyp + atomicAdd(&counts[b], 1)] = h;
	}
}

// refit of hypothesis h by the calling warp with S correspondences per lane (list = 32 S ints of shared memory)
template <int S>
__device__ __forceinline__ void refit_item(int h, const int32_t *__restrict__ cluster_offsets, const float *__restrict__ xy, const float *__restrict__ xyz,
                                           const int32_t *__restrict__ image, const Camera *__restrict__ cams, const int32_t *__restrict__ hyp_cluster,
                                           int max_lm, float thr, int lane, int *list, float *__restrict__ pose_refit, float *__restrict__ lm_err) {
	const int c = hyp_cluster[h];
	const int lo = cluster_offsets[c], n = cluster_offsets[c + 1] - lo;
	const float *cxy = xy + 2 * lo, *cxyz = xyz + 3 * lo;
	const int32_t *cim = image + lo;
	float pose[7];
#pragma unroll
	for (int j = 0; j < 7; j++) pose[j] = pose_refit[7 * (size_t)h + j];
	// inliers of `pose` in cluster order (refit_warp's list; the bucket guarantees that at most 32 S of them exist, 512 in the last one)
	float T[12];
	pose7_to_T(pose, T);
	int n_inl = 0;
	for (int i0 = 0; i0 < n; i0 += 32) {
		const int i = i0 + lane;
		bool in = false;
		if (i < n) in = proj_err(T, cams[cim[i]], cxyz[3 * i], cxyz[3 * i + 1], cxyz[3 * i + 2], cxy[2 * i], cxy[2 * i + 1]) < thr;
		const unsigned m = __ballot_sync(0xffffffffu, in);
		if (in) {
			const int k = n_inl + __popc(m & ((1u << lane) - 1));
			if (k < 32 * S) list[k] = i;
		}
		n_inl += __popc(m);
	}
	__syncwarp();
	if (n_inl > 32 * S) n_inl = 32 * S;
	float err;
	refit_S<S>(pose, n_inl, list, cxy, cxyz, cim, cams, max_lm, lane, err);
	if (lane == 0) {
		lm_err[2 * (size_t)h + 1] = err;
#pragma unroll
		for (int j = 0; j < 7; j++) pose_refit[7 * (size_t)h + j] = pose[j];
	}
	__syncwarp();
}

// a persistent grid of warps over TWO lists: the items of list B (SB correspondences per lane, the longer fits) first, then list A
template <int SA, int SB, int MINB>
__global__ void __launch_bounds__(128, MINB)
k_pose_refit_lists(const int32_t *__restrict__ cluster_offsets, const float *__restrict__ xy, const float *__restrict__ xyz,
                   const int32_t *__restrict__ image, const Camera *__restrict__ cams, const int32_t *__restrict__ hyp_cluster, int max_lm, float thr,
                   const int32_t *__restrict__ count_a, const int32_t *__restrict__ list_a, const int32_t *__restrict__ count_b,
                   const int32_t *__restrict__ list_b, float *__restrict__ pose_refit, float *__restrict__ lm_err) {
	__shared__ int s_list[4][32 * SB];
	const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
	const int na = *count_a, nb = *count_b;
	for (int it = blockIdx.x * 4 + w; it < na + nb; it += gridDim.x * 4) {
		if (it < nb) refit_item<SB>(list_b[it], cluster_offsets, xy, xyz, image, cams, hyp_cluster, max_lm, thr, lane, s_list[w], pose_refit, lm_err);
		else refit_item<SA>(list_a[it - nb], cluster_offsets, xy, xyz, image, cams, hyp_cluster, max_lm, thr, lane, s_list[w], pose_refit, lm_err);
	}
}

template <int S, int MINB>
__global__ void __launch_bounds__(128, MINB)
k_pose_refit_list(const int32_t *__restrict__ cluster_offsets, const float *__restrict__ xy, const float *__restrict__ xyz,
                  const int32_t *__restrict__ image, const Camera *__restrict__ cams, const int32_t *__restrict__ hyp_cluster, int max_lm, float thr,
                  const int32_t *__restrict__ count, const int32_t *__restrict__ list, float *__restrict__ pose_refit, float *__restrict__ lm_err) {
	__shared__ int s_list[4][32 * S];
	const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
	const int n_items = *count;
	for (int it = blockIdx.x * 4 + w; it < n_items; it += gridDim.x * 4)
		refit_item<S>(list[it], cluster_offsets, xy, xyz, image, cams, hyp_cluster, max_lm, thr, lane, s_list[w], pose_refit, lm_err);
}

// ---- kernel C: full RANSAC, one CTA per (cluster, try) task ----
// Reference semantics (RANSAC(), :188-211): sequential tests, stop at the FIRST hypothesis whose inlier
// count exceeds min_npts, refit it on its inliers. Here a round evaluates consecutive hypotheses of the task's
// stream in parallel and the lowest-numbered success wins, which is the same hypothesis the sequential loop
// would have stopped at. Latency shaping: the first round runs ONE hypothesis per warp (8 per round: no
// intra-warp divergence between hypotheses, and on real clusters hypothesis 0 usually succeeds); later rounds
// pack four per warp (32 per round). A group whose index is above an already successful one aborts its LM.
// blockDim = 32 x (warps per task, 1..8; mc_set_tuning): fewer warps per task trade the latency of one task for
// more resident tasks per SM when a frame batch brings hundreds of them. The winner does not depend on it.
__global__ void __launch_bounds__(kPoseThreads)
k_pose_ransac(const int32_t *__restrict__ cluster_offsets, const int32_t *__restrict__ n_clusters_p, int n_clusters_cap,
              const float *__restrict__ xy, const float *__restrict__ xyz, const int32_t *__restrict__ image,
              const int32_t *__restrict__ tie, const Camera *__restrict__ cams, int max_obj, int max_ransac, int max_lm, int n_align,
              int min_npts, float thr, uint64_t seed, uint8_t *__restrict__ found, float *__restrict__ pose_out,
              int32_t *__restrict__ n_tests) {
	__shared__ float s_pose[32][7];
	__shared__ int s_list[kRefitCap];
	__shared__ int s_first, s_fail;
	const int task = blockIdx.x;
	const int n_clusters = n_clusters_p ? min(*n_clusters_p, n_clusters_cap) : n_clusters_cap;
	const int c = task / max_obj;
	if (c >= n_clusters) { if (threadIdx.x == 0) { found[task] = 0; n_tests[task] = 0; } return; }
	const int lo = cluster_offsets[c], n = cluster_offsets[c + 1] - lo;
	const float *cxy = xy + 2 * lo, *cxyz = xyz + 3 * lo;
	const int32_t *cim = image + lo, *ctie = tie ? tie + lo : nullptr;
	const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, lig = lane & 7, grp = lane >> 3;
	const int nw = blockDim.x >> 5;
	const unsigned mask = 0xFFu << (8 * grp);
	const uint64_t task_seed = seed + 0x9E3779B97F4A7C15ULL * (uint64_t)(task + 1);
	if (threadIdx.x == 0) { s_first = 0x7fffffff; s_fail = 0; }
	__syncthreads();
	int tests = 0, base = 0;
	while (base < max_ransac) {
		const int hpw = base == 0 ? 1 : 4;                 // hypotheses per warp in this round
		const int slot = w * hpw + grp, h = base + slot;
		if (grp < hpw && h < max_ransac) {
			int cnt = -1;
			float pose[7] = { 0, 0, 0, 1, 0, 0, 0 }, err;
			int pos[kMaxAlign]; float quat[4];
#pragma unroll
			for (int j = 0; j < kMaxAlign; j++) pos[j] = 0;
			if (draw_sample<8>(task_seed, h, n, n_align, cxy, cim, ctie, mask, lig, pos, quat))
				cnt = fit_and_score(pos, n_align, quat, n, cxy, cxyz, cim, cams, max_lm, thr, mask, lig, pose, err, nullptr, &s_first, h);
			else if (lig == 0) s_fail = 1;               // randSample fails for every hypothesis alike -> RANSAC returns false
			if (lig == 0 && cnt > min_npts) {
				for (int j = 0; j < 7; j++) s_pose[slot][j] = pose[j];
				atomicMin(&s_first, h);
			}
		}
		__syncthreads();
		const int first = s_first;
		const int round_n = nw * hpw;
		tests = min(base + round_n, max_ransac);
		if (first != 0x7fffffff) { tests = first + 1; break; }
		if (s_fail) { tests = 0; break; }
		base += round_n;
		__syncthreads();
	}
	const int first = s_first;
	const bool ok = first != 0x7fffffff;
	if (ok && w == 0) {
		const int slot = first - base;
		float pose[7], err;
#pragma unroll
		for (int j = 0; j < 7; j++) pose[j] = s_pose[slot][j];
		refit_warp(pose, n, cxy, cxyz, cim, cams, thr, max_lm, lane, s_list, err);
		if (lane == 0)
			for (int j = 0; j < 7; j++) pose_out[7 * task + j] = pose[j];
	}
	if (threadIdx.x == 0) { found[task] = ok ? 1 : 0; n_tests[task] = tests; }
}

// ---- staged RANSAC (the default path): pose_staged.cuh instantiated with this file's lane-group LM ----
struct DefaultFit {
	static constexpr int kFitSmemFloats = 0;
	static constexpr int kRefitListInts = kRefitCap;
	static constexpr int kRefitFloatsPerPoint = 0, kRefitFloatsPerTask = 0;
	static __device__ __forceinline__ int fit(const int (&pos)[kMaxAlign], int n_align, const float (&quat)[4], int n, const float *xy, const float *xyz,
	                                          const int32_t *image, const Camera *cams, int max_lm, float thr, unsigned mask, int lig, float (&pose)[7],
	                                          float &err, const volatile int *abort_if_below, int my_index, float *) {
		return fit_and_score(pos, n_align, quat, n, xy, xyz, image, cams, max_lm, thr, mask, lig, pose, err, nullptr, abort_if_below, my_index);
	}
	static __device__ __forceinline__ bool refit(float (&pose)[7], int n, const float *xy, const float *xyz, const int32_t *image, const Camera *cams,
	                                            float thr, int max_lm, int lane, int *list, float *, float &err) {
		return refit_warp(pose, n, xy, xyz, image, cams, thr, max_lm, lane, list, err);
	}
};

// append the found poses to an object list in task order (device-side `objects->push_back`, :295-303)
__global__ void k_pose_append(const int32_t *__restrict__ cluster_model, const int32_t *__restrict__ n_clusters_p, int n_clusters_cap,
                              int max_obj, const uint8_t *__restrict__ found, const float *__restrict__ pose, int32_t *__restrict__ n_obj,
                              int obj_cap, int32_t *__restrict__ obj_model, float *__restrict__ obj_pose) {
	if (threadIdx.x != 0 || blockIdx.x != 0) return;
	const int n_clusters = n_clusters_p ? min(*n_clusters_p, n_clusters_cap) : n_clusters_cap;
	int k = *n_obj;
	for (int t = 0; t < n_clusters * max_obj; t++) {
		if (!found[t] || k >= obj_cap) continue;
		obj_model[k] = cluster_model[t / max_obj];
		for (int j = 0; j < 7; j++) obj_pose[7 * k + j] = pose[7 * t + j];
		k++;
	}
	*n_obj = k;
}

// ---- device entries ----
mc_status pose_hypotheses_device(mc_ctx *ctx, const int32_t *d_cluster_offsets, const float *d_xy, const float *d_xyz, const int32_t *d_image,
                                 const int32_t *d_hyp_cluster, const int32_t *d_sample_pos, const float *d_init_quat, int n_hyp,
                                 const mc_pose_params *pp, const int64_t *d_mask_offsets, int32_t *d_n_inliers, float *d_pose_lm,
                                 float *d_pose_refit, float *d_lm_err, uint8_t *d_mask) {
	if (!ctx->d_cams) { ctx->err = "pose: cameras not set (mc_set_cameras)"; return MC_ERR_STATE; }
	if (pp->n_pts_align < 1 || pp->n_pts_align > kMaxAlign) { ctx->err = "pose: n_pts_align must be in 1..8"; return MC_ERR_ARG; }
	if (n_hyp <= 0) return MC_OK;
	const int wpb = kPoseThreads / 32;
	// many hypotheses and no inlier masks wanted: one thread per hypothesis; otherwise one 8-lane group per hypothesis
	if (!d_mask && n_hyp >= ctx->fit_thread_min && ctx->fit_stream) {
		// persistent phase-synchronous kernel + scoring kernel (the default throughput shape)
		DevBuf &b_fit = ctx->scratch[kScrFitStream];
		MC_TRY(reserve(ctx, b_fit, 256));
		MC_CUDA(cudaMemsetAsync(b_fit.p, 0, 256, ctx->stream));
#define MC_FIT_STREAM(S, MINB)                                                                                                               \
		do {                                                                                                                                 \
			const size_t smem = (size_t)(S) * kStreamFloats * kStreamThreads * sizeof(float);                                                           \
			MC_CUDA(cudaFuncSetAttribute(k_pose_fit_stream<S, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));               \
			int per_sm = 0;                                                                                                                  \
			MC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_pose_fit_stream<S, MINB>, kStreamThreads, smem));               \
			if (per_sm < 1) per_sm = 1;                                                                                                      \
			const int64_t want = ((int64_t)n_hyp + kStreamThreads - 1) / kStreamThreads, cap = (int64_t)per_sm * ctx->num_sms;                \
			k_pose_fit_stream<S, MINB><<<(unsigned)(want < cap ? want : cap), kStreamThreads, smem, ctx->stream>>>(                          \
			    d_cluster_offsets, d_xy, d_xyz, d_image, ctx->d_cams, d_hyp_cluster, d_sample_pos, d_init_quat, n_hyp, pp->n_pts_align,      \
			    pp->max_lm_tests, (uint32_t *)b_fit.p, d_n_inliers, d_pose_lm, d_lm_err);                                                    \
		} while (0)
		if (pp->n_pts_align <= 5) MC_FIT_STREAM(5, 3);       // (4 CTAs per SM at 128 registers: measured, no gain — 5.00 vs 4.95 ms per 131072 hypotheses)
		else if (pp->n_pts_align == 6) MC_FIT_STREAM(6, 3);
		else MC_FIT_STREAM(8, 2);
#undef MC_FIT_STREAM
		MC_LAUNCH_CHECK();
		k_pose_score<<<(n_hyp + 31) / 32, 256, 0, ctx->stream>>>(d_cluster_offsets, d_xy, d_xyz, d_image, ctx->d_cams, d_hyp_cluster, n_hyp,
		                                                        pp->error_threshold, d_n_inliers, d_pose_lm);
		MC_LAUNCH_CHECK();
		// refit of the accepted ones from per-size lists
		MC_TRY(reserve(ctx, ctx->scratch[kScrRefitLists], 256 + sizeof(int32_t) * (size_t)kRefitBuckets * n_hyp));
		int32_t *counts = (int32_t *)ctx->scratch[kScrRefitLists].p, *lists = counts + 64;
		MC_CUDA(cudaMemsetAsync(counts, 0, 256, ctx->stream));
		k_refit_buckets<<<(n_hyp + 255) / 256, 256, 0, ctx->stream>>>(n_hyp, pp->min_npts_object, d_n_inliers, d_pose_lm, d_pose_refit, counts, lists);
		MC_LAUNCH_CHECK();
		const int64_t warps_cap = ((int64_t)n_hyp + 3) / 4;
#define MC_REFIT_LIST(S, MINB, B)                                                                                                            \
		do {                                                                                                                                 \
			const int64_t g = (int64_t)ctx->num_sms * (MINB);                                                                                \
			k_pose_refit_list<S, MINB><<<(unsigned)(g < warps_cap ? g : warps_cap), 128, 0, ctx->stream>>>(                                  \
			    d_cluster_offsets, d_xy, d_xyz, d_image, ctx->d_cams, d_hyp_cluster, pp->max_lm_tests, pp->error_threshold, counts + (B),    \
			    lists + (size_t)(B) * n_hyp, d_pose_refit, d_lm_err);                                                                        \
			MC_LAUNCH_CHECK();                                                                                                               \
		} while (0)
		{                                     // the two small buckets share one launch (each alone leaves the GPU half empty for one LM chain length)
			const int64_t g = (int64_t)ctx->num_sms * 3;
			k_pose_refit_lists<1, 2, 3><<<(unsigned)(g < warps_cap ? g : warps_cap), 128, 0, ctx->stream>>>(
			    d_cluster_offsets, d_xy, d_xyz, d_image, ctx->d_cams, d_hyp_cluster, pp->max_lm_tests, pp->error_threshold, counts + 0, lists,
			    counts + 1, lists + (size_t)n_hyp, d_pose_refit, d_lm_err);
			MC_LAUNCH_CHECK();
		}
		MC_REFIT_LIST(4, 2, 2);
		MC_REFIT_LIST(8, 2, 3);
		MC_REFIT_LIST(16, 2, 4);
#undef MC_REFIT_LIST
		return MC_OK;
	} else if (!d_mask && n_hyp >= ctx->fit_thread_min) {
		const int grid = (n_hyp + 127) / 128;
#define MC_FIT_THREAD(S)                                                                                                                     \
		k_pose_fit_thread<S><<<grid, 128, 0, ctx->stream>>>(d_cluster_offsets, d_xy, d_xyz, d_image, ctx->d_cams, d_hyp_cluster, d_sample_pos, \
		                                                   d_init_quat, n_hyp, pp->n_pts_align, pp->max_lm_tests, pp->error_threshold,      \
		                                                   d_n_inliers, d_pose_lm, d_lm_err)
		if (pp->n_pts_align <= 5) MC_FIT_THREAD(5);
		else if (pp->n_pts_align == 6) MC_FIT_THREAD(6);
		else MC_FIT_THREAD(8);
#undef MC_FIT_THREAD
	} else {
		k_pose_fit<<<(n_hyp + wpb * 4 - 1) / (wpb * 4), kPoseThreads, 0, ctx->stream>>>(d_cluster_offsets, d_xy, d_xyz, d_image, ctx->d_cams, d_hyp_cluster,
		                                                                              d_sample_pos, d_init_quat, n_hyp, pp->n_pts_align, pp->max_lm_tests,
		                                                                              pp->error_threshold, d_mask_offsets, d_n_inliers, d_pose_lm, d_lm_err, d_mask);
	}
	MC_LAUNCH_CHECK();
	k_pose_refit<<<(n_hyp + wpb - 1) / wpb, kPoseThreads, 0, ctx->stream>>>(d_cluster_offsets, d_xy, d_xyz, d_image, ctx->d_cams, d_hyp_cluster, n_hyp,
	                                                                      pp->max_lm_tests, pp->error_threshold, pp->min_npts_object, d_n_inliers,
	                                                                      d_pose_lm, d_pose_refit, d_lm_err);
	MC_LAUNCH_CHECK();
	return MC_OK;
}

mc_status pose_ransac_exact_device(mc_ctx *ctx, const int32_t *d_cluster_offsets, const int32_t *d_n_clusters, int n_clusters_cap, int n_points_cap,
                                   const float *d_xy, const float *d_xyz, const int32_t *d_image, const int32_t *d_tie,
                                   const mc_pose_params *pp, uint8_t *d_found, float *d_pose, int32_t *d_n_tests);      // pose_exact.cu

mc_status pose_ransac_device(mc_ctx *ctx, const int32_t *d_cluster_offsets, const int32_t *d_n_clusters, int n_clusters_cap, int n_points_cap,
                             const float *d_xy, const float *d_xyz, const int32_t *d_image, const int32_t *d_tie,
                             const mc_pose_params *pp, uint8_t *d_found, float *d_pose, int32_t *d_n_tests) {
	if (!ctx->d_cams) { ctx->err = "pose: cameras not set (mc_set_cameras)"; return MC_ERR_STATE; }
	if (pp->n_pts_align < 1 || pp->n_pts_align > kMaxAlign) { ctx->err = "pose: n_pts_align must be in 1..8"; return MC_ERR_ARG; }
	const int n_tasks = n_clusters_cap * pp->max_objects_per_cluster;
	if (n_tasks <= 0) return MC_OK;
	const int warps = ctx->pose_warps < 1 ? 1 : (ctx->pose_warps > kPoseThreads / 32 ? kPoseThreads / 32 : ctx->pose_warps);
	if (ctx->pose_exact_order)               // mc_set_option "pose_exact_order": the order-preserving LM (pose_exact.cu), bit-exact with the oracle
		return pose_ransac_exact_device(ctx, d_cluster_offsets, d_n_clusters, n_clusters_cap, n_points_cap, d_xy, d_xyz, d_image, d_tie, pp, d_found, d_pose, d_n_tests);
	if (ctx->ransac_fused && ctx->ransac_shard_world > 1) { ctx->err = "pose: the one-CTA-per-task A/B kernel has no cluster partition"; return MC_ERR_STATE; }
	if (ctx->ransac_fused) {                 // A/B aid (mc_set_option "ransac_fused"): the one-CTA-per-task kernel
		k_pose_ransac<<<n_tasks, 32 * warps, 0, ctx->stream>>>(d_cluster_offsets, d_n_clusters, n_clusters_cap, d_xy, d_xyz, d_image, d_tie, ctx->d_cams,
		                                                       pp->max_objects_per_cluster, pp->max_ransac_tests, pp->max_lm_tests, pp->n_pts_align,
		                                                       pp->min_npts_object, pp->error_threshold, pp->seed, d_found, d_pose, d_n_tests);
		MC_LAUNCH_CHECK();
		return MC_OK;
	}
	return ransac_staged_launch<DefaultFit>(ctx, d_cluster_offsets, d_n_clusters, n_clusters_cap, n_points_cap, d_xy, d_xyz, d_image, d_tie, pp, d_found, d_pose,
	                                        d_n_tests);
}

mc_status pose_append_device(mc_ctx *ctx, const int32_t *d_cluster_model, const int32_t *d_n_clusters, int n_clusters_cap, int max_obj,
                             const uint8_t *d_found, const float *d_pose, int32_t *d_n_obj, int obj_cap, int32_t *d_obj_model, float *d_obj_pose) {
	k_pose_append<<<1, 32, 0, ctx->stream>>>(d_cluster_model, d_n_clusters, n_clusters_cap, max_obj, d_found, d_pose, d_n_obj, obj_cap, d_obj_model, d_obj_pose);
	MC_LAUNCH_CHECK();
	return MC_OK;
}

} // namespace mc
