"""numpy restatement of moped's UNDISTORTED_IMAGE step (UTIL_UNDISTORT): cvInitUndistortMap + cvRemap with CV_INTER_LINEAR +
CV_WARP_FILL_OUTLIERS and fill value 0, for 8-bit gray images.

TEST INFRASTRUCTURE, like the rest of oracle/: the product (moped_b200/csrc/undistort.cuh, undistort.cu) never imports it.
Pinned by tests/golden/undistort_golden.npz (written by OpenCV) and, where cv2 can be imported, by live cv2 in
tests/test_undistort_host.py.

The arithmetic follows OpenCV's scalar loop in double precision with multiply and add kept separate (numpy never fuses them).
One known difference: with kc = 0, map entries within about 1e-13 px of zero can differ from cv2's in their residue; a map entry is
rounded to 1/32 px before use, so remapped images are unaffected."""
from __future__ import annotations

import numpy as np

INTER_BITS = 5
INTER_TAB = 1 << INTER_BITS
COEF_BITS = 15


def _inv3(a):
    """Matx33d::inv(DECOMP_LU) for a 3x3 matrix: cofactors times 1 / det"""
    det = (a[0, 0] * (a[1, 1] * a[2, 2] - a[2, 1] * a[1, 2]) - a[0, 1] * (a[1, 0] * a[2, 2] - a[2, 0] * a[1, 2]) +
           a[0, 2] * (a[1, 0] * a[2, 1] - a[2, 0] * a[1, 1]))
    d = 1.0 / det
    b = np.empty((3, 3))
    b[0, 0] = (a[1, 1] * a[2, 2] - a[1, 2] * a[2, 1]) * d
    b[0, 1] = (a[0, 2] * a[2, 1] - a[0, 1] * a[2, 2]) * d
    b[0, 2] = (a[0, 1] * a[1, 2] - a[0, 2] * a[1, 1]) * d
    b[1, 0] = (a[1, 2] * a[2, 0] - a[1, 0] * a[2, 2]) * d
    b[1, 1] = (a[0, 0] * a[2, 2] - a[0, 2] * a[2, 0]) * d
    b[1, 2] = (a[0, 2] * a[1, 0] - a[0, 0] * a[1, 2]) * d
    b[2, 0] = (a[1, 0] * a[2, 1] - a[1, 1] * a[2, 0]) * d
    b[2, 1] = (a[0, 1] * a[2, 0] - a[0, 0] * a[2, 1]) * d
    b[2, 2] = (a[0, 0] * a[1, 1] - a[0, 1] * a[1, 0]) * d
    return b


def camera_matrix(K):
    """(fx, fy, cx, cy), rounded to float32 as the C ABI takes it, as the 3x3 double matrix cv2 is given"""
    fx, fy, cx, cy = np.asarray(K, np.float32).astype(np.float64)
    return np.array([[fx, 0.0, cx], [0.0, fy, cy], [0.0, 0.0, 1.0]])


def undistort_map(K, kc, H, W):
    """cvInitUndistortMap(K, kc) with newCameraMatrix = K: float32 maps (mx, my) [H, W]. K = (fx, fy, cx, cy), kc = (k1, k2, p1,
    p2[, k3]); both are rounded to float32 first."""
    A = camera_matrix(K)
    k = np.zeros(5)
    kc32 = np.asarray(kc, np.float32).astype(np.float64)
    k[:len(kc32)] = kc32
    k1, k2, p1, p2, k3 = k
    fx, fy, u0, v0 = A[0, 0], A[1, 1], A[0, 2], A[1, 2]
    ir = _inv3(A)
    i = np.arange(H, dtype=np.float64)[:, None]

    def running(r):       # _x = i * ir[r,1] + ir[r,2], then += ir[r,0] per column, in column order
        start = i * ir[r, 1] + ir[r, 2]
        return np.add.accumulate(np.concatenate([start, np.full((H, W - 1), ir[r, 0])], axis=1), axis=1)

    with np.errstate(all="ignore"):
        xs, ys, ws = running(0), running(1), running(2)
        w = 1.0 / ws
        x = xs * w
        y = ys * w
        x2 = x * x
        y2 = y * y
        r2 = x2 + y2
        _2xy = 2 * x * y
        kr = (1 + ((k3 * r2 + k2) * r2 + k1) * r2) / (1 + ((0 * r2 + 0) * r2 + 0) * r2)
        u = fx * (x * kr + p1 * _2xy + p2 * (r2 + 2 * x2)) + u0
        v = fy * (y * kr + p1 * (r2 + 2 * y2) + p2 * _2xy) + v0
        return u.astype(np.float32), v.astype(np.float32)


def _fixed(m):
    """cvRound(32 * m) saturated to int32 (half to even; NaN -> INT32_MIN)"""
    with np.errstate(all="ignore"):
        v = np.rint(m.astype(np.float64) * INTER_TAB)
    v = np.where(np.isnan(v), -2.0 ** 31, v)
    return np.clip(v, -2.0 ** 31, 2.0 ** 31 - 1).astype(np.int64)


def remap_fixed(mx, my):
    """cvRemap's fixed-point map: the top-left source neighbour (sx, sy) saturated to int16, and the fraction index fy * 32 + fx"""
    X, Y = _fixed(mx), _fixed(my)
    sx = np.clip(X >> INTER_BITS, -32768, 32767).astype(np.int16)
    sy = np.clip(Y >> INTER_BITS, -32768, 32767).astype(np.int16)
    frac = ((Y & (INTER_TAB - 1)) * INTER_TAB + (X & (INTER_TAB - 1))).astype(np.uint16)
    return sx, sy, frac


def remap_weights():
    """initInterTab2D(INTER_LINEAR, fixed point): [1024, 4] weights of the neighbours (x, y), (x+1, y), (x, y+1), (x+1, y+1) for
    fraction index fy * 32 + fx"""
    tab = np.zeros((INTER_TAB * INTER_TAB, 4), np.int64)
    one = np.float32(1.0)
    for i in range(INTER_TAB):
        for j in range(INTER_TAB):
            b, a = np.float32(i) * np.float32(1.0 / INTER_TAB), np.float32(j) * np.float32(1.0 / INTER_TAB)
            cy, cx = (one - b, b), (one - a, a)
            t = [int(np.rint(np.float64(np.float32(cy[k1] * cx[k2]) * np.float32(1 << COEF_BITS)))) for k1 in range(2) for k2 in range(2)]
            diff = sum(t) - (1 << COEF_BITS)
            if diff:
                t[int(np.argmax(t)) if diff < 0 else int(np.argmin(t))] -= diff
            tab[i * INTER_TAB + j] = t
    return tab


def remap_linear_u8(img, maps):
    """cvRemap(img, mapx, mapy, CV_INTER_LINEAR + CV_WARP_FILL_OUTLIERS, fill 0) of one [H, W] or a batch [B, H, W] of uint8
    images; maps = (mx, my) float32 [H, W]"""
    img = np.asarray(img, np.uint8)
    batch = img.reshape((-1,) + img.shape[-2:])
    H, W = batch.shape[1:]
    sx, sy, frac = remap_fixed(*maps)
    sx, sy = sx.astype(np.int64), sy.astype(np.int64)
    wt = remap_weights()[frac]
    out = np.empty_like(batch)
    for b, im in enumerate(batch):
        s = np.zeros(sx.shape, np.int64)
        for k, (dy, dx) in enumerate(((0, 0), (0, 1), (1, 0), (1, 1))):
            yy, xx = sy + dy, sx + dx
            ok = (yy >= 0) & (yy < H) & (xx >= 0) & (xx < W)
            p = np.zeros(sx.shape, np.int64)
            p[ok] = im[yy[ok], xx[ok]]
            s += wt[..., k] * p
        out[b] = np.minimum((s + (1 << (COEF_BITS - 1))) >> COEF_BITS, 255)
    return out.reshape(img.shape)


def undistort(img, K, kc):
    """UNDISTORTED_IMAGE of one image or a batch of one camera"""
    H, W = np.asarray(img).shape[-2:]
    return remap_linear_u8(img, undistort_map(K, kc, H, W))
