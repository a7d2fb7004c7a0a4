"""UNDISTORTED_IMAGE without a GPU: the numpy restatement (oracle/undistort.py) against OpenCV — the golden file always, live cv2
when it can be imported — and the host-compiled table builder and per-pixel function of the CUDA path
(moped_b200/csrc/undistort.cuh via tests/cpp/undistort_host.cpp) against the restatement, bit for bit. The device kernel itself is
checked by tests/test_gpu_undistort.py."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import undistort as U
from undistort_cases import CAMERAS, SIZES, assert_maps_match, camera_K, images

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_f32p = np.ctypeslib.ndpointer(dtype=np.float32, flags="C_CONTIGUOUS")
_u8p = np.ctypeslib.ndpointer(dtype=np.uint8, flags="C_CONTIGUOUS")
_i16p = np.ctypeslib.ndpointer(dtype=np.int16, flags="C_CONTIGUOUS")
_u16p = np.ctypeslib.ndpointer(dtype=np.uint16, flags="C_CONTIGUOUS")


@pytest.fixture(scope="module")
def host_lib():
    out_dir = os.path.join(ROOT, "tests", "_build")
    os.makedirs(out_dir, exist_ok=True)
    out = os.path.join(out_dir, "libundistort_host.so")
    src = os.path.join(ROOT, "tests", "cpp", "undistort_host.cpp")
    deps = [src, os.path.join(ROOT, "moped_b200", "csrc", "undistort.cuh")]
    if not os.path.exists(out) or any(os.path.getmtime(d) > os.path.getmtime(out) for d in deps):
        subprocess.check_call(["g++", "-x", "c++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-Wall", "-o", out, src])
    L = C.CDLL(out)
    L.uh_maps.restype = None
    L.uh_maps.argtypes = [_f32p, _f32p, C.c_int, C.c_int, C.c_int, _f32p, _f32p]
    L.uh_entries.restype = None
    L.uh_entries.argtypes = [C.c_int, _f32p, _f32p, _i16p, _i16p, _u16p]
    L.uh_weights.restype = None
    L.uh_weights.argtypes = [_u16p]
    L.uh_undistort.restype = None
    L.uh_undistort.argtypes = [_f32p, _f32p, C.c_int, _u8p, C.c_int, C.c_int, C.c_int, _u8p]
    return L


@pytest.fixture(scope="module")
def golden():
    return dict(np.load(os.path.join(ROOT, "tests", "golden", "undistort_golden.npz")))


def test_weight_table():
    """initInterTab2D for bilinear: every fraction's four weights sum to 2^15; whole pixels weigh 2^15 on one neighbour"""
    w = U.remap_weights()
    assert (w.sum(axis=1) == 1 << 15).all() and (w >= 0).all()
    assert list(w[0]) == [1 << 15, 0, 0, 0]
    assert list(w[16 * 32 + 16]) == [1 << 13] * 4


def test_oracle_equals_golden(golden):
    cams = sorted({k.split("/")[0] for k in golden if "/" in k})
    assert cams == sorted(CAMERAS)
    n = 0
    for key in golden:
        if not key.endswith("/mx"):
            continue
        base = key[:-3]
        H, W = map(int, base.split("/")[1].split("x"))
        mx, my = U.undistort_map(golden[base + "/K"], golden[base + "/kc"], H, W)
        if base + "/rows" in golden:
            mx, my = mx[golden[base + "/rows"]], my[golden[base + "/rows"]]
        else:
            assert np.array_equal(U.remap_linear_u8(golden[base + "/img"], (mx, my)), golden[base + "/out"]), base
            assert np.array_equal(U.remap_linear_u8(golden[base + "/img"], (golden[base + "/mx"], golden[base + "/my"])), golden[base + "/out"]), base
        assert_maps_match(mx, golden[key], base + " x")
        assert_maps_match(my, golden[base + "/my"], base + " y")
        n += 1
    assert n == 3 * len(CAMERAS)


@pytest.mark.parametrize("H,W", SIZES)
def test_oracle_equals_cv2(H, W):
    cv2 = pytest.importorskip("cv2")
    K = camera_K(H, W)
    A = U.camera_matrix(K)
    ims = images(H, W)
    for name, kc in CAMERAS.items():
        kc64 = np.asarray(kc, np.float32).astype(np.float64)
        cmx, cmy = cv2.initUndistortRectifyMap(A, kc64, None, A, (W, H), cv2.CV_32FC1)
        mx, my = U.undistort_map(K, kc, H, W)
        assert_maps_match(mx, cmx, name)
        assert_maps_match(my, cmy, name)
        for kind, im in ims.items():
            ref = cv2.remap(im, cmx, cmy, cv2.INTER_LINEAR, borderMode=cv2.BORDER_CONSTANT, borderValue=0)
            assert np.array_equal(U.remap_linear_u8(im, (mx, my)), ref), (name, kind)


@pytest.mark.parametrize("H,W", SIZES)
def test_host_table_builder_equals_oracle(host_lib, H, W):
    K = camera_K(H, W)
    ims = images(H, W)
    batch = np.stack(list(ims.values()))
    w = np.zeros(1024 * 4, np.uint16)
    host_lib.uh_weights(w)
    assert np.array_equal(w.reshape(1024, 4), U.remap_weights())
    for name, kc in CAMERAS.items():
        kc32 = np.asarray(kc, np.float32)
        mx, my = np.zeros((H, W), np.float32), np.zeros((H, W), np.float32)
        host_lib.uh_maps(K, kc32, len(kc32), H, W, mx, my)
        omx, omy = U.undistort_map(K, kc, H, W)
        assert np.array_equal(mx, omx) and np.array_equal(my, omy), name
        sx, sy, fr = np.zeros(H * W, np.int16), np.zeros(H * W, np.int16), np.zeros(H * W, np.uint16)
        host_lib.uh_entries(H * W, mx.reshape(-1), my.reshape(-1), sx, sy, fr)
        osx, osy, ofr = U.remap_fixed(omx, omy)
        assert np.array_equal(sx, osx.reshape(-1)) and np.array_equal(sy, osy.reshape(-1)) and np.array_equal(fr, ofr.reshape(-1)), name
        out = np.zeros_like(batch)
        host_lib.uh_undistort(K, kc32, len(kc32), batch, len(batch), H, W, out)
        assert np.array_equal(out, U.remap_linear_u8(batch, (omx, omy))), name


def test_extreme_camera_saturates():
    """the extreme camera sends parts of the map past int16 and 32 * u past int32: those pixels read the fill value 0, and pixels
    whose neighbours straddle the border mix the image with 0"""
    H, W = 480, 640
    mx, my = U.undistort_map(camera_K(H, W), CAMERAS["extreme"], H, W)
    assert (np.abs(mx.astype(np.float64)) * 32 > 2 ** 31).any()
    sx, sy, _ = U.remap_fixed(mx, my)
    assert (sx == 32767).any() and (sx == -32768).any()
    out = U.remap_linear_u8(np.full((H, W), 255, np.uint8), (mx, my))
    assert (out == 0).any() and (out == 255).any() and ((out > 0) & (out < 255)).any()
