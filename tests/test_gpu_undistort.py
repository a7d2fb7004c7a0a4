"""UNDISTORTED_IMAGE on the device (mc_set_undistortion, mc_undistort, mc_undistort_dev, and mc_process_images with a camera-0
table) against the numpy restatement oracle/undistort.py, bit for bit."""
import os

import numpy as np
import pytest

from oracle import undistort as U
from undistort_cases import CAMERAS, SIZES, camera_K, images

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BARREL = CAMERAS["barrel"]


@pytest.fixture(scope="module")
def ctx():
    from moped_b200 import capi
    c = capi.Context(0)          # its own context: a camera-0 table would change mc_process_images for the shared one
    yield c
    c.close()


def _distinct(H, W):
    """six distinct images: random and blurred of two seeds, all 0, all 255"""
    a, b = images(H, W, 0), images(H, W, 1)
    return np.stack([a["random"], a["blurred"], b["random"], b["blurred"], a["zeros"], a["full"]])


def _batch(distinct, B):
    idx = np.arange(B) % len(distinct)
    return np.ascontiguousarray(distinct[idx]), idx


@pytest.mark.gpu
@pytest.mark.parametrize("H,W", SIZES)
def test_undistort_equals_oracle(ctx, H, W):
    import torch
    K = camera_K(H, W)
    distinct = _distinct(H, W)
    for name, kc in CAMERAS.items():
        ctx.set_undistortion(0, K, kc, H, W)
        ref = U.remap_linear_u8(distinct, U.undistort_map(K, kc, H, W))
        for B in (1, 7, 64):
            batch, idx = _batch(distinct, B)
            assert np.array_equal(ctx.undistort(batch), ref[idx]), (name, B)
        batch, idx = _batch(distinct, 64)
        d_in = torch.from_numpy(batch).cuda()
        d_out = torch.empty_like(d_in)
        torch.cuda.synchronize()
        ctx.undistort_dev(d_in.data_ptr(), 64, H, W, d_out.data_ptr())
        ctx.synchronize()
        assert np.array_equal(d_out.cpu().numpy(), ref[idx]), (name, "dev")


@pytest.mark.gpu
def test_two_cameras_replace_and_clear(ctx):
    from moped_b200 import capi
    H, W = 480, 640
    K = camera_K(H, W)
    ims = _distinct(H, W)
    ctx.set_undistortion(0, K, BARREL, H, W)
    ctx.set_undistortion(3, K, CAMERAS["pincushion"], H, W)
    assert np.array_equal(ctx.undistort(ims, 0), U.undistort(ims, K, BARREL))
    assert np.array_equal(ctx.undistort(ims, 3), U.undistort(ims, K, CAMERAS["pincushion"]))
    # setting a camera again replaces its table, also with another size
    K2 = camera_K(479, 641)
    ims2 = _distinct(479, 641)
    ctx.set_undistortion(3, K2, CAMERAS["k3"], 479, 641)
    assert np.array_equal(ctx.undistort(ims2, 3), U.undistort(ims2, K2, CAMERAS["k3"]))
    assert np.array_equal(ctx.undistort(ims, 0), U.undistort(ims, K, BARREL))
    ctx.set_undistortion(3, None, None, 0, 0)
    with pytest.raises(capi.MopedCudaError, match=r"\(-3\)"):
        ctx.undistort(ims2, 3)
    with pytest.raises(capi.MopedCudaError, match=r"\(-3\)"):
        ctx.undistort(ims, 5)
    assert np.array_equal(ctx.undistort(ims, 0), U.undistort(ims, K, BARREL))


@pytest.mark.gpu
def test_argument_errors_keep_the_table(ctx):
    from moped_b200 import capi
    H, W = 480, 640
    K = camera_K(H, W)
    ims = _distinct(H, W)
    ctx.set_undistortion(1, K, BARREL, H, W)
    want = U.undistort(ims, K, BARREL)
    nan, inf = float("nan"), float("inf")
    bad_set = [
        (-1, K, BARREL, H, W), (16, K, BARREL, H, W),                      # camera outside 0..15
        (1, K, (0.1, 0.2, 0.0), H, W), (1, K, (0.1,) * 6, H, W),         # n_kc 3 and 6
        (1, K, (nan, 0, 0, 0), H, W), (1, K, (0, 0, 0, inf, 0), H, W),   # non-finite kc
        (1, (nan, 800, 320, 240), BARREL, H, W), (1, (800, 800, inf, 240), BARREL, H, W),
        (1, (0, 800, 320, 240), BARREL, H, W), (1, (800, 0, 320, 240), BARREL, H, W),
        (1, K, BARREL, 7, W), (1, K, BARREL, H, 7), (1, K, BARREL, 32768, W), (1, K, BARREL, H, 32768),
    ]
    for args in bad_set:
        with pytest.raises(capi.MopedCudaError, match=r"\(-2\)"):
            ctx.set_undistortion(*args)
        assert np.array_equal(ctx.undistort(ims, 1), want), args
    with pytest.raises(capi.MopedCudaError, match=r"\(-2\)"):
        ctx.set_undistortion(16, None, None, 0, 0)
    for bad in (ims[:, :, :-1], ims[:, :-1, :]):                          # a size other than the table's
        with pytest.raises(capi.MopedCudaError, match=r"\(-2\)"):
            ctx.undistort(np.ascontiguousarray(bad), 1)
    with pytest.raises(capi.MopedCudaError, match=r"\(-2\)"):
        ctx.undistort(ims, 16)
    with pytest.raises(capi.MopedCudaError, match=r"\(-2\)"):
        ctx.undistort_dev(0, 1, H, W, 0, 1)
    assert np.array_equal(ctx.undistort(ims, 1), want)


@pytest.fixture(scope="module")
def real_frames():
    g = dict(np.load(os.path.join(ROOT, "tests", "golden", "real_images.npz")))
    sg = np.load(os.path.join(ROOT, "tests", "golden", "sift_golden.npz"))
    im = sg["bag4_full_double/image"]
    shifted = [np.roll(im, s, axis=1) for s in range(-4, 4)]
    return g, np.stack(shifted)


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 64])
@pytest.mark.parametrize("double_size", [0, 1])
def test_process_images_with_table(ctx, real_frames, B, double_size):
    """a camera-0 table: the same objects, poses, scores, feature counts and frame info as mc_process_images without a table on
    images the oracle undistorted; the call launches exactly the remap kernel more"""
    from moped_b200 import capi
    g, distinct = real_frames
    H, W = distinct.shape[1:]
    K = g["K"][0]
    kc = (-0.2, 0.05, 0.001, -0.0005)
    ctx.db_upload(g["db_desc"], g["db_xyz"], g["model_of_row"], len(g["n_pts"]))
    ctx.set_cameras(g["K"], g["cam_pose"])
    ctx.set_tuning(8, 8, 1)
    ref = U.remap_linear_u8(distinct, U.undistort_map(K, kc, H, W))
    idx = np.arange(B) % len(distinct)
    raw, und = np.ascontiguousarray(distinct[idx]), np.ascontiguousarray(ref[idx])

    def run(table):
        if table:
            ctx.set_undistortion(0, K, kc, H, W)
        else:
            ctx.set_undistortion(0, None, None, 0, 0)
        l0 = ctx.launches
        out = ctx.process_images(raw if table else und, bool(double_size), max_keypoints=2048, max_objects=64)
        return out, ctx.launches - l0

    run(False), run(True)                # first calls of this shape: plans, lanes and graphs
    plain, n_plain = run(False)
    with_table, n_table = run(True)
    assert n_table == n_plain + 1, (n_table, n_plain)
    assert sum(o["n_features"] for o in plain) > 0
    if double_size:                      # the bench's setting finds the planar models; at input size there may be too few features
        assert sum(len(o["model"]) for o in plain) > 0
    for a, b in zip(plain, with_table):
        assert a["n_features"] == b["n_features"]
        assert np.array_equal(a["info"], b["info"])
        assert np.array_equal(a["model"], b["model"]) and np.array_equal(a["pose"], b["pose"]) and np.array_equal(a["score"], b["score"])
    # a size other than the table's: MC_ERR_ARG before any launch
    l0 = ctx.launches
    with pytest.raises(capi.MopedCudaError, match=r"\(-2\)"):
        ctx.process_images(np.ascontiguousarray(raw[:, :-8]), bool(double_size), max_keypoints=2048, max_objects=64)
    assert ctx.launches == l0
    ctx.set_undistortion(0, None, None, 0, 0)
