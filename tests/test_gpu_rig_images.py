"""mc_process_rig_images: camera-rig frames from pixels to objects in one call (per-camera UNDISTORTED_IMAGE, SIFT on every image, the
frame's query list in camera order with imageIdx = camera, MATCH..FILTER2), bit for bit against the route a host assembles itself from
oracle-undistorted images, mc_sift_extract and mc_process_frames; against the oracle's stage chain in exact-order mode; and against
mc_process_images where a rig is one camera."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle_chain
from oracle import undistort as U

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MAX_KP = 2048
# one lens per camera: barrel, pincushion with k3, mild barrel with tangential terms
LENSES = [(-0.2, 0.05, 0.001, -0.0005), (0.1, -0.02, 0.0, 0.0005, 0.01), (-0.05, 0.0, -0.001, 0.0)]
# camera 0 at the origin; camera 1 turned 3 degrees about y and 0.1 m to the side; camera 2 turned 2 degrees about x, 0.1 m up
_S3, _C3, _S2, _C2 = np.sin(np.radians(1.5)), np.cos(np.radians(1.5)), np.sin(np.radians(1.0)), np.cos(np.radians(1.0))
POSES = np.array([[0, 0, 0, 1, 0, 0, 0], [0, _S3, 0, _C3, 0.1, 0, 0], [_S2, 0, 0, _C2, 0, 0.1, 0]], np.float32)
SOME = {2: (1,), 3: (0, 2)}        # cameras with a table in the "some" configuration


@pytest.fixture(scope="module")
def rig():
    from moped_b200 import capi
    g = dict(np.load(os.path.join(ROOT, "tests", "golden", "real_images.npz")))
    im = np.load(os.path.join(ROOT, "tests", "golden", "sift_golden.npz"))["bag4_full_double/image"]
    distinct = np.stack([np.roll(im, s, axis=1) for s in range(-4, 4)])
    H, W = distinct.shape[1:]
    K = g["K"][0]
    und = [U.remap_linear_u8(distinct, U.undistort_map(K, kc, H, W)) for kc in LENSES]
    ctx = capi.Context(0)          # its own context: the rig's tables would change mc_process_images for the shared one
    ctx.db_upload(g["db_desc"], g["db_xyz"], g["model_of_row"], len(g["n_pts"]))
    ctx.set_tuning(8, 8, 1)
    yield dict(ctx=ctx, g=g, im=im, distinct=distinct, und=und, K=K, H=H, W=W)
    ctx.close()


def _slots(B, Cn):
    """which of the 8 shifted images frame f shows on camera c"""
    return (3 * np.arange(B)[:, None] + 5 * np.arange(Cn)[None, :]) % 8


def _set_cameras(r, Cn):
    r["ctx"].set_cameras(np.tile(r["K"], (Cn, 1)), POSES[:Cn])


def _set_tables(r, tables):
    ctx = r["ctx"]
    for c in range(16):
        ctx.set_undistortion(c, None, None, 0, 0)
    for c in tables:
        ctx.set_undistortion(c, r["K"], LENSES[c], r["H"], r["W"])


def _normalise(desc):
    ss = np.zeros(len(desc), np.float32)
    for k in range(128):
        ss = ss + desc[:, k] * desc[:, k]                                  # sequential fp32 sum like MATCH_CUDA::normalise
    return desc * (1.0 / np.sqrt(ss).astype(np.float64)).astype(np.float32)[:, None]


def _host_features(r, slots, tables, double_size):
    """the route a host takes without mc_process_rig_images: each camera's images undistorted (here by the oracle; raw without a
    table), mc_sift_extract, each frame's keypoints concatenated in camera order with q_image = camera, MATCH's normalisation"""
    B, Cn = slots.shape
    per_cam = []
    for c in range(Cn):
        src = r["und"][c] if c in tables else r["distinct"]
        per_cam.append(r["ctx"].sift(np.ascontiguousarray(src[slots[:, c]]), bool(double_size), MAX_KP))
    frames = []
    for f in range(B):
        xy = [per_cam[c][f][0] for c in range(Cn)]
        q = [_normalise(per_cam[c][f][2]) for c in range(Cn)]
        img = [np.full(len(x), c, np.int32) for c, x in enumerate(xy)]
        frames.append((np.concatenate(q), np.concatenate(xy), np.concatenate(img), np.array([len(x) for x in xy], np.int32)))
    return frames


def _host_route(r, slots, tables, double_size):
    frames = _host_features(r, slots, tables, double_size)
    _set_tables(r, ())
    fo = np.concatenate([[0], np.cumsum([len(q) for q, _, _, _ in frames])]).astype(np.int32)
    out = r["ctx"].process_frames(np.concatenate([q for q, _, _, _ in frames]), np.concatenate([xy for _, xy, _, _ in frames]),
                                  np.concatenate([im for _, _, im, _ in frames]), fo, max_objects=64)
    for o, fr in zip(out, frames):
        o["n_features"] = fr[3]
    return out, frames


def _rig_call(r, slots, tables, double_size):
    _set_tables(r, tables)
    raw = np.ascontiguousarray(r["distinct"][slots])
    l0 = r["ctx"].launches
    out = r["ctx"].process_rig_images(raw, bool(double_size), max_keypoints=MAX_KP, max_objects=64)
    return out, r["ctx"].launches - l0


def _assert_same(a_list, b_list, what):
    assert len(a_list) == len(b_list)
    for f, (a, b) in enumerate(zip(a_list, b_list)):
        assert np.array_equal(np.asarray(a["n_features"]), np.asarray(b["n_features"])), (what, f)
        assert np.array_equal(a["info"], b["info"]), (what, f, a["info"], b["info"])
        assert np.array_equal(a["model"], b["model"]), (what, f, a["model"], b["model"])
        assert np.array_equal(a["pose"], b["pose"]), (what, f)
        assert np.array_equal(a["score"], b["score"]), (what, f)


@pytest.mark.parametrize("double_size", [0, 1])
@pytest.mark.parametrize("B", [1, 7])
@pytest.mark.parametrize("Cn", [2, 3])
def test_rig_call_equals_host_assembled_route(rig, Cn, B, double_size):
    r = rig
    _set_cameras(r, Cn)
    slots = _slots(B, Cn)
    found = 0
    for tables in (tuple(range(Cn)), SOME[Cn], ()):
        out, _ = _rig_call(r, slots, tables, double_size)
        want, _ = _host_route(r, slots, tables, double_size)
        _assert_same(out, want, (Cn, B, double_size, tables))
        assert all(o["n_features"].shape == (Cn,) for o in out)
        found += sum(len(o["model"]) for o in out)
        assert sum(int(o["n_features"].sum()) for o in out) > 0
    if double_size:                # the bench's setting finds the planar models
        assert found > 0
    _set_tables(r, ())


def test_exact_order_rig_frames_equal_the_oracle_chain(rig):
    """pose_exact_order: every rig frame's objects equal the oracle's chain on the features the device extracted, with each match
    projected through its own camera"""
    r = rig
    g, ctx = r["g"], r["ctx"]
    Cn, B = 2, 3
    _set_cameras(r, Cn)
    slots = _slots(B, Cn)
    tables = (1,)
    ctx.set_option("pose_exact_order", 1)
    try:
        out, _ = _rig_call(r, slots, tables, 1)
    finally:
        ctx.set_option("pose_exact_order", 0)
        _set_tables(r, ())
    frames = _host_features(r, slots, tables, 1)
    Ks = np.tile(r["K"], (Cn, 1))
    found = 0
    for f, (q, xy, img, nf) in enumerate(frames):
        assert np.array_equal(out[f]["n_features"], nf), f
        assert set(np.unique(img).tolist()) == set(range(Cn)), f
        want = oracle_chain.frame(g["db_desc"], g["db_xyz"], g["model_of_row"], len(g["n_pts"]), q, xy, img, Ks, POSES[:Cn], n_images=Cn)
        assert np.array_equal(out[f]["model"], want["model"]), (f, out[f]["model"], want["model"])
        assert np.array_equal(out[f]["pose"], want["pose"]), f
        assert np.array_equal(out[f]["score"], want["score"]), f
        found += len(want["model"])
        # the frame's objects come from both cameras' matches
        assert set(want["matches"]["image"].tolist()) == set(range(Cn)), f
    assert found > 0


def test_a_blank_camera_changes_nothing(rig):
    r = rig
    ctx = r["ctx"]
    _set_tables(r, ())
    frames = np.stack([r["im"], r["distinct"][1]])
    blank = np.zeros_like(frames)
    ctx.set_cameras(r["g"]["K"], r["g"]["cam_pose"])
    alone = ctx.process_images(frames, True, max_keypoints=MAX_KP, max_objects=64)
    assert sum(len(o["model"]) for o in alone) > 0
    ctx.set_cameras(np.tile(r["g"]["K"], (2, 1)), np.tile(r["g"]["cam_pose"], (2, 1)))
    for pos in (0, 1):
        gray = np.stack([blank, frames], axis=1) if pos == 1 else np.stack([frames, blank], axis=1)
        out = ctx.process_rig_images(gray, True, max_keypoints=MAX_KP, max_objects=64)
        for a, o in zip(alone, out):
            assert o["n_features"][1 - pos] == 0 and o["n_features"][pos] == a["n_features"], (pos, o["n_features"])
            assert np.array_equal(o["info"], a["info"]), pos
            assert np.array_equal(o["model"], a["model"]) and np.array_equal(o["pose"], a["pose"]) and np.array_equal(o["score"], a["score"]), pos


@pytest.mark.parametrize("table", [False, True])
def test_one_camera_is_process_images(rig, table):
    r = rig
    ctx = r["ctx"]
    _set_cameras(r, 1)
    _set_tables(r, (0,) if table else ())
    raw = np.ascontiguousarray(r["distinct"][_slots(5, 1)[:, 0]])

    def images():
        l0 = ctx.launches
        return ctx.process_images(raw, True, max_keypoints=MAX_KP, max_objects=64), ctx.launches - l0

    def rig_images():
        l0 = ctx.launches
        return ctx.process_rig_images(raw[:, None], True, max_keypoints=MAX_KP, max_objects=64), ctx.launches - l0

    images(), rig_images()             # first calls of this shape: plans, lanes and graphs
    a, na = images()
    b, nb = rig_images()
    assert na == nb, (na, nb)
    for x, y in zip(a, b):
        y["n_features"] = int(y["n_features"][0])
    _assert_same(a, b, table)
    assert sum(len(o["model"]) for o in a) > 0
    _set_tables(r, ())


@pytest.mark.parametrize("Cn", [2, 3])
def test_remap_is_one_launch_for_the_batch(rig, Cn):
    """tables on some cameras cost exactly one launch more than the same rig without tables on images the oracle undistorted"""
    r = rig
    ctx = r["ctx"]
    _set_cameras(r, Cn)
    B = 4
    slots = _slots(B, Cn)
    tables = SOME[Cn]
    pre = np.ascontiguousarray(np.stack([(r["und"][c] if c in tables else r["distinct"])[slots[:, c]] for c in range(Cn)], axis=1))

    def call_a():
        return _rig_call(r, slots, tables, 1)

    def call_b():
        _set_tables(r, ())
        l0 = ctx.launches
        out = ctx.process_rig_images(pre, True, max_keypoints=MAX_KP, max_objects=64)
        return out, ctx.launches - l0

    call_a(), call_b()
    a, na = call_a()
    b, nb = call_b()
    assert na == nb + 1, (na, nb)
    _assert_same(a, b, Cn)


def _raw_rig(ctx, gray, n_frames, n_cameras, H, W, max_kp=MAX_KP):
    """the C entry itself: status and n_features, also on failure"""
    p = ctx.default_params()
    n = np.zeros(max(n_frames, 1), np.int32)
    om = np.zeros(max(n_frames, 1) * 64, np.int32)
    op = np.zeros(max(n_frames, 1) * 64 * 7, np.float32)
    os_ = np.zeros(max(n_frames, 1) * 64, np.float32)
    nf = np.full(max(n_frames * n_cameras, 1), -1, np.int32)
    st = ctx.L.mc_process_rig_images(ctx.h, gray.reshape(-1), n_frames, n_cameras, H, W, 1, max_kp, C.byref(p), 64, n, om, op, os_,
                                     nf.ctypes.data, None, None)
    return st, nf


def test_errors_launch_nothing_and_keep_the_tables(rig):
    from moped_b200 import capi
    r = rig
    ctx, K, H, W = r["ctx"], r["K"], r["H"], r["W"]
    _set_cameras(r, 2)
    _set_tables(r, (0, 1))
    ims = r["distinct"][:2]
    gray = np.ascontiguousarray(np.stack([ims, ims], axis=1))          # 2 frames x 2 cameras
    ARG, STATE = -2, -3
    cases = [
        ("0 cameras", np.zeros(1, np.uint8), 1, 0, H, W, ARG),
        ("17 cameras", np.zeros(17 * H * W, np.uint8), 1, 17, H, W, ARG),
        ("65536 images", np.zeros(4096 * 16 * 64, np.uint8), 4096, 16, 8, 8, ARG),
        ("a table of another size", np.ascontiguousarray(gray[..., :-8]), 2, 2, H, W - 8, ARG),
        ("3 cameras, 2 set", np.ascontiguousarray(np.stack([ims, ims, ims], axis=1)), 2, 3, H, W, STATE),
    ]
    for what, buf, nfr, ncam, h, w, want in cases:
        l0 = ctx.launches
        st, _ = _raw_rig(ctx, buf, nfr, ncam, h, w)
        assert st == want, (what, st, ctx.L.mc_last_error(ctx.h))
        assert ctx.launches == l0, what
    # only camera 1's table has the other size: still MC_ERR_ARG before any launch
    ctx.set_undistortion(1, K, LENSES[1], H, W - 8)
    l0 = ctx.launches
    assert _raw_rig(ctx, gray, 2, 2, H, W)[0] == ARG and ctx.launches == l0
    ctx.set_undistortion(1, K, LENSES[1], H, W)
    for c in (0, 1):                                                   # the tables are still the ones set
        assert np.array_equal(ctx.undistort(ims, c), r["und"][c][:2]), c
    # no database, a database that is not 128-d
    other = capi.Context(0)
    try:
        other.set_cameras(np.tile(K, (2, 1)), POSES[:2])
        l0 = other.launches
        assert _raw_rig(other, gray, 2, 2, H, W)[0] == STATE and other.launches == l0
        rng = np.random.default_rng(3)
        other.db_upload(rng.random((300, 64), np.float32), rng.random((300, 3), np.float32), np.zeros(300, np.int32), 1)
        l0 = other.launches
        assert _raw_rig(other, gray, 2, 2, H, W)[0] == STATE and other.launches == l0
    finally:
        other.close()
    # more keypoints than max_keypoints in an image: MC_ERR_CAPACITY, n_features still per image
    _set_tables(r, ())
    full = ctx.process_rig_images(gray, True, max_keypoints=MAX_KP)
    counts = np.stack([o["n_features"] for o in full]).reshape(-1)
    blank = np.ascontiguousarray(np.stack([ims, np.zeros_like(ims)], axis=1))
    st, nf = _raw_rig(ctx, blank, 2, 2, H, W, max_kp=100)
    assert st == capi.MC_ERR_CAPACITY, st
    assert np.array_equal(nf, [counts[0], 0, counts[2], 0]), (nf, counts)
    with pytest.raises(capi.MopedCudaError, match="max_keypoints"):
        ctx.process_rig_images(gray, True, max_keypoints=100)
