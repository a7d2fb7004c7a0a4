"""mc_process_rig_cameras / _dev: camera-rig frames whose cameras differ in image size, from host or device memory. Cameras of one size
run as one SIFT batch and the groups' keypoints are merged into each frame's query list in camera order. Compared bit for bit with the
route a host assembles itself (oracle-undistorted images, per-camera mc_sift_extract, concatenation, mc_process_frames), with the
oracle's stage chain in exact-order mode, and with mc_process_rig_images / mc_process_images where every camera has one size."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle_chain
from oracle import undistort as U

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MAX_KP = 2048
LENSES = [(-0.2, 0.05, 0.001, -0.0005), (0.1, -0.02, 0.0, 0.0005, 0.01), (-0.05, 0.0, -0.001, 0.0)]
_S3, _C3, _S2, _C2 = np.sin(np.radians(1.5)), np.cos(np.radians(1.5)), np.sin(np.radians(1.0)), np.cos(np.radians(1.0))
POSES = np.array([[0, 0, 0, 1, 0, 0, 0], [0, _S3, 0, _C3, 0.1, 0, 0], [_S2, 0, 0, _C2, 0, 0.1, 0]], np.float32)
SOME = {2: (1,), 3: (0, 2)}        # cameras with a table in the "some" configuration
ARG, STATE = -2, -3
# camera kinds (rig fixture), all cut from the 640x480 bag image: A the full frame, C a 512x384 centre crop, O an odd-size 637x479
# crop (the remap's scalar-store path), U a 2x nearest upsample to 1280x960. Rigs of 2 and 3 distinct sizes, one with the sizes
# interleaved:
RIGS = ["AC", "ACA", "AOU"]


@pytest.fixture(scope="module")
def rig():
    from moped_b200 import capi
    g = dict(np.load(os.path.join(ROOT, "tests", "golden", "real_images.npz")))
    im = np.load(os.path.join(ROOT, "tests", "golden", "sift_golden.npz"))["bag4_full_double/image"]
    full = np.stack([np.roll(im, s, axis=1) for s in range(-4, 4)])
    K = g["K"][0].astype(np.float32)
    fx, fy, cx, cy = (float(v) for v in K)
    raw = {"A": full, "C": np.ascontiguousarray(full[:, 48:432, 64:576]), "O": np.ascontiguousarray(full[:, :479, 1:638]),
           "U": np.ascontiguousarray(full.repeat(2, axis=1).repeat(2, axis=2))}
    Ks = {"A": K, "C": np.float32([fx, fy, cx - 64, cy - 48]), "O": np.float32([fx, fy, cx - 1, cy]),
          "U": np.float32([2 * fx, 2 * fy, 2 * cx + 0.5, 2 * cy + 0.5])}
    ctx = capi.Context(0)
    ctx.db_upload(g["db_desc"], g["db_xyz"], g["model_of_row"], len(g["n_pts"]))
    ctx.set_tuning(8, 8, 1)
    r = dict(ctx=ctx, g=g, im=im, raw=raw, Ks=Ks, und={})
    yield r
    ctx.close()


def _undistorted(r, kind, lens):
    key = (kind, lens)
    if key not in r["und"]:
        src = r["raw"][kind]
        r["und"][key] = U.remap_linear_u8(src, U.undistort_map(r["Ks"][kind], LENSES[lens], src.shape[1], src.shape[2]))
    return r["und"][key]


def _slots(B, Cn):
    return (3 * np.arange(B)[:, None] + 5 * np.arange(Cn)[None, :]) % 8


def _set_cameras(r, kinds):
    r["ctx"].set_cameras(np.stack([r["Ks"][k] for k in kinds]), POSES[:len(kinds)])


def _set_tables(r, kinds, tables):
    ctx = r["ctx"]
    for c in range(16):
        ctx.set_undistortion(c, None, None, 0, 0)
    for c in tables:
        H, W = r["raw"][kinds[c]].shape[1:]
        ctx.set_undistortion(c, r["Ks"][kinds[c]], LENSES[c], H, W)


def _images(r, kinds, slots):
    return [np.ascontiguousarray(r["raw"][k][slots[:, c]]) for c, k in enumerate(kinds)]


def _normalise(desc):
    ss = np.zeros(len(desc), np.float32)
    for k in range(128):
        ss = ss + desc[:, k] * desc[:, k]                                  # sequential fp32 sum like MATCH_CUDA::normalise
    return desc * (1.0 / np.sqrt(ss).astype(np.float64)).astype(np.float32)[:, None]


def _host_features(r, kinds, slots, tables, double_size):
    B, Cn = slots.shape
    per_cam = []
    for c, k in enumerate(kinds):
        src = _undistorted(r, k, c) if c in tables else r["raw"][k]
        per_cam.append(r["ctx"].sift(np.ascontiguousarray(src[slots[:, c]]), bool(double_size), MAX_KP))
    frames = []
    for f in range(B):
        xy = [per_cam[c][f][0] for c in range(Cn)]
        q = [_normalise(per_cam[c][f][2]) for c in range(Cn)]
        img = [np.full(len(x), c, np.int32) for c, x in enumerate(xy)]
        frames.append((np.concatenate(q), np.concatenate(xy), np.concatenate(img), np.array([len(x) for x in xy], np.int32)))
    return frames


def _host_route(r, kinds, slots, tables, double_size):
    """what a host does without the call: each camera undistorted (by the oracle) and extracted at its own size, each frame's
    keypoints concatenated in camera order with q_image = camera, MATCH's normalisation, mc_process_frames"""
    frames = _host_features(r, kinds, slots, tables, double_size)
    _set_tables(r, kinds, ())
    fo = np.concatenate([[0], np.cumsum([len(q) for q, _, _, _ in frames])]).astype(np.int32)
    l0 = r["ctx"].launches
    out = r["ctx"].process_frames(np.concatenate([q for q, _, _, _ in frames]), np.concatenate([xy for _, xy, _, _ in frames]),
                                  np.concatenate([im for _, _, im, _ in frames]), fo, max_objects=64)
    chain = r["ctx"].launches - l0
    for o, fr in zip(out, frames):
        o["n_features"] = fr[3]
    return out, frames, chain


def _rig_call(r, kinds, slots, tables, double_size):
    _set_tables(r, kinds, tables)
    l0 = r["ctx"].launches
    out = r["ctx"].process_rig_cameras(_images(r, kinds, slots), bool(double_size), max_keypoints=MAX_KP, max_objects=64)
    return out, r["ctx"].launches - l0


def _assert_same(a_list, b_list, what):
    assert len(a_list) == len(b_list)
    for f, (a, b) in enumerate(zip(a_list, b_list)):
        assert np.array_equal(np.asarray(a["n_features"]), np.asarray(b["n_features"])), (what, f, a["n_features"], b["n_features"])
        assert np.array_equal(a["info"], b["info"]), (what, f, a["info"], b["info"])
        assert np.array_equal(a["model"], b["model"]), (what, f, a["model"], b["model"])
        assert np.array_equal(a["pose"], b["pose"]), (what, f)
        assert np.array_equal(a["score"], b["score"]), (what, f)


@pytest.mark.parametrize("double_size", [0, 1])
@pytest.mark.parametrize("B", [1, 7])
@pytest.mark.parametrize("kinds", RIGS)
def test_mixed_rig_equals_host_assembled_route(rig, kinds, B, double_size):
    r = rig
    Cn = len(kinds)
    _set_cameras(r, kinds)
    slots = _slots(B, Cn)
    found = 0
    for tables in (tuple(range(Cn)), SOME[Cn], ()):
        out, _ = _rig_call(r, kinds, slots, tables, double_size)
        want, _, _ = _host_route(r, kinds, slots, tables, double_size)
        _assert_same(out, want, (kinds, B, double_size, tables))
        assert all(o["n_features"].shape == (Cn,) for o in out)
        assert all((o["n_features"] > 0).all() for o in out)
        found += sum(len(o["model"]) for o in out)
    if double_size:
        assert found > 0
    _set_tables(r, kinds, ())


def test_exact_order_mixed_rig_frames_equal_the_oracle_chain(rig):
    r = rig
    g, ctx = r["g"], r["ctx"]
    kinds, B, tables = "AOC", 3, (1,)
    Cn = len(kinds)
    _set_cameras(r, kinds)
    slots = _slots(B, Cn)
    ctx.set_option("pose_exact_order", 1)
    try:
        out, _ = _rig_call(r, kinds, slots, tables, 1)
    finally:
        ctx.set_option("pose_exact_order", 0)
        _set_tables(r, kinds, ())
    frames = _host_features(r, kinds, slots, tables, 1)
    Ks = np.stack([r["Ks"][k] for k in kinds])
    found = 0
    for f, (q, xy, img, nf) in enumerate(frames):
        assert np.array_equal(out[f]["n_features"], nf), f
        want = oracle_chain.frame(g["db_desc"], g["db_xyz"], g["model_of_row"], len(g["n_pts"]), q, xy, img, Ks, POSES[:Cn], n_images=Cn)
        assert np.array_equal(out[f]["model"], want["model"]), (f, out[f]["model"], want["model"])
        assert np.array_equal(out[f]["pose"], want["pose"]), f
        assert np.array_equal(out[f]["score"], want["score"]), f
        found += len(want["model"])
    assert found > 0


def test_permuting_cameras_permutes_only_what_it_implies(rig):
    """(A, C, A) and (C, A, A) with the cameras' images, intrinsics, poses and tables moved along: per-camera counts follow the
    cameras, and each rig equals its own host-assembled route"""
    r = rig
    B = 3
    base = _slots(B, 3)
    for kinds, perm in (("ACA", (0, 1, 2)), ("CAA", (1, 0, 2)), ("AAC", (0, 2, 1))):
        slots = base[:, perm]
        r["ctx"].set_cameras(np.stack([r["Ks"][k] for k in kinds]), POSES[list(perm)])
        tables = tuple(j for j, p in enumerate(perm) if p in SOME[3])
        _set_tables(r, kinds, ())
        for c in tables:
            H, W = r["raw"][kinds[c]].shape[1:]
            r["ctx"].set_undistortion(c, r["Ks"][kinds[c]], LENSES[perm[c]], H, W)
        out = r["ctx"].process_rig_cameras(_images(r, kinds, slots), True, max_keypoints=MAX_KP, max_objects=64)
        if perm == (0, 1, 2):
            ref = out
        for f in range(B):
            assert np.array_equal(out[f]["n_features"], ref[f]["n_features"][list(perm)]), (kinds, f)
        # the same rig through the host route (tables by the oracle, with each camera's own lens)
        per_cam = []
        for c, k in enumerate(kinds):
            src = _undistorted(r, k, perm[c]) if c in tables else r["raw"][k]
            per_cam.append(r["ctx"].sift(np.ascontiguousarray(src[slots[:, c]]), True, MAX_KP))
        q = np.concatenate([_normalise(per_cam[c][f][2]) for f in range(B) for c in range(3)])
        xy = np.concatenate([per_cam[c][f][0] for f in range(B) for c in range(3)])
        img = np.concatenate([np.full(len(per_cam[c][f][0]), c, np.int32) for f in range(B) for c in range(3)])
        fo = np.concatenate([[0], np.cumsum([sum(len(per_cam[c][f][0]) for c in range(3)) for f in range(B)])]).astype(np.int32)
        _set_tables(r, kinds, ())
        want = r["ctx"].process_frames(q, xy, img, fo, max_objects=64)
        for o, w in zip(out, want):
            w["n_features"] = o["n_features"]
        _assert_same(out, want, kinds)


def test_a_blank_camera_of_its_own_size_changes_nothing(rig):
    r = rig
    ctx = r["ctx"]
    _set_tables(r, "A", ())
    frames = np.stack([r["im"], r["raw"]["A"][1]])
    blank = np.zeros((2, 384, 512), np.uint8)
    ctx.set_cameras(r["Ks"]["A"][None], POSES[:1])
    alone = ctx.process_images(frames, True, max_keypoints=MAX_KP, max_objects=64)
    assert sum(len(o["model"]) for o in alone) > 0
    ctx.set_cameras(np.stack([r["Ks"]["A"], r["Ks"]["A"]]), np.stack([POSES[0], POSES[0]]))
    for pos in (0, 1):
        ims = [blank, frames] if pos == 1 else [frames, blank]
        out = ctx.process_rig_cameras(ims, True, max_keypoints=MAX_KP, max_objects=64)
        for a, o in zip(alone, out):
            assert o["n_features"][1 - pos] == 0 and o["n_features"][pos] == a["n_features"], (pos, o["n_features"])
            assert np.array_equal(o["info"], a["info"]), pos
            assert np.array_equal(o["model"], a["model"]) and np.array_equal(o["pose"], a["pose"]) and np.array_equal(o["score"], a["score"]), pos


def _single_buffer_cams(buf):
    """mc_rig_camera entries for one [B][C][H][W] buffer: camera c at base + c * H * W, frame_stride C * H * W"""
    from moped_b200 import capi
    B, Cn, H, W = buf.shape
    base = buf.ctypes.data
    return (capi.RigCamera * Cn)(*[capi.RigCamera(base + c * H * W, Cn * H * W, H, W) for c in range(Cn)])


def _raw_cameras(ctx, cams, n_frames, dev=False, max_kp=MAX_KP, n_cameras=None):
    """the C entry itself: status, n_features and the per-frame outputs, also on failure"""
    Cn = (len(cams) if cams is not None else 2) if n_cameras is None else n_cameras
    p = ctx.default_params()
    B = max(n_frames, 1)
    n = np.zeros(B, np.int32)
    om = np.zeros(B * 64, np.int32)
    op = np.zeros(B * 64 * 7, np.float32)
    os_ = np.zeros(B * 64, np.float32)
    nf = np.full(max(B * Cn, 1), -1, np.int32)       # (an error returns before anything is written)
    info = np.zeros((B, 4), np.int32)
    fn = ctx.L.mc_process_rig_cameras_dev if dev else ctx.L.mc_process_rig_cameras
    st = fn(ctx.h, C.cast(cams, C.c_void_p) if cams is not None else None, Cn, n_frames, 1, max_kp, C.byref(p), 64, n, om, op, os_,
            nf.ctypes.data, info.ctypes.data, None)
    out = [dict(model=om[f * 64:f * 64 + n[f]], pose=op.reshape(-1, 64, 7)[f, :n[f]], score=os_[f * 64:f * 64 + n[f]],
                n_features=nf[f * Cn:(f + 1) * Cn], info=info[f]) for f in range(B)]
    return st, nf, out


def _ok(res):
    assert res[0] == 0, res[0]
    return res[2]


@pytest.mark.parametrize("Cn", [1, 2, 3])
@pytest.mark.parametrize("table", [False, True])
def test_one_size_is_process_rig_images(rig, Cn, table):
    r = rig
    ctx = r["ctx"]
    kinds = "A" * Cn
    _set_cameras(r, kinds)
    _set_tables(r, kinds, SOME[Cn] if Cn > 1 and table else ((0,) if table else ()))
    slots = _slots(4, Cn)
    buf = np.ascontiguousarray(r["raw"]["A"][slots])                     # [B][C][H][W]

    def counted(fn):
        l0 = ctx.launches
        out = fn()
        return out, ctx.launches - l0

    calls = {
        "rig_images": lambda: ctx.process_rig_images(buf, True, max_keypoints=MAX_KP, max_objects=64),
        "cameras, one buffer": lambda: _ok(_raw_cameras(ctx, _single_buffer_cams(buf), len(buf))),
        "cameras, one buffer each": lambda: ctx.process_rig_cameras([buf[:, c] for c in range(Cn)], True, max_keypoints=MAX_KP, max_objects=64),
    }
    if Cn == 1:
        calls["images"] = lambda: ctx.process_images(buf[:, 0], True, max_keypoints=MAX_KP, max_objects=64)
    for fn in calls.values():                                            # first calls of this shape: plans, lanes and graphs
        fn()
    ref, n_ref = counted(calls["rig_images"])
    assert sum(len(o["model"]) for o in ref) > 0
    for what, fn in calls.items():
        out, n = counted(fn)
        assert n == n_ref, (what, n, n_ref)
        if what == "images":
            out = [dict(o, n_features=np.array([o["n_features"]])) for o in out]
        _assert_same(out, ref, what)
    _set_tables(r, kinds, ())


def test_device_entry_equals_host_entry(rig):
    import torch
    r = rig
    ctx = r["ctx"]
    kinds, B, tables = "AOUC", 3, (0, 1)
    ctx.set_cameras(np.stack([r["Ks"][k] for k in kinds]), np.concatenate([POSES, POSES[:1]]))
    _set_tables(r, kinds, tables)
    ims = _images(r, kinds, _slots(B, len(kinds)))
    sizes = [im.shape[1:] for im in ims]
    ctx.process_rig_cameras(ims, True, max_keypoints=MAX_KP, max_objects=64)
    l0 = ctx.launches
    want = ctx.process_rig_cameras(ims, True, max_keypoints=MAX_KP, max_objects=64)
    n_want = ctx.launches - l0
    assert sum(len(o["model"]) for o in want) > 0
    # one device buffer per camera
    dev = [torch.from_numpy(im).cuda() for im in ims]
    # strided views into one device buffer: frame f holds every camera's image, 64 bytes apart
    offs = np.cumsum([0] + [h * w + 64 for h, w in sizes])
    stride = int(offs[-1]) + 128
    one = torch.zeros((B, stride), dtype=torch.uint8, device="cuda")
    for c, im in enumerate(ims):
        one[:, offs[c]:offs[c] + im[0].size] = torch.from_numpy(im.reshape(B, -1)).cuda()
    torch.cuda.synchronize()                                             # (the context's stream does not wait for torch's)
    layouts = {"per camera": ([t.data_ptr() for t in dev], [h * w for h, w in sizes]),
               "one buffer": ([one.data_ptr() + int(o) for o in offs[:-1]], [stride] * len(ims))}
    for what, (ptrs, strides) in layouts.items():
        ctx.process_rig_cameras_dev(ptrs, strides, sizes, B, True, max_keypoints=MAX_KP, max_objects=64)
        l0 = ctx.launches
        out = ctx.process_rig_cameras_dev(ptrs, strides, sizes, B, True, max_keypoints=MAX_KP, max_objects=64)
        assert ctx.launches - l0 == n_want, (what, ctx.launches - l0, n_want)
        _assert_same(out, want, what)
    # the images are not modified
    assert all(np.array_equal(t.cpu().numpy(), im) for t, im in zip(dev, ims))
    _set_tables(r, kinds, ())


def _sift_launches(r, B, H, W):
    import torch
    ctx = r["ctx"]
    gray = torch.zeros(B * H * W, dtype=torch.uint8, device="cuda")
    xy = torch.empty(B * MAX_KP * 2, dtype=torch.float32, device="cuda")
    desc = torch.empty(B * MAX_KP * 128, dtype=torch.float32, device="cuda")
    counts = torch.empty(B, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    l0 = ctx.launches
    ctx.sift_dev(gray.data_ptr(), B, H, W, True, MAX_KP, xy.data_ptr(), None, desc.data_ptr(), counts.data_ptr())
    n = ctx.launches - l0
    torch.cuda.synchronize()
    return n


@pytest.mark.parametrize("kinds,tables", [("ACA", (1,)), ("AOU", (0, 2)), ("AOU", ())])
def test_launches_per_size_group(rig, kinds, tables):
    """one SIFT extraction per size group, one remap per group with a table, two merge kernels, then the chain; the launches
    before the chain do not depend on the number of frames"""
    r = rig
    _set_cameras(r, kinds)
    groups = {}
    for c, k in enumerate(kinds):
        groups.setdefault(k, []).append(c)
    counts = []
    for B in (1, 3):
        slots = _slots(B, len(kinds))
        _rig_call(r, kinds, slots, tables, 1)
        out, n = _rig_call(r, kinds, slots, tables, 1)
        _host_route(r, kinds, slots, tables, 1)
        want, _, chain = _host_route(r, kinds, slots, tables, 1)
        _assert_same(out, want, (kinds, B))
        sift = sum(_sift_launches(r, B * len(cs), *r["raw"][k].shape[1:]) for k, cs in groups.items())
        remaps = sum(1 for cs in groups.values() if any(c in tables for c in cs))
        assert n == sift + remaps + 2 + chain, (B, n, sift, remaps, chain)
        counts.append(n - chain)
    assert counts[0] == counts[1], counts
    _set_tables(r, kinds, ())


def test_errors_launch_nothing_and_keep_the_tables(rig):
    from moped_b200 import capi
    r = rig
    ctx = r["ctx"]
    kinds = "AC"
    _set_cameras(r, kinds)
    _set_tables(r, kinds, (0, 1))
    ims = _images(r, kinds, _slots(2, 2))

    def cams_of(arrays, over=None):
        """one mc_rig_camera per array; over = {(camera, field): value} spoils some fields"""
        cs = (capi.RigCamera * len(arrays))(*[capi.RigCamera(a.ctypes.data, a.shape[1] * a.shape[2], a.shape[1], a.shape[2]) for a in arrays])
        for (c, field), v in (over or {}).items():
            setattr(cs[c], field, v)
        return cs

    def check(what, cams, n_frames, want, dev=False, context=ctx, n_cameras=None):
        l0 = context.launches
        st, _, _ = _raw_cameras(context, cams, n_frames, dev=dev, n_cameras=n_cameras)
        assert st == want, (what, st, context.L.mc_last_error(context.h))
        assert context.launches == l0, what

    tiny = np.zeros((1, 8, 8), np.uint8)
    for dev in (False, True):
        check("0 cameras", cams_of(ims), 2, ARG, dev, n_cameras=0)
        check("17 cameras", cams_of([tiny] * 17), 1, ARG, dev)
        check("NULL cameras", None, 2, ARG, dev)
        check("a NULL image", cams_of(ims, {(1, "gray"): None}), 2, ARG, dev)
        check("height 7", cams_of(ims, {(1, "height"): 7}), 2, ARG, dev)
        check("width 32768", cams_of(ims, {(0, "width"): 32768}), 2, ARG, dev)
        check("frame_stride below H x W", cams_of(ims, {(1, "frame_stride"): 384 * 512 - 1}), 2, ARG, dev)
        check("0 frames", cams_of(ims), 0, ARG, dev)
        check("65536 images", cams_of([tiny] * 16), 4096, ARG, dev)
        check("7282 images of one size", cams_of([tiny, tiny]), 3641, ARG, dev)
        check("a table of another size", cams_of([ims[1], ims[0]]), 2, ARG, dev)
        check("3 cameras, 2 set", cams_of(ims + [ims[0]]), 2, STATE, dev)
    # SIFT's batch limit through mc_process_images: now returned before the upload and any launch
    big = np.zeros((7282, 8, 8), np.uint8)
    _set_tables(r, kinds, ())
    l0 = ctx.launches
    with pytest.raises(capi.MopedCudaError, match=r"\(-2\)"):
        ctx.process_images(big, True, max_keypoints=16)
    assert ctx.launches == l0
    _set_tables(r, kinds, (0, 1))
    # only camera 1's table has another size
    ctx.set_undistortion(1, r["Ks"]["C"], LENSES[1], 384, 510)
    check("camera 1's table of another size", cams_of(ims), 2, ARG)
    ctx.set_undistortion(1, r["Ks"]["C"], LENSES[1], 384, 512)
    for c, k in enumerate(kinds):                                       # the tables are still the ones set
        assert np.array_equal(ctx.undistort(ims[c], c), _undistorted(r, k, c)[_slots(2, 2)[:, c]]), c
    # no database, a database that is not 128-d
    other = capi.Context(0)
    try:
        other.set_cameras(np.stack([r["Ks"][k] for k in kinds]), POSES[:2])
        check("no database", cams_of(ims), 2, STATE, context=other)
        rng = np.random.default_rng(3)
        other.db_upload(rng.random((300, 64), np.float32), rng.random((300, 3), np.float32), np.zeros(300, np.int32), 1)
        check("a 64-d database", cams_of(ims), 2, STATE, context=other)
    finally:
        other.close()
    # the context is still usable: more keypoints than max_keypoints in an image is MC_ERR_CAPACITY with the numbers found
    _set_tables(r, kinds, ())
    full = ctx.process_rig_cameras(ims, True, max_keypoints=MAX_KP)
    counts = np.stack([o["n_features"] for o in full]).reshape(-1)
    blank = [ims[0], np.zeros_like(ims[1])]
    st, nf, _ = _raw_cameras(ctx, cams_of(blank), 2, max_kp=100)
    assert st == capi.MC_ERR_CAPACITY, st
    assert np.array_equal(nf, [counts[0], 0, counts[2], 0]), (nf, counts)
    with pytest.raises(capi.MopedCudaError, match="max_keypoints"):
        ctx.process_rig_cameras(ims, True, max_keypoints=100)
