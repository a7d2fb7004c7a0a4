"""mc_extract_rig_cameras / _dev: the FEAT half of mc_process_rig_cameras with the frame-major query arrays left in the caller's device
buffers. Over the rig cases of test_gpu_rig_cameras.py: extraction followed by mc_process_frames_dev equals mc_process_rig_cameras* bit for
bit, the arrays equal the host-assembled route's, no database is needed, the launches are the rig call's minus the chain's, and every
error launches nothing."""
import ctypes as C

import numpy as np
import pytest
import torch

from test_gpu_rig_cameras import LENSES, MAX_KP, POSES, RIGS, SOME, _assert_same, _host_features, _images, _set_cameras, _set_tables, _slots, rig  # noqa: F401

pytestmark = pytest.mark.gpu
ARG, STATE, CAPACITY = -2, -3, -4


def _buffers(B, Cn, max_kp=MAX_KP):
    rows = B * Cn * max_kp
    return dict(desc=torch.full((rows, 128), float("nan"), device="cuda"), xy=torch.full((rows, 2), float("nan"), device="cuda"),
                image=torch.full((rows,), -9, dtype=torch.int32, device="cuda"))


def _extract(ctx, ims, double_size, dev, out):
    """-> (frame_offsets, n_features, launches); the images go in from the host or from one device buffer per camera"""
    B = len(ims[0])
    if dev:
        d = [torch.from_numpy(im).cuda() for im in ims]
    torch.cuda.synchronize()                                             # (the context's stream does not wait for torch's)
    l0 = ctx.launches
    ptrs = (out["desc"], out["xy"], out["image"])
    if dev:
        fo, nf, _ = ctx.extract_rig_cameras_dev([t.data_ptr() for t in d], [im.shape[1] * im.shape[2] for im in ims], [im.shape[1:] for im in ims],
                                                B, *ptrs, bool(double_size), MAX_KP)
    else:
        fo, nf, _ = ctx.extract_rig_cameras(ims, *ptrs, bool(double_size), MAX_KP)
    return fo, nf, ctx.launches - l0


def _full(ctx, ims, double_size, dev):
    if not dev:
        return ctx.process_rig_cameras(ims, bool(double_size), max_keypoints=MAX_KP, max_objects=64)
    d = [torch.from_numpy(im).cuda() for im in ims]
    torch.cuda.synchronize()
    return ctx.process_rig_cameras_dev([t.data_ptr() for t in d], [im.shape[1] * im.shape[2] for im in ims], [im.shape[1:] for im in ims], len(ims[0]),
                                       bool(double_size), max_keypoints=MAX_KP, max_objects=64)


@pytest.mark.parametrize("dev", [False, True])
@pytest.mark.parametrize("double_size", [0, 1])
@pytest.mark.parametrize("B", [1, 7])
@pytest.mark.parametrize("kinds", RIGS)
def test_extraction_then_frames_equals_the_rig_call(rig, kinds, B, double_size, dev):
    r = rig
    ctx = r["ctx"]
    Cn = len(kinds)
    _set_cameras(r, kinds)
    slots = _slots(B, Cn)
    ims = _images(r, kinds, slots)
    for tables in (tuple(range(Cn)), SOME[Cn], ()):
        _set_tables(r, kinds, tables)
        _full(ctx, ims, double_size, dev)                                # first calls of this shape: plans, lanes and graphs
        l0 = ctx.launches
        want = _full(ctx, ims, double_size, dev)
        n_full = ctx.launches - l0
        out = _buffers(B, Cn)
        _extract(ctx, ims, double_size, dev, out)
        fo, nf, n_ext = _extract(ctx, ims, double_size, dev, out)
        l0 = ctx.launches
        got = ctx.process_frames_dev(out["desc"].data_ptr(), out["xy"].data_ptr(), out["image"].data_ptr(), fo, max_objects=64)
        n_chain = ctx.launches - l0
        assert n_ext == n_full - n_chain, (kinds, tables, n_ext, n_full, n_chain)
        for f, o in enumerate(got):
            o["n_features"] = nf[f]
        _assert_same(got, want, (kinds, B, double_size, dev, tables))
        # the arrays are the host-assembled route's: per-camera extraction, concatenation in camera order, MATCH's normalisation
        frames = _host_features(r, kinds, slots, tables, double_size)
        Q = int(fo[-1])
        assert np.array_equal(fo, np.concatenate([[0], np.cumsum([len(q) for q, _, _, _ in frames])])), (fo, tables)
        assert np.array_equal(nf, np.stack([fr[3] for fr in frames]))
        assert np.array_equal(out["desc"][:Q].cpu().numpy(), np.concatenate([q for q, _, _, _ in frames]))
        assert np.array_equal(out["xy"][:Q].cpu().numpy(), np.concatenate([xy for _, xy, _, _ in frames]))
        assert np.array_equal(out["image"][:Q].cpu().numpy(), np.concatenate([im for _, _, im, _ in frames]))
    _set_tables(r, kinds, ())


def test_no_database_is_needed(rig):
    from moped_b200 import capi
    r = rig
    kinds, B = "AOU", 3
    _set_cameras(r, kinds)
    _set_tables(r, kinds, (0, 2))
    ims = _images(r, kinds, _slots(B, 3))
    with_db = _buffers(B, 3)
    fo_db, nf_db, _ = _extract(r["ctx"], ims, 1, False, with_db)
    bare = capi.Context(0)
    try:
        bare.set_cameras(np.stack([r["Ks"][k] for k in kinds]), POSES)
        for c in (0, 2):
            H, W = ims[c].shape[1:]
            bare.set_undistortion(c, r["Ks"][kinds[c]], LENSES[c], H, W)
        out = _buffers(B, 3)
        fo, nf, _ = _extract(bare, ims, 1, False, out)
    finally:
        bare.close()
    Q = int(fo[-1])
    assert Q > 0 and np.array_equal(fo, fo_db) and np.array_equal(nf, nf_db)
    for k in ("desc", "xy", "image"):
        assert torch.equal(out[k][:Q], with_db[k][:Q]), k
    _set_tables(r, kinds, ())


def _raw(ctx, cams, n_frames, out, dev=False, n_cameras=None, max_kp=MAX_KP, null=None, shift=None):
    Cn = (len(cams) if cams is not None else 2) if n_cameras is None else n_cameras
    fo = np.full(max(n_frames, 0) + 1, -1, np.int32)
    nf = np.full(max(n_frames * Cn, 1), -1, np.int32)
    ptrs = [out["desc"].data_ptr(), out["xy"].data_ptr(), out["image"].data_ptr()]
    if null is not None:
        ptrs[null] = None
    if shift is not None:                                               # (output k, bytes): a misaligned pointer
        ptrs[shift[0]] += shift[1]
    fn = ctx.L.mc_extract_rig_cameras_dev if dev else ctx.L.mc_extract_rig_cameras
    torch.cuda.synchronize()
    st = fn(ctx.h, C.cast(cams, C.c_void_p) if cams is not None else None, Cn, n_frames, 1, max_kp, *ptrs, fo, nf.ctypes.data, None)
    return st, fo, nf


def test_errors_launch_nothing(rig):
    from moped_b200 import capi
    r = rig
    ctx = r["ctx"]
    kinds = "AC"
    _set_cameras(r, kinds)
    _set_tables(r, kinds, (0, 1))
    ims = _images(r, kinds, _slots(2, 2))
    out = _buffers(2, 2)

    def cams_of(arrays, over=None):
        cs = (capi.RigCamera * len(arrays))(*[capi.RigCamera(a.ctypes.data, a.shape[1] * a.shape[2], a.shape[1], a.shape[2]) for a in arrays])
        for (c, field), v in (over or {}).items():
            setattr(cs[c], field, v)
        return cs

    def check(what, cams, n_frames, want, dev=False, **kw):
        l0 = ctx.launches
        st, fo, nf = _raw(ctx, cams, n_frames, out, dev=dev, **kw)
        assert st == want, (what, st, ctx.L.mc_last_error(ctx.h))
        assert ctx.launches == l0, what
        assert (fo == -1).all() and (nf == -1).all(), what                # nothing written either

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
        check("max_keypoints 0", cams_of(ims), 2, ARG, dev, max_kp=0)
        check("65536 images", cams_of([tiny] * 16), 4096, ARG, dev)
        check("7282 images of one size", cams_of([tiny, tiny]), 3641, ARG, dev)
        check("a table of another size", cams_of([ims[1], ims[0]]), 2, ARG, dev)
        check("3 cameras, 2 set", cams_of(ims + [ims[0]]), 2, STATE, dev)
        for k in range(3):
            check(f"NULL output {k}", cams_of(ims), 2, ARG, dev, null=k)
        for k, b in ((0, 4), (0, 8), (1, 4), (2, 2)):
            check(f"output {k} {b} bytes off its alignment", cams_of(ims), 2, ARG, dev, shift=(k, b))
    # the Python entry checks the output tensors before calling: dtype, device, contiguity, room for every row, alignment
    bad = {"a float64 desc": dict(out, desc=out["desc"].double()), "a host xy": dict(out, xy=out["xy"].cpu()),
           "an int64 image": dict(out, image=out["image"].long()), "a desc one row short": dict(out, desc=out["desc"][:-1]),
           "a strided xy": dict(out, xy=out["xy"][:, :1]), "a desc 4 bytes off": dict(out, desc=torch.zeros(out["desc"].numel() + 1, device="cuda")[1:])}
    for what, o in bad.items():
        l0 = ctx.launches
        with pytest.raises(ValueError):
            ctx.extract_rig_cameras(ims, o["desc"], o["xy"], o["image"], True, MAX_KP)
        assert ctx.launches == l0, what
    # more keypoints than max_keypoints in an image: MC_ERR_CAPACITY with the numbers found and the offsets
    _set_tables(r, kinds, ())
    st, fo, nf = _raw(ctx, cams_of(ims), 2, out)
    assert st == 0
    st, fo_small, nf_small = _raw(ctx, cams_of([ims[0], np.zeros_like(ims[1])]), 2, out, max_kp=100)
    assert st == CAPACITY, st
    assert np.array_equal(nf_small, [nf[0], 0, nf[2], 0]), (nf_small, nf)
    with pytest.raises(capi.MopedCudaError, match="max_keypoints"):
        ctx.extract_rig_cameras(ims, out["desc"], out["xy"], out["image"], True, 100)
