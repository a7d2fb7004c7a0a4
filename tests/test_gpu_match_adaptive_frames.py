"""mc_match_adaptive_frames / _dev (adaptive.cu): moped3d's depth-adaptive MATCH step for a batch of frames in one matching pass.

Bar: BIT-EXACT. One frame equals the numpy rule (tests/adaptive_rule.py, pinned to adaptive_threshold.cuh by
tests/test_match_adaptive_frames_host.py) applied to mc_match's nearest rows, and MATCH_ADAPTIVE_CUDA::emit restated in numpy; every frame
of a batch equals its own mc_match_adaptive call; the device entry equals the host entry; its output feeds mc_process_depth_frames_dev
and gives what mc_process_depth_frames gives on host-assembled lists."""
import ctypes as C

import numpy as np
import pytest
import torch

import adaptive_rule as R
from moped_b200 import capi, synth

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900, method="thread")]

DEPTHS = capi.ADAPTIVE_DEPTHS
N_MODELS = 40


@pytest.fixture(scope="module")
def db():
    return synth.make_db(N_MODELS, 500, seed=21)


@pytest.fixture(scope="module")
def ctx(db):
    c = capi.Context(0)
    c.db_upload(db["desc"], db["xyz"], db["model_of_row"], N_MODELS)
    c.set_cameras(synth.K_DEPTH, synth.CAM_IDENTITY)
    yield c
    c.close()


@pytest.fixture(scope="module")
def batch(db):
    return synth.make_adaptive_frames(db, 64, seed=22, empty=(1, 40), far=(2,))


def single(ctx, db, b, f):
    """frame f alone: mc_match_adaptive, then emit (match indices from the frame's first feature on)"""
    lo, hi = int(b["frame_offsets"][f]), int(b["frame_offsets"][f + 1])
    if hi == lo:
        nn_row, nn_dist, acc = np.zeros((0, 2), np.int32), np.zeros((0, 2), np.float32), np.zeros(0, bool)
    else:
        nn_row, nn_dist, acc = ctx.match_adaptive(b["desc"][lo:hi], b["xy"][lo:hi], b["depth"][f], b["fill_distance"][f], b["curves"])
    e = R.emit(nn_row, acc, b["xy"][lo:hi], b["image"][lo:hi], db["model_of_row"], db["xyz"], len(b["curves"]), base=lo)
    return dict(nn_row=nn_row, nn_dist=nn_dist, accepted=acc, emit=e)


@pytest.fixture(scope="module")
def singles(ctx, db, batch):
    return [single(ctx, db, batch, f) for f in range(len(batch["frame_offsets"]) - 1)]


def sub(b, n):
    """the first n frames of a batch"""
    q = int(b["frame_offsets"][n])
    out = dict(b)
    for k in ("desc", "xy", "image", "world", "fill"):
        out[k] = b[k][:q]
    out["frame_offsets"] = b["frame_offsets"][:n + 1]
    out["depth"], out["fill_distance"] = b["depth"][:n], b["fill_distance"][:n]
    return out


def run_host(ctx, b, **kw):
    return ctx.match_adaptive_frames(b["desc"], b["xy"], b["image"], b["frame_offsets"], b["depth"], b["fill_distance"], b["curves"], **kw)


def bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint32) if a.dtype == np.float32 else a


def check_frame(out, f, fo, ref, per_feature=True):
    lo, hi = int(fo[f]), int(fo[f + 1])
    e = ref["emit"]
    assert np.array_equal(out["match_offsets"][f], e["offsets"]), f
    n = int(e["offsets"][-1] - e["offsets"][0])
    assert out["frame_info"][f].tolist() == [hi - lo, n, 0], (f, out["frame_info"][f])
    s = slice(lo, lo + n)
    for k, kk in (("match_feature", "feature"), ("match_image", "image"), ("match_xy", "xy"), ("match_xyz", "xyz")):
        assert np.array_equal(bits(out[k][s]), bits(e[kk])), (f, k)
    if per_feature:
        assert np.array_equal(out["nn_row"][lo:hi], ref["nn_row"]), f
        assert np.array_equal(bits(out["nn_dist"][lo:hi]), bits(ref["nn_dist"])), f
        assert np.array_equal(out["accepted"][lo:hi], ref["accepted"]), f


def test_one_frame_equals_the_numpy_rule_on_mc_match_rows(ctx, db):
    b = synth.make_adaptive_frames(db, 1, n_features=2551, seed=23, empty=(), far=())
    W, H = b["depth"].shape[2], b["depth"].shape[1]
    b["xy"][:6] = [[W, 5], [W, H - 1], [W, H], [3, H], [W - 0.25, H - 0.25], [0, 0]]          # the reference's clamp quirk
    nn_row, nn_dist, _, _ = ctx.match(b["desc"], 1.0, capi.MATCH_TENSOR)
    acc = R.finalize(nn_row, nn_dist, b["xy"], b["depth"][0], b["fill_distance"][0], db["model_of_row"], b["curves"], DEPTHS)
    r_row, r_dist, r_acc = ctx.match_adaptive(b["desc"], b["xy"], b["depth"][0], b["fill_distance"][0], b["curves"])
    assert np.array_equal(r_row, nn_row) and np.array_equal(bits(r_dist), bits(nn_dist)) and np.array_equal(r_acc, acc)
    out = run_host(ctx, b)
    ref = dict(nn_row=nn_row, nn_dist=nn_dist, accepted=acc,
               emit=R.emit(nn_row, acc, b["xy"], b["image"], db["model_of_row"], db["xyz"], N_MODELS))
    check_frame(out, 0, b["frame_offsets"], ref)
    # accepts and rejects in every segment of the curves, only rejects beyond the depth cut
    px = R.pixel(b["xy"], W, H)
    seg = R.segment(b["curves"], db["model_of_row"][nn_row[:, 0]], b["depth"][0].reshape(-1)[px], DEPTHS[0])
    for s in range(4):
        assert acc[seg == s].any() and not acc[seg == s].all(), (R.SEGMENTS[s], np.bincount(seg, minlength=5))
    assert (seg == 4).sum() > 50 and not acc[seg == 4].any()


@pytest.mark.parametrize("n_frames", [1, 7, 64])
def test_every_frame_of_a_batch_equals_its_single_frame_call(ctx, batch, singles, n_frames):
    b = sub(batch, n_frames)
    out = run_host(ctx, b)
    assert out["status"] == 0
    fo = b["frame_offsets"]
    for f in range(n_frames):
        check_frame(out, f, fo, singles[f])
    if n_frames >= 7:
        assert out["frame_info"][1].tolist() == [0, 0, 0]                  # empty frame
        assert out["frame_info"][2][0] > 0 and out["frame_info"][2][1] == 0 and not out["accepted"][fo[2]:fo[3]].any()   # beyond the cut
    assert out["frame_info"][:, 1].sum() > 30 * n_frames


def to_dev(a, dtype=None):
    return torch.from_numpy(np.ascontiguousarray(a, dtype)).cuda()


def run_dev(ctx, b, **kw):
    Q = len(b["desc"])
    H, W = b["depth"].shape[1:]
    d = dict(q=to_dev(b["desc"], np.float32), xy=to_dev(b["xy"], np.float32), img=to_dev(b["image"], np.int32), depth=to_dev(b["depth"]),
             fill=to_dev(b["fill_distance"]))
    o = dict(match_feature=torch.zeros(Q, dtype=torch.int32, device="cuda"), match_image=torch.zeros(Q, dtype=torch.int32, device="cuda"),
             match_xy=torch.zeros((Q, 2), dtype=torch.float32, device="cuda"), match_xyz=torch.zeros((Q, 3), dtype=torch.float32, device="cuda"),
             nn_row=torch.zeros((Q, 2), dtype=torch.int32, device="cuda"), nn_dist=torch.zeros((Q, 2), dtype=torch.float32, device="cuda"),
             accepted=torch.zeros(Q, dtype=torch.uint8, device="cuda"))
    torch.cuda.synchronize()
    r = ctx.match_adaptive_frames_dev(d["q"].data_ptr(), d["xy"].data_ptr(), d["img"].data_ptr(), b["frame_offsets"], d["depth"].data_ptr(),
                                      d["fill"].data_ptr(), W, H, b["curves"], o["match_feature"].data_ptr(), o["match_image"].data_ptr(),
                                      o["match_xy"].data_ptr(), o["match_xyz"].data_ptr(), o["nn_row"].data_ptr(), o["nn_dist"].data_ptr(),
                                      o["accepted"].data_ptr(), **kw)
    return r, o, d


def test_device_entry_equals_the_host_entry(ctx, batch, singles):
    host = run_host(ctx, batch)
    r, o, _ = run_dev(ctx, batch)
    assert r["status"] == 0
    assert np.array_equal(r["match_offsets"], host["match_offsets"]) and np.array_equal(r["frame_info"], host["frame_info"])
    dev = {k: v.cpu().numpy() for k, v in o.items()}
    dev["accepted"] = dev["accepted"].astype(bool)
    dev.update(match_offsets=r["match_offsets"], frame_info=r["frame_info"])
    fo = batch["frame_offsets"]
    for f in range(len(fo) - 1):
        check_frame(dev, f, fo, singles[f])
    assert np.array_equal(dev["nn_row"], host["nn_row"]) and np.array_equal(dev["accepted"], host["accepted"])


def same_objects(a, b):
    return (np.array_equal(a["model"], b["model"]) and np.array_equal(bits(a["pose"]), bits(b["pose"]))
            and np.array_equal(bits(a["score"]), bits(b["score"])) and np.array_equal(a["info"], b["info"]))


def test_output_feeds_the_depth_frame_chain(ctx, batch, singles):
    """moped3d's MATCH -> (DEPTHPROP: per-feature world point and fill distance gathered through match_feature) -> CLUSTER..FILTER2:
    the gapped lists of the device entry against lists assembled on the host from single-frame calls, packed without gaps"""
    b = sub(batch, 16)
    fo = b["frame_offsets"]
    n_frames = len(fo) - 1
    H, W = b["depth"].shape[1:]
    r, o, d = run_dev(ctx, b)
    assert r["status"] == 0
    feat = o["match_feature"].long()
    world = to_dev(b["world"])[feat].contiguous()
    fill = to_dev(b["fill"])[feat].contiguous()
    torch.cuda.synchronize()                                                # (the context's stream does not wait for torch's)
    got = ctx.process_depth_frames_dev(r["match_offsets"], N_MODELS, o["match_image"].data_ptr(), o["match_xy"].data_ptr(), o["match_xyz"].data_ptr(),
                                       world.data_ptr(), fill.data_ptr(), d["depth"].data_ptr(), d["fill"].data_ptr(), W, H)
    rows, cat, base = [], {k: [] for k in ("feature", "image", "xy", "xyz")}, 0
    for f in range(n_frames):
        e = singles[f]["emit"]
        rows.append(e["offsets"] - e["offsets"][0] + base)
        base += int(e["offsets"][-1] - e["offsets"][0])
        for k in cat:
            cat[k].append(e[k])
    cat = {k: np.concatenate(v) for k, v in cat.items()}
    ref = ctx.process_depth_frames(np.stack(rows), N_MODELS, cat["image"], cat["xy"], cat["xyz"], b["world"][cat["feature"]], b["fill"][cat["feature"]],
                                   b["depth"], b["fill_distance"])
    for f in range(n_frames):
        assert same_objects(got[f], ref[f]), (f, got[f]["info"], ref[f]["info"])
    assert sum(int(x["info"][2]) for x in got) == base > 0
    assert sum(int(x["info"][3]) for x in got) > 0                          # clusters were formed


def test_launches_do_not_grow_with_the_batch(ctx, batch):
    counts = []
    for n in (8, 64, 8, 64):
        b = sub(batch, n)
        l0 = ctx.launches
        run_host(ctx, b)
        counts.append(ctx.launches - l0)
    assert counts[0] == counts[1] == counts[2] == counts[3] and 0 < counts[0] < 20, counts


def raw_args(ctx, b, out, **over):
    """the argument list of mc_match_adaptive_frames for batch b with outputs `out`, some replaced"""
    H, W = b["depth"].shape[1:]
    a = dict(q=b["desc"].ctypes.data, xy=b["xy"].ctypes.data, img=b["image"].ctypes.data, fo=np.ascontiguousarray(b["frame_offsets"], np.int32),
             nf=len(b["frame_offsets"]) - 1, depth=b["depth"].reshape(-1), fill=b["fill_distance"].reshape(-1), W=W, H=H,
             models=b["curves"].ctypes.data, n_models=len(b["curves"]), moff=out["moff"].reshape(-1), feat=out["feat"].ctypes.data,
             mimg=out["img"].ctypes.data, mxy=out["xy"].ctypes.data, mxyz=out["xyz"].ctypes.data)
    a.update(over)
    return [ctx.h, a["q"], a["xy"], a["img"], a["fo"], a["nf"], a["depth"], a["fill"], a["W"], a["H"], a["models"], a["n_models"],
            *[C.c_float(v) for v in DEPTHS], a["moff"], a["feat"], a["mimg"], a["mxy"], a["mxyz"], None, None, None, None]


def test_errors_return_status_and_leave_the_context_usable(ctx, db, batch, singles):
    b = sub(batch, 7)
    Q = len(b["desc"])
    out = dict(moff=np.zeros((8, N_MODELS + 1), np.int32), feat=np.zeros(Q, np.int32), img=np.zeros(Q, np.int32), xy=np.zeros((Q, 2), np.float32),
               xyz=np.zeros((Q, 3), np.float32))
    L = ctx.L
    ARG, STATE, CAPACITY = -2, -3, -4
    cases = [(ARG, dict(q=None)), (ARG, dict(feat=None)), (ARG, dict(models=None)), (ARG, dict(nf=0)), (ARG, dict(W=0)), (ARG, dict(H=0)),
             (ARG, dict(fo=np.array([5, 10], np.int32), nf=1)), (ARG, dict(fo=np.array([0, 900, 400], np.int32), nf=2)),
             (ARG, dict(n_models=N_MODELS - 1))]
    for want, over in cases:
        assert L.mc_match_adaptive_frames(*raw_args(ctx, b, out, **over)) == want, over
    # no database; object-sharded databases
    for setup in ("none", "row_base", "global_tables"):
        c2 = capi.Context(0)
        try:
            if setup == "row_base":
                c2.db_upload(db["desc"][:5000], db["xyz"][:5000], db["model_of_row"][:5000], N_MODELS, row_base=5000)
            elif setup == "global_tables":
                c2.db_upload(db["desc"][:5000], db["xyz"][:5000], db["model_of_row"][:5000], N_MODELS)
                c2.db_set_global_tables(db["xyz"], db["model_of_row"], N_MODELS)
            assert c2.L.mc_match_adaptive_frames(*raw_args(c2, b, out)) == STATE, setup
        finally:
            c2.close()
    # a frame with more than 8192 accepted matches: copies of database rows over measured plateau depth
    rng = np.random.default_rng(24)
    rows = rng.choice(len(db["desc"]), 9000, replace=False)
    seg = b["segments"]["plateau"]
    big = dict(desc=db["desc"][rows], xy=rng.uniform([0, 0], [639, 479], (9000, 2)).astype(np.float32), image=np.zeros(9000, np.int32),
               depth=np.full((480, 640), np.float32(sum(seg) / 2)), fill=np.zeros((480, 640), np.float32))
    fo0 = b["frame_offsets"]
    n0 = int(fo0[1])
    n3 = int(fo0[4] - fo0[3])
    cat = lambda k, kb: np.concatenate([b[k][:n0], big[kb], b[k][fo0[3]:fo0[4]]])
    cb = dict(desc=cat("desc", "desc"), xy=cat("xy", "xy"), image=cat("image", "image"), frame_offsets=np.array([0, n0, n0 + 9000, n0 + 9000 + n3], np.int32),
              depth=np.stack([b["depth"][0], big["depth"], b["depth"][3]]), fill_distance=np.stack([b["fill_distance"][0], big["fill"], b["fill_distance"][3]]),
              curves=b["curves"])
    with pytest.raises(capi.MopedCudaError):
        run_host(ctx, cb)
    r = run_host(ctx, cb, partial=True)
    assert r["status"] == CAPACITY and "frame 1 " in r["error"]
    assert r["frame_info"][1].tolist() == [9000, 0, 1] and (r["match_offsets"][1] == n0).all()
    assert r["accepted"][n0:n0 + 9000].sum() > 8192
    shift = dict(singles[3])
    shift["emit"] = dict(singles[3]["emit"])
    for k in ("offsets", "feature"):
        shift["emit"][k] = singles[3]["emit"][k] - fo0[3] + (n0 + 9000)
    check_frame(r, 0, cb["frame_offsets"], singles[0])
    check_frame(r, 2, cb["frame_offsets"], shift)
    rd, _, _ = run_dev(ctx, cb, partial=True)
    assert rd["status"] == CAPACITY and np.array_equal(rd["match_offsets"], r["match_offsets"]) and np.array_equal(rd["frame_info"], r["frame_info"])
    # the context still gives the reference afterwards
    ok = run_host(ctx, b)
    for f in range(7):
        check_frame(ok, f, b["frame_offsets"], singles[f])
