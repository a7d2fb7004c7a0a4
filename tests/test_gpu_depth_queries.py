"""mc_process_depth_queries / _dev / _merged_dev (depth_frames.cu): moped3d from features to objects in one call — MATCH, the per-match
gather of DEPTHPROP's depth data (fused into the compaction) and CLUSTER..FILTER2.

Bar: BIT-EXACT against the hand-stitched composition mc_match_adaptive_frames_dev -> torch gather of the per-feature world point and
fill distance through match_feature -> mc_process_depth_frames_dev, frame by frame (objects, pose and score bits, frame_info). The sharded
entry is checked against the whole-database call with one context per shard on one GPU, as tests/test_gpu_depth_sharded.py does."""
import ctypes as C

import numpy as np
import pytest
import torch

from moped_b200 import capi, synth
from moped_b200.sharding import shard_objects

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900, method="thread")]

DEPTHS = capi.ADAPTIVE_DEPTHS
N_BIG = 39                      # models of 500 rows ...
N_MODELS = N_BIG + 1            # ... and one model of a single row, a shard of its own in the sharded tests
ARG, STATE, CAPACITY = -2, -3, -4


@pytest.fixture(scope="module")
def db39():
    return synth.make_db(N_BIG, 500, seed=51)


@pytest.fixture(scope="module")
def db(db39):
    rng = np.random.default_rng(52)
    return dict(n_pts=np.append(db39["n_pts"], 1).astype(np.int32), desc=np.concatenate([db39["desc"], synth.sift_like(rng, 1)]),
                xyz=np.concatenate([db39["xyz"], rng.uniform(-0.1, 0.1, (1, 3)).astype(np.float32)]),
                model_of_row=np.append(db39["model_of_row"], N_BIG).astype(np.int32))


@pytest.fixture(scope="module")
def batch(db39):
    b = synth.make_adaptive_frames(db39, 64, seed=53, empty=(1, 40), far=(2,))
    b["curves"] = np.concatenate([b["curves"], b["curves"][:1]])
    return b


def context(db, rows=None, row_base=0):
    c = capi.Context(0)
    r0, r1 = rows if rows else (0, len(db["desc"]))
    c.db_upload(db["desc"][r0:r1], db["xyz"][r0:r1], db["model_of_row"][r0:r1], N_MODELS, row_base=row_base)
    if rows:
        c.db_set_global_tables(db["xyz"], db["model_of_row"], N_MODELS)
    c.set_cameras(synth.K_DEPTH, synth.CAM_IDENTITY)
    return c


@pytest.fixture(scope="module")
def ranks(db):
    """N -> the contexts of the N ranks; N = 1 is the context holding the whole database"""
    out = {1: [context(db)]}
    for n in (2, 3):
        shards = shard_objects(db["n_pts"][:N_BIG], n - 1) + [(N_BIG, N_MODELS, len(db["desc"]) - 1, len(db["desc"]))]
        out[n] = [context(db, (r0, r1), r0) for _, _, r0, r1 in shards]
    yield out
    for cs in out.values():
        for c in cs:
            c.close()


def sub(b, n):
    q = int(b["frame_offsets"][n])
    out = dict(b)
    for k in ("desc", "xy", "image", "world", "fill"):
        out[k] = b[k][:q]
    out["frame_offsets"] = b["frame_offsets"][:n + 1]
    out["depth"], out["fill_distance"] = b["depth"][:n], b["fill_distance"][:n]
    return out


def split(n, world):
    per, extra = divmod(n, world)
    lo = [r * per + min(r, extra) for r in range(world + 1)]
    return [(lo[r], lo[r + 1]) for r in range(world)]


def to_dev(a, dtype=None):
    return torch.from_numpy(np.ascontiguousarray(a, dtype)).cuda()


def bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint32) if a.dtype == np.float32 else a


def device_batch(b):
    return dict(q=to_dev(b["desc"], np.float32), xy=to_dev(b["xy"], np.float32), img=to_dev(b["image"], np.int32), depth=to_dev(b["depth"]),
                fill=to_dev(b["fill_distance"]), world=to_dev(b["world"], np.float32), wfill=to_dev(b["fill"], np.float32))


def params(c, variant=0):
    p = c.default_depth_params()
    p.variant = variant
    return p


def composition(c, b, d, p=None, max_objects=64):
    """the three-step route: MATCH, the caller's own gather through match_feature, then the chain"""
    Q = len(b["desc"])
    H, W = b["depth"].shape[1:]
    n = max(Q, 1)
    o = dict(feat=torch.full((n,), -9, dtype=torch.int32, device="cuda"), img=torch.zeros(n, dtype=torch.int32, device="cuda"),
             xy=torch.zeros((n, 2), device="cuda"), xyz=torch.zeros((n, 3), device="cuda"))
    torch.cuda.synchronize()
    r = c.match_adaptive_frames_dev(d["q"].data_ptr(), d["xy"].data_ptr(), d["img"].data_ptr(), b["frame_offsets"], d["depth"].data_ptr(),
                                    d["fill"].data_ptr(), W, H, b["curves"], o["feat"].data_ptr(), o["img"].data_ptr(), o["xy"].data_ptr(),
                                    o["xyz"].data_ptr(), partial=True)
    feat = o["feat"].long().clamp(min=0)
    world, fill = d["world"][feat].contiguous(), d["wfill"][feat].contiguous()
    torch.cuda.synchronize()                                # (the context's stream does not wait for torch's)
    return c.process_depth_frames_dev(r["match_offsets"], N_MODELS, o["img"].data_ptr(), o["xy"].data_ptr(), o["xyz"].data_ptr(), world.data_ptr(),
                                      fill.data_ptr(), d["depth"].data_ptr(), d["fill"].data_ptr(), W, H, params=p, max_objects=max_objects)


def one_call(c, b, d, **kw):
    H, W = b["depth"].shape[1:]
    torch.cuda.synchronize()
    return c.process_depth_queries_dev(d["q"].data_ptr(), d["xy"].data_ptr(), d["img"].data_ptr(), d["world"].data_ptr(), d["wfill"].data_ptr(),
                                       b["frame_offsets"], d["depth"].data_ptr(), d["fill"].data_ptr(), W, H, b["curves"], **kw)


def run_merged(c, packed, n_shards, b, d, lo, hi, **kw):
    H, W = b["depth"].shape[1:]
    torch.cuda.synchronize()
    return c.process_depth_queries_merged_dev(packed.data_ptr(), n_shards, d["xy"].data_ptr(), d["img"].data_ptr(), d["world"].data_ptr(),
                                              d["wfill"].data_ptr(), b["frame_offsets"], lo, hi, d["depth"].data_ptr() + 4 * lo * H * W,
                                              d["fill"].data_ptr() + 4 * lo * H * W, W, H, b["curves"], **kw)


def same(a, b):
    return (np.array_equal(a["model"], b["model"]) and np.array_equal(bits(a["pose"]), bits(b["pose"]))
            and np.array_equal(bits(a["score"]), bits(b["score"])) and np.array_equal(a["info"], b["info"]))


def gather_blocks(ctxs, d, Q):
    own = []
    acc = torch.empty(max(Q, 1), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    for c in ctxs:
        blk = torch.empty(4 * Q, dtype=torch.int32, device="cuda")
        c.match_dev(d["q"].data_ptr(), Q, 1.0, capi.MATCH_TENSOR, blk.data_ptr(), blk.data_ptr() + 8 * Q, acc.data_ptr())
        c.synchronize()
        own.append(blk)
    return torch.stack(own)


@pytest.fixture(scope="module")
def batches(batch):
    return {n: (sub(batch, n), device_batch(sub(batch, n))) for n in (1, 7, 8, 16, 64)}


@pytest.fixture(scope="module")
def reference(ranks, batches):
    """the one-call result of the 64-frame batch with default parameters (the other tests compare against it)"""
    b, d = batches[64]
    return one_call(ranks[1][0], b, d)


@pytest.mark.parametrize("linkage_cached", [1, 0])
@pytest.mark.parametrize("variant", [0, 1])
@pytest.mark.parametrize("n_frames", [1, 7, 16, 64])
def test_every_frame_equals_the_composition(ranks, batches, n_frames, variant, linkage_cached):
    c = ranks[1][0]
    b, d = batches[n_frames]
    p = params(c, variant)
    c.set_option("linkage_cached", linkage_cached)
    try:
        ref = composition(c, b, d, p)
        got = one_call(c, b, d, params=p)
    finally:
        c.set_option("linkage_cached", 1)
    assert len(got) == len(ref) == n_frames
    for f in range(n_frames):
        assert same(got[f], ref[f]), (f, got[f]["info"], ref[f]["info"])
    info = np.stack([x["info"] for x in got])
    assert (info[:, 1] == 0).all()
    if n_frames >= 7:
        assert info[1].tolist() == [0, 0, 0, 0] and info[2].tolist() == [0, 0, 0, 0]     # empty frame, frame beyond the depth cut
        assert info[:, 2].sum() > 30 * n_frames and info[:, 3].sum() > 0                 # matches and clusters
    if n_frames >= 16 and variant == 0:
        assert info[:, 0].sum() > 0                                                       # objects


def test_host_entry_equals_the_device_entry(ranks, batches, reference):
    c = ranks[1][0]
    b, _ = batches[64]
    times = np.full(2, -1.0, np.float32)
    got = c.process_depth_queries(b["desc"], b["xy"], b["image"], b["world"], b["fill"], b["frame_offsets"], b["depth"], b["fill_distance"],
                                  b["curves"], times=times)
    for f in range(64):
        assert same(got[f], reference[f]), f
    assert (times > 0).all(), times
    # stage_ms leaves the frames on their lanes: same results with and without it
    b, d = batches[64]
    timed = one_call(c, b, d, times=times)
    assert all(same(timed[f], reference[f]) for f in range(64)) and (times > 0).all()


@pytest.mark.parametrize("N", [1, 2, 3])
def test_every_rank_range_equals_the_whole_database(ranks, batches, reference, N):
    for n in (7, 64):
        b, d = batches[n]
        ref = reference if n == 64 else one_call(ranks[1][0], b, d)
        packed = gather_blocks(ranks[N], d, len(b["desc"]))
        for rank, (lo, hi) in enumerate(split(n, N)):        # uneven ranges: 7 over 2 -> 4 / 3, over 3 -> 3 / 2 / 2
            got = run_merged(ranks[N][rank], packed, N, b, d, lo, hi)
            assert len(got) == hi - lo
            for f in range(lo, hi):
                assert same(got[f - lo], ref[f]), (N, n, f, got[f - lo]["info"], ref[f]["info"])
    assert run_merged(ranks[N][0], packed, N, b, d, 3, 3) == []


def test_launches_are_those_of_the_two_calls(ranks, batches):
    c = ranks[1][0]
    for n in (8, 64):
        b, d = batches[n]
        H, W = b["depth"].shape[1:]
        Q = len(b["desc"])
        o = [torch.zeros(Q * k, dtype=dt, device="cuda") for k, dt in ((1, torch.int32), (1, torch.int32), (2, torch.float32), (3, torch.float32))]
        torch.cuda.synchronize()
        l0 = c.launches
        r = c.match_adaptive_frames_dev(d["q"].data_ptr(), d["xy"].data_ptr(), d["img"].data_ptr(), b["frame_offsets"], d["depth"].data_ptr(),
                                        d["fill"].data_ptr(), W, H, b["curves"], *[t.data_ptr() for t in o])
        l1 = c.launches
        feat = o[0].long()
        world, fill = d["world"][feat].contiguous(), d["wfill"][feat].contiguous()
        torch.cuda.synchronize()
        l2 = c.launches
        c.process_depth_frames_dev(r["match_offsets"], N_MODELS, o[1].data_ptr(), o[2].data_ptr(), o[3].data_ptr(), world.data_ptr(), fill.data_ptr(),
                                   d["depth"].data_ptr(), d["fill"].data_ptr(), W, H)
        l3 = c.launches
        one_call(c, b, d)
        l4 = c.launches
        assert l1 > l0 and l3 > l2 and l4 - l3 == (l1 - l0) + (l3 - l2), (n, l1 - l0, l3 - l2, l4 - l3)


def crowded(b, db, rows_of_model, n_rows, xy=None, seed=54):
    """batch frames 0 and 3 around one frame of n_rows copies of a model's rows at plateau depth and fill distance 0 (all accepted)"""
    rng = np.random.default_rng(seed)
    rows = np.flatnonzero(db["model_of_row"] == rows_of_model)[rng.integers(0, 500, n_rows)]
    seg = b["segments"]["plateau"]
    H, W = b["depth"].shape[1:]
    fxy = rng.uniform([0, 0], [W - 1, H - 1], (n_rows, 2)).astype(np.float32) if xy is None else xy
    depth = np.full((H, W), np.float32(sum(seg) / 2))
    fo = b["frame_offsets"]
    n0, n3 = int(fo[1]), int(fo[4] - fo[3])
    world = np.concatenate([fxy, np.ones((n_rows, 1), np.float32)], 1) * np.float32(sum(seg) / 2)
    cat = lambda k, mid: np.concatenate([b[k][:n0], mid, b[k][fo[3]:fo[4]]])
    return dict(desc=cat("desc", db["desc"][rows]), xy=cat("xy", fxy), image=cat("image", np.zeros(n_rows, np.int32)), world=cat("world", world),
                fill=cat("fill", np.zeros(n_rows, np.float32)), frame_offsets=np.array([0, n0, n0 + n_rows, n0 + n_rows + n3], np.int32),
                depth=np.stack([b["depth"][0], depth, b["depth"][3]]), fill_distance=np.stack([b["fill_distance"][0], np.zeros((H, W), np.float32),
                                                                                                 b["fill_distance"][3]]), curves=b["curves"])


def raw_args(c, b, d, res, **over):
    H, W = b["depth"].shape[1:]
    a = dict(q=d["q"].data_ptr(), xy=d["xy"].data_ptr(), img=d["img"].data_ptr(), world=d["world"].data_ptr(), wfill=d["wfill"].data_ptr(),
             fo=np.ascontiguousarray(b["frame_offsets"], np.int32), nf=len(b["frame_offsets"]) - 1, depth=d["depth"].data_ptr(),
             fill=d["fill"].data_ptr(), W=W, H=H, models=b["curves"].ctypes.data, n_models=len(b["curves"]))
    a.update(over)
    return [c.h, a["q"], a["xy"], a["img"], a["world"], a["wfill"], a["fo"], a["nf"], a["depth"], a["fill"], a["W"], a["H"], a["models"],
            a["n_models"], *[C.c_float(v) for v in DEPTHS], C.byref(params(c)), 64, *res]


def test_errors_return_status_and_leave_the_other_frames_complete(db, ranks, batches, reference):
    c = ranks[1][0]
    b, d = batches[7]
    error = lambda: c.L.mc_last_error(c.h).decode()
    # a frame over MATCH's 8192 cap: status 3
    cb = crowded(b, db, 5, 9000)
    got, st = one_call(c, cb, device_batch(cb), partial=True)
    assert st == CAPACITY and "frame 1 " in error()
    assert got[1]["info"].tolist() == [0, 3, 0, 0] and len(got[1]["model"]) == 0
    assert same(got[0], reference[0]) and same(got[2], reference[3])

    # a model with more than 2048 matches: status 4 here, while the chain alone refuses the whole batch
    cb = crowded(b, db, 5, 3000)
    dc = device_batch(cb)
    got, st = one_call(c, cb, dc, partial=True)
    assert st == CAPACITY and "frame 1 " in error()
    assert got[1]["info"][1] == 4 and got[1]["info"][2] > 2048 and got[1]["info"][0] == 0
    assert same(got[0], reference[0]) and same(got[2], reference[3])
    with pytest.raises(capi.MopedCudaError):
        composition(c, cb, dc)

    # features outside the map (x == width, x < 0) that MATCH accepts through its clamped pixel: status 1, nothing read out of range
    H, W = b["depth"].shape[1:]
    xy = np.random.default_rng(55).uniform([0, 0], [W - 1, H - 1], (300, 2)).astype(np.float32)
    xy[:3, 0], xy[3:6, 0] = W, -3.0
    cb = crowded(b, db, 7, 300, xy=xy)
    got, st = one_call(c, cb, device_batch(cb), partial=True)
    assert st == ARG and "frame 1 " in error()
    assert got[1]["info"][1] == 1 and got[1]["info"][0] == 0 and got[1]["info"][2] == 300
    assert same(got[0], reference[0]) and same(got[2], reference[3])

    # more than max_objects objects: the true count in info[0], no objects, the other frames complete
    b64, d64 = batches[64]
    counts = np.array([x["info"][0] for x in reference])
    k = int(counts.max())
    assert k >= 2, counts
    got, st = one_call(c, b64, d64, max_objects=k - 1, partial=True)
    assert st == CAPACITY and f"frame {int(np.argmax(counts))} " in error()
    for f in range(64):
        if counts[f] > k - 1:
            assert got[f]["info"].tolist() == reference[f]["info"].tolist() and len(got[f]["model"]) == 0
        else:
            assert same(got[f], reference[f]), f

    # NULL per-feature depth data with features present; an all-empty batch needs none
    n_obj, om, op, os_, info = (np.zeros(7, np.int32), np.zeros(7 * 64, np.int32), np.zeros(7 * 64 * 7, np.float32), np.zeros(7 * 64, np.float32),
                                np.zeros(7 * 4, np.int32))
    res = [n_obj, om, op, os_, info, None]
    assert c.L.mc_process_depth_queries_dev(*raw_args(c, b, d, res, world=None)) == ARG
    assert c.L.mc_process_depth_queries_dev(*raw_args(c, b, d, res, wfill=None)) == ARG
    for want, over in ((ARG, dict(q=None)), (ARG, dict(depth=None)), (ARG, dict(nf=0)), (ARG, dict(W=0)), (ARG, dict(n_models=N_MODELS - 1)),
                       (ARG, dict(fo=np.array([0, 900, 400], np.int32), nf=2))):
        assert c.L.mc_process_depth_queries_dev(*raw_args(c, b, d, res, **over)) == want, over
    empty = np.zeros(8, np.int32)
    assert c.L.mc_process_depth_queries_dev(*raw_args(c, b, d, res, fo=empty, q=None, world=None, wfill=None)) == 0
    assert (n_obj == 0).all() and (info == 0).all()

    # a row outside the tables in one gathered block (merged entry): status 2
    packed = gather_blocks(ranks[2], d, len(b["desc"]))
    fo = b["frame_offsets"]
    packed[1, 2 * (int(fo[3]) + 17)] = len(db["desc"]) + 1000
    got, st = run_merged(ranks[2][1], packed, 2, b, d, 0, 7, partial=True)
    assert st == ARG and "frame 3 " in ranks[2][1].L.mc_last_error(ranks[2][1].h).decode()
    assert got[3]["info"].tolist() == [0, 2, 0, 0]
    for f in (0, 1, 2, 4, 5, 6):
        assert same(got[f], reference[f]), f

    # no database; an object-sharded database on the whole-database entries
    c0 = capi.Context(0)
    try:
        c0.set_cameras(synth.K_DEPTH, synth.CAM_IDENTITY)
        assert c0.L.mc_process_depth_queries_dev(*raw_args(c0, b, d, res)) == STATE
    finally:
        c0.close()
    shard = ranks[2][0]
    assert shard.L.mc_process_depth_queries_dev(*raw_args(shard, b, d, res)) == STATE
    with pytest.raises(capi.MopedCudaError):
        shard.process_depth_queries(b["desc"], b["xy"], b["image"], b["world"], b["fill"], fo, b["depth"], b["fill_distance"], b["curves"])

    # the contexts still give the reference afterwards
    got = one_call(c, b64, d64)
    assert all(same(got[f], reference[f]) for f in range(64))
    got = run_merged(ranks[2][1], gather_blocks(ranks[2], d, len(b["desc"])), 2, b, d, 0, 7)
    assert all(same(got[f], reference[f]) for f in range(7))
