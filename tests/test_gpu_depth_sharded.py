"""mc_match_adaptive_frames_merged_dev (adaptive.cu): moped3d's depth-adaptive MATCH step on an object-sharded database.

One GPU stands for N ranks: N contexts each hold an object shard (row_base) plus the global coord3D / model tables, each writes its
packed block [nn_row Q x 2 | nn_dist Q x 2] with mc_match_dev, and stacking the blocks in one tensor stands for the all-gather.
Bar: BIT-EXACT against mc_match_adaptive_frames_dev on one context holding the whole database, for every frame of every range."""
import ctypes as C

import numpy as np
import pytest
import torch

from moped_b200 import capi, synth
from moped_b200.sharding import shard_objects

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900, method="thread")]

DEPTHS = capi.ADAPTIVE_DEPTHS
N_BIG = 39                      # models of 500 rows ...
N_MODELS = N_BIG + 1            # ... and one model of a single row, which is a shard of its own (its blocks carry -1 second rows)
ARG, STATE, CAPACITY = -2, -3, -4


@pytest.fixture(scope="module")
def db39():
    return synth.make_db(N_BIG, 500, seed=41)


@pytest.fixture(scope="module")
def db(db39):
    rng = np.random.default_rng(42)
    return dict(n_pts=np.append(db39["n_pts"], 1).astype(np.int32), desc=np.concatenate([db39["desc"], synth.sift_like(rng, 1)]),
                xyz=np.concatenate([db39["xyz"], rng.uniform(-0.1, 0.1, (1, 3)).astype(np.float32)]),
                model_of_row=np.append(db39["model_of_row"], N_BIG).astype(np.int32))


@pytest.fixture(scope="module")
def batch(db39):
    # frames and curves from the 500-row models (a single row has no extent to derive a curve from); the one-row model takes model 0's
    b = synth.make_adaptive_frames(db39, 64, seed=43, empty=(1, 40), far=(2,))
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
    whole = context(db)
    out = {1: [whole]}
    for n in (2, 3, 8):
        shards = shard_objects(db["n_pts"][:N_BIG], n - 1) + [(N_BIG, N_MODELS, len(db["desc"]) - 1, len(db["desc"]))]
        out[n] = [context(db, (r0, r1), r0) for _, _, r0, r1 in shards]
    yield out
    for cs in out.values():
        for c in cs:
            c.close()


def sub(b, n):
    """the first n frames of a batch"""
    q = int(b["frame_offsets"][n])
    out = dict(b)
    for k in ("desc", "xy", "image", "world", "fill"):
        out[k] = b[k][:q]
    out["frame_offsets"] = b["frame_offsets"][:n + 1]
    out["depth"], out["fill_distance"] = b["depth"][:n], b["fill_distance"][:n]
    return out


def split(n, world):
    """contiguous, possibly uneven frame ranges of `world` ranks (7 over 3: 3 / 2 / 2)"""
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
                fill=to_dev(b["fill_distance"]))


def outputs(Q):
    """per-match and per-feature outputs, filled with values no call writes"""
    n = max(Q, 1)
    return dict(match_feature=torch.full((n,), -9, dtype=torch.int32, device="cuda"), match_image=torch.full((n,), -9, dtype=torch.int32, device="cuda"),
                match_xy=torch.full((n, 2), -9.0, device="cuda"), match_xyz=torch.full((n, 3), -9.0, device="cuda"),
                nn_row=torch.full((n, 2), -9, dtype=torch.int32, device="cuda"), nn_dist=torch.full((n, 2), -9.0, device="cuda"),
                accepted=torch.full((n,), 9, dtype=torch.uint8, device="cuda"))


def host(o):
    return {k: v.cpu().numpy() for k, v in o.items()}


def gather_blocks(ctxs, d, Q):
    """every rank writes its packed block with mc_match_dev; one stacked tensor stands for the all-gather"""
    own = []
    acc = torch.empty(max(Q, 1), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    for c in ctxs:
        blk = torch.empty(4 * Q, dtype=torch.int32, device="cuda")
        c.match_dev(d["q"].data_ptr(), Q, 1.0, capi.MATCH_TENSOR, blk.data_ptr(), blk.data_ptr() + 8 * Q, acc.data_ptr())
        c.synchronize()
        own.append(blk)
    return torch.stack(own)


def run_merged(c, packed, n_shards, b, d, lo, hi, o=None, **kw):
    Q = len(b["desc"])
    H, W = b["depth"].shape[1:]
    o = outputs(Q) if o is None else o
    torch.cuda.synchronize()
    r = c.match_adaptive_frames_merged_dev(packed.data_ptr(), n_shards, d["xy"].data_ptr(), d["img"].data_ptr(), b["frame_offsets"], lo, hi,
                                           d["depth"].data_ptr() + 4 * lo * H * W, d["fill"].data_ptr() + 4 * lo * H * W, W, H, b["curves"],
                                           o["match_feature"].data_ptr(), o["match_image"].data_ptr(), o["match_xy"].data_ptr(), o["match_xyz"].data_ptr(),
                                           o["nn_row"].data_ptr(), o["nn_dist"].data_ptr(), o["accepted"].data_ptr(), **kw)
    return r, o


def run_reference(whole, b, d, **kw):
    Q = len(b["desc"])
    H, W = b["depth"].shape[1:]
    o = outputs(Q)
    torch.cuda.synchronize()
    r = whole.match_adaptive_frames_dev(d["q"].data_ptr(), d["xy"].data_ptr(), d["img"].data_ptr(), b["frame_offsets"], d["depth"].data_ptr(),
                                        d["fill"].data_ptr(), W, H, b["curves"], o["match_feature"].data_ptr(), o["match_image"].data_ptr(),
                                        o["match_xy"].data_ptr(), o["match_xyz"].data_ptr(), o["nn_row"].data_ptr(), o["nn_dist"].data_ptr(),
                                        o["accepted"].data_ptr(), **kw)
    return r, o


def check_range(r, o, ref_r, ref_o, fo, lo, hi, frames=None):
    """frames `frames` (default: all) of the range [lo, hi) equal the reference; no slot outside the range's features was written"""
    for f in (range(lo, hi) if frames is None else frames):
        i = f - lo
        a, z = int(fo[f]), int(fo[f + 1])
        assert np.array_equal(r["match_offsets"][i], ref_r["match_offsets"][f]), f
        assert np.array_equal(r["frame_info"][i], ref_r["frame_info"][f]), (f, r["frame_info"][i], ref_r["frame_info"][f])
        for k in ("nn_row", "nn_dist", "accepted"):
            assert np.array_equal(bits(o[k][a:z]), bits(ref_o[k][a:z])), (f, k)
        n = int(ref_r["frame_info"][f][1])
        for k in ("match_feature", "match_image", "match_xy", "match_xyz"):
            assert np.array_equal(bits(o[k][a:a + n]), bits(ref_o[k][a:a + n])), (f, k)
    a, z, Q = int(fo[lo]), int(fo[hi]), int(fo[-1])
    for k, v in o.items():
        outside = np.concatenate([v[:a], v[z:Q]])
        assert (outside == (9 if k == "accepted" else -9)).all(), k


@pytest.fixture(scope="module")
def references(ranks, batch):
    out = {}
    for n in (1, 7, 8, 16, 64):
        b = sub(batch, n)
        d = device_batch(b)
        r, o = run_reference(ranks[1][0], b, d)
        assert r["status"] == 0
        out[n] = (b, d, r, host(o))
    return out


_blocks = {}


def blocks(ranks, references, N, n):
    if (N, n) not in _blocks:
        b, d, _, _ = references[n]
        _blocks[(N, n)] = gather_blocks(ranks[N], d, len(b["desc"]))
    return _blocks[(N, n)]


@pytest.mark.parametrize("n_frames", [1, 7, 64])
@pytest.mark.parametrize("N", [1, 2, 3, 8])
def test_every_range_equals_the_whole_database(ranks, references, N, n_frames):
    b, d, ref_r, ref_o = references[n_frames]
    fo = b["frame_offsets"]
    packed = blocks(ranks, references, N, n_frames)
    if N > 1:                                               # the one-row shard's blocks carry -1 as the second row of every feature
        assert (packed[-1].view(-1)[1:2 * len(b["desc"]):2] == -1).all()
    r, o = run_merged(ranks[N][0], packed, N, b, d, 0, n_frames)
    assert r["status"] == 0
    check_range(r, host(o), ref_r, ref_o, fo, 0, n_frames)
    for rank, (lo, hi) in enumerate(split(n_frames, N)):     # each rank its own frames, on its own context
        r, o = run_merged(ranks[N][rank], packed, N, b, d, lo, hi)
        assert r["status"] == 0 and len(r["match_offsets"]) == hi - lo
        check_range(r, host(o), ref_r, ref_o, fo, lo, hi)
    if n_frames >= 7:
        assert ref_r["frame_info"][1].tolist() == [0, 0, 0] and ref_r["frame_info"][2][0] > 0 and ref_r["frame_info"][2][1] == 0
    assert ref_r["frame_info"][:, 1].sum() > 30 * n_frames


def same_objects(a, b):
    return (np.array_equal(a["model"], b["model"]) and np.array_equal(bits(a["pose"]), bits(b["pose"]))
            and np.array_equal(bits(a["score"]), bits(b["score"])) and np.array_equal(a["info"], b["info"]))


def depth_chain(c, r, o, b, d, lo, hi):
    """DEPTHPROP's per-feature world point and fill distance gathered through match_feature, then CLUSTER..FILTER2 for frames [lo, hi)"""
    H, W = b["depth"].shape[1:]
    feat = o["match_feature"].long().clamp(min=0)
    world = to_dev(b["world"])[feat].contiguous()
    fill = to_dev(b["fill"])[feat].contiguous()
    depth, fill_distance = d["depth"][lo:hi].contiguous(), d["fill"][lo:hi].contiguous()
    torch.cuda.synchronize()                                # (the context's stream does not wait for torch's)
    return c.process_depth_frames_dev(r["match_offsets"], N_MODELS, o["match_image"].data_ptr(), o["match_xy"].data_ptr(), o["match_xyz"].data_ptr(),
                                      world.data_ptr(), fill.data_ptr(), depth.data_ptr(), fill_distance.data_ptr(), W, H)


@pytest.mark.parametrize("N", [2, 3])
def test_ranks_chain_to_the_objects_of_the_whole_database(ranks, references, N):
    b, d, _, _ = references[16]
    whole = ranks[1][0]
    ref_r, ref_o = run_reference(whole, b, d)
    ref = depth_chain(whole, ref_r, ref_o, b, d, 0, 16)
    packed = blocks(ranks, references, N, 16)
    got = []
    for rank, (lo, hi) in enumerate(split(16, N)):
        c = ranks[N][rank]
        r, o = run_merged(c, packed, N, b, d, lo, hi)
        assert r["status"] == 0
        got += depth_chain(c, r, o, b, d, lo, hi)
    assert len(got) == len(ref) == 16
    for f in range(16):
        assert same_objects(got[f], ref[f]), (f, got[f]["info"], ref[f]["info"])
    assert sum(int(x["info"][0]) for x in got) > 0 and sum(int(x["info"][3]) for x in got) > 0     # objects and clusters were formed


def test_launches_depend_neither_on_frames_nor_on_shards(ranks, references):
    counts = []
    for N, n in ((2, 8), (2, 64), (8, 8), (8, 64), (2, 8)):
        b, d, _, _ = references[n]
        packed = blocks(ranks, references, N, n)
        c = ranks[N][0]
        l0 = c.launches
        r, _ = run_merged(c, packed, N, b, d, 0, n)
        assert r["status"] == 0
        counts.append(c.launches - l0)
    assert len(set(counts)) == 1 and 0 < counts[0] <= 2, counts


def raw_args(c, b, d, gathered, o, offsets_out, **over):
    """the argument list of mc_match_adaptive_frames_merged_dev for batch b, some entries replaced"""
    H, W = b["depth"].shape[1:]
    a = dict(packed=gathered.data_ptr(), n_shards=gathered.shape[0], xy=d["xy"].data_ptr(), img=d["img"].data_ptr(),
             fo=np.ascontiguousarray(b["frame_offsets"], np.int32), nf=len(b["frame_offsets"]) - 1, lo=0, hi=len(b["frame_offsets"]) - 1,
             depth=d["depth"].data_ptr(), fill=d["fill"].data_ptr(), W=W, H=H, models=b["curves"].ctypes.data, n_models=len(b["curves"]),
             moff=offsets_out.reshape(-1), feat=o["match_feature"].data_ptr(), mimg=o["match_image"].data_ptr(), mxy=o["match_xy"].data_ptr(),
             mxyz=o["match_xyz"].data_ptr())
    a.update(over)
    return [c.h, a["packed"], a["n_shards"], a["xy"], a["img"], a["fo"], a["nf"], a["lo"], a["hi"], a["depth"], a["fill"], a["W"], a["H"],
            a["models"], a["n_models"], *[C.c_float(v) for v in DEPTHS], a["moff"], a["feat"], a["mimg"], a["mxy"], a["mxyz"], None, None,
            None, None]


def test_errors_return_status_and_leave_the_context_usable(db, ranks, references):
    b, d, ref_r, ref_o = references[7]
    fo = b["frame_offsets"]
    Q = len(b["desc"])
    c = ranks[2][1]
    packed = blocks(ranks, references, 2, 7)
    o = outputs(Q)
    moff = np.full((8, N_MODELS + 1), -5, np.int32)
    L = c.L
    torch.cuda.synchronize()
    cases = [(ARG, dict(packed=None)), (ARG, dict(n_shards=0)), (ARG, dict(xy=None)), (ARG, dict(feat=None)), (ARG, dict(mxyz=None)),
             (ARG, dict(depth=None)), (ARG, dict(fill=None)), (ARG, dict(models=None)),
             (ARG, dict(lo=-1)), (ARG, dict(hi=8)), (ARG, dict(lo=4, hi=3)), (ARG, dict(nf=0, hi=0)),
             (ARG, dict(fo=np.zeros(65537, np.int32), nf=65536, hi=3)), (ARG, dict(fo=np.array([5, 10], np.int32), nf=1, hi=1)),
             (ARG, dict(fo=np.array([0, 900, 400], np.int32), nf=2, hi=2)), (ARG, dict(W=0)), (ARG, dict(H=0)), (ARG, dict(n_models=N_MODELS - 1))]
    for want, over in cases:
        assert L.mc_match_adaptive_frames_merged_dev(*raw_args(c, b, d, packed, o, moff, **over)) == want, over
    # an empty range: MC_OK, nothing written
    assert L.mc_match_adaptive_frames_merged_dev(*raw_args(c, b, d, packed, o, moff, lo=3, hi=3)) == 0
    assert (moff == -5).all() and (host(o)["nn_row"] == -9).all() and (host(o)["match_feature"] == -9).all()
    # no tables
    c0 = capi.Context(0)
    try:
        assert c0.L.mc_match_adaptive_frames_merged_dev(*raw_args(c0, b, d, packed, o, moff)) == STATE
    finally:
        c0.close()

    # a frame with more than 8192 accepted matches: 9000 copies of one model's rows over measured plateau depth
    rng = np.random.default_rng(44)
    m = 5
    rows = np.flatnonzero(db["model_of_row"] == m)[rng.integers(0, 500, 9000)]
    seg = b["segments"]["plateau"]
    big = dict(desc=db["desc"][rows], xy=rng.uniform([0, 0], [639, 479], (9000, 2)).astype(np.float32), image=np.zeros(9000, np.int32),
               depth=np.full((480, 640), np.float32(sum(seg) / 2)), fill=np.zeros((480, 640), np.float32))
    n0, n3 = int(fo[1]), int(fo[4] - fo[3])
    cat = lambda k, kb: np.concatenate([b[k][:n0], big[kb], b[k][fo[3]:fo[4]]])
    cb = dict(desc=cat("desc", "desc"), xy=cat("xy", "xy"), image=cat("image", "image"), frame_offsets=np.array([0, n0, n0 + 9000, n0 + 9000 + n3], np.int32),
              depth=np.stack([b["depth"][0], big["depth"], b["depth"][3]]), fill_distance=np.stack([b["fill_distance"][0], big["fill"], b["fill_distance"][3]]),
              curves=b["curves"])
    dc = device_batch(cb)
    cref_r, cref_o = run_reference(ranks[1][0], cb, dc, partial=True)
    assert cref_r["status"] == CAPACITY and cref_r["frame_info"][1].tolist() == [9000, 0, 1]
    cpacked = gather_blocks(ranks[2], dc, len(cb["desc"]))
    with pytest.raises(capi.MopedCudaError):
        run_merged(c, cpacked, 2, cb, dc, 0, 3)
    for lo in (0, 1):
        r, o2 = run_merged(c, cpacked, 2, cb, dc, lo, 3, partial=True)
        assert r["status"] == CAPACITY and "frame 1 " in r["error"]
        assert r["frame_info"][1 - lo].tolist() == [9000, 0, 1] and (r["match_offsets"][1 - lo] == n0).all()
        h = host(o2)
        assert h["accepted"][n0:n0 + 9000].sum() > 8192
        check_range(r, h, cref_r, host(cref_o), cb["frame_offsets"], lo, 3)

    # a row id outside the tables in one gathered block: rejected before any table is read
    bad = packed.clone()
    i3, i5 = int(fo[3]) + 17, int(fo[5]) + 3
    bad[1, 2 * i3] = len(db["desc"]) + 1000                 # past the last global row
    bad[0, 2 * i5 + 1] = -2                                 # negative, but not the -1 of a missing neighbour
    r, o3 = run_merged(c, bad, 2, b, d, 0, 7, partial=True)
    assert r["status"] == ARG and "frame 3 " in r["error"], r
    h = host(o3)
    for f in (3, 5):
        assert r["frame_info"][f].tolist() == [int(fo[f + 1] - fo[f]), 0, 2] and (r["match_offsets"][f] == fo[f]).all()
    assert not h["accepted"][i3] and not h["accepted"][i5]
    check_range(r, h, ref_r, ref_o, fo, 0, 7, frames=[0, 1, 2, 4, 6])

    # the context still gives the reference afterwards
    r, o4 = run_merged(c, packed, 2, b, d, 0, 7)
    assert r["status"] == 0
    check_range(r, host(o4), ref_r, ref_o, fo, 0, 7)
