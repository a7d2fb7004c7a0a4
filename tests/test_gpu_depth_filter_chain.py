"""moped3d's FILTER_PROJECTION_DEPTH as FILTER / FILTER2 of the device chain (mc_set_depth_filter with mc_process_depth_frames* and
mc_process_depth_queries*).

Bar: BIT-EXACT. With the depth filter set on a step, every frame gives what the stage-by-stage calls give with mc_filter_projection_depth
on that step (objects in order, model ids, pose and score bits, frame_info), what the oracle chain built here from oracle_chain3d's steps
and oracle.filter_depth gives, and the same through every chain entry."""
import ctypes as C
import re

import numpy as np
import pytest
import torch

import oracle_chain3d
from moped_b200 import capi, synth
from moped_b200.sharding import shard_objects
from oracle import oracle

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900, method="thread")]

ARG = -2
ALL = 100000                    # TestSampleSize above every model's keypoint count: all keypoints are test points
# (PlausibleSqDistance, DepthFraction, MinKeypointFraction). On make_depth_frame frames STRONG's penalty prunes objects the plain filter
# keeps (checked against the oracle below); MILD lowers the scores and rarely changes a decision.
STRONG = (65536.0, 0.002, 0.2)
MILD = (16384.0, 0.02, 0.2)
SETTING = (STRONG, MILD)        # per step: FILTER, FILTER2
STEPS = {"filter": (0,), "filter2": (1,), "both": (0, 1)}


def dparams(d):
    return capi.DepthFilterParams.of(*d, synth.K_DEPTH, synth.CAM_IDENTITY)


def draw_test_points(model_offsets, model_xyz, sample):
    """one table per step, each drawn with its own seed (each FILTER_PROJECTION_DEPTH instance draws its own points)"""
    return {s: oracle.filter_depth_test_points(model_offsets, model_xyz, sample, 101 + s) for s in (0, 1)}


def depth_setting(steps, tables):
    """{step: (parameters, test_offsets, test_xyz)} for the steps that run the depth filter"""
    return {s: (SETTING[s],) + tables[s] for s in steps}


def apply(ctx, setting):
    for s in (0, 1):
        if s in setting:
            d, to, tx = setting[s]
            ctx.set_depth_filter(s, dparams(d), to, tx)
        else:
            ctx.set_depth_filter(s, None)


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    c.set_cameras(synth.K_DEPTH, synth.CAM_IDENTITY)
    yield c
    c.close()


@pytest.fixture
def clean(ctx):
    yield ctx
    apply(ctx, {})


def run_batch(ctx, frs, params=None, max_objects=64):
    b = synth.stack_depth_frames(frs)
    return ctx.process_depth_frames(b["match_offsets"], len(frs[0]["match_offsets"]) - 1, b["match_image"], b["match_xy"], b["match_xyz"],
                                    b["match_world"], b["match_fill"], b["depth"], b["fill_distance"], params=params, max_objects=max_objects)


def stage_by_stage(ctx, fr, P, setting):
    """The C-ABI stage calls the way the stage classes make them (host buffers, one call per step, per model for CLUSTER); a step in
    `setting` runs mc_filter_projection_depth with the frame's depth map, the others mc_filter_projection."""
    off = fr["match_offsets"]
    matches = dict(offsets=off, image=fr["match_image"], xy=fr["match_xy"], xyz=fr["match_xyz"])
    model, co, mem = [], [0], []
    for m in range(len(off) - 1):
        lo, hi = int(off[m]), int(off[m + 1])
        if hi == lo:
            continue
        o, mm = ctx.cluster_linkage(fr["match_xy"][lo:hi], fr["match_xyz"][lo:hi], fr["match_world"][lo:hi], fr["depth"], fr["fill_distance"],
                                    P.cluster_cutoff, P.cluster_min_pts, P.cluster_use_3d_filter, P.cluster_linkage_type, P.cluster_sigma_2d,
                                    P.cluster_sigma_3d)
        for c in range(len(o) - 1):
            model.append(m); mem.append(mm[o[c]:o[c + 1]]); co.append(co[-1] + int(o[c + 1] - o[c]))
    clusters = dict(model=np.array(model, np.int32), offsets=np.array(co, np.int32),
                    members=np.concatenate(mem).astype(np.int32) if mem else np.zeros(0, np.int32))
    cauchy = oracle.cauchy_weights(fr["match_fill"], P.variant)
    objects = []

    def pose(cl, pp, alpha):
        if len(cl["model"]) == 0:
            return
        j = np.concatenate([int(off[m]) + cl["members"][cl["offsets"][k]:cl["offsets"][k + 1]] for k, m in enumerate(cl["model"])])
        tie = np.concatenate([cl["members"][cl["offsets"][k]:cl["offsets"][k + 1]] for k in range(len(cl["model"]))])
        found, p, _ = ctx.pose_depth_ransac(P.variant, cl["offsets"], fr["match_xy"][j], fr["match_xyz"][j], fr["match_world"][j], cauchy[j],
                                            fr["match_image"][j], pp, alpha, pt_tie=tie)
        for t in range(len(found)):
            if found[t]:
                objects.append((int(cl["model"][t // pp.max_objects_per_cluster]), p[t].copy()))

    def filt(step, mp, fd, ms):
        nonlocal objects
        if not objects:
            return dict(model=np.zeros(0, np.int32), offsets=np.zeros(1, np.int32), members=np.zeros(0, np.int32)), np.zeros(0, np.float32)
        om, op = np.array([o[0] for o in objects], np.int32), np.stack([o[1] for o in objects])
        if step in setting:
            d, to, tx = setting[step]
            f = ctx.filter_depth(matches, om, op, (mp, fd, d[0], ms, d[1], d[2]), to, tx, synth.K_DEPTH, synth.CAM_IDENTITY, fr["depth"],
                                 fr["fill_distance"])
        else:
            f = ctx.filter(matches, om, op, (mp, fd, ms))
        keep = f["keep"]
        order = sorted((int(om[i]), i) for i in range(len(objects)) if keep[i])
        objects = [objects[i] for i in range(len(objects)) if keep[i]]
        return dict(model=np.array([m for m, _ in order], np.int32), offsets=f["offsets"], members=f["members"]), f["score"][keep]

    pose(clusters, P.pose, P.pose_alpha)
    cl2, _ = filt(0, P.filter_min_points, P.filter_feature_distance, P.filter_min_score)
    pose(cl2, P.pose2, P.pose2_alpha)
    _, score = filt(1, P.filter2_min_points, P.filter2_feature_distance, P.filter2_min_score)
    return dict(model=np.array([o[0] for o in objects], np.int32),
                pose=np.stack([o[1] for o in objects]).astype(np.float32) if objects else np.zeros((0, 7), np.float32),
                score=np.asarray(score, np.float32), n_clusters=len(model))


def oracle_frame(fr, variant, setting):
    """The oracle chain of oracle_chain3d.frame with oracle.filter_depth on the steps in `setting`; clusters rebuilt model-major in list
    order as oracle_chain.filter_step does. Also returns how many keep decisions the penalty changed against the plain filter."""
    cams = oracle.cameras(fr["K"], fr["cam_pose"])
    dcam = oracle.cameras(synth.K_DEPTH, synth.CAM_IDENTITY)
    matches = dict(offsets=fr["match_offsets"], image=fr["match_image"], xy=fr["match_xy"], xyz=fr["match_xyz"])
    flips = 0

    def filt(step, objects, fp):
        nonlocal flips
        if not objects:
            return [], dict(model=np.zeros(0, np.int32), offsets=np.zeros(1, np.int32), members=np.zeros(0, np.int32)), np.zeros(0, np.float32)
        om, op = np.array([o[0] for o in objects], np.int32), np.stack([o[1] for o in objects]).astype(np.float32)
        f = plain = oracle.filter_objects(matches, cams, om, op, fp)
        if step in setting:
            d, to, tx = setting[step]
            f = oracle.filter_depth(matches, cams, om, op, (fp[0], fp[1], d[0], fp[2], d[1], d[2]), to, tx, dcam, fr["depth"], fr["fill_distance"])
            flips += int((f["keep"] != plain["keep"]).sum())
        keep = f["keep"]
        order = sorted((int(om[i]), i) for i in range(len(objects)) if keep[i])
        cl = dict(model=np.array([m for m, _ in order], np.int32), offsets=f["offsets"], members=f["members"])
        return [objects[i] for i in range(len(objects)) if keep[i]], cl, f["score"][keep]

    cl = oracle_chain3d.cluster_step(fr)
    objects = []
    oracle_chain3d.pose_step(fr, cl, cams, oracle_chain3d.POSE1, oracle_chain3d.ALPHA, 1, objects, variant)
    objects, cl2, _ = filt(0, objects, oracle_chain3d.FILTER1)
    oracle_chain3d.pose_step(fr, cl2, cams, oracle_chain3d.POSE2, oracle_chain3d.ALPHA, 2, objects, variant)
    objects, _, score = filt(1, objects, oracle_chain3d.FILTER2)
    return dict(model=np.array([o[0] for o in objects], np.int32),
                pose=np.stack([o[1] for o in objects]).astype(np.float32) if objects else np.zeros((0, 7), np.float32),
                score=np.asarray(score, np.float32)), flips


def bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint32) if a.dtype == np.float32 else a


def same_objects(a, b):
    return (np.array_equal(a["model"], b["model"]) and np.array_equal(bits(a["pose"]), bits(b["pose"]))
            and np.array_equal(bits(a["score"]), bits(b["score"])))


def same(a, b):
    return same_objects(a, b) and np.array_equal(a["info"], b["info"])


@pytest.fixture(scope="module")
def frames64():
    return [synth.make_depth_frame(s) for s in range(300, 364)]


@pytest.fixture(scope="module")
def tables(frames64):
    fr = frames64[0]
    return {n: draw_test_points(fr["model_offsets"], fr["model_xyz"], n) for n in (40, ALL)}


@pytest.fixture(scope="module")
def plain64(ctx, frames64):
    """the plain chain on the 64-frame batch (no depth filter set on the context yet)"""
    return run_batch(ctx, frames64)


_refs = {}


@pytest.mark.parametrize("steps", list(STEPS))
@pytest.mark.parametrize("cached", [1, 0])
@pytest.mark.parametrize("variant", [0, 1])
def test_equals_the_stage_by_stage_calls(clean, frames64, tables, plain64, variant, cached, steps):
    ctx = clean
    P = ctx.default_depth_params()
    P.variant = variant
    for sample in (40, ALL):
        setting = depth_setting(STEPS[steps], tables[sample])
        key = (variant, steps, sample)
        if key not in _refs:                              # the stage calls do not depend on linkage_cached: computed once
            apply(ctx, {})
            _refs[key] = [stage_by_stage(ctx, fr, P, setting) for fr in frames64]
        refs = _refs[key]
        apply(ctx, setting)
        ctx.set_option("linkage_cached", cached)
        try:
            for n in (1, 7, 64):
                outs = run_batch(ctx, frames64[:n], P)
                for f in range(n):
                    o, r = outs[f], refs[f]
                    assert o["info"].tolist() == [len(r["model"]), 0, int(frames64[f]["match_offsets"][-1]), r["n_clusters"]], (n, f, o["info"])
                    assert same_objects(o, r), (sample, n, f, o["model"], r["model"])
        finally:
            ctx.set_option("linkage_cached", 1)
        assert sum(len(r["model"]) for r in refs) > 20
        if variant == 0:                                   # the setting took effect: scores (and objects) differ from the plain chain
            assert any(not same_objects(o, p) for o, p in zip(outs, plain64))


@pytest.mark.parametrize("variant", [0, 1])
def test_equals_the_oracle_chain(clean, frames64, tables, variant):
    ctx = clean
    P = ctx.default_depth_params()
    P.variant = variant
    setting = {0: (STRONG,) + tables[40][0], 1: (MILD,) + tables[ALL][1]}
    apply(ctx, setting)
    frs = frames64[:6]
    outs = run_batch(ctx, frs, P)
    flips = 0
    for f, fr in enumerate(frs):
        want, n = oracle_frame(fr, variant, setting)
        flips += n
        assert same_objects(outs[f], want), (f, outs[f]["model"], want["model"], outs[f]["score"], want["score"])
    assert flips > 0, "the penalty changed no keep decision: these frames do not exercise it"


def test_empty_tables_and_cleared_steps_give_the_plain_chain(clean, frames64, tables, plain64):
    ctx = clean
    n_models = len(frames64[0]["match_offsets"]) - 1
    empty = np.zeros(n_models + 1, np.int32)
    for s in (0, 1):
        ctx.set_depth_filter(s, dparams(STRONG), empty, None)           # no test point: penalty 0
    outs = run_batch(ctx, frames64)
    assert all(same(o, p) for o, p in zip(outs, plain64))
    apply(ctx, depth_setting((0, 1), tables[ALL]))
    outs = run_batch(ctx, frames64)
    assert any(not same(o, p) for o, p in zip(outs, plain64))
    apply(ctx, {})                                                      # both steps cleared on a used context
    outs = run_batch(ctx, frames64)
    assert all(same(o, p) for o, p in zip(outs, plain64))


def test_launches(clean, frames64, tables):
    """depth-filtering both steps adds at most two launches per frame (the penalty kernel), whatever the number of test points"""
    ctx = clean

    def count(frs):
        run_batch(ctx, frs)                                              # warm: buffers reserved
        l0 = ctx.launches
        run_batch(ctx, frs)
        return ctx.launches - l0

    for n in (8, 64):
        frs = frames64[:n]
        apply(ctx, {})
        plain = count(frs)
        extra = []
        for sample in (40, ALL):
            apply(ctx, depth_setting((0, 1), tables[sample]))
            extra.append(count(frs) - plain)
        assert extra[0] == extra[1] and 0 < extra[0] <= 2 * n, (n, plain, extra)


def expect(status, fn):
    with pytest.raises(capi.MopedCudaError) as e:
        fn()
    assert re.search(r"failed \(%d\)" % status, str(e.value)), str(e.value)
    return str(e.value)


def test_errors_leave_the_setting_and_the_context_usable(clean, frames64, tables):
    ctx = clean
    frs = frames64[:8]
    setting = depth_setting((0, 1), tables[40])
    apply(ctx, setting)
    want = run_batch(ctx, frs)
    n_models = len(frs[0]["match_offsets"]) - 1
    to, tx = tables[40][0]
    p = dparams(STRONG)

    def raw(c, step, params, offs, xyz, n):
        return ctx.L.mc_set_depth_filter(c, step, C.byref(params) if params is not None else None, offs.ctypes.data if offs is not None else None,
                                         xyz.ctypes.data if xyz is not None else None, n)

    desc = to.copy(); desc[3] = desc[4] + 1
    late = to + 1
    bad = [(None, 0, p, to, tx, n_models), (ctx.h, 2, p, to, tx, n_models), (ctx.h, -1, p, to, tx, n_models), (ctx.h, 0, p, to, tx, 0),
           (ctx.h, 1, p, to, tx, -3), (ctx.h, 0, p, None, tx, n_models), (ctx.h, 0, p, late, tx, n_models), (ctx.h, 1, p, desc, tx, n_models),
           (ctx.h, 0, p, to, None, n_models)]
    for args in bad:
        assert raw(*args) == ARG, args[1:]
        got = run_batch(ctx, frs)                                        # the previous setting is still in place
        assert all(same(g, w) for g, w in zip(got, want)), args[1:]
    # a table for another number of models: refused by the chain before any launch
    for s in (0, 1):
        t11 = oracle.filter_depth_test_points(frs[0]["model_offsets"][:12], frs[0]["model_xyz"], 40, 5)
        ctx.set_depth_filter(s, dparams(SETTING[s]), *t11)
        l0 = ctx.launches
        msg = expect(ARG, lambda: run_batch(ctx, frs))
        assert "11 models" in msg and ctx.launches == l0, msg
        apply(ctx, setting)
        got = run_batch(ctx, frs)
        assert all(same(g, w) for g, w in zip(got, want)), s


# ---- the features-in entries (mc_process_depth_queries*) on an adaptive-MATCH batch ------------------------------------------------------
N_BIG = 39
N_MODELS = N_BIG + 1


@pytest.fixture(scope="module")
def qdb():
    db39 = synth.make_db(N_BIG, 500, seed=51)
    rng = np.random.default_rng(52)
    db = dict(n_pts=np.append(db39["n_pts"], 1).astype(np.int32), desc=np.concatenate([db39["desc"], synth.sift_like(rng, 1)]),
              xyz=np.concatenate([db39["xyz"], rng.uniform(-0.1, 0.1, (1, 3)).astype(np.float32)]),
              model_of_row=np.append(db39["model_of_row"], N_BIG).astype(np.int32))
    b = synth.make_adaptive_frames(db39, 64, seed=53, empty=(1, 40), far=(2,))
    b["curves"] = np.concatenate([b["curves"], b["curves"][:1]])
    return db, b


def qcontext(db, rows=None):
    c = capi.Context(0)
    r0, r1 = rows if rows else (0, len(db["desc"]))
    c.db_upload(db["desc"][r0:r1], db["xyz"][r0:r1], db["model_of_row"][r0:r1], N_MODELS, row_base=r0)
    if rows:
        c.db_set_global_tables(db["xyz"], db["model_of_row"], N_MODELS)
    c.set_cameras(synth.K_DEPTH, synth.CAM_IDENTITY)
    return c


@pytest.fixture(scope="module")
def ranks(qdb):
    db, _ = qdb
    out = {1: [qcontext(db)]}
    for n in (2, 3):
        shards = shard_objects(db["n_pts"][:N_BIG], n - 1) + [(N_BIG, N_MODELS, len(db["desc"]) - 1, len(db["desc"]))]
        out[n] = [qcontext(db, (r0, r1)) for _, _, r0, r1 in shards]
    yield out
    for cs in out.values():
        for c in cs:
            c.close()


def to_dev(a, dtype=None):
    return torch.from_numpy(np.ascontiguousarray(a, dtype)).cuda()


def sub(b, n):
    q = int(b["frame_offsets"][n])
    out = dict(b)
    for k in ("desc", "xy", "image", "world", "fill"):
        out[k] = b[k][:q]
    out["frame_offsets"] = b["frame_offsets"][:n + 1]
    out["depth"], out["fill_distance"] = b["depth"][:n], b["fill_distance"][:n]
    return out


def device_batch(b):
    return dict(q=to_dev(b["desc"], np.float32), xy=to_dev(b["xy"], np.float32), img=to_dev(b["image"], np.int32), depth=to_dev(b["depth"]),
                fill=to_dev(b["fill_distance"]), world=to_dev(b["world"], np.float32), wfill=to_dev(b["fill"], np.float32))


def composition(c, b, d):
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
    torch.cuda.synchronize()
    return c.process_depth_frames_dev(r["match_offsets"], N_MODELS, o["img"].data_ptr(), o["xy"].data_ptr(), o["xyz"].data_ptr(), world.data_ptr(),
                                      fill.data_ptr(), d["depth"].data_ptr(), d["fill"].data_ptr(), W, H)


def one_call(c, b, d):
    H, W = b["depth"].shape[1:]
    torch.cuda.synchronize()
    return c.process_depth_queries_dev(d["q"].data_ptr(), d["xy"].data_ptr(), d["img"].data_ptr(), d["world"].data_ptr(), d["wfill"].data_ptr(),
                                       b["frame_offsets"], d["depth"].data_ptr(), d["fill"].data_ptr(), W, H, b["curves"])


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


def test_every_entry_agrees(qdb, ranks):
    db, batch = qdb
    offs = np.concatenate([[0], np.cumsum(db["n_pts"])]).astype(np.int32)
    setting = {0: (STRONG,) + oracle.filter_depth_test_points(offs, db["xyz"], 40, 7),
               1: (MILD,) + oracle.filter_depth_test_points(offs, db["xyz"], ALL, 8)}
    c = ranks[1][0]
    try:
        for n in (7, 64):
            b = sub(batch, n)
            d = device_batch(b)
            plain = one_call(c, b, d)
            for cs in ranks.values():                                   # every rank holds the whole table
                for r in cs:
                    apply(r, setting)
            got = one_call(c, b, d)
            ref = composition(c, b, d)
            assert all(same(g, r) for g, r in zip(got, ref))
            if n == 64:
                assert any(not same(g, p) for g, p in zip(got, plain))
                host = c.process_depth_queries(b["desc"], b["xy"], b["image"], b["world"], b["fill"], b["frame_offsets"], b["depth"],
                                               b["fill_distance"], b["curves"])
                assert all(same(h, g) for h, g in zip(host, got))
            H, W = b["depth"].shape[1:]
            for N in (1, 2, 3):
                packed = gather_blocks(ranks[N], d, len(b["desc"]))
                per, extra = divmod(n, N)
                lo = [r * per + min(r, extra) for r in range(N + 1)]
                for rank in range(N):
                    torch.cuda.synchronize()
                    part = ranks[N][rank].process_depth_queries_merged_dev(
                        packed.data_ptr(), N, d["xy"].data_ptr(), d["img"].data_ptr(), d["world"].data_ptr(), d["wfill"].data_ptr(),
                        b["frame_offsets"], lo[rank], lo[rank + 1], d["depth"].data_ptr() + 4 * lo[rank] * H * W,
                        d["fill"].data_ptr() + 4 * lo[rank] * H * W, W, H, b["curves"])
                    assert all(same(part[f - lo[rank]], got[f]) for f in range(lo[rank], lo[rank + 1])), (n, N, rank)
            for cs in ranks.values():
                for r in cs:
                    apply(r, {})
    finally:
        for cs in ranks.values():
            for r in cs:
                apply(r, {})
