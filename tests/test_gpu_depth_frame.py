"""mc_process_depth_frames* (depth_frames.cu): moped3d's CLUSTER -> POSE -> FILTER -> POSE2 -> FILTER2 chained on the device.

Bar: BIT-EXACT. A frame must give what the stage-by-stage C-ABI calls give (mc_cluster_linkage per model, mc_pose_depth_ransac with the
match index as tie id, mc_filter_projection), what the oracle chain gives (tests/oracle_chain3d.py), and the same whatever the batch
and the number of frame lanes."""
import re

import numpy as np
import pytest

import oracle_chain3d
from moped_b200 import capi, synth
from oracle import oracle

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900, method="thread")]

GOLDEN = 0x9E3779B97F4A7C15
M64 = 0xFFFFFFFFFFFFFFFF


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    c.set_cameras(synth.K_DEPTH, synth.CAM_IDENTITY)
    yield c
    c.close()


def frames(seeds, n_models=12):
    return [synth.make_depth_frame(s, n_models=n_models) for s in seeds]


def run_batch(ctx, frs, params=None, max_objects=64, times=None):
    b = synth.stack_depth_frames(frs)
    return ctx.process_depth_frames(b["match_offsets"], len(frs[0]["match_offsets"]) - 1, b["match_image"], b["match_xy"], b["match_xyz"],
                                    b["match_world"], b["match_fill"], b["depth"], b["fill_distance"], params=params, max_objects=max_objects,
                                    times=times)


def stage_by_stage(ctx, fr, P, split=None):
    """The five C-ABI stage calls the way the stage classes make them: host buffers, one call per step (per model for CLUSTER).
    `split` (optional, 5 floats) accumulates the host seconds of each step."""
    import time
    t0 = time.perf_counter()
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
    n_clusters = len(model)
    cauchy = oracle.cauchy_weights(fr["match_fill"], P.variant)
    objects = []

    def pose(cl, pp, alpha):
        if len(cl["model"]) == 0:
            return
        j = np.concatenate([int(off[m]) + cl["members"][cl["offsets"][k]:cl["offsets"][k + 1]] for k, m in enumerate(cl["model"])])
        tie = np.concatenate([cl["members"][cl["offsets"][k]:cl["offsets"][k + 1]] for k in range(len(cl["model"]))])
        found, p, _ = ctx.pose_depth_ransac(P.variant, cl["offsets"], fr["match_xy"][j], fr["match_xyz"][j], fr["match_world"][j], cauchy[j],
                                            fr["match_image"][j], pp, alpha, pt_tie=tie)
        mo = pp.max_objects_per_cluster
        for t in range(len(found)):
            if found[t]:
                objects.append((int(cl["model"][t // mo]), p[t].copy()))

    def filt(mp, fd, ms):
        nonlocal objects
        if not objects:
            return dict(model=np.zeros(0, np.int32), offsets=np.zeros(1, np.int32), members=np.zeros(0, np.int32)), np.zeros(0, np.float32)
        om = np.array([o[0] for o in objects], np.int32)
        f = ctx.filter(matches, om, np.stack([o[1] for o in objects]), (mp, fd, ms))
        keep = f["keep"]
        surv = [objects[i] for i in range(len(objects)) if keep[i]]
        order = sorted((int(om[i]), i) for i in range(len(objects)) if keep[i])
        objects = surv
        return dict(model=np.array([m for m, _ in order], np.int32), offsets=f["offsets"], members=f["members"]), f["score"][keep]

    marks = [t0, time.perf_counter()]
    pose(clusters, P.pose, P.pose_alpha)
    marks.append(time.perf_counter())
    cl2, _ = filt(P.filter_min_points, P.filter_feature_distance, P.filter_min_score)
    marks.append(time.perf_counter())
    pose(cl2, P.pose2, P.pose2_alpha)
    marks.append(time.perf_counter())
    _, score = filt(P.filter2_min_points, P.filter2_feature_distance, P.filter2_min_score)
    marks.append(time.perf_counter())
    if split is not None:
        split += np.diff(marks)
    return dict(model=np.array([o[0] for o in objects], np.int32),
                pose=np.stack([o[1] for o in objects]).astype(np.float32) if objects else np.zeros((0, 7), np.float32),
                score=np.asarray(score, np.float32), n_clusters=n_clusters, clusters=clusters)


def same_objects(a, b):
    return (np.array_equal(a["model"], b["model"]) and np.array_equal(a["pose"].view(np.uint32), b["pose"].view(np.uint32))
            and np.array_equal(a["score"].view(np.uint32), b["score"].view(np.uint32)))


@pytest.mark.parametrize("variant", [0, 1])
@pytest.mark.parametrize("cached", [1, 0])
def test_equals_the_stage_by_stage_calls(ctx, variant, cached):
    ctx.set_option("linkage_cached", cached)
    try:
        for seed, (linkage, use3d) in zip((1, 2, 3), ((1, 2), (0, 0), (2, 1))):
            P = ctx.default_depth_params()
            P.variant = variant; P.cluster_linkage_type = linkage; P.cluster_use_3d_filter = use3d
            P.pose.seed = 11 + seed; P.pose2.seed = 23 + seed
            fr = synth.make_depth_frame(seed)
            ref = stage_by_stage(ctx, fr, P)
            out = run_batch(ctx, [fr], P)[0]
            assert out["info"][3] == ref["n_clusters"], (seed, out["info"], ref["n_clusters"])
            assert out["info"][2] == fr["match_offsets"][-1] and out["info"][1] == 0
            assert same_objects(out, ref), (seed, out["model"], ref["model"])
            if linkage == 1 and use3d == 2:
                assert len(ref["model"]) >= 4
    finally:
        ctx.set_option("linkage_cached", 1)


@pytest.mark.parametrize("variant", [0, 1])
def test_equals_the_oracle_chain(ctx, variant):
    P = ctx.default_depth_params()
    P.variant = variant
    for seed in (1, 2, 3):
        fr = synth.make_depth_frame(seed)
        o = oracle_chain3d.frame(fr, variant=variant)
        out = run_batch(ctx, [fr], P)[0]
        ref = stage_by_stage(ctx, fr, P)
        for k in ("model", "offsets", "members"):                 # the same clusters
            assert np.array_equal(ref["clusters"][k], o["clusters"][k]), (seed, k)
        assert out["info"][3] == len(o["clusters"]["model"])
        assert same_objects(out, o), (seed, out["model"], o["model"], out["pose"], o["pose"])


def with_small_models(seed):
    """every model has at most min_pts matches: no cluster"""
    fr = synth.make_depth_frame(seed)
    off = fr["match_offsets"]
    keep = np.concatenate([np.arange(off[m], min(off[m + 1], off[m] + 5)) for m in range(len(off) - 1)]).astype(np.int64)
    n = [min(int(off[m + 1] - off[m]), 5) for m in range(len(off) - 1)]
    out = dict(fr)
    out["match_offsets"] = np.concatenate([[0], np.cumsum(n)]).astype(np.int32)
    for k in ("match_image", "match_xy", "match_xyz", "match_world", "match_fill"):
        out[k] = fr[k][keep]
    return out


def empty_frame(seed):
    fr = synth.make_depth_frame(seed)
    out = dict(fr)
    out["match_offsets"] = np.zeros_like(fr["match_offsets"])
    for k in ("match_image", "match_xy", "match_xyz", "match_world", "match_fill"):
        out[k] = fr[k][:0]
    return out


def test_batches_equal_frames_one_by_one(ctx):
    import torch
    frs = frames(range(40, 100))
    frs[3] = empty_frame(3)
    frs[7] = with_small_models(7)
    frs += [empty_frame(100), with_small_models(101), frames([102])[0], frames([103])[0]]
    assert len(frs) == 64
    singles = [run_batch(ctx, [fr])[0] for fr in frs]
    assert singles[3]["info"].tolist() == [0, 0, 0, 0] and singles[7]["info"][3] == 0 and len(singles[7]["model"]) == 0
    assert sum(len(s["model"]) for s in singles) > 200
    b = synth.stack_depth_frames(frs)
    dev = {k: torch.from_numpy(np.ascontiguousarray(b[k])).cuda() for k in ("match_image", "match_xy", "match_xyz", "match_world", "match_fill",
                                                                               "depth", "fill_distance")}
    try:
        for lanes in (1, 8, 64):
            ctx.set_tuning(frame_lanes=lanes)
            for sub in (frs[:5], frs):
                outs = run_batch(ctx, sub)
                for f, (o, s) in enumerate(zip(outs, singles)):
                    assert np.array_equal(o["info"], s["info"]) and same_objects(o, s), (lanes, len(sub), f)
            outs = ctx.process_depth_frames_dev(b["match_offsets"], b["match_offsets"].shape[1] - 1, *[dev[k].data_ptr() for k in (
                "match_image", "match_xy", "match_xyz", "match_world", "match_fill", "depth", "fill_distance")], 640, 480)
            for f, (o, s) in enumerate(zip(outs, singles)):
                assert np.array_equal(o["info"], s["info"]) and same_objects(o, s), ("dev", lanes, f)
        # per-step times: the frames in order on one lane, same results
        times = np.zeros(5, np.float32)
        outs = run_batch(ctx, frs[:8], times=times)
        assert (times > 0).all(), times
        for o, s in zip(outs, singles[:8]):
            assert same_objects(o, s)
    finally:
        ctx.set_tuning(frame_lanes=8)


def test_linkage_is_batched_over_models(ctx):
    """one launch per linkage kernel whatever the number of models with matches"""
    fr = synth.make_depth_frame(5, n_models=20)
    off = fr["match_offsets"]
    m0 = int(np.argmax(np.diff(off)))
    one = dict(fr)
    lo, hi = int(off[m0]), int(off[m0 + 1])
    one["match_offsets"] = np.where(np.arange(21) <= m0, 0, hi - lo).astype(np.int32)
    for k in ("match_image", "match_xy", "match_xyz", "match_world", "match_fill"):
        one[k] = fr[k][lo:hi]
    rng = np.random.default_rng(0)
    many = dict(fr)                               # every model: its own matches, or 9 random ones
    parts, offs = {k: [] for k in ("match_image", "match_xy", "match_xyz", "match_world", "match_fill")}, [0]
    for m in range(20):
        a, b = int(off[m]), int(off[m + 1])
        if b > a:
            for k in parts:
                parts[k].append(fr[k][a:b])
        else:
            parts["match_image"].append(np.zeros(9, np.int32)); parts["match_xy"].append(rng.uniform([0, 0], [639, 479], (9, 2)).astype(np.float32))
            parts["match_xyz"].append(rng.uniform(-0.06, 0.06, (9, 3)).astype(np.float32))
            parts["match_world"].append(rng.uniform(0.5, 1.5, (9, 3)).astype(np.float32)); parts["match_fill"].append(np.zeros(9, np.float32))
        offs.append(offs[-1] + len(parts["match_image"][-1]))
    for k in parts:
        many[k] = np.concatenate(parts[k])
    many["match_offsets"] = np.array(offs, np.int32)
    assert (np.diff(many["match_offsets"]) > 0).all()
    ctx.set_tuning(frame_lanes=8)
    deltas = []
    for fr_ in (one, many, one):
        run_batch(ctx, [fr_])                       # warm: buffers reserved
        l0 = ctx.launches
        run_batch(ctx, [fr_])
        deltas.append(ctx.launches - l0)
    assert deltas[0] == deltas[1] == deltas[2], deltas


def expect(status, fn):
    with pytest.raises(capi.MopedCudaError) as e:
        fn()
    assert re.search(r"failed \(%d\)" % status, str(e.value)), str(e.value)
    return str(e.value)


def test_errors_leave_the_context_usable(ctx):
    import torch
    fr = synth.make_depth_frame(9)
    good = run_batch(ctx, [fr])[0]
    assert len(good["model"]) > 0

    def check_good():
        assert same_objects(run_batch(ctx, [fr])[0], good)

    bad = dict(fr); bad["match_xy"] = fr["match_xy"].copy(); bad["match_xy"][3] = (640.5, 10.0)
    expect(-2, lambda: run_batch(ctx, [fr, bad])); check_good()
    b = synth.stack_depth_frames([fr, bad, bad])
    dev = [torch.from_numpy(np.ascontiguousarray(b[k])).cuda() for k in ("match_image", "match_xy", "match_xyz", "match_world", "match_fill",
                                                                          "depth", "fill_distance")]
    msg = expect(-2, lambda: ctx.process_depth_frames_dev(b["match_offsets"], 12, *[t.data_ptr() for t in dev], 640, 480))
    assert "frame 1" in msg, msg
    check_good()
    for field, value in (("variant", 2), ("cluster_cutoff", -1.0)):
        P = ctx.default_depth_params(); setattr(P, field, value)
        expect(-2, lambda: run_batch(ctx, [fr], P)); check_good()
    for pp, v in (("pose", 0), ("pose2", 9)):
        P = ctx.default_depth_params(); getattr(P, pp).n_pts_align = v
        expect(-2, lambda: run_batch(ctx, [fr], P)); check_good()
    desc = dict(fr); desc["match_offsets"] = fr["match_offsets"].copy(); desc["match_offsets"][2] = desc["match_offsets"][3] + 1
    expect(-2, lambda: run_batch(ctx, [desc])); check_good()
    big = dict(fr)                                  # one model with 2049 matches
    rng = np.random.default_rng(1)
    big["match_offsets"] = np.array([0, 2049] + [2049] * 11, np.int32)
    big["match_xy"] = rng.uniform([0, 0], [639, 479], (2049, 2)).astype(np.float32)
    big["match_xyz"] = big["match_world"] = rng.uniform(0, 1, (2049, 3)).astype(np.float32)
    big["match_image"] = np.zeros(2049, np.int32); big["match_fill"] = np.zeros(2049, np.float32)
    expect(-2, lambda: run_batch(ctx, [big])); check_good()
    arena = dict(big)                               # 5 models of 2048: 2^24 similarity entries exceeded
    arena["match_offsets"] = np.array([0] + [2048 * k for k in range(1, 6)] + [10240] * 7, np.int32)
    for k in ("match_xy", "match_xyz", "match_world", "match_image", "match_fill"):
        arena[k] = np.concatenate([big[k]] * 5)[:10240]
    expect(-4, lambda: run_batch(ctx, [arena])); check_good()
    # more objects than max_objects: the true count is reported
    n = len(good["model"])
    msg = expect(-4, lambda: run_batch(ctx, [fr], max_objects=n - 1))
    check_good()
    c2 = capi.Context(0)                            # no cameras
    try:
        expect(-3, lambda: run_batch(c2, [fr]))
    finally:
        c2.close()


def test_too_many_objects_reports_the_true_count(ctx):
    import ctypes as C
    fr = synth.make_depth_frame(9)
    n = len(run_batch(ctx, [fr])[0]["model"])
    mo = max(n - 1, 1)
    P = ctx.default_depth_params()
    n_obj = np.zeros(1, np.int32)
    om, op, os_ = np.zeros(mo, np.int32), np.zeros(7 * mo, np.float32), np.zeros(mo, np.float32)
    info = np.zeros(4, np.int32)
    keep = [np.ascontiguousarray(fr[k], dtype=t).reshape(-1) for k, t in (("match_image", np.int32), ("match_xy", np.float32),
                                                                          ("match_xyz", np.float32), ("match_world", np.float32),
                                                                          ("match_fill", np.float32))]
    st = ctx.L.mc_process_depth_frames(ctx.h, fr["match_offsets"], 1, 12, *[a.ctypes.data for a in keep], fr["depth"].reshape(-1),
                                       fr["fill_distance"].reshape(-1), 640, 480, C.byref(P), mo, n_obj, om, op, os_, info, None)
    assert st == -4 and n_obj[0] == n and info[0] == n
