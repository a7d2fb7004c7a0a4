"""moped3d's linkage, depth pose and frame chain at the sizes the C ABI accepts, and on duplicate matches.

The linkage kernels run 256-thread CTAs with strided loops; mc_cluster_linkage and the frame chain accept up to 2048 matches per model
and 2^24 similarity entries per frame. Here every stage is compared with the oracle above one block (n = 255, 256, 257, 600, 1024,
2048) and at the chain's limits. Duplicate matches (SIFT's secondary orientation peaks: the same pixel, model point and world point
twice) make get3DFilterK's |dm - dw| / dm a 0/0, so the similarity matrix holds NaN, which the reference's strict > never merges on.

Bars:
  * agglomeration on the oracle's matrix: bit-identical clusters, every linkage type; average linkage with both kernels
    (mc_set_option("linkage_cached") 1 and 0; single and complete linkage always run the scan kernel);
  * mc_cluster_linkage end to end: the oracle's NaN positions, finite entries within 2e-6 (CUDA vs glibc expf / atan2f), a symmetric
    matrix, and the clusters of oracle.linkage_agglomerate on the GPU's own matrix (an ulp of expf may flip a near-tie, which the
    oracle's matrix would turn into a different merge order without any kernel being wrong);
  * depth pose on clusters of 300, 1000 and 2048 points: bit-exact hypotheses and RANSAC, team widths 32 and 8;
  * the frame chain: what the stage-by-stage calls give, for both agglomeration kernels; clusters equal to the oracle's agglomeration
    of every model's GPU matrix; POSE..FILTER2 equal to the oracle's on those clusters; a frame of exactly 2^24 similarity entries is
    accepted and one more match is a capacity error; a batch of full-size and small frames equals the frames one by one.
"""
import functools

import numpy as np
import pytest

import oracle_chain3d
from moped_b200 import capi, synth
from oracle import oracle
from test_gpu_depth_frame import expect, run_batch, same_objects, stage_by_stage
from test_gpu_depth_pose import LM, MIN_NPTS, THR, pack
from test_oracle3d_pose import ALPHA, CAM, K, make_cluster

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900, method="thread")]

SIZES = (255, 256, 257, 600, 1024, 2048)
GOLDEN = 0x9E3779B97F4A7C15
M64 = 0xFFFFFFFFFFFFFFFF


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    c.set_cameras(synth.K_DEPTH, synth.CAM_IDENTITY)
    yield c
    c.close()


# ---- linkage on one model ------------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def scene(n, dup):
    """make_linkage_scene scaled to n matches (two instances of 45 % and 30 %, the rest outliers), `dup` of them duplicated;
    n = 600 is the scene bench.py --workload linkage times (make_linkage_scene(1))"""
    if n == 600:
        xy, xyz, world, depth, dist = synth.make_linkage_scene(1)
    else:
        a, b = int(0.45 * n), int(0.3 * n)
        xy, xyz, world, depth, dist = synth.make_linkage_scene(n, n_per=(a, b), n_out=n - a - b)
    if dup:
        xy, xyz, world = synth.duplicate_matches((xy, xyz, world), dup, n)
    return xy, xyz, world, depth, dist


def scenes(n):
    return ((n, 0), (n, max(5, n // 20)))                    # and about 5 % of its matches duplicated


@functools.lru_cache(maxsize=None)
def oracle_similarity(n, dup, use3d=2):
    return oracle.linkage_similarity(*scene(n, dup), use3d_filter=use3d)


@functools.lru_cache(maxsize=None)
def oracle_clusters(n, dup, linkage):
    return oracle.linkage_agglomerate(oracle_similarity(n, dup), 0.1, 7, linkage)


@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("linkage,cached", [(1, 1), (1, 0), (0, 1), (2, 1)])
def test_agglomeration_on_the_oracles_matrix(ctx, linkage, cached, n):
    ctx.set_option("linkage_cached", cached)
    try:
        for key in scenes(n):
            Ko = oracle_similarity(*key)
            assert np.isnan(Ko).sum() == 2 * key[1], key              # one NaN pair per duplicated match
            oo, om = oracle_clusters(*key, linkage)
            go, gm = ctx.linkage_agglomerate(Ko, 0.1, 7, linkage)
            assert np.array_equal(oo, go) and np.array_equal(om, gm), (key, len(oo) - 1, len(go) - 1)
            assert len(oo) > 2                                         # something to get wrong: at least two clusters
    finally:
        ctx.set_option("linkage_cached", 1)


@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("use3d", [0, 1, 2])
def test_similarity_and_clusters_end_to_end(ctx, use3d, n):
    for key in scenes(n):
        xy, xyz, world, depth, dist = scene(*key)
        Ko = oracle_similarity(*key, use3d)
        go, gm, Kg = ctx.cluster_linkage(xy, xyz, world, depth, dist, use3d_filter=use3d, want_similarity=True)
        nan = np.isnan(Ko)
        assert nan.sum() == (2 * key[1] if use3d else 0), key
        assert np.array_equal(np.isnan(Kg), nan), key
        assert np.abs(Kg[~nan] - Ko[~nan]).max() < 2e-6, (key, np.abs(Kg[~nan] - Ko[~nan]).max())
        assert np.array_equal(Kg.view(np.uint32), Kg.T.view(np.uint32)), key
        oo, om = oracle.linkage_agglomerate(Kg, 0.1, 7, 1)
        assert np.array_equal(oo, go) and np.array_equal(om, gm), (key, len(oo) - 1, len(go) - 1)
        assert len(go) > 2


# ---- depth pose on large clusters ----------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def large_clusters():
    return [make_cluster(900 + i, n=n, outliers=o) for i, (n, o) in enumerate(((300, 0.3), (1000, 0.5), (2048, 0.2)))]


@pytest.mark.parametrize("variant", [0, 1])
def test_depth_hypotheses_on_large_clusters(ctx, variant):
    cams = oracle.cameras(K[None], CAM[None])
    ctx.set_cameras(K[None], CAM[None])
    clusters = large_clusters()
    rng = np.random.default_rng(31 + variant)
    hyp_cluster, sample_pos, init_quat = [], [], []
    for ci, cl in enumerate(clusters):
        for h in range(12):
            pos = rng.choice(cl["good"], 5, replace=False) if h % 3 else rng.choice(len(cl["xy"]), 5, replace=False)
            hyp_cluster.append(ci); sample_pos.append(pos); init_quat.append(rng.integers(0, 256, 4) / 256.0)
    hyp_cluster = np.array(hyp_cluster, np.int32); sample_pos = np.array(sample_pos, np.int32); init_quat = np.array(init_quat, np.float32)
    off, xy, xyz, world, cw, img = pack(clusters, variant)
    P = (192, LM, 1, 5, MIN_NPTS, THR)
    want = [oracle.hypothesis_depth(clusters[hyp_cluster[h]], cams, ALPHA, sample_pos[h], init_quat[h], LM, THR, MIN_NPTS, variant=variant)
            for h in range(len(hyp_cluster))]
    assert sum(o["n_inliers"] > MIN_NPTS for o in want) >= 18
    try:
        for lanes in (32, 8):
            ctx.set_option("depth_team_lanes", lanes)
            n_in, pose_lm, pose_refit, err, masks = ctx.pose_depth_hypotheses(variant, off, xy, xyz, world, cw, img, hyp_cluster, sample_pos,
                                                                              init_quat, P, ALPHA, want_mask=True)
            for h, o in enumerate(want):
                assert n_in[h] == o["n_inliers"], (lanes, h, n_in[h], o["n_inliers"])
                assert np.array_equal(masks[h], o["mask"].astype(bool)), (lanes, h)
                assert np.array_equal(err[h], o["lm_err"]), (lanes, h, err[h], o["lm_err"])
                if o["n_inliers"] >= 0:
                    assert np.array_equal(pose_lm[h], o["pose_lm"]) and np.array_equal(pose_refit[h], o["pose_refit"]), (lanes, h)
    finally:
        ctx.set_option("depth_team_lanes", 32)
        ctx.set_cameras(synth.K_DEPTH, synth.CAM_IDENTITY)


@pytest.mark.parametrize("variant", [0, 1])
def test_depth_ransac_on_large_clusters(ctx, variant):
    cams = oracle.cameras(K[None], CAM[None])
    ctx.set_cameras(K[None], CAM[None])
    clusters = large_clusters() + [make_cluster(910, n=1000, outliers=1.0)]            # junk: exhausts its tests
    off, xy, xyz, world, cw, img = pack(clusters, variant)
    max_ransac, max_obj, seed = 24, 2, 17
    P = (max_ransac, LM, max_obj, 5, MIN_NPTS, THR)
    try:
        for lanes in (32, 8):
            ctx.set_option("depth_team_lanes", lanes)
            found, pose, n_tests = ctx.pose_depth_ransac(variant, off, xy, xyz, world, cw, img, P, ALPHA, seed=seed)
            assert found[:2 * max_obj].any() and not found[-max_obj:].any(), (lanes, found)
            for task in range(len(found)):
                f, p, it = oracle.ransac_depth(clusters[task // max_obj], cams, ALPHA, (max_ransac, LM, 5, MIN_NPTS, THR),
                                               (seed + GOLDEN * (task + 1)) & M64, variant=variant)
                assert bool(found[task]) == f and n_tests[task] == it, (lanes, task, found[task], f, n_tests[task], it)
                if f:
                    assert np.array_equal(pose[task], p), (lanes, task, pose[task], p)
    finally:
        ctx.set_option("depth_team_lanes", 32)
        ctx.set_cameras(synth.K_DEPTH, synth.CAM_IDENTITY)


# ---- the frame chain at full size ----------------------------------------------------------------------------------------------------
def sized_frame(seed, sizes, junk=True):
    """make_depth_frame with instances of 2048 matches, its seen models cut to `sizes` matches (a random subset, in model order);
    the few matches of the junk models kept or dropped"""
    fr = synth.make_depth_frame(seed, pts_per_model=2048, inst_matches=(2048, 2049))
    off = fr["match_offsets"]
    counts = np.diff(off)
    seen = np.nonzero(counts >= 2048)[0]
    assert len(seen) >= len(sizes), counts
    target = np.where(counts >= 2048, 0, counts if junk else 0)
    target[seen[:len(sizes)]] = sizes
    keep = np.concatenate([np.arange(off[m], off[m] + target[m]) for m in range(len(counts))]).astype(np.int64)
    out = dict(fr)
    out["match_offsets"] = np.concatenate([[0], np.cumsum(target)]).astype(np.int32)
    for k in ("match_image", "match_xy", "match_xyz", "match_world", "match_fill"):
        out[k] = fr[k][keep]
    return out


def with_one_more_match(fr, model):
    """fr with a copy of its first match appended to `model`"""
    off = fr["match_offsets"]
    at = int(off[model + 1])
    out = dict(fr)
    out["match_offsets"] = off + (np.arange(len(off)) > model)
    for k in ("match_image", "match_xy", "match_xyz", "match_world", "match_fill"):
        out[k] = np.insert(fr[k], at, fr[k][0], axis=0)
    return out


@pytest.fixture(scope="module")
def big_frames():
    return dict(large=sized_frame(41, (257, 600, 1024, 2048)),              # models above one block, up to the per-model limit
                edge=sized_frame(42, (2048,) * 4, junk=False),              # exactly 2^24 similarity entries
                dup=synth.make_depth_frame(43, dup_frac=0.1),               # about 10 % of the matches duplicated
                small=synth.make_depth_frame(44), small2=synth.make_depth_frame(45))


def gpu_clusters(ctx, fr, P):
    """mc_cluster_linkage on every model with matches -> the clusters model-major (as oracle_chain3d.cluster_step gives them) and, per
    model, (offsets, members, similarity matrix)"""
    off = fr["match_offsets"]
    model, offsets, members, per_model = [], [0], [], {}
    for m in range(len(off) - 1):
        lo, hi = int(off[m]), int(off[m + 1])
        if hi == lo:
            continue
        per_model[m] = co, mem, _ = ctx.cluster_linkage(fr["match_xy"][lo:hi], fr["match_xyz"][lo:hi], fr["match_world"][lo:hi], fr["depth"],
                                                        fr["fill_distance"], P.cluster_cutoff, P.cluster_min_pts, P.cluster_use_3d_filter,
                                                        P.cluster_linkage_type, P.cluster_sigma_2d, P.cluster_sigma_3d, want_similarity=True)
        for c in range(len(co) - 1):
            model.append(m); members.append(mem[co[c]:co[c + 1]]); offsets.append(offsets[-1] + int(co[c + 1] - co[c]))
    cl = dict(model=np.array(model, np.int32), offsets=np.array(offsets, np.int32),
              members=np.concatenate(members).astype(np.int32) if members else np.zeros(0, np.int32))
    return cl, per_model


@pytest.mark.parametrize("name", ["large", "edge", "dup"])
def test_frame_chain_at_full_size(ctx, big_frames, name):
    """The chain does not return its clusters: they are the stage-by-stage calls' (same kernels; the same count and the same objects
    follow from them), which are checked against the oracle's agglomeration of each model's GPU matrix."""
    fr = big_frames[name]
    counts = np.diff(fr["match_offsets"])
    P = ctx.default_depth_params()
    assert (P.cluster_linkage_type, P.cluster_use_3d_filter, P.cluster_cutoff, P.cluster_min_pts) == (1, 2, np.float32(0.1), 7)
    cl, per_model = gpu_clusters(ctx, fr, P)
    for m, (go, gm, Kg) in per_model.items():
        oo, om = oracle.linkage_agglomerate(Kg, P.cluster_cutoff, P.cluster_min_pts, 1)
        assert np.array_equal(oo, go) and np.array_equal(om, gm), (name, m, len(oo) - 1, len(go) - 1)
    if name == "dup":
        assert sum(np.isnan(Kg).any() for _, _, Kg in per_model.values()) >= 3
    else:
        assert counts.max() == 2048 and (name != "edge" or int((counts.astype(np.int64) ** 2).sum()) == 1 << 24)
    o = oracle_chain3d.frame(fr, clusters=cl)
    assert len(o["model"]) >= 3, (name, o["model"])
    try:
        for cached in (1, 0):
            ctx.set_option("linkage_cached", cached)
            ref = stage_by_stage(ctx, fr, P)
            for k in ("model", "offsets", "members"):
                assert np.array_equal(ref["clusters"][k], cl[k]), (name, cached, k)
            out = run_batch(ctx, [fr], P)[0]
            assert out["info"][3] == ref["n_clusters"] and out["info"][2] == fr["match_offsets"][-1] and out["info"][1] == 0, (name, out["info"])
            assert same_objects(out, ref), (name, cached, out["model"], ref["model"])
            assert same_objects(out, o), (name, cached, out["model"], o["model"])
    finally:
        ctx.set_option("linkage_cached", 1)


def test_frame_at_the_similarity_entry_limit(ctx, big_frames):
    edge = big_frames["edge"]
    counts = np.diff(edge["match_offsets"])
    assert int((counts.astype(np.int64) ** 2).sum()) == 1 << 24 and (counts > 0).sum() == 4
    out = run_batch(ctx, [edge])[0]
    assert out["info"][1] == 0 and out["info"][3] > 0 and len(out["model"]) > 0
    over = with_one_more_match(edge, int(np.nonzero(counts == 0)[0][0]))
    assert int((np.diff(over["match_offsets"]).astype(np.int64) ** 2).sum()) == (1 << 24) + 1
    msg = expect(-4, lambda: run_batch(ctx, [over]))
    assert "2^24" in msg, msg
    assert same_objects(run_batch(ctx, [edge])[0], out)            # the context is still usable


def test_batch_of_full_size_and_small_frames(ctx, big_frames):
    frs = [big_frames[k] for k in ("large", "small", "edge", "dup", "small2")]
    singles = [run_batch(ctx, [fr])[0] for fr in frs]
    assert all(len(s["model"]) > 0 for s in singles)
    try:
        for lanes in (1, 8):                          # one lane: its buffers grow and shrink from frame to frame
            ctx.set_tuning(frame_lanes=lanes)
            outs = run_batch(ctx, frs)
            for f, (o, s) in enumerate(zip(outs, singles)):
                assert np.array_equal(o["info"], s["info"]) and same_objects(o, s), (lanes, f)
    finally:
        ctx.set_tuning(frame_lanes=8)
