"""moped_b200.sharding.RigShardStep on one card: camera-rig frames from pixels to objects on an object-sharded database.

One GPU stands for N ranks: N contexts each hold an object shard (row_base) plus the global tables, each holds the images of its own frames
only, and stacking tensors stands for the all-gathers. The rig is {640x480, 1280x720} with undistortion tables on both cameras. Bar: every
frame's objects, poses, scores, frame_info and n_features equal, bit for bit, one context holding the whole database running
mc_process_rig_cameras_dev. This also shows that a frame's results do not depend on its position in the batch: each rank runs its frames
as frames 0.. of its own list."""
import os

import numpy as np
import pytest
import torch

from moped_b200 import capi, synth
from moped_b200.sharding import RigExchange, RigShardError, RigShardStep, block_range, shard_objects

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900, method="thread")]

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MAX_KP = 2048
LENSES = [(-0.2, 0.05, 0.001, -0.0005), (0.1, -0.02, 0.0, 0.0005, 0.01)]
_S, _C = np.sin(np.radians(1.5)), np.cos(np.radians(1.5))
POSES = np.array([[0, 0, 0, 1, 0, 0, 0], [0, _S, 0, _C, 0.1, 0, 0]], np.float32)


@pytest.fixture(scope="module")
def setup():
    g = dict(np.load(os.path.join(ROOT, "tests", "golden", "real_images.npz")))
    im = np.load(os.path.join(ROOT, "tests", "golden", "sift_golden.npz"))["bag4_full_double/image"]
    full = np.stack([np.roll(im, s, axis=1) for s in range(-4, 4)])
    fx, fy, cx, cy = (float(v) for v in g["K"][0])
    # camera 0: the 640x480 bag frame; camera 1: its rows 60..419 upsampled 2x to 1280x720
    raw = [full, np.ascontiguousarray(full[:, 60:420].repeat(2, axis=1).repeat(2, axis=2))]
    Ks = np.float32([[fx, fy, cx, cy], [2 * fx, 2 * fy, 2 * cx + 0.5, 2 * (cy - 60) + 0.5]])
    # the golden database's 3 planar models (the frames show them), 12 synthetic models of 300 rows (so that 7 ranks each get a shard),
    # and a one-row model that is a shard of its own (its shard's blocks carry -1 second rows)
    extra = synth.make_db(12, 300, seed=41)
    n_models = len(g["n_pts"]) + 12
    rng = np.random.default_rng(42)
    db = dict(n_pts=np.concatenate([g["n_pts"], extra["n_pts"], [1]]),
              desc=np.concatenate([g["db_desc"], extra["desc"], synth.sift_like(rng, 1)]).astype(np.float32),
              xyz=np.concatenate([g["db_xyz"], extra["xyz"], rng.uniform(-0.1, 0.1, (1, 3))]).astype(np.float32),
              model_of_row=np.concatenate([g["model_of_row"], extra["model_of_row"] + len(g["n_pts"]), [n_models]]).astype(np.int32))
    N_MODELS = n_models + 1
    stream = torch.cuda.Stream()

    def context(rows=None):
        c = capi.Context(0)
        r0, r1 = rows if rows else (0, len(db["desc"]))
        c.db_upload(db["desc"][r0:r1], db["xyz"][r0:r1], db["model_of_row"][r0:r1], N_MODELS, row_base=r0)
        if rows:
            c.db_set_global_tables(db["xyz"], db["model_of_row"], N_MODELS)
        c.set_cameras(Ks, POSES)
        for cam in range(2):
            c.set_undistortion(cam, Ks[cam], LENSES[cam], *raw[cam].shape[1:])
        c.set_tuning(8, 8, 1)
        return c

    whole = context()
    ranks = {1: [context((0, len(db["desc"])))]}
    for n in (2, 3, 8):
        shards = shard_objects(db["n_pts"][:n_models], n - 1) + [(n_models, N_MODELS, len(db["desc"]) - 1, len(db["desc"]))]
        assert all(r1 > r0 for _, _, r0, r1 in shards)
        ranks[n] = [context((r0, r1)) for _, _, r0, r1 in shards]
    yield dict(whole=whole, ranks=ranks, raw=raw, stream=stream)
    for c in [whole] + [c for cs in ranks.values() for c in cs]:
        c.close()


def batch(s, B, blank=()):
    """per-camera device images [B][H][W] of a B-frame batch; the frames in `blank` are all zeros"""
    out = []
    for c, raw in enumerate(s["raw"]):
        a = raw[(3 * np.arange(B) + 5 * c) % 8].copy()
        a[list(blank)] = 0
        out.append(torch.from_numpy(a).cuda())
    torch.cuda.synchronize()
    return out


def cams(images, lo):
    """RigShardStep.extract's cams for frames lo.. of the batch"""
    return ([t.data_ptr() + lo * t[0].numel() for t in images], [t[0].numel() for t in images], [tuple(t.shape[1:]) for t in images])


def reference(s, images):
    B = len(images[0])
    out = s["whole"].process_rig_cameras_dev(*cams(images, 0), B, True, max_keypoints=MAX_KP, max_objects=64)
    torch.cuda.synchronize()
    return out


def drive(steps, images, n_frames, bad_rank=None):
    """moped_b200.sharding.run for N contexts in one process, the all-gathers done with torch.stack on the steps' one stream;
    bad_rank's images are described with a height of 7 (an argument error of that rank's extraction)"""
    world = len(steps)
    with torch.cuda.stream(steps[0].stream):
        heads = []
        for r, st in enumerate(steps):
            lo, hi = block_range(n_frames, world, r)
            ptrs, strides, sizes = cams(images, lo)
            if r == bad_rank:
                sizes = [(7, w) for _, w in sizes]
            heads.append(st.header(*st.extract((ptrs, strides, sizes), hi - lo)))
        headers = torch.stack(heads).cpu().numpy()
        plans = []
        errors = []
        for st in steps:                                   # every rank builds the plan from the same headers
            try:
                plans.append(RigExchange(headers, n_frames))
            except RigShardError as e:
                errors.append((e.rank, e.status, str(e)))
        if errors:
            return None, errors
        plan = plans[0]
        if plan.Q:
            gathered = torch.stack([st.send(plan).view(plan.P, 128) for st in steps])
            nn_all = torch.stack([st.match(plan, st.compact(plan, gathered)) for st in steps])
            for st in steps:
                st.merge(plan, nn_all)
        res_all = torch.stack([st.frames(plan).clone() for st in steps])
        frames = steps[0].unpack(plan, res_all)
    torch.cuda.synchronize()
    return (frames, plan), None


def assert_same(got, want, n_features, what):
    assert len(got) == len(want), what
    for f, (a, b) in enumerate(zip(got, want)):
        assert np.array_equal(a["info"], b["info"]), (what, f, a["info"], b["info"])
        assert np.array_equal(a["model"], b["model"]), (what, f, a["model"], b["model"])
        assert np.array_equal(a["pose"], b["pose"]), (what, f)
        assert np.array_equal(a["score"], b["score"]), (what, f)
        assert np.array_equal(n_features[f], b["n_features"]), (what, f, n_features[f], b["n_features"])


@pytest.mark.parametrize("B,blank", [(7, (3, 4)), (16, ())])
@pytest.mark.parametrize("N", [1, 2, 3, 8])
def test_sharded_step_equals_the_whole_database(setup, N, B, blank):
    s = setup
    images = batch(s, B, blank)
    want = reference(s, images)
    assert sum(len(o["model"]) for o in want) > 0
    steps = [RigShardStep(c, r, N, 2, B, max_keypoints=MAX_KP, max_objects=64, stream=s["stream"]) for r, c in enumerate(s["ranks"][N])]
    (got, plan), err = drive(steps, images, B)
    assert err is None, err
    assert plan.Q == sum(int(o["n_features"].sum()) for o in want)
    n_features = np.concatenate([st.n_features for st in steps])
    assert_same(got, want, n_features, (N, B))
    if N == 3 and B == 7:
        assert plan.counts[1] == 0                          # rank 1 holds the blank frames 3 and 4
    if N == 8 and B == 7:
        assert plan.frames[7] == (7, 7)                     # the last rank has no frames


def test_a_batch_without_features_skips_match(setup):
    s = setup
    images = batch(s, 7, range(7))
    want = reference(s, images)
    steps = [RigShardStep(c, r, 3, 2, 7, max_keypoints=MAX_KP, max_objects=64, stream=s["stream"]) for r, c in enumerate(s["ranks"][3])]
    matched = []
    for st in steps:
        st.match = lambda plan, q_all, _st=st: matched.append(_st.rank)
    (got, plan), err = drive(steps, images, 7)
    assert err is None and plan.Q == 0 and not matched
    assert_same(got, want, np.concatenate([st.n_features for st in steps]), "blank")


def test_an_overflow_on_one_rank_fails_every_rank_before_the_exchange(setup):
    s = setup
    images = batch(s, 7, range(3, 7))                      # only rank 0's frames (0..2 of 3 ranks) have keypoints
    steps = [RigShardStep(c, r, 3, 2, 7, max_keypoints=100, max_objects=64, stream=s["stream"]) for r, c in enumerate(s["ranks"][3])]
    sent = []
    for st in steps:
        st.send = lambda plan, _st=st: sent.append(_st.rank)
    _, errors = drive(steps, images, 7)
    assert len(errors) == 3 and all(e == errors[0] for e in errors), errors
    assert errors[0][:2] == (0, capi.MC_ERR_CAPACITY)
    assert not sent
    assert (steps[0].n_features > 100).any()               # the numbers found
    # the contexts are still usable
    images = batch(s, 7)
    steps = [RigShardStep(c, r, 3, 2, 7, max_keypoints=MAX_KP, max_objects=64, stream=s["stream"]) for r, c in enumerate(s["ranks"][3])]
    (got, _), err = drive(steps, images, 7)
    assert err is None
    assert_same(got, reference(s, images), np.concatenate([st.n_features for st in steps]), "after the error")
    # any other failure travels the same way: an argument error of rank 1's extraction
    sent.clear()
    for st in steps:
        st.send = lambda plan, _st=st: sent.append(_st.rank)
    _, errors = drive(steps, images, 7, bad_rank=1)
    assert len(errors) == 3 and all(e == errors[0] for e in errors), errors
    assert errors[0][:2] == (1, capi.MC_ERR_ARG)
    assert not sent


def test_run_over_a_one_rank_nccl_group(setup, tmp_path):
    """moped_b200.sharding.run itself, with torch.distributed collectives, on a group of one rank. The step is built without a stream:
    it makes its own and sets it on the context, and run orders it after the caller's stream, which has just written the images."""
    import torch.distributed as dist
    from moped_b200.sharding import run
    s = setup
    images = batch(s, 7, (3, 4))
    want = reference(s, images)
    dist.init_process_group("nccl", init_method=f"file://{tmp_path}/pg", rank=0, world_size=1, device_id=torch.device("cuda", 0))
    try:
        step = RigShardStep(s["ranks"][1][0], 0, 1, 2, 7, max_keypoints=MAX_KP, max_objects=64)
        assert step.stream is not None and step.stream != torch.cuda.current_stream()
        with pytest.raises(ValueError):                     # a batch larger than the step's buffers, before any collective
            run(dist.group.WORLD, step, cams(images, 0), 8)
        fresh = [torch.zeros_like(t) for t in images]
        torch.cuda.synchronize()
        for f, t in zip(fresh, images):                     # written on the current stream, not synchronised before run
            f.copy_(t)
        got = run(dist.group.WORLD, step, cams(fresh, 0), 7)
        torch.cuda.synchronize()
    finally:
        dist.destroy_process_group()
    assert_same(got, want, step.n_features, "run")
