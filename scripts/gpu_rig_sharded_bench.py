"""Camera-rig frames on an object-sharded database (moped_b200.sharding.RigShardStep) against one context holding the whole database.

Workload: a 1 M-row synthetic database (synth.make_db(1000, 1000)), the {640x480, 1280x720} rig with an undistortion table on both cameras
(the 640x480 images are a frame of the reference's timing.bag, shifted per frame; the 1280x720 images are its rows 60..419 upsampled 2x),
64-frame batches with the images already in HBM.
Arms, alternating step by step after warm-up; host clock around each step, which ends in a device synchronisation:
  whole        mc_process_rig_cameras_dev on one context holding the whole database
  shardedN     the sharded step with N shard contexts on this one card, the all-gathers done with torch.stack on the step's stream:
               N extractions of 64/N frames each, N matching passes over a 1/N shard, the merge and N frame ranges. This measures what
               extraction plus exchange cost on top of the whole-database call, not a multi-GPU speed-up.
Under torchrun with more than one GPU visible, every rank also runs moped_b200.sharding.run over NCCL, one rank per GPU (the leg
"multi_gpu"); with one GPU it is reported as not measured. Per arm: median ms per batch and frames/s, and the bytes the descriptor
all-gather moves per step (world x P x 128 x 4, P = the most query rows of one rank). Every frame of every sharded arm is checked against
the whole-database call, bit for bit. Records the card's name, power limit and max SM clock; appends one JSON line per arm to --out.

    python scripts/gpu_rig_sharded_bench.py [--out profiles/rig_sharded_bench.jsonl] [--steps 10] [--warmup 2] [--shards 2 4 8]
    torchrun --nproc-per-node G scripts/gpu_rig_sharded_bench.py ...
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from moped_b200 import capi, synth  # noqa: E402
from moped_b200.sharding import RigExchange, RigShardStep, block_range, run, shard_objects  # noqa: E402

LENSES = [(-0.2, 0.05, 0.001, -0.0005), (0.1, -0.02, 0.0, 0.0005, 0.01)]
POSES = np.array([[0, 0, 0, 1, 0, 0, 0], [0, np.sin(np.radians(1.5)), 0, np.cos(np.radians(1.5)), 0.1, 0, 0]], np.float32)
MAX_KP, MAX_OBJ, B = 2048, 16, 64


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clock = [v.strip() for v in q.stdout.strip().splitlines()[0].split(",")]
    return dict(gpu=name, power_limit=power, max_sm_clock=clock)


def rig_images(dev):
    g = dict(np.load(os.path.join(ROOT, "tests", "golden", "real_images.npz")))
    im = np.load(os.path.join(ROOT, "tests", "golden", "sift_golden.npz"))["bag4_full_double/image"]
    full = np.stack([np.roll(im, s, axis=1) for s in range(-4, 4)])
    raw = [full, np.ascontiguousarray(full[:, 60:420].repeat(2, axis=1).repeat(2, axis=2))]
    fx, fy, cx, cy = (float(v) for v in g["K"][0])
    Ks = np.float32([[fx, fy, cx, cy], [2 * fx, 2 * fy, 2 * cx + 0.5, 2 * (cy - 60) + 0.5]])
    images = [torch.from_numpy(raw[c][(3 * np.arange(B) + 5 * c) % 8]).to(dev) for c in range(2)]
    return images, Ks


def cams(images, lo):
    return ([t.data_ptr() + lo * t[0].numel() for t in images], [t[0].numel() for t in images], [tuple(t.shape[1:]) for t in images])


def context(dev, db, Ks, rows, sharded, stream=None):
    c = capi.Context(dev)
    r0, r1 = rows
    c.db_upload(db["desc"][r0:r1], db["xyz"][r0:r1], db["model_of_row"][r0:r1], len(db["n_pts"]), row_base=r0)
    if sharded:
        c.db_set_global_tables(db["xyz"], db["model_of_row"], len(db["n_pts"]))
    c.set_cameras(Ks, POSES)
    for cam, (h, w) in enumerate([(480, 640), (720, 1280)]):
        c.set_undistortion(cam, Ks[cam], LENSES[cam], h, w)
    c.set_tuning(8, 1, 1)
    if stream is not None:
        c.set_stream(stream.cuda_stream)
    return c


def drive(steps, images):
    """the sharded step for N contexts in one process; -> (frames, plan)"""
    world = len(steps)
    with torch.cuda.stream(steps[0].stream):
        heads = []
        for r, st in enumerate(steps):
            lo, hi = block_range(B, world, r)
            heads.append(st.header(*st.extract(cams(images, lo), hi - lo)))
        plan = RigExchange(torch.stack(heads).cpu().numpy(), B)
        if plan.Q:
            gathered = torch.stack([st.send(plan).view(plan.P, 128) for st in steps])
            nn_all = torch.stack([st.match(plan, st.compact(plan, gathered)) for st in steps])
            for st in steps:
                st.merge(plan, nn_all)
        frames = steps[0].unpack(plan, torch.stack([st.frames(plan) for st in steps]))
    torch.cuda.synchronize()
    return frames, plan


def same(got, want):
    return all(np.array_equal(a["info"], b["info"]) and np.array_equal(a["model"], b["model"]) and np.array_equal(a["pose"], b["pose"])
               and np.array_equal(a["score"], b["score"]) for a, b in zip(got, want)) and len(got) == len(want)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "rig_sharded_bench.jsonl"))
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--shards", type=int, nargs="+", default=[2, 4, 8])
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("gpu_rig_sharded_bench.py: no CUDA device")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    info = card()
    db = synth.make_db(1000, 1000)
    images, Ks = rig_images(local)
    rows_all = (0, len(db["desc"]))
    records = []

    if world > 1:                                          # one rank per GPU over NCCL
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        stream = torch.cuda.Stream()
        _, _, r0, r1 = shard_objects(db["n_pts"], world)[rank]
        ctx = context(local, db, Ks, (r0, r1), True, stream)
        step = RigShardStep(ctx, rank, world, 2, B, max_keypoints=MAX_KP, max_objects=MAX_OBJ, stream=stream)
        lo, hi = block_range(B, world, rank)
        mine = cams(images, lo)
        ts = []
        for i in range(a.warmup + a.steps):
            dist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            run(dist.group.WORLD, step, mine, B)
            torch.cuda.synchronize()
            if i >= a.warmup:
                ts.append((time.perf_counter() - t0) * 1e3)
        t = torch.tensor([float(np.median(ts))], device=f"cuda:{local}")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        if rank == 0:
            records.append(dict(arm="multi_gpu", gpus=world, ms=float(t.item()), frames_per_s=B / float(t.item()) * 1e3))
        dist.destroy_process_group()
        ctx.close()
    if rank == 0:
        if world == 1:
            records.append(dict(arm="multi_gpu", gpus=torch.cuda.device_count(), ms=None, note="not measured: one GPU visible"))
        whole = context(local, db, Ks, rows_all, False)
        stream = torch.cuda.Stream()
        arms = {}
        for n in a.shards:
            ctxs = [context(local, db, Ks, (r0, r1), True, stream) for _, _, r0, r1 in shard_objects(db["n_pts"], n)]
            arms[n] = [RigShardStep(c, r, n, 2, B, max_keypoints=MAX_KP, max_objects=MAX_OBJ, stream=stream) for r, c in enumerate(ctxs)]
        torch.cuda.synchronize()

        def step_whole():
            return whole.process_rig_cameras_dev(*cams(images, 0), B, True, max_keypoints=MAX_KP, max_objects=MAX_OBJ)

        want = step_whole()
        checks, gbytes = {}, {}
        for n, steps in arms.items():
            got, plan = drive(steps, images)
            checks[n] = same(got, want) and np.array_equal(np.concatenate([st.n_features for st in steps]), np.stack([w["n_features"] for w in want]))
            gbytes[n] = n * plan.P * 128 * 4
        times = {k: [] for k in ["whole"] + list(arms)}
        for i in range(a.warmup + a.steps):                 # alternating arms
            for k in times:
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                if k == "whole":
                    step_whole()
                else:
                    drive(arms[k], images)
                torch.cuda.synchronize()
                if i >= a.warmup:
                    times[k].append((time.perf_counter() - t0) * 1e3)
        Q = int(sum(int(w["n_features"].sum()) for w in want))
        records.append(dict(arm="whole", ms=float(np.median(times["whole"])), frames_per_s=B / float(np.median(times["whole"])) * 1e3, queries=Q))
        for n in arms:
            ms = float(np.median(times[n]))
            records.append(dict(arm=f"sharded{n}", shards=n, ms=ms, frames_per_s=B / ms * 1e3, overhead_ms=ms - float(np.median(times["whole"])),
                                descriptor_allgather_bytes=gbytes[n], bit_exact=bool(checks[n])))
        common = dict(info, frames=B, rig="640x480+1280x720", tables=2, db_rows=len(db["desc"]), steps=a.steps, warmup=a.warmup,
                      clock="host clock around steps ending in a device synchronise; medians over alternating arms")
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "a") as f:
            for r in records:
                line = json.dumps(dict(common, **r))
                f.write(line + "\n")
                print(line)


if __name__ == "__main__":
    main()
