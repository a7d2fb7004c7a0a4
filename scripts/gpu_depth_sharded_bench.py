"""moped3d's MATCH step on an object-sharded database (mc_match_adaptive_frames_merged_dev).

Workload: the one of scripts/gpu_depth_match_bench.py — a 1000-model, 1 M-row synthetic database and 64 frames x 2000 features
(synth.make_adaptive_frames with moped3d's DimensionPeak / DimensionFade of 150 / 50 px).

One-GPU proxy (always): N in {1, 2, 4, 8} shard contexts on one card (N = 1: the context holding the whole database). For each N:
  match_shard      mc_match_dev of all queries against one 1/N shard (what every rank runs before the all-gather)
  merged_batch     the merged entry over the N gathered blocks for the whole batch
  merged_rank      the same for the 64/N frames of one rank
next to mc_match_adaptive_frames_dev on the whole database. The gathered blocks (N x 16 bytes per feature, at most 16 MB) stay in L2
between steps; they are not flushed.

Multi-GPU leg (only with more than one visible GPU): one process per GPU (torch.multiprocessing, NCCL all_gather_into_tensor). A step of
the sharded arm is: mc_match_dev on the rank's shard -> all-gather of the packed blocks -> merged entry for the rank's frames -> DEPTHPROP's
world point and fill distance gathered through match_feature -> mc_process_depth_frames_dev on those frames. The replicated arm holds the
whole database on every rank and runs mc_match_adaptive_frames_dev on the rank's frames only, then the same chain. Both arms must give the
same objects.

Timings: host clock around work that ends in a device synchronisation, warm-up, then --steps steps. Asserts that the timed batch's MATCH
outputs equal the whole-database reference bit for bit. Records the card's name, power limit and max SM clock; appends one JSON line to
--out.

    python scripts/gpu_depth_sharded_bench.py [--out profiles/depth_sharded_bench.jsonl] [--steps 20] [--warmup 3]
"""
import argparse
import json
import os
import socket
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from moped_b200 import capi, synth  # noqa: E402
from moped_b200.sharding import shard_objects  # noqa: E402


def timed(fn, warmup, steps):
    """seconds per call of `fn` (which ends in a device synchronisation), one entry per step"""
    for _ in range(warmup):
        fn()
    out = []
    for _ in range(steps):
        t0 = time.perf_counter()
        fn()
        out.append(time.perf_counter() - t0)
    return out


def ms(t):
    return dict(median=float(np.median(t)) * 1e3, min=float(np.min(t)) * 1e3, max=float(np.max(t)) * 1e3)


def workload(a):
    db = synth.make_db(a.models, a.rows_per_model)
    b = synth.make_adaptive_frames(db, a.frames, n_features=a.features, empty=(), far=(), dimensions=capi.ADAPTIVE_DEFAULTS[4:])
    return db, b


def context(db, n_models, rows=None, device=0):
    c = capi.Context(device)
    r0, r1 = rows if rows else (0, len(db["desc"]))
    c.db_upload(db["desc"][r0:r1], db["xyz"][r0:r1], db["model_of_row"][r0:r1], n_models, row_base=r0)
    if rows:
        c.db_set_global_tables(db["xyz"], db["model_of_row"], n_models)
    c.set_cameras(synth.K_DEPTH, synth.CAM_IDENTITY)
    return c


def outputs(Q, dev):
    return dict(feat=torch.zeros(Q, dtype=torch.int32, device=dev), img=torch.zeros(Q, dtype=torch.int32, device=dev),
                xy=torch.zeros((Q, 2), dtype=torch.float32, device=dev), xyz=torch.zeros((Q, 3), dtype=torch.float32, device=dev),
                nn_row=torch.zeros((Q, 2), dtype=torch.int32, device=dev), nn_dist=torch.zeros((Q, 2), dtype=torch.float32, device=dev),
                acc=torch.zeros(Q, dtype=torch.uint8, device=dev))


def match_block(c, d, Q, blk, acc):
    c.match_dev(d["desc"].data_ptr(), Q, 1.0, capi.MATCH_TENSOR, blk.data_ptr(), blk.data_ptr() + 8 * Q, acc.data_ptr())
    c.synchronize()


def merged(c, packed, n_shards, d, fo, lo, hi, W, H, curves, o):
    return c.match_adaptive_frames_merged_dev(packed.data_ptr(), n_shards, d["xy"].data_ptr(), d["image"].data_ptr(), fo, lo, hi,
                                              d["depth"].data_ptr() + 4 * lo * H * W, d["fill_distance"].data_ptr() + 4 * lo * H * W, W, H,
                                              curves, o["feat"].data_ptr(), o["img"].data_ptr(), o["xy"].data_ptr(), o["xyz"].data_ptr(),
                                              o["nn_row"].data_ptr(), o["nn_dist"].data_ptr(), o["acc"].data_ptr())


def whole_batch(c, d, fo, W, H, curves, o):
    return c.match_adaptive_frames_dev(d["desc"].data_ptr(), d["xy"].data_ptr(), d["image"].data_ptr(), fo, d["depth"].data_ptr(),
                                       d["fill_distance"].data_ptr(), W, H, curves, o["feat"].data_ptr(), o["img"].data_ptr(), o["xy"].data_ptr(),
                                       o["xyz"].data_ptr(), o["nn_row"].data_ptr(), o["nn_dist"].data_ptr(), o["acc"].data_ptr())


def same_match(r, o, ref_r, ref_o, fo, lo, hi):
    """frames [lo, hi) of a merged call equal the whole-database reference, bit for bit"""
    assert np.array_equal(r["match_offsets"], ref_r["match_offsets"][lo:hi]) and np.array_equal(r["frame_info"], ref_r["frame_info"][lo:hi])
    a, z = int(fo[lo]), int(fo[hi])
    for k in ("nn_row", "nn_dist", "acc"):
        assert torch.equal(o[k][a:z].view(torch.int32) if o[k].dtype == torch.float32 else o[k][a:z],
                           ref_o[k][a:z].view(torch.int32) if ref_o[k].dtype == torch.float32 else ref_o[k][a:z]), k
    for f in range(lo, hi):
        s, n = int(fo[f]), int(ref_r["frame_info"][f][1])
        for k in ("feat", "img", "xy", "xyz"):
            assert torch.equal(o[k][s:s + n].view(torch.int32), ref_o[k][s:s + n].view(torch.int32)), (f, k)


def proxy(a, db, b, gpu):
    dev = torch.device("cuda", 0)
    fo, curves = b["frame_offsets"], b["curves"]
    Q, F = int(fo[-1]), a.frames
    H, W = b["depth"].shape[1:]
    d = {k: torch.from_numpy(np.ascontiguousarray(b[k])).to(dev) for k in ("desc", "xy", "image", "depth", "fill_distance")}
    whole = context(db, a.models)
    ref_o = outputs(Q, dev)
    torch.cuda.synchronize()
    t_whole = timed(lambda: whole_batch(whole, d, fo, W, H, curves, ref_o), a.warmup, a.steps)
    ref_r = whole_batch(whole, d, fo, W, H, curves, ref_o)
    assert ref_r["status"] == 0
    acc = torch.empty(Q, dtype=torch.uint8, device=dev)
    res = {}
    for N in (1, 2, 4, 8):
        ctxs = [whole] if N == 1 else [context(db, a.models, (r0, r1)) for _, _, r0, r1 in shard_objects(db["n_pts"], N)]
        packed = torch.empty((N, 4 * Q), dtype=torch.int32, device=dev)
        for r, c in enumerate(ctxs):
            match_block(c, d, Q, packed[r], acc)
        c0 = ctxs[0]
        blk = torch.empty(4 * Q, dtype=torch.int32, device=dev)
        t_match = timed(lambda: match_block(c0, d, Q, blk, acc), a.warmup, a.steps)
        assert torch.equal(blk, packed[0])
        o = outputs(Q, dev)
        torch.cuda.synchronize()
        t_batch = timed(lambda: merged(c0, packed, N, d, fo, 0, F, W, H, curves, o), a.warmup, a.steps)
        same_match(merged(c0, packed, N, d, fo, 0, F, W, H, curves, o), o, ref_r, ref_o, fo, 0, F)
        per = F // N
        t_rank = timed(lambda: merged(c0, packed, N, d, fo, 0, per, W, H, curves, o), a.warmup, a.steps)
        same_match(merged(c0, packed, N, d, fo, 0, per, W, H, curves, o), o, ref_r, ref_o, fo, 0, per)
        l0 = c0.launches
        merged(c0, packed, N, d, fo, 0, F, W, H, curves, o)
        res[N] = dict(shard_rows=int(c0.L.mc_db_rows(c0.h)), match_shard_ms=ms(t_match), merged_batch_ms=ms(t_batch), merged_rank_frames=per,
                      merged_rank_ms=ms(t_rank), gathered_bytes=int(N * 16 * Q), launches_per_merged_call=int(c0.launches - l0))
        print(f"[proxy] N={N}: match_dev on a 1/{N} shard {np.median(t_match) * 1e3:.2f} ms, merged batch {np.median(t_batch) * 1e3:.3f} ms, "
              f"merged {per} frames {np.median(t_rank) * 1e3:.3f} ms", file=sys.stderr)
        for c in ctxs:
            if c is not whole:
                c.close()
    whole.close()
    return dict(match_adaptive_frames_dev_whole_ms=ms(t_whole), match_adaptive_frames_dev_whole_frames_per_s=F / float(np.median(t_whole)),
                shards={str(k): v for k, v in res.items()})


def free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def rank_main(rank, world, a, port, queue):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), NCCL_DEBUG_FILE="/dev/stderr")
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        db, b = workload(a)
        fo, curves = b["frame_offsets"], b["curves"]
        Q, F = int(fo[-1]), a.frames
        H, W = b["depth"].shape[1:]
        per = F // world
        lo, hi = rank * per, (rank + 1) * per
        ql, qh = int(fo[lo]), int(fo[hi])
        d = {k: torch.from_numpy(np.ascontiguousarray(b[k])).to(dev) for k in ("desc", "xy", "image", "depth", "fill_distance", "world", "fill")}
        _, _, r0, r1 = shard_objects(db["n_pts"], world)[rank]
        shard, full = context(db, a.models, (r0, r1), rank), context(db, a.models, None, rank)
        own = torch.empty(4 * Q, dtype=torch.int32, device=dev)
        packed = torch.empty((world, 4 * Q), dtype=torch.int32, device=dev)
        acc = torch.empty(Q, dtype=torch.uint8, device=dev)
        o_s = outputs(Q, dev)
        # the replicated arm: the rank's frames alone, as a batch of their own
        fo_r = (fo[lo:hi + 1] - fo[lo]).astype(np.int32)
        d_r = {k: d[k][ql:qh] for k in ("desc", "xy", "image", "world", "fill")}
        d_r.update(depth=d["depth"][lo:hi], fill_distance=d["fill_distance"][lo:hi])
        o_r = outputs(qh - ql, dev)

        def chain(c, r, o, world_pts, fill):
            feat = o["feat"].long()
            wp, fl = world_pts[feat].contiguous(), fill[feat].contiguous()
            torch.cuda.synchronize(dev)
            return c.process_depth_frames_dev(r["match_offsets"], a.models, o["img"].data_ptr(), o["xy"].data_ptr(), o["xyz"].data_ptr(),
                                              wp.data_ptr(), fl.data_ptr(), d["depth"][lo].data_ptr(), d["fill_distance"][lo].data_ptr(), W, H)

        def sharded():
            match_block(shard, d, Q, own, acc)
            dist.all_gather_into_tensor(packed, own)
            torch.cuda.synchronize(dev)
            r = merged(shard, packed, world, d, fo, lo, hi, W, H, curves, o_s)
            return r, chain(shard, r, o_s, d["world"], d["fill"])

        def replicated():
            r = whole_batch(full, d_r, fo_r, W, H, curves, o_r)
            return r, chain(full, r, o_r, d_r["world"], d_r["fill"])

        def step(fn):
            def run():
                dist.barrier()
                fn()
                torch.cuda.synchronize(dev)
                dist.barrier()
            return run

        t_s = timed(step(sharded), a.warmup, a.steps)
        t_r = timed(step(replicated), a.warmup, a.steps)
        (rs, objs_s), (rr, objs_r) = sharded(), replicated()
        assert np.array_equal(rs["match_offsets"] - fo[lo], rr["match_offsets"]) and np.array_equal(rs["frame_info"], rr["frame_info"])
        assert all(np.array_equal(x["model"], y["model"]) and np.array_equal(x["pose"].view(np.uint32), y["pose"].view(np.uint32))
                   and np.array_equal(x["info"], y["info"]) for x, y in zip(objs_s, objs_r))
        med = torch.tensor([np.median(t_s), np.median(t_r)], dtype=torch.float64, device=dev)
        dist.all_reduce(med, op=dist.ReduceOp.MAX)
        if rank == 0:
            queue.put(dict(world=world, frames_per_rank=per, step_ms_sharded=float(med[0]) * 1e3, step_ms_replicated=float(med[1]) * 1e3,
                           frames_per_s_sharded=F / float(med[0]), frames_per_s_replicated=F / float(med[1])))
        shard.close()
        full.close()
    finally:
        dist.destroy_process_group()


def multi_gpu(a, world):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    queue = ctx.SimpleQueue()
    mp.start_processes(rank_main, args=(world, a, free_port(), queue), nprocs=world, join=True, start_method="spawn")
    return queue.get()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "depth_sharded_bench.jsonl"))
    ap.add_argument("--models", type=int, default=1000)
    ap.add_argument("--rows-per-model", type=int, default=1000)
    ap.add_argument("--frames", type=int, default=64)
    ap.add_argument("--features", type=int, default=2000)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("gpu_depth_sharded_bench.py: no CUDA device")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    db, b = workload(a)
    rec = dict(bench="moped3d MATCH on an object-sharded database (mc_match_adaptive_frames_merged_dev)", gpu=gpu[0], gpus_visible=len(gpu),
               db_rows=int(len(db["desc"])), models=a.models, frames=a.frames, features_per_frame=a.features, queries=int(b["frame_offsets"][-1]),
               steps=a.steps, warmup=a.warmup, one_gpu_proxy=proxy(a, db, b, gpu[0]))
    world = torch.cuda.device_count()
    rec["multi_gpu"] = multi_gpu(a, world) if world > 1 else "not measured: one GPU visible"
    rec["note"] = ("host clock around calls that end in a device synchronisation; merged outputs equal mc_match_adaptive_frames_dev on the whole "
                   "database bit for bit on the timed batch; gathered blocks L2-resident between steps")
    line = json.dumps(rec)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "a") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
