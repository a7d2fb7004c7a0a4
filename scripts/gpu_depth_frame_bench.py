"""moped3d recognition steps (CLUSTER_LINKAGE -> POSE -> FILTER -> POSE2 -> FILTER2) on the same seeded 640x480 RGB-D frames, three ways:
  (a) stage by stage: mc_cluster_linkage per model -> mc_pose_depth_ransac -> mc_filter_projection -> mc_pose_depth_ransac ->
      mc_filter_projection with host buffers, the way the stage classes call them
  (b) mc_process_depth_frames with one frame per call
  (c) 64-frame batches through mc_process_depth_frames (host arrays) and mc_process_depth_frames_dev (arrays on the device)
Asserts that every path returns the same objects (bit for bit), reports frames/s per path (windows of >= 1 s after a warm-up, repeated
for the spread) and the per-step split, and records the card's name, power limit and max SM clock.

    python scripts/gpu_depth_frame_bench.py [--out profiles/depth_frame_bench.jsonl] [--repeats 3] [--window 1.0]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from moped_b200 import capi, synth  # noqa: E402
from test_gpu_depth_frame import same_objects, stage_by_stage  # noqa: E402


def rate(fn, frames_per_call, window, repeats):
    """frames/s of `fn` over `repeats` windows of at least `window` seconds (each call ends in a device synchronisation)"""
    out = []
    for _ in range(repeats):
        n, t0 = 0, time.perf_counter()
        while True:
            fn()
            n += 1
            dt = time.perf_counter() - t0
            if dt >= window:
                break
        out.append(n * frames_per_call / dt)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "depth_frame_bench.jsonl"))
    ap.add_argument("--frames", type=int, default=64)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--window", type=float, default=1.0)
    a = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    ctx = capi.Context(0)
    ctx.set_cameras(synth.K_DEPTH, synth.CAM_IDENTITY)
    P = ctx.default_depth_params()
    frs = [synth.make_depth_frame(1000 + s) for s in range(a.frames)]
    n_models = len(frs[0]["match_offsets"]) - 1
    b = synth.stack_depth_frames(frs)
    keys = ("match_image", "match_xy", "match_xyz", "match_world", "match_fill", "depth", "fill_distance")
    dev = {k: torch.from_numpy(np.ascontiguousarray(b[k])).cuda() for k in keys}

    def one(fr, times=None):
        return ctx.process_depth_frames(fr["match_offsets"][None], n_models, fr["match_image"], fr["match_xy"], fr["match_xyz"], fr["match_world"],
                                        fr["match_fill"], fr["depth"], fr["fill_distance"], params=P, times=times)[0]

    def batch():
        return ctx.process_depth_frames(b["match_offsets"], n_models, *[b[k] for k in keys], params=P)

    def batch_dev():
        return ctx.process_depth_frames_dev(b["match_offsets"], n_models, *[dev[k].data_ptr() for k in keys], 640, 480, params=P)

    # the same objects on every path
    ref = [stage_by_stage(ctx, fr, P) for fr in frs]
    singles = [one(fr) for fr in frs]
    outs_b, outs_d = batch(), batch_dev()
    for f in range(a.frames):
        for o in (singles[f], outs_b[f], outs_d[f]):
            assert same_objects(o, ref[f]), f"frame {f}: paths disagree"
            assert o["info"][3] == ref[f]["n_clusters"]
    n_obj = sum(len(r["model"]) for r in ref)
    n_matches = int(b["match_offsets"][:, -1].sum() - b["match_offsets"][:, 0].sum())

    # per-step split: stage by stage (host clock around each synchronous call) and the chain (device time, frames in order on one lane)
    split_a = np.zeros(5)
    for fr in frs:
        stage_by_stage(ctx, fr, P, split=split_a)
    split_a_ms = (split_a / a.frames * 1e3).tolist()
    st = np.zeros(5, np.float32)
    acc = np.zeros(5)
    for fr in frs:
        one(fr, times=st)
        acc += st
    split_b_ms = (acc / a.frames).tolist()

    fps_a = rate(lambda: [stage_by_stage(ctx, fr, P) for fr in frs[:8]], 8, a.window, a.repeats)
    it = iter(range(1 << 30))
    fps_b = rate(lambda: one(frs[next(it) % a.frames]), 1, a.window, a.repeats)
    fps_c = rate(batch, a.frames, a.window, a.repeats)
    fps_cd = rate(batch_dev, a.frames, a.window, a.repeats)
    lanes = 8
    rec = dict(bench="moped3d frames: CLUSTER_LINKAGE..FILTER2", gpu=gpu, frames=a.frames, n_models=n_models, matches=n_matches, objects=n_obj,
               frame_lanes=lanes, params="mc_depth_pipeline_default_params (variant 0, linkage_cached 1)",
               fps_a_stage_by_stage=fps_a, fps_b_one_frame_per_call=fps_b, fps_c_batch64_host=fps_c, fps_c_batch64_dev=fps_cd,
               split_a_host_ms_per_frame=dict(zip(("cluster", "pose", "filter", "pose2", "filter2"), split_a_ms)),
               split_b_device_ms_per_frame=dict(zip(("cluster", "pose", "filter", "pose2", "filter2"), split_b_ms)),
               note="frames/s over windows of >= %.1f s after a warm-up (one entry per window); all paths return bit-identical objects" % a.window)
    line = json.dumps(rec)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "a") as f:
        f.write(line + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
