"""What moped3d's FILTER_PROJECTION_DEPTH costs as FILTER and FILTER2 of the device chain (mc_set_depth_filter), on two workloads:
  frames   64 seeded 640x480 RGB-D frames of synth.make_depth_frame through mc_process_depth_frames_dev (12 models of 160 keypoints):
             plain    the chain with FILTER_PROJECTION on both steps
             depth40  the depth filter on FILTER and FILTER2, 40 test points per model
             depthall the depth filter on FILTER and FILTER2, every keypoint a test point
             stages   the stage-by-stage route of a host that registers FILTER_PROJECTION_DEPTH_CUDA: mc_cluster_linkage per model,
                      mc_pose_depth_ransac, mc_filter_projection_depth on both steps (40 test points), host buffers
  queries  a 1000-model, 1 M-row database and 64 frames x 2000 features (synth.make_adaptive_frames) through mc_process_depth_queries_dev:
             plain, depth40, depthall as above (depthall: a 12 MB table of 1 M test points)
Every arm is timed with CUDA events on the context's stream (a torch stream handed to mc_set_stream) around a call, which ends in a device
synchronisation; the arms alternate round by round (`--rounds` rounds of `--steps` calls after `--warmup` calls each) and each round's
median is kept for the spread. Asserts that the depth arms equal the stage-by-stage route on the frames workload, bit for bit.
Records the card's name, power limit and max SM clock; appends one JSON line to --out.

    python scripts/gpu_depth_filter_chain_bench.py [--out profiles/depth_filter_chain_bench.jsonl] [--steps 10] [--rounds 3] [--warmup 2]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from moped_b200 import capi, synth  # noqa: E402
from test_gpu_depth_filter_chain import ALL, SETTING, apply, same_objects, stage_by_stage, draw_test_points  # noqa: E402


def timed(arms, stream, steps, rounds, warmup):
    """{arm: [median ms of each round]} with the arms alternating round by round; the events go on the contexts' stream"""
    for fn in arms.values():
        for _ in range(warmup):
            fn()
    out = {k: [] for k in arms}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for _ in range(rounds):
        for k, fn in arms.items():
            ms = []
            for _ in range(steps):
                ev[0].record(stream)
                fn()
                ev[1].record(stream)
                ev[1].synchronize()
                ms.append(ev[0].elapsed_time(ev[1]))
            out[k].append(float(np.median(ms)))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "depth_filter_chain_bench.jsonl"))
    ap.add_argument("--frames", type=int, default=64)
    ap.add_argument("--models", type=int, default=1000)
    ap.add_argument("--rows-per-model", type=int, default=1000)
    ap.add_argument("--features", type=int, default=2000)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=2)
    a = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()[0]
    stream = torch.cuda.Stream()                         # the contexts run on it: the events bracket their work

    # ---- frames: the chain alone
    ctx = capi.Context(0)
    ctx.set_stream(stream.cuda_stream)
    ctx.set_cameras(synth.K_DEPTH, synth.CAM_IDENTITY)
    P = ctx.default_depth_params()
    frs = [synth.make_depth_frame(1000 + s) for s in range(a.frames)]
    n_models = len(frs[0]["match_offsets"]) - 1
    b = synth.stack_depth_frames(frs)
    keys = ("match_image", "match_xy", "match_xyz", "match_world", "match_fill", "depth", "fill_distance")
    dev = {k: torch.from_numpy(np.ascontiguousarray(b[k])).cuda() for k in keys}
    torch.cuda.synchronize()
    H, W = b["depth"].shape[1:]
    settings = {n: {s: (SETTING[s],) + t for s, t in draw_test_points(frs[0]["model_offsets"], frs[0]["model_xyz"], n).items()} for n in (40, ALL)}

    def frames_call():
        return ctx.process_depth_frames_dev(b["match_offsets"], n_models, *[dev[k].data_ptr() for k in keys], W, H, params=P)

    current = {}

    def arm(setting):
        def run():
            if current.get("s") is not setting:          # the table is uploaded once per arm switch, not per batch
                apply(ctx, setting)
                current["s"] = setting
            return frames_call()
        return run

    stages_setting = settings[40]
    frame_arms = dict(plain=arm({}), depth40=arm(settings[40]), depthall=arm(settings[ALL]),
                      stages=lambda: [stage_by_stage(ctx, fr, P, stages_setting) for fr in frs])
    # the depth arms equal the stage-by-stage route
    apply(ctx, stages_setting)
    got = frames_call()
    ref = [stage_by_stage(ctx, fr, P, stages_setting) for fr in frs]
    assert all(same_objects(g, r) for g, r in zip(got, ref))
    objects = dict(depth40=int(sum(len(g["model"]) for g in got)))
    apply(ctx, {})
    objects["plain"] = int(sum(len(g["model"]) for g in frames_call()))
    t_frames = timed(frame_arms, stream, a.steps, a.rounds, a.warmup)
    # per-step device time (stage_ms: the frames in order on one lane). FILTER gets the same objects in every arm, so its difference is
    # the penalty's cost; FILTER2 and POSE2 see fewer objects where the penalty pruned some
    step_ms = {}
    for k, setting in (("plain", {}), ("depth40", settings[40]), ("depthall", settings[ALL])):
        apply(ctx, setting)
        ms = np.zeros((a.steps, 5), np.float32)
        for i in range(a.steps):
            ctx.process_depth_frames_dev(b["match_offsets"], n_models, *[dev[k2].data_ptr() for k2 in keys], W, H, params=P, times=ms[i])
        step_ms[k] = dict(zip(("cluster", "pose", "filter", "pose2", "filter2"), np.median(ms, 0).astype(float).tolist()))
    apply(ctx, {})
    ctx.close()

    # ---- queries: features in, objects out on the 1 M-row database
    db = synth.make_db(a.models, a.rows_per_model)
    qb = synth.make_adaptive_frames(db, a.frames, n_features=a.features, empty=(), far=(), dimensions=capi.ADAPTIVE_DEFAULTS[4:])
    qc = capi.Context(0)
    qc.set_stream(stream.cuda_stream)
    qc.db_upload(db["desc"], db["xyz"], db["model_of_row"], a.models)
    qc.set_cameras(synth.K_DEPTH, synth.CAM_IDENTITY)
    qd = {k: torch.from_numpy(np.ascontiguousarray(qb[k])).cuda() for k in ("desc", "xy", "image", "depth", "fill_distance", "world", "fill")}
    torch.cuda.synchronize()
    qH, qW = qb["depth"].shape[1:]
    offs = np.concatenate([[0], np.cumsum(db["n_pts"])]).astype(np.int32)
    qsettings = {n: {s: (SETTING[s],) + t for s, t in draw_test_points(offs, db["xyz"], n).items()} for n in (40, ALL)}
    qcurrent = {}

    def qarm(setting):
        def run():
            if qcurrent.get("s") is not setting:
                apply(qc, setting)
                qcurrent["s"] = setting
            return qc.process_depth_queries_dev(qd["desc"].data_ptr(), qd["xy"].data_ptr(), qd["image"].data_ptr(), qd["world"].data_ptr(),
                                                qd["fill"].data_ptr(), qb["frame_offsets"], qd["depth"].data_ptr(), qd["fill_distance"].data_ptr(),
                                                qW, qH, qb["curves"])
        return run

    query_arms = dict(plain=qarm({}), depth40=qarm(qsettings[40]), depthall=qarm(qsettings[ALL]))
    qobjects = {k: int(sum(len(g["model"]) for g in fn())) for k, fn in query_arms.items()}
    t_queries = timed(query_arms, stream, a.steps, a.rounds, a.warmup)
    qc.close()

    med = lambda rounds: float(np.median(rounds))
    rec = dict(bench="moped3d chain with FILTER_PROJECTION_DEPTH on FILTER and FILTER2 (mc_set_depth_filter)", gpu=gpu, steps=a.steps,
               rounds=a.rounds, warmup=a.warmup, setting=dict(filter=SETTING[0], filter2=SETTING[1]),
               frames=dict(workload=f"{a.frames} make_depth_frame frames, {n_models} models", objects=objects,
                           ms_per_batch_median={k: med(v) for k, v in t_frames.items()},
                           ms_per_batch_round_medians={k: v for k, v in t_frames.items()}, step_ms_median_one_lane=step_ms),
               queries=dict(workload=f"{a.frames} x {a.features} features, {len(db['desc'])} rows, {a.models} models", objects=qobjects,
                            ms_per_batch_median={k: med(v) for k, v in t_queries.items()},
                            ms_per_batch_round_medians={k: v for k, v in t_queries.items()},
                            stages="not measured"),
               note="CUDA events on the context's stream around each call (the call ends in a device synchronisation); arms alternate round "
                    "by round; depth arms equal the stage-by-stage route bit for bit on the frames workload")
    line = json.dumps(rec)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "a") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
