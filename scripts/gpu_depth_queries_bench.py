"""moped3d from features to objects on a frame batch (MATCH -> DEPTHPROP's depth data per match -> CLUSTER..FILTER2), three ways:
  (a) the three-step composition: mc_match_adaptive_frames_dev, a torch gather of the per-feature world point and fill distance through
      match_feature, a synchronisation, mc_process_depth_frames_dev
  (b) mc_process_depth_queries_dev: one call, arrays on the device
  (c) mc_process_depth_queries: one call, host arrays (queries, per-feature depth data and planes uploaded, objects copied back)
Workload: a 1000-model, 1 M-row synthetic database and 64 frames x 2000 features (synth.make_adaptive_frames with moped3d's
DimensionPeak / DimensionFade of 150 / 50 px), default moped3d chain parameters. The arms are timed in alternating rounds (`--rounds`
rounds of `--steps` steps per arm after `--warmup` calls each), each step a host clock around a call that ends in a device
synchronisation; the spread between rounds of the same arm is the run-to-run noise the arms are compared against. Also records the
device time of MATCH and of the chain from (b)'s stage_ms. Asserts that the three arms return identical objects on the timed batch.
Records the card's name, power limit and max SM clock; appends one JSON line to --out.

    python scripts/gpu_depth_queries_bench.py [--out profiles/depth_queries_bench.jsonl] [--steps 20] [--rounds 3] [--warmup 3]
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "depth_queries_bench.jsonl"))
    ap.add_argument("--models", type=int, default=1000)
    ap.add_argument("--rows-per-model", type=int, default=1000)
    ap.add_argument("--frames", type=int, default=64)
    ap.add_argument("--features", type=int, default=2000)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()[0]
    db = synth.make_db(a.models, a.rows_per_model)
    b = synth.make_adaptive_frames(db, a.frames, n_features=a.features, empty=(), far=(), dimensions=capi.ADAPTIVE_DEFAULTS[4:])
    fo, curves = b["frame_offsets"], b["curves"]
    Q = int(fo[-1])
    H, W = b["depth"].shape[1:]
    ctx = capi.Context(0)
    ctx.db_upload(db["desc"], db["xyz"], db["model_of_row"], a.models)
    ctx.set_cameras(synth.K_DEPTH, synth.CAM_IDENTITY)
    dev = {k: torch.from_numpy(np.ascontiguousarray(b[k])).cuda() for k in ("desc", "xy", "image", "depth", "fill_distance", "world", "fill")}
    o = dict(feat=torch.zeros(Q, dtype=torch.int32, device="cuda"), img=torch.zeros(Q, dtype=torch.int32, device="cuda"),
             xy=torch.zeros((Q, 2), dtype=torch.float32, device="cuda"), xyz=torch.zeros((Q, 3), dtype=torch.float32, device="cuda"))
    torch.cuda.synchronize()

    def composition():
        r = ctx.match_adaptive_frames_dev(dev["desc"].data_ptr(), dev["xy"].data_ptr(), dev["image"].data_ptr(), fo, dev["depth"].data_ptr(),
                                          dev["fill_distance"].data_ptr(), W, H, curves, o["feat"].data_ptr(), o["img"].data_ptr(),
                                          o["xy"].data_ptr(), o["xyz"].data_ptr())
        feat = o["feat"].long()
        world, fill = dev["world"][feat], dev["fill"][feat]
        torch.cuda.synchronize()
        return ctx.process_depth_frames_dev(r["match_offsets"], a.models, o["img"].data_ptr(), o["xy"].data_ptr(), o["xyz"].data_ptr(),
                                            world.data_ptr(), fill.data_ptr(), dev["depth"].data_ptr(), dev["fill_distance"].data_ptr(), W, H)

    def one_call_dev(times=None):
        return ctx.process_depth_queries_dev(dev["desc"].data_ptr(), dev["xy"].data_ptr(), dev["image"].data_ptr(), dev["world"].data_ptr(),
                                             dev["fill"].data_ptr(), fo, dev["depth"].data_ptr(), dev["fill_distance"].data_ptr(), W, H, curves,
                                             times=times)

    def one_call_host():
        return ctx.process_depth_queries(b["desc"], b["xy"], b["image"], b["world"], b["fill"], fo, b["depth"], b["fill_distance"], curves)

    arms = dict(a_composition=composition, b_queries_dev=one_call_dev, c_queries_host=one_call_host)
    for fn in arms.values():
        for _ in range(a.warmup):
            fn()
    t = {k: [] for k in arms}
    for _ in range(a.rounds):                       # alternate the arms: drift of the shared host hits all of them alike
        for k, fn in arms.items():
            round_t = []
            for _ in range(a.steps):
                t0 = time.perf_counter()
                fn()
                round_t.append(time.perf_counter() - t0)
            t[k].append(round_t)
    stage = np.zeros((a.steps, 2), np.float32)
    for i in range(a.steps):
        one_call_dev(stage[i])

    # the timed batch: the three arms return identical objects
    ref, got_dev, got_host = composition(), one_call_dev(), one_call_host()
    bits = lambda x: np.ascontiguousarray(x).view(np.uint32)
    for f in range(a.frames):
        for got in (got_dev, got_host):
            assert np.array_equal(got[f]["model"], ref[f]["model"]) and np.array_equal(got[f]["info"], ref[f]["info"]), f
            assert np.array_equal(bits(got[f]["pose"]), bits(ref[f]["pose"])) and np.array_equal(bits(got[f]["score"]), bits(ref[f]["score"])), f
    info = np.stack([x["info"] for x in ref])

    med = lambda x: float(np.median(x)) * 1e3
    rec = dict(bench="moped3d features to objects on a frame batch (MATCH + depth data per match + CLUSTER..FILTER2)", gpu=gpu,
               db_rows=int(len(db["desc"])), models=a.models, frames=a.frames, features_per_frame=a.features, queries=Q,
               accepted_matches=int(info[:, 2].sum()), clusters=int(info[:, 3].sum()), objects=int(info[:, 0].sum()), steps=a.steps,
               rounds=a.rounds, warmup=a.warmup,
               ms_per_batch_median={k: med(sum(v, [])) for k, v in t.items()},
               ms_per_batch_median_per_round={k: [med(r) for r in v] for k, v in t.items()},
               frames_per_s_median={k: a.frames / float(np.median(sum(v, []))) for k, v in t.items()},
               b_stage_ms_median=dict(match=float(np.median(stage[:, 0])), cluster_to_filter2=float(np.median(stage[:, 1]))),
               note="host clock around calls that end in a device synchronisation; arms alternate round by round; identical objects on the "
                    "timed batch")
    line = json.dumps(rec)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "a") as f:
        f.write(line + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
