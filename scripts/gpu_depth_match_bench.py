"""moped3d's MATCH step (MATCH_ADAPTIVE_FLANN_CPU: exact two nearest rows + depth-adaptive ratio test) on a frame batch, four ways:
  (a) mc_match_adaptive once per frame (host arrays, one matching pass, copies and a synchronisation per frame; the host-side
      bucketing of MATCH_ADAPTIVE_CUDA::emit is not included)
  (b) mc_match_adaptive_frames: the batch in one call, host arrays (planes and queries uploaded, match lists copied back)
  (c) mc_match_adaptive_frames_dev: the batch in one call, arrays on the device
  (d) mc_match_dev on the same queries: the matching pass alone (the floor of (c))
Workload: a 1000-model, 1 M-row synthetic database and 64 frames x 2000 features (synth.make_adaptive_frames with moped3d's
DimensionPeak / DimensionFade of 150 / 50 px). Warm-up, then >= `--steps` timed steps per way, each ending in a device synchronisation
(host clock). Asserts that (b), (c) give every frame exactly what (a) plus emit gives, and that (d) finds the same nearest rows.
Records the card's name, power limit and max SM clock; appends one JSON line to --out.

    python scripts/gpu_depth_match_bench.py [--out profiles/depth_match_bench.jsonl] [--steps 20] [--warmup 3]
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

import adaptive_rule as R  # noqa: E402
from moped_b200 import capi, synth  # noqa: E402


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "depth_match_bench.jsonl"))
    ap.add_argument("--models", type=int, default=1000)
    ap.add_argument("--rows-per-model", type=int, default=1000)
    ap.add_argument("--frames", type=int, default=64)
    ap.add_argument("--features", type=int, default=2000)
    ap.add_argument("--steps", type=int, default=20)
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

    def per_frame():
        return [ctx.match_adaptive(b["desc"][fo[f]:fo[f + 1]], b["xy"][fo[f]:fo[f + 1]], b["depth"][f], b["fill_distance"][f], curves)
                for f in range(a.frames)]

    def batch_host():
        return ctx.match_adaptive_frames(b["desc"], b["xy"], b["image"], fo, b["depth"], b["fill_distance"], curves)

    dev = {k: torch.from_numpy(np.ascontiguousarray(b[k])).cuda() for k in ("desc", "xy", "image", "depth", "fill_distance")}
    o = dict(feat=torch.zeros(Q, dtype=torch.int32, device="cuda"), img=torch.zeros(Q, dtype=torch.int32, device="cuda"),
             xy=torch.zeros((Q, 2), dtype=torch.float32, device="cuda"), xyz=torch.zeros((Q, 3), dtype=torch.float32, device="cuda"),
             nn_row=torch.zeros((Q, 2), dtype=torch.int32, device="cuda"), nn_dist=torch.zeros((Q, 2), dtype=torch.float32, device="cuda"),
             acc=torch.zeros(Q, dtype=torch.uint8, device="cuda"))
    torch.cuda.synchronize()

    def batch_dev():
        return ctx.match_adaptive_frames_dev(dev["desc"].data_ptr(), dev["xy"].data_ptr(), dev["image"].data_ptr(), fo, dev["depth"].data_ptr(),
                                             dev["fill_distance"].data_ptr(), W, H, curves, o["feat"].data_ptr(), o["img"].data_ptr(),
                                             o["xy"].data_ptr(), o["xyz"].data_ptr(), o["nn_row"].data_ptr(), o["nn_dist"].data_ptr(),
                                             o["acc"].data_ptr())

    f_row = torch.zeros((Q, 2), dtype=torch.int32, device="cuda")
    f_dist = torch.zeros((Q, 2), dtype=torch.float32, device="cuda")
    f_acc = torch.zeros(Q, dtype=torch.uint8, device="cuda")

    def floor():
        ctx.match_dev(dev["desc"].data_ptr(), Q, 1.0, capi.MATCH_TENSOR, f_row.data_ptr(), f_dist.data_ptr(), f_acc.data_ptr())
        ctx.synchronize()

    t_a = timed(per_frame, a.warmup, a.steps)
    t_b = timed(batch_host, a.warmup, a.steps)
    t_c = timed(batch_dev, a.warmup, a.steps)
    t_d = timed(floor, a.warmup, a.steps)

    # the timed batch: every frame of (b) and (c) equals (a) + emit; (d) finds the same rows
    singles, host, rdev = per_frame(), batch_host(), batch_dev()
    d_arr = dict(match_feature=o["feat"].cpu().numpy(), match_image=o["img"].cpu().numpy(), match_xy=o["xy"].cpu().numpy(),
                 match_xyz=o["xyz"].cpu().numpy(), nn_row=o["nn_row"].cpu().numpy(), accepted=o["acc"].cpu().numpy().astype(bool),
                 match_offsets=rdev["match_offsets"])
    floor()
    assert np.array_equal(f_row.cpu().numpy(), host["nn_row"])
    n_matches = 0
    for f in range(a.frames):
        lo, hi = int(fo[f]), int(fo[f + 1])
        nn_row, _, acc = singles[f]
        e = R.emit(nn_row, acc, b["xy"][lo:hi], b["image"][lo:hi], db["model_of_row"], db["xyz"], len(curves), base=lo)
        n = int(e["offsets"][-1] - lo)
        n_matches += n
        for out in (host, d_arr):
            assert np.array_equal(out["match_offsets"][f], e["offsets"]), f
            assert np.array_equal(out["nn_row"][lo:hi], nn_row) and np.array_equal(out["accepted"][lo:hi], acc), f
            for k, kk in (("match_feature", "feature"), ("match_image", "image"), ("match_xy", "xy"), ("match_xyz", "xyz")):
                assert np.array_equal(out[k][lo:lo + n], e[kk]), (f, k)
    ms = lambda t: dict(median=float(np.median(t)) * 1e3, mean=float(np.mean(t)) * 1e3, min=float(np.min(t)) * 1e3, max=float(np.max(t)) * 1e3)
    fps = lambda t: a.frames / float(np.median(t))
    rec = dict(bench="moped3d MATCH (depth-adaptive) on a frame batch", gpu=gpu, db_rows=int(len(db["desc"])), models=a.models, frames=a.frames,
               features_per_frame=a.features, queries=Q, accepted_matches=n_matches, steps=a.steps, warmup=a.warmup,
               ms_per_batch=dict(a_per_frame_calls=ms(t_a), b_batch_host=ms(t_b), c_batch_dev=ms(t_c), d_match_dev_floor=ms(t_d)),
               frames_per_s_median=dict(a_per_frame_calls=fps(t_a), b_batch_host=fps(t_b), c_batch_dev=fps(t_c), d_match_dev_floor=fps(t_d)),
               note="host clock around calls that end in a device synchronisation; (b) and (c) equal (a) + emit frame by frame on the timed batch")
    line = json.dumps(rec)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "a") as f:
        f.write(line + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
