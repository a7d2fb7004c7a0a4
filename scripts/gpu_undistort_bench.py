"""What UNDISTORTED_IMAGE costs on the device, and the host work it replaces, on 64-frame batches of 640x480 gray images:
  kernel   device time of one mc_undistort_dev call (one k_undistort launch) on a 64 x 640x480 batch: CUDA events around each call on
           the context's stream, after warm-up; the calls cycle through 8 input and 8 output batches (315 MB, more than the 126 MB L2),
           so the images come from HBM. Algorithmic bytes: the images read and written once plus the 8-byte-per-pixel table once.
  images   mc_process_images per 64-frame batch of the bench's `images` workload (a 640x480 frame of the reference's timing.bag, shifted
           per slot, 3 planar models) without and with a camera-0 table (a mild barrel lens), same pixels, the two arms alternating
           round by round; host clock around each call (it ends in a device synchronisation)
  cv2      cv2.remap (bilinear, constant border 0) of the same 64 frames on this host's CPU, at 1 thread and at all threads
Records the card's name, power limit and max SM clock; appends one JSON line to --out.

    python scripts/gpu_undistort_bench.py [--out profiles/undistort_bench.jsonl] [--reps 200] [--steps 10] [--rounds 5]
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

from moped_b200 import capi  # noqa: E402

KC = (-0.2, 0.05, 0.001, -0.0005)
HBM_BYTES_PER_S = 7.7e12          # HGX B200 data sheet, one GPU


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "undistort_bench.jsonl"))
    ap.add_argument("--frames", type=int, default=64)
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("gpu_undistort_bench.py: no CUDA device")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()[0]
    g = dict(np.load(os.path.join(ROOT, "tests", "golden", "real_images.npz")))
    im = np.load(os.path.join(ROOT, "tests", "golden", "sift_golden.npz"))["bag4_full_double/image"]
    frames = np.stack([np.roll(im, (i % 8) - 4, axis=1) for i in range(a.frames)])
    B, H, W = frames.shape
    K = g["K"][0]

    ctx = capi.Context(0)
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)
    ctx.set_undistortion(0, K, KC, H, W)

    # kernel: 8 input / 8 output batches in rotation
    n_buf = 8
    d_in = [torch.from_numpy(np.roll(frames, k, axis=2).copy()).cuda() for k in range(n_buf)]
    d_out = [torch.empty_like(d_in[0]) for _ in range(n_buf)]
    torch.cuda.synchronize()
    for k in range(n_buf):
        ctx.undistort_dev(d_in[k].data_ptr(), B, H, W, d_out[k].data_ptr())
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * a.reps)]
    for r in range(a.reps):
        ev[2 * r].record(stream)
        ctx.undistort_dev(d_in[r % n_buf].data_ptr(), B, H, W, d_out[r % n_buf].data_ptr())
        ev[2 * r + 1].record(stream)
    stream.synchronize()
    kms = np.array([ev[2 * r].elapsed_time(ev[2 * r + 1]) for r in range(a.reps)])
    nbytes = 2 * B * H * W + 8 * H * W
    kernel = {"ms_median": float(np.median(kms)), "ms_min": float(kms.min()), "ms_max": float(kms.max()), "reps": a.reps,
              "algorithmic_bytes": nbytes, "gb_per_s_median": nbytes / (np.median(kms) * 1e-3) / 1e9,
              "share_of_7.7TB/s": nbytes / (np.median(kms) * 1e-3) / HBM_BYTES_PER_S}

    # mc_process_images without / with the table, alternating
    ctx.db_upload(g["db_desc"], g["db_xyz"], g["model_of_row"], len(g["n_pts"]))
    ctx.set_cameras(g["K"], g["cam_pose"])
    ctx.set_tuning(8, 8, 1)
    h_frames = torch.from_numpy(frames).pin_memory().numpy()

    def use_table(k):            # outside the timed window: the table is built once per camera, not per batch
        if k == "undistorted":
            ctx.set_undistortion(0, K, KC, H, W)
        else:
            ctx.set_undistortion(0, None, None, 0, 0)

    times = {"plain": [], "undistorted": []}
    objects = {}
    for k in times:
        use_table(k)
        for _ in range(a.warmup):
            ctx.process_images(h_frames, True, max_keypoints=2048, max_objects=16)
    for _ in range(a.rounds):
        for k in times:
            use_table(k)
            ms = []
            for _ in range(a.steps):
                t0 = time.perf_counter()
                out = ctx.process_images(h_frames, True, max_keypoints=2048, max_objects=16)
                ms.append((time.perf_counter() - t0) * 1e3)
            objects[k] = int(sum(len(o["model"]) for o in out))
            times[k].append(float(np.median(ms)))
    images = {k: {"round_medians_ms": v, "median_ms": float(np.median(v)), "min_ms": float(min(v)), "max_ms": float(max(v)),
                  "objects_per_batch": objects[k]} for k, v in times.items()}

    # cv2.remap on this host's CPU
    cpu = {"cores": os.cpu_count()}
    try:
        import cv2
        from oracle import undistort as U
        mx, my = U.undistort_map(K, KC, H, W)
        for threads in (1, os.cpu_count()):
            cv2.setNumThreads(threads)
            cv2.remap(frames[0], mx, my, cv2.INTER_LINEAR, borderMode=cv2.BORDER_CONSTANT, borderValue=0)
            best = []
            for _ in range(5):
                t0 = time.perf_counter()
                for f in frames:
                    cv2.remap(f, mx, my, cv2.INTER_LINEAR, borderMode=cv2.BORDER_CONSTANT, borderValue=0)
                best.append((time.perf_counter() - t0) * 1e3)
            cpu[f"cv2_remap_ms_per_batch_{threads}_threads"] = float(np.median(best))
        cpu["cv2_version"] = cv2.__version__
    except ImportError:
        cpu["cv2"] = "not importable on this host: not measured"

    rec = {"bench": "undistort", "gpu": gpu, "frames": B, "image": f"{W}x{H} u8", "kc": KC, "kernel": kernel, "process_images": images,
           "cpu_remap": cpu}
    print(json.dumps(rec))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "a") as f:
        f.write(json.dumps(rec) + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
