"""Camera-rig frames from pixels to objects: mc_process_rig_images against the route a host assembles without it, on batches of 64 frames
of C = 1, 2 and 4 cameras at 640x480 (a frame of the reference's timing.bag, shifted per image), without and with an undistortion table on
every camera, against two databases:
  planar   the 3 planar models / 1275 descriptors of tests/golden/real_images.npz (the real frames show them)
  synth1M  synth.make_db(1000, 1000): 1 M rows, 1000 models (MATCH at the size of bench.py's flagship workload)
Arms, alternating step by step after warm-up; host clock around each call, which ends in a device synchronisation:
  rig      mc_process_rig_images on pinned host images
  host     cv2.remap per image on the host when cv2 imports (mc_undistort per camera otherwise), one mc_sift_extract for the batch with
           every descriptor copied to the host, each frame's keypoints concatenated in camera order with q_image = camera and normalised
           like MATCH, mc_process_frames
Per configuration: median ms per batch, frames/s and images/s of both arms, the rig call's stage_ms (FEAT incl. upload and remap, MATCH,
CLUSTER..FILTER2; medians), and with tables the remap kernel's device time in the rig call (torch.profiler, CUDA activities, in a pass of
its own after the timed steps) with its algorithmic bytes: per pixel 1 read, 1 written and 8 of table.
Records the card's name, power limit and max SM clock; appends one JSON line per configuration to --out.

    python scripts/gpu_rig_images_bench.py [--out profiles/rig_images_bench.jsonl] [--steps 20] [--warmup 3]
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

LENSES = [(-0.2, 0.05, 0.001, -0.0005), (0.1, -0.02, 0.0, 0.0005, 0.01), (-0.05, 0.0, -0.001, 0.0), (-0.1, 0.01, 0.0005, 0.0005)]
HBM_BYTES_PER_S = 7.7e12          # HGX B200 data sheet, one GPU
MAX_KP, MAX_OBJ = 2048, 16


def normalise(desc):
    ss = np.zeros(len(desc), np.float32)
    for k in range(128):
        ss = ss + desc[:, k] * desc[:, k]                                  # sequential fp32 sum like MATCH_CUDA::normalise
    return desc * (1.0 / np.sqrt(ss).astype(np.float64)).astype(np.float32)[:, None]


def kernel_ms(prof, name):
    """summed device time (ms) and count of the kernels whose name contains `name`"""
    tot, n = 0.0, 0
    for e in prof.key_averages():
        if name in e.key:
            tot += getattr(e, "device_time_total", 0.0) / 1e3
            n += e.count
    return tot, n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "rig_images_bench.jsonl"))
    ap.add_argument("--frames", type=int, default=64)
    ap.add_argument("--cameras", default="1,2,4")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--profile-reps", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("gpu_rig_images_bench.py: no CUDA device")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()[0]
    try:
        import cv2
        from oracle import undistort as U
        host_remap = f"cv2.remap {cv2.__version__}, {cv2.getNumThreads()} threads"
    except ImportError:
        cv2 = None
        host_remap = "mc_undistort per camera (cv2 not importable)"
    g = dict(np.load(os.path.join(ROOT, "tests", "golden", "real_images.npz")))
    im = np.load(os.path.join(ROOT, "tests", "golden", "sift_golden.npz"))["bag4_full_double/image"]
    H, W = im.shape
    K = g["K"][0]
    big = synth.make_db(1000, 1000)
    big_desc = (big["desc"] / np.linalg.norm(big["desc"], axis=1, keepdims=True)).astype(np.float32)
    dbs = {"planar": (g["db_desc"], g["db_xyz"], g["model_of_row"], len(g["n_pts"])),
           "synth1M": (big_desc, big["xyz"], big["model_of_row"], 1000)}

    ctx = capi.Context(0)
    ctx.set_tuning(8, 8, 1)
    B = a.frames
    for db_name, db in dbs.items():
        ctx.db_upload(*db)
        for Cn in [int(c) for c in a.cameras.split(",")]:
            ctx.set_cameras(np.tile(K, (Cn, 1)), np.tile(g["cam_pose"][0], (Cn, 1)))
            shifts = (np.arange(B * Cn).reshape(B, Cn) % 8) - 4
            frames = np.stack([np.stack([np.roll(im, s, axis=1) for s in row]) for row in shifts])     # [B, C, H, W]
            h_frames = torch.from_numpy(frames).pin_memory().numpy()
            for tables in (False, True):
                for c in range(Cn):
                    if tables:
                        ctx.set_undistortion(c, K, LENSES[c], H, W)
                    else:
                        ctx.set_undistortion(c, None, None, 0, 0)
                maps = [U.undistort_map(K, LENSES[c], H, W) for c in range(Cn)] if (tables and cv2 is not None) else None

                n_kp = np.zeros(B * Cn, np.int32)           # the host route's feature buffers, allocated once like a host would
                kp_xy = np.zeros((B * Cn, MAX_KP, 2), np.float32)
                kp_desc = np.zeros((B * Cn, MAX_KP, 128), np.float32)

                def rig():
                    return ctx.process_rig_images(h_frames, True, max_keypoints=MAX_KP, max_objects=MAX_OBJ, want_times=True)

                def host():
                    per_cam = []
                    for c in range(Cn):
                        ims = np.ascontiguousarray(frames[:, c])
                        if tables and cv2 is not None:
                            ims = np.stack([cv2.remap(x, maps[c][0], maps[c][1], cv2.INTER_LINEAR, borderMode=cv2.BORDER_CONSTANT, borderValue=0)
                                            for x in ims])
                        elif tables:
                            ims = ctx.undistort(ims, c)
                        per_cam.append(ims)
                    batch = np.ascontiguousarray(np.stack(per_cam, axis=1).reshape(-1))
                    ctx._check(ctx.L.mc_sift_extract(ctx.h, batch, B * Cn, H, W, 1, MAX_KP, n_kp, kp_xy.reshape(-1), None, kp_desc.reshape(-1)),
                               "mc_sift_extract")
                    q = normalise(np.concatenate([kp_desc[i, :n] for i, n in enumerate(n_kp)]))
                    xy = np.concatenate([kp_xy[i, :n] for i, n in enumerate(n_kp)])
                    img = np.repeat(np.arange(B * Cn, dtype=np.int32) % Cn, n_kp)
                    fo = np.concatenate([[0], np.cumsum(n_kp.reshape(B, Cn).sum(axis=1))]).astype(np.int32)
                    return ctx.process_frames(q, xy, img, fo, max_objects=MAX_OBJ)

                for _ in range(a.warmup):
                    rig(), host()
                ms = {"rig": [], "host": []}
                stage = []
                same = True
                for _ in range(a.steps):
                    t0 = time.perf_counter()
                    out = rig()
                    ms["rig"].append((time.perf_counter() - t0) * 1e3)
                    stage.append(out[0]["stage_ms"].copy())
                    t0 = time.perf_counter()
                    ref = host()
                    ms["host"].append((time.perf_counter() - t0) * 1e3)
                    same &= all(np.array_equal(o["model"], r["model"]) for o, r in zip(out, ref))
                rec = {"bench": "rig_images", "gpu": gpu, "db": db_name, "cameras": Cn, "frames": B, "images": B * Cn, "image": f"{W}x{H} u8",
                       "tables": tables, "steps": a.steps, "host_remap": host_remap if tables else None,
                       "objects_per_batch": int(sum(len(o["model"]) for o in out)),
                       "features_per_batch": int(sum(int(o["n_features"].sum()) for o in out)),
                       "host_route_same_models": bool(same)}
                for k, v in ms.items():
                    med = float(np.median(v))
                    rec[k] = {"median_ms": med, "min_ms": float(min(v)), "max_ms": float(max(v)), "frames_per_s": B / med * 1e3,
                              "images_per_s": B * Cn / med * 1e3}
                st = np.median(np.stack(stage), axis=0)
                rec["rig_stage_ms"] = {"feat": float(st[0]), "match": float(st[1]), "cluster_to_filter2": float(st[2])}
                if tables:
                    from torch.profiler import ProfilerActivity, profile
                    with profile(activities=[ProfilerActivity.CUDA]) as prof:
                        for _ in range(a.profile_reps):
                            rig()
                    tot, n = kernel_ms(prof, "k_undistort")
                    nbytes = 10 * B * Cn * H * W
                    kms = tot / max(n, 1)
                    rec["remap_kernel"] = {"launches": n, "calls": a.profile_reps, "ms_mean": kms, "algorithmic_bytes": nbytes,
                                           "gb_per_s": nbytes / (kms * 1e-3) / 1e9 if kms > 0 else None,
                                           "share_of_7.7TB/s": nbytes / (kms * 1e-3) / HBM_BYTES_PER_S if kms > 0 else None}
                    for c in range(Cn):
                        ctx.set_undistortion(c, None, None, 0, 0)
                print(json.dumps(rec), flush=True)
                os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
                with open(a.out, "a") as f:
                    f.write(json.dumps(rec) + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
