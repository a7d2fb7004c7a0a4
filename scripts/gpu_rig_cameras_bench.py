"""Camera rigs with cameras of different image sizes: mc_process_rig_cameras (host images) and mc_process_rig_cameras_dev (images already
in HBM) against the route a host assembles without them, on batches of 64 frames of two rigs,
  2cam   {640x480, 1280x720}
  3cam   {640x480, 640x480, 1280x720}
without and with an undistortion table on every camera, against two databases:
  planar   the 3 planar models / 1275 descriptors of tests/golden/real_images.npz (the real frames show them)
  synth1M  synth.make_db(1000, 1000): 1 M rows, 1000 models (MATCH at the size of bench.py's flagship workload)
The 640x480 images are a frame of the reference's timing.bag, shifted per image; the 1280x720 images are its rows 60..419 upsampled 2x
(nearest), with K scaled to match.
Arms, alternating step by step after warm-up; host clock around each call, which ends in a device synchronisation:
  host        mc_process_rig_cameras on pinned host images, one buffer per camera
  dev         mc_process_rig_cameras_dev on the same images, uploaded once before the timed steps
  host_route  per camera: mc_undistort where it has a table (upload, the remap kernel, download), mc_sift_extract with every descriptor
              copied to the host; each frame's keypoints concatenated in camera order with q_image = camera and normalised like MATCH;
              mc_process_frames
  rig_images  mc_process_rig_images on a rig of as many 640x480 cameras (one size: no merge), for reference
Per configuration: median ms per batch, frames/s and images/s of every arm, the host entry's stage_ms (FEAT incl. upload, remap and merge,
MATCH, CLUSTER..FILTER2; medians). A separate profiled pass (torch.profiler, CUDA activities, after the timed steps) gives the device time
of the two merge kernels, k_rig_merge_scan and k_rig_merge_interleave, with the interleave's algorithmic bytes: per keypoint 512 + 8 bytes
read and written and 4 written (imageIdx).
Records the card's name, power limit and max SM clock; appends one JSON line per configuration to --out.

    python scripts/gpu_rig_cameras_bench.py [--out profiles/rig_cameras_bench.jsonl] [--steps 10] [--warmup 2]
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

LENSES = [(-0.2, 0.05, 0.001, -0.0005), (0.1, -0.02, 0.0, 0.0005, 0.01), (-0.05, 0.0, -0.001, 0.0)]
HBM_BYTES_PER_S = 7.7e12          # HGX B200 data sheet, one GPU
MAX_KP, MAX_OBJ = 2048, 16
RIGS = {"2cam": ("vga", "hd"), "3cam": ("vga", "vga", "hd")}


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
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "rig_cameras_bench.jsonl"))
    ap.add_argument("--frames", type=int, default=64)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--profile-reps", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("gpu_rig_cameras_bench.py: no CUDA device")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()[0]
    g = dict(np.load(os.path.join(ROOT, "tests", "golden", "real_images.npz")))
    im = np.load(os.path.join(ROOT, "tests", "golden", "sift_golden.npz"))["bag4_full_double/image"]
    K = g["K"][0].astype(np.float32)
    fx, fy, cx, cy = (float(v) for v in K)
    kinds = {"vga": (lambda x: x, K),
             "hd": (lambda x: x[60:420].repeat(2, axis=0).repeat(2, axis=1), np.float32([2 * fx, 2 * fy, 2 * cx + 0.5, 2 * (cy - 60) + 0.5]))}
    big = synth.make_db(1000, 1000)
    big_desc = (big["desc"] / np.linalg.norm(big["desc"], axis=1, keepdims=True)).astype(np.float32)
    dbs = {"planar": (g["db_desc"], g["db_xyz"], g["model_of_row"], len(g["n_pts"])),
           "synth1M": (big_desc, big["xyz"], big["model_of_row"], 1000)}

    ctx = capi.Context(0)
    ref = capi.Context(0)             # the rig_images arm's own context: its 640x480 tables would clash with the mixed rig's
    for c_ in (ctx, ref):
        c_.set_tuning(8, 8, 1)
    B = a.frames
    for db_name, db in dbs.items():
        ctx.db_upload(*db)
        ref.db_upload(*db)
        for rig_name, rig in RIGS.items():
            Cn = len(rig)
            ctx.set_cameras(np.stack([kinds[k][1] for k in rig]), np.tile(g["cam_pose"][0], (Cn, 1)))
            ref.set_cameras(np.tile(K, (Cn, 1)), np.tile(g["cam_pose"][0], (Cn, 1)))
            shifts = (np.arange(B * Cn).reshape(B, Cn) % 8) - 4
            ims = [torch.from_numpy(np.ascontiguousarray(np.stack([kinds[k][0](np.roll(im, s, axis=1)) for s in shifts[:, c]]))).pin_memory().numpy()
                   for c, k in enumerate(rig)]
            sizes = [x.shape[1:] for x in ims]
            dev = [torch.from_numpy(x).cuda() for x in ims]
            torch.cuda.synchronize()
            vga = torch.from_numpy(np.ascontiguousarray(np.stack([np.stack([np.roll(im, s, axis=1) for s in row]) for row in shifts]))).pin_memory().numpy()
            for tables in (False, True):
                for c, k in enumerate(rig):
                    if tables:
                        ctx.set_undistortion(c, kinds[k][1], LENSES[c], *sizes[c])
                        ref.set_undistortion(c, K, LENSES[c], 480, 640)
                    else:
                        ctx.set_undistortion(c, None, None, 0, 0)
                        ref.set_undistortion(c, None, None, 0, 0)
                buffers = [(np.zeros(B, np.int32), np.zeros((B, MAX_KP, 2), np.float32), np.zeros((B, MAX_KP, 128), np.float32)) for _ in rig]

                def host():
                    return ctx.process_rig_cameras(ims, True, max_keypoints=MAX_KP, max_objects=MAX_OBJ, want_times=True)

                def dev_entry():
                    return ctx.process_rig_cameras_dev([t.data_ptr() for t in dev], [h * w for h, w in sizes], sizes, B, True, max_keypoints=MAX_KP,
                                                       max_objects=MAX_OBJ)

                def host_route():
                    for c in range(Cn):
                        x = ctx.undistort(ims[c], c) if tables else ims[c]
                        n, xy, desc = buffers[c]
                        H, W = sizes[c]
                        ctx._check(ctx.L.mc_sift_extract(ctx.h, np.ascontiguousarray(x).reshape(-1), B, H, W, 1, MAX_KP, n, xy.reshape(-1), None,
                                                         desc.reshape(-1)), "mc_sift_extract")
                    order = [(f, c) for f in range(B) for c in range(Cn)]
                    q = normalise(np.concatenate([buffers[c][2][f, :buffers[c][0][f]] for f, c in order]))
                    xy = np.concatenate([buffers[c][1][f, :buffers[c][0][f]] for f, c in order])
                    img = np.concatenate([np.full(buffers[c][0][f], c, np.int32) for f, c in order])
                    per_frame = np.stack([buffers[c][0] for c in range(Cn)], axis=1).sum(axis=1)
                    fo = np.concatenate([[0], np.cumsum(per_frame)]).astype(np.int32)
                    return ctx.process_frames(q, xy, img, fo, max_objects=MAX_OBJ)

                def rig_images():
                    return ref.process_rig_images(vga, True, max_keypoints=MAX_KP, max_objects=MAX_OBJ)

                arms = {"host": host, "dev": dev_entry, "host_route": host_route, "rig_images": rig_images}
                for _ in range(a.warmup):
                    for fn in arms.values():
                        fn()
                ms = {k: [] for k in arms}
                stage = []
                same = True
                for _ in range(a.steps):
                    outs = {}
                    for k, fn in arms.items():
                        t0 = time.perf_counter()
                        outs[k] = fn()
                        ms[k].append((time.perf_counter() - t0) * 1e3)
                    stage.append(outs["host"][0]["stage_ms"].copy())
                    for k in ("dev", "host_route"):
                        same &= all(np.array_equal(o["model"], r["model"]) and np.array_equal(o["pose"], r["pose"]) for o, r in zip(outs["host"], outs[k]))
                out = outs["host"]
                n_feat = int(sum(int(o["n_features"].sum()) for o in out))
                rec = {"bench": "rig_cameras", "gpu": gpu, "db": db_name, "rig": rig_name, "sizes": [f"{w}x{h}" for h, w in sizes], "frames": B,
                       "images": B * Cn, "tables": tables, "steps": a.steps, "objects_per_batch": int(sum(len(o["model"]) for o in out)),
                       "features_per_batch": n_feat, "host_dev_host_route_same_objects": bool(same),
                       "rig_images_reference": f"{Cn} x 640x480"}
                for k, v in ms.items():
                    med = float(np.median(v))
                    rec[k] = {"median_ms": med, "min_ms": float(min(v)), "max_ms": float(max(v)), "frames_per_s": B / med * 1e3,
                              "images_per_s": B * Cn / med * 1e3}
                st = np.median(np.stack(stage), axis=0)
                rec["host_stage_ms"] = {"feat": float(st[0]), "match": float(st[1]), "cluster_to_filter2": float(st[2])}
                from torch.profiler import ProfilerActivity, profile
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    for _ in range(a.profile_reps):
                        host()
                nbytes = n_feat * (2 * (512 + 8) + 4)
                for name in ("k_rig_merge_scan", "k_rig_merge_interleave"):
                    tot, n = kernel_ms(prof, name)
                    kms = tot / max(n, 1)
                    rec[name] = {"launches": n, "calls": a.profile_reps, "ms_mean": kms}
                    if name == "k_rig_merge_interleave":
                        rec[name].update(algorithmic_bytes=nbytes, gb_per_s=nbytes / (kms * 1e-3) / 1e9 if kms > 0 else None,
                                         share_of_7_7TB_s=nbytes / (kms * 1e-3) / HBM_BYTES_PER_S if kms > 0 else None)
                print(json.dumps(rec), flush=True)
                os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
                with open(a.out, "a") as f:
                    f.write(json.dumps(rec) + "\n")
            for c in range(Cn):
                ctx.set_undistortion(c, None, None, 0, 0)
                ref.set_undistortion(c, None, None, 0, 0)
    ctx.close()
    ref.close()


if __name__ == "__main__":
    main()
