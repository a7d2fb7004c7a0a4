#!/usr/bin/env python
"""bench.py — frames/s of MOPED's recognition core (MATCH..FILTER2) on the BASELINE.json workload.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json metric): synthetic 1000-object database (~1M 128-d descriptors), 640x480 frames of
2000 features, the reference's default stage parameters (config.hpp:83-120). A step = one batch of --frames
independent frames (a camera stream; BASELINE.json configs[4] batches frames the same way) through
MATCH -> CLUSTER -> POSE -> FILTER -> POSE2 -> FILTER2; value = frames/s. The latency of a single frame
(mc_process_frame) is reported beside it as `single_frame`.

ours:       value = frames/s with the features resident in HBM (mc_process_frames_dev); e2e = the same through
            the host-buffer C ABI call mc_process_frames (pinned host -> device copy of the features and
            device -> host read of the objects inside the timed region). N > 1: database sharded by object, every
            rank matches all queries of the batch against its shard, NCCL all-gather of the per-query
            (row, distance) pairs, merge, then rank r runs CLUSTER..FILTER2 for its 1/N of the frames and the
            per-frame results are all-gathered (strong scaling: the job — the batch and the database — is fixed).
reference:  the reference's own CPU stage classes (oracle/_ref, built from /root/reference) on the host
            cores; a step is a bounded sample of the same frame (see `cpu_baseline.sample`).
One JSON line on stdout (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from moped_b200 import synth  # noqa: E402
from moped_b200.sharding import ResultBlock, cluster_partition, frame_range, shard_objects  # noqa: E402

METRIC = "frames_per_s"
UNIT = "frames/s"
L2_BYTES = 126 * 1024 * 1024


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["bf16_tflops"]), float(d["hbm_gbs"]), "measured"
    return 1590.0, 6650.0, "fallback"


def measured_sustained_tflops():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["bf16_tflops_sustained"])
    except Exception:
        return None


def measured_traffic(kernel, **cfg):
    """DRAM bytes per launch of `kernel` from the committed ncu --set full capture of this configuration, or None."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        with open(p) as f:
            for e in json.load(f).get(kernel, []):
                if all(cfg.get(k) == v for k, v in e["when"].items()):
                    return {"bytes": e["dram_bytes_read"] + e["dram_bytes_write"], "source": e["source"]}
    except Exception:
        pass
    return None


def host_norm_rows(x: np.ndarray) -> np.ndarray:
    """Host-side L2 normalisation of descriptors (what the MATCH stage class does before upload,
    MATCH_ANN_CPU.hpp:54-57,94,157)."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    n = np.sqrt((x * x).sum(axis=1, dtype=np.float32)).astype(np.float32)
    return (x * (np.float32(1.0) / n)[:, None]).astype(np.float32)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(mx)) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline
# ------------------------------------------------------------------------------------------------
def reference_pl(frame):
    planted = np.nonzero(frame["src_row"] >= 0)[0]
    dis = np.nonzero(frame["src_row"] < 0)[0][:20]
    return np.sort(np.concatenate([planted, dis]))


def reference_setup(db, n_threads):
    from oracle import ref
    r = ref.Ref(n_threads)
    r.set_models(db["n_pts"], db["xyz"], db["desc"])
    r.set_images(synth.K_DEFAULT, synth.CAM_IDENTITY)
    t0 = time.time()
    r.build_match(5.0, 0.8)          # kd-tree build: excluded from the timing like the GPU database upload
    log(f"[reference] kd-tree build {time.time() - t0:.1f}s")
    return r


def reference_sample_step(r, frame, frac_inv, seed):
    """One bounded sample of a frame: (a) MATCH_ANN_CPU (eps=5, the shipped default) on a uniformly random
    1/frac_inv of the frame's features, time scaled x frac_inv (ANN matching is serial per query,
    MATCH_ANN_CPU.hpp:155-162); (b) CLUSTER..FILTER2 on the matches of the planted features + 20 distractors,
    i.e. on (all but a handful of) the matches the full frame produces.
    Returns (seconds per full frame, per-stage seconds, #objects)."""
    Q = len(frame["desc"])
    rng = np.random.default_rng(seed)
    uni = np.sort(rng.choice(Q, size=max(1, Q // frac_inv), replace=False))
    pl = reference_pl(frame)
    r.clear_frame()
    r.set_features(frame["desc"][uni], frame["xy"][uni], frame["image_idx"][uni])
    t_match = float(Q) / len(uni) * r.run_match(5.0, 0.8)
    r.set_features(frame["desc"][pl], frame["xy"][pl], frame["image_idx"][pl])
    n, times = r.run_pipeline(seed=seed)
    stage = np.array(times)
    stage[0] = t_match
    return float(stage.sum()), stage, n


def run_reference(args, rank, world):
    """--impl reference: the reference's own unmodified CPU stage classes (oracle/_ref) on the configuration of our arm. A timed step
    is ONE FULL frame of the step's batch — all its features through MATCH_ANN_CPU (eps = 5, the shipped default) and the complete
    match set through CLUSTER..FILTER2, per-stage wall clock like moped.cpp:183-191 — i.e. a bounded sample (1 of the --frames
    frames) of the workload, nothing extrapolated inside a frame. Warm-up steps use a quarter of a frame's features (they only
    page the kd-tree in). frames/s = 1 / seconds per frame: the reference processes the frames of a batch one after the other
    (Moped::processImages, moped.cpp:166-194), its stages use every host core through OpenMP."""
    if rank != 0:
        return
    from oracle import ref
    if not ref.available():
        subprocess.call(["make", "-s", "-f", os.path.join(ROOT, "oracle", "Makefile"), "ref"])
    if not ref.available():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libmoped_ref.so missing and /root/reference not present to build it"}))
        return
    cores = os.cpu_count() or 1
    db = synth.make_db(args.objects, args.pts)
    n_fr = min(args.frames, max(1, args.steps))
    frames = [synth.make_frame(db, args.features, n_visible=8, frame_id=i) for i in range(n_fr)]   # frames of our arm's first batch
    r = reference_setup(db, cores)
    for i in range(args.warmup):
        s, _, n = reference_sample_step(r, frames[i % n_fr], 4, seed=3 + i)
        log(f"[reference] warm-up {i}: {s:.2f}s/frame (quarter sample, scaled) objects={n}")
    tot = 0.0
    stages = np.zeros(6)
    n_obj = 0
    for i in range(args.steps):
        fr = frames[i % n_fr]
        r.clear_frame()
        r.set_features(fr["desc"], fr["xy"], fr["image_idx"])
        t0 = time.perf_counter()
        n, st = r.run_pipeline(seed=11 + i)
        s = time.perf_counter() - t0
        tot += s
        stages += np.array(st)
        n_obj += n
        log(f"[reference] step {i}: {s:.2f}s/frame objects={n}")
    sec = tot / args.steps
    sample = (f"per timed step: 1 full frame of the {args.frames}-frame batch ({args.features} features) through MATCH_ANN_CPU(eps=5)..FILTER2, "
              f"OpenMP on {cores} cores; kd-tree build excluded (as the GPU database upload is)")
    out = {"impl": "reference", "metric": METRIC, "value": 1.0 / sec, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": workload_config(args, world), "objects_per_frame": n_obj / args.steps,
           "stage_ms": {k: float(v / args.steps * 1e3) for k, v in zip(["match", "cluster", "pose", "filter", "pose2", "filter2"], stages)},
           "cpu_baseline": {"value": 1.0 / sec, "unit": UNIT, "cores": cores, "kind": "reference", "sample": sample},
           "e2e": {"value": 1.0 / sec, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out))


def init_nccl_quietly(dist, dev):
    """NCCL prints its banner ("NCCL version ...") on STDOUT when the communicator is created (at init with device_id, or lazily at the
    first collective), whatever NCCL_DEBUG_FILE says; rank 0's stdout must carry ONE JSON line. File descriptor 1 points at stderr while
    the process group and its communicator come up (a tiny all-reduce forces the creation), then it is restored."""
    import torch
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    try:
        dist.init_process_group("nccl", device_id=dev)
        t = torch.zeros(1, device=dev)
        dist.all_reduce(t)
        torch.cuda.synchronize(dev)
    finally:
        sys.stdout.flush()
        os.dup2(saved, 1)
        os.close(saved)


def workload_config(args, world):
    """The SAME dict on both arms (the driver compares them): the workload, and how our arm schedules it."""
    img_bytes = ((args.objects * args.pts // world + 127) // 128) * 32768
    return {"workload": f"synthetic {args.objects}-object DB ({args.objects * args.pts} x 128-d SIFT-like descriptors), "
                        f"{args.features} features/frame 640x480, MATCH..FILTER2 with config.hpp defaults; "
                        f"a step = a batch of {args.frames} independent frames",
            "db_objects": args.objects, "db_descriptors": args.objects * args.pts, "features_per_frame": args.features,
            "frames_per_step": args.frames,
            "parallelism": f"db-sharded-by-object x{world}, frames after MATCH partitioned x{world}" if world > 1 else "single-gpu",
            "l2": "db tile image > 2x L2, not flushed" if img_bytes >= 2 * L2_BYTES else "L2 flushed between steps (256 MiB write)",
            "pose_mode": args.pose_mode, "match_coarse_kind": args.coarse_kind, "match_reserve_sms": args.reserve_sms, "batches_pool": 2, "frame_lanes": args.lanes, "batch_graph": args.batch_graph, "ransac_merge_levels": args.merge_levels, "pose_warps_per_task": args.pose_warps, "match_chunks": args.chunks,
            "pipeline": (f"software-pipelined on one context: MATCH of step i+1 (mc_match_dev, coarse kernel on the MATCH partition) runs beside "
                         f"CLUSTER..FILTER2 of step i (mc_process_frames_matched_dev with deferred lane join, lanes on a {args.stage_sms}-SM stage "
                         "partition, CUDA green contexts); every step completes inside the timed region" if args.pipeline else "one mc_process_frames* call per step")}


def resolve_auto(args, world):
    """--pipeline / --stage-sms -1 = by frames per GPU: with few frames per GPU the stage chain is a ~2 ms latency chain that hides
    completely beside the next step's MATCH on a 16-SM partition; with many (64 on one GPU) it is throughput-bound on so few SMs
    and the partition costs MATCH more than it hides (measured: scripts/gpu_overlap_probe.py, profiles/overlap_r2.md)."""
    per_gpu = args.frames // max(1, world)
    if args.pipeline < 0:
        args.pipeline = 1 if per_gpu <= 16 else 0
    if args.stage_sms < 0:
        args.stage_sms = 16 if args.pipeline else 0
    if args.pipeline and args.stage_sms and args.lanes > 16:
        args.lanes = 16            # lane streams + the MATCH streams must stay below the 32 hardware connections (no false dependencies)
    if args.pose_warps <= 0:       # first-round hypotheses per RANSAC task (with levels 1 and 2 merged: 4 -> 2.74 ms, 1 -> 3.95 ms per 64 frames)
        args.pose_warps = 4
    if args.lanes <= 0:            # not pipelined: one lane per frame, all chains of a batch in one CUDA graph ("batch_graph")
        args.lanes = 16 if args.pipeline else min(64, max(1, per_gpu))
    return args


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
DUMP_LIMIT_BYTES = 64 << 20


def dump_frame_results(path, frames, max_objects, seed=0):
    """--dump-outputs: the per-frame results of one step (list of dict(model, pose, score, info) in frame order, as
    mc_process_frames_dev returns them) as .npy files under `path`, one row per frame, objects in the order the call returned them:
    frame_index [F] (frame of the batch), frame_info [F,4] {objects, status, accepted matches, clusters after CLUSTER},
    obj_model [F,MO] (-1 = empty slot), obj_pose [F,MO,7] (qx qy qz qw tx ty tz; 0 in empty slots), obj_score [F,MO].
    A batch larger than DUMP_LIMIT_BYTES keeps a fixed, seeded sample of its frames, so two runs write the same frames."""
    per_frame = 8 * (1 + 4 + max_objects) + 4 * 8 * max_objects
    idx = np.arange(len(frames))
    keep = (DUMP_LIMIT_BYTES - 4096) // per_frame             # 4096: the five .npy headers
    if len(frames) > keep:
        idx = np.sort(np.random.default_rng(seed).choice(len(frames), keep, replace=False))
    info = np.zeros((len(idx), 4), np.float64)
    model = np.full((len(idx), max_objects), -1.0, np.float64)
    pose = np.zeros((len(idx), max_objects, 7), np.float32)
    score = np.zeros((len(idx), max_objects), np.float32)
    for j, f in enumerate(idx):
        fr = frames[f]
        k = len(fr["model"])
        info[j] = fr["info"]
        model[j, :k] = fr["model"]
        pose[j, :k] = fr["pose"]
        score[j, :k] = fr["score"]
    os.makedirs(path, exist_ok=True)
    for name, a in (("frame_index", idx.astype(np.float64)), ("frame_info", info), ("obj_model", model), ("obj_pose", pose), ("obj_score", score)):
        np.save(os.path.join(path, name + ".npy"), a)


def run_ours(args, rank, world, local_rank):
    os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")   # the frame lanes are concurrent streams
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")      # NCCL's banner ("NCCL version ...") must not land on stdout beside the JSON line
    import torch
    import torch.distributed as dist
    from moped_b200 import capi

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; libmoped_cuda has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        init_nccl_quietly(dist, dev)

    log(f"[bench] rank {rank}/{world} on cuda:{local_rank}: pipeline={args.pipeline} stage_sms={args.stage_sms} lanes={args.lanes}")
    B, Q = args.frames, args.features
    if B % world:
        raise SystemExit(f"bench.py: --frames {B} must be a multiple of the number of GPUs ({world})")
    db = synth.make_db(args.objects, args.pts)
    n_pool = 2                                         # two different batches, alternated between steps
    pool = [[synth.make_frame(db, Q, n_visible=8, frame_id=p * B + i) for i in range(B)] for p in range(n_pool)]
    dbn = host_norm_rows(db["desc"])
    shards = shard_objects(db["n_pts"], world)
    o0, o1, r0, r1 = shards[rank]
    fo = (np.arange(B + 1) * Q).astype(np.int32)
    QT = B * Q

    ctx = capi.Context(local_rank)
    stream = torch.cuda.Stream()          # a real (non-default) stream shared by torch, NCCL ordering and libmoped_cuda
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)
    ctx.db_upload(dbn[r0:r1], db["xyz"][r0:r1], db["model_of_row"][r0:r1], args.objects, row_base=r0)
    if world > 1:
        ctx.db_set_global_tables(db["xyz"], db["model_of_row"], args.objects)
    ctx.set_cameras(synth.K_DEFAULT, synth.CAM_IDENTITY)
    ctx.set_profiling(True)
    ctx.set_tuning(args.lanes, args.pose_warps, args.chunks)
    ctx.set_option("match_coarse_kind", args.coarse_kind)
    ctx.set_option("match_reserve_sms", args.reserve_sms)
    ctx.set_option("batch_graph", args.batch_graph)
    ctx.set_option("ransac_merge_levels", args.merge_levels)
    if args.pose_mode == "exact":          # POSE / POSE2 with the order-preserving LM: every frame equals the oracle chain bit for bit
        ctx.set_option("pose_exact_order", 1)
    params = ctx.default_params()
    MO = 64                                            # object slots per frame in the result arrays

    # pinned host copies (e2e leg) and device-resident copies (value leg) of the two batches
    h_q = [torch.from_numpy(np.concatenate([host_norm_rows(f["desc"]) for f in fr])).pin_memory() for fr in pool]
    h_xy = [torch.from_numpy(np.concatenate([f["xy"] for f in fr])).pin_memory() for fr in pool]
    h_img = [torch.from_numpy(np.concatenate([f["image_idx"] for f in fr])).pin_memory() for fr in pool]
    d_q = [t.to(dev) for t in h_q]
    d_xy = [t.to(dev) for t in h_xy]
    d_img = [t.to(dev) for t in h_img]
    if world > 1:
        e_q = torch.empty((QT, 128), dtype=torch.float32, device=dev)
        e_xy = torch.empty((QT, 2), dtype=torch.float32, device=dev)
        e_img = torch.empty((QT,), dtype=torch.int32, device=dev)
        # this rank's (row, distance) pairs as ONE block [rows QT x 2 int32 | distances QT x 2 fp32]: mc_match_dev writes both halves in
        # place, one all-gather moves them, mc_match_merge_packed_dev reads the gathered blocks
        nn_blk = torch.empty((4 * QT,), dtype=torch.int32, device=dev)
        nn_all = torch.empty((world, 4 * QT), dtype=torch.int32, device=dev)
        nn_row = torch.empty((QT, 2), dtype=torch.int32, device=dev)
        nn_dist = torch.empty((QT, 2), dtype=torch.float32, device=dev)
        acc = torch.empty((QT,), dtype=torch.uint8, device=dev)
        q_lo, q_hi = rank * (QT // world), (rank + 1) * (QT // world)     # the slice of the batch's queries this rank uploads (e2e leg)
        f_lo, f_hi = frame_range(B, world, rank)       # frames of this rank after MATCH
        Bl = f_hi - f_lo
        blk = ResultBlock(Bl, MO)                      # written in place by mc_process_frames_matched_dev, all-gathered as one tensor
        REC = blk.words
        res_local = torch.zeros((REC,), dtype=torch.int32, device=dev)
        res_all = torch.zeros((world, REC), dtype=torch.int32, device=dev)
        res_host = torch.zeros((world, REC), dtype=torch.int32).pin_memory()
    img_bytes = ((r1 - r0 + 127) // 128) * 32768
    need_flush = img_bytes < 2 * L2_BYTES
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev) if need_flush else None

    def sharded_step(q, xy, img):
        """N > 1: shard-local MATCH of all B*Q queries, all-gather of the (row, distance) pairs, merge, this rank's
        B/N frames through CLUSTER..FILTER2, all-gather of the per-frame results, read-back."""
        ctx.match_dev(q.data_ptr(), QT, params.match_ratio, params.match_mode, nn_blk.data_ptr(), nn_blk.data_ptr() + 8 * QT, acc.data_ptr())
        dist.all_gather_into_tensor(nn_all, nn_blk)
        ctx.match_merge_packed_dev(nn_all.data_ptr(), world, QT, params.match_ratio, nn_row.data_ptr(), nn_dist.data_ptr(), acc.data_ptr())
        ctx.process_frames_matched_dev(nn_row.data_ptr(), acc.data_ptr(), xy.data_ptr(), img.data_ptr(), fo, f_lo, f_hi, params, MO,
                                       res_local.data_ptr() + 4 * blk.o_info, res_local.data_ptr() + 4 * blk.o_model,
                                       res_local.data_ptr() + 4 * blk.o_pose, res_local.data_ptr() + 4 * blk.o_score)
        dist.all_gather_into_tensor(res_all, res_local)
        res_host.copy_(res_all, non_blocking=True)
        stream.synchronize()
        info = res_host[:, :Bl * 4].numpy().reshape(B, 4)
        return int(info[:, 0].sum()), int(info[:, 2].sum())

    # ---- pipelined stream of batches (--pipeline 1) --------------------------------------------------------------------
    # ONE context, software-pipelined: MATCH of step i+1 (the context's stream; its coarse kernel on the MATCH partition of the
    # GPU) runs beside CLUSTER..FILTER2 of step i (the frame lanes, on the stage partition: mc_set_option "stage_sm_partition").
    # mc_process_frames_matched_dev returns without joining the lanes ("defer_lane_join"); the join, the all-gather of the
    # results and their read-back are enqueued AFTER the next step's MATCH. Same C-ABI calls and the same results as the
    # one-call-per-step path; buffers are triple-buffered and the host stays two steps behind the device. Every step completes
    # inside the timed region.
    if args.pipeline:
        if args.stage_sms:
            ctx.set_option("stage_sm_partition", args.stage_sms)
        ctx.set_option("defer_lane_join", 1)
        sms_match, sms_stage = ctx.sm_partition()
        pf_lo, pf_hi = frame_range(B, world, rank)
        pBl = pf_hi - pf_lo
        pblk = ResultBlock(pBl, MO)
        P = 3
        p_q = [torch.empty((QT, 128), dtype=torch.float32, device=dev) for _ in range(P)]
        p_xy = [torch.empty((QT, 2), dtype=torch.float32, device=dev) for _ in range(P)]
        p_img = [torch.empty((QT,), dtype=torch.int32, device=dev) for _ in range(P)]
        p_row = [torch.empty((QT, 2), dtype=torch.int32, device=dev) for _ in range(P)]
        p_dist = [torch.empty((QT, 2), dtype=torch.float32, device=dev) for _ in range(P)]
        p_acc = [torch.empty((QT,), dtype=torch.uint8, device=dev) for _ in range(P)]
        p_blk = [torch.empty((4 * QT,), dtype=torch.int32, device=dev) for _ in range(P)] if world > 1 else None
        p_all = [torch.empty((world, 4 * QT), dtype=torch.int32, device=dev) for _ in range(P)] if world > 1 else None
        p_res = [torch.zeros((pblk.words,), dtype=torch.int32, device=dev) for _ in range(P)]
        p_resall = [torch.zeros((world, pblk.words), dtype=torch.int32, device=dev) for _ in range(P)]
        p_reshost = [torch.zeros((world, pblk.words), dtype=torch.int32).pin_memory() for _ in range(P)]
        ev_done = [torch.cuda.Event() for _ in range(P)]

        def pipe_match(i, e2e):
            k, b = i % n_pool, i % P
            if flush is not None:
                flush.zero_()
            if e2e and world == 1:                    # host buffers in: the step's features go up inside the timed region
                p_q[b].copy_(h_q[k], non_blocking=True)
                p_xy[b].copy_(h_xy[k], non_blocking=True)
                p_img[b].copy_(h_img[k], non_blocking=True)
                q = p_q[b]
            elif e2e:                                 # N > 1: 1/N of the descriptors per rank + NVLink all-gather; coordinates of its own frames
                ql, qh = rank * (QT // world), (rank + 1) * (QT // world)
                p_q[b][ql:qh].copy_(h_q[k][ql:qh], non_blocking=True)
                dist.all_gather_into_tensor(p_q[b], p_q[b][ql:qh])
                p_xy[b][fo[pf_lo]:fo[pf_hi]].copy_(h_xy[k][fo[pf_lo]:fo[pf_hi]], non_blocking=True)
                p_img[b][fo[pf_lo]:fo[pf_hi]].copy_(h_img[k][fo[pf_lo]:fo[pf_hi]], non_blocking=True)
                q = p_q[b]
            else:
                q = d_q[k]
            if world > 1:
                ctx.match_dev(q.data_ptr(), QT, params.match_ratio, params.match_mode, p_blk[b].data_ptr(), p_blk[b].data_ptr() + 8 * QT, p_acc[b].data_ptr())
                dist.all_gather_into_tensor(p_all[b], p_blk[b])
                ctx.match_merge_packed_dev(p_all[b].data_ptr(), world, QT, params.match_ratio, p_row[b].data_ptr(), p_dist[b].data_ptr(), p_acc[b].data_ptr())
            else:
                ctx.match_dev(q.data_ptr(), QT, params.match_ratio, params.match_mode, p_row[b].data_ptr(), p_dist[b].data_ptr(), p_acc[b].data_ptr())

        def pipe_stages(i, e2e):
            k, b = i % n_pool, i % P
            xy, img = (p_xy[b], p_img[b]) if e2e else (d_xy[k], d_img[k])
            r = p_res[b]
            ctx.process_frames_matched_dev(p_row[b].data_ptr(), p_acc[b].data_ptr(), xy.data_ptr(), img.data_ptr(), fo, pf_lo, pf_hi, params, MO,
                                           r.data_ptr() + 4 * pblk.o_info, r.data_ptr() + 4 * pblk.o_model,
                                           r.data_ptr() + 4 * pblk.o_pose, r.data_ptr() + 4 * pblk.o_score)

        def pipe_finish(i):
            b = i % P
            ctx.join_lanes()                              # the stream now waits for the lanes of step i
            if world > 1:
                dist.all_gather_into_tensor(p_resall[b], p_res[b])
                p_reshost[b].copy_(p_resall[b], non_blocking=True)
            else:
                p_reshost[b][0].copy_(p_res[b], non_blocking=True)
            ev_done[b].record(stream)

        def pipe_collect(i):
            b = i % P
            ev_done[b].synchronize()
            info = p_reshost[b][:, :pBl * 4].numpy().reshape(B, 4)
            return int(info[:, 0].sum()), int(info[:, 2].sum())

        def pipe_run(n, first, e2e):
            """steps first .. first+n-1, all complete (results on the host) on return"""
            n_obj = n_match = 0
            for j in range(n):
                pipe_match(first + j, e2e)
                if j >= 1:
                    pipe_finish(first + j - 1)            # behind MATCH of step j on the stream: the lanes of step j-1 ran beside it
                pipe_stages(first + j, e2e)
                if j >= 2:
                    no, nm = pipe_collect(first + j - 2)
                    n_obj += no
                    n_match += nm
            pipe_finish(first + n - 1)
            for j in range(max(0, n - 2), n):
                no, nm = pipe_collect(first + j)
                n_obj += no
                n_match += nm
            return n_obj, n_match

        def timed_pipe(e2e, steps, warmup):
            pipe_run(warmup, 0, e2e)
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            l0 = ctx.launches
            e0.record(stream)
            n_obj, n_match = pipe_run(steps, warmup, e2e)
            e1.record(stream)                             # the last step's read-back is the last thing on the stream
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item()), ctx.launches - l0, n_obj, n_match

    last_out = []                                     # per-frame results of the latest single-GPU step_dev (--dump-outputs)

    def step_dev(i):
        k = i % n_pool
        if world == 1:
            out = ctx.process_frames_dev(d_q[k].data_ptr(), d_xy[k].data_ptr(), d_img[k].data_ptr(), fo, params, MO)
            last_out[:] = out
            return sum(len(o["model"]) for o in out), sum(int(o["info"][2]) for o in out)
        return sharded_step(d_q[k], d_xy[k], d_img[k])

    def step_e2e(i):
        k = i % n_pool
        if world == 1:
            out = ctx.process_frames(h_q[k].numpy(), h_xy[k].numpy(), h_img[k].numpy(), fo, params, MO)
            return sum(len(o["model"]) for o in out), sum(int(o["info"][2]) for o in out)
        # host buffers in: every rank uploads 1/N of the batch's descriptors and they are all-gathered over NVLink (N replicated PCIe
        # copies of the whole batch were 29 % of the 8-GPU step); coordinates / image indices only of the frames this rank runs after MATCH
        e_q[q_lo:q_hi].copy_(h_q[k][q_lo:q_hi], non_blocking=True)
        dist.all_gather_into_tensor(e_q, e_q[q_lo:q_hi])
        e_xy[fo[f_lo]:fo[f_hi]].copy_(h_xy[k][fo[f_lo]:fo[f_hi]], non_blocking=True)
        e_img[fo[f_lo]:fo[f_hi]].copy_(h_img[k][fo[f_lo]:fo[f_hi]], non_blocking=True)
        return sharded_step(e_q, e_xy, e_img)

    mtiers = []                                       # per timed step: {queries, certified by the 8-bit pass, by the fp16 pass, exact scan}
    mstats = []                                       # per timed step: {certified, fallback, candidates per query, DB splits} of its MATCH pass

    def timed(step_fn, steps, warmup, collect_kernel=False):
        for i in range(warmup):
            step_fn(i)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        kms, n_obj, n_match = [], 0, 0
        mstats.clear()
        mtiers.clear()
        l0 = ctx.launches
        for i in range(steps):
            if flush is not None:
                flush.zero_()
            ev[i][0].record(stream)
            no, nm = step_fn(warmup + i)
            ev[i][1].record(stream)
            n_obj += no
            n_match += nm
            if collect_kernel:
                kms.append(ctx.coarse_kernel_ms())
                mstats.append(ctx.match_last_stats())        # the step has completed (its results are on the host): no extra wait
                mtiers.append(ctx.match_tier_stats())
        launches = ctx.launches - l0
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        total_ms = sum(a.elapsed_time(b) for a, b in ev)
        t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), kms, launches, n_obj, n_match

    if rank == 0:
        log("[bench] setup done, timing")
    sampler = ClockSampler(local_rank)
    sampler.start()
    if args.pipeline:
        total_ms, launches, n_obj, n_match = timed_pipe(False, args.steps, args.warmup)
        clocks = sampler.stop()
        # the last timed step is step warmup + steps - 1; its all-gathered results are still in its host buffer
        dumped = pblk.unpack(p_reshost[(args.warmup + args.steps - 1) % P].numpy()) if args.dump_outputs else None
        e2e_ms, _, n_obj_e, _ = timed_pipe(True, args.steps, args.warmup)
        kms = []                                      # dominant-kernel time: a separate short pass, reading the library's event pair
        for i in range(min(args.steps, 8)):           # after every step would put the host in lock-step with the match stream
            pipe_run(1, i, False)
            kms.append(ctx.coarse_kernel_ms())
            mstats.append(ctx.match_last_stats())
            mtiers.append(ctx.match_tier_stats())
        match_stats = np.array(mstats, np.int64)
        ctx.set_option("defer_lane_join", 0)
    else:
        total_ms, kms, launches, n_obj, n_match = timed(step_dev, args.steps, args.warmup, collect_kernel=True)
        clocks = sampler.stop()
        dumped = None
        if args.dump_outputs:                          # before the e2e leg reuses the result buffers
            dumped = list(last_out) if world == 1 else blk.unpack(res_host.numpy())
        match_stats = np.array(mstats, np.int64) if mstats else np.zeros((1, 4), np.int64)
        tier_rows = list(mtiers)                      # (the e2e leg below reuses the lists)
        e2e_ms, _, _, n_obj_e, _ = timed(step_e2e, args.steps, args.warmup)
        mtiers[:] = tier_rows

    # outside the timed region: device time of MATCH vs CLUSTER..FILTER2 for one batch, and the latency of a single frame
    ms_batch = np.zeros(2, np.float32)
    lat_ms, ms_stage = None, np.zeros(6, np.float32)
    if world == 1:
        ctx.process_frames_dev(d_q[0].data_ptr(), d_xy[0].data_ptr(), d_img[0].data_ptr(), fo, params, MO, times=ms_batch)
        ctx.set_tuning(0, 8, 0)
        for _ in range(3):
            ctx.process_frame_dev(d_q[0].data_ptr(), d_xy[0].data_ptr(), d_img[0].data_ptr(), Q, params, times=ms_stage)
        t0 = time.perf_counter()
        for _ in range(10):
            ctx.process_frame_dev(d_q[0].data_ptr(), d_xy[0].data_ptr(), d_img[0].data_ptr(), Q, params)
        lat_ms = (time.perf_counter() - t0) / 10 * 1e3
        ctx.set_tuning(0, args.pose_warps, 0)

    if rank == 0:
        log(f"[bench] timed: {total_ms / args.steps:.3f} ms/step")
        peak_tf, peak_gbs, peak_src = measured_peaks()
        peak_sus = measured_sustained_tflops()
        i8 = args.coarse_kind == 1
        kname = "k_match_coarse<1> (tcgen05 kind::i8)" if i8 else "k_match_coarse<0> (tcgen05 kind::f16)"
        traffic = measured_traffic("k_match_coarse_i8" if i8 else "k_match_coarse_f16", db_descriptors=args.objects * args.pts, features_per_frame=Q,
                                   frames_per_step=B, n_gpus=world)
        if i8:      # no measured 8-bit figure in MEASURED_PEAKS.json: the 8-bit kinds run at twice the 16-bit MMA rate (4.5 vs 2.25 PF nominal)
            peak_16, peak_tf, peak_sus = peak_tf, 2.0 * peak_tf, (2.0 * peak_sus if peak_sus else None)
        tiers = np.array(mtiers, np.int64) if mtiers else np.zeros((1, 4), np.int64)
        ms_step = total_ms / args.steps
        fps = B * 1e3 / ms_step
        k_ms = float(np.mean(kms)) if kms else None
        launches_coarse = max(1, args.chunks if world == 1 else 1)
        flops = 2.0 * (QT / launches_coarse) * (r1 - r0) * 128
        achieved = flops / (k_ms * 1e-3) / 1e12 if k_ms else None
        out = {"metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
               "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
               "dtype": ("u8/s8 tensor-core coarse pass (exact int32 accumulation), f16 second-chance pass, f32 exact re-rank/LM" if i8 else
                         "f16 tensor-core coarse pass + f32 exact re-rank/LM"), "data": "synthetic",
               "config": workload_config(args, world),
               "objects_per_frame": n_obj / (args.steps * B),
               "matches_per_s": n_match / (total_ms * 1e-3),
               "query_descriptors_per_s": QT * args.steps / (total_ms * 1e-3),
               # MATCH exactness bookkeeping of the timed steps (rank 0's shard): every query is either certified by the tensor-core
               # coarse pass or re-done by the exhaustive exact scan; certified + fallback == queries
               "match_queries": int(match_stats[:, :2].sum()), "match_certified": int(match_stats[:, 0].sum()),
               "match_fallback": int(match_stats[:, 1].sum()), "match_candidates_per_query": int(match_stats[0, 2]),
               "match_db_splits": int(match_stats[0, 3]),
               # the cascade by tier (timed steps): certified by the 8-bit pass / by the fp16 pass / sent to the exhaustive scan
               "match_tiers": {"queries": int(tiers[:, 0].sum()), "certified_8bit": int(tiers[:, 1].sum()), "certified_fp16": int(tiers[:, 2].sum()),
                               "exact_scan": int(tiers[:, 3].sum())},
               "batch_ms": None if world > 1 else {"match": float(ms_batch[0]), "cluster_to_filter2": float(ms_batch[1])},
               "single_frame": None if world > 1 else {"latency_ms": lat_ms, "stage_ms": {k: float(v) for k, v in zip(["match", "cluster", "pose", "filter", "pose2", "filter2"], ms_stage)}},
               "gpu_launches": int(launches),
               "sm_partition": {"match_sms": sms_match, "stage_sms": sms_stage} if args.pipeline else None,
               "clocks": clocks,
               "e2e": {"value": B * 1e3 / (e2e_ms / args.steps), "unit": UNIT, "h2d_bytes_per_step": int(QT * (128 + 2 + 1) * 4),   # summed over the ranks
                       "d2h_bytes_per_step": int(B * (16 + 36 * MO))},
               "roofline": {"kernel": kname, "bound": "tensor", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s",
                            "frac": (achieved / peak_tf) if achieved else None, "traffic": traffic["bytes"] if traffic else None,
                            "traffic_source": traffic["source"] if traffic else None,
                            "peak_source": (f"2 x {peak_src} MEASURED_PEAKS.json bf16_tflops (burst): 8-bit operand kinds issue at twice the 16-bit MMA rate; "
                                            "integer multiply-adds counted as 2 ops like flops") if i8 else f"{peak_src} (MEASURED_PEAKS.json bf16_tflops, burst)",
                            "kernel_ms": k_ms, "frac_of_bf16_peak": (achieved / peak_16) if (i8 and achieved) else None,
                            "peak_sustained": peak_sus, "frac_of_sustained": (achieved / peak_sus) if achieved and peak_sus else None,
                            "algorithmic_flops_per_launch": flops,
                            "algorithmic_bytes_per_launch": int((r1 - r0 + 127) // 128 * (16384 if i8 else 32768) + QT * (128 if i8 else 256))}}
        if world == 1 and not args.no_cpu_baseline:
            try:
                from oracle import ref
                if ref.available():
                    cores = os.cpu_count() or 1
                    r = reference_setup(db, cores)
                    s, st, n = reference_sample_step(r, pool[0][0], 8, seed=5)
                    out["cpu_baseline"] = {"value": 1.0 / s, "unit": UNIT, "cores": cores, "kind": "reference",
                                           "sample": "1 frame: MATCH_ANN_CPU(eps=5) on a uniform 1/8 of the features, time x8 + CLUSTER..FILTER2 on the planted "
                                                     "features' matches; kd-tree build excluded",
                                           "stage_ms": {k: float(v * 1e3) for k, v in zip(["match", "cluster", "pose", "filter", "pose2", "filter2"], st)},
                                           "objects": int(n)}
                else:
                    out["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "reference", "sample": "oracle/_ref not built"}
            except Exception as e:  # the GPU numbers stand on their own
                out["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "reference", "sample": f"failed: {e}"}
        if world == 1 and args.other_configs and default_metric_config(args):
            out["other_configs"] = other_config_lines()
        if args.dump_outputs:
            dump_frame_results(args.dump_outputs, dumped, MO)
            log(f"[bench] outputs of the last timed step ({len(dumped)} frames) written to {args.dump_outputs}")
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def run_ours_cluster_partition(args, rank, world, local_rank):
    """N > 1 with fewer frames than GPUs (BASELINE configs[2] as ONE sharded frame: `--frames 1 --gpus N`), or `--partition cluster`:
    the database is sharded by object as always (every rank matches the frame's queries against its shard, one packed all-gather,
    merge), and the stages after MATCH run on EVERY rank with the RANSAC tasks of POSE and POSE2 distributed by cluster
    (mc_process_frame_sharded_dev: rank r runs the clusters c with c % N == r; two small in-place all-gathers of the task results).
    north_star: "RANSAC work is distributed by cluster". Every rank ends with the frame's objects; rank 0 reads them back."""
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    import torch
    import torch.distributed as dist
    from moped_b200 import capi

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; libmoped_cuda has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        init_nccl_quietly(dist, dev)
    B, Q = args.frames, args.features
    QT = B * Q
    db = synth.make_db(args.objects, args.pts)
    n_pool = 2
    pool = [[synth.make_frame(db, Q, n_visible=8, frame_id=p * B + i) for i in range(B)] for p in range(n_pool)]
    dbn = host_norm_rows(db["desc"])
    o0, o1, r0, r1 = shard_objects(db["n_pts"], world)[rank]
    ctx = capi.Context(local_rank)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)
    ctx.db_upload(dbn[r0:r1], db["xyz"][r0:r1], db["model_of_row"][r0:r1], args.objects, row_base=r0)
    ctx.db_set_global_tables(db["xyz"], db["model_of_row"], args.objects)
    ctx.set_cameras(synth.K_DEFAULT, synth.CAM_IDENTITY)
    ctx.set_profiling(True)
    ctx.set_tuning(args.lanes, 8, 1)                   # latency shape: 8 first-round hypotheses per task
    ctx.set_option("match_coarse_kind", args.coarse_kind)
    if args.pose_mode == "exact":
        ctx.set_option("pose_exact_order", 1)
    params = ctx.default_params()
    MO = 64
    h_q = [torch.from_numpy(np.concatenate([host_norm_rows(f["desc"]) for f in fr])).pin_memory() for fr in pool]
    h_xy = [torch.from_numpy(np.concatenate([f["xy"] for f in fr])).pin_memory() for fr in pool]
    h_img = [torch.from_numpy(np.concatenate([f["image_idx"] for f in fr])).pin_memory() for fr in pool]
    d_q, d_xy, d_img = [t.to(dev) for t in h_q], [t.to(dev) for t in h_xy], [t.to(dev) for t in h_img]
    e_q, e_xy, e_img = torch.empty_like(d_q[0]), torch.empty_like(d_xy[0]), torch.empty_like(d_img[0])
    nn_blk = torch.empty((4 * QT,), dtype=torch.int32, device=dev)
    nn_all = torch.empty((world, 4 * QT), dtype=torch.int32, device=dev)
    nn_row = torch.empty((QT, 2), dtype=torch.int32, device=dev)
    nn_dist = torch.empty((QT, 2), dtype=torch.float32, device=dev)
    acc = torch.empty((QT,), dtype=torch.uint8, device=dev)
    slot = ctx.frame_shard_slot_bytes(Q, params)
    exch = torch.zeros((world, slot), dtype=torch.uint8, device=dev)
    res = torch.zeros((B, 4 + MO * 9), dtype=torch.int32, device=dev)      # per frame: info[4] | model[MO] | pose[7 MO] | score[MO]
    res_host = torch.zeros((B, 4 + MO * 9), dtype=torch.int32).pin_memory()
    img_bytes = ((r1 - r0 + 127) // 128) * 32768
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev) if img_bytes < 2 * L2_BYTES else None
    upload_q = (QT // world) * world == QT             # 1/N of the descriptors per rank + NVLink all-gather when it divides

    def step(i, e2e):
        k = i % n_pool
        q, xy, img = d_q[k], d_xy[k], d_img[k]
        if e2e:
            if world > 1 and upload_q:
                ql, qh = rank * (QT // world), (rank + 1) * (QT // world)
                e_q[ql:qh].copy_(h_q[k][ql:qh], non_blocking=True)
                dist.all_gather_into_tensor(e_q, e_q[ql:qh])
            else:
                e_q.copy_(h_q[k], non_blocking=True)
            e_xy.copy_(h_xy[k], non_blocking=True)
            e_img.copy_(h_img[k], non_blocking=True)
            q, xy, img = e_q, e_xy, e_img
        if world > 1:
            ctx.match_dev(q.data_ptr(), QT, params.match_ratio, params.match_mode, nn_blk.data_ptr(), nn_blk.data_ptr() + 8 * QT, acc.data_ptr())
            dist.all_gather_into_tensor(nn_all, nn_blk)
            ctx.match_merge_packed_dev(nn_all.data_ptr(), world, QT, params.match_ratio, nn_row.data_ptr(), nn_dist.data_ptr(), acc.data_ptr())
        else:
            ctx.match_dev(q.data_ptr(), QT, params.match_ratio, params.match_mode, nn_row.data_ptr(), nn_dist.data_ptr(), acc.data_ptr())
        for f in range(B):
            o = res[f].data_ptr()
            a = (nn_row.data_ptr() + 8 * f * Q, acc.data_ptr() + f * Q, xy.data_ptr() + 8 * f * Q, img.data_ptr() + 4 * f * Q, Q, params, rank, world,
                 exch.data_ptr(), MO, o, o + 16, o + 16 + 4 * MO, o + 16 + 32 * MO)
            for phase in range(3):
                ctx.process_frame_sharded_dev(phase, *a)
                if phase < 2 and world > 1:
                    dist.all_gather_into_tensor(exch, exch[rank])
        res_host.copy_(res, non_blocking=True)
        stream.synchronize()
        info = res_host[:, :4].numpy()
        return int(info[:, 0].sum()), int(info[:, 2].sum())

    def timed(e2e, steps, warmup, collect=False):
        for i in range(warmup):
            step(i, e2e)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        n_obj = n_match = 0
        kms = []
        l0 = ctx.launches
        for i in range(steps):
            if flush is not None:
                flush.zero_()
            ev[i][0].record(stream)
            no, nm = step(warmup + i, e2e)
            ev[i][1].record(stream)
            n_obj += no
            n_match += nm
            if collect:
                kms.append(ctx.coarse_kernel_ms())
        launches = ctx.launches - l0
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t = torch.tensor([sum(a.elapsed_time(b) for a, b in ev)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), kms, launches, n_obj, n_match

    sampler = ClockSampler(local_rank)
    sampler.start()
    total_ms, kms, launches, n_obj, n_match = timed(False, args.steps, args.warmup, collect=True)
    clocks = sampler.stop()
    e2e_ms, _, _, _, _ = timed(True, args.steps, args.warmup)
    if rank == 0:
        peak_tf, _, peak_src = measured_peaks()
        i8 = args.coarse_kind == 1
        if i8:
            peak_tf *= 2.0
        ms_step = total_ms / args.steps
        k_ms = float(np.mean(kms)) if kms else None
        flops = 2.0 * QT * (r1 - r0) * 128
        achieved = flops / (k_ms * 1e-3) / 1e12 if k_ms else None
        cfg = workload_config(args, world)
        cfg["parallelism"] = (f"db-sharded-by-object x{world}; CLUSTER / FILTER replicated, RANSAC tasks of POSE and POSE2 distributed by cluster x{world} "
                              "(mc_process_frame_sharded_dev, two in-place all-gathers of the task results per frame)")
        cfg["pipeline"] = "one frame after the other on the context's stream"
        out = {"metric": METRIC, "value": B * 1e3 / ms_step, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
               "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
               "dtype": "u8/s8 tensor-core coarse pass (exact int32 accumulation), f16 second-chance pass, f32 exact re-rank/LM" if i8 else
                        "f16 tensor-core coarse pass + f32 exact re-rank/LM",
               "data": "synthetic", "config": cfg, "frame_latency_ms": ms_step / B,
               "objects_per_frame": n_obj / (args.steps * B), "matches_per_s": n_match / (total_ms * 1e-3),
               "gpu_launches": int(launches), "clocks": clocks,
               "e2e": {"value": B * 1e3 / (e2e_ms / args.steps), "unit": UNIT, "h2d_bytes_per_step": int(QT * 128 * 4 + world * QT * 12),
                       "d2h_bytes_per_step": int(B * (16 + 36 * MO))},
               "roofline": {"kernel": "k_match_coarse<1> (tcgen05 kind::i8)" if i8 else "k_match_coarse<0> (tcgen05 kind::f16)", "bound": "tensor",
                            "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": (achieved / peak_tf) if achieved else None, "traffic": None,
                            "peak_source": f"{'2 x ' if i8 else ''}{peak_src} MEASURED_PEAKS.json bf16_tflops (burst)", "kernel_ms": k_ms,
                            "algorithmic_flops_per_launch": flops,
                            "note": "a single frame is a latency measurement: 2000 queries give the coarse kernel 16 query tiles, far from a full wave"}}
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def default_metric_config(args):
    return (args.objects, args.pts, args.features, args.frames, args.pose_mode) == (1000, 1000, 2000, 64, "default")


def other_config_lines():
    """The other BASELINE.json configurations and the widened rows of SURVEY 8f as sub-results of the default line (single GPU): each is
    this same script run as a child process with its own timed region (device timing, W >= 3 warm-up steps, clocks sampled), and the
    child's JSON line is condensed to its headline numbers. A child that fails is reported as {"error": ...}; the main line stands."""
    import subprocess
    runs = {
        "configs[1] 100 objects, one 2000-feature frame": ["--objects", "100", "--frames", "1", "--steps", "20"],
        "configs[3] RANSAC-heavy 64 clusters x 2048 hypotheses": ["--workload", "ransac", "--steps", "5"],
        "configs[4] 64 frames x 4000 features, 1000 objects": ["--features", "4000", "--steps", "5"],
        "8f row 3 feature extraction, 64 frames 640x480": ["--workload", "sift", "--steps", "5"],
        "8f row 4 moped3d depth pose stage (bit-exact LM)": ["--workload", "depthpose", "--steps", "3"],
        "8f row 4 moped3d linkage clustering": ["--workload", "linkage", "--steps", "3"],
    }
    keep = ("metric", "value", "unit", "ms_per_step", "steps", "warmup", "gpu_launches", "dtype")
    res = {}
    for name, extra in runs.items():
        cmd = [sys.executable, os.path.abspath(__file__), "--gpus", "1", "--warmup", "3", "--no-cpu-baseline", "--other-configs", "0"] + extra
        try:
            t0 = time.perf_counter()
            r = subprocess.run(cmd, capture_output=True, text=True, timeout=240, env=dict(os.environ, RANK="0", WORLD_SIZE="1", LOCAL_RANK="0"))
            lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
            if r.returncode != 0 or not lines:
                res[name] = {"error": f"rc {r.returncode}: {(r.stderr or '').strip().splitlines()[-1:] or ''}"}
                continue
            d = json.loads(lines[-1])
            e = {k: d.get(k) for k in keep}
            e["e2e"] = (d.get("e2e") or {}).get("value")
            e["clocks_sm_mhz"] = (d.get("clocks") or {}).get("sm_mhz")
            e["throttle_reasons"] = (d.get("clocks") or {}).get("reasons")
            if d.get("single_frame"):
                e["single_frame_latency_ms"] = d["single_frame"].get("latency_ms")
            if d.get("roofline") and d["roofline"].get("frac") is not None:
                e["roofline"] = {k: d["roofline"].get(k) for k in ("kernel", "bound", "achieved", "peak", "unit", "frac")}
            e["cmd"] = "bench.py " + " ".join(extra)
            e["wall_s"] = round(time.perf_counter() - t0, 1)
            res[name] = e
        except Exception as ex:  # noqa: BLE001 - the main line stands on its own
            res[name] = {"error": str(ex)[:200]}
    return res


# ------------------------------------------------------------------------------------------------
# BASELINE.json configs[3]: RANSAC-heavy — 64 clusters x 2048 explicit hypotheses with LM refinement
# ------------------------------------------------------------------------------------------------
RANSAC_PARAMS = (600, 200, 1, 5, 6, 10.0)    # POSE defaults (config.hpp:105): LM itmax 200, 5-point samples, > 6 inliers, 10 px^2


def ransac_config(args, world):
    return {"workload": f"RANSAC-heavy (BASELINE configs[3]): {args.clusters} clusters x {args.hyp} explicit hypotheses, 80 points/cluster, 50% outliers, "
                        "sample fit (LM itmax 200) + inlier scoring + refit on inliers",
            "clusters": args.clusters, "hypotheses_per_cluster": args.hyp,
            "parallelism": f"clusters round-robin over {world} GPUs, no data-path collective" if world > 1 else "single-gpu"}


def run_ransac_reference(args, rank, world):
    """--impl reference --workload ransac: the reference's optimizeCamera/testAllPoints/refit per hypothesis (oracle/_ref) on all host
    cores, a bounded sample of the hypotheses of every cluster per step."""
    if rank != 0:
        return
    from oracle import ref
    if not ref.available():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libmoped_ref.so missing"}))
        return
    cores = os.cpu_count() or 1
    cl = synth.make_ransac_clusters(args.clusters, 80, 0.5)
    hy = synth.make_hypotheses(cl, args.hyp, 5)
    per = max(8, min(args.hyp, 32768 // args.clusters))       # hypotheses per cluster per step
    r = ransac_reference_setup(cl, cores)
    tot, nh = 0.0, 0
    for i in range(args.warmup + args.steps):
        s, n = ransac_reference_step(r, cl, hy, args, per, i)
        if i >= args.warmup:
            tot += s
            nh += n
        log(f"[reference] step {i}: {n / s:.0f} hypotheses/s")
    v = nh / tot
    out = {"impl": "reference", "metric": "hypotheses_per_s", "value": v, "unit": "hypotheses/s", "n_gpus": args.gpus, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": tot / args.steps * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
           "dtype": "f32", "data": "synthetic", "config": ransac_config(args, world),
           "cpu_baseline": {"value": v, "unit": "hypotheses/s", "cores": cores, "kind": "reference",
                            "sample": f"per step: {per} of the {args.hyp} hypotheses of each of the {args.clusters} clusters, OpenMP over hypotheses"},
           "e2e": {"value": v, "unit": "hypotheses/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out))


def ransac_reference_setup(cl, cores):
    from oracle import ref
    n_clusters = len(cl["offsets"]) - 1
    r = ref.Ref(cores)
    # one model per cluster; the cluster's correspondences are that model's matches
    n_pts = np.diff(cl["offsets"]).astype(np.int32)
    r.set_models(n_pts, cl["xyz"], np.zeros((len(cl["xyz"]), 128), np.float32) + np.float32(0.1))
    r.set_images(synth.K_DEFAULT, synth.CAM_IDENTITY)
    r.set_matches(dict(offsets=cl["offsets"], image=cl["image"], xy=cl["xy"], xyz=cl["xyz"]))
    return r


def ransac_reference_step(r, cl, hy, args, per, step):
    sec, n = 0.0, 0
    for c in range(args.clusters):
        lo = c * args.hyp + (step * per) % max(1, args.hyp - per + 1)
        members = np.arange(cl["offsets"][c + 1] - cl["offsets"][c], dtype=np.int32)
        s, _, _ = r.hypotheses_batch(c, members, hy["sample_pos"][lo:lo + per], hy["init_quat"][lo:lo + per],
                                     RANSAC_PARAMS[1], RANSAC_PARAMS[5], RANSAC_PARAMS[4])
        sec += s
        n += per
    return sec, n


def run_ransac_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from moped_b200 import capi

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; libmoped_cuda has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        init_nccl_quietly(dist, dev)
    cl = synth.make_ransac_clusters(args.clusters, 80, 0.5)
    hy = synth.make_hypotheses(cl, args.hyp, 5)
    mine = cluster_partition(hy["hyp_cluster"], world, rank)           # clusters round-robin over the ranks
    H = len(mine)
    ctx = capi.Context(local_rank)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)
    ctx.set_cameras(synth.K_DEFAULT, synth.CAM_IDENTITY)
    pp = capi.PoseParams.of(RANSAC_PARAMS)
    ctx.set_option("depth_team_lanes", args.depth_team)
    ctx.set_option("pose_fit_stream", args.fit_stream)
    h_in = [torch.from_numpy(np.ascontiguousarray(a)).pin_memory() for a in
            (cl["offsets"], cl["xy"], cl["xyz"], cl["image"], hy["hyp_cluster"][mine], hy["sample_pos"][mine], hy["init_quat"][mine])]
    d_in = [t.to(dev) for t in h_in]
    e_in = [torch.empty_like(t, device=dev) for t in h_in]
    d_out = [torch.zeros(H, dtype=torch.int32, device=dev), torch.zeros((H, 7), dtype=torch.float32, device=dev),
             torch.zeros((H, 7), dtype=torch.float32, device=dev), torch.zeros((H, 2), dtype=torch.float32, device=dev)]
    h_out = [torch.zeros(H, dtype=torch.int32).pin_memory(), torch.zeros((H, 7), dtype=torch.float32).pin_memory()]

    max_cluster = int(np.diff(cl["offsets"]).max())

    def launch(bufs):
        if args.pose_mode == "exact":      # the order-preserving LM (pose_depth.cu, variant 2 = this stage's residual): the oracle's bits
            p = [t.data_ptr() for t in bufs]
            ctx.pose_depth_hypotheses_dev(2, p[0], max_cluster, p[1], p[2], None, None, p[3], p[4], p[5], p[6], H, pp, 0.0,
                                          *[t.data_ptr() for t in d_out])
        else:
            ctx.pose_hypotheses_dev(*[t.data_ptr() for t in bufs], H, pp, *[t.data_ptr() for t in d_out])

    def step_dev(i):
        launch(d_in)

    def step_e2e(i):
        for e, h in zip(e_in, h_in):
            e.copy_(h, non_blocking=True)
        launch(e_in)
        h_out[0].copy_(d_out[0], non_blocking=True)
        h_out[1].copy_(d_out[2], non_blocking=True)
        stream.synchronize()

    def timed(fn, steps, warmup):
        for i in range(warmup):
            fn(i)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = ctx.launches
        e0.record(stream)
        for i in range(steps):
            fn(warmup + i)
        e1.record(stream)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), ctx.launches - l0

    sampler = ClockSampler(local_rank)
    sampler.start()
    total_ms, launches = timed(step_dev, args.steps, args.warmup)
    clocks = sampler.stop()
    e2e_ms, _ = timed(step_e2e, args.steps, args.warmup)
    n_in = d_out[0].cpu().numpy()
    if rank == 0:
        Htot = args.clusters * args.hyp
        ms_step = total_ms / args.steps
        out = {"metric": "hypotheses_per_s", "value": Htot * 1e3 / ms_step, "unit": "hypotheses/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
               "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
               "config": dict(ransac_config(args, world), l2="working set (a few hundred KB) is cache resident by nature; not flushed",
                              pose_mode=args.pose_mode, depth_team_lanes=args.depth_team, fit_stream=args.fit_stream),
               "accepted_fraction_rank0": float((n_in > RANSAC_PARAMS[4]).mean()), "lm_failed_fraction_rank0": float((n_in < 0).mean()),
               "gpu_launches": int(launches), "clocks": clocks,
               "e2e": {"value": Htot * 1e3 / (e2e_ms / args.steps), "unit": "hypotheses/s",
                       "h2d_bytes_per_step": int(sum(t.numel() * t.element_size() for t in h_in)),
                       "d2h_bytes_per_step": int(sum(t.numel() * t.element_size() for t in h_out))},
               "roofline": {"kernel": ("k_pose_fit_stream<5>" if args.fit_stream else "k_pose_fit_thread<5>") if args.pose_mode == "default" else "k_depth_hypotheses<2>", "bound": "fp32-issue/divergence (latency-shaped; see profiles/ for the ncu issue-slot figures)",
                            "achieved": None, "peak": None, "unit": "TFLOP/s", "frac": None, "traffic": None}}
        if not args.no_cpu_baseline and world == 1:
            try:
                from oracle import ref
                if ref.available():
                    cores = os.cpu_count() or 1
                    r = ransac_reference_setup(cl, cores)
                    per = max(8, min(args.hyp, 32768 // args.clusters))
                    ransac_reference_step(r, cl, hy, args, per, 0)
                    s, n = ransac_reference_step(r, cl, hy, args, per, 1)
                    out["cpu_baseline"] = {"value": n / s, "unit": "hypotheses/s", "cores": cores, "kind": "reference",
                                           "sample": f"{per} of the {args.hyp} hypotheses of each cluster, OpenMP over hypotheses"}
            except Exception as e:
                out["cpu_baseline"] = {"value": None, "unit": "hypotheses/s", "cores": 0, "kind": "reference", "sample": f"failed: {e}"}
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------
# --workload depthpose / linkage: moped3d's stages (SURVEY.md 8f row 4) through their host-buffer C-ABI entries, one GPU
# ------------------------------------------------------------------------------------------------
DEPTH_PARAMS = (192, 100, 4, 5, 6, 8.0)     # moped3d POSE (config.hpp:46): MaxRANSACTests, MaxLMTests, MaxObjectsPerCluster, NPtsAlign, MinNPtsObject, ErrorThreshold
DEPTH_ALPHA = 0.5


def moped3d_config(args):
    if args.workload == "depthpose":
        return {"workload": f"moped3d POSE_RANSAC_LM_DIFF_BACKPROJECTION_DEPTH: {args.clusters} clusters x {args.hyp} explicit hypotheses, 80 points/cluster, "
                            "50% outliers, sample fit (order-preserving LM, itmax 100) + consistency test + refit; bit-exact with the strict-IEEE reference",
                "clusters": args.clusters, "hypotheses_per_cluster": args.hyp, "depth_team_lanes": args.depth_team, "parallelism": "single-gpu",
                "l2": "working set (a few hundred KB) is cache resident by nature; not flushed"}
    return {"workload": "moped3d CLUSTER_LINKAGE (average linkage, 3-D filter 2): 600 matches of one model (two instances + outliers), two 320x240 depth / "
                        "fill-distance maps; a step = one mc_cluster_linkage call (host buffers in, clusters out)",
            "matches": 600, "linkage_cached": 1, "parallelism": "single-gpu", "l2": "working set (1.4 MB similarity matrix + maps) is cache resident; not flushed"}


def moped3d_inputs(args):
    if args.workload == "depthpose":
        cl = synth.make_depth_clusters(args.clusters, 80, 0.5)
        hy = synth.make_hypotheses(dict(offsets=cl["offsets"]), args.hyp, 5)
        return cl, hy
    return synth.make_linkage_scene(1), None


def moped3d_reference_rate(args, cl, hy, seconds):
    """the reference's own class (oracle/_ref, its -ffast-math flags) on ONE host core for `seconds`: units per second"""
    from oracle import ref3d
    t0 = time.perf_counter()
    n = 0
    if args.workload == "depthpose":
        per = [dict(xy=cl["xy"][a:b], xyz=cl["xyz"][a:b], world=cl["world"][a:b], fill=cl["fill"][a:b]) for a, b in zip(cl["offsets"][:-1], cl["offsets"][1:])]
        while time.perf_counter() - t0 < seconds:
            h = n % len(hy["hyp_cluster"])
            ref3d.hypothesis(per[hy["hyp_cluster"][h]], synth.K_DEPTH, synth.CAM_IDENTITY, DEPTH_ALPHA, hy["sample_pos"][h], hy["init_quat"][h],
                             DEPTH_PARAMS[1], DEPTH_PARAMS[5], DEPTH_PARAMS[4])
            n += 1
    else:
        while time.perf_counter() - t0 < seconds:
            ref3d.cluster_linkage(*cl)
            n += 1
    return n / (time.perf_counter() - t0)


def run_moped3d_reference(args, rank, world):
    if rank != 0:
        return
    from oracle import ref3d
    unit = "hypotheses/s" if args.workload == "depthpose" else "clusterings/s"
    if not ref3d.available():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libmoped3d_ref.so missing and /root/reference not present to build it"}))
        return
    cl, hy = moped3d_inputs(args)
    moped3d_reference_rate(args, cl, hy, 1.0)
    v = moped3d_reference_rate(args, cl, hy, 3.0 * max(1, args.steps))
    print(json.dumps({"impl": "reference", "metric": unit.replace("/", "_per_"), "value": v, "unit": unit, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                      "ms_per_step": None, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                      "config": moped3d_config(args),
                      "cpu_baseline": {"value": v, "unit": unit, "cores": 1, "kind": "reference",
                                       "sample": f"{3 * max(1, args.steps)} s of calls of the reference's own class on one host core (the class has no OpenMP)"},
                      "e2e": {"value": v, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def run_moped3d_ours(args, rank, world, local_rank):
    import torch
    from moped_b200 import capi
    if rank != 0:
        return                                   # one GPU: the stages' host entries; N > 1 would be N replicas
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; libmoped_cuda has no CPU fallback")
    ctx = capi.Context(local_rank)
    cl, hy = moped3d_inputs(args)
    depth = args.workload == "depthpose"
    unit = "hypotheses/s" if depth else "clusterings/s"
    if depth:
        ctx.set_cameras(synth.K_DEPTH[None], synth.CAM_IDENTITY[None])
        ctx.set_option("depth_team_lanes", args.depth_team)
        units = len(hy["hyp_cluster"])
        bytes_in = sum(cl[k].nbytes for k in ("offsets", "xy", "xyz", "world", "cauchy", "image")) + sum(hy[k].nbytes for k in hy)
        bytes_out = units * (4 + 28 + 28 + 8)

        def call():
            return ctx.pose_depth_hypotheses(0, cl["offsets"], cl["xy"], cl["xyz"], cl["world"], cl["cauchy"], cl["image"], hy["hyp_cluster"],
                                             hy["sample_pos"], hy["init_quat"], DEPTH_PARAMS, DEPTH_ALPHA, want_mask=False)
    else:
        ctx.set_option("linkage_cached", 1)
        units = 1
        bytes_in = sum(a.nbytes for a in cl)
        bytes_out = 4 * (2 * len(cl[0]) + 3)

        def call():
            return ctx.cluster_linkage(*cl)
    for _ in range(max(3, args.warmup)):
        out = call()
    sampler = ClockSampler(local_rank)
    sampler.start()
    l0 = ctx.launches
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = call()
    sec = (time.perf_counter() - t0) / args.steps       # the entries take host buffers and return host results: the call IS the end-to-end path
    launches = ctx.launches - l0
    clocks = sampler.stop()
    v = units / sec
    res = {"metric": unit.replace("/", "_per_"), "value": v, "unit": unit, "n_gpus": 1, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": sec * 1e3,
           "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": moped3d_config(args),
           "gpu_launches": int(launches), "clocks": clocks,
           "e2e": {"value": v, "unit": unit, "h2d_bytes_per_step": int(bytes_in), "d2h_bytes_per_step": int(bytes_out)},
           "roofline": {"kernel": "k_depth_hypotheses<0>" if depth else "k_link_agglomerate_cached",
                        "bound": "latency (dependent fp32 chains of the order-preserving LM / the serial merge sequence of the agglomeration: neither HBM nor tensor)",
                        "achieved": None, "peak": None, "unit": "GB/s", "frac": None, "traffic": None}}
    if depth:
        res["accepted_fraction"] = float((out[0] > DEPTH_PARAMS[4]).mean())
    else:
        res["clusters"] = int(len(out[0]) - 1)
    if not args.no_cpu_baseline:
        try:
            from oracle import ref3d
            if ref3d.available():
                moped3d_reference_rate(args, cl, hy, 1.0)
                res["cpu_baseline"] = {"value": moped3d_reference_rate(args, cl, hy, 10.0), "unit": unit, "cores": 1, "kind": "reference",
                                       "sample": "10 s of calls of the reference's own class (oracle/_ref, -ffast-math) on one host core; the class has no OpenMP"}
        except Exception as e:
            res["cpu_baseline"] = {"value": None, "unit": unit, "cores": 0, "kind": "reference", "sample": f"failed: {e}"}
    print(json.dumps(res))


# ------------------------------------------------------------------------------------------------
# --workload sift: feature extraction (SURVEY.md §8f row 3), frames/s of FEAT on 640x480 frames
# ------------------------------------------------------------------------------------------------
def sift_config(args, world):
    return {"workload": f"feature extraction (step 1, FEAT_SIFT): synthetic 640x480 grey frames (~2k SIFT keypoints each), ScaleOrigin -1 "
                        f"(doubled image, 7 octaves x 3 scales); a step = a batch of {args.frames} frames",
            "frames_per_step": args.frames, "image": "640x480 u8", "parallelism": "single-gpu" if world == 1 else f"frames partitioned x{world}"}


def sift_images(n, first=0):
    return np.stack([synth.make_image(first + i) for i in range(n)])


def run_sift_reference(args, rank, world):
    """--impl reference --workload sift: the reference's FEAT_SIFT_CPU/libsiftfast (oracle/_ref) with all host threads
    (libsiftfast parallelises inside an image with OpenMP) on a bounded sample of the step's frames."""
    if rank != 0:
        return
    from oracle import ref
    if not ref.available():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libmoped_ref.so missing and /root/reference not present to build it"}))
        return
    cores = os.cpu_count() or 1
    per = max(1, min(args.frames, 4))
    imgs = sift_images(per)
    tot, nk = 0.0, 0
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        k = sum(len(ref.sift(im, True)[0]) for im in imgs)
        dt = time.perf_counter() - t0
        if i >= args.warmup:
            tot += dt
            nk += k
        log(f"[reference] sift step {i}: {dt / per * 1e3:.1f} ms/frame, {k // per} keypoints/frame")
    fps = per * args.steps / tot
    out = {"impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": tot / args.steps / per * args.frames * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
           "data": "synthetic", "config": sift_config(args, world), "keypoints_per_frame": nk / (per * args.steps),
           "cpu_baseline": {"value": fps, "unit": UNIT, "cores": cores, "kind": "reference",
                            "sample": f"{per} of the {args.frames} frames of a step per step; libsiftfast's own OpenMP parallelism (OMP default threads)"},
           "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out))


def run_sift_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from moped_b200 import capi

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; libmoped_cuda has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        init_nccl_quietly(dist, dev)
    lo, hi = frame_range(args.frames, world, rank)                               # frames are independent: partition, no collective
    B = hi - lo
    pool = [sift_images(B, first=1000 * p + lo) for p in range(2)]               # two different batches, alternated
    H, W = pool[0].shape[1:]
    max_kp = 4096
    ctx = capi.Context(local_rank)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)
    h_gray = [torch.from_numpy(p).pin_memory() for p in pool]
    d_gray = [t.to(dev) for t in h_gray]
    e_gray = torch.empty_like(d_gray[0])
    d_xy = torch.zeros((B, max_kp, 2), dtype=torch.float32, device=dev)
    d_so = torch.zeros((B, max_kp, 2), dtype=torch.float32, device=dev)
    d_desc = torch.zeros((B, max_kp, 128), dtype=torch.float32, device=dev)
    d_cnt = torch.zeros(B, dtype=torch.int32, device=dev)
    h_cnt = torch.zeros(B, dtype=torch.int32).pin_memory()
    h_xy = torch.zeros((B, max_kp, 2), dtype=torch.float32).pin_memory()
    h_desc = torch.zeros((B, max_kp, 128), dtype=torch.float32).pin_memory()
    d2h = [0]

    def extract(gray):
        ctx.sift_dev(gray.data_ptr(), B, H, W, True, max_kp, d_xy.data_ptr(), d_so.data_ptr(), d_desc.data_ptr(), d_cnt.data_ptr())

    def step_dev(i):
        extract(d_gray[i % 2])

    def step_e2e(i):
        # the call a user makes, spelled out with pinned buffers: images up, features (counts, coord2D, descriptors) down
        e_gray.copy_(h_gray[i % 2], non_blocking=True)
        extract(e_gray)
        h_cnt.copy_(d_cnt, non_blocking=True)
        stream.synchronize()
        n = 0
        for f in range(B):
            k = min(int(h_cnt[f]), max_kp)
            h_xy[f, :k].copy_(d_xy[f, :k], non_blocking=True)
            h_desc[f, :k].copy_(d_desc[f, :k], non_blocking=True)
            n += k
        stream.synchronize()
        d2h[0] = 4 * B + n * (2 + 128) * 4

    blur_ms, blur_bytes = [], [0.0]

    def timed(fn, steps, warmup, collect=False):
        for i in range(warmup):
            fn(i)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = ctx.launches
        e0.record(stream)
        for i in range(steps):
            fn(warmup + i)
            if collect:
                ms, by = ctx.sift_profile_read()
                blur_ms.append(ms)
                blur_bytes[0] = by
        e1.record(stream)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), ctx.launches - l0

    sampler = ClockSampler(local_rank)
    sampler.start()
    total_ms, launches = timed(step_dev, args.steps, args.warmup)
    clocks = sampler.stop()
    e2e_ms, _ = timed(step_e2e, args.steps, args.warmup)
    ctx.set_profiling(True)                       # separate pass: the event pairs sit between the kernels of the step
    timed(step_dev, min(args.steps, 10), 1, collect=True)
    ctx.set_profiling(False)
    kp = int(d_cnt.sum().item())
    if rank == 0:
        ms_step = total_ms / args.steps
        _, hbm_peak, src = measured_peaks()
        kms = float(np.mean(blur_ms)) / 5.0                      # five octave-0 Gaussian+DoG launches per step
        ach = blur_bytes[0] / 5.0 / (kms * 1e-3) / 1e9
        plane_mb = B * (2 * H - 2) * (2 * W - 2) * 4 / 1e6
        # the working set of a batch (scale-space of all frames) is far larger than L2 for B >= 2; for B = 1 it is L2 resident
        l2 = (f"scale-space of a batch = {19 * 1.33 * plane_mb:.0f} MB > 126 MB L2, and two different batches alternate: not flushed"
              if 19 * 1.33 * plane_mb > 2 * L2_BYTES / 1e6 else "scale-space fits L2 at this batch size (latency case); not flushed")
        out = {"metric": METRIC, "value": args.frames * 1e3 / ms_step, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
               "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
               "dtype": "f32 (u8 pixels in)", "data": "synthetic", "config": dict(sift_config(args, world), l2=l2, max_keypoints=max_kp),
               "keypoints_per_frame_rank0": kp / B, "keypoints_per_s": kp / B * args.frames * 1e3 / ms_step,
               "gpu_launches": int(launches), "clocks": clocks,
               "e2e": {"value": args.frames * 1e3 / (e2e_ms / args.steps), "unit": UNIT, "h2d_bytes_per_step": int(B * H * W), "d2h_bytes_per_step": int(d2h[0])},
               "roofline": {"kernel": "k_sift_blur (fused Gaussian + DoG, octave 0)", "bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s",
                            "frac": ach / hbm_peak, "traffic": (measured_traffic("k_sift_blur", frames=B) or {}).get("bytes"),
                            "traffic_source": (measured_traffic("k_sift_blur", frames=B) or {}).get("source"),
                            "peak_source": f"{src} (MEASURED_PEAKS.json hbm_gbs)", "kernel_ms": kms,
                            "algorithmic_bytes_per_launch": blur_bytes[0] / 5.0,
                            "algorithmic_bytes": "per launch and frame: 1 plane read + Gaussian plane + DoG plane written, plane = 1278 x 958 x 4 B"}}
        if not args.no_cpu_baseline and world == 1:
            try:
                from oracle import ref
                if ref.available():
                    cores = os.cpu_count() or 1
                    imgs = pool[0][:4]
                    ref.sift(imgs[0], True)
                    t0 = time.perf_counter()
                    k = sum(len(ref.sift(im, True)[0]) for im in imgs)
                    dt = time.perf_counter() - t0
                    out["cpu_baseline"] = {"value": len(imgs) / dt, "unit": UNIT, "cores": cores, "kind": "reference",
                                           "sample": f"{len(imgs)} frames of the step, FEAT_SIFT_CPU/libsiftfast with its own OpenMP parallelism",
                                           "keypoints_per_frame": k / len(imgs)}
            except Exception as e:
                out["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "reference", "sample": f"failed: {e}"}
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------
# --workload images: pixels in, objects out (FEAT chained to MATCH..FILTER2 on the device, mc_process_images)
# ------------------------------------------------------------------------------------------------
def images_setup(args):
    """Real data only: the planar model database and a frame of the reference's shipped imagery (tests/golden/*.npz — the stand-in
    for BASELINE configs[0]); the frame is repeated with small horizontal shifts to fill a batch."""
    g = dict(np.load(os.path.join(ROOT, "tests", "golden", "real_images.npz")))
    sg = np.load(os.path.join(ROOT, "tests", "golden", "sift_golden.npz"))
    im = sg["bag4_full_double/image"]
    frames = np.stack([np.roll(im, (i % 8) - 4, axis=1) for i in range(args.frames)])
    return g, frames


def images_config(args, world):
    return {"workload": f"images in, objects out: FEAT_SIFT + MATCH..FILTER2 on real data (a 640x480 frame of the reference's timing.bag, shifted per slot; "
                        f"3 planar models / 1275 descriptors built from the reference's imagery); a step = a batch of {args.frames} frames",
            "frames_per_step": args.frames, "image": "640x480 u8", "parallelism": "single-gpu" if world == 1 else f"frames partitioned x{world}"}


def run_images_reference(args, rank, world):
    if rank != 0:
        return
    from oracle import ref
    if not ref.available():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libmoped_ref.so missing and /root/reference not present to build it"}))
        return
    cores = os.cpu_count() or 1
    g, frames = images_setup(args)
    r = ref.Ref(cores)
    r.set_models(g["n_pts"], g["db_xyz"], g["db_desc"])
    r.set_images(g["K"], g["cam_pose"])
    per = max(1, min(args.frames, 4))
    tot, n_obj = 0.0, 0
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        k = 0
        for f in range(per):
            xy, desc = ref.sift(frames[f], True)
            r.set_features(desc, xy, np.zeros(len(xy), np.int32))
            n, _ = r.run_pipeline(seed=3 + i)
            k += n
        dt = time.perf_counter() - t0
        if i >= args.warmup:
            tot += dt
            n_obj += k
        log(f"[reference] images step {i}: {dt / per * 1e3:.1f} ms/frame, {k / per:.1f} objects/frame")
    fps = per * args.steps / tot
    out = {"impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": tot / args.steps / per * args.frames * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
           "data": "real (reference's shipped imagery)", "config": images_config(args, world), "objects_per_frame": n_obj / (per * args.steps),
           "cpu_baseline": {"value": fps, "unit": UNIT, "cores": cores, "kind": "reference",
                            "sample": f"{per} of the {args.frames} frames of a step per step: FEAT_SIFT_CPU + MATCH_ANN_CPU(eps=5) .. FILTER2 with OpenMP"},
           "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out))


def run_images_ours(args, rank, world, local_rank):
    os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
    import torch
    import torch.distributed as dist
    from moped_b200 import capi

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; libmoped_cuda has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        init_nccl_quietly(dist, dev)
    g, frames_all = images_setup(args)
    lo, hi = frame_range(args.frames, world, rank)
    frames = np.ascontiguousarray(frames_all[lo:hi])
    B = len(frames)
    ctx = capi.Context(local_rank)
    ctx.db_upload(g["db_desc"], g["db_xyz"], g["model_of_row"], len(g["n_pts"]))
    ctx.set_cameras(g["K"], g["cam_pose"])
    ctx.set_tuning(args.lanes, args.pose_warps, 1)
    h_frames = torch.from_numpy(frames).pin_memory().numpy()

    def step(i):
        # the public call: host pixels in, objects out (H2D of the images and D2H of the objects inside)
        return ctx.process_images(h_frames, True, max_keypoints=2048, max_objects=16, want_times=(i < 0))

    for i in range(args.warmup):
        step(i)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    l0 = ctx.launches
    sampler = ClockSampler(local_rank)
    sampler.start()
    t0 = time.perf_counter()
    n_obj = n_feat = 0
    for i in range(args.steps):
        out = step(i)
        n_obj += sum(len(o["model"]) for o in out)
        n_feat += sum(o["n_features"] for o in out)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0              # every call synchronises: host wall clock = device time of the K steps
    clocks = sampler.stop()
    t = torch.tensor([dt], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    stage = step(-1)[0]["stage_ms"]
    if rank == 0:
        ms_step = float(t.item()) * 1e3 / args.steps
        fps = args.frames * 1e3 / ms_step
        out = {"metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
               "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32 (u8 pixels in; f16 tensor-core coarse matching)",
               "data": "real (reference's shipped imagery)", "config": dict(images_config(args, world), l2="not flushed (scale-space of a batch >> L2)"),
               "objects_per_frame": n_obj / (args.steps * B), "features_per_frame": n_feat / (args.steps * B),
               "stage_ms_per_batch_rank0": {"feat": float(stage[0]), "match": float(stage[1]), "cluster_to_filter2": float(stage[2])},
               "gpu_launches": int(ctx.launches - l0), "clocks": clocks,
               "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": int(frames.size), "d2h_bytes_per_step": int(B * (16 + 36 * 16) + 8 * B)},
               "note": "value == e2e here: the measured call takes host pixels and returns host objects; timed by the host clock around K synchronous calls",
               "roofline": {"kernel": "k_sift_blur (see --workload sift for the live roofline of the dominant kernel of this chain)", "bound": "hbm",
                            "achieved": None, "peak": None, "unit": "GB/s", "frac": None, "traffic": None}}
        if not args.no_cpu_baseline and world == 1:
            try:
                from oracle import ref
                if ref.available():
                    cores = os.cpu_count() or 1
                    r = ref.Ref(cores)
                    r.set_models(g["n_pts"], g["db_xyz"], g["db_desc"])
                    r.set_images(g["K"], g["cam_pose"])
                    t0 = time.perf_counter()
                    k = 0
                    for f in range(2):
                        xy, desc = ref.sift(frames[f], True)
                        r.set_features(desc, xy, np.zeros(len(xy), np.int32))
                        k += r.run_pipeline(seed=5)[0]
                    dt = time.perf_counter() - t0
                    out["cpu_baseline"] = {"value": 2 / dt, "unit": UNIT, "cores": cores, "kind": "reference", "objects_per_frame": k / 2,
                                           "sample": "2 frames of the step: FEAT_SIFT_CPU + MATCH_ANN_CPU(eps=5) .. FILTER2 with OpenMP (kd-tree build included once)"}
            except Exception as e:
                out["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "reference", "sample": f"failed: {e}"}
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--objects", type=int, default=1000)
    ap.add_argument("--pts", type=int, default=1000)
    ap.add_argument("--features", type=int, default=2000)
    ap.add_argument("--frames", type=int, default=64, help="independent frames per step (batch)")
    ap.add_argument("--lanes", type=int, default=0, help="concurrent frames after MATCH (mc_set_tuning); 0 = one per frame of a GPU's share, at most 64")
    ap.add_argument("--merge-levels", type=int, default=1, choices=[0, 1], help="frames workload: RANSAC levels 1 and 2 in one launch (mc_set_option ransac_merge_levels)")
    ap.add_argument("--batch-graph", type=int, default=1, choices=[0, 1], help="frames workload: the stage chains of a batch as ONE CUDA graph (default) or one graph per frame on the lane streams")
    ap.add_argument("--pose-warps", type=int, default=0, help="first-round hypotheses per RANSAC task (mc_set_tuning); 0 = 4")
    ap.add_argument("--chunks", type=int, default=1, help="MATCH launches per batch (mc_set_tuning)")
    ap.add_argument("--coarse-kind", type=int, default=1, choices=[0, 1], help="1 = 8-bit integer coarse pass first (default), 0 = fp16 coarse pass only; same results")
    ap.add_argument("--reserve-sms", type=int, default=0, help="SMs the persistent matching kernel leaves free for concurrent stage kernels")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--other-configs", type=int, default=1,
                    help="default line on one GPU: append the other BASELINE configurations (configs[1], [3], [4]) and the SURVEY 8f rows as "
                         "sub-results, each from a child run of this script (0 = off)")
    ap.add_argument("--stage-sms", type=int, default=-1,
                    help="--pipeline: SMs of the stage partition (CUDA green contexts; multiple of 8, 0 = no partition, -1 = pick by frames per GPU)")
    ap.add_argument("--pipeline", type=int, default=-1,
                    help="frames workload: 1 = MATCH of step i+1 runs beside CLUSTER..FILTER2 of step i (one context, SM partition); 0 = one call per step; "
                         "-1 = by frames per GPU")
    ap.add_argument("--workload", default="frames", choices=["frames", "ransac", "sift", "images", "depthpose", "linkage"],
                    help="frames = the BASELINE metric (default); ransac = BASELINE configs[3], hypotheses/s; "
                         "sift = feature extraction (SURVEY 8f row 3), frames/s of step 1; images = pixels in, objects out on real data; "
                         "depthpose / linkage = moped3d's depth-aware pose stage and linkage clustering (SURVEY 8f row 4)")
    ap.add_argument("--pose-mode", default="default", choices=["default", "exact"],
                    help="POSE / POSE2 arithmetic: default kernels (re-associating, fused multiply-add) or the order-preserving LM (bit-exact with "
                         "the oracle and the strict-IEEE build of the reference)")
    ap.add_argument("--depth-team", type=int, default=32, choices=[8, 32], help="ransac workload, --pose-mode exact: lanes per hypothesis (same bits)")
    ap.add_argument("--partition", default="auto", choices=["auto", "frame", "cluster"],
                    help="frames workload, N > 1: stages after MATCH partitioned by frame (default) or, with fewer frames than GPUs / 'cluster', "
                         "RANSAC tasks distributed by cluster on every rank (mc_process_frame_sharded_dev)")
    ap.add_argument("--fit-stream", type=int, default=1, choices=[0, 1],
                    help="ransac workload: 1 = persistent phase-synchronous thread-per-hypothesis kernel (default), 0 = the one-launch kernel; same results")
    ap.add_argument("--clusters", type=int, default=64)
    ap.add_argument("--hyp", type=int, default=2048, help="hypotheses per cluster (ransac workload)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="frames workload: after the timed steps, write the per-frame results of the last timed step as DIR/<name>.npy "
                         "(see dump_frame_results); the inputs are seeded, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    resolve_auto(args, world)
    cluster_partition_run = args.partition == "cluster" or (args.partition == "auto" and world > 1 and args.frames < world)
    if args.dump_outputs and (args.workload != "frames" or args.impl != "ours" or cluster_partition_run):
        ap.error("--dump-outputs covers the frames workload of --impl ours with the frames partitioned by GPU")
    if args.workload == "ransac":
        if args.impl == "reference":
            run_ransac_reference(args, rank, world)
        else:
            args.warmup = max(args.warmup, 3)
            run_ransac_ours(args, rank, world, local_rank)
    elif args.workload in ("depthpose", "linkage"):
        if args.workload == "depthpose" and args.hyp == 2048:
            args.hyp = 256                       # 64 x 256 = 16 384 hypotheses per call
        if args.impl == "reference":
            run_moped3d_reference(args, rank, world)
        else:
            run_moped3d_ours(args, rank, world, local_rank)
    elif args.workload == "images":
        if args.impl == "reference":
            run_images_reference(args, rank, world)
        else:
            args.warmup = max(args.warmup, 3)
            run_images_ours(args, rank, world, local_rank)
    elif args.workload == "sift":
        if args.impl == "reference":
            run_sift_reference(args, rank, world)
        else:
            args.warmup = max(args.warmup, 3)
            run_sift_ours(args, rank, world, local_rank)
    elif args.impl == "reference":
        run_reference(args, rank, world)
    elif cluster_partition_run:
        args.warmup = max(args.warmup, 3)
        run_ours_cluster_partition(args, rank, world, local_rank)
    else:
        args.warmup = max(args.warmup, 3)
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
