"""The oracle's moped3d recognition steps chained like addCudaRecognition3d registers them (moped_b200/stages/pipeline3d_cuda.hpp;
moped3d/libmoped/src/config.hpp:45-49): CLUSTER (CLUSTER_LINKAGE_CPU per model) -> POSE -> FILTER -> POSE2 -> FILTER2, on FrameData as
DEPTHPROP leaves it. The RANSAC tasks draw from the seedable streams libmoped_cuda uses (task t of a POSE call: seed + 0x9E3779B97F4A7C15 *
(t + 1); seeds 1 and 2, mc_depth_pipeline_default_params), the samples break key ties by the match index inside the model (the LmData
address order pose_depth_cuda_base.hpp passes as tie ids). Test infrastructure: what mc_process_depth_frames* must reproduce bit for bit."""
import ctypes as C

import numpy as np

from oracle import oracle
from oracle_chain import filter_step

GOLDEN = 0x9E3779B97F4A7C15
M64 = 0xFFFFFFFFFFFFFFFF
CLUSTER = dict(cutoff=0.1, min_pts=7, use3d_filter=2, linkage_type=1, sigma2d=-1.0, sigma3d=-1.0)
POSE1 = (192, 100, 4, 5, 6, 8.0)          # (MaxRANSACTests, MaxLMTests, MaxObjectsPerCluster, NPtsAlign, MinNPtsObject, ErrorThreshold)
POSE2 = (64, 250, 4, 6, 8, 5.0)
ALPHA = 0.5
FILTER1 = (6, 4096.0, 2.0)
FILTER2 = (8, 8192.0, 1e-4)


def ransac_depth_tie(xy, xyz, world, cauchy, image, tie, cams, alpha, params, seed, variant=0):
    """mo_ransac_depth* with tie ids (the key tie-break of randSample); params as POSE1. Returns (found, pose, tests)."""
    n = len(xy)
    st = C.c_uint64(int(seed))
    pose = np.zeros(7, np.float32)
    it = C.c_int(0)
    tie = np.ascontiguousarray(tie, np.int32)
    fn = oracle.lib().mo_ransac_depth_v1 if variant else oracle.lib().mo_ransac_depth
    found = fn(C.byref(st), n, np.ascontiguousarray(xy, np.float32), np.ascontiguousarray(xyz, np.float32), np.ascontiguousarray(world, np.float32),
               np.ascontiguousarray(cauchy, np.float32), np.ascontiguousarray(image, np.int32), tie.ctypes.data, cams, alpha, int(params[0]),
               int(params[1]), int(params[3]), int(params[4]), float(params[5]), pose, C.byref(it))
    return bool(found), pose, it.value


def cluster_step(fr, cluster=CLUSTER):
    """CLUSTER_LINKAGE_CPU::process: every model with matches on its own, clusters model-major."""
    off = fr["match_offsets"]
    model, offsets, members = [], [0], []
    for m in range(len(off) - 1):
        lo, hi = int(off[m]), int(off[m + 1])
        if hi == lo:
            continue
        co, mem = oracle.cluster_linkage(fr["match_xy"][lo:hi], fr["match_xyz"][lo:hi], fr["match_world"][lo:hi], fr["depth"], fr["fill_distance"],
                                         **cluster)
        for c in range(len(co) - 1):
            model.append(m)
            members.append(mem[co[c]:co[c + 1]])
            offsets.append(offsets[-1] + int(co[c + 1] - co[c]))
    return dict(model=np.array(model, np.int32), offsets=np.array(offsets, np.int32),
                members=np.concatenate(members).astype(np.int32) if members else np.zeros(0, np.int32))


def pose_step(fr, clusters, cams, params, alpha, seed, objects, variant=0):
    """POSE_RANSAC_LM_DIFF_*_DEPTH_CUDA::process: tasks = every (cluster, try), found poses appended in task order."""
    off = fr["match_offsets"]
    cauchy = oracle.cauchy_weights(fr["match_fill"], variant)
    for task in range(len(clusters["model"]) * params[2]):
        k = task // params[2]
        m = int(clusters["model"][k])
        mem = clusters["members"][clusters["offsets"][k]:clusters["offsets"][k + 1]]
        j = int(off[m]) + mem
        f, p, _ = ransac_depth_tie(fr["match_xy"][j], fr["match_xyz"][j], fr["match_world"][j], cauchy[j], fr["match_image"][j], mem, cams, alpha,
                                   params, (seed + GOLDEN * (task + 1)) & M64, variant)
        if f:
            objects.append((m, p.copy()))


def frame(fr, variant=0, seeds=(1, 2), cluster=CLUSTER, pose1=POSE1, pose2=POSE2, filter1=FILTER1, filter2=FILTER2, clusters=None):
    """One make_depth_frame frame through the five steps -> dict(model, pose, score, clusters). `clusters` (optional, as cluster_step
    returns them) replaces the CLUSTER step: POSE..FILTER2 alone."""
    cams = oracle.cameras(fr["K"], fr["cam_pose"])
    matches = dict(offsets=fr["match_offsets"], image=fr["match_image"], xy=fr["match_xy"], xyz=fr["match_xyz"])
    cl = cluster_step(fr, cluster) if clusters is None else clusters
    objects = []
    pose_step(fr, cl, cams, pose1, ALPHA, seeds[0], objects, variant)
    objects, cl2, _ = filter_step(matches, cams, objects, filter1)
    pose_step(fr, cl2, cams, pose2, ALPHA, seeds[1], objects, variant)
    objects, _, score = filter_step(matches, cams, objects, filter2)
    return dict(model=np.array([o[0] for o in objects], np.int32),
                pose=np.stack([o[1] for o in objects]).astype(np.float32) if objects else np.zeros((0, 7), np.float32),
                score=np.asarray(score, np.float32), clusters=cl)
