"""Synthetic model databases and frames of the shape BASELINE.json names (SURVEY.md §8d).

There is no network for the reference's model set (moped2/download_models.sh wgets it), so every
configuration runs on seeded synthetic data:

* model DB: ``n_obj`` objects x ``pts_per_obj`` points; coord3D ~ U(-0.1, 0.1)^3 m; descriptor =
  SIFT-like non-negative 128-d (16 cells x 8 bins ~ Gamma(0.5), L2-normalise, clip 0.2, renormalise —
  the post-processing of libs.tgz!libsiftfast-1.1-src/libsiftfast.cpp:1504-1515).
* frame: 640x480, K=(800,800,320,240), identity camera (moped2/moped_test.cpp:187-188);
  ``n_visible`` objects posed in front of the camera, ``pts_visible`` of their points projected with
  N(0, 0.5 px) noise and N(0, 0.02) descriptor noise; the rest of the Q features are distractors.

Pure numpy (make_adaptive_frames also calls the library's host-side mc_adaptive_model_init); used by tests/ and bench.py (inputs
only — no algorithm of the hot path lives here).
"""
from __future__ import annotations

import numpy as np

BASE_SEED = 20261017
K_DEFAULT = np.array([800.0, 800.0, 320.0, 240.0], dtype=np.float32)
CAM_IDENTITY = np.array([0, 0, 0, 1, 0, 0, 0], dtype=np.float32)  # quat (x,y,z,w) + t


def sift_like(rng: np.random.Generator, n: int, d: int = 128) -> np.ndarray:
    x = rng.gamma(0.5, 1.0, size=(n, d)).astype(np.float32)
    x /= np.linalg.norm(x, axis=1, keepdims=True)
    np.minimum(x, 0.2, out=x)
    x /= np.linalg.norm(x, axis=1, keepdims=True)
    return x.astype(np.float32)


def make_db(n_obj: int, pts_per_obj: int = 1000, d: int = 128, seed: int = BASE_SEED, ragged: bool = False):
    """Returns dict(n_pts[int32 n_obj], xyz[N,3], desc[N,d], model_of_row[int32 N])."""
    rng = np.random.default_rng(seed)
    if ragged:
        n_pts = rng.integers(max(8, pts_per_obj * 6 // 10), pts_per_obj * 3 + 1, size=n_obj).astype(np.int32)
    else:
        n_pts = np.full(n_obj, pts_per_obj, dtype=np.int32)
    n = int(n_pts.sum())
    xyz = rng.uniform(-0.1, 0.1, size=(n, 3)).astype(np.float32)
    desc = np.empty((n, d), dtype=np.float32)
    step = 1 << 16
    for s in range(0, n, step):
        desc[s:s + step] = sift_like(rng, min(step, n - s), d)
    model_of_row = np.repeat(np.arange(n_obj, dtype=np.int32), n_pts)
    return dict(n_pts=n_pts, xyz=xyz, desc=desc, model_of_row=model_of_row)


def quat_to_R(q: np.ndarray) -> np.ndarray:
    x, y, z, w = [float(v) for v in q]
    return np.array([
        [1 - 2 * y * y - 2 * z * z, 2 * x * y - 2 * w * z, 2 * x * z + 2 * w * y],
        [2 * x * y + 2 * w * z, 1 - 2 * x * x - 2 * z * z, 2 * y * z - 2 * w * x],
        [2 * x * z - 2 * w * y, 2 * y * z + 2 * w * x, 1 - 2 * x * x - 2 * y * y]], dtype=np.float64)


def make_frame(db, q_feats: int = 2000, n_visible: int = 8, pts_visible: int = 60, frame_id: int = 0,
               seed: int = BASE_SEED, image_idx: int = 0, K: np.ndarray = K_DEFAULT,
               pix_noise: float = 0.5, desc_noise: float = 0.02, objects=None):
    """Returns dict(desc[Q,d], xy[Q,2], image_idx[int32 Q], gt_model[int32 V], gt_pose[V,7], src_row[int32 Q])."""
    rng = np.random.default_rng(seed + 7919 * (frame_id + 1))
    n_obj = len(db["n_pts"])
    d = db["desc"].shape[1]
    starts = np.concatenate([[0], np.cumsum(db["n_pts"])])
    if objects is None:
        objects = rng.choice(n_obj, size=min(n_visible, n_obj), replace=False)
    descs, xys, src = [], [], []
    poses = []
    for o in objects:
        q = rng.normal(size=4)
        q /= np.linalg.norm(q)
        t = np.array([rng.uniform(-0.3, 0.3), rng.uniform(-0.2, 0.2), rng.uniform(0.6, 1.4)])
        poses.append(np.concatenate([q, t]).astype(np.float32))
        R = quat_to_R(q)
        npts = int(db["n_pts"][o])
        rows = starts[o] + rng.choice(npts, size=min(pts_visible, npts), replace=False)
        X = db["xyz"][rows].astype(np.float64) @ R.T + t
        u = X[:, 0] / X[:, 2] * K[0] + K[2] + rng.normal(0, pix_noise, size=len(rows))
        v = X[:, 1] / X[:, 2] * K[1] + K[3] + rng.normal(0, pix_noise, size=len(rows))
        dd = db["desc"][rows] + rng.normal(0, desc_noise, size=(len(rows), d)).astype(np.float32)
        np.maximum(dd, 0, out=dd)
        dd /= np.linalg.norm(dd, axis=1, keepdims=True)
        descs.append(dd.astype(np.float32))
        xys.append(np.stack([u, v], axis=1).astype(np.float32))
        src.append(rows.astype(np.int32))
    n_planted = sum(len(x) for x in descs)
    n_dis = max(0, q_feats - n_planted)
    descs.append(sift_like(rng, n_dis, d))
    xys.append(np.stack([rng.uniform(0, 640, n_dis), rng.uniform(0, 480, n_dis)], axis=1).astype(np.float32))
    src.append(np.full(n_dis, -1, dtype=np.int32))
    desc = np.concatenate(descs)[:q_feats]
    xy = np.concatenate(xys)[:q_feats]
    src_row = np.concatenate(src)[:q_feats]
    perm = rng.permutation(len(desc))
    return dict(desc=np.ascontiguousarray(desc[perm]), xy=np.ascontiguousarray(xy[perm]),
                image_idx=np.full(len(desc), image_idx, dtype=np.int32),
                gt_model=np.asarray(objects, dtype=np.int32), gt_pose=np.stack(poses) if poses else np.zeros((0, 7), np.float32),
                src_row=np.ascontiguousarray(src_row[perm]))


def make_ransac_clusters(n_clusters: int = 64, pts: int = 80, outlier_frac: float = 0.5, seed: int = BASE_SEED,
                         K: np.ndarray = K_DEFAULT, pix_noise: float = 0.5):
    """RANSAC-heavy config (BASELINE.json configs[3]): n_clusters clusters of `pts` 2D-3D
    correspondences, `outlier_frac` of them uniform-pixel outliers. One model per cluster.
    Returns dict(offsets[int32 n+1], xy[M,2], xyz[M,3], image[int32 M], gt_pose[n,7])."""
    rng = np.random.default_rng(seed + 104729)
    xy, xyz, poses = [], [], []
    for _ in range(n_clusters):
        q = rng.normal(size=4)
        q /= np.linalg.norm(q)
        t = np.array([rng.uniform(-0.3, 0.3), rng.uniform(-0.2, 0.2), rng.uniform(0.6, 1.4)])
        R = quat_to_R(q)
        X = rng.uniform(-0.1, 0.1, size=(pts, 3))
        Xc = X @ R.T + t
        u = Xc[:, 0] / Xc[:, 2] * K[0] + K[2] + rng.normal(0, pix_noise, pts)
        v = Xc[:, 1] / Xc[:, 2] * K[1] + K[3] + rng.normal(0, pix_noise, pts)
        n_out = int(round(pts * outlier_frac))
        out = rng.choice(pts, size=n_out, replace=False)
        u[out] = rng.uniform(0, 640, n_out)
        v[out] = rng.uniform(0, 480, n_out)
        xy.append(np.stack([u, v], axis=1))
        xyz.append(X)
        poses.append(np.concatenate([q, t]))
    offsets = (np.arange(n_clusters + 1) * pts).astype(np.int32)
    return dict(offsets=offsets, xy=np.concatenate(xy).astype(np.float32), xyz=np.concatenate(xyz).astype(np.float32),
                image=np.zeros(n_clusters * pts, dtype=np.int32), gt_pose=np.stack(poses).astype(np.float32))


def make_hypotheses(cl, n_hyp_per_cluster: int = 2048, n_pts_align: int = 5, seed: int = BASE_SEED):
    """Explicit RANSAC hypotheses for `make_ransac_clusters` output: per cluster n_hyp_per_cluster sample sets of
    n_pts_align DISTINCT point positions and an initial quaternion with components k/256 (what initPose draws,
    POSE_RANSAC_LM_DIFF_REPROJECTION_CPU.hpp:182-186). Inputs only: the parity tests draw their sets with the
    oracle's RNG stream instead. Returns dict(hyp_cluster[int32 H], sample_pos[int32 H,n], init_quat[H,4])."""
    rng = np.random.default_rng(seed + 15485863)
    n_clusters = len(cl["offsets"]) - 1
    hc, sp = [], []
    for c in range(n_clusters):
        n = int(cl["offsets"][c + 1] - cl["offsets"][c])
        keys = rng.random((n_hyp_per_cluster, n))
        sp.append(np.argsort(keys, axis=1)[:, :n_pts_align].astype(np.int32))
        hc.append(np.full(n_hyp_per_cluster, c, np.int32))
    H = n_clusters * n_hyp_per_cluster
    quat = (rng.integers(0, 256, size=(H, 4)) / 256.0).astype(np.float32)
    quat[(quat == 0).all(axis=1)] = np.array([0, 0, 0, 0.5], np.float32)
    return dict(hyp_cluster=np.concatenate(hc), sample_pos=np.ascontiguousarray(np.concatenate(sp)), init_quat=quat)


def make_image(seed: int = 0, height: int = 480, width: int = 640, n_blobs: int = 2600) -> np.ndarray:
    """A synthetic grey 640x480 frame for the feature-extraction workload: Gaussian blobs of random size, sign and
    contrast over a smooth background — blob-like structure at many scales, ~2k SIFT keypoints (BASELINE: 2k feats/frame)."""
    rng = np.random.default_rng(BASE_SEED + 7919 * seed + 13)
    im = np.zeros((height, width), np.float32)
    yy, xx = np.mgrid[0:height, 0:width].astype(np.float32)
    im += 0.15 * np.sin(xx / 97.0 + rng.uniform(0, 6)) * np.cos(yy / 71.0 + rng.uniform(0, 6))
    for _ in range(n_blobs):
        cy, cx = rng.uniform(0, height), rng.uniform(0, width)
        s = float(np.exp(rng.uniform(np.log(1.0), np.log(6.0))))
        a = rng.uniform(0.08, 0.3) * rng.choice([-1.0, 1.0])
        r = int(4 * s) + 1
        y0, y1, x0, x1 = max(0, int(cy) - r), min(height, int(cy) + r + 1), max(0, int(cx) - r), min(width, int(cx) + r + 1)
        e = rng.uniform(0.6, 1.6)
        im[y0:y1, x0:x1] += a * np.exp(-(((yy[y0:y1, x0:x1] - cy) * e) ** 2 + ((xx[y0:y1, x0:x1] - cx) / e) ** 2) / (2 * s * s))
    im = np.clip(0.5 + im, 0.0, 1.0)
    return (im * 255.0 + 0.5).astype(np.uint8)


# ---- moped3d (RGB-D) inputs: depth-aware pose stages and linkage clustering (SURVEY.md 8f row 4) ----------------------------
K_DEPTH = np.array([525.0, 525.0, 319.5, 239.5], dtype=np.float32)      # a Kinect-like camera


def make_depth_clusters(n_clusters: int = 64, pts: int = 80, outlier_frac: float = 0.5, cauchy_scale: float = 0.100, seed: int = BASE_SEED):
    """Clusters for moped3d's depth-aware pose stages: model points under a planted pose seen by the identity camera; coord2D =
    projection + pixel noise, world3D = the camera-frame point with depth noise growing with depth^2, fill distances mostly 0
    (measured depth) and sometimes up to 0.3 (hallucinated); cauchy = 1 / (1 + (fill / cauchy_scale)^2), the weight the stage
    class computes per match (POSE_RANSAC_LM_DIFF_BACKPROJECTION_DEPTH_CPU.hpp:187-190; scale 25 for the reprojection variant).
    Returns dict(offsets, xy, xyz, world, fill, cauchy, image, gt_pose)."""
    rng = np.random.default_rng(seed + 32452843)
    xy, xyz, world, cauchy, poses, fills = [], [], [], [], [], []
    K = K_DEPTH
    for _ in range(n_clusters):
        q = rng.normal(size=4)
        q /= np.linalg.norm(q)
        t = np.array([rng.uniform(-0.2, 0.2), rng.uniform(-0.15, 0.15), rng.uniform(0.6, 1.2)])
        X = rng.uniform(-0.08, 0.08, size=(pts, 3))
        cam3 = X @ quat_to_R(q).T + t
        uv = np.stack([cam3[:, 0] / cam3[:, 2] * K[0] + K[2], cam3[:, 1] / cam3[:, 2] * K[1] + K[3]], 1) + rng.normal(0, 0.4, (pts, 2))
        w = cam3 * (1 + rng.normal(0, 0.0035, (pts, 1)) * cam3[:, 2:3])
        bad = rng.random(pts) < outlier_frac
        uv[bad] = rng.uniform([0, 0], [640, 480], (int(bad.sum()), 2))
        w[bad] = w[bad] + rng.normal(0, 0.2, (int(bad.sum()), 3))
        fill = np.where(rng.random(pts) < 0.7, 0.0, rng.uniform(0, 0.3, pts)).astype(np.float32)
        f = fill / np.float32(cauchy_scale)
        xy.append(uv); xyz.append(X); world.append(w); cauchy.append((1.0 / (1 + f * f)).astype(np.float32)); fills.append(fill)
        poses.append(np.concatenate([q, t]))
    offsets = (np.arange(n_clusters + 1) * pts).astype(np.int32)
    return dict(offsets=offsets, xy=np.concatenate(xy).astype(np.float32), xyz=np.concatenate(xyz).astype(np.float32),
                world=np.concatenate(world).astype(np.float32), fill=np.concatenate(fills).astype(np.float32), cauchy=np.concatenate(cauchy).astype(np.float32),
                image=np.zeros(n_clusters * pts, dtype=np.int32), gt_pose=np.stack(poses).astype(np.float32))


def make_linkage_scene(seed: int = 1, n_per=(300, 200), n_out: int = 100, hallucinated: float = 0.2, W: int = 320, H: int = 240):
    """Matches of ONE model seen twice (two instances at different places and depths) plus outliers, a 320x240 depth map with the
    two instances as fronto-parallel patches over a slanted background, and its fill-distance map (0 = measured depth): the input
    of moped3d's CLUSTER_LINKAGE_CPU::process for one model. Returns (xy, xyz, world, depth, distance)."""
    rng = np.random.default_rng(BASE_SEED + 977 * seed)
    K = K_DEPTH * np.float32(0.5)
    depth = (1.6 + 0.002 * np.arange(W)[None, :] + 0.001 * np.arange(H)[:, None]).astype(np.float32)
    dist = np.zeros((H, W), np.float32)
    xy, xyz, world = [], [], []
    for k, n in enumerate(n_per):
        cx, cy = (90 + 140 * k + rng.uniform(-10, 10), 110 + rng.uniform(-20, 20))
        z = 0.8 + 0.35 * k
        half = 38
        depth[int(cy) - half:int(cy) + half, int(cx) - half:int(cx) + half] = z
        pts = rng.uniform(-0.07, 0.07, (n, 3)).astype(np.float32)
        u = cx + pts[:, 0] * K[0] / z + rng.normal(0, 0.3, n)
        v = cy + pts[:, 1] * K[1] / z + rng.normal(0, 0.3, n)
        zz = z + pts[:, 2] * 0.1
        xy.append(np.stack([u, v], 1)); xyz.append(pts)
        world.append(np.stack([(u - K[2]) / K[0] * zz, (v - K[3]) / K[1] * zz, zz], 1))
    ou = rng.uniform([5, 5], [W - 5, H - 5], (n_out, 2))
    xy.append(ou); xyz.append(rng.uniform(-0.07, 0.07, (n_out, 3)))
    oz = depth[ou[:, 1].astype(int), ou[:, 0].astype(int)]
    world.append(np.stack([(ou[:, 0] - K[2]) / K[0] * oz, (ou[:, 1] - K[3]) / K[1] * oz, oz], 1))
    xy, xyz, world = (np.concatenate(a).astype(np.float32) for a in (xy, xyz, world))
    holes = rng.random((H, W)) < hallucinated
    dist[holes] = rng.uniform(1, 40, int(holes.sum())).astype(np.float32)
    perm = rng.permutation(len(xy))
    return xy[perm], xyz[perm], world[perm], depth, dist


def duplicate_matches(arrays, k: int, seed: int = 0):
    """Per-match arrays (same length) with k of their rows overwritten by copies of k other rows: what SIFT's secondary orientation
    peaks give, two matches of one model with the same pixel, model point and world point. Every copied pair makes get3DFilterK's
    |dm - dw| / dm a 0/0, i.e. two NaN entries of the similarity matrix. Returns new arrays."""
    n = len(arrays[0])
    assert 2 * k <= n, (k, n)
    perm = np.random.default_rng(BASE_SEED + 7919 * seed).permutation(n)
    dst, src = perm[:k], perm[k:2 * k]
    out = [np.array(a, copy=True) for a in arrays]
    for a in out:
        a[dst] = a[src]
    return out


def make_filter_depth_scene(seed: int = 1, n_models: int = 3, pts_per_model: int = 120, W: int = 320, H: int = 240, n_wrong: int = 2):
    """A frame state for moped3d's FILTER_PROJECTION_DEPTH step (inputs only): `n_models` box-like models (keypoints on a 12 cm cube), each
    seen once at a true pose in front of a Kinect-like camera, with a depth map that shows the objects as patches at their true depth over a
    far background, a fill-distance map with holes (> 0 = hallucinated depth), matches of every model (true correspondences + outliers)
    and an object list holding, per model, the true pose (slightly perturbed), a copy of it that competes for the same features and
    `n_wrong` poses floating in free space in front of the background (what the depth penalty is there to reject).
    Returns a dict of flat arrays in the C-ABI layout."""
    rng = np.random.default_rng(BASE_SEED + 977 * seed)
    K = np.array([262.0, 262.0, W / 2.0, H / 2.0], np.float32)
    depth = np.full((H, W), 2.5, np.float32) + (0.0005 * np.arange(W)[None, :]).astype(np.float32)
    fill = np.zeros((H, W), np.float32)
    model_xyz, model_off = [], [0]
    m_off, m_xy, m_xyz = [0], [], []
    obj_model, obj_pose = [], []
    for m in range(n_models):
        pts = rng.uniform(-0.06, 0.06, (pts_per_model + 17 * m, 3)).astype(np.float32)
        model_xyz.append(pts)
        model_off.append(model_off[-1] + len(pts))
        q = rng.normal(size=4)
        q /= np.linalg.norm(q)
        t = np.array([-0.35 + 0.35 * m + rng.uniform(-0.03, 0.03), rng.uniform(-0.1, 0.1), 0.9 + 0.25 * m], np.float64)
        R = quat_to_R(q.astype(np.float32)).astype(np.float64)
        cam = pts.astype(np.float64) @ R.T + t
        u = cam[:, 0] / cam[:, 2] * K[0] + K[2]
        v = cam[:, 1] / cam[:, 2] * K[1] + K[3]
        cu, cv = int(np.clip(u.mean(), 45, W - 45)), int(np.clip(v.mean(), 45, H - 45))
        depth[cv - 40:cv + 40, cu - 40:cu + 40] = np.float32(t[2] - 0.02)
        seen = rng.random(len(pts)) < 0.5                                  # half of the keypoints are matched
        n_seen = int(seen.sum())
        xy = np.stack([u[seen] + rng.normal(0, 0.4, n_seen), v[seen] + rng.normal(0, 0.4, n_seen)], 1)
        n_out = 12
        xy = np.concatenate([xy, rng.uniform([5, 5], [W - 5, H - 5], (n_out, 2))])
        xyz = np.concatenate([pts[seen], rng.uniform(-0.06, 0.06, (n_out, 3)).astype(np.float32)])
        perm = rng.permutation(len(xy))
        m_xy.append(xy[perm]); m_xyz.append(xyz[perm])
        m_off.append(m_off[-1] + len(xy))
        true_pose = np.concatenate([q, t]).astype(np.float32)
        near = true_pose.copy(); near[4:] += rng.normal(0, 0.002, 3).astype(np.float32)
        obj_model += [m, m]
        obj_pose += [true_pose, near]
        for _ in range(n_wrong):                                            # same view direction, 60 cm in front of where the depth map says anything is
            w = true_pose.copy()
            w[4:] = (t * (0.35 / t[2])).astype(np.float32) + rng.normal(0, 0.01, 3).astype(np.float32)
            obj_model.append(m); obj_pose.append(w)
    holes = rng.random((H, W)) < 0.15
    fill[holes] = rng.uniform(1, 30, int(holes.sum())).astype(np.float32)
    order = rng.permutation(len(obj_model))                                 # the object list is not model-major
    return dict(K=K, cam_pose=CAM_IDENTITY.copy(), depth_K=K.copy(), depth_pose=CAM_IDENTITY.copy(), depth=depth, fill=fill, width=W, height=H,
                model_offsets=np.array(model_off, np.int32), model_xyz=np.concatenate(model_xyz).astype(np.float32),
                match_offsets=np.array(m_off, np.int32), match_xy=np.concatenate(m_xy).astype(np.float32),
                match_xyz=np.concatenate(m_xyz).astype(np.float32), match_image=np.zeros(m_off[-1], np.int32),
                obj_model=np.array(obj_model, np.int32)[order], obj_pose=np.stack(obj_pose).astype(np.float32)[order])


def make_depth_frame(seed: int = 1, n_models: int = 12, W: int = 640, H: int = 480, pts_per_model: int = 160, outlier_frac: float = 0.15,
                     inst_matches=(40, 71), dup_frac: float = 0.0):
    """One 640x480 RGB-D frame of moped3d's recognition steps in the C-ABI layout of mc_process_depth_frames (FrameData after DEPTHPROP,
    identity camera, Kinect-like K): about a third of the `n_models` models are seen once or twice at planted poses (40-70 matched
    keypoints each, `outlier_frac` of them at random pixels with wrong depth), a few models get a handful of junk matches (3-6, too few
    to form a cluster) and the rest none. The depth map shows every instance as a patch at its depth over a slanted background; the
    fill-distance map has holes (> 0 = hallucinated depth). A model's matches come in random (query) order, instances interleaved.
    Returns dict(match_offsets[n_models+1], match_image, match_xy, match_xyz, match_world, match_fill, depth[H,W], fill_distance[H,W],
    K, cam_pose, gt_model[V], gt_pose[V,7], junk_models, model_offsets[n_models+1], model_xyz) — the last two are every model's keypoints
    (model-major), where FILTER_PROJECTION_DEPTH draws its test points from.
    `inst_matches` = [lo, hi) of the matched keypoints per instance (at most `pts_per_model`); with `dup_frac` > 0, that fraction of every
    model's matches are copies of other matches of the model (duplicate_matches: same pixel, model point, world point and fill)."""
    rng = np.random.default_rng(BASE_SEED + 6151 * seed)
    K = K_DEPTH
    depth = (2.2 + 0.0006 * np.arange(W)[None, :] + 0.0004 * np.arange(H)[:, None]).astype(np.float32)
    fill_map = np.zeros((H, W), np.float32)
    holes = rng.random((H, W)) < 0.15
    fill_map[holes] = rng.uniform(1, 40, int(holes.sum())).astype(np.float32)
    model_pts = [np.random.default_rng(BASE_SEED + 31 * m).uniform(-0.06, 0.06, (pts_per_model, 3)) for m in range(n_models)]
    order = rng.permutation(n_models)
    n_seen = max(1, n_models // 3)
    seen, junk = order[:n_seen], order[n_seen:n_seen + max(1, n_models // 4)]
    cells = [(c, r) for r in range(3) for c in range(4)]                      # 160 x 160 cells: instances never overlap
    free = list(rng.permutation(len(cells)))
    per_model = {m: [] for m in range(n_models)}
    gt_model, gt_pose = [], []
    for m in seen:
        for _ in range(1 if rng.random() < 0.6 or len(free) < 2 else 2):
            if not free:
                break
            c, r = cells[free.pop()]
            cx, cy = 80 + 160 * c + rng.uniform(-15, 15), 80 + 160 * r + rng.uniform(-15, 15)
            z = rng.uniform(0.7, 1.1)
            t = np.array([(cx - K[2]) / K[0] * z, (cy - K[3]) / K[1] * z, z])
            q = rng.normal(size=4)
            q /= np.linalg.norm(q)
            n = int(rng.integers(*inst_matches))
            X = model_pts[m][rng.choice(pts_per_model, n, replace=False)]
            cam3 = X @ quat_to_R(q).T + t
            uv = np.stack([cam3[:, 0] / cam3[:, 2] * K[0] + K[2], cam3[:, 1] / cam3[:, 2] * K[1] + K[3]], 1) + rng.normal(0, 0.4, (n, 2))
            w = cam3 * (1 + rng.normal(0, 0.0035, (n, 1)) * cam3[:, 2:3])
            bad = rng.random(n) < outlier_frac
            uv[bad] = rng.uniform([0, 0], [W - 1, H - 1], (int(bad.sum()), 2))
            uv = np.clip(uv, 0.5, [W - 1.5, H - 1.5])
            w[bad] = w[bad] + rng.normal(0, 0.2, (int(bad.sum()), 3))
            half = 45
            depth[max(0, int(cy) - half):int(cy) + half, max(0, int(cx) - half):int(cx) + half] = np.float32(z)
            per_model[m].append((uv, X, w))
            gt_model.append(int(m)); gt_pose.append(np.concatenate([q, t]).astype(np.float32))
    for m in junk:
        n = int(rng.integers(3, 7))
        uv = rng.uniform([0, 0], [W - 1, H - 1], (n, 2))
        X = model_pts[m][rng.choice(pts_per_model, n, replace=False)]
        zz = depth[uv[:, 1].astype(int), uv[:, 0].astype(int)][:, None]
        w = np.concatenate([(uv - K[2:4]) / K[0:2] * zz, zz], 1)
        per_model[m].append((uv, X, w))
    offs, xy, xyz, world = [0], [], [], []
    for m in range(n_models):
        if per_model[m]:
            uv = np.concatenate([a[0] for a in per_model[m]]); X = np.concatenate([a[1] for a in per_model[m]])
            w = np.concatenate([a[2] for a in per_model[m]])
            perm = rng.permutation(len(uv))
            xy.append(uv[perm]); xyz.append(X[perm]); world.append(w[perm])
        offs.append(offs[-1] + (len(xy[-1]) if per_model[m] else 0))
    M = offs[-1]
    cat = lambda a, k: (np.concatenate(a) if a else np.zeros((0, k))).astype(np.float32)
    fill = np.where(rng.random(M) < 0.7, 0.0, rng.uniform(0, 0.3, M)).astype(np.float32)
    xy, xyz, world = cat(xy, 2), cat(xyz, 3), cat(world, 3)
    if dup_frac > 0:
        for m in range(n_models):
            lo, hi = offs[m], offs[m + 1]
            k = int(round(dup_frac * (hi - lo)))
            if k and 2 * k <= hi - lo:
                xy[lo:hi], xyz[lo:hi], world[lo:hi], fill[lo:hi] = duplicate_matches((xy[lo:hi], xyz[lo:hi], world[lo:hi], fill[lo:hi]), k,
                                                                                     seed=6151 * seed + m)
    return dict(match_offsets=np.array(offs, np.int32), match_image=np.zeros(M, np.int32), match_xy=xy, match_xyz=xyz,
                match_world=world, match_fill=fill, depth=depth, fill_distance=fill_map, K=K.copy(), cam_pose=CAM_IDENTITY.copy(),
                gt_model=np.array(gt_model, np.int32), gt_pose=np.stack(gt_pose) if gt_pose else np.zeros((0, 7), np.float32),
                junk_models=np.sort(junk).astype(np.int32), model_offsets=(pts_per_model * np.arange(n_models + 1)).astype(np.int32),
                model_xyz=np.concatenate(model_pts).astype(np.float32))


def stack_depth_frames(frames):
    """Frames of make_depth_frame -> the batch layout of mc_process_depth_frames: match_offsets [n_frames, n_models+1] as global
    indices into the concatenated per-match arrays, depth / fill_distance [n_frames, H, W]."""
    base, rows = 0, []
    for fr in frames:
        rows.append(fr["match_offsets"] + base)
        base += int(fr["match_offsets"][-1])
    cat = lambda k: np.concatenate([fr[k] for fr in frames])
    return dict(match_offsets=np.stack(rows).astype(np.int32), match_image=cat("match_image"), match_xy=cat("match_xy"), match_xyz=cat("match_xyz"),
                match_world=cat("match_world"), match_fill=cat("match_fill"), depth=np.stack([fr["depth"] for fr in frames]),
                fill_distance=np.stack([fr["fill_distance"] for fr in frames]))


# ---- moped3d's depth-adaptive MATCH step (MATCH_ADAPTIVE_FLANN_CPU) on frame batches -------------------------------------------------
# DimensionPeak / DimensionFade of the generator's curves. The pipeline's 150 / 50 px put twice the fade depth of make_db's 0.2 m models
# (4.2 m) beyond the 4 m depth cut, which would leave the curve's zero segment in front of the cut empty; 80 px puts it at ~2.6 m.
ADAPTIVE_DIMENSIONS = (150.0, 80.0)


def adaptive_segments(curves, maximum_depth: float = 4.0):
    """Depth intervals (lo, hi) inside the segments of ALL curves: ramp, plateau, fade, zero (beyond twice the fade depth, within
    maximum_depth) and beyond maximum_depth, each kept clear of every curve's breakpoints by a few per cent. Empty segments are left out."""
    pk_lo, pk_hi = float(curves["depth_peak"].min()), float(curves["depth_peak"].max())
    fd_lo, fd_hi = float(curves["depth_fade"].min()), float(curves["depth_fade"].max())
    seg = dict(ramp=(0.05, 0.95 * pk_lo), plateau=(1.05 * pk_hi, 0.95 * fd_lo), fade=(1.05 * fd_hi, 1.95 * fd_lo),
               zero=(2.05 * fd_hi, 0.98 * maximum_depth), beyond=(1.02 * maximum_depth, 2.0 * maximum_depth))
    return {k: v for k, v in seg.items() if v[1] > v[0]}


def make_adaptive_frames(db, n_frames: int, n_features=None, seed: int = BASE_SEED, empty=(1,), far=(2,), W: int = 640, H: int = 480,
                         maximum_depth: float = 4.0, cauchy_scale: float = 0.1, dimensions=ADAPTIVE_DIMENSIONS):
    """A batch of RGB-D frames for moped3d's MATCH step (mc_match_adaptive_frames), built on make_db / make_frame.
    * features: make_frame's planted copies of database rows and distractors, pixel coordinates clipped into the W x H map; frame f has
      `n_features` features (int, or per-frame counts; None = seeded counts in 300..2500, none a multiple of 256), frames listed in
      `empty` have none;
    * depth planes: 80 x 80 px cells, each at one depth drawn from a segment of the ratio curves (adaptive_segments: ramp, plateau,
      fade, zero, beyond maximum_depth) plus a 1 mm ramp; frames listed in `far` lie entirely beyond maximum_depth;
    * fill-distance planes: half the pixels 0 (measured depth), the rest log-uniform in 10^-2.5 .. 10^1.5 m, so the Cauchy weight of
      the fill distance goes from 1 down to ~1e-5;
    * curves: mc_adaptive_model_init over each model's bounding box with K_DEPTH, the moped3d ratio ranges and `dimensions`;
    * world / fill per feature: the depth under the feature back-projected through K_DEPTH and the fill distance under it (what
      DEPTHPROP gives moped3d's later steps).
    Returns dict(desc[Q,d], xy[Q,2], image[Q], frame_offsets[n_frames+1], depth[F,H,W], fill_distance[F,H,W], world[Q,3], fill[Q],
    curves (capi.ADAPTIVE_MODEL records), segments, maximum_depth, cauchy_scale)."""
    from . import capi
    rng = np.random.default_rng(seed + 15731)
    starts = np.concatenate([[0], np.cumsum(db["n_pts"])]).astype(np.int64)
    lo = np.minimum.reduceat(db["xyz"], starts[:-1], axis=0)
    hi = np.maximum.reduceat(db["xyz"], starts[:-1], axis=0)
    p = capi.ADAPTIVE_DEFAULTS
    curves = capi.adaptive_model_init(lo, hi, K_DEPTH, db["n_pts"], (p[0], p[1], p[2], p[3], dimensions[0], dimensions[1]))
    segs = adaptive_segments(curves, maximum_depth)
    kinds = list(segs)
    if n_features is None:
        counts = rng.integers(300, 2501, size=n_frames)
        counts[counts % 256 == 0] += 1
    else:
        counts = np.broadcast_to(np.asarray(n_features, np.int64), (n_frames,)).copy()
    counts[[f for f in empty if f < n_frames]] = 0
    desc, xy, depth, fill_map = [], [], np.empty((n_frames, H, W), np.float32), np.empty((n_frames, H, W), np.float32)
    cy, cx = np.arange(H)[:, None] // 80, np.arange(W)[None, :] // 80
    ramp = (0.001 * (np.arange(W)[None, :] % 80) / 80).astype(np.float32)
    for f in range(n_frames):
        cells = rng.integers(0, len(kinds), size=((H + 79) // 80, (W + 79) // 80))
        if f in far:
            cells[:] = kinds.index("beyond")
        bounds = np.array([segs[k] for k in kinds])[cells]
        zc = rng.uniform(bounds[..., 0], bounds[..., 1]).astype(np.float32)
        depth[f] = zc[cy, cx] + ramp
        measured = rng.random((H, W)) < 0.5
        fill_map[f] = np.where(measured, 0.0, 10.0 ** rng.uniform(-2.5, 1.5, (H, W))).astype(np.float32)
        n = int(counts[f])
        if n:
            fr = make_frame(db, n, n_visible=8, pts_visible=60, frame_id=f, seed=seed)
            desc.append(fr["desc"])
            xy.append(np.clip(fr["xy"], 0, [W - 1, H - 1]).astype(np.float32))
    d = db["desc"].shape[1]
    desc = np.concatenate(desc) if desc else np.zeros((0, d), np.float32)
    xy = np.concatenate(xy) if xy else np.zeros((0, 2), np.float32)
    offsets = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    frame_of = np.repeat(np.arange(n_frames), counts)
    px, py = xy[:, 0].astype(np.int64), xy[:, 1].astype(np.int64)
    zf = depth[frame_of, py, px]
    world = np.stack([(xy[:, 0] - K_DEPTH[2]) / K_DEPTH[0] * zf, (xy[:, 1] - K_DEPTH[3]) / K_DEPTH[1] * zf, zf], 1).astype(np.float32)
    return dict(desc=np.ascontiguousarray(desc, np.float32), xy=xy, image=np.zeros(len(desc), np.int32), frame_offsets=offsets, depth=depth,
                fill_distance=fill_map, world=world, fill=fill_map[frame_of, py, px].astype(np.float32), curves=curves, segments=segs,
                maximum_depth=float(maximum_depth), cauchy_scale=float(cauchy_scale))
