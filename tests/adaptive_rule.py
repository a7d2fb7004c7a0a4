"""numpy restatement of moped3d's depth-adaptive MATCH decision (moped_b200/csrc/adaptive_threshold.cuh) and of the match lists
MATCH_ADAPTIVE_CUDA::emit builds from it. float32 operations with the header's double promotions, every operation rounded once, so
the results are the header's bits (tests/test_match_adaptive_frames_host.py checks that against the header compiled by g++)."""
import numpy as np

F = np.float32


def ratio_curve(curves, model, depth, maximum_depth):
    """value of the curve of model[i] at depth[i] (depth may be a scalar)"""
    c = curves[np.asarray(model)]
    peak, fade, low, high = c["depth_peak"], c["depth_fade"], c["ratio_low"], c["ratio_high"]
    depth = np.broadcast_to(np.asarray(depth, np.float32), peak.shape)
    with np.errstate(all="ignore"):
        ramp = low + (depth / peak) * (high - low)
        twice = fade * F(2)
        down = ((twice - depth) / fade) * high
    out = np.where(depth < peak, ramp, np.where(depth < fade, high, np.where(depth < twice, down, F(0))))
    return np.where(depth > F(maximum_depth), F(0), out).astype(np.float32)


def cauchy_weight(fill, cauchy_scale):
    with np.errstate(all="ignore"):
        t = np.asarray(fill, np.float32) / F(cauchy_scale)
        return (1.0 / (1.0 + (t * t).astype(np.float64))).astype(np.float32)


def threshold(curves, model, depth, fill, maximum_depth, default_depth, cauchy_scale):
    w = cauchy_weight(fill, cauchy_scale)
    here = ratio_curve(curves, model, depth, maximum_depth)
    fallback = ratio_curve(curves, model, F(default_depth), maximum_depth)
    return ((w * here).astype(np.float64) + (1.0 + -w.astype(np.float64)) * fallback.astype(np.float64)).astype(np.float32)


def accept(curves, model, depth, fill, d0, d1, maximum_depth, default_depth, cauchy_scale):
    depth = np.asarray(depth, np.float32)
    with np.errstate(all="ignore"):
        ratio = np.asarray(d0, np.float32) / np.asarray(d1, np.float32)
    thr = threshold(curves, model, depth, fill, maximum_depth, default_depth, cauchy_scale)
    return ~(depth > F(maximum_depth)) & (ratio < thr)


def pixel(xy, width, height):
    """linear index of the pixel under each feature: truncation, the reference's clamp to [0, width] x [0, height], kept inside the map"""
    xy = np.asarray(xy, np.float32).reshape(-1, 2)
    x = np.clip(np.trunc(xy[:, 0]).astype(np.int64), 0, width)
    y = np.clip(np.trunc(xy[:, 1]).astype(np.int64), 0, height)
    return np.minimum(y * width + x, width * height - 1)


def finalize(nn_row, nn_dist, xy, depth, fill_distance, model_of_row, curves, depths=(4.0, 1.0, 0.1)):
    """accept flags of one frame from its nearest rows (what k_match_finalize_adaptive decides)"""
    nn_row, nn_dist = np.asarray(nn_row).reshape(-1, 2), np.asarray(nn_dist, np.float32).reshape(-1, 2)
    ok = (nn_row[:, 0] >= 0) & (nn_row[:, 1] >= 0)
    m = np.asarray(model_of_row)[np.where(ok, nn_row[:, 0], 0)]
    ok &= (m >= 0) & (m < len(curves))
    H, W = depth.shape
    px = pixel(xy, W, H)
    acc = accept(curves, np.where(ok, m, 0), depth.reshape(-1)[px], fill_distance.reshape(-1)[px], nn_dist[:, 0], nn_dist[:, 1], *depths)
    return ok & acc


def emit(nn_row, accepted, xy, image, model_of_row, db_xyz, n_models, base=0):
    """FrameData::matches after MATCH as flat model-major lists: offsets [n_models + 1] (from `base`), and per match its feature index
    (+ base), image, coord2D and the nearest row's coord3D; a model's matches in feature order."""
    idx = np.nonzero(np.asarray(accepted))[0]
    rows = np.asarray(nn_row).reshape(-1, 2)[idx, 0]
    m = np.asarray(model_of_row)[rows]
    order = np.argsort(m, kind="stable")
    idx, rows, m = idx[order], rows[order], m[order]
    offsets = (base + np.searchsorted(m, np.arange(n_models + 1), side="left")).astype(np.int32)
    return dict(offsets=offsets, feature=(base + idx).astype(np.int32), image=np.asarray(image, np.int32)[idx],
                xy=np.asarray(xy, np.float32).reshape(-1, 2)[idx], xyz=np.asarray(db_xyz, np.float32)[rows])


SEGMENTS = ("ramp", "plateau", "fade", "zero", "beyond")


def segment(curves, model, depth, maximum_depth):
    """index into SEGMENTS of the curve segment each (model, depth) falls in"""
    c = curves[np.asarray(model)]
    depth = np.asarray(depth, np.float32)
    s = np.where(depth < c["depth_peak"], 0, np.where(depth < c["depth_fade"], 1, np.where(depth < c["depth_fade"] * F(2), 2, 3)))
    return np.where(depth > F(maximum_depth), 4, s)
