"""moped3d's depth-adaptive MATCH decision without a GPU: the numpy restatement the GPU tests compare against (tests/adaptive_rule.py)
equals moped_b200/csrc/adaptive_threshold.cuh bit for bit — the header the device kernel compiles, here built by g++ -ffp-contract=off
through tests/cpp/adaptive_host.cpp — on random inputs and on the edges: every breakpoint of the curves, depths beyond maximum_depth,
fill distances of 0 and very large, and pixels at x == width / y == height. Also checks that synth.make_adaptive_frames covers every
segment of the curves."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import adaptive_rule as R
from moped_b200 import capi, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_f32p = np.ctypeslib.ndpointer(dtype=np.float32, flags="C_CONTIGUOUS")
_i32p = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
_u8p = np.ctypeslib.ndpointer(dtype=np.uint8, flags="C_CONTIGUOUS")
DEPTHS = capi.ADAPTIVE_DEPTHS


@pytest.fixture(scope="module")
def host_lib():
    out_dir = os.path.join(ROOT, "tests", "_build")
    os.makedirs(out_dir, exist_ok=True)
    out = os.path.join(out_dir, "libadaptive_host.so")
    src = os.path.join(ROOT, "tests", "cpp", "adaptive_host.cpp")
    deps = [src, os.path.join(ROOT, "moped_b200", "csrc", "adaptive_threshold.cuh"), os.path.join(ROOT, "include", "moped_cuda.h")]
    if not os.path.exists(out) or any(os.path.getmtime(d) > os.path.getmtime(out) for d in deps):
        # -ffp-contract=off: no fused multiply-add, as the device side (__fmul_rn / __fadd_rn ...); x86-64-v3 so that a contraction would show
        subprocess.check_call(["g++", "-x", "c++", "-std=c++17", "-O2", "-march=x86-64-v3", "-ffp-contract=off", "-fPIC", "-shared", "-Wall",
                               "-o", out, src])
    L = C.CDLL(out)
    L.ah_eval.restype = None
    L.ah_eval.argtypes = [C.c_int, C.c_void_p, _i32p, _f32p, _f32p, _f32p, _f32p, C.c_float, C.c_float, C.c_float, _f32p, _f32p, _u8p]
    L.ah_pixel.restype = None
    L.ah_pixel.argtypes = [C.c_int, _f32p, C.c_int, C.c_int, _i32p]
    return L


def header_eval(L, curves, model, depth, fill, d0, d1, depths=DEPTHS):
    n = len(model)
    curve, thr, acc = np.zeros(n, np.float32), np.zeros(n, np.float32), np.zeros(n, np.uint8)
    curves = np.ascontiguousarray(curves, capi.ADAPTIVE_MODEL)
    L.ah_eval(n, curves.ctypes.data, np.ascontiguousarray(model, np.int32), *[np.ascontiguousarray(a, np.float32) for a in (depth, fill, d0, d1)],
              *[float(v) for v in depths], curve, thr, acc)
    return curve, thr, acc.astype(bool)


def random_curves(rng, n):
    c = np.zeros(n, capi.ADAPTIVE_MODEL)
    c["depth_peak"] = rng.uniform(0.3, 1.5, n)
    c["depth_fade"] = c["depth_peak"] * rng.uniform(1.2, 3.0, n).astype(np.float32)
    c["ratio_low"] = rng.uniform(0.5, 0.8, n)
    c["ratio_high"] = c["ratio_low"] + rng.uniform(0.0, 0.15, n).astype(np.float32)
    return c


def edge_inputs(curves, rng):
    """every breakpoint of every curve (and the float either side), 0, the depth cut and the default depth, each with fill 0, a typical
    fill, a very large one and a huge one (t * t overflows)"""
    maxd, defd = np.float32(DEPTHS[0]), np.float32(DEPTHS[1])
    model, depth = [], []
    for m, c in enumerate(curves):
        points = [c["depth_peak"], c["depth_fade"], np.float32(c["depth_fade"] * np.float32(2)), maxd, defd, np.float32(0)]
        for p in points:
            for v in (np.nextafter(p, np.float32(-np.inf)), p, np.nextafter(p, np.float32(np.inf))):
                model.append(m); depth.append(v)
    model, depth = np.repeat(model, 4), np.repeat(np.array(depth, np.float32), 4)
    fill = np.tile(np.array([0.0, 0.07, 250.0, 3e30], np.float32), len(model) // 4)
    d1 = rng.uniform(0.2, 1.0, len(model)).astype(np.float32)
    d0 = (d1 * rng.uniform(0.0, 1.0, len(model))).astype(np.float32)
    return model.astype(np.int32), depth, fill, d0, d1


def test_numpy_rule_equals_the_header_bit_for_bit(host_lib):
    rng = np.random.default_rng(3)
    curves = random_curves(rng, 16)
    n = 200000
    model = rng.integers(0, len(curves), n).astype(np.int32)
    depth = rng.uniform(0.0, 6.0, n).astype(np.float32)
    fill = np.where(rng.random(n) < 0.3, 0.0, 10.0 ** rng.uniform(-4, 3, n)).astype(np.float32)
    d1 = rng.uniform(0.05, 1.5, n).astype(np.float32)
    d0 = (d1 * rng.uniform(0.3, 1.0, n)).astype(np.float32)
    d1[:50] = 0                                                               # ratio inf / nan: rejected on both sides
    em, ed, ef, e0, e1 = edge_inputs(curves, rng)
    model, depth, fill, d0, d1 = (np.concatenate(a) for a in ((model, em), (depth, ed), (fill, ef), (d0, e0), (d1, e1)))
    curve, thr, acc = header_eval(host_lib, curves, model, depth, fill, d0, d1)
    assert np.array_equal(curve.view(np.uint32), R.ratio_curve(curves, model, depth, DEPTHS[0]).view(np.uint32))
    assert np.array_equal(thr.view(np.uint32), R.threshold(curves, model, depth, fill, *DEPTHS).view(np.uint32))
    assert np.array_equal(acc, R.accept(curves, model, depth, fill, d0, d1, *DEPTHS))
    seg = R.segment(curves, model, depth, DEPTHS[0])
    for s in range(4):                                                        # accepts and rejects in every segment inside the cut
        assert acc[seg == s].any() and not acc[seg == s].all(), R.SEGMENTS[s]
    assert not acc[seg == 4].any() and (seg == 4).sum() > 1000
    w = R.cauchy_weight(fill, DEPTHS[2])
    assert w.max() == 1 and w.min() == 0                                      # fill 0 and a fill whose square overflows


def test_other_stage_constants(host_lib):
    """maximum_depth / default_depth / cauchy_scale are parameters of the entry: a default depth in the fade segment, a depth cut
    inside the curves, a wide Cauchy kernel"""
    rng = np.random.default_rng(4)
    curves = random_curves(rng, 8)
    n = 50000
    model = rng.integers(0, len(curves), n).astype(np.int32)
    depth = rng.uniform(0.0, 4.0, n).astype(np.float32)
    fill = (10.0 ** rng.uniform(-3, 2, n)).astype(np.float32)
    d1 = rng.uniform(0.05, 1.5, n).astype(np.float32)
    d0 = (d1 * rng.uniform(0.3, 1.0, n)).astype(np.float32)
    for depths in ((2.5, 2.2, 0.5), (1.1, 0.4, 25.0)):
        curve, thr, acc = header_eval(host_lib, curves, model, depth, fill, d0, d1, depths)
        assert np.array_equal(curve.view(np.uint32), R.ratio_curve(curves, model, depth, depths[0]).view(np.uint32))
        assert np.array_equal(thr.view(np.uint32), R.threshold(curves, model, depth, fill, *depths).view(np.uint32))
        assert np.array_equal(acc, R.accept(curves, model, depth, fill, d0, d1, *depths))


def test_pixel_lookup_equals_the_header(host_lib):
    """truncation, the reference's clamp to [0, width] x [0, height] and the index kept inside the map: x == width reads the next
    row's first pixel, x == width on the last row the map's last pixel"""
    rng = np.random.default_rng(5)
    W, H = 640, 480
    xy = np.stack([rng.uniform(-5, W + 5, 20000), rng.uniform(-5, H + 5, 20000)], 1).astype(np.float32)
    edges = np.array([[W, 0], [W, 17], [W, H - 1], [W, H], [0, H], [W - 1, H], [W - 0.001, H - 0.001], [-0.5, -0.5], [-1.0, 3.0], [0, 0],
                      [W + 3, H + 3], [639.99994, 479.99997]], np.float32)
    xy = np.ascontiguousarray(np.concatenate([xy, edges]))
    px = np.zeros(len(xy), np.int32)
    host_lib.ah_pixel(len(xy), xy, W, H, px)
    assert np.array_equal(px, R.pixel(xy, W, H))
    e = px[-len(edges):]
    assert e[0] == W and e[1] == 18 * W and e[2] == H * W - 1 and e[3] == H * W - 1 and e[4] == H * W - 1 and e[7] == 0


def test_synth_frames_cover_every_segment():
    db = synth.make_db(24, 400, seed=11)
    b = synth.make_adaptive_frames(db, 6, seed=11, empty=(1,), far=(2,))
    fo, curves = b["frame_offsets"], b["curves"]
    counts = np.diff(fo)
    assert counts[1] == 0 and (counts[[0, 2, 3, 4, 5]] > 0).all() and not (counts % 256 == 0)[counts > 0].any()
    assert len(set(counts.tolist())) == len(counts)
    assert (b["depth"][2] > b["maximum_depth"]).all()
    assert set(b["segments"]) == set(R.SEGMENTS)
    # the depth under every feature lies in the same segment of EVERY model's curve (segments are clear of all breakpoints)
    H, W = b["depth"].shape[1:]
    frame_of = np.repeat(np.arange(len(counts)), counts)
    px = R.pixel(b["xy"], W, H)
    z = b["depth"].reshape(len(counts), -1)[frame_of, px]
    seg = np.stack([R.segment(curves, np.full(len(z), m), z, b["maximum_depth"]) for m in range(len(curves))])
    assert (seg == seg[0]).all()
    hist = np.bincount(seg[0], minlength=5)
    assert (hist > 200).all(), hist
    w = R.cauchy_weight(b["fill"], b["cauchy_scale"])
    assert (w == 1).mean() > 0.3 and w.min() < 1e-3 and ((w > 0.1) & (w < 0.9)).any()
    assert np.array_equal(b["fill"], b["fill_distance"].reshape(len(counts), -1)[frame_of, px])
    assert ((b["xy"] >= 0) & (b["xy"] < [W, H])).all()
    assert np.allclose(b["world"][:, 2], z)
