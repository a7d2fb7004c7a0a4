"""The DEVICE SOURCE of the cached-row-maximum agglomeration (moped_b200/csrc/linkage_cached.cuh, the kernel behind
mc_set_option("linkage_cached")) compiled by g++ with the 256 threads of its block emulated by a loop (tests/cpp/linkage_host.cpp),
against the oracle's hierarchicalCluster (oracle/moped_linkage_oracle.c, bit-identical to the strict build of moped3d's
CLUSTER_LINKAGE_CPU): identical clusters on tie-heavy quantised matrices (where the reference's scan-order tie rule and its
erase-and-skip quirk decide), on real-valued ones and on matrices with NaN entries (duplicate matches make get3DFilterK a 0/0; the
reference's strict > never merges on a NaN), threads of a phase visited in ascending and in descending order. The CUDA
kernel itself is checked on the device by tests/test_gpu_depth_pose.py::test_cached_agglomeration_equals_default_kernel."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_f32p = np.ctypeslib.ndpointer(dtype=np.float32, flags="C_CONTIGUOUS")
_i32p = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")


@pytest.fixture(scope="module")
def host_lib():
    out_dir = os.path.join(ROOT, "tests", "_build")
    os.makedirs(out_dir, exist_ok=True)
    out = os.path.join(out_dir, "liblinkage_host.so")
    src = os.path.join(ROOT, "tests", "cpp", "linkage_host.cpp")
    deps = [src] + [os.path.join(ROOT, "moped_b200", "csrc", f) for f in ("linkage_cached.cuh", "simt_phases.cuh")]
    if not os.path.exists(out) or any(os.path.getmtime(d) > os.path.getmtime(out) for d in deps):
        subprocess.check_call(["g++", "-x", "c++", "-std=c++17", "-O2", "-march=x86-64-v3", "-ffp-contract=off", "-fPIC", "-shared", "-Wall",
                               "-o", out, src])
    L = C.CDLL(out)
    L.lh_agglomerate.restype = None
    L.lh_agglomerate.argtypes = [C.c_int, C.c_int, _f32p, C.c_float, C.c_int, _i32p, _i32p, _i32p]
    return L


def run_host(L, K, cutoff, min_pts, order):
    n = len(K)
    cnt = np.zeros(1, np.int32); off = np.zeros(n + 2, np.int32); mem = np.zeros(n + 1, np.int32)
    L.lh_agglomerate(order, n, np.ascontiguousarray(K, np.float32), cutoff, min_pts, cnt, off, mem)
    c = int(cnt[0])
    return off[:c + 1].copy(), mem[:off[c]].copy()


def random_similarity(rng, n, quantised):
    if quantised:
        levels = int(rng.integers(2, 6))
        K = rng.integers(0, levels + 1, (n, n)).astype(np.float32) / levels
    else:
        K = rng.random((n, n)).astype(np.float32)
    K = np.maximum(K, K.T)
    np.fill_diagonal(K, 1.0)
    return K


def nan_sprinkled(rng, K, frac):
    """K with a fraction `frac` of its off-diagonal pairs set to NaN on both sides"""
    K = K.copy()
    n = len(K)
    i, j = np.triu_indices(n, 1)
    pick = rng.random(len(i)) < frac
    K[i[pick], j[pick]] = np.nan; K[j[pick], i[pick]] = np.nan
    return K


def duplicate_scene_similarity(seed, n_dup, use3d):
    """the similarity matrix of make_linkage_scene(seed) with n_dup of its matches duplicated: 2 * n_dup NaN entries for
    use3d 1 and 2"""
    from moped_b200 import synth
    xy, xyz, world, depth, dist = synth.make_linkage_scene(seed)
    xy, xyz, world = synth.duplicate_matches((xy, xyz, world), n_dup, seed)
    return oracle.linkage_similarity(xy, xyz, world, depth, dist, use3d_filter=use3d)


def test_cached_agglomeration_equals_oracle(host_lib):
    rng = np.random.default_rng(0)
    merged = 0
    for case in range(240):
        n = int(rng.integers(1, 70)) if case % 8 else int(rng.integers(250, 330))       # a few cases above the block width
        K = random_similarity(rng, n, case % 2 == 1)
        cutoff = float(rng.choice([0.1, 0.2, 0.5, 0.75, 1.0]))
        min_pts = int(rng.integers(0, 4))
        oo, om = oracle.linkage_agglomerate(K, cutoff, min_pts, 1)
        for order in (0, 1):
            co, cm = run_host(host_lib, K, cutoff, min_pts, order)
            assert np.array_equal(oo, co) and np.array_equal(om, cm), (case, n, cutoff, min_pts, order)
        merged += n - (len(oo) - 1)
    assert merged > 2000
    # NaN similarities: the 600-match scene with duplicated matches, and random matrices with NaN pairs
    nan_cases = [(duplicate_scene_similarity(seed, 5 + 11 * (seed % 6), 1 + seed % 2), 0.1, 7) for seed in range(8)]
    for case in range(60):
        n = int(rng.integers(2, 321))
        K = nan_sprinkled(rng, random_similarity(rng, n, case % 2 == 1), float(rng.choice([0.001, 0.01, 0.03, 0.1])))
        nan_cases.append((K, float(rng.choice([0.1, 0.2, 0.5, 0.75])), int(rng.integers(0, 4))))
    assert sum(np.isnan(K).any() for K, _, _ in nan_cases) >= 50
    for case, (K, cutoff, min_pts) in enumerate(nan_cases):
        oo, om = oracle.linkage_agglomerate(K, cutoff, min_pts, 1)
        for order in (0, 1):
            co, cm = run_host(host_lib, K, cutoff, min_pts, order)
            assert np.array_equal(oo, co) and np.array_equal(om, cm), ("nan", case, len(K), cutoff, min_pts, order)


def test_cached_agglomeration_on_clustered_scenes(host_lib):
    """Block-structured similarities like the stage produces (a few objects + outliers), 600 matches: the size the first timing
    was taken at (profiles/linkage_bench_r1j.jsonl)."""
    rng = np.random.default_rng(3)
    for n, groups in ((240, 3), (600, 4)):
        g = rng.integers(0, groups + 1, n)                       # group `groups` = outliers
        base = (g[:, None] == g[None, :]) & (g[:, None] < groups)
        K = np.where(base, 0.6 + 0.4 * rng.random((n, n)), 0.05 * rng.random((n, n))).astype(np.float32)
        K = np.maximum(K, K.T); np.fill_diagonal(K, 1.0)
        oo, om = oracle.linkage_agglomerate(K, 0.1, 7, 1)
        co, cm = run_host(host_lib, K, 0.1, 7, 0)
        assert np.array_equal(oo, co) and np.array_equal(om, cm), n
        assert len(oo) - 1 == groups
