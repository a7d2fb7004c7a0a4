"""Host-side logic of bench.py (no GPU): the schedule bench.py picks from the frames per GPU, the sub-result runner of the
default line (child JSON lines condensed, a failing child reported without losing the main line), the file layout of
--dump-outputs, and the file-descriptor redirection that keeps NCCL's banner off stdout."""
import argparse
import json
import os
import subprocess
import sys
import types

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def _args(**kw):
    d = dict(frames=64, pipeline=-1, stage_sms=-1, lanes=0, pose_warps=0, objects=1000, pts=1000, features=2000, pose_mode="default")
    d.update(kw)
    return argparse.Namespace(**d)


def test_schedule_by_frames_per_gpu():
    a = bench.resolve_auto(_args(), 1)                      # 64 frames on one GPU: one call per step, a lane per frame
    assert (a.pipeline, a.stage_sms, a.lanes, a.pose_warps) == (0, 0, 64, 4)
    a = bench.resolve_auto(_args(), 2)
    assert (a.pipeline, a.lanes) == (0, 32)
    a = bench.resolve_auto(_args(), 4)                      # <= 16 frames per GPU: MATCH of step i+1 beside the stages of step i
    assert (a.pipeline, a.stage_sms, a.lanes) == (1, 16, 16)
    a = bench.resolve_auto(_args(), 8)
    assert (a.pipeline, a.stage_sms, a.lanes) == (1, 16, 16)
    a = bench.resolve_auto(_args(frames=1), 1)              # configs[1]: a single frame
    assert (a.pipeline, a.stage_sms, a.lanes) == (1, 16, 16)
    a = bench.resolve_auto(_args(lanes=8, pose_warps=2, pipeline=0, stage_sms=0), 1)      # explicit flags win
    assert (a.pipeline, a.lanes, a.pose_warps) == (0, 8, 2)


def test_both_arms_describe_the_same_configuration():
    a, b = bench.resolve_auto(_args(coarse_kind=1, reserve_sms=0, batch_graph=1, merge_levels=1, chunks=1), 1), \
        bench.resolve_auto(_args(coarse_kind=1, reserve_sms=0, batch_graph=1, merge_levels=1, chunks=1), 1)
    assert bench.workload_config(a, 1) == bench.workload_config(b, 1)
    c = bench.workload_config(a, 1)
    assert c["db_descriptors"] == 1000000 and c["features_per_frame"] == 2000 and c["frames_per_step"] == 64
    assert bench.default_metric_config(a) and not bench.default_metric_config(_args(features=4000))


def test_other_config_lines_condense_children_and_survive_failures(monkeypatch):
    calls = []

    def fake_run(cmd, **kw):
        calls.append(cmd)
        if "sift" in cmd:                                                         # one child fails
            return types.SimpleNamespace(returncode=3, stdout="", stderr="boom\nlast line")
        line = {"metric": "frames_per_s", "value": 12.5, "unit": "frames/s", "ms_per_step": 80.0, "steps": 5, "warmup": 3, "gpu_launches": 7, "dtype": "f32",
                "e2e": {"value": 11.0}, "clocks": {"sm_mhz": 1965.0, "reasons": []}, "single_frame": {"latency_ms": 1.5},
                "roofline": {"kernel": "k", "bound": "tensor", "achieved": 1.0, "peak": 2.0, "unit": "TFLOP/s", "frac": 0.5}}
        return types.SimpleNamespace(returncode=0, stdout="NCCL version 2.28\n" + json.dumps(line) + "\n", stderr="")

    monkeypatch.setattr(subprocess, "run", fake_run)
    res = bench.other_config_lines()
    assert len(res) == 6 and len(calls) == 6
    assert all("--other-configs" in c and c[c.index("--other-configs") + 1] == "0" for c in calls)      # children never recurse
    ok = [v for v in res.values() if "error" not in v]
    bad = [v for v in res.values() if "error" in v]
    assert len(ok) == 5 and len(bad) == 1 and "rc 3" in bad[0]["error"]
    assert all(v["value"] == 12.5 and v["e2e"] == 11.0 and v["roofline"]["frac"] == 0.5 and v["single_frame_latency_ms"] == 1.5 for v in ok)
    json.dumps(res)                                                               # must fit into the main JSON line


def _frames(n, mo, seed=1):
    rng = np.random.default_rng(seed)
    out = []
    for f in range(n):
        k = int(rng.integers(0, mo + 1))
        out.append(dict(model=rng.integers(0, 1000, k).astype(np.int32), pose=rng.standard_normal((k, 7)).astype(np.float32),
                        score=rng.random(k).astype(np.float32), info=np.array([k, 0, int(rng.integers(0, 500)), int(rng.integers(0, 9))], np.int32)))
    return out


def test_dump_outputs_writes_every_frame_as_float_arrays(tmp_path):
    frames = _frames(5, 4)
    bench.dump_frame_results(str(tmp_path / "d"), frames, 4)
    a = {n: np.load(tmp_path / "d" / (n + ".npy")) for n in ("frame_index", "frame_info", "obj_model", "obj_pose", "obj_score")}
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    assert a["frame_index"].tolist() == [0, 1, 2, 3, 4]
    assert a["obj_model"].shape == (5, 4) and a["obj_pose"].shape == (5, 4, 7) and a["obj_score"].shape == (5, 4)
    for f, fr in enumerate(frames):
        k = len(fr["model"])
        assert np.array_equal(a["frame_info"][f], fr["info"])
        assert np.array_equal(a["obj_model"][f, :k], fr["model"]) and (a["obj_model"][f, k:] == -1).all()
        assert np.array_equal(a["obj_pose"][f, :k], fr["pose"]) and (a["obj_pose"][f, k:] == 0).all()
        assert np.array_equal(a["obj_score"][f, :k], fr["score"])


def test_dump_outputs_of_a_large_batch_is_a_fixed_sample_under_the_limit(tmp_path, monkeypatch):
    mo = 64
    per_frame = 8 * (1 + 4 + mo) + 4 * 8 * mo
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 4096 + 10 * per_frame)
    frames = _frames(40, mo)
    bench.dump_frame_results(str(tmp_path / "a"), frames, mo)
    bench.dump_frame_results(str(tmp_path / "b"), frames, mo)
    total = sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a"))
    assert total <= bench.DUMP_LIMIT_BYTES
    idx = np.load(tmp_path / "a" / "frame_index.npy")
    assert len(idx) == 10 and len(set(idx.tolist())) == 10 and (np.diff(idx) > 0).all()
    for n in os.listdir(tmp_path / "a"):
        assert np.array_equal(np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n))
    model = np.load(tmp_path / "a" / "obj_model.npy")
    for j, f in enumerate(idx.astype(int)):
        assert np.array_equal(model[j, :len(frames[f]["model"])], frames[f]["model"])


@pytest.mark.gpu
@pytest.mark.parametrize("pipeline,steps", [(0, 3), (1, 4)])
def test_dump_outputs_hold_the_last_timed_step(tmp_path, pipeline, steps):
    """bench.py --dump-outputs on a small batch, one call per step and software-pipelined. bench alternates two batches, step i
    running batch i % 2. The objects its timed region counted equal those of exactly steps warmup .. warmup + steps - 1 (a run of
    any other number of steps counts a different total, both batches finding objects), and the files equal what mc_process_frames
    returns for the batch of step warmup + steps - 1."""
    from moped_b200 import capi, synth
    objects, pts, Q, B, warmup = 20, 500, 1000, 4, 3
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--objects", str(objects), "--pts", str(pts), "--features", str(Q),
                        "--frames", str(B), "--steps", str(steps), "--warmup", str(warmup), "--pipeline", str(pipeline), "--no-cpu-baseline",
                        "--other-configs", "0", "--dump-outputs", str(tmp_path / "got")], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
    assert line["steps"] == steps and line["warmup"] == warmup
    db = synth.make_db(objects, pts)
    fo = (np.arange(B + 1) * Q).astype(np.int32)
    ctx = capi.Context(0)
    try:
        ctx.db_upload(bench.host_norm_rows(db["desc"]), db["xyz"], db["model_of_row"], objects)
        ctx.set_cameras(synth.K_DEFAULT, synth.CAM_IDENTITY)
        ctx.set_tuning(B, 4, 1)
        for opt in ("match_coarse_kind", "batch_graph", "ransac_merge_levels"):
            ctx.set_option(opt, 1)
        want = []
        for p in range(2):
            fr = [synth.make_frame(db, Q, n_visible=8, frame_id=p * B + i) for i in range(B)]
            want.append(ctx.process_frames(np.concatenate([bench.host_norm_rows(f["desc"]) for f in fr]), np.concatenate([f["xy"] for f in fr]),
                                           np.concatenate([f["image_idx"] for f in fr]), fo))
    finally:
        ctx.close()
    n_objects = [sum(len(o["model"]) for o in w) for w in want]
    assert min(n_objects) > 0
    assert round(line["objects_per_frame"] * steps * B) == sum(n_objects[i % 2] for i in range(warmup, warmup + steps))
    last = (warmup + steps - 1) % 2
    assert [o["model"].tolist() for o in want[last]] != [o["model"].tolist() for o in want[1 - last]]     # the two batches tell apart
    bench.dump_frame_results(str(tmp_path / "want"), want[last], 64)
    for name in sorted(os.listdir(tmp_path / "want")):
        g, w = np.load(tmp_path / "got" / name), np.load(tmp_path / "want" / name)
        assert g.shape == w.shape and g.dtype == w.dtype, name
        if name in ("obj_pose.npy", "obj_score.npy"):
            assert np.allclose(g, w, rtol=0, atol=1e-5), (name, np.abs(g - w).max())
        else:
            assert np.array_equal(g, w), name


def test_stdout_is_restored_after_the_quiet_nccl_init(capfd):
    class FakeDist:
        def init_process_group(self, *a, **k):
            os.write(1, b"NCCL version banner\n")                                 # what NCCL does: straight to file descriptor 1

        def all_reduce(self, t):
            pass

    fake_torch = types.SimpleNamespace(zeros=lambda *a, **k: 0, cuda=types.SimpleNamespace(synchronize=lambda *a, **k: None))
    saved = sys.modules.get("torch")
    sys.modules["torch"] = fake_torch
    try:
        bench.init_nccl_quietly(FakeDist(), None)
    finally:
        if saved is not None:
            sys.modules["torch"] = saved
        else:
            del sys.modules["torch"]
    os.write(1, b"{\"json\": 1}\n")
    out, err = capfd.readouterr()
    assert "banner" not in out and "banner" in err and out.strip() == '{"json": 1}'
