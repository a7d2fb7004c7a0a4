"""The oracle's moped3d recognition chain (tests/oracle_chain3d.py) on synthetic RGB-D frames (synth.make_depth_frame): it recovers every
planted instance and finds nothing for the models that only have a handful of junk matches. No GPU needed."""
import numpy as np
import pytest

import oracle_chain3d
from conftest import quat_angle
from moped_b200 import synth


@pytest.mark.parametrize("variant", [0, 1])
def test_oracle_chain_recovers_the_planted_instances(oracle_mod, variant):
    """Within 1 cm / 60 mrad with the shipped back-projection stage (variant 0); the reprojection stage finds the same instances."""
    for seed in (1, 2, 3):
        fr = synth.make_depth_frame(seed)
        out = oracle_chain3d.frame(fr, variant=variant)
        assert len(fr["gt_model"]) >= 4
        assert sorted(out["model"].tolist()) == sorted(fr["gt_model"].tolist()), (seed, out["model"], fr["gt_model"])
        for m, g in zip(fr["gt_model"], fr["gt_pose"]):
            if variant:
                continue
            hits = [p for mm, p in zip(out["model"], out["pose"]) if mm == m
                    and np.abs(p[4:] - g[4:]).max() < 0.01 and quat_angle(p[:4], g[:4]) < 0.06]
            assert hits, (seed, int(m), out["model"])
        assert not set(out["model"].tolist()) & set(fr["junk_models"].tolist()), (seed, out["model"], fr["junk_models"])


def test_depth_frame_layout():
    fr = synth.make_depth_frame(4, n_models=9)
    off = fr["match_offsets"]
    assert off[0] == 0 and np.all(np.diff(off) >= 0) and len(off) == 10
    M = int(off[-1])
    for k, w in (("match_xy", 2), ("match_xyz", 3), ("match_world", 3)):
        assert fr[k].shape == (M, w) and fr[k].dtype == np.float32
    assert fr["match_fill"].shape == (M,) and fr["match_image"].shape == (M,)
    assert fr["depth"].shape == (480, 640) and fr["fill_distance"].shape == (480, 640)
    xy = fr["match_xy"]
    assert (xy >= 0).all() and (xy[:, 0] < 640).all() and (xy[:, 1] < 480).all()
    assert (fr["fill_distance"] > 0).any() and (fr["fill_distance"] == 0).any()
    for m in fr["junk_models"]:
        assert 3 <= off[m + 1] - off[m] <= 6
    b = synth.stack_depth_frames([fr, synth.make_depth_frame(5, n_models=9)])
    assert b["match_offsets"].shape == (2, 10) and b["match_offsets"][1, 0] == M
    assert b["depth"].shape == (2, 480, 640) and len(b["match_xy"]) == b["match_offsets"][1, -1]
