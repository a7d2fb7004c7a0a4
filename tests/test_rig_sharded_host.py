"""moped_b200.sharding.run on CPU over gloo (world 2 and 3): the exchange logic of the object-sharded step from pixels to objects, with
stand-ins for the library calls. Frame f's extraction yields n(f) descriptor rows that spell (frame, keypoint), so the compacted query list
shows the bases, P and the compaction order; the stand-in MATCH / frame calls record what they were given. Also: the status exchange
(every rank raises the same error before the descriptor all-gather), ranks without frames, and batches without any feature (no MATCH)."""
import os
import socket
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KP = 6                       # max_keypoints of the stand-in extraction (one camera)


def n_feat(f, blank):
    return 0 if f in blank else 1 + (3 * f + 2) % KP


def _fake_step_class():
    import torch
    from moped_b200.sharding import RigShardStep

    class FakeStep(RigShardStep):
        """RigShardStep with the library calls replaced: `cams` = (first frame, frames that come out blank, failing status)"""

        def __init__(self, *a, **kw):
            super().__init__(None, *a, device="cpu", **kw)
            self.log = {}

        def extract(self, cams, n_local):
            lo, blank, status = cams
            counts = [n_feat(lo + j, blank) for j in range(n_local)]
            self.fo = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
            self.n_features = np.array(counts, np.int32).reshape(-1, 1)
            for j, n in enumerate(counts):
                for i in range(n):
                    self.desc[self.fo[j] + i] = float(1000 * (lo + j) + i)
            self.desc[self.fo[-1]:] = -1.0                 # rows past the rank's list: never part of the query list
            return status, int(self.fo[-1]) if status == 0 else 0

        def send(self, plan):
            self.log["sent"] = True
            return super().send(plan)

        def match(self, plan, q_all):
            self.log["q_all"] = q_all[:plan.Q, 0].clone().numpy()
            assert bool((q_all[:plan.Q] == q_all[:plan.Q, :1]).all())
            return torch.full((4 * plan.Q,), 10 + self.rank, dtype=torch.int32)

        def merge(self, plan, nn_all):
            self.log["nn_all"] = nn_all.numpy().copy()

        def frames(self, plan):
            lo, hi = plan.frames[self.rank]
            b = self.block
            self.res.zero_()
            for s in range(hi - lo):                          # info = {0 objects, frame, its first global row, Q}
                self.res[b.o_info + 4 * s:b.o_info + 4 * s + 4] = torch.tensor([0, lo + s, int(plan.base[self.rank]) + int(self.fo[s]), plan.Q])
            return self.res

    return FakeStep


# (n_frames, frames that come out blank, failing rank or None). World 2: an even split, a batch without features (Q = 0), a failure.
# World 3: 7 frames over 3 ranks with rank 1's frames blank (Q_1 = 0), 2 frames (rank 2 has none), a failure, 16 uneven frames.
CASES = {2: [(5, (), None), (3, (0, 1, 2), None), (4, (1,), 0)],
         3: [(7, (3, 4), None), (2, (), None), (7, (), 1), (16, (0, 5, 6, 7, 8, 9), None)]}


def _rank(rank, world, port, q):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    from moped_b200.sharding import RigShardError, block_range, run
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    FakeStep = _fake_step_class()
    out = []
    for n_frames, blank, failing in CASES[world]:
        step = FakeStep(rank, world, 1, n_frames, max_keypoints=KP, max_objects=3, params=object())
        lo, hi = block_range(n_frames, world, rank)
        status = -4 if rank == failing else 0
        try:
            frames = run(None, step, (lo, blank, status), n_frames)
            out.append(dict(frames=[fr["info"].tolist() for fr in frames], log=step.log, n_features=step.n_features.reshape(-1).tolist()))
        except RigShardError as e:
            out.append(dict(error=(e.rank, e.status, str(e)), log=step.log))
    q.put((rank, out))
    dist.destroy_process_group()


def _spawn(world):
    import torch.multiprocessing as mp
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_rank, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=300) for _ in procs)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    return [res[r] for r in range(world)]


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_rig_step_exchange(world):
    from moped_b200.sharding import block_range
    per_rank = _spawn(world)
    for k, (n_frames, blank, failing) in enumerate(CASES[world]):
        res = [per_rank[r][k] for r in range(world)]
        counts = [n_feat(f, blank) for f in range(n_frames)]
        if failing is not None:
            # the same error on every rank, raised after the status exchange and before the descriptor all-gather
            assert all(r.get("error") == res[0]["error"] for r in res), res
            assert res[0]["error"][:2] == (failing, -4)
            assert not any(r["log"].get("sent") for r in res)
            continue
        ranges = [block_range(n_frames, world, r) for r in range(world)]
        q_r = [sum(counts[lo:hi]) for lo, hi in ranges]
        Q = sum(q_r)
        want_rows = [1000 * f + i for f in range(n_frames) for i in range(counts[f])]
        first_row = np.concatenate([[0], np.cumsum(counts)[:-1]])
        for r in range(world):
            lo, hi = ranges[r]
            assert res[r]["n_features"] == counts[lo:hi]
            # every rank gets every frame, in frame order, each with its global first row (base + local offset)
            assert res[r]["frames"] == [[0, f, int(first_row[f]), Q] for f in range(n_frames)], (r, res[r]["frames"])
            if Q == 0:
                assert "sent" not in res[r]["log"] and "q_all" not in res[r]["log"]         # no exchange, no MATCH
                continue
            assert res[r]["log"]["sent"]
            assert res[r]["log"]["q_all"].tolist() == want_rows                           # compaction in rank (= frame) order
            nn_all = res[r]["log"]["nn_all"]
            assert nn_all.shape == (world, 4 * Q) and nn_all.tolist() == [[10 + s] * (4 * Q) for s in range(world)]


def test_exchange_plan_and_block_range():
    from moped_b200.sharding import RigExchange, RigShardError, block_range
    assert [block_range(7, 3, r) for r in range(3)] == [(0, 3), (3, 5), (5, 7)]
    assert [block_range(7, 8, r) for r in range(8)] == [(r, r + 1) for r in range(7)] + [(7, 7)]
    p = RigExchange(np.array([[0, 5], [0, 0], [0, 9]]), 7)
    assert p.Q == 14 and p.P == 9 and p.base.tolist() == [0, 5, 5] and p.frames == [(0, 3), (3, 5), (5, 7)]
    with pytest.raises(RigShardError) as e:
        RigExchange(np.array([[0, 5], [-4, 0], [-2, 0]]), 7)
    assert (e.value.rank, e.value.status) == (1, -4)
