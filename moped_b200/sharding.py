"""Host-side sharding of the model database by object (SURVEY.md §8e): contiguous object ranges balanced by
descriptor count. Rank r uploads rows [row_lo, row_hi) with row_base = row_lo (mc_db_upload) plus the two small
global tables (mc_db_set_global_tables); per-query (row, distance) pairs of all shards are exchanged with one
all-gather and merged by mc_match_merge_dev (smaller distance first, then smaller global row id)."""
from __future__ import annotations

import numpy as np


def shard_objects(n_pts: np.ndarray, world: int):
    """-> list of (obj_lo, obj_hi, row_lo, row_hi) per rank."""
    n_pts = np.asarray(n_pts)
    cum = np.concatenate([[0], np.cumsum(n_pts)])
    total = cum[-1]
    bounds = [0]
    for r in range(1, world):
        b = int(np.searchsorted(cum, total * r / world))
        bounds.append(min(max(b, bounds[-1]), len(n_pts)))
    bounds.append(len(n_pts))
    return [(bounds[r], bounds[r + 1], int(cum[bounds[r]]), int(cum[bounds[r + 1]])) for r in range(world)]


def frame_range(n_frames: int, world: int, rank: int):
    """Frames of a batch that rank `rank` runs through CLUSTER..FILTER2 after the merged MATCH: contiguous blocks
    of n_frames / world (so that the all-gathered per-rank result blocks are in frame order)."""
    if n_frames % world:
        raise ValueError(f"{n_frames} frames do not split evenly over {world} ranks")
    per = n_frames // world
    return rank * per, (rank + 1) * per


class ResultBlock:
    """Layout of one rank's result block for `frames` frames with `max_objects` slots each, in int32 words:
    info[frames,4] | model[frames,MO] | score[frames,MO] (f32 bits) | pose[frames,MO*7] (f32 bits).
    mc_process_frames_matched_dev writes the four regions in place; one all-gather moves the block."""

    def __init__(self, frames: int, max_objects: int):
        self.frames, self.mo = frames, max_objects
        self.o_info = 0
        self.o_model = frames * 4
        self.o_score = frames * (4 + max_objects)
        self.o_pose = frames * (4 + 2 * max_objects)
        self.words = frames * (4 + 9 * max_objects)

    def unpack(self, blocks: np.ndarray, counts=None):
        """blocks: [world, words] int32 (the all-gathered blocks) -> list of per-frame dict(model, pose, score, info)
        in frame order. counts (optional): frames written in each block, when ranks hold fewer frames than the block's."""
        blocks = np.asarray(blocks, dtype=np.int32).reshape(-1, self.words)
        out = []
        for r, b in enumerate(blocks):
            info = b[self.o_info:self.o_model].reshape(self.frames, 4)
            model = b[self.o_model:self.o_score].reshape(self.frames, self.mo)
            score = b[self.o_score:self.o_pose].view(np.float32).reshape(self.frames, self.mo)
            pose = b[self.o_pose:self.words].view(np.float32).reshape(self.frames, self.mo, 7)
            for f in range(self.frames if counts is None else counts[r]):
                k = min(int(info[f, 0]), self.mo)
                out.append(dict(model=model[f, :k].copy(), pose=pose[f, :k].copy(), score=score[f, :k].copy(), info=info[f].copy()))
        return out


def cluster_partition(hyp_cluster: np.ndarray, world: int, rank: int) -> np.ndarray:
    """RANSAC work distributed by cluster (north_star; BASELINE configs[3]): cluster c belongs to rank c % world, so a
    rank owns every hypothesis of its clusters and no data-path collective is needed. Returns the indices (ascending)
    of the hypotheses rank `rank` evaluates; the union over ranks is a partition of range(len(hyp_cluster))."""
    return np.nonzero(np.asarray(hyp_cluster) % world == rank)[0]


RANSAC_STREAM_STRIDE = 0x9E3779B97F4A7C15      # task t of a call draws from seed + stride * (t + 1)  (pose.cu / pose_depth.cu)


def block_range(n: int, world: int, rank: int):
    """Rank `rank`'s contiguous block [lo, hi) of n items split as evenly as possible, the first n % world ranks one item longer
    (7 over 3 ranks: 3 / 2 / 2; 7 over 8 ranks: the last rank has none)."""
    per, extra = divmod(n, world)
    lo = rank * per + min(rank, extra)
    return lo, lo + per + (1 if rank < extra else 0)


def ransac_cluster_range(n_clusters: int, world: int, rank: int):
    """Full RANSAC (mc_pose_ransac / mc_pose_depth_ransac) distributed by cluster: rank r runs the contiguous cluster block
    [lo, hi) — contiguous, so that one seed offset (ransac_shard_seed) keeps every task on the random stream it has in a
    single-GPU call and the result does not depend on the number of ranks."""
    return block_range(n_clusters, world, rank)


def ransac_shard_seed(seed: int, first_cluster: int, max_objects_per_cluster: int) -> int:
    """The `seed` a shard passes so that its LOCAL task t (cluster first_cluster + t // MaxObjectsPerCluster) draws from the
    stream of GLOBAL task first_cluster * MaxObjectsPerCluster + t: seed + stride * first_task, modulo 2^64."""
    return (seed + RANSAC_STREAM_STRIDE * first_cluster * max_objects_per_cluster) & 0xFFFFFFFFFFFFFFFF


def ransac_task_owner(task: int, max_objects_per_cluster: int, world: int) -> int:
    """Frame pipeline with the RANSAC work distributed by cluster (mc_process_frame_sharded_dev): task t = (cluster, try) belongs to the
    rank that owns its cluster, cluster c -> rank c % world (the cluster count is only known on the device, so the deal is round-robin)."""
    return (task // max_objects_per_cluster) % world


def select_task_records(records: np.ndarray, max_objects_per_cluster: int) -> np.ndarray:
    """What k_shard_select does after the all-gather: records[r][t] is rank r's record of task t (zeros unless r owns t); the result
    takes every task from its owner."""
    world, n_tasks = records.shape[:2]
    owner = (np.arange(n_tasks) // max_objects_per_cluster) % world
    return records[owner, np.arange(n_tasks)]


# ---- camera-rig frames from pixels to objects on an object-sharded database ------------------------------------------------------

class RigShardError(RuntimeError):
    """A rank's extraction failed (status = the mc_status mc_extract_rig_cameras_dev returned there: -4 for a frame over max_keypoints,
    -2 for a bad argument such as an image size, ...); every rank raises the same error after the status exchange, before any later
    collective."""

    def __init__(self, rank: int, status: int):
        super().__init__(f"sharded rig step: rank {rank}'s feature extraction failed ({status})")
        self.rank, self.status = rank, status


class RigExchange:
    """What every rank knows after the all-gather of the (status, Q_r) headers [world, 2]: counts[r] = Q_r, base[r] = rank r's first
    row in the batch's query list, Q = sum, P = max (rows per rank in the descriptor all-gather), frames[r] = (lo_r, hi_r)."""

    def __init__(self, headers, n_frames: int):
        h = np.asarray(headers, dtype=np.int64).reshape(-1, 2)
        self.world = len(h)
        bad = np.nonzero(h[:, 0])[0]
        if len(bad):
            raise RigShardError(int(bad[0]), int(h[bad[0], 0]))
        self.counts = h[:, 1].copy()
        self.base = np.concatenate([[0], np.cumsum(self.counts)[:-1]]).astype(np.int64)
        self.Q, self.P = int(self.counts.sum()), int(self.counts.max())
        self.frames = [block_range(n_frames, self.world, r) for r in range(self.world)]


class RigShardStep:
    """One rank of an object-sharded database running camera-rig batches from pixels to objects. The rank's context holds its shard
    (mc_db_upload with row_base) and the global tables (mc_db_set_global_tables); the rank holds the images of its frames [lo_r, hi_r)
    (block_range) only. The step, with `run` doing the collectives:
      1 extract      mc_extract_rig_cameras_dev of the rank's frames into local buffers (skipped without frames: Q_r = 0)
      2 plan         all-gather of (status, Q_r) -> Q, P and the bases; a failed rank makes every rank raise here
      3 send         all-gather of the first P local descriptor rows of every rank -> [world][P][128]
      4 compact      the ranks' Q_r rows into one [Q][128] query list, in rank (= frame) order, with world device copies
      5 match/merge  mc_match_dev on the shard, all-gather of the packed blocks, mc_match_merge_packed_dev (skipped when Q = 0)
      6 frames       mc_process_frames_matched_dev on the rank's own frames, with its local xy / image / frame offsets and the merged
                     nearest neighbours from row base[r] on; xy and image never leave the rank
      7 unpack       all-gather of the ResultBlocks -> every frame of the batch in frame order
    The step's library calls and its torch copies and collectives run in order on one stream: `stream`, or a new torch stream when it is
    None, is set as the context's stream (mc_set_stream), and `run` enqueues everything on it. A step without a context (a stand-in for
    the library calls) has no stream. Buffers hold the frames of one rank of a batch of up to `max_frames` frames."""

    def __init__(self, ctx, rank: int, world: int, n_cameras: int, max_frames: int, max_keypoints: int = 4096, max_objects: int = 64,
                 double_size: bool = True, params=None, device="cuda", stream=None):
        import torch
        self.torch = torch
        self.ctx, self.rank, self.world, self.device = ctx, rank, world, torch.device(device)
        self.n_cameras, self.max_keypoints, self.max_objects, self.double_size = n_cameras, max_keypoints, max_objects, double_size
        self.params = params if params is not None or ctx is None else ctx.default_params()
        self.F = -(-max_frames // world)                       # most frames a rank holds
        cap = self.F * n_cameras * max_keypoints                # rows the extraction may write
        self.desc = torch.empty((cap, 128), dtype=torch.float32, device=self.device)
        self.xy = torch.empty((cap, 2), dtype=torch.float32, device=self.device)
        self.image = torch.empty((cap,), dtype=torch.int32, device=self.device)
        self.block = ResultBlock(self.F, max_objects)
        self.res = torch.zeros((self.block.words,), dtype=torch.int32, device=self.device)
        self.max_frames = max_frames
        self.stream = None
        if ctx is not None:                                    # never the context's private stream, which torch's work would not wait for
            self.stream = stream if stream is not None else torch.cuda.Stream(self.device)
            ctx.set_stream(self.stream.cuda_stream)
        self.fo = np.zeros(1, np.int32)
        self.n_features = np.zeros((0, n_cameras), np.int32)

    def extract(self, cams, n_local: int):
        """step 1: cams = (ptrs, strides, sizes) of the rank's images, frame 0 = the rank's first frame -> (status, Q_r); any failure
        of the call comes back as its status, for the exchange"""
        if n_local > self.F:
            raise ValueError(f"{n_local} frames on one rank; the step's buffers hold {self.F} (max_frames {self.max_frames} over {self.world} ranks)")
        if n_local == 0:
            self.fo, self.n_features = np.zeros(1, np.int32), np.zeros((0, self.n_cameras), np.int32)
            return 0, 0
        ptrs, strides, sizes = cams
        self.fo, self.n_features, _, st = self.ctx.extract_rig_cameras_dev(ptrs, strides, sizes, n_local, self.desc, self.xy, self.image,
                                                                          self.double_size, self.max_keypoints, partial=True)
        return st, int(self.fo[-1]) if st == 0 else 0

    def header(self, status: int, q: int):
        return self.torch.tensor([status, q], dtype=self.torch.int32, device=self.device)

    def send(self, plan: RigExchange):
        """step 3's input: the first P rows of the local buffer (P <= its capacity on every rank, so no copy)"""
        return self.desc[:plan.P].reshape(-1)

    def compact(self, plan: RigExchange, gathered):
        """step 4: gathered [world, P, 128] -> [Q, 128], rank r's Q_r rows at base[r]"""
        q_all = self.torch.empty((max(plan.Q, 1), 128), dtype=self.torch.float32, device=self.device)
        for r in range(plan.world):
            if plan.counts[r]:
                q_all[plan.base[r]:plan.base[r] + plan.counts[r]].copy_(gathered[r, :plan.counts[r]])
        return q_all

    def match(self, plan: RigExchange, q_all):
        """step 5a: this shard's two nearest rows of every query as one packed block [nn_row Q x 2 | nn_dist Q x 2]"""
        Q = plan.Q
        blk = self.torch.empty((4 * Q,), dtype=self.torch.int32, device=self.device)
        self.acc = self.torch.empty((Q,), dtype=self.torch.uint8, device=self.device)
        self.ctx.match_dev(q_all.data_ptr(), Q, self.params.match_ratio, self.params.match_mode, blk.data_ptr(), blk.data_ptr() + 8 * Q,
                           self.acc.data_ptr())
        return blk

    def merge(self, plan: RigExchange, nn_all):
        """step 5b: nn_all [world, 4 Q], the gathered blocks -> the global two nearest rows and the ratio test"""
        Q = plan.Q
        self.nn_row = self.torch.empty((Q, 2), dtype=self.torch.int32, device=self.device)
        nn_dist = self.torch.empty((Q, 2), dtype=self.torch.float32, device=self.device)
        self.ctx.match_merge_packed_dev(nn_all.data_ptr(), plan.world, Q, self.params.match_ratio, self.nn_row.data_ptr(), nn_dist.data_ptr(),
                                        self.acc.data_ptr())

    def frames(self, plan: RigExchange):
        """step 6: CLUSTER..FILTER2 of the rank's frames into its ResultBlock"""
        lo, hi = plan.frames[self.rank]
        if hi > lo:
            if plan.Q == 0:                                    # no features anywhere: nothing is read from the neighbour arrays
                self.nn_row = self.torch.zeros((1, 2), dtype=self.torch.int32, device=self.device)
                self.acc = self.torch.zeros((1,), dtype=self.torch.uint8, device=self.device)
            b, blk, base = int(plan.base[self.rank]), self.block, self.res.data_ptr()
            self.ctx.process_frames_matched_dev(self.nn_row.data_ptr() + 8 * b, self.acc.data_ptr() + b, self.xy.data_ptr(), self.image.data_ptr(),
                                                self.fo, 0, hi - lo, self.params, self.max_objects, base + 4 * blk.o_info, base + 4 * blk.o_model,
                                                base + 4 * blk.o_pose, base + 4 * blk.o_score)
        return self.res

    def unpack(self, plan: RigExchange, res_all):
        """step 7: res_all [world, words], the gathered blocks -> one dict(model, pose, score, info) per frame of the batch"""
        return self.block.unpack(res_all.cpu().numpy(), [hi - lo for lo, hi in plan.frames])


def run(group, step: RigShardStep, cams, n_frames: int):
    """One sharded step over the process group `group` (one rank per member, step.rank = the member's rank): cams = the rank's images
    as RigShardStep.extract takes them, n_frames = frames of the whole batch. Returns the frames of the whole batch in frame order
    (dict(model, pose, score, info)); step.n_features holds the counts of the rank's own frames. Raises RigShardError on every rank
    when any rank's extraction failed, and ValueError on every rank (before any collective) when n_frames exceeds the step's max_frames.
    The step's stream first waits for the caller's current stream, so images written there before the call are complete."""
    import contextlib

    import torch
    import torch.distributed as dist
    if n_frames > step.max_frames:
        raise ValueError(f"a batch of {n_frames} frames; the step was built for up to {step.max_frames}")
    lo, hi = block_range(n_frames, step.world, step.rank)
    if step.stream is not None:
        step.stream.wait_stream(torch.cuda.current_stream(step.device))
    with torch.cuda.stream(step.stream) if step.stream is not None else contextlib.nullcontext():
        st, q = step.extract(cams, hi - lo)
        # the gathered tensors are flat ([world * n], viewed as [world][n]): the layout every backend accepts
        headers = torch.empty((step.world * 2,), dtype=torch.int32, device=step.device)
        dist.all_gather_into_tensor(headers, step.header(st, q), group=group)
        plan = RigExchange(headers.cpu().numpy(), n_frames)
        if plan.Q:
            gathered = torch.empty((step.world * plan.P * 128,), dtype=torch.float32, device=step.device)
            dist.all_gather_into_tensor(gathered, step.send(plan), group=group)
            blk = step.match(plan, step.compact(plan, gathered.view(step.world, plan.P, 128)))
            nn_all = torch.empty((step.world * 4 * plan.Q,), dtype=torch.int32, device=step.device)
            dist.all_gather_into_tensor(nn_all, blk, group=group)
            step.merge(plan, nn_all.view(step.world, 4 * plan.Q))
        res = step.frames(plan)
        res_all = torch.empty((step.world * step.block.words,), dtype=torch.int32, device=step.device)
        dist.all_gather_into_tensor(res_all, res, group=group)
        return step.unpack(plan, res_all.view(step.world, step.block.words))
