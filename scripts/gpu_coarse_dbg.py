"""Timing of the coarse matching kernels on the bench's MATCH pass (1 M rows x 128 000 queries of the synthetic workload), run on the
GPU box:  python scripts/gpu_coarse_dbg.py [label]   — per coarse kind (8-bit cascade / fp16 only) and reserved-SM count: device
time of the dominant kernel (events inside the library), of the whole mc_match_dev pass, and the cascade's tier counts.
MOPED_LIB selects another build of the library (e.g. one compiled with -DMC_COARSE_DBG=1). DBG_SAVE=DIR writes every configuration's
nn_row / nn_dist / accepted to DIR as .npy files, so that the results of two builds can be compared array by array."""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402
from moped_b200 import capi, synth  # noqa: E402

label = sys.argv[1] if len(sys.argv) > 1 else "default"
if os.environ.get("DBG_OLD"):          # a build of the library from before the cascade: no tier statistics
    capi.SIGNATURES.pop("mc_match_tier_stats", None)
OBJ, B, Q = int(os.environ.get("DBG_OBJECTS", 1000)), int(os.environ.get("DBG_FRAMES", 64)), 2000


def nrm(x):
    n = np.sqrt((x * x).sum(1, dtype=np.float32))
    return (x / n[:, None]).astype(np.float32)


db = synth.make_db(OBJ, 1000)
dbn = nrm(db["desc"])
qn = np.concatenate([nrm(synth.make_frame(db, Q, n_visible=8, frame_id=i)["desc"]) for i in range(B)])
QT = len(qn)
q = torch.from_numpy(qn).cuda()
ctx = capi.Context(0)
ctx.db_upload(dbn, db["xyz"], db["model_of_row"], OBJ)
ctx.set_profiling(True)
nn_row = torch.empty((QT, 2), dtype=torch.int32, device="cuda")
nn_dist = torch.empty((QT, 2), dtype=torch.float32, device="cuda")
acc = torch.empty((QT,), dtype=torch.uint8, device="cuda")
ref = None
import subprocess  # noqa: E402
old_lib = bool(os.environ.get("DBG_OLD"))
configs = ((0, 0, 0),) if old_lib else tuple(tuple(int(v) for v in c.split(":")) for c in os.environ.get("DBG_CONFIGS", "1:0:1,1:0:0,0:0:1,0:0:0,1:8:1").split(","))
splits_list = [int(v) for v in os.environ.get("DBG_SPLITS", "0").split(",")]
for kind, reserve, stagger, splits in [(c[0], c[1], c[2], sp) for c in configs for sp in splits_list]:
    if not old_lib:
        ctx.set_option("match_splits", splits)
        ctx.set_option("match_coarse_kind", kind)
        ctx.set_option("match_reserve_sms", reserve)
        ctx.set_option("match_stagger", stagger)
    ms, tot = [], []
    smi = subprocess.Popen(["nvidia-smi", "--id=0", "--query-gpu=clocks.sm,power.draw", "--format=csv,noheader,nounits", "-lms", "20"],
                           stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
    for i in range(int(os.environ.get("DBG_ITERS", 12))):
        import time
        torch.cuda.synchronize()
        t0 = time.perf_counter()                 # (the context runs its own stream: wall clock around the synchronised pass, launch overhead included)
        ctx.match_dev(q.data_ptr(), QT, 0.8, capi.MATCH_TENSOR, nn_row.data_ptr(), nn_dist.data_ptr(), acc.data_ptr())
        ctx.synchronize()
        tot.append((time.perf_counter() - t0) * 1e3)
        torch.cuda.synchronize()
        ms.append(ctx.coarse_kernel_ms())
    smi.terminate()
    clk = [ln.split(",") for ln in smi.stdout.read().strip().splitlines() if "," in ln]
    sm_mhz = float(np.median([float(c[0]) for c in clk])) if clk else None
    watts = float(np.median([float(c[1]) for c in clk])) if clk else None
    res = (nn_row.cpu().numpy().copy(), nn_dist.cpu().numpy().copy(), acc.cpu().numpy().copy())
    same = True if ref is None else all(np.array_equal(a, b) for a, b in zip(ref, res))
    ref = ref or res
    if os.environ.get("DBG_SAVE"):
        os.makedirs(os.environ["DBG_SAVE"], exist_ok=True)
        for name, arr in zip(("nn_row", "nn_dist", "accepted"), res):
            np.save(os.path.join(os.environ["DBG_SAVE"], f"k{kind}_r{reserve}_s{stagger}_p{splits}_{name}.npy"), arr)
    km = float(np.median(ms[2:]))
    print(json.dumps({"label": label, "coarse_kind": kind, "reserve_sms": reserve, "stagger": stagger, "splits": splits, "rows": len(dbn), "queries": QT, "coarse_ms": km, "match_ms": float(np.median(tot[2:])),
                      "tera_ops": 2.0 * len(dbn) * QT * 128 / (km * 1e-3) / 1e12,
                      "sm_mhz": sm_mhz, "watts": watts, "clock_samples": len(clk),
                      "tiers": None if old_lib else ctx.match_tier_stats().tolist(), "stats": ctx.match_last_stats().tolist(), "same_bits_as_first": same}), flush=True)
