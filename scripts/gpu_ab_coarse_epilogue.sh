#!/bin/bash
# A/B of the coarse kernel's epilogue on one GPU, A = a build of the previous commit, B = this tree:
#   git stash / checkout the previous commit; MOPED_LIB=$PWD/moped_b200/lib/libmoped_cuda_parent.so python -m moped_b200.build --force
#   back to this tree; python -m moped_b200.build --force; the libmoped_cuda_dbg{1,2,3}.so libraries compiled with -DMC_COARSE_DBG=n
# Part "coarse": alternates A and B three times on the coarse kernel of the 1 M x 128 000 pass, compares their results array by
# array, then times the DBG decomposition and the 125 k-row shard. Part "bench": alternates A and B three times on bench.py's
# default line and compares the dumped results. Everything goes to OUTDIR.   usage: gpu_ab_coarse_epilogue.sh coarse|bench OUTDIR
set -u
if [ $# -ne 2 ] || { [ "$1" != coarse ] && [ "$1" != bench ]; }; then echo "usage: $0 coarse|bench OUTDIR" >&2; exit 2; fi
PART=$1
O=$2; mkdir -p "$O"
A=$PWD/moped_b200/lib/libmoped_cuda_parent.so; B=$PWD/moped_b200/lib/libmoped_cuda.so
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm,temperature.gpu --format=csv | tee -a $O/gpu.txt
cmp_dirs() {   # cmp_dirs PREFIX: are the .npy files of PREFIX_A<r> and PREFIX_B<r> equal, for r = 1..3?
  python - "$1" <<'PY'
import os, sys, numpy as np
p = sys.argv[1]
def same(a, b):
    fa, fb = sorted(os.listdir(a)), sorted(os.listdir(b))
    return fa == fb and len(fa) > 0 and all(np.array_equal(np.load(os.path.join(a, f)), np.load(os.path.join(b, f))) for f in fa if f.endswith(".npy"))
print({f"{p}_A{r}_vs_B{r}": same(f"{p}_A{r}", f"{p}_B{r}") for r in (1, 2, 3) if os.path.isdir(f"{p}_A{r}") and os.path.isdir(f"{p}_B{r}")})
PY
}
if [ "$PART" = coarse ]; then
  for r in 1 2 3; do
    for v in A B; do
      L=$A; [ $v = B ] && L=$B
      MOPED_LIB=$L DBG_CONFIGS=1:0:1 DBG_ITERS=10 DBG_SAVE=$O/nn_$v$r timeout 200 python scripts/gpu_coarse_dbg.py ab_$v$r 2>>$O/err.txt | tee -a $O/coarse_ab.jsonl
    done
  done
  cmp_dirs $O/nn | tee -a $O/compare.txt
  for d in 1 2 3; do
    MOPED_LIB=$PWD/moped_b200/lib/libmoped_cuda_dbg$d.so DBG_CONFIGS=1:0:1 DBG_ITERS=8 timeout 200 python scripts/gpu_coarse_dbg.py dbg$d 2>>$O/err.txt | tee -a $O/coarse_dbg.jsonl
  done
  for v in A B; do
    L=$A; [ $v = B ] && L=$B
    MOPED_LIB=$L DBG_OBJECTS=125 DBG_CONFIGS=1:0:1 timeout 200 python scripts/gpu_coarse_dbg.py shard125k_$v 2>>$O/err.txt | tee -a $O/coarse_125k.jsonl
  done
else
  for r in 1 2 3; do
    for v in A B; do
      L=$A; [ $v = B ] && L=$B
      MOPED_LIB=$L timeout 200 python bench.py --gpus 1 --steps 20 --warmup 3 --other-configs 0 --no-cpu-baseline --dump-outputs $O/dump_$v$r \
        2>>$O/err.txt | grep '^{' | tee $O/bench_$v$r.json | cut -c1-200
    done
  done
  cmp_dirs $O/dump | tee -a $O/compare.txt
fi
