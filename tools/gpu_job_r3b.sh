#!/bin/bash
# round-3 GPU job B: endpoint lifecycle.  The gpu suite (with the [cuda] lifecycle cases), a sweep of lifecycle
# seeds on the product library, smoke, and the flagship's dumped outputs and time against the parent commit's
# library (maelstrom_b200/libmaelstrom_b200_base.so, built from a worktree of the parent).
# Usage: tools/gpu_job_r3b.sh OUTDIR [SEEDS]  (logs, bench JSON lines and dumped outputs go to OUTDIR)
O=${1:?usage: gpu_job_r3b.sh OUTDIR [SEEDS]}
SEEDS=${2:-0:400}
mkdir -p $O
BASE=$PWD/maelstrom_b200/libmaelstrom_b200_base.so
NEW=$PWD/maelstrom_b200/libmaelstrom_b200.so
nvidia-smi --query-gpu=name,power.limit,clocks.sm,clocks.max.sm,clocks.mem --format=csv > $O/gpu.csv 2>&1
cat $O/gpu.csv
python -c "import __graft_entry__ as G; G.build()" > $O/build.log 2>&1 || { echo "build failed"; tail $O/build.log; exit 1; }
timeout 900 python -m pytest tests -q -m gpu -p no:cacheprovider > $O/pytest_gpu.log 2>&1
echo "pytest rc=$?" >> $O/pytest_gpu.log
tail -n 3 $O/pytest_gpu.log
MS_LIFECYCLE_SEEDS=$SEEDS timeout 1200 python -m pytest tests/test_lifecycle_fuzz.py -q -m gpu -k scenario \
  -p no:cacheprovider > $O/lifecycle_cuda.log 2>&1
echo "lifecycle seeds $SEEDS rc=$?" >> $O/lifecycle_cuda.log
tail -n 3 $O/lifecycle_cuda.log
timeout 300 python -c "import __graft_entry__ as G; G.smoke()" > $O/smoke.log 2>&1
echo "smoke rc=$?" >> $O/smoke.log
tail -n 2 $O/smoke.log
# what the timed steps computed, both libraries
for v in base new; do
  if [ $v = base ]; then L=$BASE; else L=$NEW; fi
  MS_B200_LIB=$L timeout 300 python bench.py --steps 10 --warmup 3 --no-cpu --no-e2e --dump-outputs $O/dump_$v > $O/dump_$v.json 2> $O/dump_$v.err
done
python - <<PY > $O/dump_compare.txt 2>&1
import glob, os, numpy as np
a, b = "$O/dump_base", "$O/dump_new"
fa = sorted(os.path.basename(f) for f in glob.glob(a + "/*.npy"))
fb = sorted(os.path.basename(f) for f in glob.glob(b + "/*.npy"))
print("files", len(fa), len(fb), fa == fb)
bad = [f for f in fa if f in fb and not np.array_equal(np.load(a + "/" + f), np.load(b + "/" + f))]
print("differ:", bad)
print("IDENTICAL" if fa == fb and fa and not bad else "DIFFERENT")
PY
cat $O/dump_compare.txt
# flagship, alternating base / new, twice each
for k in 1 2; do
  for v in base new; do
    if [ $v = base ]; then L=$BASE; else L=$NEW; fi
    MS_B200_LIB=$L timeout 300 python bench.py --gpus 1 --steps 10 --warmup 3 > $O/flag_${v}_$k.json 2> $O/flag_${v}_$k.err
    echo "rc=$?" >> $O/flag_${v}_$k.err
    tail -c 400 $O/flag_${v}_$k.json
  done
done
