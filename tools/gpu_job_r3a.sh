#!/bin/bash
# round-3 GPU job A: compact gossip records (key / body ring planes).  A/B of the flagship against the parent
# commit's library (maelstrom_b200/libmaelstrom_b200_base.so, built from a worktree of the parent), output
# equality, the other configs, the gpu suite, smoke and a memcheck pass over the broadcast parity cases.
# Usage: tools/gpu_job_r3a.sh OUTDIR (logs, bench JSON lines and dumped outputs go there)
O=${1:?usage: gpu_job_r3a.sh OUTDIR}
mkdir -p $O
BASE=$PWD/maelstrom_b200/libmaelstrom_b200_base.so
NEW=$PWD/maelstrom_b200/libmaelstrom_b200.so
nvidia-smi --query-gpu=name,power.limit,clocks.sm,clocks.max.sm,clocks.mem --format=csv > $O/gpu.csv 2>&1
cat $O/gpu.csv
python -c "import __graft_entry__ as G; G.build()" > $O/build.log 2>&1 || { echo "build failed"; tail $O/build.log; exit 1; }
# flagship, alternating base / new, three times each (device arm only)
for k in 1 2 3; do
  for v in base new; do
    if [ $v = base ]; then L=$BASE; else L=$NEW; fi
    MS_B200_LIB=$L timeout 300 python bench.py --steps 10 --warmup 3 --no-cpu --no-e2e > $O/flag_${v}_$k.json 2> $O/flag_${v}_$k.err
    echo "rc=$?" >> $O/flag_${v}_$k.err
  done
done
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
# the default bench (with the e2e leg), base and new
MS_B200_LIB=$BASE timeout 600 python bench.py --steps 10 --warmup 3 > $O/bench_default_base.json 2> $O/bench_default_base.err
timeout 600 python bench.py --steps 10 --warmup 3 > $O/bench_default.json 2> $O/bench_default.err
# the other configs, base and new alternating, twice each
for k in 1 2; do
  for c in broadcast-lat1:6 gset16k:3 raft64k:6 txn256k:6; do
    cfg=${c%%:*}; st=${c##*:}
    for v in base new; do
      if [ $v = base ]; then L=$BASE; else L=$NEW; fi
      MS_B200_LIB=$L timeout 300 python bench.py --config $cfg --steps $st --warmup 3 --no-cpu --no-e2e > $O/cfg_${cfg}_${v}_$k.json 2> $O/cfg_${cfg}_${v}_$k.err
    done
  done
done
timeout 900 python -m pytest tests -m gpu -q -p no:cacheprovider > $O/pytest_gpu.log 2>&1
echo "pytest rc=$?" >> $O/pytest_gpu.log
timeout 300 python __graft_entry__.py smoke > $O/smoke.log 2>&1
echo "smoke rc=$?" >> $O/smoke.log
python - <<PY > $O/summary.txt 2>&1
import json, statistics
def val(f):
    try:
        d = json.load(open(f)); return d["ms_per_step"], d["value"]
    except Exception as e:
        return None, str(e)
for v in ("base", "new"):
    ms = [val("$O/flag_%s_%d.json" % (v, k))[0] for k in (1, 2, 3)]
    print("flagship", v, "ms_per_step", ms, "median", statistics.median([m for m in ms if m is not None] or [0]))
for f in ("bench_default_base", "bench_default"):
    try:
        d = json.load(open("$O/%s.json" % f)); print(f, "value", d["value"], "e2e", d["e2e"]["value"])
    except Exception as e:
        print(f, e)
for c in ("broadcast-lat1", "gset16k", "raft64k", "txn256k"):
    print(c, "base", [val("$O/cfg_%s_base_%d.json" % (c, k))[0] for k in (1, 2)],
          "new", [val("$O/cfg_%s_new_%d.json" % (c, k))[0] for k in (1, 2)])
PY
cat $O/summary.txt
tail -n 2 $O/pytest_gpu.log $O/smoke.log
# memcheck over the broadcast parity cases on the GPU (the ring layout changed: out-of-bounds is the risk)
if command -v compute-sanitizer > /dev/null; then
  timeout 900 compute-sanitizer --tool memcheck --error-exitcode 9 python -m pytest tests/test_gpu_parity.py \
    tests/test_compact_gossip.py -m gpu -q -p no:cacheprovider -k "cuda and not heavy and not 4096 and not smoke" \
    > $O/memcheck.log 2>&1
  echo "memcheck rc=$?" >> $O/memcheck.log
  tail -n 4 $O/memcheck.log
else
  echo "compute-sanitizer not available" | tee $O/memcheck.log
fi
