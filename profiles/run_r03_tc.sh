#!/bin/bash
# Tensor-core scan round: micro-benchmark, GPU suite, smoke, and the bench A/B of the POPC scan (ISX_TC_SCAN=0) against
# the tensor-core scan on the same build, alternating, with output dumps compared file by file.
# Usage: profiles/run_r03_tc.sh OUTDIR   (from the repository root; everything the run writes goes to OUTDIR)
OUT=${1:?usage: run_r03_tc.sh OUTDIR}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm --format=csv | tee $OUT/r03_tc_b200.txt
nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -o $OUT/tc_hamming profiles/microbench/tc_hamming.cu \
  && timeout 120 $OUT/tc_hamming 2>&1 | tee -a $OUT/r03_tc_b200.txt
timeout 900 python -m pytest tests/test_gpu_tc_scan.py -x -q 2>&1 | tail -15
for i in 1 2 3; do
  for tc in 0 1; do
    ISX_TC_SCAN=$tc timeout 600 python bench.py > $OUT/r03_cfg3_n1_tc${tc}_$i.json 2> $OUT/r03_cfg3_n1_tc${tc}_$i.err
    echo "bench tc=$tc run $i rc=$?"
  done
done
for tc in 0 1; do
  ISX_TC_SCAN=$tc timeout 600 python bench.py --steps 1 --warmup 1 --dump-outputs $OUT/dump_tc$tc > /dev/null 2>&1; echo "dump tc=$tc rc=$?"
done
OUT="$OUT" python - <<'PY'
import json, glob, os
import numpy as np
for f in sorted(glob.glob(os.environ["OUT"] + "/r03_cfg3_n1_tc*.json")):
    try:
        d = json.loads(open(f).read().strip().splitlines()[-1])
        print(os.path.basename(f), round(d["ms_per_step"], 2), "e2e", round(d["e2e"]["ms_per_step"], 2), "bit_exact", d["parity"]["bit_exact"], d.get("clocks"))
    except Exception as e:
        print(f, "unreadable", e)
a, b = sorted(glob.glob(os.environ["OUT"] + "/dump_tc0/**/*.npy", recursive=True)), sorted(glob.glob(os.environ["OUT"] + "/dump_tc1/**/*.npy", recursive=True))
same = len(a) == len(b) > 0 and all(open(x, "rb").read() == open(y, "rb").read() for x, y in zip(a, b))
print("dumps", len(a), len(b), "byte-identical" if same else "DIFFER")
PY
timeout 1500 python -m pytest tests -m gpu -x -q 2>&1 | tail -4
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -1
rm -rf $OUT/dump_tc0 $OUT/dump_tc1 $OUT/tc_hamming
