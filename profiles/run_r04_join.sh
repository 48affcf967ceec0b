#!/bin/bash
# Self-join round: the join's own GPU tests, the 10 M-row join measurement with its parity check, then the whole GPU
# suite, smoke() and the default bench line (the existing scan kernels are unchanged; the bench line shows it).
# Usage: profiles/run_r04_join.sh OUTDIR [join|suite]   (from the repository root; everything the run writes goes to
# OUTDIR; "join" runs the first half only, "suite" the second)
OUT=${1:?usage: run_r04_join.sh OUTDIR [join|suite]}
PART=${2:-all}
mkdir -p "$OUT"
if [ "$PART" != suite ]; then
timeout 900 python -m pytest tests/test_gpu_self_join.py -x -q 2>&1 | tail -5 | tee $OUT/r04_gpu_self_join_tests.txt
timeout 1200 python profiles/join_bench.py --out $OUT/r04_join_10M.json 2> $OUT/r04_join_10M.err; echo "join_bench rc=$?"
timeout 600 python bench.py > $OUT/r04_cfg3_n1.json 2> $OUT/r04_cfg3_n1.err; echo "bench rc=$?"
fi
[ "$PART" = join ] && exit 0
timeout 1800 python -m pytest tests -m gpu -q 2>&1 | tail -4 | tee $OUT/r04_gpu_suite.txt
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -1 | tee -a $OUT/r04_gpu_suite.txt
