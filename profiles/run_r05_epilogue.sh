#!/bin/bash
# Packed 16-bit compare epilogue of the tensor-core scan (DESIGN.md §3.0): the card and its clocks, the micro-benchmark
# (packed-read check, s32 and s16x2 epilogue rates at 1 and 2 CTAs per SM), bench A/B of the parent commit's library
# against this build, the GPU suite and smoke().
# The parent library is built from the parent commit (make -C iscc_search_b200/csrc in a checkout of it) and placed at
# ab_libs/parent/libisx_b200.so (ignored by git); bench.py loads it through ISX_LIB_PATH. A/B: three alternating cfg3
# pairs, --dump-outputs of both compared byte for byte, one pair each of a cfg5-shaped run (100 M rows of 256 bits,
# 20 000 queries: every compare 8 words) and of cfg4 at 100 M rows (threshold mode).
# Usage: profiles/run_r05_epilogue.sh OUTDIR [quick]   (from the repository root; everything the run writes goes to
# OUTDIR; "quick" stops after the micro-benchmark, the tensor-core tests and one cfg3 pair)
OUT=${1:?usage: run_r05_epilogue.sh OUTDIR [quick]}
MODE=${2:-all}
PARENT=ab_libs/parent/libisx_b200.so
mkdir -p "$OUT"
[ -f "$PARENT" ] || { echo "missing $PARENT"; exit 1; }
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm,clocks_throttle_reasons.active --format=csv | tee $OUT/r05_tc_b200.txt
nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -o $OUT/tc_hamming profiles/microbench/tc_hamming.cu \
  && timeout 300 $OUT/tc_hamming 2>&1 | tee -a $OUT/r05_tc_b200.txt

bench() {   # bench NAME parent|new ARGS...
    local name=$1 arm=$2
    shift 2
    if [ "$arm" = parent ]; then
        ISX_LIB_PATH=$PARENT timeout 900 python bench.py --no-cpu-baseline "$@" > $OUT/$name.json 2> $OUT/$name.err
    else
        timeout 900 python bench.py --no-cpu-baseline "$@" > $OUT/$name.json 2> $OUT/$name.err
    fi
    echo "$name rc=$?"
}

if [ "$MODE" = quick ]; then
    timeout 900 python -m pytest tests/test_gpu_tc_epilogue.py tests/test_gpu_tc_scan.py -q 2>&1 | tail -15
    bench r05_cfg3_n1_parent_1 parent
    bench r05_cfg3_n1_new_1 new
else
    for i in 1 2 3; do
        bench r05_cfg3_n1_parent_$i parent
        bench r05_cfg3_n1_new_$i new
    done
    ISX_LIB_PATH=$PARENT timeout 900 python bench.py --no-cpu-baseline --steps 1 --warmup 1 --dump-outputs $OUT/dump_parent > /dev/null 2>&1
    echo "dump parent rc=$?"
    timeout 900 python bench.py --no-cpu-baseline --steps 1 --warmup 1 --dump-outputs $OUT/dump_new > /dev/null 2>&1
    echo "dump new rc=$?"
    bench r05_cfg5_100M_parent parent --config cfg5 --rows 100000000 --queries 20000
    bench r05_cfg5_100M_new new --config cfg5 --rows 100000000 --queries 20000
    bench r05_cfg4_100M_parent parent --config cfg4 --rows 100000000
    bench r05_cfg4_100M_new new --config cfg4 --rows 100000000
fi

OUT="$OUT" python - <<'PY' | tee $OUT/r05_summary.txt
import glob, json, os, statistics
out = os.environ["OUT"]
arms = {}
for f in sorted(glob.glob(out + "/r05_*.json")):
    name = os.path.basename(f)[:-5]
    try:
        d = json.loads(open(f).read().strip().splitlines()[-1])
    except Exception as e:
        print(name, "unreadable", e)
        continue
    c = d.get("clocks", {})
    print(f"{name:26s} ms_per_step {d['ms_per_step']:9.2f}  bit_exact {d['parity']['bit_exact']}  "
          f"sm_mhz {c.get('sm_mhz')}  reasons {c.get('reasons')}")
    arms.setdefault(name.rsplit("_", 1)[0] if name[-1].isdigit() else name, []).append(d["ms_per_step"])
for shape in ("r05_cfg3_n1", "r05_cfg5_100M", "r05_cfg4_100M"):
    p, n = arms.get(shape + "_parent"), arms.get(shape + "_new")
    if p and n:
        mp, mn = statistics.median(p), statistics.median(n)
        print(f"{shape}: parent median {mp:.2f} ms {sorted(p)}, new median {mn:.2f} ms {sorted(n)}: "
              f"{100 * (1 - mn / mp):.1f} % lower, every new run faster than every parent run: {max(n) < min(p)}")
a = sorted(glob.glob(out + "/dump_parent/**/*.npy", recursive=True))
b = sorted(glob.glob(out + "/dump_new/**/*.npy", recursive=True))
if a or b:
    same = len(a) == len(b) > 0 and all(os.path.basename(x) == os.path.basename(y) and open(x, "rb").read() == open(y, "rb").read()
                                        for x, y in zip(a, b))
    print("cfg3 dumps", len(a), len(b), "byte-identical" if same else "DIFFER")
PY

if [ "$MODE" != quick ]; then
    timeout 1800 python -m pytest tests -m gpu -q 2>&1 | tail -4 | tee $OUT/r05_gpu_suite.txt
    timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -1 | tee -a $OUT/r05_gpu_suite.txt
fi
rm -rf $OUT/dump_parent $OUT/dump_new $OUT/tc_hamming
