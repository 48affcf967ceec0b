"""Time the store self-join (isx_self_join) on the device and check its parity at that scale.

    python profiles/join_bench.py [--rows 10000000] [--thr 1/8] [--out profiles/r04_join_10M.json]

Builds a synthetic store on the device (isx_synth_rows_device + isx_add_device: mixed 64..256-bit rows, every
`--dup-every`-th row repeats the code of the row `--dup-back` before it, cut to its own length), runs one join to warm
up, then times one join between device synchronisations with CUDA events and runs one more with profiling on for the
scan time. Parity: for a seeded sample of rows, the partners the join reports must equal those of the CPU oracle's
exact threshold top-k over all rows (oracle synth_topk, regenerating the rows). Prints one JSON line; exits 1 on a
mismatch.
"""

import argparse
import json
import subprocess
import sys
from fractions import Fraction
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from iscc_search_b200 import _lib  # noqa: E402
from oracle import c_oracle  # noqa: E402


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", "0"], capture_output=True, text=True)
    if r.returncode != 0:
        return {"card": None, "nvidia_smi": r.stderr.strip()[-200:]}
    name, power, sm, sm_max = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
    return {"card": name, "power_limit_w": power, "sm_clock_mhz": sm, "sm_max_mhz": sm_max}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--lengths", default="8,16,24,32")
    ap.add_argument("--dup-every", type=int, default=1000)
    ap.add_argument("--dup-back", type=int, default=777)
    ap.add_argument("--thr", default="1/8", help="NPHD threshold as a fraction")
    ap.add_argument("--sample", type=int, default=64, help="rows whose partners are checked against the oracle")
    ap.add_argument("--k", type=int, default=4096, help="oracle top-k per sampled row (must exceed its partner count)")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    import torch

    lengths = tuple(int(x) for x in args.lengths.split(","))
    thr = Fraction(args.thr)
    thr_t = (thr.numerator, thr.denominator)

    st = _lib.Store(key_bytes=8, max_bytes=32)
    dev = torch.device("cuda", 0)
    chunk = min(8_000_000, args.rows)
    d_keys = torch.empty(chunk * 8, dtype=torch.uint8, device=dev)
    d_codes = torch.empty(chunk * 32, dtype=torch.uint8, device=dev)
    d_lens = torch.empty(chunk, dtype=torch.uint8, device=dev)
    for c0 in range(0, args.rows, chunk):
        cn = min(chunk, args.rows - c0)
        st.synth_rows_device(args.seed, c0, cn, d_keys.data_ptr(), d_codes.data_ptr(), d_lens.data_ptr(), lengths=lengths,
                             dup_every=args.dup_every, dup_back=args.dup_back)
        st.add_device(d_keys.data_ptr(), d_codes.data_ptr(), d_lens.data_ptr(), cn)
    del d_keys, d_codes, d_lens
    torch.cuda.empty_cache()

    st.self_join(thr_t)   # warm-up: modules, rank tables, working memory
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    total = ctypes_join(st, thr_t)   # synchronous: returns after the sort finished on the store's stream
    e1.record()
    torch.cuda.synchronize()
    join_ms = e0.elapsed_time(e1)
    timed = st.stats()
    info = gpu_info()   # right after the timed join, in the same command
    st.set_profiling(True)
    ka, kb, h, nb = st.self_join(thr_t)
    prof = st.stats()
    st.set_profiling(False)

    # half random rows, half planted duplicates and the rows they copy (each of those has at least one partner)
    rng = np.random.default_rng(args.seed + 17)
    n_s = min(args.sample, args.rows)
    dups = np.arange(args.dup_every - 1, args.rows, args.dup_every) if args.dup_every else np.zeros(0, dtype=np.int64)
    dups = dups[dups >= args.dup_back]
    picked = rng.choice(dups, size=min(n_s // 4, len(dups)), replace=False) if len(dups) else dups
    planted = np.concatenate([picked, picked - args.dup_back]).astype(np.int64)
    rest = rng.choice(args.rows, size=n_s - len(planted), replace=False)
    sample = np.unique(np.concatenate([planted, rest]))
    rows = [c_oracle.synth_rows(int(i), 1, args.seed, lengths=lengths, dup_every=args.dup_every, dup_back=args.dup_back) for i in sample]
    skeys = np.array([r[0][0] for r in rows], dtype=np.uint64)
    queries = np.concatenate([r[2] for r in rows])
    qlens = np.concatenate([r[3] for r in rows])
    okeys, _, oh, onb, ocnt = c_oracle.synth_topk(args.rows, args.seed, queries, qlens, args.k, lengths=lengths, dup_every=args.dup_every,
                                                  dup_back=args.dup_back, max_h_over_n=thr_t)
    mismatches = []
    for j, key in enumerate(skeys):
        c = int(ocnt[j])
        if c >= args.k:
            mismatches.append({"row": int(sample[j]), "why": f"oracle k={args.k} too small"})
            continue
        exp = sorted((int(okeys[j, t]), int(oh[j, t]), int(onb[j, t])) for t in range(c) if okeys[j, t] != key)
        ia, ib = np.nonzero(ka == key)[0], np.nonzero(kb == key)[0]
        got = sorted([(int(kb[i]), int(h[i]), int(nb[i])) for i in ia] + [(int(ka[i]), int(h[i]), int(nb[i])) for i in ib])
        if got != exp:
            mismatches.append({"row": int(sample[j]), "expected": len(exp), "got": len(got)})
    ordered = bool(np.all((ka[:-1] < ka[1:]) | ((ka[:-1] == ka[1:]) & (kb[:-1] < kb[1:])))) and bool(np.all(ka < kb))
    partners = int(sum(int(ocnt[j]) - 1 for j in range(len(skeys))))
    res = {
        "what": "isx_self_join", "rows": args.rows, "lengths": list(lengths), "dup_every": args.dup_every, "dup_back": args.dup_back,
        "threshold": f"{thr.numerator}/{thr.denominator}", "join_s": round(join_ms / 1e3, 3), "pairs_scored": int(timed["pairs"]),
        "pairs_per_s": float(f"{timed['pairs'] / (join_ms / 1e3):.4g}"), "pairs_found": int(total), "scan_ms": round(prof["scan_ms"], 1),
        "profiled_total_ms": round(prof["total_ms"], 1), "scan_launches": int(timed["scan_launches"]), "chunks": int(timed["passes"]),
        "candidates": int(timed["candidates"]), "overflow_rescan_rows": int(timed["fallback_queries"]),
        "parity": not mismatches and ordered and len(h) == total, "parity_sample_rows": len(skeys), "parity_sample_partners": partners,
        "mismatches": mismatches[:8], **info,
    }
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).write_text(line + "\n")
    st.close()
    return 0 if res["parity"] else 1


def ctypes_join(st, thr):
    """The join alone (no fetch): isx_self_join, returning the number of pairs."""
    import ctypes

    total = ctypes.c_uint64()
    _lib.check(_lib.lib().isx_self_join(st.handle, thr[0], thr[1], ctypes.byref(total)))
    return int(total.value)


if __name__ == "__main__":
    sys.exit(main())
