"""
GPU tests of the tensor-core scan's compare epilogue (csrc/tc.cuh, tc_compare_tile): accumulators and bounds are compared
as packed 16-bit halves, so the edges of that encoding are checked here against the CPU oracle and against the POPC scan
(ISX_TC_SCAN=0, read once per process, hence a subprocess):
  * rows exactly on a fixed threshold and one bit past it, at every compared length 1..32 bytes
  * the accumulator extremes: acc = -256 (all-ones rows, all-ones query) and acc = +256 (all-ones rows, all-zero query,
    a threshold that accepts every row)
  * query tiles whose width is not a multiple of 32, so that padding columns are read
  * byte-granular mixed lengths in top-k mode
"""

import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from iscc_search_b200 import synth
from iscc_search_b200._lib import Store
from tests.helpers import assert_same_topk, make_store_arrays, oracle_topk

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent
QUERIES_PER_LENGTH = 64   # the smallest query tile that takes the tensor-core scan


def _flip(rng, code, L, nflip):
    bits = np.unpackbits(code[:L])
    bits[rng.choice(8 * L, size=nflip, replace=False)] ^= 1
    out = code.copy()
    out[:L] = np.packbits(bits)
    return out


def bound_case(thr, per_length=QUERIES_PER_LENGTH, lengths=tuple(range(1, 33)), row_steps=(0,), n_fill=2048):
    """
    For every query length L of `lengths`, `per_length` random queries of L bytes (one count for all lengths, or one per
    length). Per query and per step s of `row_steps`, the row length Lr is the length s places from L in `lengths` (where
    that exists); one row of Lr bytes lies exactly on the threshold (h = floor(thr * 8m), m = min(L, Lr)) and one a bit
    past it. A row longer than its query holds 0xFF past the query's length, so that those bytes differ from the query's
    zero padding. Plus `n_fill` random rows of the lengths.
    -> (keys, codes, lens, queries, qlens, on_rows, past_rows, owner): owner[i] is the query of on_rows[i] / past_rows[i]
    """
    num, den = thr
    rng = np.random.default_rng(6100 + 10 * num + den)
    counts = [per_length] * len(lengths) if np.isscalar(per_length) else list(per_length)
    queries, qlens, rows, lens, on_rows, past_rows, owner = [], [], [], [], [], [], []
    for i, L in enumerate(lengths):
        for _ in range(counts[i]):
            q = np.zeros(32, dtype=np.uint8)
            q[:L] = rng.integers(0, 256, size=L, dtype=np.uint8)
            for s in row_steps:
                if not 0 <= i + s < len(lengths):
                    continue
                Lr = lengths[i + s]
                m = min(L, Lr)
                hb = num * 8 * m // den
                for pos, nflip in ((on_rows, hb), (past_rows, hb + 1)):
                    row = _flip(rng, q, m, nflip)
                    row[m:Lr] = 0xFF
                    row[Lr:] = 0
                    pos.append(len(rows))
                    rows.append(row)
                    lens.append(Lr)
                owner.append(len(queries))
            queries.append(q)
            qlens.append(L)
    fill_lens = np.asarray(lengths, dtype=np.uint8)[rng.integers(0, len(lengths), size=n_fill)]
    fill = rng.integers(0, 256, size=(n_fill, 32), dtype=np.uint8)
    fill[np.arange(32)[None, :] >= fill_lens[:, None]] = 0
    codes = np.concatenate([np.stack(rows), fill])
    lens = np.concatenate([np.array(lens, dtype=np.uint8), fill_lens])
    keys = synth.make_keys(0, len(lens), 6101 + num)
    return (keys, codes, lens, np.stack(queries), np.array(qlens, dtype=np.uint8), np.array(on_rows), np.array(past_rows),
            np.array(owner))


def ones_case():
    """300 all-ones rows among random ones (32 bytes) against 64 all-ones queries: acc = -256 for the all-ones rows."""
    rng = np.random.default_rng(6201)
    codes = np.concatenate([np.full((300, 32), 0xFF, dtype=np.uint8), rng.integers(0, 256, size=(4000, 32), dtype=np.uint8)])
    lens = np.full(len(codes), 32, dtype=np.uint8)
    queries = np.full((QUERIES_PER_LENGTH, 32), 0xFF, dtype=np.uint8)
    return synth.make_keys(0, len(lens), 6202), codes, lens, queries, np.full(QUERIES_PER_LENGTH, 32, dtype=np.uint8)


def zeros_case():
    """1000 all-ones rows among random ones (32 bytes) against 64 all-zero queries: acc = +256 for the all-ones rows."""
    rng = np.random.default_rng(6301)
    codes = np.concatenate([np.full((1000, 32), 0xFF, dtype=np.uint8), rng.integers(0, 256, size=(500, 32), dtype=np.uint8)])
    lens = np.full(len(codes), 32, dtype=np.uint8)
    queries = np.zeros((QUERIES_PER_LENGTH, 32), dtype=np.uint8)
    return synth.make_keys(0, len(lens), 6302), codes, lens, queries, np.full(QUERIES_PER_LENGTH, 32, dtype=np.uint8)


MIXED_QUERY_LENGTHS = (1, 3, 8, 13, 20, 31, 32)


def mixed_case():
    """150 000 rows of every length 1..32 bytes, 64 queries at each of MIXED_QUERY_LENGTHS."""
    all_lengths = tuple(range(1, 33))
    keys, codes, lens = make_store_arrays(150_000, 6401, lengths=all_lengths)
    qs = [synth.make_queries(QUERIES_PER_LENGTH, len(keys), 6402 + L, 6401, lengths=(L,), row_lengths=all_lengths)
          for L in MIXED_QUERY_LENGTHS]
    return keys, codes, lens, np.concatenate([q for q, _ in qs]), np.concatenate([ql for _, ql in qs])


def _search(case, k, thr=None):
    keys, codes, lens, queries, qlens = case[:5]
    st = Store(key_bytes=8, max_bytes=32)
    try:
        st.add(keys, codes, lens)
        got = st.search(queries, qlens, k, thr=thr)[:4]
        return got, st.stats()
    finally:
        st.close()


def _check(case, k, thr=None):
    keys, codes, lens, queries, qlens = case[:5]
    (gk, gh, gn, gc), stats = _search(case, k, thr)
    rows, h, nb, cnt = oracle_topk(keys, codes, lens, queries, qlens, k, thr)
    assert_same_topk(gk, gh, gn, gc, keys, rows, h, nb, cnt)
    return (gk, gh, gn, gc), stats


def check_bound_rows(case, gk, gc):
    """Every row planted on the bound is in its query's result, every row one bit past it is not."""
    keys, on_rows, past_rows, owner = case[0], case[5], case[6], case[7]
    for on, past, q in zip(on_rows, past_rows, owner):
        got = set(gk[q, : gc[q]].tolist())
        assert int(keys[on]) in got, f"query {q}: the row on the bound is missing"
        assert int(keys[past]) not in got, f"query {q}: the row past the bound is returned"


# 64 queries per length: every length tile takes the tensor-core scan; 16: every tile takes the POPC scan (k_scan)
@pytest.mark.parametrize("thr,per_length", [((1, 8), 64), ((3, 10), 64), ((1, 8), 16), ((3, 10), 16)],
                         ids=["thr0", "thr1", "thr0-popc", "thr1-popc"])
def test_rows_on_the_bound_every_length(cuda, thr, per_length):
    case = bound_case(thr, per_length)
    k = 2048   # above the count of any query (a 1-byte query compares one byte of every row)
    (gk, _, _, gc), stats = _check(case, k, thr)
    if per_length >= QUERIES_PER_LENGTH:
        assert stats["issued_popc"] == 0   # only tensor-core launches
    else:
        assert stats["issued_popc"] > 0   # tiles of 16 queries: the POPC scan
    assert (gc < k).all()              # every row within the threshold is in the result
    check_bound_rows(case, gk, gc)


def test_accumulator_minus_256(cuda):
    (_, gh, _, gc), _ = _check(ones_case(), 400)
    assert (gc == 400).all() and (gh[:, :300] == 0).all()


def test_accumulator_plus_256_every_row_returns(cuda):
    case = zeros_case()
    n = len(case[0])
    (_, gh, _, gc), stats = _check(case, n, thr=(1, 1))
    assert (gc == n).all()                     # every row passes
    assert ((gh == 256).sum(axis=1) == 1000).all()
    assert stats["fallback_queries"] == 0      # emitted by the tensor-core scan, not by the exact re-scan


@pytest.fixture(scope="module")
def wide_store(cuda):
    # 1.25 M rows of one length: 1221 blocks of 1024 rows, at least 4 waves of 2 CTAs on 148 SMs, so the main range of a
    # search keeps all T <= 256 queries of a length in one CTA (tile width T); its first, shorter ranges split them
    n = 1_250_000
    keys, codes, lens = make_store_arrays(n, 6501, lengths=(32,))
    st = Store(key_bytes=8, max_bytes=32)
    st.add(keys, codes, lens)
    yield st, keys, codes, lens
    st.close()


@pytest.mark.parametrize("T", [64, 65, 97, 250, 256])
def test_padding_columns(wide_store, T):
    st, keys, codes, lens = wide_store
    q, ql = synth.make_queries(T, len(keys), 6600 + T, 6501, lengths=(32,), row_lengths=(32,))
    gk, gh, gn, gc, _ = st.search(q, ql, 50)
    assert st.stats()["issued_popc"] == 0   # only tensor-core launches
    rows, h, nb, cnt = oracle_topk(keys, codes, lens, q, ql, 50)
    assert_same_topk(gk, gh, gn, gc, keys, rows, h, nb, cnt)


def test_mixed_lengths_topk(cuda):
    _check(mixed_case(), 100)


_AB_SCRIPT = r"""
import json, sys
import numpy as np
sys.path.insert(0, sys.argv[1])
from tests import test_gpu_tc_epilogue as t
out, popc = {}, {}
for name, case, k, thr in (("bound", t.bound_case((1, 8)), 2048, (1, 8)), ("plus256", t.zeros_case(), 1500, (1, 1)),
                           ("mixed", t.mixed_case(), 100, None)):
    (gk, gh, gn, gc), stats = t._search(case, k, thr)
    out.update({name + "_keys": gk, name + "_h": gh, name + "_nb": gn, name + "_cnt": gc})
    popc[name] = stats["issued_popc"]
np.savez(sys.argv[2], **out)
print(json.dumps(popc))
"""


def test_same_results_as_popc_scan(cuda, tmp_path):
    out = {}
    for flag in ("1", "0"):
        env = dict(os.environ, ISX_TC_SCAN=flag)
        r = subprocess.run([sys.executable, "-c", _AB_SCRIPT, str(ROOT), str(tmp_path / f"tc{flag}.npz")], capture_output=True,
                           text=True, timeout=600, cwd=str(ROOT), env=env)
        assert r.returncode == 0, r.stderr[-2000:]
        out[flag] = (json.loads(r.stdout.strip().splitlines()[-1]), np.load(tmp_path / f"tc{flag}.npz"))
    assert out["1"][0]["bound"] == 0 and out["0"][0]["bound"] > 0   # each arm took the path it names
    for name in out["1"][1].files:
        assert np.array_equal(out["1"][1][name], out["0"][1][name]), name
