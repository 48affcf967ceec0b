"""
GPU tests of the tensor-core batch scan (csrc/tc.cuh, k_scan_tc): batches whose query tiles hold >= 64 queries of one
length take it. Exact parity with the CPU oracle over lengths, k, threshold mode, 128-bit keys, candidate overflow and
multi-tile batches; identity with the POPC scan (ISX_TC_SCAN=0, read once per process, hence a subprocess); and a check
through stats() that the tensor-core path was taken.
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


@pytest.fixture(scope="module")
def mixed_store(cuda):
    n = 120_000
    keys, codes, lens = make_store_arrays(n, 3101)
    st = Store(key_bytes=8, max_bytes=32)
    st.add(keys, codes, lens)
    yield st, keys, codes, lens
    st.close()


def _check(st, keys, codes, lens, queries, qlens, k, thr=None):
    gk, gh, gn, gc, _ = st.search(queries, qlens, k, thr=thr)
    rows, h, nb, cnt = oracle_topk(keys, codes, lens, queries, qlens, k, thr)
    assert_same_topk(gk, gh, gn, gc, keys, rows, h, nb, cnt)


@pytest.mark.parametrize("length", [8, 16, 24, 32])
def test_uniform_length(cuda, length):
    n = 100_000
    keys, codes, lens = make_store_arrays(n, 3200 + length, lengths=(length,))
    st = Store(key_bytes=8, max_bytes=32)
    try:
        st.add(keys, codes, lens)
        q, ql = synth.make_queries(160, n, 3300 + length, 3200 + length, lengths=(length,), row_lengths=(length,))
        _check(st, keys, codes, lens, q, ql, 100)
        assert st.stats()["issued_popc"] == 0   # only tensor-core launches
    finally:
        st.close()


def test_byte_granular_lengths(cuda):
    n = 90_000
    lengths = (5, 13, 30)
    keys, codes, lens = make_store_arrays(n, 3401, lengths=lengths)
    st = Store(key_bytes=8, max_bytes=32)
    try:
        st.add(keys, codes, lens)
        q, ql = synth.make_queries(300, n, 3402, 3401, lengths=lengths, row_lengths=lengths)
        _check(st, keys, codes, lens, q, ql, 50)
    finally:
        st.close()


@pytest.mark.parametrize("k", [1, 100, 1000, 4096])
def test_mixed_lengths_every_query_length(mixed_store, k):
    st, keys, codes, lens = mixed_store
    q, ql = synth.make_queries(400, len(keys), 3500 + k, 3101)
    assert set(np.unique(ql).tolist()) == set(synth.STANDARD_LENGTHS)
    _check(st, keys, codes, lens, q, ql, k)


def test_threshold_mode(mixed_store):
    st, keys, codes, lens = mixed_store
    q, ql = synth.make_queries(300, len(keys), 3601, 3101)
    _check(st, keys, codes, lens, q, ql, 200, thr=(3, 8))


def test_128_bit_keys(cuda):
    rng = np.random.default_rng(3701)
    n = 60_000
    codes = np.zeros((n, 32), dtype=np.uint8)
    codes[:, :16] = rng.integers(0, 256, size=(n, 16), dtype=np.uint8)
    lens = np.full(n, 16, dtype=np.uint8)
    hi = rng.integers(0, 2**20, size=n, dtype=np.uint64)      # many equal high halves: order decided by the low half
    lo = rng.permutation(n).astype(np.uint64)
    keys = np.zeros((n, 16), dtype=np.uint8)
    keys[:, :8] = hi.astype(">u8").view(np.uint8).reshape(n, 8)
    keys[:, 8:] = lo.astype(">u8").view(np.uint8).reshape(n, 8)
    st = Store(key_bytes=16, max_bytes=16, fixed_len=16)
    try:
        st.add(keys, codes, lens)
        q, ql = codes[:96].copy(), lens[:96].copy()
        gk, gh, gn, gc, _ = st.search(q, ql, 64)
        rows, h, nb, cnt = oracle_topk(hi, codes, lens, q, ql, 64, keys_lo=lo)
        assert_same_topk(gk, gh, gn, gc, hi, rows, h, nb, cnt, keys_lo=lo)
    finally:
        st.close()


def test_mass_duplicates_overflow(cuda):
    # 200K rows share one code, 100K more are one bit away: every query of the batch overflows its candidate list and is
    # answered by the exact re-scan
    n, k = 300_000, 10
    keys = synth.make_keys(0, n, 3801)
    codes = np.zeros((n, 32), dtype=np.uint8)
    codes[:, :8] = np.arange(8, dtype=np.uint8) + 1
    codes[2 * n // 3:, 0] ^= 0x80
    lens = np.full(n, 8, dtype=np.uint8)
    st = Store(key_bytes=8, max_bytes=32)
    try:
        st.add(keys, codes, lens)
        q = np.repeat(codes[:1], 64, axis=0)
        q[32:] = codes[n - 1]
        ql = np.full(64, 8, dtype=np.uint8)
        gk, gh, gn, gc, _ = st.search(q, ql, k)
        assert st.stats()["fallback_queries"] == 64
        rows, h, nb, cnt = oracle_topk(keys, codes, lens, q, ql, k)
        assert_same_topk(gk, gh, gn, gc, keys, rows, h, nb, cnt)
    finally:
        st.close()


def test_batch_spanning_several_tiles(cuda):
    n = 40_000
    keys, codes, lens = make_store_arrays(n, 3901)
    st = Store(key_bytes=8, max_bytes=32)
    try:
        st.add(keys, codes, lens)
        q, ql = synth.make_queries(9000, n, 3902, 3901, lengths=(16,))
        _check(st, keys, codes, lens, q, ql, 20)
    finally:
        st.close()


_AB_SCRIPT = r"""
import json, sys
import numpy as np
sys.path.insert(0, sys.argv[1])
from iscc_search_b200._lib import Store
from tests.helpers import make_store_arrays
from iscc_search_b200 import synth
keys, codes, lens = make_store_arrays(150_000, 4001)
st = Store(key_bytes=8, max_bytes=32)
st.add(keys, codes, lens)
q, ql = synth.make_queries(700, len(keys), 4002, 4001)
gk, gh, gn, gc, _ = st.search(q, ql, 300)
np.savez(sys.argv[2], keys=gk, h=gh, nb=gn, cnt=gc)
print(json.dumps({"issued_popc": st.stats()["issued_popc"]}))
st.close()
"""


def test_same_results_as_popc_scan(cuda, tmp_path):
    out = {}
    for flag in ("1", "0"):
        env = dict(os.environ, ISX_TC_SCAN=flag)
        r = subprocess.run([sys.executable, "-c", _AB_SCRIPT, str(ROOT), str(tmp_path / f"tc{flag}.npz")], capture_output=True,
                           text=True, timeout=600, cwd=str(ROOT), env=env)
        assert r.returncode == 0, r.stderr[-2000:]
        out[flag] = (json.loads(r.stdout.strip().splitlines()[-1]), np.load(tmp_path / f"tc{flag}.npz"))
    assert out["1"][0]["issued_popc"] == 0 and out["0"][0]["issued_popc"] > 0   # each arm took the path it names
    for name in ("keys", "h", "nb", "cnt"):
        assert np.array_equal(out["1"][1][name], out["0"][1][name]), name
