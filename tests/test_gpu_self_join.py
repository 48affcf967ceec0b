"""
GPU tests of the store self-join (isx_self_join / isx_join_fetch, csrc/join.cuh): every pair of stored rows within an
exact rational threshold, once, with key_a < key_b, in (key_a, key_b) order. Each test compares the complete pair list
(keys, h, nbits, order, count) with the CPU oracle self-join (oracle/self_join.py).
"""

import json
import os
import subprocess
import sys
from fractions import Fraction
from pathlib import Path

import numpy as np
import pytest

from iscc_search_b200 import ShardedIndex128, ShardedNphdIndex, synth
from iscc_search_b200._lib import Store
from oracle import c_oracle
from oracle.self_join import self_join as oracle_self_join
from tests.helpers import make_store_arrays

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent


def plant_near_duplicates(keys, codes, lens, n_new, seed, flips=(0, 1, 2, 4), key_start=None):
    """Append n_new rows: copies of random rows with r bit flips inside their length, and 8-byte prefixes of long rows."""
    rng = np.random.default_rng(seed)
    n = len(lens)
    src = rng.integers(0, n, size=n_new)
    new_codes = codes[src].copy()
    new_lens = lens[src].copy()
    half = n_new // 2
    for i in range(half):   # near copies
        r = flips[i % len(flips)]
        for bit in rng.choice(8 * int(new_lens[i]), size=r, replace=False):
            new_codes[i, bit // 8] ^= np.uint8(1 << (bit % 8))
    for i in range(half, n_new):   # prefixes: a shorter row equal to the start of a longer one
        L = int(new_lens[i])
        if L > 8:
            p = 8 if L <= 16 else int(rng.choice([8, 16]))
            new_codes[i, p:] = 0
            new_lens[i] = p
    new_keys = synth.make_keys(n if key_start is None else key_start, n_new, seed)
    return (np.concatenate([keys, new_keys]), np.concatenate([codes, new_codes]), np.concatenate([lens, new_lens]))


def expected(keys, codes, lens, thr, keys_lo=None):
    ra, rb, h, nb = oracle_self_join(keys, keys_lo, codes, lens, thr)
    if keys_lo is None:
        return keys[ra], keys[rb], h, nb
    return synth.keys128_bytes(keys[ra], keys_lo[ra]), synth.keys128_bytes(keys[rb], keys_lo[rb]), h, nb


def assert_same_pairs(got, exp):
    ga, gb, gh, gn = got
    ea, eb, eh, en = exp
    assert len(gh) == len(eh), f"pair count {len(gh)} != {len(eh)}"
    assert np.array_equal(ga, ea), "key_a / order differ"
    assert np.array_equal(gb, eb), "key_b / order differ"
    assert np.array_equal(gh, eh), "hamming differs"
    assert np.array_equal(gn, en), "nbits differs"


@pytest.fixture(scope="module")
def mixed_store(cuda):
    keys, codes, lens = make_store_arrays(36_000, 5101)
    keys, codes, lens = plant_near_duplicates(keys, codes, lens, 4_000, 5102)
    st = Store(key_bytes=8, max_bytes=32)
    st.add(keys, codes, lens)
    yield st, keys, codes, lens
    st.close()


@pytest.mark.parametrize("thr", [(0, 1), (1, 64), (1, 8), (1, 4)])
def test_mixed_lengths_planted_duplicates(mixed_store, thr):
    st, keys, codes, lens = mixed_store
    got = st.self_join(thr)
    assert_same_pairs(got, expected(keys, codes, lens, thr))
    s = st.stats()
    assert s["scan_launches"] > 0 and s["pairs"] > 0 and s["passes"] > 0


def test_byte_granular_lengths_and_small_bucket(cuda):
    # lengths 5, 13, 30 plus a 7-byte bucket of 40 rows: that bucket's chunk has fewer than 64 queries (POPC scan k_scan)
    keys, codes, lens = make_store_arrays(20_000, 5201, lengths=(5, 13, 30))
    small = 40
    sk = synth.make_keys(50_000, small, 5202)
    sl = np.full(small, 7, dtype=np.uint8)
    sc = codes[:small].copy()
    sc[:, 7:] = 0
    sc[: small // 2, 5] ^= 1   # 7-byte rows that start like a stored row; half of them differ in their 6th byte
    keys, codes, lens = np.concatenate([keys, sk]), np.concatenate([codes, sc]), np.concatenate([lens, sl])
    keys, codes, lens = plant_near_duplicates(keys, codes, lens, 2_000, 5203, key_start=60_000)
    st = Store(key_bytes=8, max_bytes=32)
    try:
        st.add(keys, codes, lens)
        for thr in [(0, 1), (1, 10), (1, 5)]:
            assert_same_pairs(st.self_join(thr), expected(keys, codes, lens, thr))
    finally:
        st.close()


@pytest.mark.parametrize("bits", [0, 8])
def test_128_bit_keys_index(cuda, bits):
    n = 30_000
    khi, klo, codes, lens = c_oracle.synth_rows(0, n, 5301, lengths=(8,), key_mode=1, cpa=64, dup_every=7, dup_back=3)
    idx = ShardedIndex128(ndim=64)
    try:
        idx.add(synth.keys128_bytes(khi, klo), codes[:, :8])
        res = idx.self_join(bits)
        got = (res.keys_a, res.keys_b, res.hamming, res.nbits)
        exp = expected(khi, codes, lens, (bits, 64), keys_lo=klo)
        assert_same_pairs(got, exp)
        assert len(res) >= n // 7 - 1   # the planted duplicates
        assert np.array_equal(res.distances, res.hamming.astype(np.float32))
    finally:
        idx.close()


def test_mass_duplicates_force_overflow_rescan(cuda):
    n_rand, n_dup = 20_000, 3_000
    keys, codes, lens = make_store_arrays(n_rand + n_dup, 5401, lengths=(8,))
    codes[n_rand:] = codes[0]
    st = Store(key_bytes=8, max_bytes=32)
    try:
        st.add(keys, codes, lens)
        got = st.self_join((0, 1))
        group = n_dup + 1   # row 0 carries the code too
        assert len(got[2]) == group * (group - 1) // 2
        assert st.stats()["fallback_queries"] > 0
        assert_same_pairs(got, expected(keys, codes, lens, (0, 1)))
    finally:
        st.close()


def test_empty_single_and_everything(cuda):
    st = Store(key_bytes=8, max_bytes=32)
    try:
        ka, kb, h, nb = st.self_join((1, 4))
        assert len(ka) == len(kb) == len(h) == len(nb) == 0
        keys, codes, lens = make_store_arrays(300, 5501)
        st.add(keys[:1], codes[:1], lens[:1])
        assert len(st.self_join((1, 1))[2]) == 0
        st.add(keys, codes, lens)
        got = st.self_join((1, 1))
        assert len(got[2]) == 300 * 299 // 2
        assert_same_pairs(got, expected(keys, codes, lens, (1, 1)))
    finally:
        st.close()


def test_after_remove_and_add(cuda):
    keys, codes, lens = make_store_arrays(12_000, 5601)
    keys, codes, lens = plant_near_duplicates(keys, codes, lens, 3_000, 5602)
    st = Store(key_bytes=8, max_bytes=32)
    try:
        st.add(keys, codes, lens)
        thr = (1, 8)
        assert_same_pairs(st.self_join(thr), expected(keys, codes, lens, thr))
        rm = np.random.default_rng(5603).choice(len(keys), size=2_500, replace=False)   # swap-remove moves rows
        st.remove(keys[rm], len(rm))
        live = np.ones(len(keys), dtype=bool)
        live[rm] = False
        keys, codes, lens = keys[live], codes[live], lens[live]
        assert_same_pairs(st.self_join(thr), expected(keys, codes, lens, thr))
        k2, c2, l2 = plant_near_duplicates(keys, codes, lens, 1_500, 5604, key_start=100_000)
        st.add(k2[len(keys):], c2[len(keys):], l2[len(keys):])
        assert_same_pairs(st.self_join(thr), expected(k2, c2, l2, thr))
    finally:
        st.close()


def test_lifecycle_and_paging(cuda):
    keys, codes, lens = make_store_arrays(8_000, 5701)
    keys, codes, lens = plant_near_duplicates(keys, codes, lens, 2_000, 5702)
    st = Store(key_bytes=8, max_bytes=32)
    try:
        st.add(keys, codes, lens)
        thr = (1, 4)
        full = st.self_join(thr)
        n = len(full[2])
        assert n > 1000
        pages = [st.join_fetch(i0, min(333, n - i0)) for i0 in range(0, n, 333)]
        for j in range(4):
            assert np.array_equal(np.concatenate([p[j] for p in pages]), full[j])
        with pytest.raises(ValueError, match="outside"):
            st.join_fetch(n - 1, 2)
        st.search(codes[:4], lens[:4], 5)
        with pytest.raises(ValueError, match="no self-join result"):
            st.join_fetch(0, 1)
        st.self_join(thr)
        st.add(synth.make_keys(900_000, 1, 1), codes[:1], lens[:1])
        with pytest.raises(ValueError, match="no self-join result"):
            st.join_fetch(0, 1)
        st.self_join(thr)
        st.release_scratch()
        with pytest.raises(ValueError, match="no self-join result"):
            st.join_fetch(0, 1)
    finally:
        st.close()
    idx = ShardedNphdIndex(max_dim=256)
    try:
        idx.add(keys, [bytes(codes[i, : lens[i]]) for i in range(len(keys))])
        with pytest.raises(ValueError, match="float"):
            idx.self_join(0.25)
        res = idx.self_join(Fraction(1, 4))
        assert_same_pairs((res.keys_a, res.keys_b, res.hamming, res.nbits), full)
        assert np.array_equal(res.distances, (res.hamming.astype(np.float32) / res.nbits.astype(np.float32)).astype(np.float32))
        assert len(idx.self_join((1, 4))) == len(res)
    finally:
        idx.close()


_AB_SCRIPT = r"""
import json, sys
import numpy as np
sys.path.insert(0, sys.argv[1])
from iscc_search_b200._lib import Store
from tests.helpers import make_store_arrays
from tests.test_gpu_self_join import plant_near_duplicates
keys, codes, lens = make_store_arrays(30_000, 5801)
keys, codes, lens = plant_near_duplicates(keys, codes, lens, 5_000, 5802)
st = Store(key_bytes=8, max_bytes=32)
st.add(keys, codes, lens)
ka, kb, h, nb = st.self_join((3, 16))
np.savez(sys.argv[2], ka=ka, kb=kb, h=h, nb=nb)
print(json.dumps({"issued_popc": st.stats()["issued_popc"], "pairs": int(len(h))}))
st.close()
"""


def test_same_results_without_tensor_core_scan(cuda, tmp_path):
    out = {}
    for flag in ("1", "0"):
        env = dict(os.environ, ISX_TC_SCAN=flag)
        r = subprocess.run([sys.executable, "-c", _AB_SCRIPT, str(ROOT), str(tmp_path / f"tc{flag}.npz")], capture_output=True,
                           text=True, timeout=600, cwd=str(ROOT), env=env)
        assert r.returncode == 0, r.stderr[-2000:]
        out[flag] = (json.loads(r.stdout.strip().splitlines()[-1]), np.load(tmp_path / f"tc{flag}.npz"))
    assert out["0"][0]["issued_popc"] > 0 and out["1"][0]["issued_popc"] < out["0"][0]["issued_popc"]
    assert out["1"][0]["pairs"] > 0
    for name in ("ka", "kb", "h", "nb"):
        assert np.array_equal(out["1"][1][name], out["0"][1][name]), name
