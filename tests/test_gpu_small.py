"""
Small-batch path (csrc/small.cuh: one cooperative launch per search, TMA ring, fused bootstrap and select): by default
every request of <= 4 queries takes it (ISX_SMALL_MAXQ, at most 8). Parity against the oracle for each shape the launch
plan distinguishes, and equality with the general path (ISX_SMALL_PATH=0 is read once per process, so the general path
is exercised here by batches of 5+ queries carrying the same queries). Every compared length, rows on the bound and the
ISX_SMALL_* switches: tests/test_gpu_scan_edges.py.
"""

import numpy as np
import pytest

from iscc_search_b200 import _lib, synth
from tests.helpers import assert_same_topk, make_store_arrays, oracle_topk

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def mixed_store(cuda):
    n = 400_000
    keys, codes, lens = make_store_arrays(n, 41)
    st = _lib.Store(key_bytes=8, max_bytes=32)
    st.add(keys, codes, lens)
    yield st, keys, codes, lens
    st.close()


@pytest.mark.parametrize("q,k", [(1, 100), (2, 10), (4, 100), (5, 100), (8, 1000), (3, 2048)])
def test_small_batches_mixed_lengths_equal_oracle(mixed_store, q, k):
    st, keys, codes, lens = mixed_store
    queries, qlens = synth.make_queries(q, len(keys), 100 + q, 41)
    gk, gh, gn, gc, _ = st.search(queries, qlens, k)
    if q <= 4:
        assert st.stats()["kernel_launches"] == 1, "the small-batch path was expected to answer this request in one launch"
    rows, h, nb, cnt = oracle_topk(keys, codes, lens, queries, qlens, k)
    assert_same_topk(gk, gh, gn, gc, keys, rows, h, nb, cnt)


def test_each_single_query_length_and_general_path_agreement(mixed_store):
    st, keys, codes, lens = mixed_store
    queries, qlens = synth.make_queries(24, len(keys), 7, 41)
    big = st.search(queries, qlens, 50)                       # 24 queries: general path
    assert st.stats()["kernel_launches"] > 1
    for i in range(24):                                       # one by one: small path
        gk, gh, gn, gc, _ = st.search(queries[i:i + 1], qlens[i:i + 1], 50)
        assert st.stats()["kernel_launches"] == 1
        assert np.array_equal(gk[0], big[0][i]) and np.array_equal(gh[0], big[1][i]) and np.array_equal(gn[0], big[2][i])
        assert gc[0] == big[3][i]


def test_small_path_threshold_mode_codes_out_and_128bit_keys(cuda):
    n, seed = 250_000, 4
    st = _lib.Store(key_bytes=16, max_bytes=8, fixed_len=8)
    l8 = np.full(n, 8, dtype=np.uint8)
    codes = synth.make_codes(0, n, seed, l8, dup_every=16, dup_back=65)
    hi, lo = synth.make_keys128(0, n, seed, 64)
    st.add(synth.keys128_bytes(hi, lo), codes, l8)
    qs = np.ascontiguousarray(codes[[14, 206, 4110, 77_774]])
    qs[3, 0] ^= 0x81
    ql = np.full(4, 8, dtype=np.uint8)
    for kk, thr in ((400, (16, 64)), (1000, (0, 64)), (7, None)):
        gk, gh, gn, gc, gcodes = st.search(qs, ql, kk, thr, with_codes=True)
        assert st.stats()["kernel_launches"] == 1
        rows, h, nb, cnt = oracle_topk(hi, codes, l8, qs, ql, kk, thr, keys_lo=lo)
        assert_same_topk(gk, gh, gn, gc, hi, rows, h, nb, cnt, keys_lo=lo)
        for i in range(4):
            c = int(cnt[i])
            assert np.array_equal(gcodes[i, :c], codes[rows[i, :c]])
    st.close()


def test_small_path_tiny_stores_and_k_beyond_rows(cuda):
    for n in (1, 37, 1023, 1025, 5000):
        keys, codes, lens = make_store_arrays(n, 5 + n)
        st = _lib.Store(key_bytes=8, max_bytes=32)
        st.add(keys, codes, lens)
        queries, qlens = synth.make_queries(3, n, 6, 5 + n)
        for k in (1, 50, 3000):
            gk, gh, gn, gc, _ = st.search(queries, qlens, k)
            rows, h, nb, cnt = oracle_topk(keys, codes, lens, queries, qlens, k, use_c=False)
            assert_same_topk(gk, gh, gn, gc, keys, rows, h, nb, cnt)
        st.close()


def test_small_path_mass_duplicates_fall_back_to_the_general_path(cuda):
    # 150K rows share one code: far more ties than the fused select sorts -> the general path answers, still exact
    n, dup_n, k = 100_000, 150_000, 100
    keys, codes, lens = make_store_arrays(n, 61)
    dup_keys = synth.make_keys(10**9, dup_n, 77)
    dup_codes = np.zeros((dup_n, 32), dtype=np.uint8)
    dup_codes[:, :16] = 0xA7
    dup_lens = np.full(dup_n, 16, dtype=np.uint8)
    st = _lib.Store(key_bytes=8, max_bytes=32)
    st.add(np.concatenate([keys, dup_keys]), np.concatenate([codes, dup_codes]), np.concatenate([lens, dup_lens]))
    q = np.ascontiguousarray(dup_codes[:1])
    ql = dup_lens[:1].copy()
    for _ in range(2):   # twice: the small path's per-query state must be clean again after the fall-back
        gk, gh, gn, gc, _ = st.search(q, ql, k)
        assert gc[0] == k and (gh[0] == 0).all()
        assert np.array_equal(gk[0], np.sort(dup_keys)[:k])
    # and an ordinary query right behind it
    queries, qlens = synth.make_queries(2, n, 62, 61)
    gk, gh, gn, gc, _ = st.search(queries, qlens, k)
    rows, h, nb, cnt = oracle_topk(np.concatenate([keys, dup_keys]), np.concatenate([codes, dup_codes]), np.concatenate([lens, dup_lens]),
                                   queries, qlens, k)
    assert_same_topk(gk, gh, gn, gc, np.concatenate([keys, dup_keys]), rows, h, nb, cnt)
    st.close()


def test_small_path_device_queries_and_device_results(mixed_store):
    import torch

    from iscc_search_b200.sharded import ShardedSearcher

    st, keys, codes, lens = mixed_store
    dev = torch.device("cuda", 0)
    queries, qlens = synth.make_queries(4, len(keys), 9, 41)
    searcher = ShardedSearcher(st, 0, 1, None, dev)
    gk, gh, gn, gc = (a.copy() for a in searcher.search(queries, qlens, 64))
    assert st.stats()["kernel_launches"] == 1
    rows, h, nb, cnt = oracle_topk(keys, codes, lens, queries, qlens, 64)
    assert_same_topk(gk, gh, gn, gc, keys, rows, h, nb, cnt)
    st.set_stream(None)


def test_small_path_repeated_searches_keep_state_clean(mixed_store):
    st, keys, codes, lens = mixed_store
    queries, qlens = synth.make_queries(8, len(keys), 11, 41)
    rows, h, nb, cnt = oracle_topk(keys, codes, lens, queries, qlens, 20)
    for rep in range(5):
        sel = np.roll(np.arange(8), rep)[: 1 + rep]
        gk, gh, gn, gc, _ = st.search(np.ascontiguousarray(queries[sel]), np.ascontiguousarray(qlens[sel]), 20)
        assert_same_topk(gk, gh, gn, gc, keys, rows[sel], h[sel], nb[sel], cnt[sel])


def test_small_path_heavy_ties_are_cut_by_key(cuda):
    # 64-bit codes only: distances are coarse, the tie group at the k-th distance holds hundreds of rows, so the fused
    # select has to find the pivot key among the ties (radix pass in shared memory) - 64- and 128-bit keys
    n = 1_500_000
    l8 = np.full(n, 8, dtype=np.uint8)
    codes = synth.make_codes(0, n, 17, l8)
    keys = synth.make_keys(0, n, 17)
    hi, lo = synth.make_keys128(0, n, 17, 64)
    queries, qlens = synth.make_queries(4, n, 18, 17, lengths=(8,), row_lengths=(8,), mixed_rows=False)
    st = _lib.Store(key_bytes=8, max_bytes=8, fixed_len=8)
    st.add(keys, codes, l8)
    st2 = _lib.Store(key_bytes=16, max_bytes=8, fixed_len=8)
    st2.add(synth.keys128_bytes(hi, lo), codes, l8)
    for k in (100, 700, 2048):
        gk, gh, gn, gc, _ = st.search(queries, qlens, k)
        assert st.stats()["kernel_launches"] == 1
        rows, h, nb, cnt = oracle_topk(keys, codes, l8, queries, qlens, k)
        assert_same_topk(gk, gh, gn, gc, keys, rows, h, nb, cnt)
        gk, gh, gn, gc, _ = st2.search(queries, qlens, k)
        rows, h, nb, cnt = oracle_topk(hi, codes, l8, queries, qlens, k, keys_lo=lo)
        assert_same_topk(gk, gh, gn, gc, hi, rows, h, nb, cnt, keys_lo=lo)
    st.close()
    st2.close()
