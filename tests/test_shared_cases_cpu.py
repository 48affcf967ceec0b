"""
CPU checks of what tests/test_gpu_shared_thresholds.py builds on: the probe rows sit at exactly the distances the probe
bound is reasoned from, the two length sets land on either side of the 512-rank cut-off of sharing (the library's own
rank table), the skewed shards have the promised shape, and the host merge of per-shard oracle lists equals the oracle over
the union. No GPU needed.
"""

import numpy as np
import pytest

from iscc_search_b200 import synth
from iscc_search_b200.sharded import owner_of
from oracle import c_oracle, nphd_oracle
from tests import test_gpu_shared_thresholds as sh
from tests.helpers import assert_same_topk, make_store_arrays, oracle_topk


@pytest.mark.parametrize("world", [2, 3, 8])
def test_probe_rows_at_exact_distances(world):
    n_rows = 4096
    extra = [8, 13, 31] if world == 3 else []
    case, P = sh.probe_case(world, n_rows, d=8, seed=world, extra_lengths=extra)
    assert len(np.unique(case.hi)) == len(case.hi)
    for r, (keys, lo, codes, lens) in enumerate(case.shards):
        h, nb = nphd_oracle.prefix_hamming(codes, lens, P, 32)
        if r == 0:
            assert len(lens) == sh.K and not h.any() and (nb == 256).all()
            continue
        at_d = np.zeros(len(lens), dtype=bool)
        at_d[sh.PROBE_EVERY - 1:n_rows:sh.PROBE_EVERY] = True
        assert (h[at_d] == 8).all() and (nb[at_d] == 256).all() and at_d.sum() == n_rows // sh.PROBE_EVERY
        assert (h[~at_d].astype(int) * 256 > 8 * nb[~at_d].astype(int) * 4).all()   # every other row beyond 4 D
        if r == 1 and extra:
            assert lens[n_rows:].tolist() == extra and (h[n_rows:] == nb[n_rows:]).all()   # h/nbits = 1
        else:
            assert len(lens) == n_rows
        assert len(np.unique(codes, axis=0)) == len(lens)


def test_probe_sizing():
    for world in (2, 3, 8):
        span, n1 = sh.warm_span(world), sh.probe_n1(world)
        assert span == {2: 32, 3: 21, 8: 8}[world]
        # the warm-up ranges run only when the shard has more than 4 first ranges of blocks
        assert sh.probe_rows(world) // sh.BLOCK_ROWS > 4 * span
        # the first warm-up range holds N1 / 8 probe rows
        assert span * sh.BLOCK_ROWS // sh.PROBE_EVERY * 8 == n1
        # the 64-block bootstrap sample holds >= k probe rows, so it starts the threshold at D
        assert 64 * sh.BLOCK_ROWS // sh.PROBE_EVERY >= sh.K
    # an item of one block stages at most 1024 records for a CTA's <= 256 queries (the stage holds 1024)
    assert 256 * sh.BLOCK_ROWS // sh.PROBE_EVERY <= 1024


def test_cut_lengths_sit_on_either_side_of_the_share_cap():
    lo, hi = sh.cut_lengths()
    r_lo, r_hi = sh.rank_count(lo), sh.rank_count(hi)
    assert r_lo <= sh.SHARE_RCAP < r_hi
    assert sh.rank_count([32]) == 257 and 32 in lo
    assert len(set(hi) - set(lo)) == 1 and max(len(lo), len(hi)) < sh.K   # the extra rows fit on a rank with < k rows
    # greedy maximum: no single further length keeps R within the cap
    assert all(sh.rank_count(lo + [L]) > sh.SHARE_RCAP for L in range(1, 33) if L not in lo)
    assert r_lo > 480


@pytest.mark.parametrize("few", [37, 0])
def test_skew_case_shape(few):
    case = sh.skew_case(20_000, 43, 3, few)
    keys, codes, lens = make_store_arrays(20_000, 43)
    assert sorted(case.hi.tolist()) == sorted(keys.tolist())
    r0, r1, r2 = case.shards
    assert len(r1[3]) == few and set(r1[3].tolist()) <= {8}
    assert 24 in set(r2[3].tolist()) and 24 not in set(r0[3].tolist()) | set(r1[3].tolist())
    assert len(r0[3]) > 5000 and len(r2[3]) > 5000


def test_prefix_pairs_against_brute_force():
    keys, codes, lens = sh.prefix_planted(600, 5, 40)
    exp = set()
    for a in range(len(lens)):
        for b in range(a + 1, len(lens)):
            m = min(lens[a], lens[b])
            if np.array_equal(codes[a, :m], codes[b, :m]):
                exp.add((*sorted((int(keys[a]), int(keys[b]))), 8 * int(m)))
    assert len(exp) >= 40 and sh.prefix_pairs(keys, codes, lens) == sorted(exp)


def _shard_lists(case, queries, qlens, k, thr, key16):
    parts = []
    for keys, lo, codes, lens in case.shards:
        rows, h, nb, cnt = oracle_topk(keys, codes, lens, queries, qlens, k, thr, keys_lo=lo)
        safe = np.where(rows >= 0, rows, 0)
        kk = keys[safe] if not key16 else synth.keys128_bytes(keys[safe].ravel(), lo[safe].ravel()).reshape(*rows.shape, 16)
        parts.append((kk, h, nb, cnt))
    return parts


@pytest.mark.parametrize("thr", [None, (1, 8)])
@pytest.mark.parametrize("world", [2, 3, 5])
def test_merge_of_shard_oracles_equals_union_oracle(world, thr):
    keys, codes, lens = make_store_arrays(6000, 61)
    # cross-length ties at equal h/nbits: 8-byte prefixes of 16-byte rows
    codes[:50, :8], lens[:50] = codes[50:100, :8], 8
    codes[:50, 8:] = 0
    case = sh.split(keys, codes, lens, owner_of(keys, world), world)
    queries, qlens = synth.make_queries(40, 6000, 62, 61)
    queries[:5] = codes[50:55]
    qlens[:5] = lens[50:55]
    k = 30
    gk, gh, gn, gc = sh.merge_topk(_shard_lists(case, queries, qlens, k, thr, False), k)
    rows, h, nb, cnt = oracle_topk(case.hi, case.codes, case.lens, queries, qlens, k, thr)
    assert_same_topk(gk, gh, gn, gc, case.hi, rows, h, nb, cnt)


def test_merge_sixteen_byte_keys_shared_high_half():
    hi, lo, codes, lens = c_oracle.synth_rows(0, 8000, 48, lengths=(8,), key_mode=1, cpa=64, dup_every=16, dup_back=5)
    case = sh.split(hi, codes, lens, owner_of(hi ^ lo, 4), 4, lo=lo)
    queries, qlens = synth.make_queries(24, 8000, 14, 48, lengths=(8,), row_lengths=(8,), mixed_rows=False)
    for k, thr in ((200, (16, 64)), (50, (0, 1)), (7, None)):
        gk, gh, gn, gc = sh.merge_topk(_shard_lists(case, queries, qlens, k, thr, True), k)
        rows, h, nb, cnt = oracle_topk(case.hi, case.codes, case.lens, queries, qlens, k, thr, keys_lo=case.lo)
        assert cnt.max() > 1
        assert_same_topk(gk, gh, gn, gc, case.hi, rows, h, nb, cnt, keys_lo=case.lo)
