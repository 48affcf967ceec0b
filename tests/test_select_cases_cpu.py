"""
CPU checks of what tests/test_gpu_select_edges.py builds on: the planted-tie case builder against the numpy oracle, the
restated host arithmetic (sort capacities, regimes, first-of-asset limit) against hand-computed values, and the merge
reference. No GPU needed.
"""

from fractions import Fraction

import numpy as np
import pytest

from oracle import nphd_oracle
from tests import test_gpu_select_edges as sel

B200_OPTIN = 232448   # 227 KB opt-in shared memory per block
SM86_OPTIN = 101376   # 99 KB


def _distances(case, q):
    return nphd_oracle.prefix_hamming(case.codes, case.lens, case.queries[q], 32)


@pytest.mark.parametrize("key_bytes", (8, 16))
def test_planted_ties_distances_counts_and_keys(key_bytes):
    counts = [(5, 300), (40, 3), (7, 90), (0, 513), (12, 12)]
    case = sel.planted_ties(counts, key_bytes, seed=3, cross=(2,), n_fill=2000)
    assert len(case.lens) == sum(a + b for a, b in counts) + 2000
    for q, (n_lt, n_eq) in enumerate(counts):
        h, nb = _distances(case, q)
        lt, eq = case.groups[q]
        assert len(lt) == n_lt and len(eq) == n_eq
        assert (h[lt].astype(int) * 8 < nb[lt]).all()                  # strictly below 1/8
        assert (h[eq].astype(int) * 8 == nb[eq]).all()                 # exactly 1/8, whatever the row's length
        within = np.flatnonzero(h.astype(int) * 8 <= nb)
        assert sorted(within.tolist()) == sorted(lt.tolist() + eq.tolist()), f"query {q}: a foreign row within 1/8"
        lens = set(case.lens[eq].tolist())
        assert lens == ({8, 16, 32} if q == 2 else {32})
        assert len(np.unique(case.codes[eq], axis=0)) > 1
    # exact counts: a k in n_lt + 1 .. n_lt + n_eq cuts the group at d, so total_le is the whole group
    assert [sel.exact_counts(case, 10)[q] for q in (0, 2, 3)] == [(305, 10), (97, 10), (513, 10)]
    assert [sel.exact_counts(case, 10, sel.THR)[q] for q in (0, 2, 3)] == [(305, 10), (97, 10), (513, 10)]
    assert sel.exact_counts(case, 24)[4] == (24, 24) and sel.exact_counts(case, 41)[1] == (43, 41)
    assert sel.exact_counts(case, 400, sel.THR)[1] == (43, 43)        # fewer than k within the threshold
    assert sel.exact_counts(case, 10)[1][0] < 40                       # k below n_lt: d* is under the tie distance
    # the rows agree with the oracle's top-k: the group's rows lead in (h/n, key) order
    res = nphd_oracle.topk(case.hi, case.lo, case.codes, case.lens, case.queries[:1], case.qlens[:1], 305)[0]
    assert sorted(res[0].tolist()) == sorted(case.groups[0][0].tolist() + case.groups[0][1].tolist())
    # key layouts
    hi, lo = case.hi, case.lo if case.lo is not None else np.zeros_like(case.hi)
    g = [np.concatenate(case.groups[q]) for q in range(len(counts))]
    assert len(np.unique(np.stack([hi, lo], axis=1), axis=0)) == len(hi)
    if key_bytes == 8:
        assert hi[g[0]].min() == 0 and hi[g[1]].max() == sel.U64_MAX
        for q in (1, 4):   # small groups share the top 7 bytes: the pivot is decided in byte 7
            assert len(np.unique(hi[g[q]] >> np.uint64(8))) <= 2
    else:
        for q in (0, 1, 3, 4):
            assert len(np.unique(hi[g[q]])) == 1                        # ties share the high half
        assert hi[g[1]][0] == sel.U64_MAX and lo[g[1]].max() == sel.U64_MAX and lo[g[0]].min() == 0
        his = np.unique(hi[g[2]])
        assert len(his) == 4 and len(np.unique(his >> np.uint64(8))) == 1   # high halves differ in the last byte only


def test_host_arithmetic_hand_values():
    assert sel.max_sort_cap(B200_OPTIN, 8) == 8192 and sel.max_sort_cap(B200_OPTIN, 16) == 8192
    assert sel.max_sort_cap(SM86_OPTIN, 8) == 4096 and sel.max_sort_cap(SM86_OPTIN, 16) == 2048
    cm = 8192
    assert [sel.sort_cap(k, cm) for k in (1, 256, 257, 1024, 1025, 2048, 2049, 8192, 65536)] == \
        [1024, 1024, 2048, 4096, 8192, 8192, cm, cm, cm]
    assert sel.sort_cap(2049, 2048) == 2048 and sel.sort_cap(100, 2048) == 1024
    assert sel.small_path_takes(4, 2048) and not sel.small_path_takes(5, 10) and not sel.small_path_takes(1, 2049)
    assert sel.first_of_asset_max_count(B200_OPTIN) == 8192 and sel.first_of_asset_max_count(SM86_OPTIN) == 4096
    assert sel.candidate_capacity(10) == 32768 and sel.candidate_capacity(9000) == 380928
    # regimes: (k, total_le, cap)
    assert sel.select_regime(256, 256, 1024) == "S1" and sel.select_regime(256, 1024, 1024) == "S1"
    assert sel.select_regime(256, 1025, 1024) == "S2" and sel.select_regime(8192, 8193, 8192) == "S2"
    assert sel.select_regime(8193, 8193, 8192) == "B1" and sel.select_regime(8193, 8194, 8192) == "B2"
    assert sel.select_regime(65536, 8193, 8192) == "B1" and sel.select_regime(65536, 8192, 8192) == "S1"
    assert sel.select_regime(10, 400_000, 1024) == "S2"


def test_select_cases_land_in_their_regimes_and_cover_every_one():
    seen = set()
    for cm in (8192, 4096):
        for k in sel.SMALL_KS + (cm, cm + 1, 10007, 65536):
            cap = sel.sort_cap(k, cm)
            for name, n_lt, n_eq, mode, regime in sel.select_cases(k, cap, cm):
                total = n_lt + n_eq
                assert n_lt < k or mode == "thr", name
                assert total >= k if mode == "topk" else total <= k, name   # top-k cases cut the tie group at d*
                assert sel.select_regime(k, total, cap) == regime, (k, name)
                seen.add(regime + ("_big_scratch" if k > cm and regime[0] == "S" else ""))
                seen.update(["one_winner"] if n_lt == k - 1 and n_eq >= 2 else [])
                seen.update(["all_win"] if total == k else [])
                seen.update(["on_cap"] if total == cap else ["past_cap"] if total == cap + 1 else [])
    assert seen >= {"S1", "S2", "B1", "B2", "S1_big_scratch", "one_winner", "all_win", "on_cap", "past_cap"}, seen


@pytest.mark.parametrize("key_bytes", (8, 16))
def test_merge_reference(key_bytes):
    G, Q, k = 3, 4, 7
    counts = np.array([[0, 3, 7, 12], [7, 0, 2, 9], [1, 7, 7, 0]], dtype=np.uint32)
    h, n, hi, lo, cnt, expected = sel.merge_case(G, Q, k, counts, key_bytes, seed=5)
    for q in range(Q):
        recs = []
        for g in range(G):
            m = min(int(cnt[g, q]), k)
            r = [(int(h[g, q, j]), int(n[g, q, j]), int(hi[g, q, j]), int(lo[g, q, j])) for j in range(m)]
            assert r == sorted(r, key=lambda t: (Fraction(t[0], t[1]), t[2], t[3]))   # each shard list is sorted
            recs += r
        assert len({(t[2], t[3]) for t in recs}) == len(recs)               # keys unique over all shards
        assert expected[q] == sorted(recs, key=lambda t: (Fraction(t[0], t[1]), t[2], t[3]))[:k]
        assert all(t[1] in (64, 128, 192, 256) and t[0] * 8 in (0, t[1], 4 * t[1]) for t in recs)
    assert any(len({t[1] for t in e if Fraction(t[0], t[1]) == Fraction(1, 8)}) > 1 for e in expected)
