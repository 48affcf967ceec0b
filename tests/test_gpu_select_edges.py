"""
GPU edge tests of the selection stage, each compared bit-exactly with the C oracle, each asserting the regime it is named
for before it compares:
  A. `k_select` (csrc/kernels.cuh) at every cutoff of its four regimes - shared-memory sort without (S1) and with (S2) the
     radix pivot over the ties at d*, global-scratch sort without (B1) and with (B2) it - for 8- and 16-byte keys, with
     `total_le` (rows with rank <= d*) on k, k + 1, the sort capacity and one past it, in top-k and threshold mode
  B. the small path's fused select (csrc/small.cuh `small_select`): radix cut off at 256 survivors and on at 257, one
     launch at 4096 rows within d*, the fall-back at 4097 and the request after it, k = 2048 with 128-bit ties
  C. the exact re-scan of overflowed queries inside a batch of many tiles, on 1, 2 and 4 tile lanes, with the
     shared-memory and the global-scratch select after it
  D. `k_merge` on synthetic per-shard lists against a plain sort by (Fraction(h, n), key)
  E. the largest count `first_of_asset_out` accepts, and the refusal one above it
Every planted group of part A and B sits at distance <= 32 of 256 bits from its query; random rows and the other queries'
groups sit near 128, so the counts of a case are exact by construction and are re-counted from the oracle's distances.
"""

import json
import os
import subprocess
import sys
from fractions import Fraction
from pathlib import Path

import numpy as np
import pytest

from iscc_search_b200 import _lib, synth
from iscc_search_b200._lib import Store
from iscc_search_b200.sharded import record_layout
from oracle import nphd_oracle
from tests.helpers import oracle_topk

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent
U64_MAX = 2**64 - 1

# ---- host arithmetic of csrc/isx.cu, restated ------------------------------------------------------------------------
SMALL_MAX_Q = 4          # the small path takes requests of <= 4 queries (ISX_SMALL_MAXQ)
SMALL_SORT_CAP = 4096    # survivors its fused select sorts (kSmallSortCap); more go to the general path
SMALL_MAX_K = SMALL_SORT_CAP // 2
SMALL_RADIX_MIN = 256    # it cuts the ties by radix only above this many survivors


def select_smem(cap, key_bytes):
    return cap * (8 * (2 if key_bytes == 16 else 1) + 12) + 64


def max_sort_cap(smem_optin, key_bytes):
    """Entries the shared-memory sort of `k_select` holds at most."""
    cap = 1024
    while select_smem(cap * 2, key_bytes) + 2048 <= smem_optin:
        cap *= 2
    return cap


def sort_cap(k, cap_max):
    """The sort capacity of a search with count k: the first power of two >= 4k, in [1024, cap_max]."""
    c = 1024
    while c < 4 * k and c < cap_max:
        c *= 2
    return min(cap_max, max(1024, c))


def small_path_takes(n_queries, k):
    return n_queries <= SMALL_MAX_Q and k <= SMALL_MAX_K


def select_regime(k, total_le, cap):
    """'S1' | 'S2' | 'B1' | 'B2': shared or global-scratch sort, without or with the radix pivot over the ties at d*."""
    n_out = min(k, total_le)
    big = n_out > cap
    pivot = total_le > n_out and (total_le > cap or big)
    return ("B" if big else "S") + ("2" if pivot else "1")


def candidate_capacity(k):
    """Candidate list entries per query of the batch path (C): more rows within the running threshold overflow it."""
    r0 = max(1, (2 * k + 1023) // 1024)
    c = max(r0 * 1024 + 40 * k + 2048, 32768)
    return min((c + 1023) // 1024 * 1024, 1 << 26)


def first_of_asset_max_count(smem_optin):
    """Largest count `first_of_asset_out` accepts: its table of H >= 2 * count slots (a power of two) takes 12 H + 16 bytes."""
    h = 2
    while h * 2 * 12 + 16 + 2048 <= smem_optin:
        h *= 2
    return h // 2


def device_smem_optin():
    import torch

    return torch.cuda.get_device_properties(0).shared_memory_per_block_optin


# ---- case builder ----------------------------------------------------------------------------------------------------
D_TIE = 32        # every planted tie group sits at h = 32 of 256 bits: fraction 1/8
THR = (1, 8)      # the threshold through the tie rank
N_FILL = 4000     # random 32-byte rows
N_PATTERNS = 16   # flip masks per distance: planted rows are not all the same code


def _masks(rng, n_bits, h):
    """N_PATTERNS masks of n_bits // 8 bytes, each with exactly h bits set."""
    m = np.zeros((N_PATTERNS, n_bits), dtype=np.uint8)
    for j in range(N_PATTERNS):
        m[j, rng.choice(n_bits, h, replace=False)] = 1
    return np.packbits(m, axis=1)


def _group_keys(rng, q, n, key_bytes):
    """
    Keys of query q's planted group (n rows), chosen so that the radix pivot is decided in the last key byte:
      8 bytes:  one contiguous range, so the rows share all top bytes above the range's width (the top 7 when n <= 256);
                query 0's range starts at key 0, query 1's ends at 2**64 - 1 (the empty-slot value)
      16 bytes: every row shares the high half, the low half is a contiguous range - the pivot lies in bytes 8..15;
                query 1's group has high half 2**64 - 1 and ends at (2**64 - 1, 2**64 - 1); query 2's high halves
                differ only in their last byte (four sub-groups)
    -> (hi, lo) uint64[n]
    """
    off = np.arange(n, dtype=np.uint64)
    v = min(q, 3)
    if key_bytes == 8:
        if v == 0:
            hi = off
        elif v == 1:
            hi = np.uint64(U64_MAX - n + 1) + off
        else:
            hi = (np.uint64(int(rng.integers(1, 2**39))) << np.uint64(24)) + off
        return hi, np.zeros(n, dtype=np.uint64)
    top = np.uint64(int(rng.integers(1, 2**62)) << 2)
    if v == 0:
        return np.full(n, top, dtype=np.uint64), off
    if v == 1:
        return np.full(n, U64_MAX, dtype=np.uint64), np.uint64(U64_MAX - n + 1) + off
    if v == 2:
        return (top & ~np.uint64(0xFF)) | (off % np.uint64(4)), off
    return np.full(n, top, dtype=np.uint64), (np.uint64(int(rng.integers(1, 2**39))) << np.uint64(24)) + off


class Case:
    """A store and queries with known planted groups: keys hi/lo uint64 (lo None for 8-byte keys), codes, lens, queries."""

    def __init__(self, key_bytes, hi, lo, codes, lens, queries, groups):
        self.key_bytes, self.hi, self.lo = key_bytes, hi, lo
        self.codes, self.lens, self.queries = codes, lens, queries
        self.qlens = np.full(len(queries), 32, dtype=np.uint8)
        self.groups = groups   # per query: (row indices below d, row indices at d)

    def store_keys(self, rows=slice(None)):
        if self.key_bytes == 8:
            return np.ascontiguousarray(self.hi[rows])
        return keys16(self.hi[rows], self.lo[rows])

    def store(self):
        st = Store(key_bytes=self.key_bytes, max_bytes=32)
        st.add(self.store_keys(), self.codes, self.lens)
        assert st.size() == len(self.lens)
        return st


def keys16(hi, lo):
    n = len(hi)
    k = np.zeros((n, 16), dtype=np.uint8)
    k[:, :8] = hi.astype(">u8").view(np.uint8).reshape(n, 8)
    k[:, 8:] = lo.astype(">u8").view(np.uint8).reshape(n, 8)
    return k


def planted_ties(counts, key_bytes, seed, d=D_TIE, cross=(), n_fill=N_FILL):
    """
    One 32-byte query per entry of `counts` = [(n_lt, n_eq)]: n_lt rows strictly below distance d (h uniform in 0..d-1)
    and n_eq rows at exactly d, by flipping bits of the query. Queries in `cross` get cross-length ties: every third tie
    row is 8 bytes at h = d/4 and every third 16 bytes at h = d/2 - the same fraction, cut by key. Plus n_fill random rows.
    """
    rng = np.random.default_rng(seed)
    queries = rng.integers(0, 256, size=(len(counts), 32), dtype=np.uint8)
    lt_bank = np.stack([_masks(rng, 256, h) for h in range(d)])
    eq_bank = {32: _masks(rng, 256, d), 16: _masks(rng, 128, d // 2), 8: _masks(rng, 64, d // 4)}
    his, los, codes, lens, groups = [], [], [], [], []
    n0 = 0
    for q, (n_lt, n_eq) in enumerate(counts):
        n = n_lt + n_eq
        c = np.zeros((n, 32), dtype=np.uint8)
        ln = np.full(n, 32, dtype=np.uint8)
        h_lt = rng.integers(0, d, size=n_lt)
        c[:n_lt] = queries[q] ^ lt_bank[h_lt, np.arange(n_lt) % N_PATTERNS]
        j = np.arange(n_eq)
        eq_len = np.where(j % 3 == 1, 8, np.where(j % 3 == 2, 16, 32)) if q in cross else np.full(n_eq, 32)
        for L in (8, 16, 32):
            sel = np.flatnonzero(eq_len == L)
            c[n_lt + sel, :L] = queries[q, :L] ^ eq_bank[L][sel % N_PATTERNS]
            ln[n_lt + sel] = L
        hi, lo = _group_keys(rng, q, n, key_bytes)
        perm = rng.permutation(n)   # rows below d and at d interleave in key order
        his.append(hi[perm])
        los.append(lo[perm])
        codes.append(c)
        lens.append(ln)
        groups.append((n0 + np.arange(n_lt), n0 + n_lt + np.arange(n_eq)))
        n0 += n
    codes.append(rng.integers(0, 256, size=(n_fill, 32), dtype=np.uint8))
    lens.append(np.full(n_fill, 32, dtype=np.uint8))
    his.append(synth.make_keys(0, n_fill, seed))
    los.append(synth.make_keys(0, n_fill, seed + 1) if key_bytes == 16 else np.zeros(n_fill, dtype=np.uint64))
    hi, lo = np.concatenate(his), np.concatenate(los)
    assert len(np.unique(np.stack([hi, lo], axis=1), axis=0)) == len(hi), "keys must be unique"
    return Case(key_bytes, hi, lo if key_bytes == 16 else None, np.concatenate(codes), np.concatenate(lens), queries, groups)


def exact_counts(case, k, thr=None):
    """From the oracle's exact distances, per query -> (total_le, n_out): rows with rank <= d*, and rows returned."""
    out = []
    for q in range(len(case.queries)):
        h, nb = nphd_oracle.prefix_hamming(case.codes, case.lens, case.queries[q], 32)
        d = h.astype(np.int64) * (nphd_oracle.LCM_BITS // nb.astype(np.int64))   # h / n as an exact integer
        if thr is not None:
            d = d[h.astype(np.int64) * thr[1] <= thr[0] * nb.astype(np.int64)]
        total_le = len(d) if len(d) < k else int((d <= np.partition(d, k - 1)[k - 1]).sum())
        out.append((total_le, min(k, total_le)))
    return out


def _key_pairs(got_keys, key_bytes):
    """Search output keys -> (hi, lo) uint64 arrays of the same leading shape."""
    if key_bytes == 8:
        return got_keys, np.zeros_like(got_keys)
    g = np.ascontiguousarray(got_keys)
    return g[..., :8].copy().view(">u8")[..., 0].astype(np.uint64), g[..., 8:].copy().view(">u8")[..., 0].astype(np.uint64)


def check_exact(case, got, k, thr=None, queries=None):
    """Bit-exact against the C oracle: counts, keys in order, h, nbits, stored codes, and the padding past the count."""
    gk, gh, gn, gc, gcodes = got
    qi = np.arange(len(case.queries)) if queries is None else np.asarray(queries)
    rows, h, nb, cnt = oracle_topk(case.hi, case.codes, case.lens, case.queries[qi], case.qlens[qi], k, thr, keys_lo=case.lo)
    assert np.array_equal(gc.astype(np.int64), cnt.astype(np.int64)), f"counts {gc.tolist()} != {cnt.tolist()}"
    ghi, glo = _key_pairs(gk, case.key_bytes)
    lo = case.lo if case.lo is not None else np.zeros_like(case.hi)
    for i in range(len(qi)):
        c = int(cnt[i])
        r = rows[i, :c]
        assert np.array_equal(ghi[i, :c], case.hi[r]) and np.array_equal(glo[i, :c], lo[r]), f"query {qi[i]}: keys/order differ"
        assert np.array_equal(gh[i, :c], h[i, :c]) and np.array_equal(gn[i, :c], nb[i, :c]), f"query {qi[i]}: h/nbits differ"
        if gcodes is not None:
            assert np.array_equal(gcodes[i, :c], case.codes[r]), f"query {qi[i]}: codes differ"
        assert (ghi[i, c:] == U64_MAX).all(), f"query {qi[i]}: key padding"
        assert case.key_bytes == 8 or (glo[i, c:] == U64_MAX).all(), f"query {qi[i]}: key padding"
        assert (gh[i, c:] == 0xFFFF).all() and (gn[i, c:] == 1).all(), f"query {qi[i]}: h/nbits padding"


# ---- A. k_select at every cutoff (>= 5 queries: the batch path) -------------------------------------------------------
SMALL_KS = (256, 257, 1024, 1025, 2048, 2049)
BIG_KS = ("cap_max+1", 10007, 65536)


def select_cases(k, cap, cap_max):
    """
    -> [(name, n_lt, n_eq, mode, regime)], mode 'topk' or 'thr': the search in which the case is named for `regime`
    (queries are searched in both modes and compared in both; queries 2 and 4 carry cross-length ties).
    """
    if k <= cap_max:
        cases = [("all_ties_win", k - k // 2, k // 2, "topk", "S1"),          # total_le = k
                 ("one_tie_loses", k // 2, k - k // 2 + 1, "topk", "S1"),     # total_le = k + 1
                 ("full_capacity", k - 1, cap - k + 1, "topk", "S1"),         # total_le = cap
                 ("one_winner_past_capacity", k - 1, cap - k + 2, "topk", "S2"),   # total_le = cap + 1
                 ("many_ties", k // 2, 3 * cap - k // 2, "topk", "S2")]
        if k == cap_max:   # total_le = cap_max exactly full; cap_max + 1 with every row below d* but one kept
            cases[1] = ("one_winner_past_capacity_k", 1, k, "topk", "S2")
        return cases
    return [("all_ties_win", k - 300, 300, "topk", "B1"),                    # total_le = k
            ("one_winner", k - 1, 2, "topk", "B2"),                          # total_le = k + 1
            ("many_ties", k // 2, 2 * k, "topk", "B2"),                      # more survivors than the scratch holds
            ("below_k_on_threshold", max(k - 1, cap + 1) - 500, 500, "thr", "B1"),   # cap < total_le = k - 1 (or k)
            ("just_past_capacity", cap - 99, 100, "thr", "B1"),              # total_le = cap + 1
            ("at_capacity", cap - 100, 100, "thr", "S1"),                    # total_le = cap, big scratch present
            ("few", 60, 40, "thr", "S1")]


@pytest.fixture(scope="module")
def cap_max_of(cuda):
    optin = device_smem_optin()
    return {kb: max_sort_cap(optin, kb) for kb in (8, 16)}


@pytest.mark.parametrize("key_bytes", (8, 16))
@pytest.mark.parametrize("k", SMALL_KS + ("cap_max",) + BIG_KS)
def test_k_select_regimes(cap_max_of, key_bytes, k):
    cap_max = cap_max_of[key_bytes]
    k = {"cap_max": cap_max, "cap_max+1": cap_max + 1}.get(k, k)
    cap = sort_cap(k, cap_max)
    cases = select_cases(k, cap, cap_max)
    case = planted_ties([(a, b) for _, a, b, _, _ in cases], key_bytes, seed=k * 7 + key_bytes, cross=(2, 4))
    assert not small_path_takes(len(cases), k)
    st = case.store()
    try:
        for mode, thr in (("topk", None), ("thr", THR)):
            counts = exact_counts(case, k, thr)
            for (name, n_lt, n_eq, m, regime), (total_le, n_out) in zip(cases, counts):
                if m == mode:
                    assert total_le == n_lt + n_eq, f"{name}: planted {n_lt + n_eq}, within d* {total_le}"
                    assert select_regime(k, total_le, cap) == regime, f"{name}: k {k}, total_le {total_le}, cap {cap}"
            got = st.search(case.queries, case.qlens, k, thr=thr, with_codes=True)
            stats = st.stats()
            assert stats["fallback_queries"] == 0 and stats["kernel_launches"] > 1
            check_exact(case, got, k, thr)
    finally:
        st.close()


# ---- B. the small path's fused select (<= 4 queries) ------------------------------------------------------------------
SMALL_CASES = (("no_radix_cut", 50, 206), ("radix_cut", 50, 207), ("one_launch_full", 99, 3997), ("falls_back", 60, 4037))


@pytest.mark.parametrize("key_bytes", (8, 16))
def test_small_select_cutoffs(cuda, key_bytes):
    k = 100
    case = planted_ties([(a, b) for _, a, b in SMALL_CASES], key_bytes, seed=500 + key_bytes, cross=(1,))
    totals = [t for t, _ in exact_counts(case, k)]
    assert totals == [SMALL_RADIX_MIN, SMALL_RADIX_MIN + 1, SMALL_SORT_CAP, SMALL_SORT_CAP + 1]
    st = case.store()
    try:
        def run(qs):
            qs = np.asarray(qs)
            got = st.search(case.queries[qs], case.qlens[qs], k, with_codes=True)
            check_exact(case, got, k, queries=qs)
            return st.stats()["kernel_launches"]

        assert small_path_takes(3, k)
        assert run([0, 1, 2]) == 1                 # 256 and 257 survivors, 4096 within d*: one launch
        for qs in ([3], [0, 3], [1, 2, 3]):        # 4097 within d*: the request falls back, still exact
            assert run(qs) > 1, qs
            assert run([0, 1, 2]) == 1             # and the next small request is answered in one launch again
        assert run([2]) == 1 and run([1]) == 1
    finally:
        st.close()


@pytest.mark.parametrize("key_bytes", (8, 16))
def test_small_select_k_2048_ties_share_high_half(cuda, key_bytes):
    k = SMALL_MAX_K
    counts = [(1000, 3000), (k - 1, 2), (100, 2200), (k - 600, 600)]   # radix cut; one winner; cut; every tie wins
    case = planted_ties(counts, key_bytes, seed=600 + key_bytes, cross=(2,))
    assert [t for t, _ in exact_counts(case, k)] == [a + b for a, b in counts]
    st = case.store()
    try:
        for qs in ([0, 1, 2, 3], [0], [1, 3]):
            qs = np.asarray(qs)
            got = st.search(case.queries[qs], case.qlens[qs], k, with_codes=True)
            assert st.stats()["kernel_launches"] == 1, qs
            check_exact(case, got, k, queries=qs)
    finally:
        st.close()


# ---- C. overflow re-scan inside a tiled batch -------------------------------------------------------------------------
RESCAN_LENGTHS = (8, 16, 32)
RESCAN_PER_LENGTH = 100       # ISX_MAX_TILE=64: two tiles of 50 per length, six tiles
RESCAN_TARGETS = (10, 170, 240)   # one query of each length, in the first or second tile of its length
RESCAN_KS = (10, 9000)
RESCAN_FILL = 400_000


def rescan_case():
    """
    300 queries of 8, 16 and 32 bytes with 128-bit keys. Three of them are prefixes of one 32-byte code X stored
    candidate_capacity(9000) + 8192 times (tie keys share the high half), so they overflow their candidate list at every
    k searched. The other queries are at least 44/64, 80/128 or 150/256 bits from X, so the copies never enter their
    lists, and the random rows (400 000, every length) keep their running thresholds far below the copies.
    """
    rng = np.random.default_rng(7300)
    x = rng.integers(0, 256, size=32, dtype=np.uint8)
    n_dup = candidate_capacity(max(RESCAN_KS)) + 8192
    qlens = np.repeat(np.array(RESCAN_LENGTHS, dtype=np.uint8), RESCAN_PER_LENGTH)
    flips = rng.random((len(qlens), 256)) < 0.75
    for L, need in ((8, 44), (16, 80), (32, 150)):
        flips[:, : 8 * L][flips[:, : 8 * L].sum(axis=1) < need] = True
    queries = x ^ np.packbits(flips, axis=1)
    queries[RESCAN_TARGETS, :] = x
    queries[np.arange(32)[None, :] >= qlens[:, None]] = 0
    fill_lens = np.array(RESCAN_LENGTHS, dtype=np.uint8)[rng.integers(0, 3, size=RESCAN_FILL)]
    fill = rng.integers(0, 256, size=(RESCAN_FILL, 32), dtype=np.uint8)
    fill[np.arange(32)[None, :] >= fill_lens[:, None]] = 0
    codes = np.concatenate([fill, np.repeat(x[None], n_dup, axis=0)])
    lens = np.concatenate([fill_lens, np.full(n_dup, 32, dtype=np.uint8)])
    hi = np.concatenate([synth.make_keys(0, RESCAN_FILL, 7301), np.full(n_dup, 0x5EED << 40, dtype=np.uint64)])
    lo = np.concatenate([synth.make_keys(0, RESCAN_FILL, 7302), rng.permutation(n_dup).astype(np.uint64) << np.uint64(5)])
    case = Case(16, hi, lo, codes, lens, queries, None)
    case.qlens = qlens
    return case


_RESCAN_ARM_SCRIPT = r"""
import json, sys
import numpy as np
sys.path.insert(0, sys.argv[1])
from tests import test_gpu_select_edges as t
case = t.rescan_case()
st = case.store()
out, fb = {}, {}
for k in t.RESCAN_KS:
    gk, gh, gn, gc, codes = st.search(case.queries, case.qlens, k, with_codes=True)
    s = st.stats()
    fb[k] = [s["fallback_queries"], s["passes"]]
    out.update({f"k{k}_keys": gk, f"k{k}_h": gh, f"k{k}_nb": gn, f"k{k}_cnt": gc, f"k{k}_codes": codes})
st.close()
np.savez(sys.argv[2], **out)
print(json.dumps(fb))
"""


_ENV_SWITCHES = ("ISX_MAX_TILE", "ISX_TILE_LANES", "ISX_TILE_BALANCE", "ISX_SMALL_PATH", "ISX_TC_SCAN", "ISX_STAGE")


def _run_arm(script, env, out_path):
    """Run `script` in a fresh interpreter with the switches `env` -> (its last stdout line as JSON, npz)."""
    full = {k: v for k, v in os.environ.items() if k not in _ENV_SWITCHES}
    full.update(env)
    r = subprocess.run([sys.executable, "-c", script, str(ROOT), str(out_path)], capture_output=True, text=True,
                       timeout=1200, cwd=str(ROOT), env=full)
    assert r.returncode == 0, r.stderr[-2000:]
    return json.loads(r.stdout.strip().splitlines()[-1]), np.load(out_path)


def test_overflow_rescan_in_tiled_batch_on_every_lane_count(cuda, tmp_path):
    arms = {lanes: _run_arm(_RESCAN_ARM_SCRIPT, {"ISX_MAX_TILE": "64", "ISX_TILE_LANES": str(lanes)}, tmp_path / f"l{lanes}.npz")
            for lanes in (1, 2, 4)}
    for lanes, (fb, res) in arms.items():
        for k in RESCAN_KS:
            assert fb[str(k)] == [len(RESCAN_TARGETS), 6], f"lanes {lanes}, k {k}: (fallback queries, tiles) {fb[str(k)]}"
        for f in arms[1][1].files:
            assert np.array_equal(res[f], arms[1][1][f]), f"lanes {lanes}: {f}"
    case = rescan_case()
    cap_max = max_sort_cap(device_smem_optin(), 16)
    res = arms[2][1]
    for k in RESCAN_KS:
        for q in RESCAN_TARGETS:   # every copy of X is at d* = 0: more rows than the list holds, k of them returned
            h, nb = nphd_oracle.prefix_hamming(case.codes, case.lens, case.queries[q], case.qlens[q])
            total_le = int((h == 0).sum())
            assert total_le > candidate_capacity(k)
            assert select_regime(k, total_le, sort_cap(k, cap_max)) == ("B2" if k > cap_max else "S2")
        got = tuple(res[f"k{k}_{f}"] for f in ("keys", "h", "nb", "cnt", "codes"))
        check_exact(case, got, k)
    assert max(RESCAN_KS) > cap_max


# ---- D. k_merge against a plain reference -----------------------------------------------------------------------------
# equal fractions at every compared length: 1/8 = 8/64 = 16/128 = 24/192 = 32/256, and 0, 1/2 the same way
FRACTIONS = [(f * n // 8, n) for f in (0, 1, 4) for n in (64, 128, 192, 256)]


def merge_case(G, Q, k, counts, key_bytes, seed):
    """
    Per shard g and query q a sorted list of min(counts[g][q], k) records (h, n, hi, lo), garbage past it; keys unique
    over all shards, interleaved across shards, drawn from equal fractions at different nbits. 16-byte keys share the
    high half in a query. -> (h, n, hi, lo) uint[G][Q][k], cnt uint32[G][Q], expected [(h, n, hi, lo)] per query
    """
    rng = np.random.default_rng(seed)
    h = rng.integers(0, 2**16, size=(G, Q, k), dtype=np.uint16)
    n = rng.integers(0, 2**16, size=(G, Q, k), dtype=np.uint16)
    hi = rng.integers(0, 2**63, size=(G, Q, k), dtype=np.uint64)
    lo = rng.integers(0, 2**63, size=(G, Q, k), dtype=np.uint64)
    cnt = np.asarray(counts, dtype=np.uint32).reshape(G, Q)
    expected = []
    for q in range(Q):
        m = [min(int(cnt[g, q]), k) for g in range(G)]
        keys = rng.permutation(4 * sum(m) + 4)[: sum(m)].astype(np.uint64)   # unique, shard membership random
        shared_hi = np.uint64(int(rng.integers(0, 2**64 - 1, dtype=np.uint64)))
        recs, i0 = [], 0
        for g in range(G):
            fr = [FRACTIONS[j] for j in rng.integers(0, len(FRACTIONS), size=m[g])]
            if key_bytes == 16:
                r = [(a, b, int(shared_hi), int(keys[i0 + j])) for j, (a, b) in enumerate(fr)]
            else:
                r = [(a, b, int(keys[i0 + j]) * 0x9E3779B97F4A7C15 % 2**64, 0) for j, (a, b) in enumerate(fr)]
            i0 += m[g]
            r.sort(key=lambda t: (Fraction(t[0], t[1]), t[2], t[3]))
            for j, t in enumerate(r):
                h[g, q, j], n[g, q, j], hi[g, q, j], lo[g, q, j] = t
            recs += r
        recs.sort(key=lambda t: (Fraction(t[0], t[1]), t[2], t[3]))
        expected.append(recs[:k])
    return h, n, hi, lo, cnt, expected


MERGE_SHAPES = [(G, k) for G in (1, 2, 3, 8) for k in (1, 7, 1000)]


@pytest.fixture(scope="module")
def merge_store(cuda):
    st = Store(key_bytes=8, max_bytes=32)   # only lends its stream to the merge
    yield st
    st.close()


@pytest.mark.parametrize("packed", (False, True), ids=("dense", "packed"))
@pytest.mark.parametrize("key_bytes", (8, 16))
@pytest.mark.parametrize("G,k", MERGE_SHAPES)
def test_merge_kernel_against_sorted_reference(merge_store, G, k, key_bytes, packed):
    import torch

    Q = 6
    rng = np.random.default_rng(G * 1000 + k)
    # per query: empty shards, fewer than k, exactly k, more than k (clamped), and a mix
    per_q = [[0] * G, [max(0, k - 1 - g) for g in range(G)], [k] * G, [k + 5 + g for g in range(G)],
             [(0, k // 2, k, 3 * k)[g % 4] for g in range(G)], rng.integers(0, 2 * k + 1, size=G).tolist()]
    counts = np.array(per_q, dtype=np.uint32).T   # [G][Q]
    h, n, hi, lo, cnt, expected = merge_case(G, Q, k, counts, key_bytes, seed=G * 31 + k + key_bytes)
    dev = torch.device("cuda", 0)
    if packed:   # per-shard buffers back to back, as an all-gather of `record_layout` buffers delivers them
        off, size = record_layout(Q, k)
        buf = np.zeros(G * size, dtype=np.uint8)
        for g in range(G):
            b = buf[g * size:(g + 1) * size]
            for name, a in (("khi", hi[g]), ("klo", lo[g]), ("h", h[g]), ("n", n[g]), ("cnt", cnt[g])):
                raw = np.ascontiguousarray(a).view(np.uint8).ravel()
                b[off[name]: off[name] + len(raw)] = raw
        d_in = torch.from_numpy(buf).to(dev)
        src = [d_in.data_ptr() + off[f] for f in ("khi", "klo", "h", "n", "cnt")]
        stride = size
    else:   # dense [G][Q][k] arrays per field
        signed = {2: np.int16, 4: np.int32, 8: np.int64}
        d_in = [torch.from_numpy(np.ascontiguousarray(a).view(signed[a.itemsize])).to(dev) for a in (hi, lo, h, n, cnt)]
        src = [a.data_ptr() for a in d_in]
        stride = 0
    out = [torch.zeros(Q * k, dtype=torch.int64, device=dev), torch.zeros(Q * k, dtype=torch.int64, device=dev),
           torch.zeros(Q * k, dtype=torch.int16, device=dev), torch.zeros(Q * k, dtype=torch.int16, device=dev),
           torch.zeros(Q, dtype=torch.int32, device=dev)]
    torch.cuda.synchronize()
    _lib.check(_lib.lib().isx_merge_device(merge_store.handle, G, Q, k, stride, *src, *[o.data_ptr() for o in out], 1))
    gkhi, gklo, gh, gn = (o.cpu().numpy().view(t).reshape(Q, k) for o, t in zip(out, (np.uint64, np.uint64, np.uint16, np.uint16)))
    gc = out[4].cpu().numpy().view(np.uint32)
    for q in range(Q):
        exp = expected[q]
        c = len(exp)
        assert gc[q] == c == min(k, sum(min(int(x), k) for x in counts[:, q])), f"query {q}: count"
        got = list(zip(gh[q, :c].tolist(), gn[q, :c].tolist(), gkhi[q, :c].tolist(), gklo[q, :c].tolist()))
        assert got == [tuple(int(v) for v in t) for t in exp], f"query {q}: records differ"
        assert (gkhi[q, c:] == U64_MAX).all() and (gklo[q, c:] == U64_MAX).all(), f"query {q}: key padding"
        assert (gh[q, c:] == 0xFFFF).all() and (gn[q, c:] == 1).all(), f"query {q}: h/nbits padding"


# ---- E. first-of-asset: the largest accepted count and the refusal above it ---------------------------------------------
def test_first_of_asset_largest_count_and_refusal(cuda):
    kmax = first_of_asset_max_count(device_smem_optin())
    rng = np.random.default_rng(11)
    n, nq = kmax + 4000, 3
    assets = rng.integers(0, 2000, size=n, dtype=np.uint64)
    assets[:40] = np.uint64(U64_MAX)                       # the asset id that equals the table's empty marker
    lo = np.arange(n, dtype=np.uint64)
    vecs = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    vecs[:, 8:] = 0
    lens = np.full(n, 8, dtype=np.uint8)
    st = Store(key_bytes=16, max_bytes=8, fixed_len=8)
    try:
        st.add(keys16(assets, lo), vecs, lens)
        q, ql = np.ascontiguousarray(vecs[:nq]), np.ascontiguousarray(lens[:nq])
        first = np.zeros((nq, kmax), dtype=np.uint8)
        gk, gh, gn, gc, _ = st.search(q, ql, kmax, first_of_asset=first)
        assert (gc == kmax).all()
        ghi, _ = _key_pairs(gk, 16)
        for i in range(nq):
            _, first_idx = np.unique(ghi[i], return_index=True)
            expect = np.zeros(kmax, dtype=np.uint8)
            expect[first_idx] = 1
            assert np.array_equal(first[i], expect), f"query {i}: first-of-asset flags"
        # one above: refused with ISX_ELIMIT, and the message states the bound the check enforces
        k = kmax + 1
        out = [np.zeros((nq, k, 16), dtype=np.uint8), np.zeros((nq, k), dtype=np.uint16), np.zeros((nq, k), dtype=np.uint16),
               np.zeros(nq, dtype=np.uint32), None, np.zeros((nq, k), dtype=np.uint8)]
        L = _lib.lib()
        rc = L.isx_search(st.handle, _lib.ptr(q), _lib.ptr(ql), nq, k, 0, 0, *[_lib.ptr(a) for a in out])
        assert rc == _lib.ISX_ELIMIT
        assert f"count <= {kmax}" in L.isx_last_error().decode(), L.isx_last_error()
    finally:
        st.close()
