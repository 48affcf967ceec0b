"""
GPU edge tests of every scan path, each compared bit-exactly with the CPU oracle, each asserting the path it exercises:
  A. the small path (csrc/small.cuh) at every compared length 1..32 bytes: every word count of `small_consume`, units of
     16/8/5/4/3/2 blocks straddling a segment boundary, partial last words, rows exactly on the bound, the fall-back to
     the general path at its limits, and the same bytes under ISX_SMALL_WIDE=0, ISX_SMALL_DYNAMIC=1 and ISX_SMALL_MAXQ=8
  B. the POPC scan (`k_scan`, csrc/kernels.cuh) on length tiles of 1, 3, 5 and 63 queries, and at the cutoffs of its
     lower-bound filter tiers, with rows that differ from the query only past the compared length
  C. removed rows whose bytes stay past a segment's live count, on the small path, `k_scan`, `k_scan_tc`, the self-join
     and a saved and reloaded store, including a bucket whose last segment was emptied and refilled
  D. the candidate stage of the scans: full (ISX_STAGE=64) and absent (ISX_STAGE=0) give the same bytes as the default
Path markers are deterministic statistics: the small path answers in one launch, the tensor-core scan issues no POPC, the
POPC scan does. Environment switches are read once per process, so the arms of A and D run in subprocesses.
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
from oracle import self_join as join_oracle
from tests.helpers import assert_same_topk, make_store_arrays, oracle_topk
from tests.test_gpu_tc_epilogue import bound_case, check_bound_rows

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent
_ENV_SWITCHES = ("ISX_SMALL_WIDE", "ISX_SMALL_DYNAMIC", "ISX_SMALL_MAXQ", "ISX_SMALL_PATH", "ISX_TC_SCAN", "ISX_STAGE")


def _run_arm(script, env, out_path, *args):
    """Run `script` in a fresh interpreter with the switches `env` (and no other) -> (its last stdout line as JSON, npz)."""
    full = {k: v for k, v in os.environ.items() if k not in _ENV_SWITCHES}
    full.update(env)
    r = subprocess.run([sys.executable, "-c", script, str(ROOT), str(out_path), *args], capture_output=True, text=True,
                       timeout=900, cwd=str(ROOT), env=full)
    assert r.returncode == 0, r.stderr[-2000:]
    return json.loads(r.stdout.strip().splitlines()[-1]), np.load(out_path)


def _rank_in_length(lens):
    """Position of every row among the rows of its length, in array order."""
    order = np.argsort(lens, kind="stable")
    sl = lens[order]
    rank = np.empty(len(lens), dtype=np.int64)
    rank[order] = np.arange(len(lens)) - np.searchsorted(sl, sl, side="left")
    return rank


# ---- A. the small path -------------------------------------------------------------------------------------------------
# Eight lengths per store, one per word count, R <= 1024 rank classes (857, 753, 881, 705): together every length 1..32.
SMALL_STORES = ((1, 5, 9, 13, 17, 21, 25, 29), (2, 7, 10, 15, 18, 23, 26, 30), (3, 6, 11, 14, 19, 22, 27, 31),
                (4, 8, 12, 16, 20, 24, 28, 32))
# 1/5 rather than a looser second threshold: a 1-byte query compares one byte of every row, and the rows within its
# threshold must stay under the fused select's 4096 for the small path to answer
SMALL_THRESHOLDS = ((1, 8), (1, 5))
SMALL_FIRST_ADD = 3000       # rows per length in the first add: each bucket's first segment holds 4096 rows
SMALL_FILL = 8 * 6500        # ~6 500 rows per length: a 4096-row segment and part of a 16 384-row one, 7 blocks
SMALL_REQUESTS = (1, 2, 3, 4)


def small_case(lengths, thr):
    # 3 queries per length; per query, rows on / past the bound one length shorter, equal and one length longer
    return bound_case(thr, 3, lengths, row_steps=(-1, 0, 1), n_fill=SMALL_FILL)


def build_two_segment_store(case, seed):
    """The rows in a fixed random order, in two adds: every bucket spans a 4096-row segment and a larger one."""
    keys, codes, lens = case[:3]
    order = np.random.default_rng(seed).permutation(len(lens))
    rank = _rank_in_length(lens[order])
    st = Store(key_bytes=8, max_bytes=32)
    for sel in (rank < SMALL_FIRST_ADD, rank >= SMALL_FIRST_ADD):
        idx = order[sel]
        st.add(np.ascontiguousarray(keys[idx]), np.ascontiguousarray(codes[idx]), np.ascontiguousarray(lens[idx]))
    return st


def search_in_requests(st, queries, qlens, k, thr, sizes, seed):
    """All queries in a fixed random order, in requests of `sizes` queries (cycled) -> (keys, h, nbits, counts), launches."""
    n = len(qlens)
    order = np.random.default_rng(seed).permutation(n)
    gk = np.zeros((n, k), dtype=np.uint64)
    gh = np.zeros((n, k), dtype=np.uint16)
    gn = np.zeros((n, k), dtype=np.uint16)
    gc = np.zeros(n, dtype=np.uint32)
    launches = []
    i = j = 0
    while i < n:
        idx = order[i: i + sizes[j % len(sizes)]]
        r = st.search(np.ascontiguousarray(queries[idx]), np.ascontiguousarray(qlens[idx]), k, thr=thr)
        gk[idx], gh[idx], gn[idx], gc[idx] = r[:4]
        launches.append(st.stats()["kernel_launches"])
        i += len(idx)
        j += 1
    return (gk, gh, gn, gc), launches


def small_runs(stores, sizes):
    """Every search of part A -> yields (name, case, k, thr, (keys, h, nbits, counts), launches per request)."""
    for lengths in stores:
        for thr in SMALL_THRESHOLDS:
            case = small_case(lengths, thr)
            st = build_two_segment_store(case, lengths[0])
            try:
                searches = [(2048, thr)] + ([(1, None), (100, None)] if thr == SMALL_THRESHOLDS[0] else [])
                for k, t in searches:
                    got, launches = search_in_requests(st, case[3], case[4], k, t, sizes, 31 * lengths[0] + k)
                    yield f"L{lengths[0]}_t{thr[1]}_k{k}_{'thr' if t else 'topk'}", case, k, t, got, launches
            finally:
                st.close()


@pytest.mark.parametrize("lengths", SMALL_STORES, ids=[f"L{s[0]}" for s in SMALL_STORES])
def test_small_path_every_compared_length(cuda, lengths):
    lens = small_case(lengths, SMALL_THRESHOLDS[0])[2]
    per_len = np.bincount(lens, minlength=33)[list(lengths)]
    assert (per_len > 4096).all() and ((per_len + 1023) // 1024 == 7).all()   # 7 blocks: no multiple of any unit size
    for name, case, k, thr, got, launches in small_runs([lengths], SMALL_REQUESTS):
        assert all(n == 1 for n in launches), f"{name}: a request left the small path ({launches})"
        rows, h, nb, cnt = oracle_topk(*case[:5], k, thr)
        assert_same_topk(*got, case[0], rows, h, nb, cnt)
        if thr is not None:
            assert (got[3] < k).all(), name   # every row within the threshold is in the result
            check_bound_rows(case, got[0], got[3])


def test_small_path_limits_fall_back_exactly(cuda):
    case = small_case(SMALL_STORES[3], SMALL_THRESHOLDS[0])
    st = build_two_segment_store(case, 5)
    q, ql = np.ascontiguousarray(case[3][[0, 9, 23]]), np.ascontiguousarray(case[4][[0, 9, 23]])
    gk, gh, gn, gc, _ = st.search(q, ql, 2049)   # one above the largest k the small path takes
    assert st.stats()["kernel_launches"] > 1
    assert_same_topk(gk, gh, gn, gc, case[0], *oracle_topk(*case[:3], q, ql, 2049))
    st.close()
    nine = (2, 4, 8, 12, 16, 20, 24, 28, 32)   # one length more than the small path's ranges, R = 705
    case = bound_case((1, 8), 1, nine, n_fill=9000)
    st = Store(key_bytes=8, max_bytes=32)
    st.add(*case[:3])
    q, ql = np.ascontiguousarray(case[3][[0, 4, 8]]), np.ascontiguousarray(case[4][[0, 4, 8]])
    for k, thr in ((100, None), (2048, (1, 8))):
        gk, gh, gn, gc, _ = st.search(q, ql, k, thr=thr)
        assert st.stats()["kernel_launches"] > 1
        assert_same_topk(gk, gh, gn, gc, case[0], *oracle_topk(*case[:3], q, ql, k, thr))
    st.close()


_SMALL_ARM_SCRIPT = r"""
import json, sys
import numpy as np
sys.path.insert(0, sys.argv[1])
from tests import test_gpu_scan_edges as t
out, launches = {}, []
for name, case, k, thr, got, ln in t.small_runs(t.SMALL_STORES, tuple(json.loads(sys.argv[3]))):
    out.update({name + "_keys": got[0], name + "_h": got[1], name + "_nb": got[2], name + "_cnt": got[3]})
    launches += ln
np.savez(sys.argv[2], **out)
print(json.dumps(launches))
"""


def test_small_path_switches_give_the_same_bytes(cuda, tmp_path):
    arms = {"default": ({}, SMALL_REQUESTS), "narrow_ring": ({"ISX_SMALL_WIDE": "0"}, SMALL_REQUESTS),
            "dynamic_units": ({"ISX_SMALL_DYNAMIC": "1"}, SMALL_REQUESTS), "maxq8": ({"ISX_SMALL_MAXQ": "8"}, (5, 6, 7, 8))}
    out = {name: _run_arm(_SMALL_ARM_SCRIPT, env, tmp_path / f"{name}.npz", json.dumps(sizes)) for name, (env, sizes) in arms.items()}
    for name, (launches, res) in out.items():
        assert launches and all(n == 1 for n in launches), f"{name}: a request left the small path"
        for f in out["default"][1].files:
            assert np.array_equal(res[f], out["default"][1][f]), f"{name}: {f}"


# ---- B. the POPC scan --------------------------------------------------------------------------------------------------
def test_popc_scan_tiles_of_1_3_5_63_queries(cuda):
    case = bound_case((1, 8), (1, 3, 5, 63), (7, 13, 26, 32), row_steps=(-1, 0, 1))
    st = Store(key_bytes=8, max_bytes=32)
    st.add(*case[:3])
    gk, gh, gn, gc, _ = st.search(case[3], case[4], 2048, thr=(1, 8))
    assert st.stats()["issued_popc"] > 0
    st.close()
    assert_same_topk(gk, gh, gn, gc, case[0], *oracle_topk(*case[:5], 2048, (1, 8)))
    assert (gc < 2048).all()
    check_bound_rows(case, gk, gc)


# cutoffs of the lower-bound filter tiers per word count (csrc/kernels.cuh, LowerBound::kCutoff3 and kCutoff2): a query
# whose Hamming bound is at or below one scans with that tier's folds
TIER_CUTOFFS = {2: (17,), 4: (38,), 5: (50,), 6: (48, 60), 7: (61,), 8: (70, 82)}
# per word count one length whose last compared word is full and one where it is partial
TIER_LENGTHS = (6, 8, 14, 16, 19, 20, 23, 24, 26, 28, 30, 32)
TIER_QUERIES = 16   # one length tile of 16 queries: the POPC scan


def tier_case(L):
    """
    16 queries of L bytes. Per query and cutoff c of L's word count, rows at h = c and h = c + 1, half of them with as many
    flips as fit in the last compared word; each once of length L and once of 32 bytes with 0xFF past L. Plus random rows
    of every length. -> (keys, codes, lens, queries, qlens, planted): planted = [(query, row, h)]
    """
    rng = np.random.default_rng(7100 + L)
    last0 = 32 * ((L + 3) // 4 - 1)   # first bit of the last compared word
    queries = np.zeros((TIER_QUERIES, 32), dtype=np.uint8)
    queries[:, :L] = rng.integers(0, 256, size=(TIER_QUERIES, L), dtype=np.uint8)
    rows, lens, planted = [], [], []
    for qi in range(TIER_QUERIES):
        for c in TIER_CUTOFFS[(L + 3) // 4]:
            for h in (c, c + 1):
                for in_last in (False, True):
                    if in_last:
                        n_last = min(h, 8 * L - last0)
                        pos = np.concatenate([last0 + rng.choice(8 * L - last0, n_last, replace=False),
                                              rng.choice(last0, h - n_last, replace=False)])
                    else:
                        pos = rng.choice(8 * L, h, replace=False)
                    bits = np.unpackbits(queries[qi])
                    bits[pos] ^= 1
                    for Lr in ((L, 32) if L < 32 else (L,)):
                        row = np.packbits(bits)
                        row[L:Lr] = 0xFF
                        planted.append((qi, len(rows), h))
                        rows.append(row)
                        lens.append(Lr)
    n_fill = 3000
    fill_lens = rng.integers(1, 33, size=n_fill).astype(np.uint8)
    fill = rng.integers(0, 256, size=(n_fill, 32), dtype=np.uint8)
    fill[np.arange(32)[None, :] >= fill_lens[:, None]] = 0
    codes = np.concatenate([np.stack(rows), fill])
    lens = np.concatenate([np.array(lens, dtype=np.uint8), fill_lens])
    return synth.make_keys(0, len(lens), 7100 + L), codes, lens, queries, np.full(TIER_QUERIES, L, dtype=np.uint8), planted


@pytest.mark.parametrize("L", TIER_LENGTHS)
def test_popc_scan_tier_cutoffs(cuda, L):
    keys, codes, lens, queries, qlens, planted = tier_case(L)
    st = Store(key_bytes=8, max_bytes=32)
    st.add(keys, codes, lens)
    k = 1024   # above every count
    try:
        for c in TIER_CUTOFFS[(L + 3) // 4]:
            for bound in (c, c + 1):   # the tier's last bound, and the first one past it
                thr = (bound, 8 * L)
                gk, gh, gn, gc, _ = st.search(queries, qlens, k, thr=thr)
                assert st.stats()["issued_popc"] > 0
                assert_same_topk(gk, gh, gn, gc, keys, *oracle_topk(keys, codes, lens, queries, qlens, k, thr))
                assert (gc < k).all()
                for qi, row, h in planted:
                    got = int(keys[row]) in set(gk[qi, : gc[qi]].tolist())
                    assert got == (h <= bound), f"bound {bound}: query {qi}, row at h = {h}, length {lens[row]}"
    finally:
        st.close()


# ---- C. removed rows past the live count -------------------------------------------------------------------------------
STALE_Q = 64        # 32-byte queries: one tensor-core tile
STALE_TWINS = 4     # twins (h = 0 rows) per query for each way of leaving bytes past the live count


def stale_store():
    """
    A store in which every query has 6 live twins and 12 removed ones whose bytes stay in partly live blocks:
      (a) bucket 32: the twins are the bucket's tail rows, removed: their bytes stay past n
      (b) bucket 24: twins in the middle of the segment are removed, the tail twins move into the holes: copies of live
          rows stay past n
      (c) bucket 13: its last segment is emptied by removes that also take the last 600 rows (twins among them) of the
          4096-row segment before it; an `add` and an `add_device` then fill the emptied segment, so the bucket holds a
          partly filled segment in the middle of its block list
    -> (store, live keys, codes, lens, removed keys, queries, qlens)
    """
    import torch

    rng = np.random.default_rng(8100)
    queries = rng.integers(0, 256, size=(STALE_Q, 32), dtype=np.uint8)
    qlens = np.full(STALE_Q, 32, dtype=np.uint8)
    parts, is_twin = [], []   # (codes, lens) in the order the rows are added; which of them are twins

    def part(codes_twins, L):
        codes, twin = codes_twins
        codes[:, L:] = 0
        parts.append((codes, np.full(len(codes), L, dtype=np.uint8)))
        is_twin.append(twin)
        return len(parts) - 1

    def fill(n):
        return rng.integers(0, 256, size=(n, 32), dtype=np.uint8), np.zeros(n, dtype=bool)

    def twins(per):
        return np.repeat(queries, per, axis=0), np.ones(STALE_Q * per, dtype=bool)

    def mixed(tw, n_fill):   # twins shuffled among random rows
        perm = rng.permutation(len(tw[0]) + n_fill)
        return np.concatenate([tw[0], fill(n_fill)[0]])[perm], perm < len(tw[0])

    tw = STALE_Q * STALE_TWINS
    # first add: bucket 32 ends 256 rows into block 8; bucket 24 ends 256 rows into block 4; bucket 13 fills exactly
    # one 4096-row segment, its last 600 rows in block 3
    first = [part(fill(3000), 8), part(fill(8692), 32), a_tail := part(twins(STALE_TWINS), 32),
             b_mid := part(mixed(twins(STALE_TWINS), 4696 - tw), 24), part(twins(STALE_TWINS), 24),
             part(fill(3496), 13), c_dead := part(mixed(twins(STALE_TWINS), 600 - tw), 13)]
    c_seg1 = part(fill(2000), 13)
    c_add = part(mixed(twins(1), 1500 - STALE_Q), 13)
    c_dev = part(mixed(twins(1), 700 - STALE_Q), 13)
    starts = np.cumsum([0] + [len(c) for c, _ in parts])
    keys = synth.make_keys(0, int(starts[-1]), 8101)
    codes = np.concatenate([c for c, _ in parts])
    lens = np.concatenate([ln for _, ln in parts])
    rows = [np.arange(starts[i], starts[i + 1]) for i in range(len(parts))]
    cat = lambda ids: np.concatenate([rows[i] for i in ids])   # noqa: E731
    alive = np.zeros(len(keys), dtype=bool)
    st = Store(key_bytes=8, max_bytes=32)
    for ids in (first, [c_seg1]):
        r = cat(ids)
        st.add(keys[r], codes[r], lens[r])
        alive[r] = True
    dead = [rows[a_tail][::-1], rows[b_mid][is_twin[b_mid]], np.concatenate([rows[c_dead], rows[c_seg1]])[::-1]]
    for r in dead:   # (a) and (c) tail first, (b) in row order
        removed, n = st.remove(np.ascontiguousarray(keys[r]), len(r))
        assert n == len(r)
        alive[r] = False
    r = rows[c_add]
    st.add(keys[r], codes[r], lens[r])
    alive[r] = True
    r = rows[c_dev]
    dev = torch.device("cuda", 0)
    d_keys = torch.from_numpy(keys[r].view(np.int64)).to(dev)
    d_codes = torch.from_numpy(codes[r]).to(dev)
    d_lens = torch.from_numpy(lens[r]).to(dev)
    torch.cuda.synchronize()
    st.add_device(d_keys.data_ptr(), d_codes.data_ptr(), d_lens.data_ptr(), len(r))
    alive[r] = True
    assert st.size() == int(alive.sum())
    return st, keys[alive], codes[alive], lens[alive], keys[np.concatenate(dead)], queries, qlens


@pytest.fixture(scope="module")
def stale(cuda):
    case = stale_store()
    yield case
    case[0].close()


def check_survivors(st, case, queries, qlens, k):
    """Exact top-k over the surviving rows, codes included; no removed key, no key twice. -> stats of the search."""
    _, keys, codes, lens, removed = case[:5]
    gk, gh, gn, gc, gcodes = st.search(queries, qlens, k, with_codes=True)
    stats = st.stats()
    rows, h, nb, cnt = oracle_topk(keys, codes, lens, queries, qlens, k)
    assert_same_topk(gk, gh, gn, gc, keys, rows, h, nb, cnt)
    gone = set(removed.tolist())
    for i in range(len(qlens)):
        c = int(cnt[i])
        assert np.array_equal(gcodes[i, :c], codes[rows[i, :c]]), f"query {i}: codes differ"
        got = gk[i, :c].tolist()
        assert len(set(got)) == c and not gone.intersection(got), f"query {i}: a removed or repeated key"
    assert (h[:, :6] == 0).all() and (h[:, 6:] > 0).all()   # the six live twins lead every result
    return stats


def _all_paths(st, case):
    queries, qlens = case[5], case[6]
    for k in (1, 10):   # small path: requests of 4 queries; the phase-0 sample must not count the removed twins
        for i in range(0, 16, 4):
            check_survivors(st, case, queries[i: i + 4], qlens[i: i + 4], k)
            assert st.stats()["kernel_launches"] == 1
    assert check_survivors(st, case, queries[:16], qlens[:16], 10)["issued_popc"] > 0     # one 16-query tile: k_scan
    assert check_survivors(st, case, queries, qlens, 10)["issued_popc"] == 0              # one 64-query tile: k_scan_tc


def _check_join(st, case, thr):
    _, keys, codes, lens = case[:4]
    ka, kb, h, nb = st.self_join(thr)
    ra, rb, eh, en = join_oracle.self_join(keys, None, codes, lens, thr)
    assert len(ka) == len(ra)
    assert np.array_equal(ka, keys[ra]) and np.array_equal(kb, keys[rb])
    assert np.array_equal(h, eh) and np.array_equal(nb, en)
    assert (ka != kb).all()
    return len(ka)


def test_stale_rows_every_scan_path(stale):
    _all_paths(stale[0], stale)


@pytest.mark.parametrize("thr", [(0, 1), (1, 8)])
def test_stale_rows_self_join(stale, thr):
    # the live twins of a query pair up among themselves at h = 0: 15 pairs per query at least
    assert _check_join(stale[0], stale, thr) >= STALE_Q * 15


def test_stale_rows_after_save_and_load(stale, tmp_path):
    stale[0].save(tmp_path / "stale.isx")
    st = Store(key_bytes=8, max_bytes=32)
    try:
        st.load(tmp_path / "stale.isx")
        assert st.size() == len(stale[1])
        _all_paths(st, stale)
        _check_join(st, stale, (0, 1))
    finally:
        st.close()


# ---- D. stage capacity -------------------------------------------------------------------------------------------------
def stage_cases():
    """-> [(name, keys, codes, lens, queries, qlens, k, thr)]"""
    out = []
    keys, codes, lens = make_store_arrays(50_000, 9101)
    q, ql = synth.make_queries(16, len(keys), 9102, 9101)
    out.append(("loose", keys, codes, lens, q, ql, 4096, (1, 2)))   # about half of all rows within the threshold
    keys, codes, lens = make_store_arrays(150_000, 9201, lengths=(32,))
    q, ql = synth.make_queries(2048, len(keys), 9202, 9201, lengths=(32,), row_lengths=(32,))
    out.append(("tile2048", keys, codes, lens, q, ql, 10, None))   # the widest tile: the least room for a stage
    keys, codes, lens = make_store_arrays(100_000, 9301)
    dup_n = 150_000
    dup_codes = np.zeros((dup_n, 32), dtype=np.uint8)
    dup_codes[:, :16] = 0xA7
    q, ql = synth.make_queries(7, len(keys), 9302, 9301)
    out.append(("mass_dup", np.concatenate([keys, synth.make_keys(10**9, dup_n, 9303)]), np.concatenate([codes, dup_codes]),
                np.concatenate([lens, np.full(dup_n, 16, dtype=np.uint8)]), np.concatenate([dup_codes[:1], q]),
                np.concatenate([np.array([16], dtype=np.uint8), ql]), 100, None))   # 150 000 ties overflow the list
    return out


_STAGE_ARM_SCRIPT = r"""
import json, sys
import numpy as np
sys.path.insert(0, sys.argv[1])
from tests import test_gpu_scan_edges as t
from iscc_search_b200._lib import Store
out, popc = {}, {}
for name, keys, codes, lens, q, ql, k, thr in t.stage_cases():
    st = Store(key_bytes=8, max_bytes=32)
    st.add(keys, codes, lens)
    gk, gh, gn, gc, _ = st.search(q, ql, k, thr=thr)
    popc[name] = st.stats()["issued_popc"]
    st.close()
    out.update({name + "_keys": gk, name + "_h": gh, name + "_nb": gn, name + "_cnt": gc})
np.savez(sys.argv[2], **out)
print(json.dumps(popc))
"""


def test_stage_capacity_never_changes_the_result(cuda, tmp_path):
    arms = {"default": {}, "popc": {"ISX_TC_SCAN": "0"}, "popc_stage64": {"ISX_TC_SCAN": "0", "ISX_STAGE": "64"},
            "popc_no_stage": {"ISX_TC_SCAN": "0", "ISX_STAGE": "0"}}
    out = {name: _run_arm(_STAGE_ARM_SCRIPT, env, tmp_path / f"{name}.npz") for name, env in arms.items()}
    assert out["default"][0]["tile2048"] == 0   # the 2048-query tile takes the tensor-core scan by default
    for name in ("popc", "popc_stage64", "popc_no_stage"):
        assert all(v > 0 for v in out[name][0].values()), name
        for f in out["default"][1].files:
            assert np.array_equal(out[name][1][f], out["default"][1][f]), f"{name}: {f}"
    res = out["default"][1]
    for name, keys, codes, lens, q, ql, k, thr in stage_cases():
        assert_same_topk(res[name + "_keys"], res[name + "_h"], res[name + "_nb"], res[name + "_cnt"], keys,
                         *oracle_topk(keys, codes, lens, q, ql, k, thr))
