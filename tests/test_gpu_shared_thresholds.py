"""
GPU edge tests of cross-rank threshold sharing (include/isx.h `isx_share_*`, DESIGN.md §4) on ONE device: W worker
processes, each with its own store and home histograms, attach to each other through CUDA IPC exactly as the ranks of a
multi-GPU box do (on a box with more GPUs rank r takes device r % n). The parent drives every rank over a pipe and replaces
the collectives of `ShardedSearcher` by a host barrier: per batch reset -> device synchronise -> barrier -> the union of
the stored-length masks -> search -> barrier (no rank may zero its homes while a peer can still count into them). The
ranks' results are merged on the host by (h/nbits, key) and compared bit-exactly with the C oracle over the union of all
shards.

Exact results alone cannot show that peer counts reached the kernels (an unshared search is exact too), so the probe
batch measures it: Q copies of a code P; rank 0 holds k copies of P, every other probe rank random rows with every
256th row at exactly D bits from P (N1 of them). A rank that does not share emits every one of its Q * N1 rows at D;
searched after rank 0, a rank that reads the shared histograms finds k rows at distance 0 there at its first
re-derivation and emits at most the rows at D of its first warm-up range, Q * N1 / 8.
"""

import math
import multiprocessing as mp
import os
import sys
import time
import traceback
from multiprocessing.connection import wait
from pathlib import Path

import numpy as np
import pytest

from iscc_search_b200 import synth
from iscc_search_b200.sharded import owner_of
from tests.helpers import assert_same_topk, make_store_arrays, oracle_topk

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent

SHARE_RCAP = 512            # distance ranks per query the shared histograms hold (kShareRcap); beyond it sharing is off
BLOCK_ROWS = 1024
LCM = 8 * math.lcm(*range(1, 33))   # h * (LCM / nbits) orders h/nbits exactly for every nbits = 8..256; < 2**63
BARRIER_S = 300
CALL_S = 900
K = 100

# ---- case builders (checked on the CPU by tests/test_shared_cases_cpu.py) ----------------------------------------------


def rank_count(lengths):
    """R, the number of distinct h/(8m) over the compared-length classes `lengths` (the library's own rank table)."""
    import ctypes

    from iscc_search_b200 import _lib

    rank = np.zeros((33, 257), dtype=np.uint16)
    R = ctypes.c_uint32()
    _lib.check(_lib.lib().isx_selftest_rank_table(sum(1 << (L - 1) for L in lengths), _lib.ptr(rank), None, 0, ctypes.byref(R)))
    return int(R.value)


def cut_lengths():
    """(lo, hi): stored-length sets of 32-byte probe queries, greedily grown from {32} while R <= 512, and lo plus the first
    length that would pass 512."""
    lo, over = [32], None
    for L in range(31, 0, -1):
        if rank_count(lo + [L]) <= SHARE_RCAP:
            lo.append(L)
        elif over is None:
            over = L
    return sorted(lo), sorted(lo + [over])


def warm_span(world):
    """Blocks of the first warm-up range of a >= 64-query tile while shared (csrc/isx.cu: max(8, 64 / world))."""
    return max(8, 64 // world)


PROBE_EVERY = 256   # one probe row in 256: a 1024-row block holds 4, so an item of <= 256 queries stages <= 1024 records


def probe_rows(world):
    """Rows per probe rank: 8 first warm-up ranges."""
    return 8 * warm_span(world) * BLOCK_ROWS


def probe_n1(world):
    """Rows at distance D per probe rank; the first warm-up range holds N1 / 8 of them."""
    return probe_rows(world) // PROBE_EVERY


class Case:
    """Rows of every rank (keys hi, keys lo or None, codes, lens) and their union."""

    def __init__(self, shards):
        self.shards = shards
        self.hi = np.concatenate([s[0] for s in shards])
        self.lo = None if shards[0][1] is None else np.concatenate([s[1] for s in shards])
        self.codes = np.concatenate([s[2] for s in shards])
        self.lens = np.concatenate([s[3] for s in shards])


def split(keys, codes, lens, own, world, lo=None):
    return Case([(keys[own == r], None if lo is None else lo[own == r], codes[own == r], lens[own == r]) for r in range(world)])


def near_rows(P, n, d, rng):
    """n copies of P with d bits flipped in each: d distinct bytes, one bit in each."""
    codes = np.repeat(P[None, :], n, axis=0)
    pos = np.argsort(rng.random((n, 32)), axis=1)[:, :d]
    bit = (1 << rng.integers(0, 8, (n, d))).astype(np.uint8)
    np.bitwise_xor.at(codes, (np.arange(n)[:, None], pos), bit)
    return codes


def probe_case(world, n_rows, d=8, seed=0, extra_lengths=(), key0=7 << 40):
    """
    -> (Case, P). Rank 0: K copies of P (32 bytes). Every other rank: n_rows random 32-byte rows, of which every
    PROBE_EVERY-th is at exactly d bits from P. Rank 1 when `extra_lengths` is given also holds one row per extra length,
    the complement of P's prefix (h/nbits = 1, so they only add distance classes).
    """
    rng = np.random.default_rng(seed)
    P = np.zeros(32, dtype=np.uint8)
    P[:] = rng.integers(0, 256, 32, dtype=np.uint8)
    shards, start = [], key0
    for r in range(world):
        if r == 0:
            codes, lens = np.repeat(P[None, :], K, axis=0), np.full(K, 32, dtype=np.uint8)
        else:
            codes = rng.integers(0, 256, (n_rows, 32), dtype=np.uint8)
            codes[PROBE_EVERY - 1::PROBE_EVERY] = near_rows(P, n_rows // PROBE_EVERY, d, rng)
            lens = np.full(n_rows, 32, dtype=np.uint8)
            if r == 1 and extra_lengths:
                extra = np.zeros((len(extra_lengths), 32), dtype=np.uint8)
                for i, L in enumerate(extra_lengths):
                    extra[i, :L] = ~P[:L]
                codes = np.concatenate([codes, extra])
                lens = np.concatenate([lens, np.asarray(extra_lengths, dtype=np.uint8)])
        shards.append((synth.make_keys(start, len(codes), 91), None, codes, lens))
        start += len(codes)
    return Case(shards), P


def mixed_queries(per_len, n_rows, seed, data_seed, lengths=synth.STANDARD_LENGTHS):
    """Exactly per_len queries of every length in `lengths`, near stored rows (synth.make_queries)."""
    parts = [synth.make_queries(per_len, n_rows, seed + 17 * L, data_seed, lengths=(L,)) for L in lengths]
    return np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts])


def skew_case(n, seed, world, few):
    """Mixed rows; every 24-byte row on the last rank, `few` 8-byte rows (< K) on rank 1, the rest on rank 0 or the last."""
    keys, codes, lens = make_store_arrays(n, seed)
    own = owner_of(keys, world)
    own[own == 1] = 0
    own[np.flatnonzero((own == 0) & (lens == 8))[:few]] = 1
    own[lens == 24] = world - 1
    return split(keys, codes, lens, own, world)


def prefix_planted(n, seed, n_plant):
    """Mixed rows plus n_plant 8-byte rows that repeat the first 8 bytes of longer rows (self-join pairs at h = 0)."""
    keys, codes, lens = make_store_arrays(n, seed)
    src = np.flatnonzero(lens > 8)[:n_plant]
    pc = np.zeros((n_plant, 32), dtype=np.uint8)
    pc[:, :8] = codes[src, :8]
    return (np.concatenate([keys, synth.make_keys(10**9, n_plant, seed)]), np.concatenate([codes, pc]),
            np.concatenate([lens, np.full(n_plant, 8, dtype=np.uint8)]))


def prefix_pairs(keys, codes, lens):
    """Reference of a self-join at threshold 0: every pair whose codes agree on the shorter length, (key_a, key_b) order."""
    out = set()
    for m in np.unique(lens).tolist():
        idx = np.flatnonzero(lens >= m)
        _, inv = np.unique(np.ascontiguousarray(codes[idx, :m]).view(f"V{m}").ravel(), return_inverse=True)
        order = np.argsort(inv, kind="stable")
        grp = np.split(idx[order], np.flatnonzero(np.diff(inv[order])) + 1)
        for g in grp:
            if len(g) < 2:
                continue
            for a in g[lens[g] == m]:
                for b in g:
                    if a != b:
                        ka, kb = sorted((int(keys[a]), int(keys[b])))
                        out.add((ka, kb, 8 * m))
    return sorted(out)


def merge_topk(parts, k):
    """Host merge of per-rank (keys, h, nbits, counts) into the global top-k by (h/nbits, key), keys in Store form."""
    Q = len(parts[0][3])
    k16 = parts[0][0].ndim == 3
    mk = np.zeros_like(parts[0][0])
    mh = np.zeros((Q, k), dtype=np.uint16)
    mn = np.zeros((Q, k), dtype=np.uint16)
    mc = np.zeros(Q, dtype=np.uint32)
    for q in range(Q):
        c = [int(p[3][q]) for p in parts]
        key = np.concatenate([p[0][q, :n] for p, n in zip(parts, c)])
        h = np.concatenate([p[1][q, :n] for p, n in zip(parts, c)]).astype(np.int64)
        nb = np.concatenate([p[2][q, :n] for p, n in zip(parts, c)]).astype(np.int64)
        if k16:
            hi = np.ascontiguousarray(key[:, :8]).view(">u8").ravel().astype(np.uint64)
            lo = np.ascontiguousarray(key[:, 8:]).view(">u8").ravel().astype(np.uint64)
        else:
            hi, lo = key, np.zeros(len(key), dtype=np.uint64)
        order = np.lexsort((lo, hi, h * (LCM // np.maximum(nb, 1))))[:k]
        n = len(order)
        mk[q, :n], mh[q, :n], mn[q, :n], mc[q] = key[order], h[order], nb[order], n
    return mk, mh, mn, mc


def check_merged(case, parts, queries, qlens, k, thr=None):
    rows, h, nb, cnt = oracle_topk(case.hi, case.codes, case.lens, queries, qlens, k, thr, keys_lo=case.lo)
    gk, gh, gn, gc = merge_topk(parts, k)
    assert_same_topk(gk, gh, gn, gc, case.hi, rows, h, nb, cnt, keys_lo=case.lo)


def keys_arg(shard):
    hi, lo = shard[0], shard[1]
    return hi if lo is None else synth.keys128_bytes(hi, lo)


# ---- the rank process ---------------------------------------------------------------------------------------------------


def _rank_main(rank, world, conn, barrier, env):
    """One rank: serves commands from the parent until it sends None. Every reply is ("ok", value) or ("err", message)."""
    try:
        os.environ.update(env)   # the library reads its knobs once per process, at the first search
        if str(ROOT) not in sys.path:
            sys.path.insert(0, str(ROOT))
        import ctypes

        import torch

        from iscc_search_b200 import _lib

        L = _lib.lib()
        dev = rank % torch.cuda.device_count()
        torch.cuda.set_device(dev)
        stores = {}
    except BaseException:
        conn.send(("err", f"rank {rank}: start: {traceback.format_exc()}"))
        return

    def search_device(st, queries, qlens, k, thr):
        q = len(qlens)
        d_q = torch.from_numpy(np.ascontiguousarray(queries)).to(dev)
        khi, klo = (torch.empty(q * k, dtype=torch.int64, device=dev) for _ in range(2))
        h, nb = (torch.empty(q * k, dtype=torch.int16, device=dev) for _ in range(2))
        cnt = torch.empty(q, dtype=torch.int32, device=dev)
        torch.cuda.synchronize(dev)   # the upload ran on torch's stream, the search runs on the store's own
        tn, td = (0, 0) if thr is None else thr
        _lib.check(L.isx_search_device(st.handle, d_q.data_ptr(), 1, _lib.ptr(np.ascontiguousarray(qlens)), q, k, tn, td,
                                       khi.data_ptr(), klo.data_ptr(), h.data_ptr(), nb.data_ptr(), cnt.data_ptr(), 1))
        hi = khi.cpu().numpy().view(np.uint64).reshape(q, k)
        keys = hi if st.key_bytes == 8 else synth.keys128_bytes(hi.ravel(), klo.cpu().numpy().view(np.uint64)).reshape(q, k, 16)
        return keys, h.cpu().numpy().view(np.uint16).reshape(q, k), nb.cpu().numpy().view(np.uint16).reshape(q, k), \
            cnt.cpu().numpy().view(np.uint32)

    def run(name, queries, qlens, k, thr, device_queries):
        st = stores[name]
        if device_queries:
            out = search_device(st, queries, qlens, k, thr)
        else:
            out = st.search(queries, qlens, k, thr)[:4]
        return out + (st.stats(),)

    def batch(name, queries, qlens, k, thr=None, gmask=0, device_queries=False, sequenced=False):
        """One armed batch, the protocol of include/isx.h with the host barrier in place of the collectives."""
        st = stores[name]
        _lib.check(L.isx_share_reset(st.handle))
        torch.cuda.synchronize(dev)    # the zeroing is on the store's stream: done before any peer may count here
        barrier.wait()
        _lib.check(L.isx_share_set_lengths(st.handle, gmask))
        if sequenced:                  # rank 0 first, each rank after the previous one has finished
            for r in range(world):
                if r == rank:
                    res = run(name, queries, qlens, k, thr, device_queries)
                barrier.wait()
        else:
            res = run(name, queries, qlens, k, thr, device_queries)
        barrier.wait()                 # the fence of the all-gather: no rank resets while a peer can still count into it
        return res

    def open_store(name, key_bytes, keys, codes, lens, max_bytes=32, fixed_len=0):
        st = _lib.Store(device=dev, key_bytes=key_bytes, max_bytes=max_bytes, fixed_len=fixed_len)
        stores[name] = st
        if len(lens):
            st.add(np.ascontiguousarray(keys), np.ascontiguousarray(codes), np.ascontiguousarray(lens))
        return st.size(), st.length_mask()

    def add(name, keys, codes, lens):
        stores[name].add(np.ascontiguousarray(keys), np.ascontiguousarray(codes), np.ascontiguousarray(lens))
        return stores[name].length_mask()

    def share(name, max_queries):
        handle = (ctypes.c_ubyte * 64)()
        _lib.check(L.isx_share_init(stores[name].handle, world, rank, max_queries, handle))
        return bytes(handle)

    def attach(name, handles):
        for r, hb in enumerate(handles):
            if r != rank:
                _lib.check(L.isx_share_attach(stores[name].handle, r, (ctypes.c_ubyte * 64)(*hb)))

    def search(name, queries, qlens, k, thr=None):
        return run(name, queries, qlens, k, thr, False)

    def match_all(name, query, thr):
        return stores[name].match_all(query, thr)

    def self_join(name, thr):
        return stores[name].self_join(thr)

    handlers = dict(batch=batch, open=open_store, add=add, share=share, attach=attach, search=search, match_all=match_all,
                    self_join=self_join)
    conn.send(("ok", dev))
    try:
        while True:
            msg = conn.recv()
            if msg is None:
                break
            cmd, kw = msg
            try:
                conn.send(("ok", handlers[cmd](**kw)))
            except BaseException:
                conn.send(("err", f"rank {rank}: {cmd}: {traceback.format_exc()}"))
    finally:
        for st in stores.values():
            st.close()


class Ranks:
    """W rank processes on this machine's GPUs (rank r on device r % n), started with spawn: CUDA is live in the parent."""

    def __init__(self, world, env=None):
        ctx = mp.get_context("spawn")
        self.world = world
        self.barrier = ctx.Barrier(world, timeout=BARRIER_S)
        self.procs, self.conns = [], []
        try:
            for r in range(world):
                a, b = ctx.Pipe()
                p = ctx.Process(target=_rank_main, args=(r, world, b, self.barrier, dict(env or {})), daemon=True)
                p.start()
                b.close()
                self.procs.append(p)
                self.conns.append(a)
            self._collect("start")
        except BaseException:
            self.close()
            raise

    def _collect(self, cmd):
        """Replies of all ranks, taken as they arrive: the first error aborts the barrier, so the peers waiting there
        report at once instead of at its timeout."""
        out, errors = [None] * self.world, []
        waiting = dict(zip(self.conns, range(self.world)))
        deadline = time.monotonic() + CALL_S
        while waiting:
            ready = wait(list(waiting), timeout=max(0.0, deadline - time.monotonic()))
            if not ready:
                errors += [f"rank {r}: no reply to {cmd} within {CALL_S} s" for r in waiting.values()]
                self.barrier.abort()
                break
            for c in ready:
                r = waiting.pop(c)
                try:
                    status, val = c.recv()
                except EOFError:
                    status, val = "err", f"rank {r}: process ended during {cmd} (exit code {self.procs[r].exitcode})"
                if status == "err":
                    errors.append(val)
                    self.barrier.abort()    # releases the peers waiting for this rank
                out[r] = val
        if errors:
            self.barrier.reset()
            pytest.fail("\n".join(errors), pytrace=False)
        return out

    def call(self, cmd, per_rank=None, **common):
        """Send `cmd` to every rank (common kwargs plus per_rank[r]) and return the ranks' replies."""
        for r, c in enumerate(self.conns):
            c.send((cmd, dict(common, **(per_rank[r] if per_rank else {}))))
        return self._collect(cmd)

    def close(self):
        for c in self.conns:
            try:
                c.send(None)
            except (OSError, BrokenPipeError):
                pass
        for p in self.procs:
            p.join(timeout=60)
        for p in self.procs:
            if p.is_alive():
                p.terminate()
                p.join(timeout=10)
            if p.is_alive():
                p.kill()
                p.join()
        for c in self.conns:
            c.close()


class Group:
    """A running set of ranks plus the stores each of them opened (name -> Case)."""

    def __init__(self, world, env=None):
        self.ranks = Ranks(world, env)
        self.world = world
        self.cases = {}
        self.masks = {}

    def open(self, name, case, key_bytes=8, max_queries=16384, **kw):
        per = [dict(keys=keys_arg(s), codes=s[2], lens=s[3]) for s in case.shards]
        res = self.ranks.call("open", per, name=name, key_bytes=key_bytes, **kw)
        assert [n for n, _ in res] == [len(s[3]) for s in case.shards]
        self.masks[name] = [m for _, m in res]
        handles = self.ranks.call("share", name=name, max_queries=max_queries)
        self.ranks.call("attach", name=name, handles=handles)
        self.cases[name] = case

    def gmask(self, name):
        m = 0
        for x in self.masks[name]:
            m |= x
        return m

    def batch(self, name, queries, qlens, k, thr=None, **kw):
        return self.ranks.call("batch", name=name, queries=queries, qlens=qlens, k=k, thr=thr, gmask=self.gmask(name), **kw)

    def search(self, name, queries, qlens, k, thr=None):
        return self.ranks.call("search", name=name, queries=queries, qlens=qlens, k=k, thr=thr)

    def checked(self, name, queries, qlens, k, thr=None, **kw):
        """An armed batch, merged and compared with the oracle over the union; -> the ranks' stats."""
        res = self.batch(name, queries, qlens, k, thr, **kw)
        check_merged(self.cases[name], [r[:4] for r in res], queries, qlens, k, thr)
        return [r[4] for r in res]

    def close(self):
        self.ranks.close()


def probe_queries(P, q):
    return np.repeat(P[None, :], q, axis=0), np.full(q, 32, dtype=np.uint8)


def assert_probe(stats, q, n1, shared, ranks):
    """
    Candidates of the probe ranks. Unshared, a rank's own counts never take its threshold below D, so it emits all its
    Q * N1 rows at D. Shared, the first re-derivation reads rank 0's k counts at distance 0, so at most the rows at D of
    the first warm-up range, Q * N1 / 8, are emitted; Q * N1 / 4 is asserted. Observed on a B200 (1000 W): exactly Q * N1 / 8
    on every probe rank, 8 192 of 65 536 at world 2 and 2 048 of 16 384 at world 8.
    Probe rows are sparse on purpose: a CTA stages at most 1024 records per item, and past that only 32 re-derivations
    per flush are noted, so a probe whose every row passes keeps most queries' thresholds loose for many items (a dense
    probe, every row at D, emitted 13 336 576 of 16 777 216 at world 2 with sharing on).
    """
    for r in ranks:
        c = stats[r]["candidates"]
        if shared:
            assert c <= q * n1 // 4, f"rank {r}: {c} candidates of {q * n1} rows at D: peer counts did not tighten the threshold"
        else:
            assert c >= q * n1, f"rank {r}: {c} candidates < {q * n1}: some rows at D were not emitted"


# ---- world 2: owner split of mixed rows, default knobs -----------------------------------------------------------------
N2 = 400_000


@pytest.fixture(scope="module")
def w2(cuda):
    g = Group(2)
    try:
        keys, codes, lens = prefix_planted(N2, 41, 200)
        g.open("mix", split(keys, codes, lens, owner_of(keys, 2), 2))
        case, g.P = probe_case(2, probe_rows(2), seed=2)
        g.open("probe", case)
        yield g
    finally:
        g.close()


def test_w2_tensor_core_tiles_device_queries(w2):
    q, ql = mixed_queries(96, N2, 1, 41)
    stats = w2.checked("mix", q, ql, K, device_queries=True)
    assert all(s["issued_popc"] == 0 for s in stats), "every tile of >= 64 queries runs on the tensor cores"


def test_w2_popc_tiles(w2):
    q, ql = mixed_queries(20, N2, 2, 41)
    stats = w2.checked("mix", q, ql, K)
    assert all(s["issued_popc"] > 0 for s in stats), "tiles of < 64 queries run k_scan"


def test_w2_small_path_then_armed_batch(w2):
    q, ql = mixed_queries(1, N2, 3, 41, lengths=(8, 16, 32))
    stats = w2.checked("mix", q, ql, 10)
    assert all(s["kernel_launches"] == 1 for s in stats), "a request of <= 4 queries is one launch of the small path"
    q, ql = mixed_queries(64, N2, 4, 41)
    w2.checked("mix", q, ql, K)


def test_w2_threshold_mode(w2):
    q, ql = mixed_queries(64, N2, 5, 41)
    w2.checked("mix", q, ql, K, thr=(1, 8))


@pytest.mark.parametrize("k", [1, 100, "sort_cap+1"])
def test_w2_counts(w2, k):
    import torch

    from tests.test_gpu_select_edges import max_sort_cap

    if k == "sort_cap+1":
        k = max_sort_cap(torch.cuda.get_device_properties(0).shared_memory_per_block_optin, 8) + 1
    q, ql = mixed_queries(64, N2, 6, 41)
    w2.checked("mix", q, ql, k)


def test_w2_unarmed_calls_between_armed_batches(w2):
    case = w2.cases["mix"]
    q, ql = mixed_queries(64, N2, 7, 41)
    w2.checked("mix", q, ql, K)
    # unarmed on both ranks: each rank's own top-k, not a share of the merged one
    for r, res in enumerate(w2.search("mix", q, ql, K)):
        s = case.shards[r]
        rows, h, nb, cnt = oracle_topk(s[0], s[2], s[3], q, ql, K)
        assert_same_topk(*res[:4], s[0], rows, h, nb, cnt)
    query = bytes(q[0, : ql[0]])
    for r, (gk, gh, gn) in enumerate(w2.ranks.call("match_all", name="mix", query=query, thr=(1, 4))):
        s = case.shards[r]
        rows, h, nb, cnt = oracle_topk(s[0], s[2], s[3], q[:1], ql[:1], len(s[3]), (1, 4))
        exp = sorted(zip(s[0][rows[0, : cnt[0]]].tolist(), h[0, : cnt[0]].tolist(), nb[0, : cnt[0]].tolist()))
        assert sorted(zip(gk.tolist(), gh.tolist(), gn.tolist())) == exp
    for r, (ka, kb, h, nb) in enumerate(w2.ranks.call("self_join", name="mix", thr=(0, 1))):
        s = case.shards[r]
        exp = prefix_pairs(s[0], s[2], s[3])
        assert len(exp) > 20
        assert list(zip(ka.tolist(), kb.tolist(), nb.tolist())) == exp and not h.any()
    w2.checked("mix", q, ql, K)


def test_w2_probe_peer_counts_reach_the_kernels(w2):
    n1, Q = probe_n1(2), 64
    q, ql = probe_queries(w2.P, Q)
    stats = w2.checked("probe", q, ql, K, sequenced=True)
    assert_probe(stats, Q, n1, True, [1])
    res = w2.search("probe", q, ql, K)
    check_merged(w2.cases["probe"], [r[:4] for r in res], q, ql, K)
    assert_probe([r[4] for r in res], Q, n1, False, [1])


RESCAN_ROWS = 12 << 20   # > 3 first waves of the POPC scan (444 CTAs x one 8-block item = 3.6 M rows)


def test_w2_overflow_rescan_repeats_when_the_local_histogram_under_counts(w2):
    """
    The grow-and-repeat loop of the exact re-scan (csrc/isx.cu), which only sharing needs. Rank 0 holds K copies of P,
    rank 1 holds 12 M rows, each 1 bit from P. 8 queries (one POPC tile, no warm-up ranges) are searched on rank 1 after
    rank 0. Its first items emit every row, far more than the candidate list holds. Their flushes read rank 0's K counts at
    distance 0, and the threshold drops below distance 1, so later rows are skipped. The overflowed query's local histogram
    thus counts fewer rows within d* than the shard holds. The first re-scan, sized from that count, overflows again, and
    the second one, sized from what the first saw, completes. Unarmed, the local count is exact and one re-scan suffices.
    """
    rng = np.random.default_rng(21)
    P = rng.integers(0, 256, 32, dtype=np.uint8)
    near = np.repeat(P[None, :], RESCAN_ROWS, axis=0)
    flip = np.arange(RESCAN_ROWS) % 256
    near[np.arange(RESCAN_ROWS), flip // 8] ^= (1 << (flip % 8)).astype(np.uint8)
    lens = np.full(RESCAN_ROWS, 32, dtype=np.uint8)
    case = Case([(synth.make_keys(0, K, 23), None, np.repeat(P[None, :], K, axis=0), lens[:K]),
                 (synth.make_keys(K, RESCAN_ROWS, 23), None, near, lens)])
    w2.open("rescan", case)
    q, ql = probe_queries(P, 8)
    armed = w2.batch("rescan", q, ql, K, sequenced=True)
    check_merged(case, [r[:4] for r in armed], q, ql, K)
    unarmed = w2.search("rescan", q, ql, K)
    check_merged(case, [r[:4] for r in unarmed], q, ql, K)
    # rank 1's own list is its exact local top-k in both runs, the K smallest keys at h = 1: the repeated re-scan
    # truncated nothing
    keys1 = case.shards[1][0]
    exp = np.sort(keys1)[:K]
    for res in (armed[1], unarmed[1]):
        assert (res[3] == K).all() and (res[1] == 1).all() and (res[0] == exp[None, :]).all()
    a, u = armed[1][4], unarmed[1][4]
    assert a["issued_popc"] > 0 and u["passes"] == a["passes"] == 1
    assert a["fallback_queries"] == u["fallback_queries"] == 8
    assert a["candidates"] < u["candidates"] == 8 * RESCAN_ROWS, "the shared threshold skipped some rows at distance 1"
    # unarmed: init + scan + select per re-scanned query once; armed: at least one query repeats them
    assert a["kernel_launches"] > u["kernel_launches"], (a["kernel_launches"], u["kernel_launches"])


def test_w2_mass_duplicates_overflow_rescan_while_shared(w2):
    """Last in the group: it adds rows. 45 000 copies of one code per rank overflow every rank's candidate list."""
    dup_n = 45_000 * 2
    dup_keys = synth.make_keys(2 * 10**9, dup_n, 77)
    dup_codes = np.zeros((dup_n, 32), dtype=np.uint8)
    dup_codes[:, :16] = 0xA7
    dup_lens = np.full(dup_n, 16, dtype=np.uint8)
    own = owner_of(dup_keys, 2)
    w2.masks["mix"] = w2.ranks.call("add", [dict(keys=dup_keys[own == r], codes=dup_codes[own == r], lens=dup_lens[own == r])
                                            for r in range(2)], name="mix")
    old = w2.cases["mix"]
    w2.cases["mix"] = Case([(np.concatenate([s[0], dup_keys[own == r]]), None, np.concatenate([s[2], dup_codes[own == r]]),
                             np.concatenate([s[3], dup_lens[own == r]])) for r, s in enumerate(old.shards)])
    q, ql = mixed_queries(63, N2, 8, 41, lengths=(16,))
    q, ql = np.concatenate([dup_codes[:1], q]), np.concatenate([dup_lens[:1], ql])
    stats = w2.checked("mix", q, ql, K)
    # one tile of 64 queries (the tensor-core scan); the re-scans' own POPC launches count in issued_popc
    assert all(s["fallback_queries"] >= 1 and s["passes"] == 1 for s in stats)


# ---- world 3: skewed shards, both cut-offs of sharing -----------------------------------------------------------------
N3 = 150_000
MAXQ3 = 300


@pytest.fixture(scope="module")
def w3(cuda):
    g = Group(3)
    try:
        g.open("few", skew_case(N3, 43, 3, 37), max_queries=MAXQ3)
        g.open("empty", skew_case(N3, 43, 3, 0), max_queries=MAXQ3)
        lo, hi = cut_lengths()
        for name, lengths in (("cut_lo", lo), ("cut_hi", hi)):
            case, g.P = probe_case(3, probe_rows(3), seed=3, extra_lengths=[L for L in lengths if L != 32])
            g.open(name, case, max_queries=MAXQ3)
        yield g
    finally:
        g.close()


@pytest.mark.parametrize("q", [MAXQ3, MAXQ3 + 1])
@pytest.mark.parametrize("name", ["few", "empty"])
def test_w3_skewed_shards(w3, name, q):
    assert len(set(w3.masks[name])) == 3, "every rank stores a different set of lengths"
    assert w3.cases[name].shards[1][3].size < K
    queries, qlens = mixed_queries(MAXQ3 // 4, N3, 11, 43)
    queries, qlens = queries[:q], qlens[:q]
    if q > MAXQ3:
        extra = synth.make_queries(1, N3, 12, 43, lengths=(16,))
        queries, qlens = np.concatenate([queries, extra[0]]), np.concatenate([qlens, extra[1]])
    stats = w3.checked(name, queries, qlens, K)
    assert all(s["issued_popc"] == 0 for s in stats), "75 or 76 queries per length: every tile on the tensor cores"


@pytest.mark.parametrize("name,q,shared", [("cut_lo", MAXQ3, True), ("cut_lo", MAXQ3 + 1, False), ("cut_hi", MAXQ3, False)])
def test_w3_probe_cutoffs(w3, name, q, shared):
    lo, hi = cut_lengths()
    assert rank_count(lo) <= SHARE_RCAP < rank_count(hi)
    n1 = probe_n1(3)
    queries, qlens = probe_queries(w3.P, q)
    stats = w3.checked(name, queries, qlens, K, sequenced=True)
    assert_probe(stats, q, n1, shared, [1, 2])   # the decision is the same on both probe ranks


def test_w3_probe_unarmed_replay(w3):
    n1, q = probe_n1(3), MAXQ3
    queries, qlens = probe_queries(w3.P, q)
    res = w3.search("cut_lo", queries, qlens, K)
    check_merged(w3.cases["cut_lo"], [r[:4] for r in res], queries, qlens, K)
    assert_probe([r[4] for r in res], q, n1, False, [1, 2])


# ---- world 4: many small tiles in flight on four lanes ------------------------------------------------------------------
N4 = 200_000


@pytest.fixture(scope="module")
def w4(cuda):
    g = Group(4, env={"ISX_MAX_TILE": "64", "ISX_TILE_LANES": "4"})
    try:
        keys, codes, lens = make_store_arrays(N4, 44)
        g.open("mix", split(keys, codes, lens, owner_of(keys, 4), 4))
        yield g
    finally:
        g.close()


def test_w4_many_tiles_then_permuted_batch(w4):
    q, ql = mixed_queries(512, N4, 12, 44)   # 8 tiles of 64 per length, all on the tensor cores
    stats = w4.checked("mix", q, ql, K)
    assert all(s["passes"] == 32 and s["issued_popc"] == 0 for s in stats)
    perm = np.random.default_rng(13).permutation(len(ql))
    w4.checked("mix", np.ascontiguousarray(q[perm]), np.ascontiguousarray(ql[perm]), K)


# ---- world 8: 16-byte keys on a fixed-length store (cfg4 shape at test size) ----------------------------------------------
N8 = 1_000_000


@pytest.fixture(scope="module")
def w8(cuda):
    from oracle import c_oracle

    g = Group(8)
    try:
        hi, lo, codes, lens = c_oracle.synth_rows(0, N8, 48, lengths=(8,), key_mode=1, cpa=64, dup_every=16, dup_back=5)
        g.open("simprint", split(hi, codes, lens, owner_of(hi ^ lo, 8), 8, lo=lo), key_bytes=16, max_bytes=8, fixed_len=8)
        case, g.P = probe_case(8, probe_rows(8), seed=8)
        g.open("probe", case)
        yield g
    finally:
        g.close()


@pytest.mark.parametrize("bits,k", [(16, 4000), (0, 1000)])
def test_w8_keys16_threshold(w8, bits, k):
    q, ql = synth.make_queries(64, N8, 14, 48, lengths=(8,), row_lengths=(8,), mixed_rows=False)
    stats = w8.checked("simprint", q, ql, k, thr=(bits, 64))
    assert all(s["issued_popc"] == 0 and s["passes"] == 1 and s["fallback_queries"] == 0 for s in stats)


def test_w8_probe_peer_counts_reach_the_kernels(w8):
    n1, Q = probe_n1(8), 64
    q, ql = probe_queries(w8.P, Q)
    stats = w8.checked("probe", q, ql, K, sequenced=True)
    assert_probe(stats, Q, n1, True, range(1, 8))
