"""torchrun worker for the N>1 tests: gloo (CPU: layout + collective plumbing only) or nccl (real sharded search)."""
import argparse
import os
import sys
from pathlib import Path

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from iscc_search_b200 import synth  # noqa: E402
from iscc_search_b200.sharded import owner_of, record_layout  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--backend", default="gloo")
ap.add_argument("--out", required=True)
args = ap.parse_args()
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])

if args.backend == "nccl":
    from iscc_search_b200 import _lib
    from iscc_search_b200.sharded import ShardedSearcher
    from tests.helpers import make_store_arrays

    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
    n, q, k = 400_000, 128, 100
    keys, codes, lens = make_store_arrays(n, 31)
    queries, qlens = synth.make_queries(q, n, 32, 31)
    sel = owner_of(keys, world) == rank
    st = _lib.Store(device=rank, key_bytes=8, max_bytes=32)
    st.add(np.ascontiguousarray(keys[sel]), np.ascontiguousarray(codes[sel]), np.ascontiguousarray(lens[sel]))
    searcher = ShardedSearcher(st, rank, world, None, torch.device("cuda", rank))
    gk, gh, gn, gc = (a.copy() for a in searcher.search(queries, qlens, k))
    # a second batch right behind the first: different query order, exercises the reset -> barrier -> search protocol
    perm = np.random.default_rng(7).permutation(q)
    gk2, gh2, gn2, gc2 = (a.copy() for a in searcher.search(np.ascontiguousarray(queries[perm]), np.ascontiguousarray(qlens[perm]), k))
    inv = np.argsort(perm)
    # 80 queries of every length: every tile has >= 64 queries, so the shared thresholds run through k_scan_tc
    tc = [synth.make_queries(80, n, 40 + L, 31, lengths=(L,)) for L in synth.STANDARD_LENGTHS]
    qtc, qltc = np.concatenate([t[0] for t in tc]), np.concatenate([t[1] for t in tc])
    gktc, ghtc, gntc, gctc = (a.copy() for a in searcher.search(qtc, qltc, k))
    popc_tc = st.stats()["issued_popc"]
    # third batch: 150K extra rows sharing ONE code -> every rank's candidate buffer overflows for that query and the
    # exact re-scan path runs while thresholds are shared; the merged result must be the 100 smallest keys among the ties
    dup_n = 45_000 * world   # > the candidate buffer (32768) on every rank
    dup_keys = synth.make_keys(10**9, dup_n, 77)
    dup_codes = np.zeros((dup_n, 32), dtype=np.uint8)
    dup_codes[:, :16] = 0xA7
    dup_lens = np.full(dup_n, 16, dtype=np.uint8)
    dsel = owner_of(dup_keys, world) == rank
    st.add(np.ascontiguousarray(dup_keys[dsel]), np.ascontiguousarray(dup_codes[dsel]), np.ascontiguousarray(dup_lens[dsel]))
    q3 = np.concatenate([dup_codes[:1], queries[:7]])
    ql3 = np.concatenate([dup_lens[:1], qlens[:7]])
    gk3, gh3, gn3, gc3 = (a.copy() for a in searcher.search(q3, ql3, k))
    fb = st.stats()["fallback_queries"]
    if rank == 0:
        np.savez(args.out.replace(".npz", "_dup.npz"), keys=gk3, h=gh3, nb=gn3, cnt=gc3, fallback=fb, dup_n=dup_n)
    # fourth batch, fresh stores whose shards hold DIFFERENT length buckets (192-bit rows only on rank 0, 128-bit rows
    # only on the last rank): the rank tables must still agree across ranks (global class mask), else the shared
    # histograms are indexed inconsistently and true neighbours are dropped
    st4 = _lib.Store(device=rank, key_bytes=8, max_bytes=32)
    own = owner_of(keys, world)
    own[lens == 24] = 0
    own[lens == 16] = world - 1
    sel4 = own == rank
    st4.add(np.ascontiguousarray(keys[sel4]), np.ascontiguousarray(codes[sel4]), np.ascontiguousarray(lens[sel4]))
    masks = [None] * world
    dist.all_gather_object(masks, st4.length_mask())
    s4 = ShardedSearcher(st4, rank, world, None, torch.device("cuda", rank))
    gk4, gh4, gn4, gc4 = (a.copy() for a in s4.search(queries, qlens, k))
    if rank == 0:
        np.savez(args.out.replace(".npz", "_skew.npz"), keys=gk4, h=gh4, nb=gn4, cnt=gc4, masks=np.array(masks, dtype=np.int64),
                 shared=s4.shared)
    if rank == 0:
        np.savez(args.out, keys=gk, h=gh, nb=gn, cnt=gc, keys2=gk2[inv], h2=gh2[inv], nb2=gn2[inv], cnt2=gc2[inv], n=n, q=q, k=k,
                 shared=searcher.shared, keys_tc=gktc, h_tc=ghtc, nb_tc=gntc, cnt_tc=gctc, popc_tc=popc_tc)
    dist.barrier()
    dist.destroy_process_group()
else:
    # CPU: every rank packs a deterministic fake record buffer; the all-gather must deliver them in
    # rank order with the stride `record_layout` promises (what isx_merge_device indexes by).
    dist.init_process_group("gloo")
    q, k = 5, 7
    off, size = record_layout(q, k)
    local = torch.zeros(size, dtype=torch.uint8)
    raw = local.numpy()
    raw[off["khi"]: off["khi"] + q * k * 8].view(np.uint64)[:] = np.arange(q * k, dtype=np.uint64) * 10 + rank
    raw[off["h"]: off["h"] + q * k * 2].view(np.uint16)[:] = rank + 1
    raw[off["n"]: off["n"] + q * k * 2].view(np.uint16)[:] = 64
    raw[off["cnt"]: off["cnt"] + q * 4].view(np.uint32)[:] = k - rank
    gathered = torch.zeros(size * world, dtype=torch.uint8)
    dist.all_gather_into_tensor(gathered, local)
    # stored-length masks differ per rank (rank r holds codes of 8*(r+1) bytes, rank 0 also 5-byte codes): every rank
    # must come out with the union
    from iscc_search_b200.sharded import global_length_mask

    local_mask = (1 << (8 * (rank + 1) - 1)) | ((1 << 4) if rank == 0 else 0)
    gmask = global_length_mask(local_mask, dist)
    all_masks = [None] * world
    dist.all_gather_object(all_masks, gmask)
    if rank == 0:
        np.savez(args.out, gathered=gathered.numpy(), size=size, world=world, q=q, k=k, gmasks=np.array(all_masks, dtype=np.int64))
    dist.barrier()
    dist.destroy_process_group()
