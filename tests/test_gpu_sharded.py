"""
Multi-shard path: (1) single-GPU emulation - S stores on one device searched separately, their packed
record buffers concatenated exactly as an all-gather delivers them, merged by `isx_merge_device`;
(2) real 2-rank NCCL run when the box has >= 2 GPUs. The merged result must be byte-identical to
the un-sharded oracle (result independent of the shard count, SURVEY.md 8e).
"""

import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from iscc_search_b200 import _lib, synth
from iscc_search_b200.sharded import ShardedSearcher, owner_of, record_layout
from tests.helpers import assert_same_topk, make_store_arrays, oracle_topk

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent


@pytest.mark.parametrize("shards", [2, 3, 8])
def test_emulated_shards_merge_equals_unsharded_oracle(cuda, shards):
    import torch

    n, q, k = 150_000, 96, 100
    keys, codes, lens = make_store_arrays(n, 21)
    queries, qlens = synth.make_queries(q, n, 22, 21)
    own = owner_of(keys, shards)
    stores = []
    for r in range(shards):
        st = _lib.Store(key_bytes=8, max_bytes=32)
        sel = own == r
        st.add(np.ascontiguousarray(keys[sel]), np.ascontiguousarray(codes[sel]), np.ascontiguousarray(lens[sel]))
        stores.append(st)
    assert sum(st.size() for st in stores) == n
    dev = torch.device("cuda", 0)
    d_q = torch.from_numpy(queries).to(dev)
    off, size = record_layout(q, k)
    gathered = torch.zeros(size * shards, dtype=torch.uint8, device=dev)
    for r, st in enumerate(stores):
        buf, _, _ = ShardedSearcher(st, r, 1, None, dev).search_device(d_q, qlens, k)
        torch.cuda.synchronize()
        gathered[r * size:(r + 1) * size] = buf[:size]
    merged = torch.zeros(size, dtype=torch.uint8, device=dev)
    g0, m0 = gathered.data_ptr(), merged.data_ptr()
    st0 = stores[0]
    st0.set_stream(torch.cuda.current_stream(dev).cuda_stream)
    _lib.check(_lib.lib().isx_merge_device(st0.handle, shards, q, k, size, g0 + off["khi"], g0 + off["klo"], g0 + off["h"],
                                           g0 + off["n"], g0 + off["cnt"], m0 + off["khi"], m0 + off["klo"], m0 + off["h"],
                                           m0 + off["n"], m0 + off["cnt"], 1))
    raw = merged.cpu().numpy()
    qk = q * k
    gk = raw[off["khi"]: off["khi"] + qk * 8].view(np.uint64).reshape(q, k)
    gh = raw[off["h"]: off["h"] + qk * 2].view(np.uint16).reshape(q, k)
    gn = raw[off["n"]: off["n"] + qk * 2].view(np.uint16).reshape(q, k)
    gc = raw[off["cnt"]: off["cnt"] + q * 4].view(np.uint32)
    rows, h, nb, cnt = oracle_topk(keys, codes, lens, queries, qlens, k)
    assert_same_topk(gk, gh, gn, gc, keys, rows, h, nb, cnt)
    for st in stores:
        st.close()


def test_emulated_shards_with_fewer_rows_than_k(cuda):
    import torch

    n, q, k, shards = 37, 6, 50, 4
    keys, codes, lens = make_store_arrays(n, 5)
    queries, qlens = synth.make_queries(q, n, 6, 5)
    own = owner_of(keys, shards)
    dev = torch.device("cuda", 0)
    d_q = torch.from_numpy(queries).to(dev)
    off, size = record_layout(q, k)
    gathered = torch.zeros(size * shards, dtype=torch.uint8, device=dev)
    stores = []
    for r in range(shards):
        st = _lib.Store(key_bytes=8, max_bytes=32)
        sel = own == r
        if sel.any():
            st.add(np.ascontiguousarray(keys[sel]), np.ascontiguousarray(codes[sel]), np.ascontiguousarray(lens[sel]))
        buf, _, _ = ShardedSearcher(st, r, 1, None, dev).search_device(d_q, qlens, k)
        torch.cuda.synchronize()
        gathered[r * size:(r + 1) * size] = buf[:size]
        stores.append(st)
    merged = torch.zeros(size, dtype=torch.uint8, device=dev)
    g0, m0 = gathered.data_ptr(), merged.data_ptr()
    _lib.check(_lib.lib().isx_merge_device(stores[0].handle, shards, q, k, size, g0 + off["khi"], g0 + off["klo"], g0 + off["h"],
                                           g0 + off["n"], g0 + off["cnt"], m0 + off["khi"], m0 + off["klo"], m0 + off["h"],
                                           m0 + off["n"], m0 + off["cnt"], 1))
    raw = merged.cpu().numpy()
    qk = q * k
    gk = raw[off["khi"]: off["khi"] + qk * 8].view(np.uint64).reshape(q, k)
    gh = raw[off["h"]: off["h"] + qk * 2].view(np.uint16).reshape(q, k)
    gn = raw[off["n"]: off["n"] + qk * 2].view(np.uint16).reshape(q, k)
    gc = raw[off["cnt"]: off["cnt"] + q * 4].view(np.uint32)
    rows, h, nb, cnt = oracle_topk(keys, codes, lens, queries, qlens, k, use_c=False)
    assert (gc == n).all()
    assert_same_topk(gk, gh, gn, gc, keys, rows, h, nb, cnt)
    for st in stores:
        st.close()


def _n_gpus():
    import ctypes

    n = ctypes.c_int()
    return n.value if _lib.lib().isx_device_count(ctypes.byref(n)) == 0 else 0


@pytest.mark.parametrize("world", [2, 4, 8])
def test_multi_rank_nccl_search_with_shared_thresholds_equals_oracle(cuda, tmp_path, world):
    if _n_gpus() < world:
        pytest.skip(f"needs {world} GPUs on one machine")
    out = tmp_path / "result.npz"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(29533 + world), str(ROOT / "tests" / "sharded_worker.py"), "--backend", "nccl", "--out", str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=str(ROOT), env=dict(os.environ))
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    d = np.load(out)
    n, q, k = int(d["n"]), int(d["q"]), int(d["k"])
    assert bool(d["shared"]), "threshold sharing over peer memory was not active"
    keys, codes, lens = make_store_arrays(n, 31)
    queries, qlens = synth.make_queries(q, n, 32, 31)
    rows, h, nb, cnt = oracle_topk(keys, codes, lens, queries, qlens, k)
    # two batches were searched back to back (reset/fence protocol of the shared histograms): both must be exact
    assert_same_topk(d["keys"], d["h"], d["nb"], d["cnt"], keys, rows, h, nb, cnt)
    assert_same_topk(d["keys2"], d["h2"], d["nb2"], d["cnt2"], keys, rows, h, nb, cnt)
    # >= 64 queries per length: the tensor-core scan with shared thresholds
    tc = [synth.make_queries(80, n, 40 + L, 31, lengths=(L,)) for L in synth.STANDARD_LENGTHS]
    qtc, qltc = np.concatenate([t[0] for t in tc]), np.concatenate([t[1] for t in tc])
    assert int(d["popc_tc"]) == 0, "every tile of the batch was meant to run on the tensor cores"
    rows_tc, h_tc, nb_tc, cnt_tc = oracle_topk(keys, codes, lens, qtc, qltc, k)
    assert_same_topk(d["keys_tc"], d["h_tc"], d["nb_tc"], d["cnt_tc"], keys, rows_tc, h_tc, nb_tc, cnt_tc)
    # third batch: mass duplicates -> candidate overflow + exact re-scan on every rank, thresholds still shared
    dd = np.load(str(out).replace(".npz", "_dup.npz"))
    dup_n = int(dd["dup_n"])
    assert int(dd["fallback"]) >= 1
    dup_keys = synth.make_keys(10**9, dup_n, 77)
    dup_codes = np.zeros((dup_n, 32), dtype=np.uint8)
    dup_codes[:, :16] = 0xA7
    all_keys = np.concatenate([keys, dup_keys])
    all_codes = np.concatenate([codes, dup_codes])
    all_lens = np.concatenate([lens, np.full(dup_n, 16, dtype=np.uint8)])
    q3 = np.concatenate([dup_codes[:1], queries[:7]])
    ql3 = np.concatenate([np.array([16], dtype=np.uint8), qlens[:7]])
    rows3, h3, nb3, cnt3 = oracle_topk(all_keys, all_codes, all_lens, q3, ql3, k)
    assert_same_topk(dd["keys"], dd["h"], dd["nb"], dd["cnt"], all_keys, rows3, h3, nb3, cnt3)
    # fourth batch: shards with different length buckets (ADVICE r1: rank tables must come from the global class mask)
    ds = np.load(str(out).replace(".npz", "_skew.npz"))
    assert bool(ds["shared"])
    assert len(set(ds["masks"].tolist())) > 1, "the shards were meant to hold different length buckets"
    assert_same_topk(ds["keys"], ds["h"], ds["nb"], ds["cnt"], keys, rows, h, nb, cnt)
