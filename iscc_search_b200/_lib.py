"""
ctypes binding of libisx_b200.so (C ABI declared in include/isx.h).

There is deliberately NO fallback: if the shared library is missing or no B200 is visible, every
entry point raises. The product path never imports anything from `oracle/`.
"""

import ctypes
import os
import subprocess
from pathlib import Path

import numpy as np

_PKG = Path(__file__).resolve().parent
SO_PATH = Path(os.environ["ISX_LIB_PATH"]).resolve() if os.environ.get("ISX_LIB_PATH") else _PKG / "libisx_b200.so"  # override: A/B of builds
CSRC = _PKG / "csrc"

ISX_EINVAL, ISX_ECUDA, ISX_ENOMEM, ISX_EIO, ISX_ELIMIT = -1, -2, -3, -4, -5


class IsxError(RuntimeError):
    """CUDA / allocation / IO failure inside libisx_b200."""


class IsxStats(ctypes.Structure):
    _fields_ = [
        ("kernel_launches", ctypes.c_uint64),
        ("scan_launches", ctypes.c_uint64),
        ("scan_ms", ctypes.c_float),
        ("select_ms", ctypes.c_float),
        ("total_ms", ctypes.c_float),
        ("pairs", ctypes.c_uint64),
        ("algo_bytes", ctypes.c_uint64),
        ("algo_popc", ctypes.c_uint64),
        ("candidates", ctypes.c_uint64),
        ("fallback_queries", ctypes.c_uint64),
        ("passes", ctypes.c_uint64),
        ("issued_popc", ctypes.c_uint64),
    ]

    def as_dict(self):
        return {name: getattr(self, name) for name, _ in self._fields_}


_lib = None

# every symbol include/isx.h declares (tests check the .so exports all of them)
SYMBOLS = (
    "isx_last_error", "isx_abi_version", "isx_device_count", "isx_open", "isx_close", "isx_set_stream",
    "isx_set_profiling", "isx_get_stats", "isx_add", "isx_add_device", "isx_synth_rows_device", "isx_remove", "isx_contains", "isx_get", "isx_size",
    "isx_clear", "isx_release_scratch", "isx_device_bytes", "isx_length_mask", "isx_save", "isx_load", "isx_search",
    "isx_search_device", "isx_merge_device", "isx_max_k", "isx_match_all", "isx_self_join", "isx_join_fetch", "isx_score_segments", "isx_share_init", "isx_share_attach",
    "isx_share_reset", "isx_share_set_lengths", "isx_selftest_rank_table", "isx_selftest_keymap", "isx_selftest_distance",
)


def build(force=False):
    # type: (bool) -> Path
    """Compile csrc/ for sm_100a with nvcc (in-tree, so the .so ships with the repo snapshot)."""
    srcs = [CSRC / "isx.cu", CSRC / "kernels.cuh", CSRC / "small.cuh", CSRC / "tc.cuh", CSRC / "join.cuh", CSRC / "keymap.hpp", _PKG.parent / "include" / "isx.h"]
    stale = not SO_PATH.exists() or any(p.stat().st_mtime > SO_PATH.stat().st_mtime for p in srcs)
    if force or stale:
        r = subprocess.run(["make", "-C", str(CSRC)], capture_output=True, text=True)
        if r.returncode != 0:
            raise IsxError("building libisx_b200.so failed:\n" + r.stdout + r.stderr)
    return SO_PATH


def lib():
    """Load the shared library (once). Raises IsxError when it is not built - no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not SO_PATH.exists():
        raise IsxError(
            f"{SO_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). iscc_search_b200 has no CPU fallback."
        )
    L = ctypes.CDLL(str(SO_PATH))
    vp, cp = ctypes.c_void_p, ctypes.c_char_p
    u32, u64, sz, ci = ctypes.c_uint32, ctypes.c_uint64, ctypes.c_size_t, ctypes.c_int
    P = ctypes.POINTER
    L.isx_last_error.restype = cp
    L.isx_last_error.argtypes = []
    L.isx_abi_version.restype = ci
    L.isx_device_count.argtypes = [P(ci)]
    L.isx_open.argtypes = [P(vp), ci, u32, u32, u32]
    L.isx_close.argtypes = [vp]
    L.isx_set_stream.argtypes = [vp, vp]
    L.isx_set_profiling.argtypes = [vp, ci]
    L.isx_get_stats.argtypes = [vp, P(IsxStats)]
    L.isx_add.argtypes = [vp, vp, vp, vp, sz, vp]
    L.isx_remove.argtypes = [vp, vp, sz, vp, P(u64)]
    L.isx_add_device.argtypes = [vp, vp, vp, vp, u32, sz]
    L.isx_synth_rows_device.argtypes = [vp, u64, u64, sz, vp, u32, u32, u32, u32, u32, vp, vp, vp]
    L.isx_contains.argtypes = [vp, vp, sz, vp]
    L.isx_get.argtypes = [vp, vp, sz, vp, vp]
    L.isx_size.argtypes = [vp, P(u64)]
    L.isx_clear.argtypes = [vp]
    L.isx_device_bytes.argtypes = [vp, P(u64)]
    L.isx_release_scratch.argtypes = [vp, P(u64)]
    L.isx_length_mask.argtypes = [vp, P(u32)]
    L.isx_save.argtypes = [vp, cp]
    L.isx_load.argtypes = [vp, cp]
    L.isx_search.argtypes = [vp, vp, vp, sz, u32, u32, u32, vp, vp, vp, vp, vp, vp]
    L.isx_search_device.argtypes = [vp, vp, ci, vp, sz, u32, u32, u32, vp, vp, vp, vp, vp, ci]
    L.isx_merge_device.argtypes = [vp, u32, sz, u32, sz, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, ci]
    L.isx_max_k.argtypes = [vp, P(u32)]
    L.isx_match_all.argtypes = [vp, vp, u32, u32, u32, sz, vp, vp, vp, P(u64)]
    L.isx_self_join.argtypes = [vp, u32, u32, P(u64)]
    L.isx_join_fetch.argtypes = [vp, u64, sz, vp, vp, vp, vp]
    L.isx_score_segments.argtypes = [vp, vp, sz, vp, vp, vp, sz, vp, u32, vp]
    L.isx_share_init.argtypes = [vp, u32, u32, u32, vp]
    L.isx_share_attach.argtypes = [vp, u32, vp]
    L.isx_share_reset.argtypes = [vp]
    L.isx_share_set_lengths.argtypes = [vp, u32]
    L.isx_selftest_rank_table.argtypes = [u32, vp, vp, u32, P(u32)]
    L.isx_selftest_keymap.argtypes = [u64, u64, u32]
    L.isx_selftest_distance.argtypes = [u64, u64]
    for name in SYMBOLS:
        if name != "isx_last_error":
            getattr(L, name).restype = ci
    if L.isx_abi_version() != 1:
        raise IsxError("libisx_b200.so ABI version mismatch")
    _lib = L
    return L


def check(rc):
    # type: (int) -> None
    """Map a negative return code to the exception class the reference's callers expect."""
    if rc == 0:
        return
    msg = lib().isx_last_error().decode("utf-8", "replace")
    if rc in (ISX_EINVAL, ISX_ELIMIT):
        raise ValueError(msg)
    if rc == ISX_ENOMEM:
        raise MemoryError(msg)
    if rc == ISX_EIO:
        raise OSError(msg)
    raise IsxError(msg)


def ptr(a):
    # type: (np.ndarray|None) -> int|None
    return None if a is None else a.ctypes.data


class Store:
    """Thin owner of one `isx_store_t*` (one device, this process)."""

    def __init__(self, device=0, key_bytes=8, max_bytes=32, fixed_len=0):
        self._h = ctypes.c_void_p()
        self.key_bytes = key_bytes
        self.max_bytes = max_bytes
        self.fixed_len = fixed_len
        self.device = device
        check(lib().isx_open(ctypes.byref(self._h), device, key_bytes, max_bytes, fixed_len))

    # -- lifecycle
    def close(self):
        if self._h:
            lib().isx_close(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):  # pragma: no cover - best effort
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self):
        if not self._h:
            raise ValueError("store is closed")
        return self._h

    # -- rows
    def size(self):
        n = ctypes.c_uint64()
        check(lib().isx_size(self.handle, ctypes.byref(n)))
        return int(n.value)

    def device_bytes(self):
        n = ctypes.c_uint64()
        check(lib().isx_device_bytes(self.handle, ctypes.byref(n)))
        return int(n.value)

    def length_mask(self):
        m = ctypes.c_uint32()
        check(lib().isx_length_mask(self.handle, ctypes.byref(m)))
        return int(m.value)

    def max_k(self):
        m = ctypes.c_uint32()
        check(lib().isx_max_k(self.handle, ctypes.byref(m)))
        return int(m.value)

    def clear(self):
        check(lib().isx_clear(self.handle))

    def release_scratch(self):
        # type: () -> int
        """Free the per-search working memory (re-grows on demand); returns the bytes freed."""
        n = ctypes.c_uint64()
        check(lib().isx_release_scratch(self.handle, ctypes.byref(n)))
        return int(n.value)

    def add(self, keys, codes, lens):
        # type: (np.ndarray, np.ndarray, np.ndarray) -> np.ndarray
        n = len(lens)
        added = np.zeros(n, dtype=np.uint8)
        check(lib().isx_add(self.handle, ptr(keys), ptr(codes), ptr(lens), n, ptr(added)))
        return added

    def add_device(self, d_keys, d_codes, d_lens, n, uniform_len=0):
        # type: (int, int, int|None, int, int) -> None
        """Bulk append of n rows from DEVICE pointers; keys promised unique and absent (include/isx.h: isx_add_device)."""
        check(lib().isx_add_device(self.handle, d_keys, d_codes, d_lens, uniform_len, n))

    def synth_rows_device(self, seed, start, n, d_keys, d_codes, d_lens, lengths=(8, 16, 24, 32), key_mode=0, cpa=64, dup_every=0, dup_back=0):
        """Rows [start, start+n) of the synthetic data set (synth.py) generated on the device into caller-owned buffers."""
        ln = np.ascontiguousarray(lengths, dtype=np.uint8)
        check(lib().isx_synth_rows_device(self.handle, seed, start, n, ptr(ln), len(ln), key_mode, cpa, dup_every, dup_back, d_keys, d_codes, d_lens))

    def remove(self, keys, n):
        removed = np.zeros(n, dtype=np.uint8)
        cnt = ctypes.c_uint64()
        check(lib().isx_remove(self.handle, ptr(keys), n, ptr(removed), ctypes.byref(cnt)))
        return removed, int(cnt.value)

    def contains(self, keys, n):
        present = np.zeros(n, dtype=np.uint8)
        check(lib().isx_contains(self.handle, ptr(keys), n, ptr(present)))
        return present.astype(bool)

    def get(self, keys, n):
        codes = np.zeros((n, 32), dtype=np.uint8)
        lens = np.zeros(n, dtype=np.uint8)
        check(lib().isx_get(self.handle, ptr(keys), n, ptr(codes), ptr(lens)))
        return codes, lens

    def save(self, path):
        check(lib().isx_save(self.handle, os.fsencode(str(path))))

    def load(self, path):
        check(lib().isx_load(self.handle, os.fsencode(str(path))))

    # -- search
    def search(self, queries, qlens, k, thr=None, with_codes=False, first_of_asset=None):
        # type: (np.ndarray, np.ndarray, int, tuple[int,int]|None, bool, np.ndarray|None) -> tuple
        """
        -> (keys, hamming uint16[Q,k], nbits uint16[Q,k], counts uint32[Q], codes|None).
        `first_of_asset`: optional uint8[Q,k] output, 1 where a record is the best of its asset within its query.
        """
        q = len(qlens)
        if k < 1:
            raise ValueError("`count` must be >= 1")
        keys = np.zeros((q, k), dtype=np.uint64) if self.key_bytes == 8 else np.zeros((q, k, 16), dtype=np.uint8)
        h = np.zeros((q, k), dtype=np.uint16)
        nb = np.zeros((q, k), dtype=np.uint16)
        counts = np.zeros(q, dtype=np.uint32)
        codes = np.zeros((q, k, 32), dtype=np.uint8) if with_codes else None
        tn, td = (0, 0) if thr is None else thr
        check(lib().isx_search(self.handle, ptr(queries), ptr(qlens), q, k, tn, td, ptr(keys), ptr(h), ptr(nb), ptr(counts), ptr(codes),
                               ptr(first_of_asset)))
        return keys, h, nb, counts, codes

    def score_segments(self, seg, rec_qi, rec_sim, rec_idf, q_idf):
        # type: (np.ndarray, np.ndarray, np.ndarray, np.ndarray, np.ndarray) -> np.ndarray
        """Per-asset IDF-weighted simprint scores on the device (include/isx.h: isx_score_segments)."""
        seg = np.ascontiguousarray(seg, dtype=np.uint32)
        rec_qi = np.ascontiguousarray(rec_qi, dtype=np.uint32)
        rec_sim = np.ascontiguousarray(rec_sim, dtype=np.float64)
        rec_idf = np.ascontiguousarray(rec_idf, dtype=np.float64)
        q_idf = np.ascontiguousarray(q_idf, dtype=np.float64)
        n_assets = len(seg) - 1
        out = np.zeros(n_assets, dtype=np.float64)
        check(lib().isx_score_segments(self.handle, ptr(seg), n_assets, ptr(rec_qi), ptr(rec_sim), ptr(rec_idf), len(rec_qi), ptr(q_idf),
                                       len(q_idf), ptr(out)))
        return out

    def match_all(self, query, thr=(0, 1), max_out=4096):
        # type: (bytes, tuple[int,int], int) -> tuple
        """All rows within the threshold of one query: (keys, hamming, nbits), unordered; grows the buffer until all fit."""
        q = np.zeros(32, dtype=np.uint8)
        qb = bytes(query)
        q[: len(qb)] = np.frombuffer(qb, dtype=np.uint8)
        while True:
            keys = np.zeros(max_out, dtype=np.uint64) if self.key_bytes == 8 else np.zeros((max_out, 16), dtype=np.uint8)
            h = np.zeros(max_out, dtype=np.uint16)
            nb = np.zeros(max_out, dtype=np.uint16)
            total = ctypes.c_uint64()
            check(lib().isx_match_all(self.handle, ptr(q), len(qb), thr[0], thr[1], max_out, ptr(keys), ptr(h), ptr(nb), ctypes.byref(total)))
            if total.value <= max_out:
                n = int(total.value)
                return keys[:n], h[:n], nb[:n]
            max_out = int(total.value) + 1024

    def self_join(self, thr, page=1 << 22):
        # type: (tuple[int,int], int) -> tuple
        """
        Every pair of stored rows within h/nbits <= thr[0]/thr[1] (include/isx.h: isx_self_join), fetched in pages of
        `page` records -> (keys_a, keys_b, hamming uint16[n], nbits uint16[n]) with key_a < key_b, ascending (key_a, key_b).
        Keys have the form of `search`: uint64[n], or uint8[n,16] for 16-byte keys.
        """
        total = ctypes.c_uint64()
        check(lib().isx_self_join(self.handle, thr[0], thr[1], ctypes.byref(total)))
        n = int(total.value)
        shape = (n,) if self.key_bytes == 8 else (n, 16)
        dt = np.uint64 if self.key_bytes == 8 else np.uint8
        ka, kb = np.zeros(shape, dtype=dt), np.zeros(shape, dtype=dt)
        h, nb = np.zeros(n, dtype=np.uint16), np.zeros(n, dtype=np.uint16)
        for i0 in range(0, n, page):
            c = min(page, n - i0)
            check(lib().isx_join_fetch(self.handle, i0, c, ptr(ka[i0:]), ptr(kb[i0:]), ptr(h[i0:]), ptr(nb[i0:])))
        return ka, kb, h, nb

    def join_fetch(self, first, n):
        # type: (int, int) -> tuple
        """Records [first, first+n) of the last self_join (include/isx.h: isx_join_fetch)."""
        shape = (n,) if self.key_bytes == 8 else (n, 16)
        dt = np.uint64 if self.key_bytes == 8 else np.uint8
        ka, kb = np.zeros(shape, dtype=dt), np.zeros(shape, dtype=dt)
        h, nb = np.zeros(n, dtype=np.uint16), np.zeros(n, dtype=np.uint16)
        check(lib().isx_join_fetch(self.handle, first, n, ptr(ka), ptr(kb), ptr(h), ptr(nb)))
        return ka, kb, h, nb

    def set_stream(self, cuda_stream):
        """
        Run all work of this store on the given CUDA stream handle (e.g. `torch.cuda.current_stream().cuda_stream`).
        torch's default stream has handle 0, which the C ABI reads as "use the store's own stream"; it is passed as
        cudaStreamLegacy (0x1) so that the store really shares torch's stream and stays ordered with its collectives.
        `None` restores the store's own non-blocking stream.
        """
        if cuda_stream is None:
            check(lib().isx_set_stream(self.handle, None))
        else:
            check(lib().isx_set_stream(self.handle, ctypes.c_void_p(cuda_stream if cuda_stream else 1)))

    def set_profiling(self, enabled):
        check(lib().isx_set_profiling(self.handle, 1 if enabled else 0))

    def stats(self):
        st = IsxStats()
        check(lib().isx_get_stats(self.handle, ctypes.byref(st)))
        return st.as_dict()
