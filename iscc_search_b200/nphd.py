"""
HBM-resident drop-ins for the two `iscc_usearch` classes iscc-search instantiates:

* `ShardedNphdIndex`  - /root/reference/iscc_search/indexes/usearch/index.py:34, 1617-1625, 1732-1740
                        (variable-length ISCC-UNIT bodies, uint64 ISCC-ID keys, NPHD metric)
* `ShardedIndex128`   - /root/reference/iscc_search/indexes/simprint/usearch_core.py:26, 73-83
                        (fixed-ndim simprints, 128-bit composite keys, Hamming metric)

Same method names, argument meaning and error behaviour; the HNSW/shard knobs are accepted and
ignored (search here is exact). All arithmetic happens in libisx_b200.so on the GPU; this module
only converts arguments and rebuilds the float distances the reference consumes:
NPHD distance = float32(h) / float32(nbits) (index.py:2041-2043 reads `float(distance)`),
Hamming distance = float32(h) (tests/test_usearch_search.py:122-167).
"""

from fractions import Fraction
from pathlib import Path

import numpy as np

from iscc_search_b200._lib import Store
from iscc_search_b200.matches import BatchMatches, JoinPairs, Matches

MAX_BYTES = 32
SNAPSHOT_NAME = "store.isx"


def _as_u64_keys(keys):
    # type: (object) -> tuple[np.ndarray, bool]
    """int | iterable of ints | uint64 array -> (uint64[n], was_scalar)."""
    if isinstance(keys, (int, np.integer)):
        k = int(keys)
        if k < 0 or k >= 2**64:
            raise ValueError(f"key {k} outside uint64 range")
        return np.array([k], dtype=np.uint64), True
    if isinstance(keys, np.ndarray) and keys.dtype == np.uint64:
        return np.ascontiguousarray(keys.ravel()), False
    items = [int(k) for k in (keys.ravel() if isinstance(keys, np.ndarray) else keys)]
    if any(k < 0 or k >= 2**64 for k in items):
        raise ValueError("key outside uint64 range")
    return np.array(items, dtype=np.uint64), False


def _pack_vectors(vectors, n_expected=None, fixed_len=0, max_bytes=MAX_BYTES):
    # type: (object, int|None, int, int) -> tuple[np.ndarray, np.ndarray]
    """bytes | uint8 1-D | 2-D array | list of bytes/arrays -> (codes uint8[n,32], lens uint8[n])."""
    if isinstance(vectors, (bytes, bytearray, memoryview)):
        vectors = [bytes(vectors)]
    elif isinstance(vectors, np.ndarray) and vectors.ndim == 1:
        vectors = [vectors]
    if isinstance(vectors, np.ndarray) and vectors.ndim == 2:
        n, L = vectors.shape
        if not 1 <= L <= max_bytes:
            raise ValueError(f"vector length {L} bytes outside 1..{max_bytes}")
        codes = np.zeros((n, MAX_BYTES), dtype=np.uint8)
        codes[:, :L] = vectors.astype(np.uint8, copy=False)
        lens = np.full(n, L, dtype=np.uint8)
    else:
        n = len(vectors)
        codes = np.zeros((n, MAX_BYTES), dtype=np.uint8)
        lens = np.zeros(n, dtype=np.uint8)
        for i, v in enumerate(vectors):
            b = v.astype(np.uint8, copy=False).tobytes() if isinstance(v, np.ndarray) else bytes(v)
            if not 1 <= len(b) <= max_bytes:
                raise ValueError(f"vector {i}: length {len(b)} bytes outside 1..{max_bytes}")
            codes[i, : len(b)] = np.frombuffer(b, dtype=np.uint8)
            lens[i] = len(b)
    if fixed_len and np.any(lens != fixed_len):
        raise ValueError(f"vectors must have exactly {fixed_len * 8} bits")
    if n_expected is not None and n != n_expected:
        raise ValueError(f"number of keys ({n_expected}) and vectors ({n}) differ")
    return codes, lens


def _rational_threshold(threshold):
    # type: (object) -> tuple[int, int]
    """Fraction | (num, den) of non-negative ints below 2**32 -> (num, den). A float is refused."""
    if isinstance(threshold, (float, np.floating)):
        raise ValueError(
            "self_join needs an exact rational threshold (fractions.Fraction or a (num, den) pair): a float is not one "
            "rational cut, since h/nbits for different code lengths falls on different sides of its rounded value"
        )
    if isinstance(threshold, Fraction):
        num, den = threshold.numerator, threshold.denominator
    elif isinstance(threshold, tuple) and len(threshold) == 2 and all(
        isinstance(v, (int, np.integer)) and not isinstance(v, bool) for v in threshold
    ):
        num, den = int(threshold[0]), int(threshold[1])
    else:
        raise ValueError("threshold must be a fractions.Fraction or a (num, den) pair of ints")
    if not (0 <= num < 2**32 and 0 < den < 2**32):
        raise ValueError(f"threshold {num}/{den}: num and den must be non-negative ints below 2**32, den > 0")
    return num, den


class _IndexBase:
    """Shared lifecycle / bookkeeping of both drop-in classes."""

    _key_bytes = 8

    def _init_store(self, path, max_bytes, fixed_len, device):
        self.path = Path(path) if path is not None else None
        self._store = Store(device=device, key_bytes=self._key_bytes, max_bytes=max_bytes, fixed_len=fixed_len)
        self._dirty = 0
        if self.path is not None:
            self.path.mkdir(parents=True, exist_ok=True)
            snap = self.path / SNAPSHOT_NAME
            if snap.exists():
                self._store.load(snap)

    # usearch / iscc-usearch surface -------------------------------------------------------
    @property
    def size(self):
        return self._store.size()

    def __len__(self):
        return self._store.size()

    @property
    def dirty(self):
        """Unsaved key mutations (auto-flush trigger, index.py:469-478)."""
        return self._dirty

    @property
    def max_count(self):
        """Largest `count` one search accepts (isx_max_k)."""
        return self._store.max_k()

    @property
    def shard_count(self):
        """No file shards: the store is one HBM-resident unit (0 when empty)."""
        return 1 if self._store.size() else 0

    @property
    def serialized_length(self):
        """Bytes a snapshot of the live rows takes (keys + codes), cf. common.py:71-108."""
        return self._store.size() * (self._key_bytes + MAX_BYTES)

    @property
    def _active_shard_path(self):
        return self.path / SNAPSHOT_NAME if self.path is not None else None

    @property
    def memory_usage(self):
        return self._store.device_bytes()

    def save(self):
        """Write the snapshot (atomic rename); clears the dirty counter (index.py:883-913)."""
        if self.path is not None:
            self._store.save(self.path / SNAPSHOT_NAME)
        self._dirty = 0

    def drain_rotations(self):
        """No background shard rotation exists here; kept for interface parity (index.py:934-936)."""

    def reset(self):
        """Release all in-memory (HBM) rows without touching the snapshot (index.py:1699)."""
        self._store.clear()
        self._dirty = 0

    def close(self):
        """Save and release resources (usearch_core.py:310-313)."""
        if self._store is None:
            return
        if self._dirty and self.path is not None:
            self.save()
        self._store.close()
        self._store = None

    def stats(self):
        return self._store.stats()

    def release_scratch(self):
        """Free the store's per-search working memory (include/isx.h: isx_release_scratch); returns the bytes freed."""
        return self._store.release_scratch()


class ShardedNphdIndex(_IndexBase):
    """
    Exact NPHD index over variable-length codes with uint64 keys.

    Mirrors the constructor the reference calls (index.py:1617-1625); `connectivity`,
    `expansion_*`, `shard_size`, `background_rotation` are HNSW / file-shard knobs with no meaning
    for an exact HBM scan and are ignored.
    """

    _key_bytes = 8

    def __init__(self, max_dim=256, path=None, connectivity=16, expansion_add=128, expansion_search=64,
                 shard_size=512 * 1024 * 1024, background_rotation=False, device=0, **_ignored):
        if max_dim < 8 or max_dim > 256 or max_dim % 8:
            raise ValueError("max_dim must be a multiple of 8 bits in 8..256")
        self.max_dim = max_dim
        self._init_store(path, max_dim // 8, 0, device)

    # -- mutation
    def add(self, keys, vectors):
        """
        Add vectors (mixed lengths allowed). A key that already exists is silently skipped, first
        wins (tests/test_usearch_add.py:53-63). Returns the keys as uint64 array like usearch.
        """
        k, _ = _as_u64_keys(keys)
        codes, lens = _pack_vectors(vectors, len(k), 0, self.max_dim // 8)
        if len(k) == 0:
            return k
        added = self._store.add(k, codes, lens)
        self._dirty += int(added.sum())
        return k

    def remove(self, keys):
        """Remove keys; missing keys are ignored. Returns the number removed (tests/test_usearch_remove.py:19-141)."""
        k, _ = _as_u64_keys(keys)
        if len(k) == 0:
            return 0
        _, cnt = self._store.remove(k, len(k))
        self._dirty += cnt
        return cnt

    # -- lookup
    def contains(self, keys):
        k, scalar = _as_u64_keys(keys)
        if len(k) == 0:
            return np.zeros(0, dtype=bool)
        res = self._store.contains(k, len(k))
        return bool(res[0]) if scalar else res

    def __contains__(self, key):
        return bool(self.contains(int(key)))

    def get(self, keys):
        """Stored body WITHOUT padding as uint8 array, or None (tests/test_indexes_usearch_persistence.py:704-706)."""
        k, scalar = _as_u64_keys(keys)
        if len(k) == 0:
            return []
        codes, lens = self._store.get(k, len(k))
        out = [codes[i, : lens[i]].copy() if lens[i] else None for i in range(len(k))]
        return out[0] if scalar else out

    # -- search
    def search(self, vectors, count=10, exact=True, **_ignored):
        """
        Exact top-`count` by NPHD. 1-D input -> Matches, 2-D / list input -> BatchMatches
        (tests/test_usearch_search.py:173-215, 374-429). `count=0` raises ValueError (:678-685).
        """
        if count < 1:
            raise ValueError("`count` must be >= 1")
        queries, qlens = _pack_vectors(vectors, None, 0, self.max_dim // 8)
        single = len(qlens) == 1  # usearch returns a bare Matches for exactly one query vector, 1-D or (1, n)
        kk = max(1, min(int(count), max(self._store.size(), 1)))
        keys, h, nb, counts, _ = self._store.search(queries, qlens, kk)
        dist = (h.astype(np.float32) / np.maximum(nb, 1).astype(np.float32)).astype(np.float32)
        n_rows = self._store.size()
        if single:
            c = int(counts[0])
            return Matches(keys=keys[0, :c], distances=dist[0, :c], hamming=h[0, :c], nbits=nb[0, :c],
                           visited_members=n_rows, computed_distances=n_rows)
        return BatchMatches(keys=keys, distances=dist, counts=counts.astype(np.int64), hamming=h, nbits=nb,
                            visited_members=n_rows * len(qlens), computed_distances=n_rows * len(qlens))

    def self_join(self, threshold):
        # type: (Fraction|tuple[int, int]) -> JoinPairs
        """
        Every pair of stored codes that are near-duplicates of each other: NPHD h/nbits <= threshold, with
        nbits = 8 * the shorter code's length in bytes, as an exact rational rule (the one `search` thresholds use).
        `threshold` is a `fractions.Fraction` or a `(num, den)` pair of non-negative ints below 2**32; a float raises
        ValueError. `Fraction(0)` gives exact duplicates plus codes that are a prefix of a longer stored code.

        Each pair comes back once with key_a < key_b, in ascending (key_a, key_b) order; `distances` are the float32
        values `search` returns for the same pair. All pairs are computed on the GPU and returned in full (MemoryError
        when they do not fit in device memory). This is not usearch's `Index.join`, which computes a one-to-one
        matching between two indexes.
        """
        ka, kb, h, nb = self._store.self_join(_rational_threshold(threshold))
        dist = (h.astype(np.float32) / np.maximum(nb, 1).astype(np.float32)).astype(np.float32)
        return JoinPairs(keys_a=ka, keys_b=kb, hamming=h, nbits=nb, distances=dist)


class ShardedIndex128(_IndexBase):
    """
    Exact Hamming index over fixed-`ndim` binary vectors with 128-bit composite keys
    (`iscc_id_body(8) + offset(4) + size(4)`, big-endian - lmdb_ops.py:30-49).
    Constructor mirrors usearch_core.py:73-83; only metric="hamming", dtype="b1" exist.
    """

    _key_bytes = 16

    def __init__(self, ndim=128, metric="hamming", dtype="b1", path=None, connectivity=8, expansion_add=16,
                 expansion_search=512, shard_size=1024 * 1024 * 1024, background_rotation=False, device=0, **_ignored):
        if str(metric).lower() not in ("hamming", "metrickind.hamming") or str(dtype).lower() not in ("b1", "scalarkind.b1"):
            raise ValueError("ShardedIndex128 on B200 supports metric='hamming', dtype='b1' only")
        if ndim < 8 or ndim > 256 or ndim % 8:
            raise ValueError("ndim must be a multiple of 8 bits in 8..256")
        self.ndim = ndim
        self._init_store(path, ndim // 8, ndim // 8, device)

    def score_segments(self, seg, rec_qi, rec_sim, rec_idf, q_idf):
        """Per-asset simprint scores on this index's device (include/isx.h: isx_score_segments)."""
        return self._store.score_segments(seg, rec_qi, rec_sim, rec_idf, q_idf)

    def _normalize_batch_keys(self, keys):
        # type: (object) -> np.ndarray
        """list of 16-byte keys (or array) -> structured-free `V16` array (one row per key), usearch_core.py:100."""
        if isinstance(keys, np.ndarray) and keys.dtype == np.dtype("V16"):
            return keys
        if isinstance(keys, (bytes, bytearray)):
            keys = [bytes(keys)]
        if isinstance(keys, np.ndarray) and keys.dtype == np.uint8 and keys.ndim == 2 and keys.shape[1] == 16:
            return np.ascontiguousarray(keys).view("V16").ravel()
        out = np.zeros(len(keys), dtype="V16")
        buf = out.view(np.uint8).reshape(len(keys), 16)
        for i, k in enumerate(keys):
            b = bytes(k)
            if len(b) != 16:
                raise ValueError(f"key {i}: expected 16 bytes, got {len(b)}")
            buf[i] = np.frombuffer(b, dtype=np.uint8)
        return out

    def _raw_keys(self, keys):
        arr = self._normalize_batch_keys(keys)
        return np.ascontiguousarray(arr.view(np.uint8).reshape(-1, 16))

    def add(self, keys, vectors):
        k = self._raw_keys(keys)
        codes, lens = _pack_vectors(vectors, len(k), self.ndim // 8, self.ndim // 8)
        if len(k) == 0:
            return self._normalize_batch_keys(keys)
        added = self._store.add(k, codes, lens)
        self._dirty += int(added.sum())
        return self._normalize_batch_keys(keys)

    def remove(self, keys):
        k = self._raw_keys(keys)
        if len(k) == 0:
            return 0
        _, cnt = self._store.remove(k, len(k))
        self._dirty += cnt
        return cnt

    def contains(self, keys):
        scalar = isinstance(keys, (bytes, bytearray))
        k = self._raw_keys(keys)
        if len(k) == 0:
            return np.zeros(0, dtype=bool)
        res = self._store.contains(k, len(k))
        return bool(res[0]) if scalar else res

    def __contains__(self, key):
        return bool(self.contains(bytes(key)))

    def get(self, keys):
        scalar = isinstance(keys, (bytes, bytearray))
        k = self._raw_keys(keys)
        if len(k) == 0:
            return []
        codes, lens = self._store.get(k, len(k))
        out = [codes[i, : lens[i]].copy() if lens[i] else None for i in range(len(k))]
        return out[0] if scalar else out

    def search(self, vectors, count=10, exact=True, threshold_bits=None, with_vectors=False, with_first=False, **_ignored):
        """
        Exact top-`count` by Hamming distance; distances are raw bit counts as float32.
        A single 1-D query returns a bare `Matches` (usearch_core.py:167-169), a batch `BatchMatches`.
        `threshold_bits` (extension): keep only rows with h <= threshold_bits (h == 0: equality join).
        `with_vectors` (extension): also return the matched stored codes (replaces `.get` per match).
        `with_first` (extension): also return per-record flags marking the best record of every asset
        (asset = first 8 key bytes) within its query - the grouping of usearch_core.py:187-196, done on the device.
        """
        if count < 1:
            raise ValueError("`count` must be >= 1")
        queries, qlens = _pack_vectors(vectors, None, self.ndim // 8, self.ndim // 8)
        single = len(qlens) == 1  # bare Matches for one query (usearch_core.py:167-169), also for a (1, n) array
        kk = max(1, min(int(count), max(self._store.size(), 1)))
        thr = None if threshold_bits is None else (int(threshold_bits), self.ndim)
        first = np.zeros((len(qlens), kk), dtype=np.uint8) if with_first else None
        keys, h, nb, counts, codes = self._store.search(queries, qlens, kk, thr, with_vectors, first)
        dist = h.astype(np.float32)
        nbytes = self.ndim // 8
        vec = codes[:, :, :nbytes] if codes is not None else None
        n_rows = self._store.size()
        if single:
            c = int(counts[0])
            return Matches(keys=keys[0, :c], distances=dist[0, :c], hamming=h[0, :c], nbits=nb[0, :c],
                           vectors=None if vec is None else vec[0, :c], first=None if first is None else first[0, :c],
                           visited_members=n_rows, computed_distances=n_rows)
        return BatchMatches(keys=keys, distances=dist, counts=counts.astype(np.int64), hamming=h, nbits=nb, vectors=vec, first=first,
                            visited_members=n_rows * len(qlens), computed_distances=n_rows * len(qlens))

    def self_join(self, threshold_bits):
        # type: (int) -> JoinPairs
        """
        Every pair of stored vectors within `threshold_bits` (0..ndim) Hamming bits of each other (0: exact duplicates).
        Each pair comes back once with key_a < key_b (16-byte keys compared bytewise), in ascending (key_a, key_b)
        order; keys are uint8[n,16] like `search` results and `distances` are float32(h). Computed on the GPU and
        returned in full (MemoryError when the pairs do not fit in device memory). This is not usearch's `Index.join`,
        which computes a one-to-one matching between two indexes.
        """
        if isinstance(threshold_bits, bool) or not isinstance(threshold_bits, (int, np.integer)):
            raise ValueError("threshold_bits must be an int")
        t = int(threshold_bits)
        if not 0 <= t <= self.ndim:
            raise ValueError(f"threshold_bits must be in 0..{self.ndim}, got {t}")
        ka, kb, h, nb = self._store.self_join((t, self.ndim))
        return JoinPairs(keys_a=ka, keys_b=kb, hamming=h, nbits=nb, distances=h.astype(np.float32))


class _MultiScratch:
    def release_scratch(self):
        """Free the per-search working memory of every device's store."""
        return sum(shard.release_scratch() for shard in self.shards)


class MultiDeviceNphdIndex(_MultiScratch):
    """
    `ShardedNphdIndex` row-sharded over several GPUs of ONE process.

    iscc-search serves from a single process (cli/serve.py:43-50, manager.py:43-46), so the protocol backend reaches all
    GPUs of the box through one store handle per device: a key lives on the device `splitmix64(key) % G` selects
    (`sharded.owner_of`), every device answers its own exact top-`count` concurrently (one host thread per device; the
    C ABI releases the GIL) and the G sorted lists are merged on the host under the store's total order - exact rational
    h/n, then key - so the result is identical to a single-device index. For one process per GPU with an NCCL
    all-gather and a device merge see `sharded.ShardedSearcher`.
    """

    def __init__(self, max_dim=256, path=None, devices=(0,), **kw):
        from concurrent.futures import ThreadPoolExecutor

        if not devices:
            raise ValueError("devices must name at least one GPU")
        self.max_dim = max_dim
        self.path = Path(path) if path is not None else None
        self.devices = tuple(int(d) for d in devices)
        self.shards = [ShardedNphdIndex(max_dim=max_dim, path=None if self.path is None else self.path / f"shard{i}", device=d, **kw)
                       for i, d in enumerate(self.devices)]
        self._pool = ThreadPoolExecutor(max_workers=len(self.shards), thread_name_prefix="isx-dev")

    def _owner(self, keys):
        from iscc_search_b200.sharded import owner_of

        return owner_of(keys, len(self.shards))

    def _map(self, fn):
        return list(self._pool.map(fn, self.shards))

    # -- mutation: every key has exactly one home shard; a key present anywhere is a duplicate (first wins)
    def add(self, keys, vectors):
        k, _ = _as_u64_keys(keys)
        codes, lens = _pack_vectors(vectors, len(k), 0, self.max_dim // 8)
        if len(k) == 0:
            return k
        owner = self._owner(k)
        for g, shard in enumerate(self.shards):
            sel = np.nonzero(owner == g)[0]
            if len(sel):
                shard.add(k[sel], [codes[i, : lens[i]] for i in sel])
        return k

    def remove(self, keys):
        k, _ = _as_u64_keys(keys)
        if len(k) == 0:
            return 0
        owner = self._owner(k)
        return sum(shard.remove(k[owner == g]) for g, shard in enumerate(self.shards) if np.any(owner == g))

    def contains(self, keys):
        k, scalar = _as_u64_keys(keys)
        if len(k) == 0:
            return np.zeros(0, dtype=bool)
        owner = self._owner(k)
        res = np.zeros(len(k), dtype=bool)
        for g, shard in enumerate(self.shards):
            sel = np.nonzero(owner == g)[0]
            if len(sel):
                res[sel] = shard.contains(k[sel])
        return bool(res[0]) if scalar else res

    def __contains__(self, key):
        return bool(self.contains(int(key)))

    def get(self, keys):
        k, scalar = _as_u64_keys(keys)
        owner = self._owner(k) if len(k) else []
        out = [self.shards[int(g)].get(int(key)) for key, g in zip(k, owner)]
        return out[0] if scalar else out

    # -- search: all shards concurrently, host merge under (h/n, key)
    def search(self, vectors, count=10, exact=True, **_ignored):
        if count < 1:
            raise ValueError("`count` must be >= 1")
        queries, qlens = _pack_vectors(vectors, None, 0, self.max_dim // 8)
        q = len(qlens)
        qlist = [queries[i, : qlens[i]] for i in range(q)]
        parts = self._map(lambda shard: shard.search(qlist, count=count) if shard.size else None)
        parts = [p for p in parts if p is not None]
        n_rows = self.size
        merged = []
        for i in range(q):
            per = [p if q == 1 else p[i] for p in parts]
            keys = np.concatenate([m.keys for m in per]) if per else np.zeros(0, dtype=np.uint64)
            h = np.concatenate([m.hamming for m in per]).astype(np.int64) if per else np.zeros(0, dtype=np.int64)
            nb = np.concatenate([m.nbits for m in per]).astype(np.int64) if per else np.zeros(0, dtype=np.int64)
            if len(keys):
                lcm = int(np.lcm.reduce(np.unique(nb)))
                order = np.lexsort((keys, h * (lcm // nb)))[:count]  # exact: h/n ascending as integers over a common denominator
            else:
                order = np.zeros(0, dtype=np.int64)
            merged.append((keys[order], h[order].astype(np.uint16), nb[order].astype(np.uint16)))
        if q == 1:
            keys, h, nb = merged[0]
            return Matches(keys=keys, distances=(h.astype(np.float32) / np.maximum(nb, 1).astype(np.float32)).astype(np.float32),
                           hamming=h, nbits=nb, visited_members=n_rows, computed_distances=n_rows)
        kk = max(1, max(len(m[0]) for m in merged))
        keys = np.zeros((q, kk), dtype=np.uint64)
        h = np.zeros((q, kk), dtype=np.uint16)
        nb = np.zeros((q, kk), dtype=np.uint16)
        counts = np.zeros(q, dtype=np.int64)
        for i, (mk, mh, mn) in enumerate(merged):
            c = len(mk)
            keys[i, :c], h[i, :c], nb[i, :c], counts[i] = mk, mh, mn, c
        dist = (h.astype(np.float32) / np.maximum(nb, 1).astype(np.float32)).astype(np.float32)
        return BatchMatches(keys=keys, distances=dist, counts=counts, hamming=h, nbits=nb,
                            visited_members=n_rows * q, computed_distances=n_rows * q)

    # -- bookkeeping: sums / fan-out over the shards
    size = property(lambda self: sum(s.size for s in self.shards))
    dirty = property(lambda self: sum(s.dirty for s in self.shards))
    shard_count = property(lambda self: sum(s.shard_count for s in self.shards))
    serialized_length = property(lambda self: sum(s.serialized_length for s in self.shards))
    memory_usage = property(lambda self: sum(s.memory_usage for s in self.shards))
    max_count = property(lambda self: min(s.max_count for s in self.shards))
    _active_shard_path = property(lambda self: None)

    def __len__(self):
        return self.size

    def save(self):
        for s in self.shards:
            s.save()

    def drain_rotations(self):
        pass

    def reset(self):
        for s in self.shards:
            s.reset()

    def close(self):
        for s in self.shards:
            s.close()
        self._pool.shutdown(wait=True)

    def stats(self):
        return [s.stats() for s in self.shards]


class MultiDeviceIndex128(_MultiScratch):
    """
    `ShardedIndex128` row-sharded over several GPUs of ONE process (see `MultiDeviceNphdIndex`).

    A composite key lives on the device its asset selects (`splitmix64(first 8 key bytes) % G`), so all chunks of an
    asset share a device and the per-shard "best record of its asset" flags stay valid after the merge. Every device
    answers its own exact top-`count` (threshold pushed down), the host merges under (Hamming distance, 16-byte key).
    """

    def __init__(self, ndim=128, metric="hamming", dtype="b1", path=None, devices=(0,), **kw):
        from concurrent.futures import ThreadPoolExecutor

        if not devices:
            raise ValueError("devices must name at least one GPU")
        self.ndim = ndim
        self.path = Path(path) if path is not None else None
        self.devices = tuple(int(d) for d in devices)
        self.shards = [ShardedIndex128(ndim=ndim, metric=metric, dtype=dtype, path=None if self.path is None else self.path / f"shard{i}",
                                       device=d, **kw) for i, d in enumerate(self.devices)]
        self._pool = ThreadPoolExecutor(max_workers=len(self.shards), thread_name_prefix="isx-dev")

    _normalize_batch_keys = ShardedIndex128._normalize_batch_keys
    _raw_keys = ShardedIndex128._raw_keys

    def score_segments(self, seg, rec_qi, rec_sim, rec_idf, q_idf):
        """Per-asset simprint scores (pure arithmetic on host-provided records): any of the devices will do."""
        return self.shards[0].score_segments(seg, rec_qi, rec_sim, rec_idf, q_idf)

    def _owner(self, raw_keys):
        from iscc_search_b200.sharded import owner_of

        asset = np.ascontiguousarray(raw_keys[:, :8]).view(">u8").ravel().astype(np.uint64)
        return owner_of(asset, len(self.shards))

    def add(self, keys, vectors):
        k = self._raw_keys(keys)
        codes, _lens = _pack_vectors(vectors, len(k), self.ndim // 8, self.ndim // 8)
        if len(k):
            owner = self._owner(k)
            for g, shard in enumerate(self.shards):
                sel = np.nonzero(owner == g)[0]
                if len(sel):
                    shard.add(k[sel], codes[sel, : self.ndim // 8])
        return self._normalize_batch_keys(keys)

    def remove(self, keys):
        k = self._raw_keys(keys)
        if len(k) == 0:
            return 0
        owner = self._owner(k)
        return sum(shard.remove(k[owner == g]) for g, shard in enumerate(self.shards) if np.any(owner == g))

    def contains(self, keys):
        scalar = isinstance(keys, (bytes, bytearray))
        k = self._raw_keys(keys)
        if len(k) == 0:
            return np.zeros(0, dtype=bool)
        owner = self._owner(k)
        res = np.zeros(len(k), dtype=bool)
        for g, shard in enumerate(self.shards):
            sel = np.nonzero(owner == g)[0]
            if len(sel):
                res[sel] = shard.contains(k[sel])
        return bool(res[0]) if scalar else res

    def __contains__(self, key):
        return bool(self.contains(bytes(key)))

    def get(self, keys):
        scalar = isinstance(keys, (bytes, bytearray))
        k = self._raw_keys(keys)
        owner = self._owner(k) if len(k) else []
        out = [self.shards[int(g)].get(bytes(key)) for key, g in zip(k, owner)]
        return out[0] if scalar else out

    def search(self, vectors, count=10, exact=True, threshold_bits=None, with_vectors=False, with_first=False, **_ignored):
        if count < 1:
            raise ValueError("`count` must be >= 1")
        queries, qlens = _pack_vectors(vectors, None, self.ndim // 8, self.ndim // 8)
        q, nbytes = len(qlens), self.ndim // 8
        batch = np.ascontiguousarray(queries[:, :nbytes])
        parts = list(self._pool.map(lambda shard: shard.search(batch, count=count, threshold_bits=threshold_bits, with_vectors=with_vectors,
                                                               with_first=with_first) if shard.size else None, self.shards))
        parts = [p for p in parts if p is not None]
        n_rows = self.size
        merged = []
        for i in range(q):
            per = [p if q == 1 else p[i] for p in parts]
            per = [m for m in per if len(m)]
            if per:
                keys = np.concatenate([np.asarray(m.keys, dtype=np.uint8).reshape(-1, 16) for m in per])
                h = np.concatenate([m.hamming for m in per])
                hi = np.ascontiguousarray(keys[:, :8]).view(">u8").ravel()
                lo = np.ascontiguousarray(keys[:, 8:]).view(">u8").ravel()
                order = np.lexsort((lo, hi, h))[:count]
                rec = {"keys": keys[order], "h": h[order], "nb": np.concatenate([m.nbits for m in per])[order],
                       "vec": np.concatenate([m.vectors for m in per])[order] if with_vectors else None,
                       "first": np.concatenate([m.first for m in per])[order] if with_first else None}
            else:
                rec = {"keys": np.zeros((0, 16), dtype=np.uint8), "h": np.zeros(0, dtype=np.uint16), "nb": np.zeros(0, dtype=np.uint16),
                       "vec": np.zeros((0, nbytes), dtype=np.uint8) if with_vectors else None,
                       "first": np.zeros(0, dtype=np.uint8) if with_first else None}
            merged.append(rec)
        if q == 1:
            r = merged[0]
            return Matches(keys=r["keys"], distances=r["h"].astype(np.float32), hamming=r["h"], nbits=r["nb"], vectors=r["vec"],
                           first=r["first"], visited_members=n_rows, computed_distances=n_rows)
        kk = max(1, max(len(r["h"]) for r in merged))
        keys = np.zeros((q, kk, 16), dtype=np.uint8)
        h = np.zeros((q, kk), dtype=np.uint16)
        nb = np.zeros((q, kk), dtype=np.uint16)
        vec = np.zeros((q, kk, nbytes), dtype=np.uint8) if with_vectors else None
        first = np.zeros((q, kk), dtype=np.uint8) if with_first else None
        counts = np.zeros(q, dtype=np.int64)
        for i, r in enumerate(merged):
            c = len(r["h"])
            keys[i, :c], h[i, :c], nb[i, :c], counts[i] = r["keys"], r["h"], r["nb"], c
            if with_vectors:
                vec[i, :c] = r["vec"]
            if with_first:
                first[i, :c] = r["first"]
        return BatchMatches(keys=keys, distances=h.astype(np.float32), counts=counts, hamming=h, nbits=nb, vectors=vec, first=first,
                            visited_members=n_rows * q, computed_distances=n_rows * q)

    size = property(lambda self: sum(s.size for s in self.shards))
    dirty = property(lambda self: sum(s.dirty for s in self.shards))
    shard_count = property(lambda self: sum(s.shard_count for s in self.shards))
    serialized_length = property(lambda self: sum(s.serialized_length for s in self.shards))
    memory_usage = property(lambda self: sum(s.memory_usage for s in self.shards))
    max_count = property(lambda self: min(s.max_count for s in self.shards))
    _active_shard_path = property(lambda self: None)

    def __len__(self):
        return self.size

    def save(self):
        for s in self.shards:
            s.save()

    def drain_rotations(self):
        pass

    def reset(self):
        for s in self.shards:
            s.reset()

    def close(self):
        for s in self.shards:
            s.close()
        self._pool.shutdown(wait=True)
