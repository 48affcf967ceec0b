"""
Result containers with the surface of `usearch.index.Matches` / `BatchMatches` that iscc-search
touches (`.keys`, `.distances`, `len()`, indexing, `.to_list()`, `.counts`), pinned by
/root/reference/tests/test_usearch_search.py:20-119, 324-372, 484-566.
Extra (exact integer) fields: `.hamming`, `.nbits`, `.vectors` (matched stored codes).
"""

from dataclasses import dataclass, field

import numpy as np


@dataclass
class Match:
    key: object
    distance: float

    def to_tuple(self):
        return self.key, self.distance


@dataclass
class Matches:
    keys: np.ndarray  # uint64[c] or list[bytes] view (128-bit keys: uint8[c,16])
    distances: np.ndarray  # float32[c]
    hamming: np.ndarray = None  # uint16[c]
    nbits: np.ndarray = None  # uint16[c]
    vectors: np.ndarray = None  # uint8[c,32] matched stored codes (optional)
    first: np.ndarray = None  # uint8[c] 1 where the record is the best of its asset (optional, 128-bit keys)
    visited_members: int = 0
    computed_distances: int = 0

    def __len__(self):
        return len(self.keys)

    def _key(self, i):
        k = self.keys[i]
        return bytes(k) if isinstance(k, np.ndarray) else int(k)

    def __getitem__(self, i):
        if isinstance(i, slice):
            raise TypeError("Matches supports integer indexing only")
        if i < 0 or i >= len(self):
            raise IndexError(f"`index` must be an integer under {len(self)}")
        return Match(self._key(i), float(self.distances[i]))

    def to_list(self):
        return [(self._key(i), float(self.distances[i])) for i in range(len(self))]

    def __repr__(self):
        return f"usearch.Matches({len(self)})"


@dataclass
class BatchMatches:
    keys: np.ndarray  # [Q,k]
    distances: np.ndarray  # float32[Q,k]
    counts: np.ndarray  # int64[Q]
    hamming: np.ndarray = None
    nbits: np.ndarray = None
    vectors: np.ndarray = None
    first: np.ndarray = None
    visited_members: int = 0
    computed_distances: int = 0

    def __len__(self):
        return len(self.counts)

    def __getitem__(self, i):
        if i < 0 or i >= len(self):
            raise IndexError(f"`index` must be an integer under {len(self)}")
        c = int(self.counts[i])
        return Matches(
            keys=self.keys[i, :c],
            distances=self.distances[i, :c],
            hamming=None if self.hamming is None else self.hamming[i, :c],
            nbits=None if self.nbits is None else self.nbits[i, :c],
            vectors=None if self.vectors is None else self.vectors[i, :c],
            first=None if self.first is None else self.first[i, :c],
            visited_members=self.visited_members // max(len(self), 1),
            computed_distances=self.computed_distances // max(len(self), 1),
        )

    def to_list(self):
        out = []
        for i in range(len(self)):
            out.extend(self[i].to_list())
        return out

    def __repr__(self):
        return f"usearch.BatchMatches({int(np.sum(self.counts))} across {len(self)} queries)"


@dataclass
class JoinPairs:
    """
    Result of a self-join (`ShardedNphdIndex.self_join`, `ShardedIndex128.self_join`): every pair of stored rows within a
    threshold, once, as (keys_a[i], keys_b[i]) with keys_a[i] < keys_b[i], in ascending (key_a, key_b) order.
    Keys have the form of the index's search results (uint64[n], or uint8[n,16] for 128-bit keys).
    """

    keys_a: np.ndarray
    keys_b: np.ndarray
    hamming: np.ndarray  # uint16[n]
    nbits: np.ndarray  # uint16[n]: 8 * the shorter code's length in bytes
    distances: np.ndarray  # float32[n], the float `search` returns for the same pair

    def __len__(self):
        return len(self.hamming)

    def __repr__(self):
        return f"JoinPairs({len(self)})"
