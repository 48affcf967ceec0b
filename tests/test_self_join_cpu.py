"""
CPU tests of the self-join's host side: the oracle self-join (oracle/self_join.py) against a brute-force double loop,
and the argument checks and result conversion of ShardedNphdIndex.self_join / ShardedIndex128.self_join on a store
double answered by that oracle.
"""

from fractions import Fraction

import numpy as np
import pytest

from iscc_search_b200 import JoinPairs, ShardedIndex128, ShardedNphdIndex, synth
from oracle.self_join import self_join as oracle_self_join
from tests.fakes import OracleStore


def brute_force(keys_hi, keys_lo, codes, lens, thr):
    lo = np.zeros_like(keys_hi) if keys_lo is None else keys_lo
    out = []
    n = len(lens)
    for i in range(n):
        for j in range(i + 1, n):
            m = min(int(lens[i]), int(lens[j]))
            h = int(np.unpackbits(codes[i, :m] ^ codes[j, :m]).sum())
            if h * thr[1] <= thr[0] * 8 * m:
                a, b = (i, j) if (int(keys_hi[i]), int(lo[i])) < (int(keys_hi[j]), int(lo[j])) else (j, i)
                out.append(((int(keys_hi[a]), int(lo[a]), int(keys_hi[b]), int(lo[b])), a, b, h, 8 * m))
    out.sort()
    return out


def _tiny_store(n, seed, lengths=(1, 2, 3, 8)):
    lens = synth.make_lengths(0, n, seed, lengths)
    codes = synth.make_codes(0, n, seed, lens)
    # near duplicates and prefixes
    codes[n // 2: n // 2 + 10] = codes[:10]
    lens[n // 2: n // 2 + 10] = lens[:10]
    codes[n // 2 + 5: n // 2 + 10, 0] ^= 1
    return codes, lens


@pytest.mark.parametrize("thr", [(0, 1), (1, 8), (1, 4), (3, 7), (1, 1)])
def test_oracle_self_join_matches_brute_force(thr):
    n = 160
    codes, lens = _tiny_store(n, 11)
    keys = synth.make_keys(0, n, 11)
    ra, rb, h, nb = oracle_self_join(keys, None, codes, lens, thr, batch=37)
    ref = brute_force(keys, None, codes, lens, thr)
    assert [(a, b, hh, nn) for _, a, b, hh, nn in ref] == list(zip(ra.tolist(), rb.tolist(), h.tolist(), nb.tolist()))


def test_oracle_self_join_128_bit_keys():
    n = 120
    codes, lens = _tiny_store(n, 12, lengths=(2,))
    hi = (np.arange(n, dtype=np.uint64) % 5).astype(np.uint64)   # equal high halves: the low half decides
    lo = np.random.default_rng(12).permutation(n).astype(np.uint64)
    ra, rb, h, nb = oracle_self_join(hi, lo, codes, lens, (1, 8))
    ref = brute_force(hi, lo, codes, lens, (1, 8))
    assert len(ref) > 0
    assert [(a, b, hh, nn) for _, a, b, hh, nn in ref] == list(zip(ra.tolist(), rb.tolist(), h.tolist(), nb.tolist()))


def test_oracle_self_join_empty_and_single():
    for n in (0, 1):
        codes, lens = np.zeros((n, 32), np.uint8), np.full(n, 8, np.uint8)
        ra, rb, h, nb = oracle_self_join(np.arange(n, dtype=np.uint64), None, codes, lens, (1, 1))
        assert len(ra) == len(rb) == len(h) == len(nb) == 0


class JoinOracleStore(OracleStore):
    """Store double with self_join answered by the oracle self-join, in the key form of the C ABI."""

    calls = []

    def self_join(self, thr, page=1 << 22):
        JoinOracleStore.calls.append(thr)
        ks, hi, lo, codes, lens = self._arrays()
        ra, rb, h, nb = oracle_self_join(hi, lo, codes, lens, thr)
        if self.key_bytes == 8:
            return hi[ra], hi[rb], h, nb
        return synth.keys128_bytes(hi[ra], lo[ra]), synth.keys128_bytes(hi[rb], lo[rb]), h, nb


@pytest.fixture
def join_store(monkeypatch):
    monkeypatch.setattr("iscc_search_b200.nphd.Store", JoinOracleStore)
    JoinOracleStore.calls = []
    return JoinOracleStore


def test_nphd_self_join_threshold_forms(join_store):
    idx = ShardedNphdIndex(max_dim=256)
    keys = np.array([5, 3, 9, 7], dtype=np.uint64)
    idx.add(keys, [b"\x01\x02\x03\x04\x05\x06\x07\x08", b"\x01\x02\x03\x04\x05\x06\x07\x09", b"\x01\x02\x03\x04\x05\x06\x07\x08" * 2,
                   b"\xff" * 8])
    res = idx.self_join(Fraction(1, 64))
    assert join_store.calls[-1] == (1, 64)
    assert isinstance(res, JoinPairs) and len(res) == 3
    assert res.keys_a.tolist() == [3, 3, 5] and res.keys_b.tolist() == [5, 9, 9]
    assert res.hamming.tolist() == [1, 1, 0] and res.nbits.tolist() == [64, 64, 64]
    assert res.distances.dtype == np.float32
    assert np.array_equal(res.distances, np.float32(res.hamming) / np.float32(res.nbits))
    assert len(idx.self_join((0, 1))) == 1
    assert join_store.calls[-1] == (0, 1)
    assert len(idx.self_join(Fraction(0))) == 1
    assert len(idx.self_join((np.uint32(1), np.uint32(1)))) == 6


@pytest.mark.parametrize("bad", [0.25, np.float32(0.5), 1, "1/4", (1,), (1, 0), (-1, 4), (1, 2**32), (2**32, 1), (1.0, 4), (True, 4),
                                 Fraction(1, 2**32), Fraction(-1, 4)])
def test_nphd_self_join_rejects_bad_thresholds(join_store, bad):
    idx = ShardedNphdIndex(max_dim=256)
    with pytest.raises(ValueError):
        idx.self_join(bad)
    assert join_store.calls == []


def test_nphd_self_join_float_message(join_store):
    idx = ShardedNphdIndex(max_dim=256)
    with pytest.raises(ValueError, match="float"):
        idx.self_join(0.125)


def test_index128_self_join(join_store):
    idx = ShardedIndex128(ndim=64)
    hi = np.array([2, 1, 1, 3], dtype=np.uint64)
    lo = np.array([0, 9, 4, 0], dtype=np.uint64)
    keys = synth.keys128_bytes(hi, lo)
    vec = np.zeros((4, 8), dtype=np.uint8)
    vec[1, 0] = 1
    vec[3] = 0xFF
    idx.add(keys, vec)
    res = idx.self_join(1)
    assert join_store.calls[-1] == (1, 64)
    assert res.keys_a.shape == (3, 16) and res.keys_a.dtype == np.uint8
    exp_a = synth.keys128_bytes(np.array([1, 1, 1], np.uint64), np.array([4, 4, 9], np.uint64))
    exp_b = synth.keys128_bytes(np.array([1, 2, 2], np.uint64), np.array([9, 0, 0], np.uint64))
    assert np.array_equal(res.keys_a, exp_a) and np.array_equal(res.keys_b, exp_b)
    assert res.hamming.tolist() == [1, 0, 1]
    assert np.array_equal(res.distances, res.hamming.astype(np.float32))
    assert len(idx.self_join(0)) == 1
    assert len(idx.self_join(64)) == 6
    for bad in (-1, 65, 1.0, True, "1", None):
        with pytest.raises(ValueError):
            idx.self_join(bad)
