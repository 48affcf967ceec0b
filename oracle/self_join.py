"""
ORACLE - TEST INFRASTRUCTURE ONLY (see oracle/nphd_oracle.py header). Self-join of a store on the CPU: every row is a
query of the C oracle's exact threshold top-k over all rows (k grown until no query is cut), the self match is dropped
and each pair is kept from the side of its smaller key. Shares no code with the GPU kernels.
Never imported from `iscc_search_b200/`.
"""

import numpy as np

from oracle import c_oracle


def self_join(keys_hi, keys_lo, codes, lens, thr, batch=1024, n_threads=0):
    # type: (np.ndarray, np.ndarray|None, np.ndarray, np.ndarray, tuple[int, int], int, int) -> tuple
    """
    Every unordered pair of distinct rows with h * thr[1] <= thr[0] * nbits (nbits = 8 * min(len a, len b)).

    :return: (rows_a int64[n], rows_b int64[n], h uint16[n], nbits uint16[n]): row indices into the input with
             key(row_a) < key(row_b) (keys compared as (hi, lo)), in ascending (key_a, key_b) order.
    """
    keys_hi = np.ascontiguousarray(keys_hi, dtype=np.uint64)
    lo = np.zeros_like(keys_hi) if keys_lo is None else np.ascontiguousarray(keys_lo, dtype=np.uint64)
    codes = np.ascontiguousarray(codes, dtype=np.uint8)
    lens = np.ascontiguousarray(lens, dtype=np.uint8)
    n = len(lens)
    out_a, out_b, out_h, out_n = [], [], [], []
    for q0 in range(0, n, batch):
        q1 = min(n, q0 + batch)
        k = min(n, 64)
        while True:
            rows, h, nb, cnt = c_oracle.topk(keys_hi, keys_lo, codes, lens, codes[q0:q1], lens[q0:q1], k, thr, n_threads)
            if k >= n or int(cnt.max(initial=0)) < k:
                break
            k = min(n, 4 * k)
        for i in range(q1 - q0):
            c = int(cnt[i])
            r = rows[i, :c]
            q = q0 + i
            # the query's own smaller key keeps the pair (the partner sees it from the other side with the roles swapped)
            keep = (r != q) & ((keys_hi[q] < keys_hi[r]) | ((keys_hi[q] == keys_hi[r]) & (lo[q] < lo[r])))
            out_a.append(np.full(int(keep.sum()), q, dtype=np.int64))
            out_b.append(r[keep])
            out_h.append(h[i, :c][keep])
            out_n.append(nb[i, :c][keep])
    if not out_a:
        e = np.zeros(0, dtype=np.int64)
        return e, e.copy(), np.zeros(0, np.uint16), np.zeros(0, np.uint16)
    ra, rb = np.concatenate(out_a), np.concatenate(out_b)
    h, nb = np.concatenate(out_h), np.concatenate(out_n)
    order = np.lexsort((lo[rb], keys_hi[rb], lo[ra], keys_hi[ra]))
    return ra[order], rb[order], h[order], nb[order]
