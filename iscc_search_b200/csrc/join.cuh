// join.cuh - kernels of the store self-join (isx_self_join, DESIGN.md §3.7): every unordered pair of stored rows within a
// rational NPHD threshold. The pairs are scored by the ordinary fixed-threshold scan (k_scan / k_scan_tc with
// update_tau = 0); the kernels here turn stored rows into a query tile and candidate lists into canonical pair records.
#pragma once
#include <cub/device/device_radix_sort.cuh>
#include <cuda/std/tuple>

#include "kernels.cuh"

namespace isx {

// one pair record: the two keys with key_a < key_b (8-byte keys: uint64 order; 16-byte keys: (hi, lo) = bytewise
// big-endian order). The value beside it packs h | nbits << 16.
struct JoinKey8 { uint64_t a, b; };
struct JoinKey16 { uint64_t a_hi, a_lo, b_hi, b_lo; };
struct JoinKey8Bits {
    __host__ __device__ cuda::std::tuple<uint64_t&, uint64_t&> operator()(JoinKey8& k) const { return {k.a, k.b}; }
};
struct JoinKey16Bits {
    __host__ __device__ cuda::std::tuple<uint64_t&, uint64_t&, uint64_t&, uint64_t&> operator()(JoinKey16& k) const {
        return {k.a_hi, k.a_lo, k.b_hi, k.b_lo};
    }
};
__device__ __forceinline__ void put_join_key(JoinKey8* out, uint64_t slot, uint64_t ahi, uint64_t, uint64_t bhi, uint64_t) {
    out[slot] = JoinKey8{ahi, bhi};
}
__device__ __forceinline__ void put_join_key(JoinKey16* out, uint64_t slot, uint64_t ahi, uint64_t alo, uint64_t bhi, uint64_t blo) {
    out[slot] = JoinKey16{ahi, alo, bhi, blo};
}

// Stored rows -> query words [T][8] (the form ScanParams::queries takes), bytes past the code's length zeroed. Query i is
// row rows[i] of segment `seg`, or row row0 + i when `rows` is null. 8 threads per query, one word each.
__global__ void k_rows_as_queries(const SegDesc* segs, uint32_t seg, uint32_t row0, const uint32_t* rows, uint32_t T, uint32_t* dst) {
    const uint32_t i = (blockIdx.x * blockDim.x + threadIdx.x) >> 3, w = threadIdx.x & 7;
    if (i >= T) return;
    const SegDesc& sd = segs[seg];
    const uint32_t row = rows ? rows[i] : row0 + i, L = sd.len_bytes;
    uint32_t v = 0;
    if (4 * w < L) {
        v = sd.planes[(size_t)w * sd.cap + row];
        if (4 * w + 4 > L) v &= (1u << (8 * (L - 4 * w))) - 1u;
    }
    dst[(size_t)i * 8 + w] = v;
}

struct JoinParams {
    const SegDesc* segs;
    const uint64_t* cand;          // [T][C] candidate lists of the scan
    const uint32_t* cand_cnt;      // [T] exact counts (may exceed C)
    uint32_t C, T;
    uint32_t seg, row0;            // query i = row rows[i] (or row0 + i) of segment seg
    const uint32_t* rows;
    unsigned long long* counter;   // records appended so far (counts past cap too)
    uint64_t cap;                  // records the output holds
    uint32_t* vals;                // [cap] h | nbits << 16
};

// Candidate lists -> pair records, one warp per query. The scan of a chunk starts at the chunk's first block, so its own
// rows meet each other (and themselves) from both sides: a partner in the query's segment at or before the query row is
// dropped, which leaves every pair once. Lists that overflowed (count > C) are skipped: the driver re-scans those queries.
template <class K>
__global__ void k_join_pairs(const JoinParams p, K* keys) {
    const uint32_t q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (q >= p.T) return;   // whole warps
    const uint32_t cnt = p.cand_cnt[q];
    if (cnt > p.C) return;
    const SegDesc& qs = p.segs[p.seg];
    const uint32_t qrow = p.rows ? p.rows[q] : p.row0 + q;
    const uint64_t qhi = qs.khi[qrow], qlo = qs.klo ? qs.klo[qrow] : 0ull;
    const uint64_t* list = p.cand + (size_t)q * p.C;
    for (uint32_t j0 = 0; j0 < cnt; j0 += 32) {
        const uint32_t j = j0 + lane;
        uint64_t c = 0;
        bool keep = false;
        if (j < cnt) {
            c = list[j];
            keep = !(cand_seg(c) == p.seg && cand_row(c) <= qrow);
        }
        const unsigned bal = __ballot_sync(0xffffffffu, keep);
        if (!bal) continue;
        const int leader = __ffs(bal) - 1;
        unsigned long long base = 0;
        if ((int)lane == leader) base = atomicAdd(p.counter, (unsigned long long)__popc(bal));
        base = __shfl_sync(0xffffffffu, base, leader);
        const uint64_t slot = base + (uint64_t)__popc(bal & ((1u << lane) - 1u));
        if (keep && slot < p.cap) {   // beyond cap a record is counted only: the driver reports the total
            const SegDesc& ps = p.segs[cand_seg(c)];
            const uint32_t r = cand_row(c);
            const uint64_t phi = ps.khi[r], plo = ps.klo ? ps.klo[r] : 0ull;
            if (phi < qhi || (phi == qhi && plo < qlo)) put_join_key(keys, slot, phi, plo, qhi, qlo);
            else put_join_key(keys, slot, qhi, qlo, phi, plo);
            p.vals[slot] = cand_h(c) | ((8u * min(qs.len_bytes, ps.len_bytes)) << 16);
        }
    }
}

}  // namespace isx
