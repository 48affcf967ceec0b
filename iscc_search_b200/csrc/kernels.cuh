// kernels.cuh - sm_100a kernels of the exact NPHD / Hamming top-k path.
//
// Replaces the native metric + exact scan of `usearch-iscc` behind
//   /root/reference/iscc_search/indexes/usearch/index.py:2037           (ShardedNphdIndex.search)
//   /root/reference/iscc_search/indexes/simprint/usearch_core.py:165    (ShardedIndex128.search)
// Formula: NPHD(a,b) = popc(a[:m]^b[:m]) / (8m), m = min(len) bytes
//   (/root/reference/docs/explanation/similarity-search.md:24-32).
//
// Data layout in HBM (see DESIGN.md): per code length L a bucket of segments; a segment holds
// `cap` rows as 32-bit WORD PLANES plane[w][row], w < ceil(L/4), so a query that shares only m
// bytes with the bucket streams just the first ceil(m/4) planes, each with perfectly coalesced
// 128-bit loads (4 rows per LDG.128). Keys live in separate arrays touched only for winners.
//
// Selection is an exact counting select on the tiny integer distance domain: every (m, h) pair is
// mapped to the dense rank of the rational h/(8m); per query a global histogram over ranks plus
// a running rank threshold tau (always >= the true k-th rank) decides which rows are emitted as
// candidates; the final kernel cuts at the exact k-th rank and breaks ties by key.
#pragma once
#include <cstdint>
#ifndef ISX_PAIR_VOTE
#define ISX_PAIR_VOTE 0
#endif
#include <cuda_runtime.h>

namespace isx {

constexpr int kMaxBytes = 32;
constexpr int kThreads = 256;          // scan CTA
constexpr int kRowsPerStep = kThreads * 4;  // one LDG.128 per plane per thread = 4 rows
constexpr int kMaxTile = 2048;         // queries resident in shared memory per launch
constexpr int kSelectThreads = 1024;
constexpr uint32_t kRowBits = 22;      // rows per segment <= 4 Mi
constexpr uint32_t kSegBits = 16;      // segments per store <= 65536
constexpr uint32_t kHBits = 9;         // hamming <= 256
constexpr uint32_t kRankBits = 13;     // dense ranks < 8192
constexpr int kMaxRanks = 8;           // GPUs of one box sharing thresholds through peer memory

struct SegDesc {
    uint32_t* planes;   // [words][cap]
    uint64_t* khi;      // [cap]
    uint64_t* klo;      // [cap] or nullptr (8-byte keys)
    uint32_t cap;       // allocated rows (multiple of 4096)
    uint32_t n;         // live rows
    uint32_t len_bytes; // code length of the bucket
    uint32_t words;     // ceil(len_bytes / 4)
};

struct ScanParams {
    const SegDesc* segs;
    const uint2* blocks;         // (segment id, first row) of every live 1024-row block, bucket order
    uint32_t block_begin, block_end;  // this launch: blocks of ONE bucket (uniform m / WE)
    uint32_t blocks_per_item;    // consecutive blocks a CTA takes per work item (multiple of G)
    const uint32_t* queries;     // [T][8] words, little-endian words of the zero padded code
    uint32_t T;                  // queries in this launch (<= kMaxTile)
    uint32_t qlen_bytes;         // length of every query of this launch
    uint32_t* tau;               // [T] running rank threshold
    uint32_t* hist;              // [T][R]
    uint32_t* cand_cnt;          // [T]
    uint64_t* cand;              // [T][C]
    uint32_t* overflow;          // [T]
    uint32_t C, R, k;
    const uint16_t* rank_tab;    // [33][257]: rank of h/(8m)
    const uint16_t* hmax_tab;    // [33][R]:  max h with rank(m, h) <= r
    uint32_t update_tau;         // 0: fixed threshold (exact re-scan)
    uint32_t tighten_shift;      // a query's threshold is re-derived whenever its candidate count crosses a multiple of 2^shift
    uint32_t q_split;            // queries per CTA along gridDim.y (small ranges are split over queries
                                 // so the bootstrap rounds still fill the chip)
    uint32_t stage_cap;          // candidate records a CTA stages in shared memory between two flushes (0: emit straight to HBM)
    // Cross-rank threshold sharing (multi-GPU): rank histograms of ALL ranks are summed in peer memory
    // over NVLink (CUDA IPC mapped). Query gq = g_q0 + q lives on rank gq % g_world, slot gq / g_world.
    // Every emission is also counted there (fire-and-forget remote RED); thresholds are tightened from the
    // global counts, i.e. against k rows found ANYWHERE, so a shard stops emitting rows that cannot reach
    // the merged top-k. g_world == 0: disabled (single GPU / emulated shards).
    uint32_t* g_hist[kMaxRanks];
    uint32_t g_world, g_rcap, g_q0;
};

__device__ __forceinline__ uint64_t pack_cand(uint32_t rank, uint32_t h, uint32_t seg, uint32_t row) {
    return ((uint64_t)rank << (kHBits + kSegBits + kRowBits)) | ((uint64_t)h << (kSegBits + kRowBits)) |
           ((uint64_t)seg << kRowBits) | row;
}
__device__ __forceinline__ uint32_t cand_rank(uint64_t c) { return (uint32_t)(c >> (kHBits + kSegBits + kRowBits)); }
__device__ __forceinline__ uint32_t cand_h(uint64_t c) { return (uint32_t)(c >> (kSegBits + kRowBits)) & ((1u << kHBits) - 1); }
__device__ __forceinline__ uint32_t cand_seg(uint64_t c) { return (uint32_t)(c >> kRowBits) & ((1u << kSegBits) - 1); }
__device__ __forceinline__ uint32_t cand_row(uint64_t c) { return (uint32_t)c & ((1u << kRowBits) - 1); }

__device__ __forceinline__ uint4 ldg_stream(const uint32_t* p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}

__device__ __forceinline__ uint32_t ld_sys(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p));  // peer memory: never a stale L1 line
    return v;
}

// Tighten tau[q] to the smallest rank t with (observed) sum_{r<=t} hist[q][r] >= k. Observed counts only under-count, so
// t is always >= the true k-th rank. One warp; the bins are fetched 8 x 32 at a time (one round trip to L2 - or over
// NVLink to the home rank of the shared histograms - per 256 ranks instead of one per 32).
__device__ __noinline__ void tighten_tau(const ScanParams& p, uint32_t q, uint32_t lane) {
    const uint32_t tcur = __ldcg(&p.tau[q]);
    const bool shared = p.g_world != 0;
    const uint32_t gq = p.g_q0 + q;
    const uint32_t* hq = shared ? p.g_hist[gq % p.g_world] + (size_t)(gq / p.g_world) * p.g_rcap : p.hist + (size_t)q * p.R;
    uint32_t cum = 0;
    for (uint32_t base = 0; base <= tcur; base += 256) {
        uint32_t v[8];
#pragma unroll
        for (int j = 0; j < 8; j++) {
            const uint32_t r = base + 32 * j + lane;
            v[j] = (r <= tcur) ? (shared ? ld_sys(&hq[r]) : __ldcg(&hq[r])) : 0u;
        }
#pragma unroll
        for (int j = 0; j < 8; j++) {
            uint32_t incl = v[j];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= (uint32_t)o) incl += t;
            }
            const unsigned hit = __ballot_sync(0xffffffffu, cum + incl >= p.k);
            if (hit) {
                const uint32_t t = base + 32 * j + (uint32_t)(__ffs(hit) - 1);
                if (lane == 0 && t < tcur) atomicMin(&p.tau[q], t);
                return;
            }
            cum += __shfl_sync(0xffffffffu, incl, 31);
            if (base + 32 * (j + 1) > tcur) return;
        }
    }
}

// Rare path, entered by the WHOLE warp when any lane has a row within the running threshold of
// query q: per row slot one ballot, one slot-allocating atomic per warp, fire-and-forget histogram
// updates. `s_rank` is the rank row of this launch's compared length (shared memory).
// Threshold feedback lives here too: the warp whose emission makes the query's candidate count cross a multiple of
// 2^tighten_shift (~k/4 new candidates anywhere on this GPU) re-derives the threshold from the histogram. The
// threshold follows "k rows found" only logarithmically in the rows scanned, so that is ~100 re-derivations per query
// and search instead of one per CTA and work item in which the query emitted (which cost 25 % of a small shard's scan).
__device__ __noinline__ void emit_group(const ScanParams& p, uint32_t q, uint32_t hmax, uint32_t d0, uint32_t d1, uint32_t d2,
                                        uint32_t d3, uint32_t seg, uint32_t row0, uint32_t seg_n, const uint16_t* s_rank,
                                        unsigned char* dirty) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t d[4] = {d0, d1, d2, d3};
    bool any = false, crossed = false;
#pragma unroll
    for (int r = 0; r < 4; r++) {
        const bool e = (d[r] <= hmax) && (row0 + r < seg_n);  // padding rows of the last block never emit
        const unsigned bal = __ballot_sync(0xffffffffu, e);
        if (bal == 0) continue;
        any = true;
        const int leader = __ffs(bal) - 1;
        uint32_t base = 0;
        if ((int)lane == leader) base = atomicAdd(&p.cand_cnt[q], (uint32_t)__popc(bal));
        base = __shfl_sync(0xffffffffu, base, leader);
        crossed |= ((base + (uint32_t)__popc(bal)) >> p.tighten_shift) != (base >> p.tighten_shift);
        if (e) {
            const uint32_t rank = s_rank[d[r]];
            atomicAdd(&p.hist[(size_t)q * p.R + rank], 1u);
            if (p.g_world) {
                const uint32_t gq = p.g_q0 + q;
                atomicAdd(&p.g_hist[gq % p.g_world][(size_t)(gq / p.g_world) * p.g_rcap + rank], 1u);  // NVLink RED
            }
            const uint32_t slot = base + __popc(bal & ((1u << lane) - 1u));
            if (slot < p.C) p.cand[(size_t)q * p.C + slot] = pack_cand(rank, d[r], seg, row0 + r);
            else p.overflow[q] = 1u;
        }
    }
    if (dirty && any && lane == 0) dirty[q] = 1;
    if (crossed && p.update_tau) {
        __threadfence();   // this warp's own counts are visible to the sweep (others' are at worst missed: under-count)
        tighten_tau(p, q, lane);
    }
}

// ---- staged emission ---------------------------------------------------------------------------
// emit_group pays one RETURNING global atomic (a round trip to L2, ~1 us with the warp stalled) per emitting row slot.
// While the thresholds are loose - the warm-up ranges of every tile, the first items of the bulk launch, k = 1000 - that
// round trip, not the popcounts, bounds the scan. So a CTA appends its candidates to a shared-memory stage (one
// shared-memory atomic each) and flushes the stage at the end of every work item with all 256 threads: the slot
// allocations of a whole item are in flight together, and the threshold is re-derived there. Thresholds are only re-read
// at item boundaries anyway, so deferring the histogram updates to the same point changes nothing a CTA can observe.
// A record that finds the stage full is written straight to HBM (stage_direct), so capacity never affects the result;
// if such a record crosses a tighten milestone, its query is noted in a short pending list that the flush serves too.
// Layout behind the tables of k_scan: u64 cand[cap] | u32 query[cap] | u32 counters[4] | u32 pending[kStagePending].
// The counters only grow: [0] records appended, [1] records flushed, [2] pending noted, [3] pending served - a flush
// moves [1] and [3] up between two barriers, emitters (which run outside that window) index relative to them.
constexpr uint32_t kStagePending = 32;
struct Stage {
    uint64_t* cand;
    uint32_t* query;
    uint32_t* counters;
    uint32_t* pending;
};
__host__ __device__ constexpr size_t stage_bytes(uint32_t cap) { return 8 + (size_t)cap * 12 + 16 + kStagePending * 4; }
__device__ __forceinline__ Stage stage_of(const ScanParams& p, const uint16_t* s_rank) {
    uintptr_t a = (reinterpret_cast<uintptr_t>(s_rank + 258 + p.R) + 7) & ~(uintptr_t)7;
    Stage st;
    st.cand = reinterpret_cast<uint64_t*>(a);
    st.query = reinterpret_cast<uint32_t*>(st.cand + p.stage_cap);
    st.counters = st.query + p.stage_cap;
    st.pending = st.counters + 4;
    return st;
}

// one candidate of query q to HBM, by one thread; returns whether the query's count crossed a tighten milestone
__device__ __forceinline__ bool stage_direct(const ScanParams& p, uint32_t q, uint64_t c) {
    const uint32_t rank = cand_rank(c);
    const uint32_t slot = atomicAdd(&p.cand_cnt[q], 1u);
    atomicAdd(&p.hist[(size_t)q * p.R + rank], 1u);
    if (p.g_world) {
        const uint32_t gq = p.g_q0 + q;
        atomicAdd(&p.g_hist[gq % p.g_world][(size_t)(gq / p.g_world) * p.g_rcap + rank], 1u);  // NVLink RED
    }
    if (slot < p.C) p.cand[(size_t)q * p.C + slot] = c;
    else p.overflow[q] = 1u;
    return ((slot + 1) >> p.tighten_shift) != (slot >> p.tighten_shift);
}

// one candidate of query q to the stage, by one thread (straight to HBM when the stage is full)
__device__ __forceinline__ void stage_push(const ScanParams& p, const Stage& st, uint32_t q, uint64_t c) {
    const uint32_t idx = atomicAdd(&st.counters[0], 1u) - st.counters[1];
    if (idx < p.stage_cap) {
        st.cand[idx] = c;
        st.query[idx] = q;
    } else if (stage_direct(p, q, c)) {
        const uint32_t j = atomicAdd(&st.counters[2], 1u) - st.counters[3];
        if (j < kStagePending) st.pending[j] = q;   // beyond that: the threshold just stays looser for a while
    }
}

// entered by the whole warp when any lane has a row of the group within the bound of query q
__device__ __noinline__ void stage_group(const ScanParams& p, uint32_t q, uint32_t hmax, uint32_t d0, uint32_t d1, uint32_t d2,
                                         uint32_t d3, uint32_t seg, uint32_t row0, uint32_t seg_n, const uint16_t* s_rank) {
    if (p.stage_cap == 0) {   // no room for a stage next to a maximal query tile: the warp-aggregated direct path
        emit_group(p, q, hmax, d0, d1, d2, d3, seg, row0, seg_n, s_rank, nullptr);
        return;
    }
    const Stage st = stage_of(p, s_rank);
    const uint32_t d[4] = {d0, d1, d2, d3};
#pragma unroll
    for (int r = 0; r < 4; r++) {
        if (d[r] <= hmax && row0 + r < seg_n)   // padding rows of the last block never emit
            stage_push(p, st, q, pack_cand(s_rank[d[r]], d[r], seg, row0 + r));
    }
}

// all threads of the CTA, called between two barriers with no emitter in between
__device__ __noinline__ void stage_flush(const ScanParams& p, const uint16_t* s_rank) {
    const Stage st = stage_of(p, s_rank);
    const uint32_t appended = st.counters[0], noted = st.counters[2];
    const uint32_t n = min(appended - st.counters[1], p.stage_cap);
    const uint32_t n_pending = min(noted - st.counters[3], kStagePending);
    if (appended == st.counters[1] && n_pending == 0) return;   // CTA-uniform: nothing staged since the last flush
    __syncthreads();                                            // everyone has read the counters
    if (threadIdx.x == 0) { st.counters[1] = appended; st.counters[3] = noted; }
    const uint32_t lane = threadIdx.x & 31;
    for (uint32_t i0 = threadIdx.x & ~31u; i0 < n; i0 += kThreads) {   // warp-uniform trip count
        const uint32_t i = i0 + lane;
        uint32_t q = 0;
        bool crossed = false;
        if (i < n) {
            q = st.query[i];
            crossed = stage_direct(p, q, st.cand[i]);
        }
        if (p.update_tau) {
            unsigned bal = __ballot_sync(0xffffffffu, crossed);
            if (bal) __threadfence();   // this warp's counts are visible to its sweeps (others' are at worst missed: under-count)
            while (bal) {
                const int l = __ffs(bal) - 1;
                bal &= bal - 1;
                tighten_tau(p, __shfl_sync(0xffffffffu, q, l), lane);
            }
        }
    }
    if (p.update_tau)
        for (uint32_t j = threadIdx.x >> 5; j < n_pending; j += kThreads / 32) tighten_tau(p, st.pending[j], lane);
}

// Hamming distance of one row (word r of each plane vector) to the query, WE words, last word masked.
// Carry-save compression: the POPC pipe issues 16 lanes/clk/SM against 64 for LOP3 and both overlap
// (profiles/microbench), so three XOR words are first folded by a full adder (2 LOP3) into a sum and a
// carry word: popc(x0)+popc(x1)+popc(x2) = popc(s) + 2*popc(c). 8 words need 5 POPC instead of 8.
// The pure arithmetic helpers below are __host__ __device__ so that the library's host-side self test
// (isx_selftest_distance, CPU test-suite) runs the very same template code against a naive popcount.
#ifdef __CUDA_ARCH__
#define ISX_UNROLL _Pragma("unroll")
#else
#define ISX_UNROLL
#endif
__host__ __device__ __forceinline__ uint32_t popc32(uint32_t x) {
#ifdef __CUDA_ARCH__
    return (uint32_t)__popc(x);
#else
    return (uint32_t)__builtin_popcount(x);
#endif
}

template <int WE>
__host__ __device__ __forceinline__ uint32_t pair_distance(const uint32_t (&x)[WE]) {
    auto csa_s = [](uint32_t a, uint32_t b, uint32_t c) { return a ^ b ^ c; };
    auto csa_c = [](uint32_t a, uint32_t b, uint32_t c) { return (a & b) | (c & (a ^ b)); };
    if constexpr (WE == 1) return popc32(x[0]);
    else if constexpr (WE == 2) return popc32(x[0]) + popc32(x[1]);
    else if constexpr (WE == 3) return popc32(csa_s(x[0], x[1], x[2])) + 2 * popc32(csa_c(x[0], x[1], x[2]));
    else if constexpr (WE == 4) return popc32(csa_s(x[0], x[1], x[2])) + popc32(x[3]) + 2 * popc32(csa_c(x[0], x[1], x[2]));
    else if constexpr (WE == 5)
        return popc32(csa_s(x[0], x[1], x[2])) + popc32(x[3]) + popc32(x[4]) + 2 * popc32(csa_c(x[0], x[1], x[2]));
    else if constexpr (WE == 6)
        return popc32(csa_s(x[0], x[1], x[2])) + popc32(csa_s(x[3], x[4], x[5])) +
               2 * (popc32(csa_c(x[0], x[1], x[2])) + popc32(csa_c(x[3], x[4], x[5])));
    else if constexpr (WE == 7) {
        uint32_t s0 = csa_s(x[0], x[1], x[2]), s1 = csa_s(x[3], x[4], x[5]);
        return popc32(csa_s(s0, s1, x[6])) +
               2 * (popc32(csa_c(x[0], x[1], x[2])) + popc32(csa_c(x[3], x[4], x[5])) + popc32(csa_c(s0, s1, x[6])));
    } else {
        uint32_t s0 = csa_s(x[0], x[1], x[2]), s1 = csa_s(x[3], x[4], x[5]);
        return popc32(csa_s(s0, s1, x[6])) + popc32(x[7]) +
               2 * (popc32(csa_c(x[0], x[1], x[2])) + popc32(csa_c(x[3], x[4], x[5])) + popc32(csa_c(s0, s1, x[6])));
    }
}

__host__ __device__ __forceinline__ uint32_t comp(const uint4& v, int r) { return r == 0 ? v.x : r == 1 ? v.y : r == 2 ? v.z : v.w; }

// Cheap LOWER bounds of the distance: popc(x0 | x1 [| x2]) <= popc(x0) + popc(x1) [+ popc(x2)], one POPC per
// group of F words (the OR rides in the XOR's LOP3). A row whose bound already exceeds the query's current
// Hamming bound cannot be a candidate, so once the running threshold is tight the exact distance is only
// evaluated for the rare warp slots where some lane's bound passes. Exact by construction (the bound never
// over-estimates). Two tiers: folds of 3 words (6, 7, 8 words: 2, 3, 3 POPC) when the bound is very tight,
// folds of 2 words (2, 4, 5, 6, 8 words: 1, 2, 3, 3, 4 POPC) otherwise.
// Cutoffs = largest Hamming bound for which the filter is expected to reject almost every random row:
// mean - 2.75 sigma of the bound under uniformly random codes (an OR of f words ~ Bin(32, 1 - 2^-f)).
template <int WE>
struct LowerBound {
    static constexpr uint32_t kCutoff3 = WE == 6 ? 48u : WE == 7 ? 61u : WE == 8 ? 70u : 0u;
    static constexpr uint32_t kCutoff2 = WE == 2 ? 17u : WE == 4 ? 38u : WE == 5 ? 50u : WE == 6 ? 60u : WE == 8 ? 82u : 0u;
    // bound of row r of a 4-row group straight from the planes
    template <int F>
    __host__ __device__ __forceinline__ static uint32_t eval(const uint4 (&a)[WE], const uint32_t (&qv)[WE], int r, uint32_t mask_last) {
        uint32_t acc = 0;
        ISX_UNROLL
        for (int w = 0; w < WE; w += F) {
            // the fold that holds the last word starts with it: (a ^ q) & mask is ONE LOP3 there, and every further
            // word of a fold is one LOP3 (t | (a ^ q)); starting from an unmasked word costs an extra instruction
            const bool has_last = (w + F >= WE);
            uint32_t t = has_last ? ((comp(a[WE - 1], r) ^ qv[WE - 1]) & mask_last) : 0u;
            ISX_UNROLL
            for (int j = 0; j < F; j++) {
                if (w + j < WE && !(has_last && w + j == WE - 1)) t |= comp(a[w + j], r) ^ qv[w + j];
            }
            acc += popc32(t);
        }
        return acc;
    }
    template <int F>
    __device__ __forceinline__ static uint32_t min4(const uint4 (&a)[WE], const uint32_t (&qv)[WE], uint32_t mask_last) {
        return min(min(eval<F>(a, qv, 0, mask_last), eval<F>(a, qv, 1, mask_last)),
                   min(eval<F>(a, qv, 2, mask_last), eval<F>(a, qv, 3, mask_last)));
    }
};

// WE: words compared per pair (1..8). G: groups of 4 rows a thread keeps in flight.
// Work split: CTA x of the launch owns a contiguous, balanced share of the launch's block range and
// re-reads the running thresholds every `blocks_per_item` blocks.
template <int WE, int G, int MINB = 3>
__global__ void __launch_bounds__(kThreads, MINB) k_scan(const __grid_constant__ ScanParams p) {
    constexpr int QW = (WE <= 4) ? 4 : 8;  // query words kept per query in shared memory
    constexpr bool kInRec = WE < QW;       // a free word of the record carries the query's bound | tier: one address stream, no extra LDS
    extern __shared__ uint4 smem_raw[];
    const uint32_t tid = threadIdx.x;
    const uint32_t q0 = blockIdx.y * p.q_split;                 // first query of this CTA's sub-tile
    const uint32_t T = min(p.q_split, p.T - q0);
    uint32_t* qw = reinterpret_cast<uint32_t*>(smem_raw);       // [q_split][QW]
    uint16_t* hm = reinterpret_cast<uint16_t*>(qw + (size_t)p.q_split * QW);   // [q_split] bound | tier << 12 (h <= 256 needs 9 bits)
    uint16_t* s_rank = hm + ((p.q_split + 1) & ~1u);                 // [258] rank of h at this compared length
    uint16_t* s_hrow = s_rank + 258;                                 // [R rounded up to even] largest h within rank r

    for (uint32_t i = tid; i < T * QW; i += kThreads) {
        uint32_t q = i / QW, w = i % QW;
        qw[i] = (w < WE) ? p.queries[(size_t)(q0 + q) * 8 + w] : 0u;
    }

    // every block of this launch belongs to one bucket: m, the last-word mask and the threshold row are uniform
    const uint32_t seg_len = p.segs[p.blocks[p.block_begin].x].len_bytes;
    const uint32_t m = min(p.qlen_bytes, seg_len);               // bytes compared
    const uint32_t mask_last = (m & 3u) ? ((1u << (8u * (m & 3u))) - 1u) : 0xffffffffu;
    const uint16_t* hrow = s_hrow;
    for (uint32_t i = tid; i < 257; i += kThreads) s_rank[i] = p.rank_tab[m * 257 + i];
    for (uint32_t i = tid; i < p.R; i += kThreads) s_hrow[i] = p.hmax_tab[(size_t)m * p.R + i];
    if (p.stage_cap && tid < 4) stage_of(p, s_rank).counters[tid] = 0;
    __syncthreads();

    // shares are whole groups of G blocks, so only the launch's very last group can be partial (a partial group costs a
    // full pass over the query tile: with 6-7 blocks per CTA on a small shard that was 14-25 % of the work)
    const uint64_t n_groups = ((uint64_t)(p.block_end - p.block_begin) + G - 1) / G;
    const uint32_t my_lo = p.block_begin + G * (uint32_t)(n_groups * blockIdx.x / gridDim.x);
    const uint32_t my_hi = min(p.block_end, p.block_begin + G * (uint32_t)(n_groups * (blockIdx.x + 1) / gridDim.x));
    // small tiles (one query per thread at most): the next item's bound is fetched while this item streams
    const bool prefetch = (T <= kThreads);
    // bound of a query + its filter tier (uniform per query): 3 = folds of three words, 2 = folds of two, 0 = none
    auto pack_bound = [](uint32_t h) -> uint16_t {
        const uint32_t tier = h <= LowerBound<WE>::kCutoff3 ? 3u : h <= LowerBound<WE>::kCutoff2 ? 2u : 0u;
        return (uint16_t)(h | (tier << 12));
    };
    uint16_t hm_next = 0;
    if (prefetch && tid < T) hm_next = pack_bound(hrow[__ldcg(&p.tau[q0 + tid])]);

    // item size ramps G, 2G, 4G .. blocks_per_item: the first bounds a CTA works with are the loosest
    uint32_t item_blocks = p.update_tau ? G : p.blocks_per_item;
    uint32_t n_items_done = 0;
    for (uint32_t b_lo = my_lo; b_lo < my_hi; n_items_done++) {
        const uint32_t b_hi = min(b_lo + item_blocks, my_hi);
        __syncthreads();  // previous item's readers of hm are done, its candidates are staged
        if (p.stage_cap) stage_flush(p, s_rank);
        if (prefetch && n_items_done >= 3) {                  // steady state: bound fetched during the previous item
            if (tid < T) { if (kInRec) qw[(size_t)tid * QW + QW - 1] = hm_next; else hm[tid] = hm_next; }
        } else {                                              // ramp-up items: always the freshest bound
            for (uint32_t q = tid; q < T; q += kThreads) {
                const uint16_t v = pack_bound(hrow[__ldcg(&p.tau[q0 + q])]);
                if (kInRec) qw[(size_t)q * QW + QW - 1] = v; else hm[q] = v;
            }
        }
        __syncthreads();
        if (prefetch && tid < T && p.update_tau) hm_next = pack_bound(hrow[__ldcg(&p.tau[q0 + tid])]);  // lands during the item

        for (uint32_t b = b_lo; b < b_hi; b += G) {
            uint4 a[G][WE];
            uint32_t seg_id[G], row0[G], seg_n[G];
#pragma unroll
            for (int g = 0; g < G; g++) {
                const bool live = (b + g < b_hi);
                const uint2 blk = p.blocks[live ? b + g : b];
                const SegDesc* sd = p.segs + blk.x;
                seg_id[g] = blk.x;
                row0[g] = blk.y + tid * 4;
                seg_n[g] = live ? sd->n : 0u;      // a dead group never emits
                const uint32_t* base = sd->planes + row0[g];
                const uint32_t cap = sd->cap;
#pragma unroll
                for (int w = 0; w < WE; w++) a[g][w] = ldg_stream(base + (size_t)w * cap);
            }

#pragma unroll 1
            for (uint32_t q = 0; q < T; q++) {
                uint32_t qv[WE];
                uint32_t hv;
                {
                    const uint4* qp = reinterpret_cast<const uint4*>(qw + (size_t)q * QW);
                    uint4 v0 = qp[0];
                    qv[0] = v0.x;
                    if (WE > 1) qv[1] = v0.y;
                    if (WE > 2) qv[2] = v0.z;
                    if (WE > 3) qv[3] = v0.w;
                    hv = v0.w;
                    if (WE > 4) {
                        uint4 v1 = qp[1];
                        qv[4] = v1.x;
                        if (WE > 5) qv[5] = v1.y;
                        if (WE > 6) qv[6] = v1.z;
                        if (WE > 7) qv[7] = v1.w;
                        hv = v1.w;
                    }
                    if (!kInRec) hv = hm[q];
                }
                const uint32_t hmax = hv & 0xfffu;
                const uint32_t tier = hv >> 12;   // filter tier, uniform per query
                auto exact_and_emit = [&](int g) {
                    uint32_t d[4];
#pragma unroll
                    for (int r = 0; r < 4; r++) {
                        uint32_t x[WE];
#pragma unroll
                        for (int w = 0; w < WE; w++) x[w] = (comp(a[g][w], r) ^ qv[w]) & ((w == WE - 1) ? mask_last : 0xffffffffu);
                        d[r] = pair_distance<WE>(x);
                    }
                    const uint32_t dmin = min(min(d[0], d[1]), min(d[2], d[3]));
                    if (__any_sync(0xffffffffu, dmin <= hmax))
                        stage_group(p, q0 + q, hmax, d[0], d[1], d[2], d[3], seg_id[g], row0[g], seg_n[g], s_rank);
                };
                auto bound_of = [&](int g) -> uint32_t {
                    return (LowerBound<WE>::kCutoff3 && tier == 3) ? LowerBound<WE>::template min4<3>(a[g], qv, mask_last)
                                                                   : LowerBound<WE>::template min4<2>(a[g], qv, mask_last);
                };
#if ISX_PAIR_VOTE
                if (tier && G >= 2) {   // A/B variant: one vote per PAIR of 4-row groups, per-group votes only when the pair passes
#pragma unroll
                    for (int g = 0; g + 1 < G; g += 2) {
                        const uint32_t lb0 = bound_of(g), lb1 = bound_of(g + 1);
                        if (!__any_sync(0xffffffffu, min(lb0, lb1) <= hmax)) continue;
                        if (__any_sync(0xffffffffu, lb0 <= hmax)) exact_and_emit(g);
                        if (__any_sync(0xffffffffu, lb1 <= hmax)) exact_and_emit(g + 1);
                    }
                    continue;
                }
#endif
#pragma unroll
                for (int g = 0; g < G; g++) {
                    if (tier) {
                        if (!__any_sync(0xffffffffu, bound_of(g) <= hmax)) continue;  // no lane can have a candidate in this slot
                    }
                    exact_and_emit(g);
                }
            }
        }

        b_lo = b_hi;
        item_blocks = min(item_blocks * 2, p.blocks_per_item);
    }
    if (p.stage_cap) {
        __syncthreads();
        stage_flush(p, s_rank);
    }
}

// ---------------------------------------------------------------------------------------------
// Threshold bootstrap: exact rank histogram of a SAMPLE of rows (blocks [block_begin, block_end) of
// one bucket) per query, no candidates emitted. The k-th smallest rank of a subset is an upper
// bound of the k-th smallest rank of the whole store, so tau = that rank is a safe first threshold.
// grid = (sample blocks, queries). The sample is stratified over the buckets (a slice of the first
// blocks of every bucket, proportional to its size), so the bound fits the whole store.
struct SampleParams {
    uint32_t bucket_first_block[kMaxBytes + 1];  // [L] first block of bucket L in the block list
    uint32_t prefix[kMaxBytes + 2];              // [L] sample blocks taken from buckets < L; [33] = total
    uint32_t q_per_cta;                          // queries one CTA histograms for its block (shared-memory bound)
    uint32_t tail_only;                          // 1: only rows in the lower tail (h <= mean - 1.5 sigma of a random pair) are
                                                 // counted - the k-th rank of the sample lies there whenever 4k <= rows / 16
};

// One CTA = one sampled block of 1024 rows x a sub-tile of queries: the rows are loaded once (4 per thread) and scored
// against every query of the sub-tile, each query with its own shared-memory histogram (round 1 launched one CTA per
// (block, query): 82 000 CTAs of a microsecond each for a 1250-query tile).
template <int WE>
__device__ __forceinline__ void sample_body(const ScanParams& p, const SampleParams& sp, const SegDesc& sd, uint32_t blk_row, uint32_t m,
                                            uint32_t q0, uint32_t nq, uint32_t* s_hist, const uint16_t* s_rank) {
    const uint32_t tid = threadIdx.x;
    const uint32_t mask_last = (m & 3u) ? ((1u << (8u * (m & 3u))) - 1u) : 0xffffffffu;
    const uint32_t row0 = blk_row + tid * 4;
    uint4 a[WE];
#pragma unroll
    for (int w = 0; w < WE; w++) a[w] = ldg_stream(sd.planes + (size_t)w * sd.cap + row0);
    const float mean = 4.0f * (float)m, sigma = sqrtf(2.0f * (float)m);
    const uint32_t hcut = sp.tail_only ? (uint32_t)fmaxf(0.0f, mean - 1.5f * sigma) : 8u * m;
    for (uint32_t qi = 0; qi < nq; qi++) {
        const uint32_t* qsrc = p.queries + (size_t)(q0 + qi) * 8;
        uint32_t x0[WE], x1[WE], x2[WE], x3[WE];
#pragma unroll
        for (int w = 0; w < WE; w++) {
            const uint32_t qv = __ldg(&qsrc[w]);
            const uint32_t mk = (w == WE - 1) ? mask_last : 0xffffffffu;
            x0[w] = (a[w].x ^ qv) & mk; x1[w] = (a[w].y ^ qv) & mk; x2[w] = (a[w].z ^ qv) & mk; x3[w] = (a[w].w ^ qv) & mk;
        }
        const uint32_t d[4] = {pair_distance<WE>(x0), pair_distance<WE>(x1), pair_distance<WE>(x2), pair_distance<WE>(x3)};
#pragma unroll
        for (int r = 0; r < 4; r++)
            if (d[r] <= hcut && row0 + r < sd.n) atomicAdd(&s_hist[qi * p.R + s_rank[d[r]]], 1u);
    }
}

__global__ void __launch_bounds__(kThreads) k_sample(const __grid_constant__ ScanParams p, const __grid_constant__ SampleParams sp,
                                                      uint32_t* __restrict__ sample_hist) {
    extern __shared__ uint4 smem_raw[];
    uint32_t* s_hist = reinterpret_cast<uint32_t*>(smem_raw);                       // [q_per_cta][R]
    uint16_t* s_rank = reinterpret_cast<uint16_t*>(s_hist + (size_t)sp.q_per_cta * p.R);   // [258]
    const uint32_t tid = threadIdx.x;
    const uint32_t q0 = blockIdx.y * sp.q_per_cta, nq = min(sp.q_per_cta, p.T - q0);
    uint32_t L = 1;
    while (L < kMaxBytes && blockIdx.x >= sp.prefix[L + 1]) L++;    // bucket of this sample block (uniform)
    const uint2 blk = p.blocks[sp.bucket_first_block[L] + (blockIdx.x - sp.prefix[L])];
    const SegDesc sd = p.segs[blk.x];
    const uint32_t m = min(p.qlen_bytes, sd.len_bytes);
    for (uint32_t i = tid; i < nq * p.R; i += kThreads) s_hist[i] = 0;
    for (uint32_t i = tid; i < 257; i += kThreads) s_rank[i] = p.rank_tab[m * 257 + i];
    __syncthreads();
    switch ((m + 3) / 4) {
        case 1: sample_body<1>(p, sp, sd, blk.y, m, q0, nq, s_hist, s_rank); break;
        case 2: sample_body<2>(p, sp, sd, blk.y, m, q0, nq, s_hist, s_rank); break;
        case 3: sample_body<3>(p, sp, sd, blk.y, m, q0, nq, s_hist, s_rank); break;
        case 4: sample_body<4>(p, sp, sd, blk.y, m, q0, nq, s_hist, s_rank); break;
        case 5: sample_body<5>(p, sp, sd, blk.y, m, q0, nq, s_hist, s_rank); break;
        case 6: sample_body<6>(p, sp, sd, blk.y, m, q0, nq, s_hist, s_rank); break;
        case 7: sample_body<7>(p, sp, sd, blk.y, m, q0, nq, s_hist, s_rank); break;
        default: sample_body<8>(p, sp, sd, blk.y, m, q0, nq, s_hist, s_rank); break;
    }
    __syncthreads();
    for (uint32_t i = tid; i < nq * p.R; i += kThreads) {
        const uint32_t v = s_hist[i];
        if (v) atomicAdd(&sample_hist[(size_t)q0 * p.R + i], v);
    }
}

// tau[q] = min(tau[q], smallest rank whose cumulative SAMPLE count reaches k). One warp per query.
__global__ void k_sample_tau(const uint32_t* __restrict__ sample_hist, uint32_t* tau, uint32_t T, uint32_t R, uint32_t k) {
    const uint32_t q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (q >= T) return;
    const uint32_t tcur = tau[q];
    const uint32_t* hq = sample_hist + (size_t)q * R;
    uint32_t cum = 0;
    for (uint32_t base = 0; base <= tcur; base += 32) {
        const uint32_t r = base + lane;
        uint32_t incl = (r <= tcur) ? hq[r] : 0u;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= (uint32_t)o) incl += t;
        }
        const unsigned hit = __ballot_sync(0xffffffffu, cum + incl >= k);
        if (hit) {
            if (lane == 0) tau[q] = min(tcur, base + (uint32_t)(__ffs(hit) - 1));
            return;
        }
        cum += __shfl_sync(0xffffffffu, incl, 31);
    }
}

// ---------------------------------------------------------------------------------------------
// per-query state reset
__global__ void k_init_queries(uint32_t* tau, uint32_t* hist, uint32_t* sample_hist, uint32_t* cand_cnt, uint32_t* overflow,
                               uint32_t T, uint32_t R, uint32_t tau_init) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t total = (size_t)T * R;
    for (size_t j = i; j < total; j += (size_t)gridDim.x * blockDim.x) { hist[j] = 0; if (sample_hist) sample_hist[j] = 0; }
    if (i < T) { tau[i] = tau_init; cand_cnt[i] = 0; overflow[i] = 0; }
}

// ---------------------------------------------------------------------------------------------
// Final exact selection: one CTA per query.
struct BigRec { uint64_t hi, lo; uint32_t rank, cidx; };  // sort record of the large-k path (global scratch)

struct SelectParams {
    const SegDesc* segs;
    const uint32_t* hist;      // [T][R]
    const uint32_t* cand_cnt;  // [T]
    const uint64_t* cand;      // [T][C]  (or one big list when `single_list`)
    const uint32_t* overflow;  // [T]
    const uint32_t* qmap;      // [T] -> output row (original query index)
    uint32_t C, R, k, T;
    uint32_t qlen_bytes;
    uint32_t sort_cap;         // entries that fit in shared memory
    uint32_t key_words;        // 1 (uint64 keys) | 2 (128-bit keys)
    uint32_t tau_init;         // threshold rank (R-1 = none)
    uint64_t* out_khi; uint64_t* out_klo; uint16_t* out_h; uint16_t* out_n; uint32_t* out_cnt;
    uint8_t* out_codes;        // optional [Q][k][32]
    uint32_t* fallback_info;   // [T][2]: (needs fallback, count_le(d*)) for overflowed queries
    uint32_t skip_overflowed;  // 1 in the normal pass; 0 in the fallback pass (lists are complete)
    // k beyond the shared-memory sort capacity: winners are sorted in this global scratch instead
    // ([T][big_P] records of BigRec, big_P = power of two >= k); nullptr when k <= sort_cap
    BigRec* big_scratch;
    uint32_t big_P;
};

struct SortKey { uint32_t rank; uint64_t hi, lo; };
__device__ __forceinline__ bool key_less(const SortKey& a, const SortKey& b) {
    if (a.rank != b.rank) return a.rank < b.rank;
    if (a.hi != b.hi) return a.hi < b.hi;
    return a.lo < b.lo;
}

__global__ void __launch_bounds__(kSelectThreads) k_select(const SelectParams p) {
    extern __shared__ uint4 smem_raw[];
    // shared layout: khi[cap] | klo[cap] (if key_words==2) | rk[cap] | cidx[cap] | perm[cap] (u16 or u32)
    const uint32_t cap = p.sort_cap;
    uint64_t* s_khi = reinterpret_cast<uint64_t*>(smem_raw);
    uint64_t* s_klo = s_khi + cap;
    uint32_t* s_rk = reinterpret_cast<uint32_t*>(s_klo + (p.key_words == 2 ? cap : 0));
    uint32_t* s_cidx = s_rk + cap;
    uint32_t* s_perm = s_cidx + cap;
    __shared__ uint32_t s_scan[kSelectThreads / 32];
    __shared__ uint32_t s_dstar, s_count_lt, s_total_le, s_fill;
    __shared__ uint32_t s_hist[256];
    __shared__ uint32_t s_need;

    const uint32_t q = blockIdx.x;
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t oq = p.qmap[q];
    const uint32_t* hq = p.hist + (size_t)q * p.R;
    const uint32_t n_list = min(p.cand_cnt[q], p.C);

    // ---- 1. exact k-th rank d* from the histogram (block-wide scan over R bins) ----
    if (tid == 0) { s_dstar = p.R; s_count_lt = 0; s_total_le = 0; s_fill = 0; }
    __syncthreads();
    uint32_t carry = 0;
    for (uint32_t base = 0; base < p.R; base += kSelectThreads) {
        uint32_t r = base + tid;
        uint32_t v = (r < p.R && r <= p.tau_init) ? hq[r] : 0u;
        uint32_t incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= (uint32_t)o) incl += t;
        }
        if (lane == 31) s_scan[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            uint32_t w = s_scan[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                uint32_t t = __shfl_up_sync(0xffffffffu, w, o);
                if (lane >= (uint32_t)o) w += t;
            }
            s_scan[lane] = w;  // inclusive warp totals
        }
        __syncthreads();
        uint32_t before = carry + (warp ? s_scan[warp - 1] : 0u);
        uint32_t cum_incl = before + incl;
        uint32_t cum_excl = cum_incl - v;
        if (r < p.R && cum_excl < p.k && cum_incl >= p.k) { s_dstar = r; s_count_lt = cum_excl; s_total_le = cum_incl; }
        carry += s_scan[kSelectThreads / 32 - 1];
        __syncthreads();
        if (s_dstar != p.R) break;
    }
    __syncthreads();
    if (s_dstar == p.R) {  // fewer than k rows within the threshold: take them all
        if (tid == 0) { s_dstar = min(p.tau_init, p.R - 1); s_count_lt = carry; s_total_le = carry; }
        __syncthreads();
    }
    const uint32_t dstar = s_dstar;
    const uint32_t total_le = s_total_le;               // rows with rank <= d*
    const uint32_t n_out = min(p.k, total_le);

    if (p.skip_overflowed && p.overflow[q]) {
        // candidate list truncated: the histogram still gives d* and the number of rows within it, which is
        // what the host needs to size the exact re-scan of this query
        if (tid == 0) { p.fallback_info[2 * q] = dstar; p.fallback_info[2 * q + 1] = total_le; p.out_cnt[oq] = 0; }
        return;
    }

    const uint64_t* list = p.cand + (size_t)q * p.C;
    uint64_t pivot_hi = ~0ull, pivot_lo = ~0ull;  // ties with key <= pivot are winners

    const bool big = n_out > cap;                       // the winners do not fit the shared-memory sort
    const bool use_pivot = total_le > n_out && (total_le > cap || big);  // ties at d* must be cut by key
    if (use_pivot) {
        // ---- 2b. too many survivors for shared memory: radix-select the r-th smallest key among
        //          the ties at d*, most significant byte first (keys are unique inside a store) ----
        uint32_t need = p.k - s_count_lt;  // >= 1
        uint64_t pre_hi = 0, pre_lo = 0;
        const int n_bytes = (p.key_words == 2) ? 16 : 8;
        for (int b = 0; b < n_bytes; b++) {
            for (uint32_t i = tid; i < 256; i += kSelectThreads) s_hist[i] = 0;
            __syncthreads();
            for (uint32_t i = tid; i < n_list; i += kSelectThreads) {
                uint64_t c = list[i];
                if (cand_rank(c) != dstar) continue;
                const SegDesc& sd = p.segs[cand_seg(c)];
                uint64_t hi = sd.khi[cand_row(c)];
                uint64_t lo = (p.key_words == 2) ? sd.klo[cand_row(c)] : 0ull;
                // top b bytes must equal the prefix found so far
                bool match;
                uint32_t digit;
                if (p.key_words == 2) {
                    if (b < 8) {
                        match = (b == 0) || ((hi >> (64 - 8 * b)) == (pre_hi >> (64 - 8 * b)));
                        digit = (uint32_t)(hi >> (56 - 8 * b)) & 0xffu;
                    } else {
                        int bb = b - 8;
                        match = (hi == pre_hi) && ((bb == 0) || ((lo >> (64 - 8 * bb)) == (pre_lo >> (64 - 8 * bb))));
                        digit = (uint32_t)(lo >> (56 - 8 * bb)) & 0xffu;
                    }
                } else {
                    match = (b == 0) || ((hi >> (64 - 8 * b)) == (pre_hi >> (64 - 8 * b)));
                    digit = (uint32_t)(hi >> (56 - 8 * b)) & 0xffu;
                }
                if (match) atomicAdd(&s_hist[digit], 1u);
            }
            __syncthreads();
            if (tid == 0) {
                uint32_t cum = 0, dsel = 255;
                for (uint32_t d = 0; d < 256; d++) {
                    if (cum + s_hist[d] >= need) { dsel = d; break; }
                    cum += s_hist[d];
                }
                s_need = need - cum;
                s_fill = dsel;
            }
            __syncthreads();
            need = s_need;
            uint64_t dsel = s_fill;
            if (p.key_words == 2 && b >= 8) pre_lo |= dsel << (56 - 8 * (b - 8));
            else pre_hi |= dsel << (56 - 8 * b);
            __syncthreads();
        }
        pivot_hi = pre_hi;
        pivot_lo = (p.key_words == 2) ? pre_lo : ~0ull;
        if (p.key_words == 1) pivot_lo = 0;
        if (tid == 0) s_fill = 0;
        __syncthreads();
    }

    if (big) {
        // ---- large k: winners -> global scratch, bitonic sort there (L2 resident), write out ----
        BigRec* rec = p.big_scratch + (size_t)q * p.big_P;
        for (uint32_t i = tid; i < n_list; i += kSelectThreads) {
            uint64_t c = list[i];
            uint32_t rk = cand_rank(c);
            if (rk > dstar) continue;
            const SegDesc& sd = p.segs[cand_seg(c)];
            uint64_t hi = sd.khi[cand_row(c)];
            uint64_t lo = (p.key_words == 2) ? sd.klo[cand_row(c)] : 0ull;
            if (use_pivot && rk == dstar) {
                bool le = (hi < pivot_hi) || (hi == pivot_hi && lo <= pivot_lo);
                if (!le) continue;
            }
            uint32_t slot = atomicAdd(&s_fill, 1u);
            if (slot < p.big_P) rec[slot] = BigRec{hi, lo, rk, i};
        }
        __syncthreads();
        const uint32_t n_surv = min(s_fill, p.big_P);
        uint32_t P = 1;
        while (P < n_surv) P <<= 1;
        for (uint32_t i = n_surv + tid; i < P; i += kSelectThreads) rec[i] = BigRec{~0ull, ~0ull, 0xffffffffu, 0};  // +inf padding
        __syncthreads();
        for (uint32_t size = 2; size <= P; size <<= 1) {
            for (uint32_t stride = size >> 1; stride > 0; stride >>= 1) {
                for (uint32_t i = tid; i < (P >> 1); i += kSelectThreads) {
                    uint32_t lo_i = 2 * i - (i & (stride - 1));
                    uint32_t hi_i = lo_i + stride;
                    bool asc = ((lo_i & size) == 0);
                    BigRec a = rec[lo_i], b = rec[hi_i];
                    SortKey ka{a.rank, a.hi, a.lo}, kb{b.rank, b.hi, b.lo};
                    if (key_less(kb, ka) == asc) { rec[lo_i] = b; rec[hi_i] = a; }
                }
                __syncthreads();
            }
        }
        const uint32_t n_write = min(n_out, n_surv);
        for (uint32_t j = tid; j < p.k; j += kSelectThreads) {
            size_t o = (size_t)oq * p.k + j;
            if (j < n_write) {
                const BigRec r = rec[j];
                uint64_t c = list[r.cidx];
                const SegDesc& sd = p.segs[cand_seg(c)];
                p.out_khi[o] = r.hi;
                p.out_klo[o] = (p.key_words == 2) ? r.lo : 0ull;
                p.out_h[o] = (uint16_t)cand_h(c);
                p.out_n[o] = (uint16_t)(8u * min(p.qlen_bytes, sd.len_bytes));
            } else {
                p.out_khi[o] = ~0ull; p.out_klo[o] = ~0ull; p.out_h[o] = 0xffffu; p.out_n[o] = 1;
            }
        }
        if (p.out_codes) {
            for (uint32_t j = tid; j < n_write * 8; j += kSelectThreads) {
                uint32_t w = j & 7;
                uint64_t c = list[rec[j >> 3].cidx];
                const SegDesc& sd = p.segs[cand_seg(c)];
                uint32_t v = (w < sd.words) ? sd.planes[(size_t)w * sd.cap + cand_row(c)] : 0u;
                reinterpret_cast<uint32_t*>(p.out_codes)[((size_t)oq * p.k + (j >> 3)) * 8 + w] = v;
            }
        }
        if (tid == 0) p.out_cnt[oq] = n_write;
        return;
    }

    // ---- 2. gather survivors (rank < d*, or rank == d* and key <= pivot) into shared memory ----
    for (uint32_t i = tid; i < n_list; i += kSelectThreads) {
        uint64_t c = list[i];
        uint32_t rk = cand_rank(c);
        if (rk > dstar) continue;
        const SegDesc& sd = p.segs[cand_seg(c)];
        uint64_t hi = sd.khi[cand_row(c)];
        uint64_t lo = (p.key_words == 2) ? sd.klo[cand_row(c)] : 0ull;
        if (use_pivot && rk == dstar) {
            bool le = (hi < pivot_hi) || (hi == pivot_hi && lo <= pivot_lo);
            if (!le) continue;
        }
        uint32_t slot = atomicAdd(&s_fill, 1u);
        if (slot < cap) {
            s_khi[slot] = hi;
            if (p.key_words == 2) s_klo[slot] = lo;
            s_rk[slot] = rk;
            s_cidx[slot] = i;
        }
    }
    __syncthreads();
    const uint32_t n_surv = min(s_fill, cap);
    uint32_t P = 1;
    while (P < n_surv) P <<= 1;
    for (uint32_t i = tid; i < P; i += kSelectThreads) s_perm[i] = (i < n_surv) ? i : 0xffffffffu;
    __syncthreads();

    // ---- 3. bitonic sort of the permutation by (rank, key) ----
    for (uint32_t size = 2; size <= P; size <<= 1) {
        for (uint32_t stride = size >> 1; stride > 0; stride >>= 1) {
            for (uint32_t i = tid; i < (P >> 1); i += kSelectThreads) {
                uint32_t lo_i = 2 * i - (i & (stride - 1));
                uint32_t hi_i = lo_i + stride;
                bool asc = ((lo_i & size) == 0);
                uint32_t pa = s_perm[lo_i], pb = s_perm[hi_i];
                bool b_lt_a;
                if (pb == 0xffffffffu) b_lt_a = false;
                else if (pa == 0xffffffffu) b_lt_a = true;
                else {
                    SortKey ka{s_rk[pa], s_khi[pa], (p.key_words == 2) ? s_klo[pa] : 0ull};
                    SortKey kb{s_rk[pb], s_khi[pb], (p.key_words == 2) ? s_klo[pb] : 0ull};
                    b_lt_a = key_less(kb, ka);
                }
                if (b_lt_a == asc) { s_perm[lo_i] = pb; s_perm[hi_i] = pa; }
            }
            __syncthreads();
        }
    }

    // ---- 4. write the first n_out rows ----
    const uint32_t n_write = min(n_out, n_surv);
    for (uint32_t j = tid; j < p.k; j += kSelectThreads) {
        size_t o = (size_t)oq * p.k + j;
        if (j < n_write) {
            uint32_t e = s_perm[j];
            uint64_t c = list[s_cidx[e]];
            const SegDesc& sd = p.segs[cand_seg(c)];
            p.out_khi[o] = s_khi[e];
            p.out_klo[o] = (p.key_words == 2) ? s_klo[e] : 0ull;
            p.out_h[o] = (uint16_t)cand_h(c);
            p.out_n[o] = (uint16_t)(8u * min(p.qlen_bytes, sd.len_bytes));
        } else {
            p.out_khi[o] = ~0ull; p.out_klo[o] = ~0ull; p.out_h[o] = 0xffffu; p.out_n[o] = 1;
        }
    }
    if (p.out_codes) {
        // stored code of every winner: words strided by cap in the segment's planes
        for (uint32_t j = tid; j < n_write * 8; j += kSelectThreads) {
            uint32_t e = s_perm[j >> 3], w = j & 7;
            uint64_t c = list[s_cidx[e]];
            const SegDesc& sd = p.segs[cand_seg(c)];
            uint32_t v = (w < sd.words) ? sd.planes[(size_t)w * sd.cap + cand_row(c)] : 0u;
            reinterpret_cast<uint32_t*>(p.out_codes)[((size_t)oq * p.k + (j >> 3)) * 8 + w] = v;
        }
    }
    if (tid == 0) p.out_cnt[oq] = n_write;
}

// ---------------------------------------------------------------------------------------------
// Multi-shard merge: every record finds its global position as the number of records (over all
// shards) that order before it - each shard list is already sorted, so that is a sum of binary
// searches. Order: (h/n as exact rational, key). Keys are unique across shards.
__device__ __forceinline__ bool rec_less(uint32_t h1, uint32_t n1, uint64_t hi1, uint64_t lo1, uint32_t h2, uint32_t n2,
                                         uint64_t hi2, uint64_t lo2) {
    uint32_t a = h1 * n2, b = h2 * n1;  // <= 65535 * 256 fits
    if (a != b) return a < b;
    if (hi1 != hi2) return hi1 < hi2;
    return lo1 < lo2;
}

// Field arrays of shard g start `stride` BYTES after those of shard g-1 (packed per-rank buffers as
// an all-gather delivers them); stride 0 = dense [g][q][k] arrays per field.
template <class T>
__device__ __forceinline__ const T* shard_ptr(const T* base, uint32_t g, size_t stride, size_t dense_elems) {
    return stride ? reinterpret_cast<const T*>(reinterpret_cast<const char*>(base) + (size_t)g * stride) : base + (size_t)g * dense_elems;
}

__global__ void k_merge(uint32_t G, uint32_t Q, uint32_t k, size_t stride, const uint64_t* khi, const uint64_t* klo,
                        const uint16_t* hh, const uint16_t* nn, const uint32_t* cnt, uint64_t* o_khi, uint64_t* o_klo,
                        uint16_t* o_h, uint16_t* o_n, uint32_t* o_cnt) {
    const uint32_t q = blockIdx.x;
    const size_t QK = (size_t)Q * k;
    uint32_t total = 0;
    for (uint32_t g = 0; g < G; g++) total += min(shard_ptr(cnt, g, stride, Q)[q], k);
    const uint32_t n_out = min(total, k);
    for (uint32_t e = threadIdx.x; e < G * k; e += blockDim.x) {
        uint32_t g = e / k, j = e % k;
        if (j >= min(shard_ptr(cnt, g, stride, Q)[q], k)) continue;
        size_t src = (size_t)q * k + j;
        uint32_t h1 = shard_ptr(hh, g, stride, QK)[src], n1 = shard_ptr(nn, g, stride, QK)[src];
        uint64_t hi1 = shard_ptr(khi, g, stride, QK)[src], lo1 = shard_ptr(klo, g, stride, QK)[src];
        uint32_t pos = j;  // records of the own list before it
        for (uint32_t g2 = 0; g2 < G; g2++) {
            if (g2 == g) continue;
            const uint16_t* h2 = shard_ptr(hh, g2, stride, QK) + (size_t)q * k;
            const uint16_t* n2 = shard_ptr(nn, g2, stride, QK) + (size_t)q * k;
            const uint64_t* hi2 = shard_ptr(khi, g2, stride, QK) + (size_t)q * k;
            const uint64_t* lo2 = shard_ptr(klo, g2, stride, QK) + (size_t)q * k;
            uint32_t lo_i = 0, hi_i = min(shard_ptr(cnt, g2, stride, Q)[q], k);
            while (lo_i < hi_i) {  // first index whose record is not less than ours
                uint32_t mid = (lo_i + hi_i) >> 1;
                if (rec_less(h2[mid], n2[mid], hi2[mid], lo2[mid], h1, n1, hi1, lo1)) lo_i = mid + 1;
                else hi_i = mid;
            }
            pos += lo_i;
        }
        if (pos < k) {
            size_t o = (size_t)q * k + pos;
            o_khi[o] = hi1; o_klo[o] = lo1; o_h[o] = (uint16_t)h1; o_n[o] = (uint16_t)n1;
        }
    }
    for (uint32_t j = n_out + threadIdx.x; j < k; j += blockDim.x) {
        size_t o = (size_t)q * k + j;
        o_khi[o] = ~0ull; o_klo[o] = ~0ull; o_h[o] = 0xffffu; o_n[o] = 1;
    }
    if (threadIdx.x == 0) o_cnt[q] = n_out;
}

// ---------------------------------------------------------------------------------------------
// Store maintenance kernels.
// dest[i] = (segment << 32) | row, or ~0 to skip row i of the staged batch.
__global__ void k_scatter_rows(const SegDesc* segs, const uint64_t* dest, const uint8_t* codes, const uint8_t* keys,
                               uint32_t key_bytes, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint64_t d = dest[i];
    if (d == ~0ull) return;
    const SegDesc sd = segs[(uint32_t)(d >> 32)];
    uint32_t row = (uint32_t)d;
    const uint32_t* c = reinterpret_cast<const uint32_t*>(codes + i * kMaxBytes);
    for (uint32_t w = 0; w < sd.words; w++) sd.planes[(size_t)w * sd.cap + row] = c[w];
    if (key_bytes == 8) {
        sd.khi[row] = reinterpret_cast<const uint64_t*>(keys)[i];
    } else {
        const uint8_t* kb = keys + i * 16;
        uint64_t hi = 0, lo = 0;
        for (int b = 0; b < 8; b++) { hi = (hi << 8) | kb[b]; lo = (lo << 8) | kb[8 + b]; }
        sd.khi[row] = hi; sd.klo[row] = lo;
    }
}

// ---------------------------------------------------------------------------------------------
// Bulk append from DEVICE memory (isx_add_device): rows of one length class go to consecutive free rows, described
// by a few spans (tail of the last segment + fresh segments). Row i takes the next index of its class (mixed lengths:
// one warp-aggregated atomic per class and warp; uniform length: the index is i itself).
struct BulkSpan { uint32_t seg, row0, first, pad; };  // class-relative rows [first, next span's first) -> seg rows row0..
constexpr int kMaxBulkSpans = 96;
struct BulkPlan {
    uint32_t span_lo[kMaxBytes + 2];  // spans of length class L: [span_lo[L], span_lo[L+1])
    BulkSpan spans[kMaxBulkSpans];
};

__global__ void k_len_hist(const uint8_t* __restrict__ lens, size_t n, uint32_t* __restrict__ hist /*256*/) {
    __shared__ uint32_t sh[256];
    sh[threadIdx.x] = 0;
    __syncthreads();
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) atomicAdd(&sh[lens[i]], 1u);
    __syncthreads();
    if (sh[threadIdx.x]) atomicAdd(&hist[threadIdx.x], sh[threadIdx.x]);
}

__global__ void k_scatter_bulk(const SegDesc* segs, const __grid_constant__ BulkPlan plan, uint32_t* cursor /*[33]*/, const uint8_t* keys,
                               const uint8_t* codes, const uint8_t* lens, uint32_t uniform_len, uint32_t key_bytes, size_t n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t L = lens ? lens[i] : uniform_len;
    uint32_t idx;
    if (lens) {
        const unsigned grp = __match_any_sync(__activemask(), L);
        const int leader = __ffs(grp) - 1;
        const uint32_t lane = threadIdx.x & 31;
        uint32_t base = 0;
        if ((int)lane == leader) base = atomicAdd(&cursor[L], (uint32_t)__popc(grp));
        base = __shfl_sync(grp, base, leader);
        idx = base + __popc(grp & ((1u << lane) - 1u));
    } else {
        idx = (uint32_t)i;
    }
    uint32_t sp = plan.span_lo[L + 1] - 1;
    while (sp > plan.span_lo[L] && plan.spans[sp].first > idx) sp--;
    const BulkSpan span = plan.spans[sp];
    const SegDesc sd = segs[span.seg];
    const uint32_t row = span.row0 + (idx - span.first);
    const uint32_t* c = reinterpret_cast<const uint32_t*>(codes + i * kMaxBytes);
    for (uint32_t w = 0; w < sd.words; w++) {
        uint32_t v = c[w];
        if (4 * w + 4 > L) v &= (1u << (8 * (L - 4 * w))) - 1u;  // bytes beyond the code's length are never stored
        sd.planes[(size_t)w * sd.cap + row] = v;
    }
    if (key_bytes == 8) {
        sd.khi[row] = reinterpret_cast<const uint64_t*>(keys)[i];
    } else {
        const uint8_t* kb = keys + i * 16;
        uint64_t hi = 0, lo = 0;
        for (int b = 0; b < 8; b++) { hi = (hi << 8) | kb[b]; lo = (lo << 8) | kb[8 + b]; }
        sd.khi[row] = hi; sd.klo[row] = lo;
    }
}

// ---------------------------------------------------------------------------------------------
// Synthetic rows of SURVEY.md 8d on the device (definition: iscc_search_b200/synth.py; the CPU checker regenerates
// the same rows): word w of row i = splitmix64(seed ^ (4i + w)), length = lengths[mix(i) % n_lengths], key = bijective
// mix of i (key_mode 0, uint64) or the chunk pointer asset8|offset4|size4 as 16 big-endian bytes (key_mode 1).
// 1 B rows never cross PCIe: they are generated next to the store and appended with isx_add_device.
struct SynthParams {
    uint64_t seed, start;
    uint8_t lengths[8];
    uint32_t n_lengths, key_mode, cpa, dup_every, dup_back;
};
__device__ __forceinline__ uint64_t splitmix64_dev(uint64_t x) {
    uint64_t z = x + 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
__global__ void k_synth_rows(const __grid_constant__ SynthParams g, size_t n, uint8_t* keys, uint8_t* codes, uint8_t* lens) {
    const size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const uint64_t i = g.start + j;
    const uint32_t L = g.lengths[g.n_lengths > 1 ? (uint32_t)(splitmix64_dev(i ^ (g.seed + 0x1234567ull)) % g.n_lengths) : 0u];
    const uint64_t src = (g.dup_every && i % g.dup_every == g.dup_every - 1 && i >= g.dup_back) ? i - g.dup_back : i;
    uint64_t w[4];
#pragma unroll
    for (int k = 0; k < 4; k++) {
        uint64_t v = splitmix64_dev(g.seed ^ (src * 4 + k));
        const uint32_t lo = 8u * k;
        if (L <= lo) v = 0;
        else if (L < lo + 8) v &= (1ull << (8 * (L - lo))) - 1ull;
        w[k] = v;
    }
    uint4* c = reinterpret_cast<uint4*>(codes + j * kMaxBytes);
    c[0] = make_uint4((uint32_t)w[0], (uint32_t)(w[0] >> 32), (uint32_t)w[1], (uint32_t)(w[1] >> 32));
    c[1] = make_uint4((uint32_t)w[2], (uint32_t)(w[2] >> 32), (uint32_t)w[3], (uint32_t)(w[3] >> 32));
    if (lens) lens[j] = (uint8_t)L;
    const uint64_t kc = g.seed * 0x51ED27ull + 0xA5A5A5A5ull;
    if (g.key_mode == 0) {
        reinterpret_cast<uint64_t*>(keys)[j] = splitmix64_dev(i ^ kc);
    } else {
        const uint64_t hi = splitmix64_dev((i / g.cpa) ^ kc);
        const uint64_t lo = ((uint64_t)((uint32_t)(i % g.cpa) * 4096u) << 32) | 4096u;
        uint8_t* kb = keys + j * 16;
#pragma unroll
        for (int b = 0; b < 8; b++) { kb[b] = (uint8_t)(hi >> (56 - 8 * b)); kb[8 + b] = (uint8_t)(lo >> (56 - 8 * b)); }
    }
}

// Row moves of a batch of swap-removes: move[i] = (dst seg, dst row, src seg, src row). The host resolves chains
// (a row moved into a hole that is removed later in the same batch) to NET moves first: every source is a row beyond the
// bucket's final size, every destination a live row below it, so the moves are independent - one warp each, lane w
// copies word w, lanes 8 and 9 the key halves. A bulk update of 10^5 assets is one launch of 10^5 warps.
__global__ void k_move_rows(const SegDesc* segs, const uint4* moves, size_t n) {
    const size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t lane = threadIdx.x & 31;
    if (i >= n) return;
    const uint4 mv = moves[i];
    const SegDesc d = segs[mv.x], s = segs[mv.z];
    if (lane < d.words) d.planes[(size_t)lane * d.cap + mv.y] = s.planes[(size_t)lane * s.cap + mv.w];
    if (lane == 8) d.khi[mv.y] = s.khi[mv.w];
    if (lane == 9 && d.klo) d.klo[mv.y] = s.klo[mv.w];
}

// Simprint grouping on the device (SURVEY 8f row 2): per query, flag the FIRST (= best, lists are sorted) record of
// every asset, asset = high 8 bytes of the 128-bit composite key (usearch_core.py:187-196 keeps exactly that record
// per (asset, query)). One CTA per query, open-addressing table in shared memory: slot -> (asset, smallest index).
__global__ void k_first_per_asset(const uint64_t* khi, const uint32_t* cnt, uint32_t k, uint32_t H, uint8_t* first) {
    extern __shared__ uint4 smem_raw[];
    unsigned long long* s_asset = reinterpret_cast<unsigned long long*>(smem_raw);  // [H], ~0 = empty slot
    uint32_t* s_min = reinterpret_cast<uint32_t*>(s_asset + H);                      // [H]
    __shared__ uint32_t s_all_ones_min;  // the one asset id that collides with the empty marker is tracked apart
    const uint32_t q = blockIdx.x, n = min(cnt[q], k), mask = H - 1;
    const uint64_t* kq = khi + (size_t)q * k;
    for (uint32_t i = threadIdx.x; i < H; i += blockDim.x) { s_asset[i] = ~0ull; s_min[i] = 0xffffffffu; }
    if (threadIdx.x == 0) s_all_ones_min = 0xffffffffu;
    __syncthreads();
    for (uint32_t j = threadIdx.x; j < n; j += blockDim.x) {
        const unsigned long long a = kq[j];
        if (a == ~0ull) { atomicMin(&s_all_ones_min, j); continue; }
        uint32_t h = (uint32_t)((a * 0x9E3779B97F4A7C15ull) >> 40) & mask;
        for (;;) {
            const unsigned long long prev = atomicCAS(&s_asset[h], ~0ull, a);
            if (prev == ~0ull || prev == a) { atomicMin(&s_min[h], j); break; }
            h = (h + 1) & mask;
        }
    }
    __syncthreads();
    for (uint32_t j = threadIdx.x; j < k; j += blockDim.x) {
        uint8_t f = 0;
        if (j < n) {
            const unsigned long long a = kq[j];
            if (a == ~0ull) f = (s_all_ones_min == j);
            else {
                uint32_t h = (uint32_t)((a * 0x9E3779B97F4A7C15ull) >> 40) & mask;
                while (s_asset[h] != a) h = (h + 1) & mask;
                f = (s_min[h] == j);
            }
        }
        first[(size_t)q * k + j] = f;
    }
}

// ---------------------------------------------------------------------------------------------
// Simprint asset scoring (SURVEY 8f row 2): the IDF-weighted similarity of usearch_core.py:199-269 as a segmented
// reduce. Input: the best record of every (asset, query simprint) pair, grouped by asset, ascending query index inside
// an asset - rec_qi / rec_sim / rec_idf, segment a = records [seg[a], seg[a+1]). One thread per asset walks its segment
// in order and then the query simprints the asset did NOT match, exactly the order in which the reference's Python
// adds the terms; every operation is an explicitly rounded IEEE double (__dadd_rn / __dmul_rn / __ddiv_rn: no FMA
// contraction), so the scores are bit-identical to the reference's floats.
__global__ void k_score_segments(const uint32_t* __restrict__ seg, const uint32_t* __restrict__ rec_qi, const double* __restrict__ rec_sim,
                                 const double* __restrict__ rec_idf, const double* __restrict__ q_idf, uint32_t n_assets, uint32_t S,
                                 double* __restrict__ score) {
    const uint32_t a = blockIdx.x * blockDim.x + threadIdx.x;
    if (a >= n_assets) return;
    const uint32_t lo = seg[a], hi = seg[a + 1];
    double total = 0.0, weighted = 0.0;
    for (uint32_t i = lo; i < hi; i++) {          // matched query simprints, ascending query index
        const double idf = rec_idf[i];
        total = __dadd_rn(total, idf);
        weighted = __dadd_rn(weighted, __dmul_rn(idf, rec_sim[i]));
    }
    uint32_t i = lo;
    for (uint32_t q = 0; q < S; q++) {            // then every query simprint without a match (coverage penalty)
        if (i < hi && rec_qi[i] == q) { i++; continue; }
        total = __dadd_rn(total, q_idf[q]);
    }
    score[a] = total > 0.0 ? __ddiv_rn(weighted, total) : 0.0;
}

// queries (device, caller order) -> group order: dst[i] = src[order[i]], 32 bytes per query, bytes beyond the
// query's length zeroed (8 threads per query, one word each)
__global__ void k_gather_queries(const uint32_t* src, const uint32_t* order, const uint8_t* qlens_sorted, uint32_t* dst, uint32_t Q) {
    uint32_t i = (blockIdx.x * blockDim.x + threadIdx.x) >> 3, w = threadIdx.x & 7;
    if (i >= Q) return;
    uint32_t v = src[(size_t)order[i] * 8 + w];
    const uint32_t L = qlens_sorted[i];
    if (4 * w >= L) v = 0;
    else if (4 * w + 4 > L) v &= (1u << (8 * (L - 4 * w))) - 1u;
    dst[(size_t)i * 8 + w] = v;
}

// candidate list -> (key, h, nbits) records, list order (used by the unbounded match-all mode)
__global__ void k_gather_cands(const SegDesc* segs, const uint64_t* cand, uint32_t n, uint32_t qlen_bytes, uint64_t* khi,
                               uint64_t* klo, uint16_t* hh, uint16_t* nn) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint64_t c = cand[i];
    const SegDesc& sd = segs[cand_seg(c)];
    khi[i] = sd.khi[cand_row(c)];
    klo[i] = sd.klo ? sd.klo[cand_row(c)] : 0ull;
    hh[i] = (uint16_t)cand_h(c);
    nn[i] = (uint16_t)(8u * min(qlen_bytes, sd.len_bytes));
}

// loc[i] = (segment << 32) | row or ~0; out: 32-byte zero padded rows
__global__ void k_gather_rows(const SegDesc* segs, const uint64_t* loc, uint8_t* out, size_t n) {
    size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 3;
    uint32_t w = threadIdx.x & 7;
    if (i >= n) return;
    uint64_t d = loc[i];
    uint32_t v = 0;
    if (d != ~0ull) {
        const SegDesc sd = segs[(uint32_t)(d >> 32)];
        if (w < sd.words) v = sd.planes[(size_t)w * sd.cap + (uint32_t)d];
    }
    reinterpret_cast<uint32_t*>(out)[i * 8 + w] = v;
}

}  // namespace isx
