// tc.cuh - the batch scan on the tensor cores: exact Hamming distances with tcgen05 int8 MMA (sm_100a).
//
// Rows are expanded to 0/1 bytes (a), queries to +-1 bytes (b' = 1 - 2b, 0 past the compared length). Over the compared
// bits acc = sum a * b' = popc(a) - 2 popc(a & b), so h = popc(a ^ b) = acc + popc(b[:m]): an int8 MMA with int32
// accumulators, exact. One 32-bit plane word is one K = 32 step of tcgen05.mma.kind::i8, a WE-word compare is WE MMAs per
// (128-row x N-query) tile. The bit order inside a word is free as long as rows and queries share it: K byte 4j + i of a
// word holds bit 8i + j, i.e. the 32 bytes of a word are the eight u32 (w >> j) & 0x01010101, j = 0..7.
//
// k_scan_tc keeps the contract of k_scan (ScanParams, block range of one bucket, running thresholds re-read at item
// boundaries with the same ramp, histograms, stage, candidate lists, overflow flags, threshold feedback); only the
// per-pair arithmetic moves from the POPC pipe to the tensor core. A pair passes when acc <= t_q = bound_q - popc(q[:m]).
#pragma once
#include "kernels.cuh"
#include "small.cuh"   // smem_u32, mbarrier primitives

namespace isx {

// ---- encoding (host and device: isx_selftest_distance checks it against a naive popcount) ---------------------------
// u32 j (0..7) of the 32 row bytes of word w: byte i = bit 8i + j of w, as 0/1
__host__ __device__ __forceinline__ uint32_t tc_row_bytes(uint32_t w, int j) { return (w >> j) & 0x01010101u; }
// the same for a query word of which only the low `nbits` bits are compared: byte i = 1 - 2 * bit (+1 / -1 as s8), 0 past nbits
__host__ __device__ __forceinline__ uint32_t tc_query_bytes(uint32_t w, int j, uint32_t nbits) {
    uint32_t valid = 0;
    for (int i = 0; i < 4; i++)
        if ((uint32_t)(8 * i + j) < nbits) valid |= 1u << (8 * i);
    return valid | (tc_row_bytes(w, j) & valid) * 0xfeu;
}
__host__ __device__ __forceinline__ uint32_t tc_word_bits(uint32_t m, uint32_t w) {   // compared bits of word w at length m
    const int b = 8 * (int)m - 32 * (int)w;
    return b <= 0 ? 0u : b >= 32 ? 32u : (uint32_t)b;
}
__host__ __device__ __forceinline__ uint32_t tc_hamming(int32_t acc, uint32_t popc_q) { return (uint32_t)(acc + (int32_t)popc_q); }

// ---- tcgen05 plumbing -----------------------------------------------------------------------------------------------
constexpr int kTcRows = 128;        // MMA M: rows per tile = TMEM lanes
constexpr int kTcMaxN = 256;        // MMA N: queries per CTA
constexpr int kTcMinBlocksPerSm = 2;

// operands are K-major without swizzle: 8 x 16-byte core matrices, K-adjacent ones 128 B apart (LBO), 8-row groups
// 8 * KB apart (SBO), KB = 32 * WE bytes per row. Byte kb of row r sits at tc_off(r, kb).
__host__ __device__ __forceinline__ uint32_t tc_off(uint32_t r, uint32_t kb, uint32_t KB) {
    return (r >> 3) * (8 * KB) + (kb >> 4) * 128 + (r & 7) * 16 + (kb & 15);
}

__device__ __forceinline__ uint64_t tc_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
    return (uint64_t)((saddr & 0x3ffffu) >> 4) | ((uint64_t)(lbo >> 4) << 16) | ((uint64_t)(sbo >> 4) << 32) | (1ull << 46);
}
// kind::i8 instruction descriptor: D s32, A and B s8, both K-major, N x M
__device__ __forceinline__ uint32_t tc_idesc(uint32_t n) {
    return (2u << 4) | (1u << 7) | (1u << 10) | ((n >> 3) << 17) | ((uint32_t)(kTcRows >> 4) << 24);
}
__device__ __forceinline__ void tc_mma(uint32_t tmem_d, uint64_t a, uint64_t b, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
                 :: "r"(tmem_d), "l"(a), "l"(b), "r"(idesc), "r"(accumulate));
}
__device__ __forceinline__ void tc_commit(uint64_t* mbar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(smem_u32(mbar)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// 32 consecutive accumulator columns of this thread's TMEM lane; the wait is tied to the registers so no use moves above it
// (the micro-benchmark's 32-bit reference for tmem_ld32_pack16)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
                 "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                   "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
                   "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
                   "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                 : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]),
                   "+r"(v[8]), "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15]),
                   "+r"(v[16]), "+r"(v[17]), "+r"(v[18]), "+r"(v[19]), "+r"(v[20]), "+r"(v[21]), "+r"(v[22]), "+r"(v[23]),
                   "+r"(v[24]), "+r"(v[25]), "+r"(v[26]), "+r"(v[27]), "+r"(v[28]), "+r"(v[29]), "+r"(v[30]), "+r"(v[31])
                 :: "memory");
}
// the same 32 columns as 16-bit values, two per register: v[i] holds the low 16 bits of column 2i in its low half and of
// column 2i + 1 in its high half. Asynchronous: no use of v before tmem_wait_ld(v). The memory clobber keeps the load
// where it is issued, ahead of the shared-memory reads of the compare it is meant to overlap.
__device__ __forceinline__ void tmem_ld32_pack16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.pack::16b.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                   "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                 : "r"(taddr) : "memory");
}
// waits for every TMEM load this thread issued; tied to v so that no use of v moves above it
__device__ __forceinline__ void tmem_wait_ld(uint32_t (&v)[16]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]),
                   "+r"(v[8]), "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15])
                 :: "memory");
}
__device__ __forceinline__ uint32_t ld_nc_u32(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}

// TMEM columns a CTA allocates for N query columns (a power of two >= 32)
__host__ __device__ constexpr uint32_t tc_tmem_cols(uint32_t n) { return n <= 32 ? 32u : n <= 64 ? 64u : n <= 128 ? 128u : 256u; }
__host__ __device__ constexpr uint32_t tc_round32(uint32_t n) { return (n + 31u) & ~31u; }
// shared memory of k_scan_tc before the stage: A tile | B (queries) | t_q | popc_q | mbarrier + TMEM slot | s_rank | s_hrow
__host__ __device__ constexpr size_t tc_smem_bytes(uint32_t we, uint32_t q_split, uint32_t R) {
    return (size_t)kTcRows * 32 * we + (size_t)tc_round32(q_split) * 32 * we + (size_t)tc_round32(q_split) * 8 + 16 + 258 * 2 +
           ((size_t)R + 2) * 2;
}

// one passing pair of the tensor-core scan, by one thread: the same record as k_scan, through the stage
__device__ __noinline__ void tc_emit(const ScanParams& p, uint32_t q, uint32_t h, uint32_t seg, uint32_t row, const uint16_t* s_rank) {
    const uint64_t rec = pack_cand(s_rank[h], h, seg, row);
    if (p.stage_cap) stage_push(p, stage_of(p, s_rank), q, rec);
    else stage_direct(p, q, rec);   // no room for a stage: straight to HBM
}

// The compare epilogue of one tile for one thread: its TMEM lane (taddr: lane << 16, column 0), 32-column chunks
// c = c0, c0 + 2, ... < nc. s_nt holds -t_q as s16, two columns per u32 in the order of tmem_ld32_pack16, so one
// VIADDMNMX.S16x2 takes min(m, acc - t_q) of two pairs; four independent minima per chunk, and the load of the warp's next
// chunk is in flight while a chunk is compared. on_pass(c, v) runs in the live lanes with acc <= t_q in some column of
// chunk c, after every TMEM load of the thread has completed.
// No 16-bit sum wraps: |acc| <= 256 (at most 256 compared bits), |t_q| <= 256 (0 <= hmax <= 8m and 0 <= popc(q) <= 8m,
// m <= 32), and padding columns (acc = 0) hold -t = 0x4000.
template <typename OnPass>
__device__ __forceinline__ void tc_compare_tile(uint32_t taddr, uint32_t c0, uint32_t nc, const uint32_t* s_nt, bool live,
                                                OnPass&& on_pass) {
    uint32_t va[16], vb[16];
    auto compare = [&](uint32_t c, uint32_t (&cur)[16], uint32_t (&nxt)[16], bool next_in_flight) {
        const uint4* nt = reinterpret_cast<const uint4*>(s_nt + c * 16);
        uint32_t m0 = 0x7fff7fffu, m1 = 0x7fff7fffu, m2 = 0x7fff7fffu, m3 = 0x7fff7fffu;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const uint4 t = nt[j];
            m0 = __viaddmin_s16x2(cur[4 * j], t.x, m0);
            m1 = __viaddmin_s16x2(cur[4 * j + 1], t.y, m1);
            m2 = __viaddmin_s16x2(cur[4 * j + 2], t.z, m2);
            m3 = __viaddmin_s16x2(cur[4 * j + 3], t.w, m3);
        }
        const uint32_t mn = __vimin3_s16x2(m0, m1, __vmins2(m2, m3));
        const bool hit = live && min((int32_t)(int16_t)mn, (int32_t)mn >> 16) <= 0;
        if (__any_sync(0xffffffffu, hit)) {   // rare
            if (next_in_flight) tmem_wait_ld(nxt);   // warp-uniform; no call is made with a TMEM load in flight
            if (hit) on_pass(c, cur);
        }
    };
    if (c0 >= nc) return;
    tmem_ld32_pack16(taddr + c0 * 32, va);
    tmem_wait_ld(va);
    // Two chunks per iteration, so that the buffers swap without copies. The __syncwarp() after each load keeps it where
    // it is: without it ptxas schedules the load after the compare it should overlap, next to the vote.
    for (uint32_t c = c0;; c += 4) {
        const bool b_next = c + 2 < nc;
        if (b_next) tmem_ld32_pack16(taddr + (c + 2) * 32, vb);
        __syncwarp();
        compare(c, va, vb, b_next);
        if (!b_next) return;
        tmem_wait_ld(vb);
        const bool a_next = c + 4 < nc;
        if (a_next) tmem_ld32_pack16(taddr + (c + 4) * 32, va);
        __syncwarp();
        compare(c + 2, vb, va, a_next);
        if (!a_next) return;
        tmem_wait_ld(va);
    }
}

// WE: words compared per pair (1..8). One CTA = one query sub-tile of <= 256 queries (gridDim.y) x a contiguous share of
// the launch's blocks (gridDim.x). Per 128-row tile: all 8 warps expand the rows into shared memory, one thread issues WE
// MMAs into the TMEM accumulator and commits them to an mbarrier while the next tile's words are fetched, then every warp
// reads its 32 TMEM lanes (warps w and w + 4 split the columns) as packed 16-bit values, compares two accumulators per
// instruction with their queries' t_q (tc_compare_tile) and takes the rare emit path when some lane passes. Two CTAs per
// SM overlap one's MMA with the other's epilogue.
template <int WE>
__global__ void __launch_bounds__(kThreads, kTcMinBlocksPerSm) k_scan_tc(const __grid_constant__ ScanParams p) {
    constexpr uint32_t KB = 32 * WE;                      // K bytes per row
    constexpr int PER = (kTcRows * WE + kThreads - 1) / kThreads;   // plane words a thread expands per tile
    extern __shared__ __align__(1024) uint8_t smem_tc[];
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t q0 = blockIdx.y * p.q_split;
    const uint32_t T = min(p.q_split, p.T - q0);
    const uint32_t N = tc_round32(T);                     // MMA N (multiple of 32 <= 256)
    const uint32_t NB = tc_round32(p.q_split);            // B rows reserved (same for every CTA of the launch)
    uint8_t* sA = smem_tc;
    uint8_t* sB = sA + kTcRows * KB;
    uint32_t* s_nt = reinterpret_cast<uint32_t*>(sB + (size_t)NB * KB);   // -t_q, packed (tc_compare_tile); NB / 2 used
    uint32_t* s_pq = s_nt + NB;
    uint64_t* mbar = reinterpret_cast<uint64_t*>(s_pq + NB);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(mbar + 1);
    uint16_t* s_rank = reinterpret_cast<uint16_t*>(tmem_slot + 2);
    uint16_t* s_hrow = s_rank + 258;

    const uint32_t seg_len = p.segs[p.blocks[p.block_begin].x].len_bytes;
    const uint32_t m = min(p.qlen_bytes, seg_len);

    // queries -> +-1 bytes (0 past 8m bits and for padding columns), popc of the compared bits
    for (uint32_t i = tid; i < N * WE; i += kThreads) {
        const uint32_t q = i / WE, w = i % WE;
        const uint32_t nb = q < T ? tc_word_bits(m, w) : 0u;
        const uint32_t v = q < T ? p.queries[(size_t)(q0 + q) * 8 + w] : 0u;
        uint4* dst = reinterpret_cast<uint4*>(sB + tc_off(q, 32 * w, KB));
        dst[0] = make_uint4(tc_query_bytes(v, 0, nb), tc_query_bytes(v, 1, nb), tc_query_bytes(v, 2, nb), tc_query_bytes(v, 3, nb));
        dst[8] = make_uint4(tc_query_bytes(v, 4, nb), tc_query_bytes(v, 5, nb), tc_query_bytes(v, 6, nb), tc_query_bytes(v, 7, nb));
    }
    for (uint32_t q = tid; q < N; q += kThreads) {
        uint32_t c = 0;
        if (q < T)
            for (int w = 0; w < WE; w++) {
                const uint32_t nb = tc_word_bits(m, w);
                c += popc32(p.queries[(size_t)(q0 + q) * 8 + w] & (nb >= 32 ? 0xffffffffu : (1u << nb) - 1u));
            }
        s_pq[q] = c;
    }
    for (uint32_t i = tid; i < 257; i += kThreads) s_rank[i] = p.rank_tab[m * 257 + i];
    for (uint32_t i = tid; i < p.R; i += kThreads) s_hrow[i] = p.hmax_tab[(size_t)m * p.R + i];
    if (p.stage_cap && tid < 4) stage_of(p, s_rank).counters[tid] = 0;
    if (tid == 0) {
        mbar_init(mbar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    fence_async_smem();
    const uint32_t ncols = tc_tmem_cols(N);
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(tmem_slot)), "r"(ncols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    const uint32_t idesc = tc_idesc(N);
    const uint32_t a_addr = smem_u32(sA), b_addr = smem_u32(sB);
    const uint32_t lane_base = (warp & 3) * 32;           // the TMEM lanes this warp may read
    const uint32_t col0 = warp >> 2;                      // first 32-column chunk (warps w and w + 4 alternate)
    uint32_t phase = 0;

    const uint32_t n_blocks = p.block_end - p.block_begin;
    const uint32_t my_lo = p.block_begin + (uint32_t)((uint64_t)n_blocks * blockIdx.x / gridDim.x);
    const uint32_t my_hi = p.block_begin + (uint32_t)((uint64_t)n_blocks * (blockIdx.x + 1) / gridDim.x);
    constexpr uint32_t kTiles = kRowsPerStep / kTcRows;    // 128-row tiles per block

    auto load_tile = [&](uint32_t ti, uint32_t (&v)[PER]) {
        const uint2 blk = p.blocks[ti / kTiles];
        const SegDesc* sd = p.segs + blk.x;
        const uint32_t* base = sd->planes + blk.y + (ti % kTiles) * kTcRows;
        const uint32_t cap = sd->cap;
#pragma unroll
        for (int k = 0; k < PER; k++) {
            const uint32_t i = tid + kThreads * k;
            if (i < kTcRows * WE) v[k] = ld_nc_u32(base + (size_t)(i / kTcRows) * cap + (i % kTcRows));
        }
    };

    uint32_t item_blocks = p.update_tau ? 1u : p.blocks_per_item;
    for (uint32_t b_lo = my_lo; b_lo < my_hi;) {
        const uint32_t b_hi = min(b_lo + item_blocks, my_hi);
        __syncthreads();   // the previous item's readers of s_nt are done, its candidates are staged
        if (p.stage_cap) stage_flush(p, s_rank);
        for (uint32_t i = tid; i < N / 2; i += kThreads) {
            uint32_t w = 0;
            for (uint32_t hf = 0; hf < 2; hf++) {
                const uint32_t q = 2 * i + hf;
                const int32_t nt = q < T ? (int32_t)s_pq[q] - (int32_t)s_hrow[__ldcg(&p.tau[q0 + q])] : 0x4000;   // padding never passes
                w |= ((uint32_t)nt & 0xffffu) << (16 * hf);
            }
            s_nt[i] = w;
        }
        __syncthreads();

        uint32_t v[PER];
        load_tile(b_lo * kTiles, v);
        for (uint32_t ti = b_lo * kTiles; ti < b_hi * kTiles; ti++) {
#pragma unroll
            for (int k = 0; k < PER; k++) {
                const uint32_t i = tid + kThreads * k;
                if (i < kTcRows * WE) {
                    const uint32_t r = i % kTcRows, w = i / kTcRows;
                    uint4* dst = reinterpret_cast<uint4*>(sA + tc_off(r, 32 * w, KB));
                    dst[0] = make_uint4(tc_row_bytes(v[k], 0), tc_row_bytes(v[k], 1), tc_row_bytes(v[k], 2), tc_row_bytes(v[k], 3));
                    dst[8] = make_uint4(tc_row_bytes(v[k], 4), tc_row_bytes(v[k], 5), tc_row_bytes(v[k], 6), tc_row_bytes(v[k], 7));
                }
            }
            fence_async_smem();
            __syncthreads();   // A tile written; every lane's TMEM reads of the previous tile are complete
            if (tid == 0) {
                tc_fence_after();
#pragma unroll
                for (int s = 0; s < WE; s++)
                    tc_mma(tmem, tc_desc(a_addr + 256 * s, 128, 8 * KB), tc_desc(b_addr + 256 * s, 128, 8 * KB), idesc, s > 0);
                tc_commit(mbar);
            }
            if (ti + 1 < b_hi * kTiles) load_tile(ti + 1, v);   // lands while the MMA and this tile's epilogue run
            mbar_wait(mbar, phase);
            phase ^= 1;
            tc_fence_after();

            const uint2 blk = p.blocks[ti / kTiles];
            const uint32_t row = blk.y + (ti % kTiles) * kTcRows + lane_base + lane;
            const bool live = row < p.segs[blk.x].n;           // padding rows of the last block never emit
            tc_compare_tile(tmem + (lane_base << 16), col0, N / 32, s_nt, live, [&](uint32_t c, const uint32_t (&v)[16]) {
#pragma unroll
                for (int i = 0; i < 16; i++) {   // unrolled: v stays in registers
                    const uint32_t nt = s_nt[c * 16 + i];
#pragma unroll
                    for (int hf = 0; hf < 2; hf++) {   // sign-extend each half: the exact acc and -t_q
                        const int32_t acc = hf ? (int32_t)v[i] >> 16 : (int32_t)(int16_t)v[i];
                        const int32_t neg_t = hf ? (int32_t)nt >> 16 : (int32_t)(int16_t)nt;
                        const uint32_t q = c * 32 + 2 * i + hf;
                        if (acc + neg_t <= 0) tc_emit(p, q0 + q, tc_hamming(acc, s_pq[q]), blk.x, row, s_rank);
                    }
                }
            });
            tc_fence_before();
        }
        b_lo = b_hi;
        item_blocks = min(item_blocks * 2, p.blocks_per_item);
    }
    __syncthreads();
    if (p.stage_cap) stage_flush(p, s_rank);
    if (warp == 0) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem), "r"(ncols) : "memory");
    }
}

}  // namespace isx
