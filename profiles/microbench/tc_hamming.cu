// Micro-benchmark of the tensor-core Hamming scan's three stages on B200 (sm_100a), with the very helpers of
// iscc_search_b200/csrc/tc.cuh:
//   * correctness: one 128-row x 256-query tile at every word count WE = 1..8 and a byte-granular length, against a naive
//     popcount (h = acc + popc(q[:m]) for every pair); and the packed read the kernel's epilogue uses
//     (tcgen05.ld.32x32b.x16.pack::16b) against the low 16 bits of the 32-bit read, column for column
//   * MMA: tcgen05.mma.kind::i8 M=128 N=256 K=32 issued back to back by one thread into one accumulator, one CTA per SM
//   * epilogue, s32: tcgen05.ld.32x32b.x32 + one compare-and-min per value on one chain + vote (the kernel's epilogue
//     before the packed compare), 8 warps (columns split) and 4
//   * epilogue, s16x2: tc_compare_tile of tc.cuh, the kernel's epilogue (packed reads, two pairs per VIADDMNMX.S16x2,
//     four chains, next chunk in flight), 8 warps
//   * expansion: plane words -> 0/1 bytes in the K-major shared-memory layout
// Both epilogues also run with 2 CTAs per SM, as k_scan_tc does (the line says on how many SMs the two CTAs' timed
// regions overlapped). Rates are per SM per clock: each CTA records its SM and its start and end clock, an SM's time is
// its span from the first start to the last end. The SM clock is read from
// the device (cudaDevAttrClockRate); the card's power limit and current clocks are read by nvidia-smi in the same run.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -o tc_hamming tc_hamming.cu
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <vector>

#include "../../iscc_search_b200/csrc/tc.cuh"

using namespace isx;
#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e), __FILE__, __LINE__); exit(1);} } while (0)

constexpr int kN = 256;

// shared memory: A [128][KB] | B [256][KB] | mbarrier | TMEM slot | s32 bounds [256] | packed s16 bounds [128]
template <int WE>
__global__ void __launch_bounds__(256, 2) k_tile(const uint32_t* rows, const uint32_t* queries, uint32_t m, int32_t* out, int mode,
                                                 int iters, unsigned long long* clk) {
    constexpr uint32_t KB = 32 * WE;
    extern __shared__ __align__(1024) uint8_t sm[];
    uint8_t* sA = sm;
    uint8_t* sB = sA + 128 * KB;
    uint64_t* mbar = reinterpret_cast<uint64_t*>(sB + kN * KB);
    uint32_t* slot = reinterpret_cast<uint32_t*>(mbar + 1);
    int32_t* s_t = reinterpret_cast<int32_t*>(slot + 2);
    uint32_t* s_nt = reinterpret_cast<uint32_t*>(s_t + kN);
    const uint32_t tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    for (uint32_t i = tid; i < kN * WE; i += 256) {
        const uint32_t q = i / WE, w = i % WE, nb = tc_word_bits(m, w), v = queries[q * 8 + w];
        uint4* d = reinterpret_cast<uint4*>(sB + tc_off(q, 32 * w, KB));
        d[0] = make_uint4(tc_query_bytes(v, 0, nb), tc_query_bytes(v, 1, nb), tc_query_bytes(v, 2, nb), tc_query_bytes(v, 3, nb));
        d[8] = make_uint4(tc_query_bytes(v, 4, nb), tc_query_bytes(v, 5, nb), tc_query_bytes(v, 6, nb), tc_query_bytes(v, 7, nb));
    }
    for (uint32_t i = tid; i < kN; i += 256) s_t[i] = -1000 - (int32_t)i;   // nothing passes: the vote path only
    for (uint32_t i = tid; i < kN / 2; i += 256) s_nt[i] = (1000u + 2 * i) | (1001u + 2 * i) << 16;   // the same, as -t in s16
    auto expand = [&](uint32_t salt) {
        for (uint32_t i = tid; i < 128 * WE; i += 256) {
            const uint32_t r = i % 128, w = i / 128, v = rows[r * 8 + w] ^ salt;
            uint4* d = reinterpret_cast<uint4*>(sA + tc_off(r, 32 * w, KB));
            d[0] = make_uint4(tc_row_bytes(v, 0), tc_row_bytes(v, 1), tc_row_bytes(v, 2), tc_row_bytes(v, 3));
            d[8] = make_uint4(tc_row_bytes(v, 4), tc_row_bytes(v, 5), tc_row_bytes(v, 6), tc_row_bytes(v, 7));
        }
    };
    expand(0);
    if (tid == 0) { mbar_init(mbar, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
    fence_async_smem();
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(slot)), "r"(256) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *slot;
    const uint32_t idesc = tc_idesc(kN), a = smem_u32(sA), b = smem_u32(sB);
    uint32_t phase = 0;
    auto mma_tile = [&](int reps) {
        if (tid == 0) {
            tc_fence_after();
            for (int r = 0; r < reps; r++)
#pragma unroll
                for (int s = 0; s < WE; s++) tc_mma(tmem, tc_desc(a + 256 * s, 128, 8 * KB), tc_desc(b + 256 * s, 128, 8 * KB), idesc, s > 0);
            tc_commit(mbar);
        }
        mbar_wait(mbar, phase);
        phase ^= 1;
        tc_fence_after();
    };
    const uint32_t lane_base = (warp & 3) * 32;
    int32_t sink = 0x7fffffff;
    auto epilogue = [&](uint32_t first_warp_half, uint32_t step) {
        for (uint32_t c = first_warp_half; c < kN / 32; c += step) {
            uint32_t acc[32];
            tmem_ld32(tmem + (lane_base << 16) + c * 32, acc);
            const int4* tq = reinterpret_cast<const int4*>(s_t + c * 32);
            int32_t mn = 0x7fffffff;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const int4 t = tq[j];
                mn = min(mn, (int32_t)acc[4 * j] - t.x); mn = min(mn, (int32_t)acc[4 * j + 1] - t.y);
                mn = min(mn, (int32_t)acc[4 * j + 2] - t.z); mn = min(mn, (int32_t)acc[4 * j + 3] - t.w);
            }
            if (__any_sync(0xffffffffu, mn <= 0)) sink = min(sink, mn);
        }
    };
    __syncthreads();
    unsigned long long t0 = clock64();
    if (mode == 0) {                      // correctness: one tile, every accumulator out, then the packed read of it
        mma_tile(1);
        for (uint32_t c = 0; c < kN / 32; c++) {
            if ((warp >> 2) != (c & 1)) continue;
            uint32_t acc[32], v[16];
            tmem_ld32(tmem + (lane_base << 16) + c * 32, acc);
#pragma unroll
            for (int j = 0; j < 32; j++) out[(lane_base + lane) * kN + c * 32 + j] = (int32_t)acc[j];
            tmem_ld32_pack16(tmem + (lane_base << 16) + c * 32, v);
            tmem_wait_ld(v);
#pragma unroll
            for (int j = 0; j < 16; j++) out[128 * kN + (lane_base + lane) * (kN / 2) + c * 16 + j] = (int32_t)v[j];
        }
    } else if (mode == 1) {               // MMA rate
        mma_tile(iters);
    } else if (mode == 2 || mode == 3) {  // s32 epilogue rate, 8 warps (columns split) or 4 warps (all columns)
        mma_tile(1);
        for (int it = 0; it < iters; it++)
            if (mode == 2) epilogue(warp >> 2, 2);
            else if (warp < 4) epilogue(0, 1);
    } else if (mode == 5) {               // s16x2 epilogue rate (tc_compare_tile), 8 warps
        mma_tile(1);
        for (int it = 0; it < iters; it++)
            tc_compare_tile(tmem + (lane_base << 16), warp >> 2, kN / 32, s_nt, true,
                            [&](uint32_t c, const uint32_t (&v)[16]) { sink = min(sink, (int32_t)(v[0] ^ v[15] ^ c)); });
    } else {                              // expansion rate
        for (int it = 0; it < iters; it++) { expand((uint32_t)it); __syncthreads(); }
    }
    tc_fence_before();
    __syncthreads();
    unsigned long long t1 = clock64();
    if (tid == 0) {
        uint32_t smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        clk[3 * blockIdx.x] = smid;
        clk[3 * blockIdx.x + 1] = t0;
        clk[3 * blockIdx.x + 2] = t1;
    }
    if (sink == 12345) out[0] = sink;
    if (warp == 0) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem), "r"(256) : "memory");
    }
}

static uint64_t rng = 88172645463325252ull;
static uint32_t next32() { rng ^= rng << 13; rng ^= rng >> 7; rng ^= rng << 17; return (uint32_t)rng; }

template <int WE>
static bool run_we(uint32_t m, int sms, bool timing, uint32_t* d_rows, uint32_t* d_q, int32_t* d_out, unsigned long long* d_clk,
                   int clock_khz) {
    const size_t smem = 128 * 32 * WE + kN * 32 * WE + 16 + kN * 4 + kN * 2;
    CK(cudaFuncSetAttribute(k_tile<WE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    std::vector<uint32_t> rows(128 * 8), qs(kN * 8);
    for (auto& v : rows) v = next32();
    for (auto& v : qs) v = next32();
    for (int r = 0; r < 8; r++) for (int w = 0; w < 8; w++) rows[r * 8 + w] = qs[r * 8 + w] ^ (next32() & next32() & next32());
    CK(cudaMemcpy(d_rows, rows.data(), rows.size() * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_q, qs.data(), qs.size() * 4, cudaMemcpyHostToDevice));
    k_tile<WE><<<1, 256, smem>>>(d_rows, d_q, m, d_out, 0, 1, d_clk);
    CK(cudaDeviceSynchronize());
    std::vector<int32_t> out(128 * kN + 128 * kN / 2);
    CK(cudaMemcpy(out.data(), d_out, out.size() * 4, cudaMemcpyDeviceToHost));
    int bad = 0, bad16 = 0, neg = 0;
    for (int r = 0; r < 128; r++)
        for (int q = 0; q < kN; q++) {   // packed word j of a lane: column 2j in the low half, 2j + 1 in the high half
            const uint32_t w = (uint32_t)out[128 * kN + r * (kN / 2) + q / 2];
            const uint16_t half = (uint16_t)(w >> (16 * (q & 1)));
            neg += out[r * kN + q] < 0;
            if (half != (uint16_t)out[r * kN + q] && bad16++ < 3)
                printf("  packed mismatch WE=%d m=%u row %d column %d: acc %d packed half 0x%04x\n", WE, m, r, q, out[r * kN + q], half);
        }
    for (int r = 0; r < 128; r++)
        for (int q = 0; q < kN; q++) {
            uint32_t h = 0, pq = 0;
            for (int w = 0; w < WE; w++) {
                const uint32_t nb = tc_word_bits(m, w), mk = nb >= 32 ? ~0u : (1u << nb) - 1u;
                h += __builtin_popcount((rows[r * 8 + w] ^ qs[q * 8 + w]) & mk);
                pq += __builtin_popcount(qs[q * 8 + w] & mk);
            }
            if (tc_hamming(out[r * kN + q], pq) != h && bad++ < 3)
                printf("  mismatch WE=%d m=%u row %d query %d: acc %d popc_q %u naive h %u\n", WE, m, r, q, out[r * kN + q], pq, h);
        }
    printf("CHECK WE=%d m=%2u  128x%d tile: %s; packed 16-bit read: %s (%d of %d accumulators negative)\n", WE, m, kN,
           bad ? "MISMATCH" : "exact", bad16 ? "MISMATCH" : "exact", neg, 128 * kN);
    bad += bad16 + (neg == 0);   // the check must see negative accumulators
    if (!timing || bad) return bad == 0;
    auto rate = [&](int mode, int iters, int per_sm, double work_per_iter, const char* what) {
        const int ctas = sms * per_sm;
        k_tile<WE><<<ctas, 256, smem>>>(d_rows, d_q, m, d_out, mode, iters, d_clk);   // warm
        CK(cudaDeviceSynchronize());
        cudaEvent_t e0, e1;
        CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
        CK(cudaEventRecord(e0));
        k_tile<WE><<<ctas, 256, smem>>>(d_rows, d_q, m, d_out, mode, iters, d_clk);
        CK(cudaEventRecord(e1));
        CK(cudaDeviceSynchronize());
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, e0, e1));
        std::vector<unsigned long long> clk(3 * ctas);
        CK(cudaMemcpy(clk.data(), d_clk, clk.size() * 8, cudaMemcpyDeviceToHost));
        // per SM: first start, last end, latest start, earliest end (the CTAs ran together when latest start < earliest end)
        std::vector<unsigned long long> lo(sms, ~0ull), hi(sms, 0), lo_end(sms, ~0ull), hi_start(sms, 0);
        std::vector<int> n(sms, 0);
        for (int b = 0; b < ctas; b++) {
            const int s = (int)clk[3 * b];
            lo[s] = std::min(lo[s], clk[3 * b + 1]);
            hi[s] = std::max(hi[s], clk[3 * b + 2]);
            hi_start[s] = std::max(hi_start[s], clk[3 * b + 1]);
            lo_end[s] = std::min(lo_end[s], clk[3 * b + 2]);
            n[s]++;
        }
        unsigned long long span = 0;   // the slowest SM
        int together = 0;
        for (int s = 0; s < sms; s++) {
            if (n[s]) span = std::max(span, hi[s] - lo[s]);
            together += n[s] == per_sm && hi_start[s] < lo_end[s];
        }
        printf("RATE WE=%d %-40s ms=%8.3f clk/SM=%10llu  %s/SM/clk=%8.1f  (at %d MHz: %.3g /s per GPU)", WE, what, ms, span,
               mode == 1 ? "MAC" : "pairs", work_per_iter * iters * per_sm / (double)span, clock_khz / 1000,
               work_per_iter * iters * ctas / (ms * 1e-3));
        if (per_sm > 1) printf("  [%d CTAs ran together on %d of %d SMs]", per_sm, together, sms);
        printf("\n");
        CK(cudaEventDestroy(e0)); CK(cudaEventDestroy(e1));
    };
    rate(1, 4096, 1, 128.0 * kN * 32 * WE, "mma M128 N256 K32xWE");
    rate(2, 512, 1, 128.0 * kN, "epilogue s32   8 warps, 1 CTA/SM");
    rate(5, 512, 1, 128.0 * kN, "epilogue s16x2 8 warps, 1 CTA/SM");
    rate(2, 512, 2, 128.0 * kN, "epilogue s32   8 warps, 2 CTA/SM");
    rate(5, 512, 2, 128.0 * kN, "epilogue s16x2 8 warps, 2 CTA/SM");
    rate(3, 512, 1, 128.0 * kN, "epilogue s32   4 warps, 1 CTA/SM");
    rate(4, 2048, 1, 128.0 * WE, "expansion (words; pairs=words)");
    return true;
}

int main() {
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, 0));
    int clock_khz = 0;
    CK(cudaDeviceGetAttribute(&clock_khz, cudaDevAttrClockRate, 0));
    printf("device=%s sms=%d clockRate_kHz=%d\n", prop.name, prop.multiProcessorCount, clock_khz);
    uint32_t *d_rows, *d_q;
    int32_t* d_out;
    unsigned long long* d_clk;
    CK(cudaMalloc(&d_rows, 128 * 8 * 4)); CK(cudaMalloc(&d_q, kN * 8 * 4)); CK(cudaMalloc(&d_out, (128 * kN + 128 * kN / 2) * 4));
    CK(cudaMalloc(&d_clk, 2 * prop.multiProcessorCount * 3 * 8));
    const int sms = prop.multiProcessorCount;
    bool ok = true;
    ok &= run_we<1>(4, sms, false, d_rows, d_q, d_out, d_clk, clock_khz);
    ok &= run_we<2>(8, sms, true, d_rows, d_q, d_out, d_clk, clock_khz);
    ok &= run_we<3>(11, sms, false, d_rows, d_q, d_out, d_clk, clock_khz);
    ok &= run_we<4>(16, sms, true, d_rows, d_q, d_out, d_clk, clock_khz);
    ok &= run_we<4>(13, sms, false, d_rows, d_q, d_out, d_clk, clock_khz);
    ok &= run_we<5>(17, sms, false, d_rows, d_q, d_out, d_clk, clock_khz);
    ok &= run_we<6>(24, sms, true, d_rows, d_q, d_out, d_clk, clock_khz);
    ok &= run_we<7>(26, sms, false, d_rows, d_q, d_out, d_clk, clock_khz);
    ok &= run_we<8>(32, sms, true, d_rows, d_q, d_out, d_clk, clock_khz);
    ok &= run_we<8>(30, sms, false, d_rows, d_q, d_out, d_clk, clock_khz);
    printf("%s\n", ok ? "ALL EXACT" : "SOME MISMATCH");
    return ok ? 0 : 1;
}
