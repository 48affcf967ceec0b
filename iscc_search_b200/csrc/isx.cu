// isx.cu - store management + C ABI of libisx_b200.so (see include/isx.h for the contract and the
// reference interfaces each entry point replaces).
//
// Host side: exact key map, length buckets of plane-major segments in HBM, swap-remove (rows stay
// dense, no tombstones in the scan), launch planning for the scan (bootstrap rounds that tighten
// the per-query rank threshold before the bulk of the store is streamed), exact fallback re-scan
// for queries whose candidate buffer overflowed.
#include <algorithm>
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <numeric>
#include <shared_mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/isx.h"
#include "kernels.cuh"
#include "join.cuh"
#include "keymap.hpp"
#include "small.cuh"
#include "tc.cuh"

namespace isx {

static thread_local std::string g_err;

static int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define CU(expr)                                                                                   \
    do {                                                                                           \
        cudaError_t _e = (expr);                                                                   \
        if (_e != cudaSuccess)                                                                     \
            return fail(_e == cudaErrorMemoryAllocation ? ISX_ENOMEM : ISX_ECUDA, "%s failed: %s (%s:%d)", #expr, \
                        cudaGetErrorString(_e), __FILE__, __LINE__);                               \
    } while (0)

constexpr uint32_t kMinSegRows = 4096;
constexpr uint32_t kMaxSegRows = 1u << kRowBits;  // 4 Mi rows
constexpr uint32_t kBlockRows = kRowsPerStep;     // 1024
constexpr int kMaxLanes = 4;                      // query tiles of one batch in flight at a time (each with its own per-query state)
constexpr uint32_t kMaxK = 65536;                 // beyond the shared-memory sort capacity winners are sorted in global scratch

// growable device buffer
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return 0;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        size_t want = bytes + bytes / 4 + 256;
        CU(cudaMalloc(&p, want));
        cap = want;
        return 0;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <class T>
    T* as() const { return reinterpret_cast<T*>(p); }
};

struct PinnedBuf {
    void* p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return 0;
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
        size_t want = bytes + bytes / 4 + 256;
        CU(cudaMallocHost(&p, want));
        cap = want;
        return 0;
    }
    void release() {
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
    }
    template <class T>
    T* as() const { return reinterpret_cast<T*>(p); }
};

struct Segment {
    void* d_mem = nullptr;  // one allocation: planes | khi | klo
    SegDesc desc{};
    uint32_t len_bytes = 0;
    std::vector<uint64_t> h_khi, h_klo;  // host mirror of the keys (needed to re-point the moved row on swap-remove)
    uint32_t mirrored = 0;               // rows [0, mirrored) are in the host mirror and the key map (bulk appends lag behind)
    size_t bytes = 0;
};

// rank tables for one set of compared-length classes
struct RankTables {
    uint32_t class_mask = 0;  // bit m-1: m bytes compared
    uint32_t R = 0;
    std::vector<uint16_t> rank;  // [33][257]
    std::vector<uint16_t> hmax;  // [33][R]
    std::vector<uint32_t> frac_h, frac_n;  // representative fraction of every rank (for thresholds)
    DevBuf d_rank, d_hmax;
};

}  // namespace isx

using namespace isx;

struct isx_store {
    int device = 0;
    uint32_t key_bytes = 8, max_bytes = 32, fixed_len = 0;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    cudaStream_t side[3] = {nullptr, nullptr, nullptr};  // the launches of one pass run concurrently (tails overlap)
    cudaEvent_t fork_ev = nullptr, join_ev[3] = {nullptr, nullptr, nullptr};
    // two tile lanes: consecutive query tiles of a batch run on alternating streams with their own per-query state, so the
    // bootstrap / select of one tile and the tail of its scan launches overlap the next tile's scan
    cudaStream_t lane_stream[kMaxLanes] = {}, lane_side[kMaxLanes][3] = {};
    cudaEvent_t lane_fork[kMaxLanes] = {}, lane_join[kMaxLanes][3] = {};
    cudaEvent_t lanes_begin = nullptr, lane_done[kMaxLanes] = {};
    bool profiling = false;

    std::shared_mutex rows_mu;  // shared: search/get/contains; exclusive: add/remove/clear/load
    std::mutex work_mu;         // serialises users of the scratch buffers below

    KeyMap map;
    std::atomic<bool> map_stale{false};        // rows were bulk-appended from device memory (isx_add_device): the key map and
                                               // the host key mirrors are completed lazily by the first keyed operation
    uint64_t n_rows = 0;                       // live rows (== map.size() when the map is current)
    std::vector<Segment> segs;                 // global segment ids
    std::vector<uint32_t> bucket_segs[kMaxBytes + 1];
    uint64_t bucket_rows[kMaxBytes + 1] = {0};
    uint64_t device_bytes = 0;
    uint64_t version = 0;  // bumped by every mutation

    // device mirrors
    DevBuf d_segs;
    bool segs_dirty = true;
    DevBuf d_blocks, d_bdesc;
    uint64_t blocks_version = ~0ull;
    std::vector<uint2> h_blocks;
    uint32_t bucket_block_lo[kMaxBytes + 2] = {0};  // block range of bucket L: [lo[L], lo[L+1])

    RankTables tables;

    // cross-rank threshold sharing (see ScanParams::g_hist)
    uint32_t share_world = 0, share_rank = 0, share_maxq = 0;
    static constexpr uint32_t kShareRcap = 512;   // ranks per query in the shared histograms (385 for 64..256-bit codes)
    uint32_t* share_local = nullptr;              // this rank's home histograms (cudaMalloc, IPC exported)
    uint32_t* share_ptrs[kMaxRanks] = {nullptr};  // [r] = rank r's home histograms mapped into this process
    size_t share_bytes = 0;
    uint32_t share_len_mask = 0;                  // union of the stored-length masks of ALL ranks (isx_share_set_lengths)
    bool share_armed = false;                     // set by isx_share_reset, consumed by the next search: only a search that
                                                  // follows reset + barrier may count into / read the shared histograms

    // scratch
    DevBuf d_stage_codes, d_stage_keys, d_stage_dest, d_moves, d_bulk;
    DevBuf d_queries, d_tau, d_hist, d_shist, d_cnt, d_ovf, d_cand, d_qmap, d_fb, d_fb_cand;
    DevBuf d_out_khi, d_out_klo, d_out_h, d_out_n, d_out_cnt, d_out_codes, d_bigsort;
    PinnedBuf h_queries, h_qmap, h_flags, h_out;
    // small-batch path (k_scan_small): per-query state kept clean between searches, results land in mapped pinned memory
    DevBuf d_small;                 // tau[8] | cnt[8] | ovf[8] | hist[8][R] | shist[8][R]
    uint32_t small_R = 0;           // R the state was laid out (and zeroed) for
    PinnedBuf h_small_info;         // [8][4] status words written by the kernel
    PinnedBuf h_small_dbg;
    bool small_ok = true;           // cooperative launch available
    int small_smem_max = -1;        // dynamic shared memory k_scan_small may use on this device (set on first use)
    // function attributes are per device: the scan kernels whose shared-memory limit this store has raised, bit WE
    uint32_t scan_attr_done = 0, scan_tc_attr_done = 0;
    // isx_search (host results): the fused select writes straight into the pinned result block (no D2H copies)
    uint64_t* small_host_khi = nullptr; uint64_t* small_host_klo = nullptr; uint16_t* small_host_h = nullptr;
    uint16_t* small_host_n = nullptr; uint32_t* small_host_cnt = nullptr;
    bool small_host_valid = false, small_host_used = false;
    // self-join (isx_self_join): the sorted pair records of the last join, in d_join_keys / d_join_vals [join_cur] (the
    // other buffer of each pair is the sort's scratch); valid until the next search or match, a mutation (version), or
    // release_scratch
    DevBuf d_join_keys[2], d_join_vals[2], d_join_tmp, d_join_rows, d_join_cnt;
    uint32_t join_cur = 0;
    uint64_t join_total = 0, join_version = 0;
    bool join_valid = false;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    std::vector<cudaEvent_t> tile_events;  // 3 per tile, grown on demand (profiling only)
    isx_stats_t stats{};
    int sm_count = 148;
    int max_smem_optin = 0;
    int smem_per_sm = 0;
};

namespace isx {

static inline Key128 load_key(const isx_store* s, const void* keys, size_t i) {
    if (s->key_bytes == 8) return Key128{reinterpret_cast<const uint64_t*>(keys)[i], 0};
    const uint8_t* kb = reinterpret_cast<const uint8_t*>(keys) + i * 16;
    uint64_t hi = 0, lo = 0;
    for (int b = 0; b < 8; b++) { hi = (hi << 8) | kb[b]; lo = (lo << 8) | kb[8 + b]; }
    return Key128{hi, lo};
}
static inline void store_key(const isx_store* s, void* keys, size_t i, uint64_t hi, uint64_t lo) {
    if (s->key_bytes == 8) { reinterpret_cast<uint64_t*>(keys)[i] = hi; return; }
    uint8_t* kb = reinterpret_cast<uint8_t*>(keys) + i * 16;
    for (int b = 0; b < 8; b++) { kb[b] = (uint8_t)(hi >> (56 - 8 * b)); kb[8 + b] = (uint8_t)(lo >> (56 - 8 * b)); }
}

static int set_device(isx_store* s) {
    CU(cudaSetDevice(s->device));
    return 0;
}

static int new_segment(isx_store* s, uint32_t len_bytes, uint32_t cap, bool mirror = true) {
    if (s->segs.size() >= (1u << kSegBits)) return fail(ISX_ENOMEM, "segment table full (%u segments)", 1u << kSegBits);
    Segment sg;
    uint32_t words = (len_bytes + 3) / 4;
    size_t plane_bytes = (size_t)words * cap * 4;
    size_t key_bytes = (size_t)cap * 8;
    size_t total = plane_bytes + key_bytes * (s->key_bytes == 16 ? 2 : 1);
    CU(cudaMalloc(&sg.d_mem, total));
    CU(cudaMemsetAsync(sg.d_mem, 0, total, s->stream));
    sg.bytes = total;
    sg.len_bytes = len_bytes;
    sg.desc.planes = reinterpret_cast<uint32_t*>(sg.d_mem);
    sg.desc.khi = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(sg.d_mem) + plane_bytes);
    sg.desc.klo = s->key_bytes == 16 ? sg.desc.khi + cap : nullptr;
    sg.desc.cap = cap;
    sg.desc.n = 0;
    sg.desc.len_bytes = len_bytes;
    sg.desc.words = words;
    if (mirror) {
        sg.h_khi.resize(cap);
        if (s->key_bytes == 16) sg.h_klo.resize(cap);
    }
    s->device_bytes += total;
    s->bucket_segs[len_bytes].push_back((uint32_t)s->segs.size());
    s->segs.push_back(std::move(sg));
    s->segs_dirty = true;
    return 0;
}

static int upload_segs(isx_store* s) {
    if (!s->segs_dirty) return 0;
    size_t n = std::max<size_t>(s->segs.size(), 1);
    std::vector<SegDesc> h(n);
    for (size_t i = 0; i < s->segs.size(); i++) h[i] = s->segs[i].desc;
    if (s->d_segs.ensure(n * sizeof(SegDesc))) return ISX_ECUDA;
    // pageable source: cudaMemcpyAsync stages it before returning, so the vector may die afterwards
    CU(cudaMemcpyAsync(s->d_segs.p, h.data(), n * sizeof(SegDesc), cudaMemcpyHostToDevice, s->stream));
    CU(cudaStreamSynchronize(s->stream));
    s->segs_dirty = false;
    return 0;
}

static int upload_blocks(isx_store* s) {
    if (s->blocks_version == s->version) return 0;
    s->h_blocks.clear();
    for (uint32_t L = 1; L <= kMaxBytes; L++) {
        s->bucket_block_lo[L] = (uint32_t)s->h_blocks.size();
        for (uint32_t sid : s->bucket_segs[L]) {
            uint32_t n = s->segs[sid].desc.n;
            for (uint32_t r = 0; r < n; r += kBlockRows) s->h_blocks.push_back(make_uint2(sid, r));
        }
    }
    s->bucket_block_lo[kMaxBytes + 1] = (uint32_t)s->h_blocks.size();
    size_t bytes = std::max<size_t>(s->h_blocks.size(), 1) * sizeof(uint2);
    if (s->d_blocks.ensure(bytes) || s->d_bdesc.ensure(std::max<size_t>(s->h_blocks.size(), 1) * sizeof(BlockDesc))) return ISX_ECUDA;
    if (!s->h_blocks.empty()) {
        std::vector<BlockDesc> bd(s->h_blocks.size());
        for (size_t i = 0; i < bd.size(); i++) {
            const SegDesc& d = s->segs[s->h_blocks[i].x].desc;
            bd[i] = BlockDesc{d.planes + s->h_blocks[i].y, d.cap, s->h_blocks[i].x, s->h_blocks[i].y, d.n, {0, 0}};
        }
        CU(cudaMemcpyAsync(s->d_blocks.p, s->h_blocks.data(), s->h_blocks.size() * sizeof(uint2), cudaMemcpyHostToDevice, s->stream));
        CU(cudaMemcpyAsync(s->d_bdesc.p, bd.data(), bd.size() * sizeof(BlockDesc), cudaMemcpyHostToDevice, s->stream));
        CU(cudaStreamSynchronize(s->stream));
    }
    s->blocks_version = s->version;
    return 0;
}

// Complete the key map + host key mirrors after bulk appends (caller holds rows_mu exclusively and work_mu).
static int sync_map(isx_store* s) {
    if (!s->map_stale.load()) return 0;
    CU(cudaSetDevice(s->device));
    s->map.reserve(s->n_rows);
    for (size_t sid = 0; sid < s->segs.size(); sid++) {
        Segment& sg = s->segs[sid];
        const uint32_t n = sg.desc.n, m0 = sg.mirrored;
        if (m0 >= n) continue;
        if (sg.h_khi.size() < sg.desc.cap) sg.h_khi.resize(sg.desc.cap);
        if (s->key_bytes == 16 && sg.h_klo.size() < sg.desc.cap) sg.h_klo.resize(sg.desc.cap);
        CU(cudaMemcpyAsync(sg.h_khi.data() + m0, sg.desc.khi + m0, (size_t)(n - m0) * 8, cudaMemcpyDeviceToHost, s->stream));
        if (s->key_bytes == 16) CU(cudaMemcpyAsync(sg.h_klo.data() + m0, sg.desc.klo + m0, (size_t)(n - m0) * 8, cudaMemcpyDeviceToHost, s->stream));
        CU(cudaStreamSynchronize(s->stream));
        for (uint32_t r = m0; r < n; r++) {
            const Key128 key{sg.h_khi[r], s->key_bytes == 16 ? sg.h_klo[r] : 0};
            if (!s->map.insert(key, ((uint64_t)sid << 32) | r))
                return fail(ISX_EINVAL, "isx_add_device: bulk-appended keys were not unique (key %016llx%016llx is stored twice); the key map "
                                        "cannot be completed - clear or reload the store (searches still work)",
                            (unsigned long long)key.hi, (unsigned long long)key.lo);
        }
        sg.mirrored = n;
    }
    s->map_stale.store(false);
    return 0;
}

// keyed operations call this BEFORE taking their own locks
static int ensure_map(isx_store* s) {
    if (!s->map_stale.load()) return 0;
    std::unique_lock<std::shared_mutex> g(s->rows_mu);
    std::lock_guard<std::mutex> gw(s->work_mu);
    return sync_map(s);
}

// ---- rank tables -------------------------------------------------------------------------------
// Dense rank of every rational h/(8m) over the compared-length classes in `mask`; exact integer
// order via cross multiplication. hmax[m][r] = largest h with rank(m,h) <= r.
static int compute_tables(uint32_t mask, RankTables& t) {
    struct F { uint32_t h, n, m; };
    std::vector<F> fr;
    for (uint32_t m = 1; m <= kMaxBytes; m++)
        if (mask & (1u << (m - 1)))
            for (uint32_t h = 0; h <= 8 * m; h++) fr.push_back(F{h, 8 * m, m});
    std::sort(fr.begin(), fr.end(), [](const F& a, const F& b) {
        uint64_t x = (uint64_t)a.h * b.n, y = (uint64_t)b.h * a.n;
        if (x != y) return x < y;
        return a.n < b.n;
    });
    t.rank.assign(33 * 257, 0xffff);
    t.frac_h.clear();
    t.frac_n.clear();
    uint32_t r = 0;
    for (size_t i = 0; i < fr.size(); i++) {
        if (i > 0 && (uint64_t)fr[i].h * fr[i - 1].n != (uint64_t)fr[i - 1].h * fr[i].n) r++;
        if (t.frac_h.size() <= r) { t.frac_h.push_back(fr[i].h); t.frac_n.push_back(fr[i].n); }
        t.rank[fr[i].m * 257 + fr[i].h] = (uint16_t)r;
    }
    t.R = fr.empty() ? 1 : r + 1;
    if (t.R >= (1u << kRankBits)) return fail(ISX_EINVAL, "too many distinct distances (%u)", t.R);
    t.hmax.assign((size_t)33 * t.R, 0);
    for (uint32_t m = 1; m <= kMaxBytes; m++) {
        if (!(mask & (1u << (m - 1)))) continue;
        uint32_t h = 0;
        for (uint32_t rr = 0; rr < t.R; rr++) {
            while (h + 1 <= 8 * m && t.rank[m * 257 + h + 1] <= rr) h++;
            t.hmax[(size_t)m * t.R + rr] = (uint16_t)h;
        }
    }
    t.class_mask = mask;
    return 0;
}

static int build_tables(isx_store* s, uint32_t mask) {
    RankTables& t = s->tables;
    if (t.class_mask == mask && t.R) return 0;
    t.class_mask = 0;
    int rc = compute_tables(mask, t);
    if (rc) return rc;
    t.class_mask = 0;  // set again only after the upload succeeded
    if (t.d_rank.ensure(t.rank.size() * 2) || t.d_hmax.ensure(t.hmax.size() * 2)) return ISX_ECUDA;
    CU(cudaMemcpyAsync(t.d_rank.p, t.rank.data(), t.rank.size() * 2, cudaMemcpyHostToDevice, s->stream));
    CU(cudaMemcpyAsync(t.d_hmax.p, t.hmax.data(), t.hmax.size() * 2, cudaMemcpyHostToDevice, s->stream));
    CU(cudaStreamSynchronize(s->stream));
    t.class_mask = mask;
    return 0;
}

// ---- scan launch dispatch ----------------------------------------------------------------------
template <int WE, int G, int MINB = 3>
static int launch_scan_t(isx_store* s, ScanParams& p, uint32_t grid_cap_per_sm, cudaStream_t stream) {
    constexpr int QW = (WE <= 4) ? 4 : 8;
    size_t smem = (size_t)p.q_split * (QW * 4 + 2) + 4 + 258 * 2 + ((size_t)p.R + 2) * 2 + 32;
    // candidate stage (kernels.cuh "staged emission"): as many records as keep MINB CTAs of this size on an SM, at most 1024
    {
        static const int env_stage = [] { const char* e = getenv("ISX_STAGE"); return e ? atoi(e) : 1024; }();
        const size_t per_cta = (size_t)s->smem_per_sm / MINB - 1024;   // the driver reserves 1 KB per CTA
        size_t cap = per_cta > smem + stage_bytes(0) ? (per_cta - smem - stage_bytes(0)) / 12 : 0;
        cap = std::min<size_t>(cap, (size_t)std::max(0, env_stage)) & ~(size_t)31;
        p.stage_cap = cap >= 64 ? (uint32_t)cap : 0;
        if (p.stage_cap) smem += stage_bytes(p.stage_cap);
    }
    if (!(s->scan_attr_done & (1u << WE))) {
        CU(cudaFuncSetAttribute(k_scan<WE, G, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, s->max_smem_optin));
        s->scan_attr_done |= 1u << WE;
    }
    uint32_t n_blocks = p.block_end - p.block_begin;
    uint32_t n_groups = (n_blocks + G - 1) / G;
    if (n_groups == 0) return 0;
    const uint32_t cap = (uint32_t)s->sm_count * grid_cap_per_sm;
    const uint32_t per = (n_groups + cap - 1) / cap;   // groups per CTA
    const uint32_t gx = (n_groups + per - 1) / per;    // equal shares (they differ by at most one group)
    dim3 grid(gx, (p.T + p.q_split - 1) / p.q_split, 1);
    k_scan<WE, G, MINB><<<grid, kThreads, smem, stream>>>(p);
    CU(cudaGetLastError());
    s->stats.kernel_launches++;
    s->stats.scan_launches++;
    return 0;
}

// ---- tensor-core scan (tc.cuh) ----
template <int WE>
static int launch_scan_tc_t(isx_store* s, ScanParams& p, cudaStream_t stream) {
    size_t smem = tc_smem_bytes(WE, p.q_split, p.R) + 8;   // + alignment of the stage
    {
        const size_t per_cta = (size_t)s->smem_per_sm / kTcMinBlocksPerSm - 1024;
        size_t cap = per_cta > smem + stage_bytes(0) ? (per_cta - smem - stage_bytes(0)) / 12 : 0;
        cap = std::min<size_t>(cap, 1024) & ~(size_t)31;
        p.stage_cap = cap >= 64 ? (uint32_t)cap : 0;
        if (p.stage_cap) smem += stage_bytes(p.stage_cap);
    }
    if (!(s->scan_tc_attr_done & (1u << WE))) {
        CU(cudaFuncSetAttribute(k_scan_tc<WE>, cudaFuncAttributeMaxDynamicSharedMemorySize, s->max_smem_optin));
        s->scan_tc_attr_done |= 1u << WE;
    }
    const uint32_t n_blocks = p.block_end - p.block_begin;
    if (n_blocks == 0) return 0;
    const uint32_t gx = std::min<uint32_t>(n_blocks, (uint32_t)s->sm_count * kTcMinBlocksPerSm);
    dim3 grid(gx, (p.T + p.q_split - 1) / p.q_split, 1);
    k_scan_tc<WE><<<grid, kThreads, smem, stream>>>(p);
    CU(cudaGetLastError());
    s->stats.kernel_launches++;
    s->stats.scan_launches++;
    return 0;
}

// ISX_TC_SCAN=0 keeps every launch on the POPC scan (A/B on the same build); ISX_TC_MIN_T sets the smallest query tile
// that takes the tensor-core scan (below it the MMA's N would be mostly padding)
static bool use_tc_scan(uint32_t T) {
    static const bool env_on = [] { const char* e = getenv("ISX_TC_SCAN"); return !(e && e[0] == '0'); }();
    static const uint32_t env_min_t = [] { const char* e = getenv("ISX_TC_MIN_T"); return e ? (uint32_t)std::max(1, atoi(e)) : 64u; }();
    return env_on && T >= env_min_t;
}

static int launch_scan_tc(isx_store* s, ScanParams& p, uint32_t we, uint32_t bpi_hint, cudaStream_t stream) {
    p.blocks_per_item = std::max<uint32_t>(1, bpi_hint);
    // <= 256 queries per CTA (the MMA's N); small ranges split the tile further, down to 64 queries, so ~4 waves of CTAs exist
    const uint32_t n_blocks = std::max<uint32_t>(1, p.block_end - p.block_begin);
    const uint32_t want = (uint32_t)s->sm_count * kTcMinBlocksPerSm * 4;
    uint32_t splits = (p.T + kTcMaxN - 1) / kTcMaxN;
    if (n_blocks * splits < want) splits = std::max(splits, std::min((want + n_blocks - 1) / n_blocks, std::max<uint32_t>(1, p.T / 64)));
    p.q_split = (p.T + splits - 1) / splits;
    switch (we) {
        case 1: return launch_scan_tc_t<1>(s, p, stream);
        case 2: return launch_scan_tc_t<2>(s, p, stream);
        case 3: return launch_scan_tc_t<3>(s, p, stream);
        case 4: return launch_scan_tc_t<4>(s, p, stream);
        case 5: return launch_scan_tc_t<5>(s, p, stream);
        case 6: return launch_scan_tc_t<6>(s, p, stream);
        case 7: return launch_scan_tc_t<7>(s, p, stream);
        case 8: return launch_scan_tc_t<8>(s, p, stream);
    }
    return fail(ISX_EINVAL, "bad word count %u", we);
}

static uint32_t groups_for(uint32_t we) { return we <= 2 ? 4 : (we <= 4 ? 2 : 1); }

static int launch_scan(isx_store* s, ScanParams& p, uint32_t we, uint32_t bpi_hint, cudaStream_t stream) {
    uint32_t G = groups_for(we);
    p.blocks_per_item = std::max(G, (bpi_hint / G) * G);
    const uint32_t per_sm = 3;  // resident CTAs per SM (register bound, __launch_bounds__(256, 3); 4 CTAs of 64
                                // registers measured no faster - the POPC pipe, not occupancy, is the limit)
    // small ranges: split the query tile over gridDim.y so ~8 waves of CTAs exist. Finer work units cut the tail of a launch
    // whose CTAs all take equally long (measured on a 12.5 M-row shard, 8192 queries: 2 waves 81.7 ms, 4 waves 80.4, 8 waves 78.4)
    {
        uint32_t n_items = (p.block_end - p.block_begin + G - 1) / G;
        static const uint32_t env_waves = [] { const char* e = getenv("ISX_SPLIT_WAVES"); return e ? (uint32_t)std::max(1, atoi(e)) : 8u; }();
        uint32_t want = (uint32_t)s->sm_count * per_sm * env_waves;
        uint32_t splits = n_items >= want ? 1 : std::min<uint32_t>(p.T, (want + n_items - 1) / n_items);
        splits = std::min<uint32_t>(splits, std::max<uint32_t>(1, p.T / 32));  // >= 32 queries per CTA: its set-up (tables, tile) must stay small next to its work
        splits = std::max<uint32_t>(splits, (p.T + kMaxTile - 1) / kMaxTile);   // a CTA holds at most kMaxTile queries in shared memory
        p.q_split = (p.T + splits - 1) / splits;
    }
    switch (we) {
        case 1: return launch_scan_t<1, 4>(s, p, per_sm, stream);
        case 2: return launch_scan_t<2, 4>(s, p, per_sm, stream);
        case 3: return launch_scan_t<3, 2>(s, p, per_sm, stream);
        case 4: return launch_scan_t<4, 2>(s, p, per_sm, stream);
        case 5: return launch_scan_t<5, 1>(s, p, per_sm, stream);
        case 6: return launch_scan_t<6, 1>(s, p, per_sm, stream);
        case 7: return launch_scan_t<7, 1>(s, p, per_sm, stream);
        case 8: return launch_scan_t<8, 1>(s, p, per_sm, stream);
    }
    return fail(ISX_EINVAL, "bad word count %u", we);
}

// Scan block range [b0, b1) of the global block list for one tile of queries; the range may span
// several buckets, each bucket portion is one launch (uniform compared length).
static int scan_range(isx_store* s, ScanParams& p, uint32_t b0, uint32_t b1, uint32_t bpi_hint, int lane = -1) {
    cudaStream_t main_stream = lane < 0 ? s->stream : s->lane_stream[lane];
    cudaStream_t* sides = lane < 0 ? s->side : s->lane_side[lane];
    cudaEvent_t fork_ev = lane < 0 ? s->fork_ev : s->lane_fork[lane];
    cudaEvent_t* join_ev = lane < 0 ? s->join_ev : s->lane_join[lane];
    // buckets with L >= Lq all compare m = Lq bytes: they form ONE launch; shorter buckets one launch each.
    // The launches of a pass are independent (they only share the monotone thresholds), so the 2nd..4th go to
    // side streams forked from / joined back into the store's stream: their ramp-up and tails overlap.
    int n_launch = 0, side_used = 0;
    for (uint32_t L = 1; L <= kMaxBytes; L++) {
        const uint32_t Lhi = (L >= p.qlen_bytes) ? kMaxBytes : L;  // last bucket of this launch
        uint32_t lo = std::max(b0, s->bucket_block_lo[L]), hi = std::min(b1, s->bucket_block_lo[Lhi + 1]);
        if (lo < hi) {
            uint32_t m = std::min(p.qlen_bytes, L);
            p.block_begin = lo;
            p.block_end = hi;
            cudaStream_t stream = main_stream;
            if (n_launch > 0 && side_used < 3) {
                if (side_used == 0) CU(cudaEventRecord(fork_ev, main_stream));
                stream = sides[side_used];
                CU(cudaStreamWaitEvent(stream, fork_ev, 0));
            }
            const bool tc = use_tc_scan(p.T);
            int rc = tc ? launch_scan_tc(s, p, (m + 3) / 4, bpi_hint, stream) : launch_scan(s, p, (m + 3) / 4, bpi_hint, stream);
            if (rc) return rc;
            if (stream != main_stream) {
                CU(cudaEventRecord(join_ev[side_used], stream));
                side_used++;
            }
            n_launch++;
            uint64_t rows = 0;  // live rows in the range: whole buckets from the bucket counters, partial ones block by block
            for (uint32_t Lb = L; Lb <= Lhi; Lb++) {
                const uint32_t blo = std::max(lo, s->bucket_block_lo[Lb]), bhi = std::min(hi, s->bucket_block_lo[Lb + 1]);
                if (blo >= bhi) continue;
                if (blo == s->bucket_block_lo[Lb] && bhi == s->bucket_block_lo[Lb + 1]) { rows += s->bucket_rows[Lb]; continue; }
                for (uint32_t b = blo; b < bhi; b++) {  // last block of a segment may be partial
                    const SegDesc& d = s->segs[s->h_blocks[b].x].desc;
                    rows += std::min<uint32_t>(kBlockRows, d.n - s->h_blocks[b].y);
                }
            }
            s->stats.pairs += rows * p.T;
            s->stats.algo_bytes += rows * m;
            s->stats.algo_popc += rows * p.T * ((m + 3) / 4);
            static const uint32_t kCsaPopc[9] = {0, 1, 1, 2, 2, 3, 2, 3, 3};  // steady state: OR-fold lower-bound filter (3-word folds for 6..8 words, 2-word folds for 2, 4, 5) else carry-save
            if (!tc) s->stats.issued_popc += rows * p.T * kCsaPopc[(m + 3) / 4];   // the tensor-core scan issues no POPC
        }
        if (Lhi == kMaxBytes) break;
    }
    for (int i = 0; i < side_used; i++) CU(cudaStreamWaitEvent(main_stream, join_ev[i], 0));
    return 0;
}

static size_t select_smem(uint32_t cap, uint32_t key_words) { return (size_t)cap * (8 * key_words + 12) + 64; }

static uint32_t max_sort_cap(const isx_store* s) {
    uint32_t key_words = s->key_bytes == 16 ? 2 : 1;
    uint32_t cap = 1024;
    while (select_smem(cap * 2, key_words) + 2048 <= (size_t)s->max_smem_optin) cap *= 2;
    return cap;
}

struct SearchOut {
    uint64_t* khi; uint64_t* klo; uint16_t* h; uint16_t* n; uint32_t* cnt; uint8_t* codes;
};

// ---- small-batch path: the whole search in one cooperative launch (small.cuh) --------------------------------
// Returns 0 and *done = true when every query was answered; *done = false when the caller has to run the general
// path (not eligible, or a query overflowed its candidate list / has more ties than the fused select sorts).
static int search_small(isx_store* s, const uint8_t* queries, bool q_on_device, const uint8_t* qlens, size_t Q, uint32_t k,
                        uint32_t tau_init, const SearchOut& out, bool* done) {
    *done = false;
    static const bool env_on = [] { const char* e = getenv("ISX_SMALL_PATH"); return !(e && e[0] == '0'); }();
    static const uint32_t env_sample = [] { const char* e = getenv("ISX_SMALL_SAMPLE"); return e ? (uint32_t)std::max(1, atoi(e)) : 1u; }();
    const RankTables& tb = s->tables;
    const uint32_t R = tb.R;
    static const size_t env_maxq = [] { const char* e = getenv("ISX_SMALL_MAXQ"); return e ? (size_t)std::max(1, std::min(atoi(e), kSmallT)) : (size_t)4; }();
    if (!env_on || !s->small_ok || Q > env_maxq || k > kSmallSortCap / 2 || R > kSmallMaxR || s->h_blocks.empty()) return 0;
    static const bool env_wide = [] { const char* e = getenv("ISX_SMALL_WIDE"); return e ? e[0] != '0' : true; }();
    static const bool env_hint = [] { const char* e = getenv("ISX_SMALL_L2HINT"); return e ? e[0] != '0' : true; }();
    const uint32_t chunks = env_wide ? 16 : 8;
    isx_stats_t& st = s->stats;
    SmallParams p{};
    p.l2_evict_first = env_hint ? 1 : 0;
    // static round-robin units by default; ISX_SMALL_DYNAMIC=1 claims them from a global counter (no tail wait, but
    // measured 4-8 % slower on 192/256-bit compares, 2 % faster on 64/128-bit: profiles/r02_small_path.txt)
    static const bool env_dynamic = [] { const char* e = getenv("ISX_SMALL_DYNAMIC"); return e && e[0] == '1'; }();
    p.static_units = env_dynamic ? 0 : 1;
    uint32_t max_lq = 0;
    for (size_t i = 0; i < Q; i++) max_lq = std::max<uint32_t>(max_lq, qlens[i]);
    uint64_t algo_bytes = 0, pairs = 0, algo_popc = 0;
    for (uint32_t L = 1; L <= kMaxBytes; L++) {
        const uint32_t nb = s->bucket_block_lo[L + 1] - s->bucket_block_lo[L];
        if (!nb) continue;
        if (p.n_ranges == (uint32_t)kSmallRanges) return 0;
        SmallRange& rg = p.ranges[p.n_ranges++];
        rg.we = (std::min(max_lq, L) + 3) / 4;
        rg.bpu = chunks / rg.we;
        rg.block0 = s->bucket_block_lo[L];
        rg.n_blocks = nb;
        rg.unit0 = p.n_units;
        rg.n_units = (nb + rg.bpu - 1) / rg.bpu;
        rg.len_bytes = L;
        p.n_units += rg.n_units;
        algo_bytes += s->bucket_rows[L] * std::min(max_lq, L);
        for (size_t i = 0; i < Q; i++) {
            const uint32_t m = std::min<uint32_t>(qlens[i], L);
            pairs += s->bucket_rows[L];
            algo_popc += s->bucket_rows[L] * ((m + 3) / 4);
        }
    }
    // candidate buffer as in the general path
    const uint32_t r0 = std::max<uint32_t>(1, (2 * k + kBlockRows - 1) / kBlockRows);
    uint64_t C64 = std::max<uint64_t>((uint64_t)r0 * kBlockRows + 40ull * k + 2048, 32768);
    const uint32_t C = (uint32_t)((C64 + 1023) / 1024 * 1024);
    const size_t state_words = 3 * (size_t)kSmallT + 2 * (size_t)kSmallT * R + 4;   // + the unit counter
    if (s->d_cand.ensure((size_t)kSmallT * C * 8) || s->h_small_info.ensure(kSmallT * 16) || s->d_out_klo.ensure(Q * (size_t)k * 8)) return ISX_ENOMEM;
    if (s->small_R != R || s->d_small.cap < state_words * 4) {
        if (s->d_small.ensure(state_words * 4)) return ISX_ENOMEM;
        CU(cudaMemsetAsync(s->d_small.p, 0, state_words * 4, s->stream));
        CU(cudaMemsetAsync(s->d_small.p, 0xff, kSmallT * 4, s->stream));   // tau = ~0
        s->small_R = R;
    }
    uint32_t* base = s->d_small.as<uint32_t>();
    p.tau = base; p.cand_cnt = base + kSmallT; p.overflow = base + 2 * kSmallT;
    p.hist = base + 3 * kSmallT; p.shist = p.hist + (size_t)kSmallT * R;
    p.unit_counter = p.shist + (size_t)kSmallT * R;
    p.cand = s->d_cand.as<uint64_t>();
    p.bdesc = s->d_bdesc.as<BlockDesc>();
    p.segs = s->d_segs.as<SegDesc>();
    p.T = (uint32_t)Q;
    p.C = C; p.R = R; p.k = k; p.tau_init = tau_init;
    p.rank_tab = tb.d_rank.as<uint16_t>();
    p.hmax_tab = tb.d_hmax.as<uint16_t>();
    for (size_t i = 0; i < Q; i++) {
        p.qlen[i] = qlens[i];
        p.qsrc[i] = (uint32_t)i;
        if (!q_on_device) memcpy(p.qwords[i], queries + i * 32, 32);
    }
    p.d_queries = q_on_device ? reinterpret_cast<const uint32_t*>(queries) : nullptr;
    const uint32_t grid = (uint32_t)s->sm_count;
    p.sample_units = env_sample;
    p.sample_stride = std::max<uint32_t>(1, p.n_units / (grid * p.sample_units));
    p.out_khi = out.khi; p.out_klo = out.klo ? out.klo : s->d_out_klo.as<uint64_t>(); p.out_h = out.h; p.out_n = out.n;
    p.out_cnt = out.cnt; p.out_codes = out.codes;
    if (s->small_host_valid) {
        p.out_khi = s->small_host_khi; p.out_h = s->small_host_h; p.out_n = s->small_host_n; p.out_cnt = s->small_host_cnt;
        if (s->key_bytes == 16) p.out_klo = s->small_host_klo;
    }
    p.key_words = s->key_bytes == 16 ? 2 : 1;
    p.info = s->h_small_info.as<uint32_t>();
    static const bool env_dbg = [] { const char* e = getenv("ISX_SMALL_DEBUG"); return e && e[0] == '1'; }();
    if (env_dbg) {
        if (s->h_small_dbg.ensure((size_t)s->sm_count * 128)) return ISX_ENOMEM;
        memset(s->h_small_dbg.p, 0, (size_t)s->sm_count * 128);
        p.dbg = s->h_small_dbg.as<unsigned long long>();
    }
    const void* kern = env_wide ? (const void*)k_scan_small<3, 16> : (const void*)k_scan_small<5, 8>;
    const size_t smem = (env_wide ? sizeof(SmallSharedT<3, 16>) : sizeof(SmallSharedT<5, 8>)) + (size_t)Q * R * 4;
    // function attributes are per device: remembered per store (one store = one device), not in a process-wide static
    if (s->small_smem_max < 0) {
        cudaFuncAttributes fa;
        CU(cudaFuncGetAttributes(&fa, kern));
        CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, s->max_smem_optin - (int)fa.sharedSizeBytes));
        s->small_smem_max = s->max_smem_optin - (int)fa.sharedSizeBytes;
    }
    const int smem_max = s->small_smem_max;
    if (smem > (size_t)smem_max) return 0;
    if (s->profiling) CU(cudaEventRecord(s->ev[0], s->stream));
    void* args[] = {&p};
    cudaError_t e = cudaLaunchCooperativeKernel(kern, dim3(grid), dim3(kSmallThreads), args, smem, s->stream);
    if (e != cudaSuccess) {
        cudaGetLastError();
        s->small_ok = false;   // e.g. cooperative launches unsupported under this context (MPS): general path from now on
        return 0;
    }
    if (s->profiling) CU(cudaEventRecord(s->ev[3], s->stream));
    CU(cudaStreamSynchronize(s->stream));
    st.kernel_launches = 1;
    st.scan_launches = 1;
    st.passes = 1;
    st.pairs = pairs; st.algo_bytes = algo_bytes; st.algo_popc = algo_popc; st.issued_popc = algo_popc;
    if (s->profiling) {
        float t = 0;
        CU(cudaEventElapsedTime(&t, s->ev[0], s->ev[3]));
        st.total_ms = t;
        st.scan_ms = t;
    }
    if (env_dbg) {
        const unsigned long long* d = s->h_small_dbg.as<unsigned long long>();
        for (int b : {0, s->sm_count - 1})
            fprintf(stderr, "[isx small dbg] cta %3d: setup %llu | phase0 %llu | sync+tau %llu | phase1 %llu | sync %llu | select %llu clk"
                    " (dstar+list %llu, filter %llu, keys %llu, sort %llu [radix %lld, compact %lld], write %llu) info: cands %u d* %u total_le %u\n", b,
                    d[b * 16 + 1] - d[b * 16], d[b * 16 + 2] - d[b * 16 + 1], d[b * 16 + 3] - d[b * 16 + 2], d[b * 16 + 4] - d[b * 16 + 3],
                    d[b * 16 + 5] - d[b * 16 + 4], d[b * 16 + 6] - d[b * 16 + 5], d[b * 16 + 7] - d[b * 16 + 5], d[b * 16 + 8] - d[b * 16 + 7],
                    d[b * 16 + 9] - d[b * 16 + 8], d[b * 16 + 10] - d[b * 16 + 9], (long long)(d[b * 16 + 12] - d[b * 16 + 9]), (long long)(d[b * 16 + 13] - d[b * 16 + 12]),
                    d[b * 16 + 11] - d[b * 16 + 10], s->h_small_info.as<uint32_t>()[1], s->h_small_info.as<uint32_t>()[2], s->h_small_info.as<uint32_t>()[3]);
    }
    const uint32_t* info = s->h_small_info.as<uint32_t>();
    bool clean = true;
    for (size_t i = 0; i < Q; i++) {
        st.candidates += info[4 * i + 1];
        if (info[4 * i] != 0) clean = false;
    }
    if (!clean) {
        // rare: candidate overflow (mass duplicates) or more ties than the fused select sorts - the general path
        // answers the whole batch; the per-query state of the small path is reset
        CU(cudaMemsetAsync(s->d_small.p, 0, state_words * 4, s->stream));
        CU(cudaMemsetAsync(s->d_small.p, 0xff, kSmallT * 4, s->stream));
        return 0;
    }
    *done = true;
    s->small_host_used = s->small_host_valid;
    return 0;
}

// Core: all pointers in `out` are DEVICE pointers laid out [Q][k]. `queries` host or device.
static int search_core(isx_store* s, const uint8_t* queries, bool q_on_device, const uint8_t* qlens, size_t Q, uint32_t k,
                       uint32_t thr_num, uint32_t thr_den, const SearchOut& out) {
    isx_stats_t& st = s->stats;
    st = isx_stats_t{};
    s->join_valid = false;
    const bool share_armed = s->share_armed;  // consumed by this call whatever happens next
    s->share_armed = false;
    if (Q == 0) return 0;
    if (k < 1) return fail(ISX_EINVAL, "`count` must be >= 1");
    const uint32_t key_words = s->key_bytes == 16 ? 2 : 1;
    const uint32_t cap_max = max_sort_cap(s);
    if (k > kMaxK) return fail(ISX_ELIMIT, "count %u exceeds the supported maximum %u", k, kMaxK);
    for (size_t i = 0; i < Q; i++) {
        uint32_t L = qlens[i];
        if (L < 1 || L > s->max_bytes) return fail(ISX_EINVAL, "query %zu: length %u bytes outside 1..%u", i, L, s->max_bytes);
        if (s->fixed_len && L != s->fixed_len) return fail(ISX_EINVAL, "query %zu: length %u bytes, index expects %u", i, L, s->fixed_len);
    }
    int rc;
    if ((rc = upload_segs(s)) || (rc = upload_blocks(s))) return rc;
    const uint32_t n_blocks_total = (uint32_t)s->h_blocks.size();

    // group queries by length (stable): order[] lists original indices
    std::vector<uint32_t> order(Q);
    std::iota(order.begin(), order.end(), 0u);
    std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return qlens[a] < qlens[b]; });

    // compared-length classes present
    uint32_t qmask = 0, bmask = 0, cmask = 0;
    for (size_t i = 0; i < Q; i++) qmask |= 1u << (qlens[i] - 1);
    for (uint32_t L = 1; L <= kMaxBytes; L++) if (s->bucket_rows[L]) bmask |= 1u << (L - 1);
    // Shared thresholds index the peer histograms by dense rank, so every rank must build the SAME rank table:
    // the compared-length classes come from the union of the lengths stored on any rank, not from the local rows.
    if (s->share_world > 1 && share_armed) bmask |= s->share_len_mask;
    for (uint32_t a = 1; a <= kMaxBytes; a++) {
        if (!(qmask & (1u << (a - 1)))) continue;
        cmask |= 1u << (a - 1);  // keeps the table non-empty for an empty store
        for (uint32_t b = 1; b <= kMaxBytes; b++)
            if (bmask & (1u << (b - 1))) cmask |= 1u << (std::min(a, b) - 1);
    }
    if ((rc = build_tables(s, cmask))) return rc;
    const RankTables& tb = s->tables;
    const uint32_t R = tb.R;
    uint32_t tau_init = R - 1;
    if (thr_den) {  // largest rank whose fraction is <= thr_num / thr_den (rank 0 = distance 0 always qualifies)
        uint32_t r = 0;
        while (r + 1 < R && (uint64_t)tb.frac_h[r + 1] * thr_den <= (uint64_t)thr_num * tb.frac_n[r + 1]) r++;
        tau_init = r;
    }

    {   // one or a handful of queries: the whole search is one cooperative launch (small.cuh)
        bool done = false;
        if ((rc = search_small(s, queries, q_on_device, qlens, Q, k, tau_init, out, &done))) return rc;
        if (done) return 0;
        st = isx_stats_t{};
    }

    // candidate buffer per query: a few k for the logarithmic tail of the running threshold plus slack for the
    // rows accepted before the first feedback (first wave of the bulk launch); overflow is handled exactly anyway
    const uint32_t r0 = std::max<uint32_t>(1, (2 * k + kBlockRows - 1) / kBlockRows);
    uint64_t C64 = (uint64_t)r0 * kBlockRows + 40ull * k + 2048;
    C64 = std::max<uint64_t>(C64, 32768);  // slack for the delayed threshold feedback of the first wave
    C64 = (C64 + 1023) / 1024 * 1024;
    const uint32_t C = (uint32_t)std::min<uint64_t>(C64, 1u << 26);

    // tile size from a scratch budget
    const size_t per_query = (size_t)C * 8 + (size_t)R * 4 + 64;
    const size_t budget = (size_t)6 << 30;
    // queries per tile (one pass over the store): up to 2 x kMaxTile - a launch then splits the tile over gridDim.y so that a
    // CTA keeps at most kMaxTile queries in shared memory; fewer, larger tiles halve the per-tile fixed work (bootstrap
    // sample, warm-up ranges, select) of a 10 000-query batch
    static const size_t env_tile = [] { const char* e = getenv("ISX_MAX_TILE"); return e ? (size_t)std::max(64, atoi(e)) : (size_t)kMaxTile; }();
    uint32_t tile_max = (uint32_t)std::max<size_t>(1, std::min<size_t>(env_tile, budget / per_query));
    tile_max = std::min<uint32_t>(tile_max, (uint32_t)Q);

    uint32_t big_P = 0;
    if (k > cap_max) {  // large k: global-memory sort scratch, one region per query of the tile
        big_P = 1;
        while (big_P < k) big_P <<= 1;
        if (s->d_bigsort.ensure((size_t)kMaxLanes * tile_max * big_P * sizeof(BigRec))) return ISX_ENOMEM;
    }
    // per-query state of a tile, twice (two tile lanes) when the batch has more than one tile
    static const size_t env_lanes = [] { const char* e = getenv("ISX_TILE_LANES"); return e ? (size_t)std::max(1, std::min(atoi(e), kMaxLanes)) : (size_t)2; }();
    const bool multi_tile = Q > tile_max || [&] { uint32_t m = 0; for (size_t i = 0; i < Q; i++) m |= 1u << (qlens[i] - 1); return (m & (m - 1)) != 0; }();
    const size_t n_sets = multi_tile ? env_lanes : 1;
    if (s->d_queries.ensure(Q * 32) || s->d_qmap.ensure(Q * 4) || s->d_tau.ensure(n_sets * tile_max * 4) ||
        s->d_hist.ensure(n_sets * tile_max * R * 4) || s->d_shist.ensure(n_sets * tile_max * R * 4) || s->d_cnt.ensure(n_sets * tile_max * 4) ||
        s->d_ovf.ensure(n_sets * tile_max * 4) || s->d_cand.ensure(n_sets * tile_max * C * 8) ||
        s->d_fb.ensure(n_sets * tile_max * 8) || s->h_flags.ensure((size_t)tile_max * 16))
        return ISX_ECUDA;

    // queries in group order on the device + the map back to original positions
    if (s->h_qmap.ensure(Q * 4)) return ISX_ECUDA;
    memcpy(s->h_qmap.p, order.data(), Q * 4);
    CU(cudaMemcpyAsync(s->d_qmap.p, s->h_qmap.p, Q * 4, cudaMemcpyHostToDevice, s->stream));
    if (!q_on_device) {
        if (s->h_queries.ensure(Q * 32)) return ISX_ECUDA;
        uint8_t* hq = s->h_queries.as<uint8_t>();
        for (size_t i = 0; i < Q; i++) {
            const uint8_t* src = queries + (size_t)order[i] * 32;
            uint32_t L = qlens[order[i]];
            memcpy(hq + i * 32, src, L);
            memset(hq + i * 32 + L, 0, 32 - L);
        }
        CU(cudaMemcpyAsync(s->d_queries.p, hq, Q * 32, cudaMemcpyHostToDevice, s->stream));
    } else {
        // device queries: one gather kernel into group order (also zero-pads beyond each query's length)
        if (s->h_queries.ensure(Q) || s->d_stage_dest.ensure(Q)) return ISX_ECUDA;
        uint8_t* hl = s->h_queries.as<uint8_t>();
        for (size_t i = 0; i < Q; i++) hl[i] = qlens[order[i]];
        CU(cudaMemcpyAsync(s->d_stage_dest.p, hl, Q, cudaMemcpyHostToDevice, s->stream));
        k_gather_queries<<<(unsigned)((Q * 8 + 255) / 256), 256, 0, s->stream>>>(reinterpret_cast<const uint32_t*>(queries), s->d_qmap.as<uint32_t>(),
                                                                               s->d_stage_dest.as<uint8_t>(), s->d_queries.as<uint32_t>(), (uint32_t)Q);
        CU(cudaGetLastError());
        st.kernel_launches++;
    }

    if (s->profiling) CU(cudaEventRecord(s->ev[0], s->stream));
    const uint32_t sort_cap = std::min<uint32_t>(cap_max, std::max<uint32_t>(1024, [&] { uint32_t c = 1024; while (c < 4 * k && c < cap_max) c *= 2; return c; }()));
    const size_t sel_smem = select_smem(sort_cap, key_words);
    {
        cudaFuncAttributes fa;
        CU(cudaFuncGetAttributes(&fa, k_select));
        CU(cudaFuncSetAttribute(k_select, cudaFuncAttributeMaxDynamicSharedMemorySize, s->max_smem_optin - (int)fa.sharedSizeBytes));
    }

    // ---- all tiles are enqueued without host synchronisation; overflow flags, candidate counts and the
    //      (d*, count<=d*) pairs of every tile land in pinned memory and are inspected once at the end ----
    struct Tile { size_t t0; uint32_t T, Lq; };
    std::vector<Tile> tiles;
    for (size_t g0 = 0; g0 < Q;) {
        const uint32_t Lq = qlens[order[g0]];
        size_t g1 = g0;
        while (g1 < Q && qlens[order[g1]] == Lq) g1++;
        {   // equal tiles per query length (2500 queries -> 2 x 1250, not 2048 + 452: the small tail tile ran at low efficiency)
            static const bool env_balance = [] { const char* e = getenv("ISX_TILE_BALANCE"); return !(e && e[0] == '0'); }();
            const size_t n = g1 - g0, n_tiles = (n + tile_max - 1) / tile_max;
            const size_t step = env_balance ? (n + n_tiles - 1) / n_tiles : tile_max;
            for (size_t t0 = g0; t0 < g1; t0 += step) tiles.push_back(Tile{t0, (uint32_t)std::min<size_t>(step, g1 - t0), Lq});
        }
        g0 = g1;
    }
    if (s->h_flags.ensure(Q * 16)) return ISX_ENOMEM;
    uint32_t* hf_ovf = s->h_flags.as<uint32_t>();  // [Q] overflow flags | [Q] candidate counts | [Q][2] (d*, count_le)
    uint32_t* hf_cnt = hf_ovf + Q;
    uint32_t* hf_info = hf_cnt + Q;
    if (s->profiling)
        while (s->tile_events.size() < tiles.size() * 3) {
            cudaEvent_t e;
            CU(cudaEventCreate(&e));
            s->tile_events.push_back(e);
        }

    // shared (cross-rank) histograms need every rank to see the same query batch in the same order
    const bool share_on = s->share_world > 1 && share_armed && R <= isx_store::kShareRcap && Q <= s->share_maxq;
    auto make_params = [&](const Tile& t, size_t set = 0) {
        ScanParams p{};
        p.segs = s->d_segs.as<SegDesc>();
        p.blocks = s->d_blocks.as<uint2>();
        p.queries = s->d_queries.as<uint32_t>() + t.t0 * 8;
        p.T = t.T;
        p.qlen_bytes = t.Lq;
        p.tau = s->d_tau.as<uint32_t>() + set * tile_max;
        p.hist = s->d_hist.as<uint32_t>() + set * tile_max * R;
        p.cand_cnt = s->d_cnt.as<uint32_t>() + set * tile_max;
        p.cand = s->d_cand.as<uint64_t>() + set * tile_max * C;
        p.overflow = s->d_ovf.as<uint32_t>() + set * tile_max;
        p.C = C; p.R = R; p.k = k;
        p.rank_tab = tb.d_rank.as<uint16_t>();
        p.hmax_tab = tb.d_hmax.as<uint16_t>();
        p.update_tau = 1;
        {   // threshold feedback every 2^sh new candidates of a query: ~k/4, at least 16. A small store on its own (no shared
            // thresholds) re-derives less often, at the first power of two >= 2k: with the staged emission a re-derivation
            // costs more there than the few candidates it saves (12.5 M rows, k = 100: 16 -> 73.8 ms per step, 64 -> 72.8,
            // 256 -> 70.8, 1024 -> 73.4), while at 100 M rows 256 is 0.7 % slower than 16 and on 2 GPUs with shared thresholds
            // 16..256 measure the same (profiles/r02m_shift_sweep.txt, r02m_n2_shift.txt, r02n_cfg3_n1.json)
            const bool sparse_feedback = !share_on && s->n_rows <= (32u << 20);
            uint32_t step = sparse_feedback ? std::max<uint32_t>(2 * k, 16) : std::max<uint32_t>(k / 4, 16), sh = 0;
            while ((2u << sh) <= step) sh++;
            if (sparse_feedback && (1u << sh) < step) sh++;
            static const int env_shift = [] { const char* e = getenv("ISX_TIGHTEN_SHIFT"); return e ? atoi(e) : -1; }();
            p.tighten_shift = env_shift >= 0 ? (uint32_t)env_shift : sh;
        }
        if (share_on) {
            for (uint32_t r = 0; r < s->share_world; r++) p.g_hist[r] = s->share_ptrs[r];
            p.g_world = s->share_world;
            p.g_rcap = isx_store::kShareRcap;
            p.g_q0 = (uint32_t)t.t0;
        }
        return p;
    };
    auto make_select = [&](const Tile& t, const ScanParams& p, size_t set = 0) {
        SelectParams sp{};
        sp.segs = p.segs; sp.hist = p.hist; sp.cand_cnt = p.cand_cnt; sp.cand = p.cand; sp.overflow = p.overflow;
        sp.qmap = s->d_qmap.as<uint32_t>() + t.t0;
        sp.C = C; sp.R = R; sp.k = k; sp.T = t.T; sp.qlen_bytes = t.Lq; sp.sort_cap = sort_cap; sp.key_words = key_words;
        sp.tau_init = tau_init;
        sp.out_khi = out.khi; sp.out_klo = out.klo; sp.out_h = out.h; sp.out_n = out.n; sp.out_cnt = out.cnt;
        sp.out_codes = out.codes;
        sp.fallback_info = s->d_fb.as<uint32_t>() + set * tile_max * 2;
        sp.skip_overflowed = 1;
        sp.big_scratch = big_P ? s->d_bigsort.as<BigRec>() + set * tile_max * big_P : nullptr;
        sp.big_P = big_P;
        return sp;
    };

    const bool lanes = n_sets > 1 && tiles.size() > 1;
    if (lanes) {   // the tile lanes start after everything enqueued so far (query upload, tables)
        CU(cudaEventRecord(s->lanes_begin, s->stream));
        for (size_t l = 0; l < n_sets; l++) CU(cudaStreamWaitEvent(s->lane_stream[l], s->lanes_begin, 0));
    }
    for (size_t ti = 0; ti < tiles.size(); ti++) {
        const Tile& t = tiles[ti];
        const uint32_t T = t.T, Lq = t.Lq;
        const int lane = lanes ? (int)(ti % n_sets) : -1;
        const size_t set = lanes ? (ti % n_sets) : 0;
        cudaStream_t ts = lanes ? s->lane_stream[lane] : s->stream;
        uint32_t* d_shist = s->d_shist.as<uint32_t>() + set * tile_max * R;
        st.passes++;
        ScanParams p = make_params(t, set);
        {
            size_t total = (size_t)T * R;
            uint32_t grid = (uint32_t)std::min<size_t>((total + 255) / 256, (size_t)s->sm_count * 8);
            grid = std::max<uint32_t>(grid, (T + 255) / 256);
            k_init_queries<<<grid, 256, 0, ts>>>(p.tau, p.hist, d_shist, p.cand_cnt, p.overflow, T, R, tau_init);
            CU(cudaGetLastError());
            st.kernel_launches++;
        }
        if (s->profiling) CU(cudaEventRecord(s->tile_events[3 * ti], ts));
        // threshold bootstrap from a stratified row sample (no emission), then one launch per compared length
        if (n_blocks_total > 0) {
            // batches: 64 blocks, refined by the two warm-up ranges below; small tiles: ~1 % of the store, because
            // their threshold feedback is slow relative to the scan (the first items of all CTAs run at once)
            // (sampling only 64 / world blocks per rank under shared thresholds was tried on 8 GPUs: 66.7 vs 65.2 ms per step,
            //  the looser first bounds cost more than the smaller sample saves - profiles/r02i_cfg3_n8.json)
            static const uint32_t env_sample = [] { const char* e = getenv("ISX_SAMPLE_BLOCKS"); return e ? (uint32_t)std::max(1, atoi(e)) : 64u; }();
            uint32_t want = T >= 64 ? env_sample : std::min<uint32_t>(1024, std::max<uint32_t>(64, n_blocks_total / 128));
            want = std::max<uint32_t>(want, (4 * k + kBlockRows - 1) / kBlockRows);
            SampleParams sp{};
            uint32_t total = 0;
            for (uint32_t L = 1; L <= kMaxBytes; L++) {
                uint32_t nb = s->bucket_block_lo[L + 1] - s->bucket_block_lo[L];
                uint32_t take = nb ? std::min<uint32_t>(nb, std::max<uint32_t>(1, (uint32_t)(((uint64_t)want * nb + n_blocks_total - 1) / n_blocks_total))) : 0;
                sp.bucket_first_block[L] = s->bucket_block_lo[L];
                sp.prefix[L] = total;
                total += take;
            }
            sp.prefix[kMaxBytes + 1] = total;
            // queries per sample CTA: their histograms share 32 KB of shared memory (21 queries at R = 385)
            sp.q_per_cta = std::max<uint32_t>(1, std::min<uint32_t>(T, (32u * 1024) / (R * 4)));
            sp.tail_only = (uint64_t)4 * k * 16 <= (uint64_t)total * kBlockRows ? 1 : 0;
            size_t smem = (size_t)sp.q_per_cta * R * 4 + 258 * 2 + 16;
            if (smem > 48 * 1024) CU(cudaFuncSetAttribute(k_sample, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            k_sample<<<dim3(total, (T + sp.q_per_cta - 1) / sp.q_per_cta, 1), kThreads, smem, ts>>>(p, sp, d_shist);
            CU(cudaGetLastError());
            k_sample_tau<<<(T * 32 + 255) / 256, 256, 0, ts>>>(d_shist, p.tau, T, R, k);
            CU(cudaGetLastError());
            st.kernel_launches += 2;
        }
        const uint32_t bpi_main = T >= 64 ? 4 : (T >= 8 ? 8 : 16);
        // Batches: the first wave of the bulk launch covers ~1.8 M rows before any threshold feedback, so the
        // threshold is first tightened on two short ranges (64 and 512 blocks) that are split over query
        // sub-tiles (gridDim.y) to fill the chip; every range is scanned exactly once.
        uint32_t done = 0;
        if (T >= 64) {
            // with shared thresholds all ranks warm up at once on `world` times the rows: each rank's share of the two
            // ranges shrinks accordingly (the ranges run at low occupancy, 5 % of a 12.5 M-row shard otherwise)
            const uint32_t w = share_on ? s->share_world : 1;
            static const int env_warm = [] { const char* e = getenv("ISX_WARM_RANGES"); return e ? atoi(e) : 2; }();
            int wi = 0;
            for (uint32_t span : {std::max(8u, 64u / w), std::max(64u, 512u / w)}) {
                if (wi++ >= env_warm || n_blocks_total - done <= span * 4) break;
                if ((rc = scan_range(s, p, done, done + span, bpi_main, lane))) return rc;
                done += span;
            }
        }
        if ((rc = scan_range(s, p, done, n_blocks_total, bpi_main, lane))) return rc;
        if (s->profiling) CU(cudaEventRecord(s->tile_events[3 * ti + 1], ts));

        SelectParams sp = make_select(t, p, set);
        k_select<<<T, kSelectThreads, sel_smem, ts>>>(sp);
        CU(cudaGetLastError());
        st.kernel_launches++;
        if (s->profiling) CU(cudaEventRecord(s->tile_events[3 * ti + 2], ts));
        // per-tile flags to pinned memory, no synchronisation (the state buffers are reused two tiles later in stream order)
        CU(cudaMemcpyAsync(hf_ovf + t.t0, p.overflow, (size_t)T * 4, cudaMemcpyDeviceToHost, ts));
        CU(cudaMemcpyAsync(hf_cnt + t.t0, p.cand_cnt, (size_t)T * 4, cudaMemcpyDeviceToHost, ts));
        CU(cudaMemcpyAsync(hf_info + 2 * t.t0, sp.fallback_info, (size_t)T * 8, cudaMemcpyDeviceToHost, ts));
        (void)Lq;
    }
    if (lanes) {
        for (size_t l = 0; l < n_sets; l++) {
            CU(cudaEventRecord(s->lane_done[l], s->lane_stream[l]));
            CU(cudaStreamWaitEvent(s->stream, s->lane_done[l], 0));
        }
    }
    CU(cudaStreamSynchronize(s->stream));
    if (s->profiling) {
        for (size_t ti = 0; ti < tiles.size(); ti++) {
            float a = 0, b = 0;
            CU(cudaEventElapsedTime(&a, s->tile_events[3 * ti], s->tile_events[3 * ti + 1]));
            CU(cudaEventElapsedTime(&b, s->tile_events[3 * ti + 1], s->tile_events[3 * ti + 2]));
            st.scan_ms += a;
            st.select_ms += b;
        }
    }
    for (size_t i = 0; i < Q; i++) st.candidates += hf_cnt[i];

    // exact re-scan of overflowed queries, one at a time: their histogram was still exact, so d* and the
    // number of rows with rank <= d* are known; collect exactly those rows with the fixed threshold d*.
    for (const Tile& t : tiles) {
        for (uint32_t qi = 0; qi < t.T; qi++) {
            if (!hf_ovf[t.t0 + qi]) continue;
            st.fallback_queries++;
            const uint32_t dstar = hf_info[2 * (t.t0 + qi)], count_le = hf_info[2 * (t.t0 + qi) + 1];
            // With shared thresholds the local histogram may under-count beyond the final global threshold, so the
            // buffer size is a first guess: the re-scan is repeated with a doubled buffer until nothing is dropped.
            size_t C2 = (size_t)count_le + 1024;
            for (;;) {
                if (s->d_fb_cand.ensure(C2 * 8)) return ISX_ENOMEM;
                ScanParams p2 = make_params(t);
                p2.queries += (size_t)qi * 8;
                p2.T = 1;
                p2.cand = s->d_fb_cand.as<uint64_t>();
                p2.C = (uint32_t)std::min<size_t>(C2, 0xffffffffu);
                p2.update_tau = 0;
                p2.g_world = 0;  // local, fixed threshold
                k_init_queries<<<std::max<uint32_t>(1, (R + 255) / 256), 256, 0, s->stream>>>(p2.tau, p2.hist, nullptr, p2.cand_cnt, p2.overflow, 1, R, dstar);
                CU(cudaGetLastError());
                st.kernel_launches++;
                if (s->profiling) CU(cudaEventRecord(s->ev[1], s->stream));
                if ((rc = scan_range(s, p2, 0, n_blocks_total, 16))) return rc;
                if (s->profiling) CU(cudaEventRecord(s->ev[2], s->stream));
                SelectParams sp2 = make_select(t, p2);
                sp2.cand = p2.cand; sp2.C = p2.C; sp2.T = 1; sp2.qmap += qi; sp2.tau_init = dstar;
                sp2.skip_overflowed = 1;  // a still-too-small buffer is reported, not silently truncated
                k_select<<<1, kSelectThreads, sel_smem, s->stream>>>(sp2);
                CU(cudaGetLastError());
                st.kernel_launches++;
                if (s->profiling) CU(cudaEventRecord(s->ev[3], s->stream));
                uint32_t again = 0, seen = 0;
                CU(cudaMemcpyAsync(&again, p2.overflow, 4, cudaMemcpyDeviceToHost, s->stream));
                CU(cudaMemcpyAsync(&seen, p2.cand_cnt, 4, cudaMemcpyDeviceToHost, s->stream));
                CU(cudaStreamSynchronize(s->stream));
                if (s->profiling) {
                    float a = 0, b = 0;
                    CU(cudaEventElapsedTime(&a, s->ev[1], s->ev[2]));
                    CU(cudaEventElapsedTime(&b, s->ev[2], s->ev[3]));
                    st.scan_ms += a;
                    st.select_ms += b;
                }
                if (!again) break;
                C2 = (size_t)seen + 1024;
            }
        }
    }
    if (s->profiling) {
        CU(cudaEventRecord(s->ev[3], s->stream));
        CU(cudaStreamSynchronize(s->stream));
        float t = 0;
        CU(cudaEventElapsedTime(&t, s->ev[0], s->ev[3]));
        st.total_ms = t;
    }
    return 0;
}

// ---- self-join (join.cuh, DESIGN.md §3.7) ------------------------------------------------------------------------------
constexpr uint32_t kJoinCap = 1024;   // candidate list per query of a chunk; a query with more partners is re-scanned exactly

// grow a device buffer to at least `want` bytes, keeping its first `used` bytes; ISX_ENOMEM (no message, the error state
// cleared) when the device has no room - the caller decides what that means
static int grow_keep(isx_store* s, DevBuf& b, size_t used, size_t want) {
    if (want <= b.cap) return 0;
    void* p = nullptr;
    size_t bytes = want + want / 4 + 256;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e != cudaSuccess) { cudaGetLastError(); bytes = want; e = cudaMalloc(&p, bytes); }
    if (e != cudaSuccess) { cudaGetLastError(); return ISX_ENOMEM; }
    if (used) {
        e = cudaMemcpyAsync(p, b.p, used, cudaMemcpyDeviceToDevice, s->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s->stream);
        if (e != cudaSuccess) { cudaFree(p); return fail(ISX_ECUDA, "self-join: copying the pair records failed: %s", cudaGetErrorString(e)); }
    }
    if (b.p) cudaFree(b.p);
    b.p = p;
    b.cap = bytes;
    return 0;
}

static void release_join(isx_store* s) {
    for (DevBuf* b : {&s->d_join_keys[0], &s->d_join_keys[1], &s->d_join_vals[0], &s->d_join_vals[1], &s->d_join_tmp}) b->release();
    s->join_valid = false;
    s->join_total = 0;
}

// Every unordered pair of stored rows with h * thr_den <= thr_num * nbits, sorted by (key_a, key_b), left in d_join_*.
// The live blocks are walked in list order (ascending length, segments in order) in chunks of <= kMaxTile rows of one
// segment; a chunk's rows become a query tile that is scanned with a fixed threshold against [chunk's first block, end):
// the rest of its own bucket and every longer bucket. So a pair of different lengths is scored once, from its shorter row,
// and a pair of one length from its earlier row; k_join_pairs drops what a chunk sees of itself from the other side.
static int self_join_core(isx_store* s, uint32_t thr_num, uint32_t thr_den, uint64_t* total_out) {
    isx_stats_t& st = s->stats;
    st = isx_stats_t{};
    s->join_valid = false;   // the record buffers of the last join are reused
    s->join_total = 0;
    int rc;
    if ((rc = upload_segs(s)) || (rc = upload_blocks(s))) return rc;
    const uint32_t n_blocks_total = (uint32_t)s->h_blocks.size();
    const bool wide = s->key_bytes == 16;
    const size_t kb = wide ? sizeof(JoinKey16) : sizeof(JoinKey8);
    uint32_t mask = 0;   // the compared lengths of all pairs are exactly the stored lengths
    for (uint32_t L = 1; L <= kMaxBytes; L++) if (s->bucket_rows[L]) mask |= 1u << (L - 1);
    if (n_blocks_total == 0 || s->n_rows < 2) {
        s->join_valid = true;
        s->join_version = s->version;
        return 0;
    }
    if ((rc = build_tables(s, mask))) return rc;
    const RankTables& tb = s->tables;
    const uint32_t R = tb.R;
    uint32_t tau = 0;   // largest rank whose fraction is <= thr_num / thr_den
    while (tau + 1 < R && (uint64_t)tb.frac_h[tau + 1] * thr_den <= (uint64_t)thr_num * tb.frac_n[tau + 1]) tau++;
    const uint32_t TM = kMaxTile, C = kJoinCap;
    if (s->d_queries.ensure((size_t)TM * 32) || s->d_tau.ensure((size_t)TM * 4) || s->d_hist.ensure((size_t)TM * R * 4) ||
        s->d_cnt.ensure((size_t)TM * 4) || s->d_ovf.ensure((size_t)TM * 4) || s->d_cand.ensure((size_t)TM * C * 8) ||
        s->d_join_rows.ensure((size_t)TM * 4) || s->d_join_cnt.ensure(8) || s->h_flags.ensure((size_t)TM * 4 + 16) ||
        s->h_qmap.ensure((size_t)TM * 4))
        return ISX_ENOMEM;
    CU(cudaMemsetAsync(s->d_join_cnt.p, 0, 8, s->stream));
    uint32_t* h_cnt = s->h_flags.as<uint32_t>();
    unsigned long long* h_pairs = reinterpret_cast<unsigned long long*>(s->h_flags.as<uint8_t>() + (size_t)TM * 4);
    uint64_t cap = std::min<uint64_t>(s->d_join_keys[0].cap / kb, s->d_join_vals[0].cap / 4);   // pair records the output holds
    bool counting_only = false;   // the device had no room for more records: the join only counts from here on

    // scan a tile of T rows of segment `seg` (rows row0.. or the device list d_rows) against [b0, end); on return the
    // exact candidate counts are in h_cnt and the records appended so far in *h_pairs
    auto scan_tile = [&](uint32_t seg, uint32_t row0, const uint32_t* d_rows, uint32_t T, uint32_t b0, uint32_t Ct) -> int {
        k_rows_as_queries<<<(T * 8 + 255) / 256, 256, 0, s->stream>>>(s->d_segs.as<SegDesc>(), seg, row0, d_rows, T, s->d_queries.as<uint32_t>());
        CU(cudaGetLastError());
        k_init_queries<<<std::max<uint32_t>(1, std::min<uint32_t>((T * R + 255) / 256, (uint32_t)s->sm_count * 8)), 256, 0, s->stream>>>(
            s->d_tau.as<uint32_t>(), s->d_hist.as<uint32_t>(), nullptr, s->d_cnt.as<uint32_t>(), s->d_ovf.as<uint32_t>(), T, R, tau);
        CU(cudaGetLastError());
        st.kernel_launches += 2;
        ScanParams p{};
        p.segs = s->d_segs.as<SegDesc>();
        p.blocks = s->d_blocks.as<uint2>();
        p.queries = s->d_queries.as<uint32_t>();
        p.T = T;
        p.qlen_bytes = s->segs[seg].len_bytes;
        p.tau = s->d_tau.as<uint32_t>();
        p.hist = s->d_hist.as<uint32_t>();
        p.cand_cnt = s->d_cnt.as<uint32_t>();
        p.cand = s->d_cand.as<uint64_t>();
        p.overflow = s->d_ovf.as<uint32_t>();
        p.C = Ct; p.R = R; p.k = 1;
        p.rank_tab = tb.d_rank.as<uint16_t>();
        p.hmax_tab = tb.d_hmax.as<uint16_t>();
        p.update_tau = 0;   // fixed threshold: every row within it is emitted
        if (s->profiling) CU(cudaEventRecord(s->ev[1], s->stream));
        int rc2 = scan_range(s, p, b0, n_blocks_total, T >= 64 ? 4 : 16);
        if (rc2) return rc2;
        if (s->profiling) CU(cudaEventRecord(s->ev[2], s->stream));
        CU(cudaMemcpyAsync(h_cnt, p.cand_cnt, (size_t)T * 4, cudaMemcpyDeviceToHost, s->stream));
        CU(cudaMemcpyAsync(h_pairs, s->d_join_cnt.p, 8, cudaMemcpyDeviceToHost, s->stream));
        CU(cudaStreamSynchronize(s->stream));
        if (s->profiling) {
            float t = 0;
            CU(cudaEventElapsedTime(&t, s->ev[1], s->ev[2]));
            st.scan_ms += t;
        }
        return 0;
    };
    // candidate lists of the tile just scanned -> pair records; `bound` >= the records it can append
    auto append = [&](uint32_t seg, uint32_t row0, const uint32_t* d_rows, uint32_t T, uint32_t Ct, uint64_t bound) -> int {
        const uint64_t have = *h_pairs, need = have + bound;
        if (!counting_only && need > cap) {
            const uint64_t used = std::min(have, cap);
            int rc2 = grow_keep(s, s->d_join_keys[0], used * kb, need * kb);
            if (!rc2) rc2 = grow_keep(s, s->d_join_vals[0], used * 4, need * 4);
            if (rc2 && rc2 != ISX_ENOMEM) return rc2;
            counting_only = rc2 == ISX_ENOMEM;
            cap = std::min<uint64_t>(s->d_join_keys[0].cap / kb, s->d_join_vals[0].cap / 4);
        }
        JoinParams jp{};
        jp.segs = s->d_segs.as<SegDesc>();
        jp.cand = s->d_cand.as<uint64_t>();
        jp.cand_cnt = s->d_cnt.as<uint32_t>();
        jp.C = Ct; jp.T = T; jp.seg = seg; jp.row0 = row0; jp.rows = d_rows;
        jp.counter = s->d_join_cnt.as<unsigned long long>();
        jp.cap = cap;
        jp.vals = s->d_join_vals[0].as<uint32_t>();
        const unsigned grid = (T * 32 + 255) / 256;
        if (wide) k_join_pairs<JoinKey16><<<grid, 256, 0, s->stream>>>(jp, s->d_join_keys[0].as<JoinKey16>());
        else k_join_pairs<JoinKey8><<<grid, 256, 0, s->stream>>>(jp, s->d_join_keys[0].as<JoinKey8>());
        CU(cudaGetLastError());
        st.kernel_launches++;
        return 0;
    };

    std::vector<uint32_t> ovf_rows, ovf_cnt;
    for (uint32_t b0 = 0; b0 < n_blocks_total; b0++) {
        const uint32_t seg = s->h_blocks[b0].x, row0 = s->h_blocks[b0].y;
        if (row0 % TM) continue;   // chunks start every kMaxTile rows of a segment (two blocks; capacities are multiples of 4096)
        const uint32_t T = std::min<uint32_t>(TM, s->segs[seg].desc.n - row0);
        st.passes++;
        if ((rc = scan_tile(seg, row0, nullptr, T, b0, C))) return rc;
        uint64_t bound = 0;
        ovf_rows.clear();
        ovf_cnt.clear();
        for (uint32_t i = 0; i < T; i++) {
            st.candidates += h_cnt[i];
            if (h_cnt[i] <= C) bound += h_cnt[i];
            else { ovf_rows.push_back(row0 + i); ovf_cnt.push_back(h_cnt[i]); }
        }
        if ((rc = append(seg, row0, nullptr, T, C, bound))) return rc;
        // queries whose list overflowed: re-scanned together, with C = their largest count (so nothing overflows again),
        // in as few tiles as a 1 GB candidate budget allows
        st.fallback_queries += ovf_rows.size();
        for (size_t i0 = 0; i0 < ovf_rows.size();) {
            size_t i1 = i0;
            uint32_t Ct = 0;
            while (i1 < ovf_rows.size()) {
                const uint32_t c = std::max(Ct, ovf_cnt[i1]);
                if (i1 > i0 && (uint64_t)(i1 - i0 + 1) * c * 8 > ((uint64_t)1 << 30)) break;
                Ct = c;
                i1++;
            }
            const uint32_t To = (uint32_t)(i1 - i0);
            if (s->d_cand.ensure((size_t)To * Ct * 8)) return ISX_ENOMEM;
            memcpy(s->h_qmap.p, ovf_rows.data() + i0, (size_t)To * 4);
            CU(cudaMemcpyAsync(s->d_join_rows.p, s->h_qmap.p, (size_t)To * 4, cudaMemcpyHostToDevice, s->stream));
            if ((rc = scan_tile(seg, 0, s->d_join_rows.as<uint32_t>(), To, b0, Ct))) return rc;
            uint64_t bound2 = 0;
            for (uint32_t i = 0; i < To; i++) {
                if (h_cnt[i] != ovf_cnt[i0 + i])
                    return fail(ISX_ECUDA, "self-join: the re-scan of an overflowed row found %u partners, the first scan %u", h_cnt[i], ovf_cnt[i0 + i]);
                bound2 += h_cnt[i];
            }
            if ((rc = append(seg, 0, s->d_join_rows.as<uint32_t>(), To, Ct, bound2))) return rc;
            i0 = i1;
        }
    }
    CU(cudaMemcpyAsync(h_pairs, s->d_join_cnt.p, 8, cudaMemcpyDeviceToHost, s->stream));
    CU(cudaStreamSynchronize(s->stream));
    const uint64_t total = *h_pairs;
    *total_out = total;
    const size_t per_pair = 2 * (kb + 4);
    auto no_room = [&]() {
        release_join(s);
        return fail(ISX_ENOMEM, "self-join found %llu pairs; they do not fit in device memory (%zu bytes per pair with the sort)",
                    (unsigned long long)total, per_pair);
    };
    if (counting_only || total > cap) return no_room();
    if (total > 1) {   // sort by (key_a, key_b) on the device: LSD radix passes over the key words
        if (grow_keep(s, s->d_join_keys[1], 0, total * kb) || grow_keep(s, s->d_join_vals[1], 0, total * 4)) return no_room();
        size_t tmp_bytes = 0;
        cudaError_t e;
        if (wide) {
            cub::DoubleBuffer<JoinKey16> dk(s->d_join_keys[0].as<JoinKey16>(), s->d_join_keys[1].as<JoinKey16>());
            cub::DoubleBuffer<uint32_t> dv(s->d_join_vals[0].as<uint32_t>(), s->d_join_vals[1].as<uint32_t>());
            CU(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, dk, dv, total, JoinKey16Bits{}, s->stream));
            if (grow_keep(s, s->d_join_tmp, 0, tmp_bytes)) return no_room();
            e = cub::DeviceRadixSort::SortPairs(s->d_join_tmp.p, tmp_bytes, dk, dv, total, JoinKey16Bits{}, s->stream);
            s->join_cur = (uint32_t)dk.selector;
        } else {
            cub::DoubleBuffer<JoinKey8> dk(s->d_join_keys[0].as<JoinKey8>(), s->d_join_keys[1].as<JoinKey8>());
            cub::DoubleBuffer<uint32_t> dv(s->d_join_vals[0].as<uint32_t>(), s->d_join_vals[1].as<uint32_t>());
            CU(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, dk, dv, total, JoinKey8Bits{}, s->stream));
            if (grow_keep(s, s->d_join_tmp, 0, tmp_bytes)) return no_room();
            e = cub::DeviceRadixSort::SortPairs(s->d_join_tmp.p, tmp_bytes, dk, dv, total, JoinKey8Bits{}, s->stream);
            s->join_cur = (uint32_t)dk.selector;
        }
        CU(e);
        CU(cudaStreamSynchronize(s->stream));
        st.kernel_launches++;   // the sort counts as one step (CUB launches several kernels)
    } else {
        s->join_cur = 0;
    }
    s->join_total = total;
    s->join_version = s->version;
    s->join_valid = true;
    return 0;
}

}  // namespace isx

// =================================================================================================
// C ABI
// =================================================================================================
extern "C" {

const char* isx_last_error(void) { return g_err.c_str(); }
int isx_abi_version(void) { return ISX_ABI_VERSION; }

int isx_device_count(int* n_out) {
    if (!n_out) return fail(ISX_EINVAL, "n_out is NULL");
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) { *n_out = 0; return fail(ISX_ECUDA, "cudaGetDeviceCount: %s", cudaGetErrorString(e)); }
    *n_out = n;
    return 0;
}

int isx_open(isx_store_t** out, int device, uint32_t key_bytes, uint32_t max_bytes, uint32_t fixed_len) {
    if (!out) return fail(ISX_EINVAL, "out is NULL");
    *out = nullptr;
    if (key_bytes != 8 && key_bytes != 16) return fail(ISX_EINVAL, "key_bytes must be 8 or 16, got %u", key_bytes);
    if (max_bytes < 1 || max_bytes > ISX_MAX_BYTES) return fail(ISX_EINVAL, "max_bytes must be 1..32, got %u", max_bytes);
    if (fixed_len > max_bytes) return fail(ISX_EINVAL, "fixed_len %u exceeds max_bytes %u", fixed_len, max_bytes);
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(ISX_ECUDA, "no CUDA device available (%s) - this library has no CPU fallback", e != cudaSuccess ? cudaGetErrorString(e) : "0 devices");
    if (device < 0 || device >= n) return fail(ISX_EINVAL, "device %d out of range (have %d)", device, n);
    CU(cudaSetDevice(device));
    isx_store* s = new (std::nothrow) isx_store();
    if (!s) return fail(ISX_ENOMEM, "out of host memory");
    s->device = device;
    s->key_bytes = key_bytes;
    s->max_bytes = max_bytes;
    s->fixed_len = fixed_len;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { delete s; return fail(ISX_ECUDA, "cudaGetDeviceProperties failed"); }
    if (prop.major < 10) { delete s; return fail(ISX_ECUDA, "device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, prop.major, prop.minor); }
    s->sm_count = prop.multiProcessorCount;
    s->max_smem_optin = (int)prop.sharedMemPerBlockOptin;
    s->smem_per_sm = (int)prop.sharedMemPerMultiprocessor;
    s->small_ok = prop.cooperativeLaunch != 0;
    if (cudaStreamCreateWithFlags(&s->own_stream, cudaStreamNonBlocking) != cudaSuccess) { delete s; return fail(ISX_ECUDA, "cudaStreamCreate failed"); }
    s->stream = s->own_stream;
    for (auto& ev : s->ev)
        if (cudaEventCreate(&ev) != cudaSuccess) { delete s; return fail(ISX_ECUDA, "cudaEventCreate failed"); }
    for (int i = 0; i < 3; i++) {
        if (cudaStreamCreateWithFlags(&s->side[i], cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreateWithFlags(&s->join_ev[i], cudaEventDisableTiming) != cudaSuccess) { delete s; return fail(ISX_ECUDA, "side stream setup failed"); }
    }
    if (cudaEventCreateWithFlags(&s->fork_ev, cudaEventDisableTiming) != cudaSuccess) { delete s; return fail(ISX_ECUDA, "cudaEventCreate failed"); }
    {
        bool ok = cudaEventCreateWithFlags(&s->lanes_begin, cudaEventDisableTiming) == cudaSuccess;
        for (int l = 0; l < kMaxLanes && ok; l++) {
            ok = ok && cudaStreamCreateWithFlags(&s->lane_stream[l], cudaStreamNonBlocking) == cudaSuccess &&
                 cudaEventCreateWithFlags(&s->lane_fork[l], cudaEventDisableTiming) == cudaSuccess &&
                 cudaEventCreateWithFlags(&s->lane_done[l], cudaEventDisableTiming) == cudaSuccess;
            for (int i = 0; i < 3 && ok; i++)
                ok = cudaStreamCreateWithFlags(&s->lane_side[l][i], cudaStreamNonBlocking) == cudaSuccess &&
                     cudaEventCreateWithFlags(&s->lane_join[l][i], cudaEventDisableTiming) == cudaSuccess;
        }
        if (!ok) { delete s; return fail(ISX_ECUDA, "tile lane stream setup failed"); }
    }
    *out = s;
    return 0;
}

static void free_rows(isx_store* s) {
    for (auto& sg : s->segs) if (sg.d_mem) cudaFree(sg.d_mem);
    s->segs.clear();
    for (auto& v : s->bucket_segs) v.clear();
    memset(s->bucket_rows, 0, sizeof s->bucket_rows);
    s->device_bytes = 0;
    s->map.clear();
    s->map_stale.store(false);
    s->n_rows = 0;
    s->segs_dirty = true;
    s->version++;
}

int isx_close(isx_store_t* s) {
    if (!s) return 0;
    {   // wait for searches / mutations in flight on other threads (they hold rows_mu shared or work_mu); a call that
        // arrives after this point is a use-after-close of the caller, as with any handle
        std::unique_lock<std::shared_mutex> g(s->rows_mu);
        std::lock_guard<std::mutex> gw(s->work_mu);
        cudaSetDevice(s->device);
        cudaStreamSynchronize(s->stream);
        free_rows(s);
    }
    DevBuf* bufs[] = {&s->d_segs, &s->d_blocks, &s->tables.d_rank, &s->tables.d_hmax, &s->d_stage_codes, &s->d_stage_keys,
                      &s->d_stage_dest, &s->d_moves, &s->d_queries, &s->d_tau, &s->d_hist, &s->d_shist, &s->d_cnt, &s->d_ovf, &s->d_cand,
                      &s->d_qmap, &s->d_fb, &s->d_fb_cand, &s->d_out_khi, &s->d_out_klo, &s->d_out_h, &s->d_out_n,
                      &s->d_out_cnt, &s->d_out_codes, &s->d_bigsort, &s->d_bdesc, &s->d_bulk, &s->d_small,
                      &s->d_join_keys[0], &s->d_join_keys[1], &s->d_join_vals[0], &s->d_join_vals[1], &s->d_join_tmp,
                      &s->d_join_rows, &s->d_join_cnt};
    for (DevBuf* b : bufs) b->release();
    PinnedBuf* pbufs[] = {&s->h_queries, &s->h_qmap, &s->h_flags, &s->h_out, &s->h_small_info, &s->h_small_dbg};
    for (PinnedBuf* b : pbufs) b->release();
    for (uint32_t r = 0; r < s->share_world; r++)
        if (r != s->share_rank && s->share_ptrs[r]) cudaIpcCloseMemHandle(s->share_ptrs[r]);
    if (s->share_local) cudaFree(s->share_local);
    for (auto& ev : s->ev) if (ev) cudaEventDestroy(ev);
    for (auto& ev : s->tile_events) cudaEventDestroy(ev);
    for (int i = 0; i < 3; i++) { if (s->side[i]) cudaStreamDestroy(s->side[i]); if (s->join_ev[i]) cudaEventDestroy(s->join_ev[i]); }
    if (s->fork_ev) cudaEventDestroy(s->fork_ev);
    if (s->lanes_begin) cudaEventDestroy(s->lanes_begin);
    for (int l = 0; l < kMaxLanes; l++) {
        for (int i = 0; i < 3; i++) { if (s->lane_side[l][i]) cudaStreamDestroy(s->lane_side[l][i]); if (s->lane_join[l][i]) cudaEventDestroy(s->lane_join[l][i]); }
        if (s->lane_fork[l]) cudaEventDestroy(s->lane_fork[l]);
        if (s->lane_done[l]) cudaEventDestroy(s->lane_done[l]);
        if (s->lane_stream[l]) cudaStreamDestroy(s->lane_stream[l]);
    }
    if (s->own_stream) cudaStreamDestroy(s->own_stream);
    delete s;
    return 0;
}

int isx_release_scratch(isx_store_t* s, uint64_t* bytes_freed) {
    if (!s) return fail(ISX_EINVAL, "store is NULL");
    std::shared_lock<std::shared_mutex> g(s->rows_mu);
    std::lock_guard<std::mutex> gw(s->work_mu);
    int rc = set_device(s);
    if (rc) return rc;
    CU(cudaStreamSynchronize(s->stream));
    // per-search working memory only (candidate lists, histograms, result and staging buffers): everything re-grows on
    // demand; rows, keys, descriptors, rank tables and the small-batch state stay
    DevBuf* bufs[] = {&s->d_stage_codes, &s->d_stage_keys, &s->d_stage_dest, &s->d_moves, &s->d_queries, &s->d_tau, &s->d_hist, &s->d_shist,
                      &s->d_cnt, &s->d_ovf, &s->d_cand, &s->d_qmap, &s->d_fb, &s->d_fb_cand, &s->d_out_khi, &s->d_out_klo, &s->d_out_h,
                      &s->d_out_n, &s->d_out_cnt, &s->d_out_codes, &s->d_bigsort, &s->d_bulk, &s->d_join_keys[0], &s->d_join_keys[1],
                      &s->d_join_vals[0], &s->d_join_vals[1], &s->d_join_tmp, &s->d_join_rows, &s->d_join_cnt};
    s->join_valid = false;   // the self-join result lives in this working memory
    uint64_t freed = 0;
    for (DevBuf* b : bufs) { freed += b->cap; b->release(); }
    if (bytes_freed) *bytes_freed = freed;
    return 0;
}

int isx_set_stream(isx_store_t* s, void* cuda_stream) {
    if (!s) return fail(ISX_EINVAL, "store is NULL");
    std::lock_guard<std::mutex> g(s->work_mu);
    s->stream = cuda_stream ? reinterpret_cast<cudaStream_t>(cuda_stream) : s->own_stream;
    return 0;
}

int isx_set_profiling(isx_store_t* s, int enabled) {
    if (!s) return fail(ISX_EINVAL, "store is NULL");
    s->profiling = enabled != 0;
    return 0;
}

int isx_get_stats(isx_store_t* s, isx_stats_t* out) {
    if (!s || !out) return fail(ISX_EINVAL, "NULL argument");
    std::lock_guard<std::mutex> g(s->work_mu);
    *out = s->stats;
    return 0;
}

int isx_size(isx_store_t* s, uint64_t* n_out) {
    if (!s || !n_out) return fail(ISX_EINVAL, "NULL argument");
    std::shared_lock<std::shared_mutex> g(s->rows_mu);
    *n_out = s->n_rows;
    return 0;
}

int isx_device_bytes(isx_store_t* s, uint64_t* n_out) {
    if (!s || !n_out) return fail(ISX_EINVAL, "NULL argument");
    std::shared_lock<std::shared_mutex> g(s->rows_mu);
    *n_out = s->device_bytes;
    return 0;
}

int isx_length_mask(isx_store_t* s, uint32_t* mask_out) {
    if (!s || !mask_out) return fail(ISX_EINVAL, "NULL argument");
    std::shared_lock<std::shared_mutex> g(s->rows_mu);
    uint32_t m = 0;
    for (uint32_t L = 1; L <= kMaxBytes; L++) if (s->bucket_rows[L]) m |= 1u << (L - 1);
    *mask_out = m;
    return 0;
}

int isx_max_k(isx_store_t* s, uint32_t* k_out) {
    if (!s || !k_out) return fail(ISX_EINVAL, "NULL argument");
    *k_out = kMaxK;
    return 0;
}

int isx_clear(isx_store_t* s) {
    if (!s) return fail(ISX_EINVAL, "store is NULL");
    std::unique_lock<std::shared_mutex> g(s->rows_mu);
    int rc = set_device(s);
    if (rc) return rc;
    CU(cudaStreamSynchronize(s->stream));
    free_rows(s);
    return 0;
}

int isx_add(isx_store_t* s, const void* keys, const uint8_t* codes, const uint8_t* lens, size_t n, uint8_t* added) {
    if (!s) return fail(ISX_EINVAL, "store is NULL");
    if (n == 0) return 0;
    if (!keys || !codes || !lens) return fail(ISX_EINVAL, "NULL input array");
    std::unique_lock<std::shared_mutex> g(s->rows_mu);
    std::lock_guard<std::mutex> gw(s->work_mu);
    int rc = set_device(s);
    if (rc) return rc;
    if ((rc = sync_map(s))) return rc;
    for (size_t i = 0; i < n; i++) {
        uint32_t L = lens[i];
        if (L < 1 || L > s->max_bytes) return fail(ISX_EINVAL, "row %zu: code length %u bytes outside 1..%u", i, L, s->max_bytes);
        if (s->fixed_len && L != s->fixed_len) return fail(ISX_EINVAL, "row %zu: code length %u bytes, index expects %u", i, L, s->fixed_len);
    }
    // staging buffers first: an allocation failure must not leave the key map ahead of the device rows
    {
        const size_t cn0 = std::min<size_t>((size_t)4 << 20, n);
        if (s->d_stage_codes.ensure(cn0 * 32) || s->d_stage_keys.ensure(cn0 * s->key_bytes) || s->d_stage_dest.ensure(cn0 * 8)) return ISX_ENOMEM;
    }
    s->map.reserve(s->map.size() + n);
    // rows needed per bucket (upper bound: duplicates are skipped later) so big batches get big segments
    uint64_t need[kMaxBytes + 1] = {0};
    for (size_t i = 0; i < n; i++) need[lens[i]]++;

    std::vector<uint64_t> dest(n, ~0ull);
    const size_t PF = 16;
    for (size_t i = 0; i < std::min(n, PF); i++) s->map.prefetch(load_key(s, keys, i));
    size_t n_added = 0;
    for (size_t i = 0; i < n; i++) {
        if (i + PF < n) s->map.prefetch(load_key(s, keys, i + PF));
        Key128 key = load_key(s, keys, i);
        uint32_t L = lens[i];
        uint64_t dummy;
        if (s->map.find(key, &dummy)) { if (added) added[i] = 0; need[L]--; continue; }
        // segment with room in bucket L
        auto& bs = s->bucket_segs[L];
        if (bs.empty() || s->segs[bs.back()].desc.n == s->segs[bs.back()].desc.cap) {
            uint32_t grow = bs.empty() ? kMinSegRows : std::min<uint64_t>((uint64_t)s->segs[bs.back()].desc.cap * 4, kMaxSegRows);
            uint64_t want = std::max<uint64_t>(grow, std::min<uint64_t>(need[L], kMaxSegRows));
            uint32_t cap = (uint32_t)((want + kMinSegRows - 1) / kMinSegRows * kMinSegRows);
            if ((rc = new_segment(s, L, cap))) return rc;
        }
        uint32_t sid = bs.back();
        Segment& sg = s->segs[sid];
        uint32_t row = sg.desc.n++;
        sg.mirrored = sg.desc.n;
        sg.h_khi[row] = key.hi;
        if (s->key_bytes == 16) sg.h_klo[row] = key.lo;
        uint64_t loc = ((uint64_t)sid << 32) | row;
        s->map.insert(key, loc);
        dest[i] = loc;
        s->bucket_rows[L]++;
        s->n_rows++;
        need[L]--;
        if (added) added[i] = 1;
        n_added++;
    }
    if (n_added == 0) return 0;
    s->segs_dirty = true;
    s->version++;
    if ((rc = upload_segs(s))) return rc;
    // stage + scatter in chunks (bounded staging memory)
    const size_t CH = (size_t)4 << 20;
    for (size_t c0 = 0; c0 < n; c0 += CH) {
        size_t cn = std::min(CH, n - c0);
        if (s->d_stage_codes.ensure(cn * 32) || s->d_stage_keys.ensure(cn * s->key_bytes) || s->d_stage_dest.ensure(cn * 8)) return ISX_ENOMEM;
        CU(cudaMemcpyAsync(s->d_stage_codes.p, codes + c0 * 32, cn * 32, cudaMemcpyHostToDevice, s->stream));
        CU(cudaMemcpyAsync(s->d_stage_keys.p, reinterpret_cast<const uint8_t*>(keys) + c0 * s->key_bytes, cn * s->key_bytes, cudaMemcpyHostToDevice, s->stream));
        CU(cudaMemcpyAsync(s->d_stage_dest.p, dest.data() + c0, cn * 8, cudaMemcpyHostToDevice, s->stream));
        k_scatter_rows<<<(unsigned)((cn + 255) / 256), 256, 0, s->stream>>>(s->d_segs.as<SegDesc>(), s->d_stage_dest.as<uint64_t>(),
                                                                            s->d_stage_codes.as<uint8_t>(), s->d_stage_keys.as<uint8_t>(),
                                                                            s->key_bytes, cn);
        CU(cudaGetLastError());
        CU(cudaStreamSynchronize(s->stream));
    }
    return 0;
}

int isx_remove(isx_store_t* s, const void* keys, size_t n, uint8_t* removed, uint64_t* n_removed) {
    if (!s) return fail(ISX_EINVAL, "store is NULL");
    if (n_removed) *n_removed = 0;
    if (n == 0) return 0;
    if (!keys) return fail(ISX_EINVAL, "NULL input array");
    std::unique_lock<std::shared_mutex> g(s->rows_mu);
    std::lock_guard<std::mutex> gw(s->work_mu);
    int rc = set_device(s);
    if (rc) return rc;
    if ((rc = sync_map(s))) return rc;
    // Swap-remove on the host mirrors, one key at a time; the device copies are deferred: `origin` maps a row that now
    // holds moved data to the ORIGINAL location of that data, so a chain (row moved into a hole, hole removed again
    // later in the batch) collapses to one net move - or to none when the moved row was removed as well.
    std::unordered_map<uint64_t, uint64_t> origin;
    uint64_t cnt = 0;
    for (size_t i = 0; i < n; i++) {
        Key128 key = load_key(s, keys, i);
        uint64_t loc;
        if (!s->map.find(key, &loc)) { if (removed) removed[i] = 0; continue; }
        uint32_t sid = (uint32_t)(loc >> 32), row = (uint32_t)loc;
        uint32_t L = s->segs[sid].len_bytes;
        // last live row of the bucket
        auto& bs = s->bucket_segs[L];
        size_t li = bs.size();
        while (li > 0 && s->segs[bs[li - 1]].desc.n == 0) li--;
        uint32_t lsid = bs[li - 1];
        Segment& last = s->segs[lsid];
        uint32_t lrow = last.desc.n - 1;
        const uint64_t last_loc = ((uint64_t)lsid << 32) | lrow;
        s->map.erase(key);
        origin.erase(loc);   // whatever was moved here before is gone now
        if (last_loc != loc) {
            Key128 moved{last.h_khi[lrow], s->key_bytes == 16 ? last.h_klo[lrow] : 0};
            Segment& dst = s->segs[sid];
            dst.h_khi[row] = moved.hi;
            if (s->key_bytes == 16) dst.h_klo[row] = moved.lo;
            s->map.update(moved, loc);
            auto it = origin.find(last_loc);
            const uint64_t src = it == origin.end() ? last_loc : it->second;
            if (it != origin.end()) origin.erase(it);
            origin[loc] = src;
        }
        last.desc.n--;
        last.mirrored = last.desc.n;
        s->bucket_rows[L]--;
        s->n_rows--;
        if (removed) removed[i] = 1;
        cnt++;
    }
    if (n_removed) *n_removed = cnt;
    if (cnt == 0) return 0;
    std::vector<uint4> moves;
    moves.reserve(origin.size());
    for (const auto& kv : origin)
        moves.push_back(make_uint4((uint32_t)(kv.first >> 32), (uint32_t)kv.first, (uint32_t)(kv.second >> 32), (uint32_t)kv.second));
    s->segs_dirty = true;
    s->version++;
    if ((rc = upload_segs(s))) return rc;
    if (!moves.empty()) {
        if (s->d_moves.ensure(moves.size() * sizeof(uint4))) return ISX_ENOMEM;
        CU(cudaMemcpyAsync(s->d_moves.p, moves.data(), moves.size() * sizeof(uint4), cudaMemcpyHostToDevice, s->stream));
        k_move_rows<<<(unsigned)((moves.size() * 32 + 255) / 256), 256, 0, s->stream>>>(s->d_segs.as<SegDesc>(), s->d_moves.as<uint4>(), moves.size());
        CU(cudaGetLastError());
        CU(cudaStreamSynchronize(s->stream));
    }
    return 0;
}

// rows [i0, i0+cn) of a device batch -> free rows of their length buckets (caller holds both locks)
static int add_device_chunk(isx_store* s, const uint8_t* d_keys, const uint8_t* d_codes, const uint8_t* d_lens, uint32_t uniform_len, size_t cn) {
    int rc;
    uint32_t counts[256] = {0};
    if (s->d_bulk.ensure(256 * 4 + 64 * 4)) return ISX_ENOMEM;
    uint32_t* d_hist = s->d_bulk.as<uint32_t>();
    uint32_t* d_cursor = d_hist + 256;
    CU(cudaMemsetAsync(d_hist, 0, (256 + 64) * 4, s->stream));
    if (d_lens) {
        k_len_hist<<<std::min<size_t>((cn + 4095) / 4096, (size_t)s->sm_count * 8), 256, 0, s->stream>>>(d_lens, cn, d_hist);
        CU(cudaGetLastError());
        CU(cudaMemcpyAsync(counts, d_hist, sizeof counts, cudaMemcpyDeviceToHost, s->stream));
        CU(cudaStreamSynchronize(s->stream));
    } else {
        counts[uniform_len] = (uint32_t)cn;
    }
    for (uint32_t L = 0; L < 256; L++) {
        if (!counts[L]) continue;
        if (L < 1 || L > s->max_bytes) return fail(ISX_EINVAL, "isx_add_device: code length %u bytes outside 1..%u", L, s->max_bytes);
        if (s->fixed_len && L != s->fixed_len) return fail(ISX_EINVAL, "isx_add_device: code length %u bytes, index expects %u", L, s->fixed_len);
    }
    // plan: spans of free rows per length class (tail of the bucket's last segment, then fresh segments); nothing is
    // committed to the descriptors before the whole plan fits
    struct Pending { uint32_t L, sid, row0, cnt; };
    std::vector<Pending> pend;
    std::vector<std::pair<uint32_t, uint32_t>> fresh;  // (L, cap) segments to create
    BulkPlan plan{};
    uint32_t n_spans = 0;
    for (uint32_t L = 1; L <= kMaxBytes; L++) {
        plan.span_lo[L] = n_spans;
        uint64_t left = counts[L], first = 0;
        if (!left) continue;
        auto& bs = s->bucket_segs[L];
        uint32_t last_cap = 0;
        if (!bs.empty()) {
            const SegDesc& d = s->segs[bs.back()].desc;
            last_cap = d.cap;
            if (d.n < d.cap) {
                const uint32_t take = (uint32_t)std::min<uint64_t>(left, d.cap - d.n);
                pend.push_back({L, bs.back(), d.n, take});
                if (n_spans < kMaxBulkSpans) plan.spans[n_spans] = BulkSpan{bs.back(), d.n, (uint32_t)first, 0};
                n_spans++; first += take; left -= take;
            }
        }
        uint32_t next_sid = (uint32_t)(s->segs.size() + fresh.size());
        while (left) {
            const uint32_t grow = last_cap ? (uint32_t)std::min<uint64_t>((uint64_t)last_cap * 4, kMaxSegRows) : kMinSegRows;
            const uint64_t want = std::max<uint64_t>(grow, std::min<uint64_t>(left, kMaxSegRows));
            const uint32_t cap = (uint32_t)((want + kMinSegRows - 1) / kMinSegRows * kMinSegRows);
            const uint32_t take = (uint32_t)std::min<uint64_t>(left, cap);
            fresh.push_back({L, cap});
            pend.push_back({L, next_sid, 0, take});
            if (n_spans < kMaxBulkSpans) plan.spans[n_spans] = BulkSpan{next_sid, 0, (uint32_t)first, 0};
            n_spans++; next_sid++; first += take; left -= take; last_cap = cap;
        }
    }
    plan.span_lo[kMaxBytes + 1] = n_spans;
    if (n_spans > kMaxBulkSpans) return ISX_ELIMIT;  // caller splits the chunk
    for (auto& f : fresh)
        if ((rc = new_segment(s, f.first, f.second, /*mirror=*/false))) return rc;
    if ((rc = upload_segs(s))) return rc;  // plane / key pointers of the fresh segments (row counts still the old ones)
    k_scatter_bulk<<<(unsigned)((cn + 255) / 256), 256, 0, s->stream>>>(s->d_segs.as<SegDesc>(), plan, d_cursor, d_keys, d_codes, d_lens,
                                                                        uniform_len, s->key_bytes, cn);
    CU(cudaGetLastError());
    for (const Pending& pd : pend) {
        s->segs[pd.sid].desc.n = pd.row0 + pd.cnt;
        s->bucket_rows[pd.L] += pd.cnt;
        s->n_rows += pd.cnt;
    }
    s->segs_dirty = true;
    s->version++;
    s->map_stale.store(true);
    return 0;
}

int isx_add_device(isx_store_t* s, const void* d_keys, const uint8_t* d_codes, const uint8_t* d_lens, uint32_t uniform_len, size_t n) {
    if (!s) return fail(ISX_EINVAL, "store is NULL");
    if (n == 0) return 0;
    if (!d_keys || !d_codes) return fail(ISX_EINVAL, "NULL input array");
    if (!d_lens && (uniform_len < 1 || uniform_len > s->max_bytes || (s->fixed_len && uniform_len != s->fixed_len)))
        return fail(ISX_EINVAL, "isx_add_device: uniform_len %u bytes not accepted by this index", uniform_len);
    std::unique_lock<std::shared_mutex> g(s->rows_mu);
    std::lock_guard<std::mutex> gw(s->work_mu);
    int rc = set_device(s);
    if (rc) return rc;
    const uint8_t* keys = reinterpret_cast<const uint8_t*>(d_keys);
    size_t chunk = (size_t)16 << 20;
    for (size_t i0 = 0; i0 < n;) {
        const size_t cn = std::min(chunk, n - i0);
        rc = add_device_chunk(s, keys + i0 * s->key_bytes, d_codes + i0 * 32, d_lens ? d_lens + i0 : nullptr, uniform_len, cn);
        if (rc == ISX_ELIMIT && chunk > 4096) { chunk /= 2; continue; }  // too many spans for one launch: smaller chunks
        if (rc) return rc == ISX_ELIMIT ? fail(ISX_ELIMIT, "isx_add_device: cannot plan the append") : rc;
        i0 += cn;
    }
    if ((rc = upload_segs(s))) return rc;
    CU(cudaStreamSynchronize(s->stream));  // the caller may reuse its buffers when this returns
    return 0;
}

int isx_synth_rows_device(isx_store_t* s, uint64_t seed, uint64_t start, size_t n, const uint8_t* lengths, uint32_t n_lengths,
                          uint32_t key_mode, uint32_t chunks_per_asset, uint32_t dup_every, uint32_t dup_back, void* d_keys,
                          uint8_t* d_codes, uint8_t* d_lens) {
    if (!s) return fail(ISX_EINVAL, "store is NULL");
    if (n == 0) return 0;
    if (!lengths || n_lengths < 1 || n_lengths > 8 || !d_keys || !d_codes) return fail(ISX_EINVAL, "bad argument");
    if (key_mode > 1 || (key_mode == 1 && chunks_per_asset < 1)) return fail(ISX_EINVAL, "bad key_mode / chunks_per_asset");
    std::lock_guard<std::mutex> gw(s->work_mu);
    int rc = set_device(s);
    if (rc) return rc;
    SynthParams g{};
    g.seed = seed; g.start = start; g.n_lengths = n_lengths; g.key_mode = key_mode; g.cpa = chunks_per_asset;
    g.dup_every = dup_every; g.dup_back = dup_back;
    for (uint32_t i = 0; i < n_lengths; i++) {
        if (lengths[i] < 1 || lengths[i] > kMaxBytes) return fail(ISX_EINVAL, "length %u outside 1..32", lengths[i]);
        g.lengths[i] = lengths[i];
    }
    k_synth_rows<<<(unsigned)((n + 255) / 256), 256, 0, s->stream>>>(g, n, reinterpret_cast<uint8_t*>(d_keys), d_codes, d_lens);
    CU(cudaGetLastError());
    return 0;
}

int isx_contains(isx_store_t* s, const void* keys, size_t n, uint8_t* present) {
    if (!s) return fail(ISX_EINVAL, "store is NULL");
    if (n == 0) return 0;
    if (!keys || !present) return fail(ISX_EINVAL, "NULL argument");
    if (int rc0 = ensure_map(s)) return rc0;
    std::shared_lock<std::shared_mutex> g(s->rows_mu);
    for (size_t i = 0; i < n; i++) {
        uint64_t loc;
        present[i] = s->map.find(load_key(s, keys, i), &loc) ? 1 : 0;
    }
    return 0;
}

int isx_get(isx_store_t* s, const void* keys, size_t n, uint8_t* codes_out, uint8_t* lens_out) {
    if (!s) return fail(ISX_EINVAL, "store is NULL");
    if (n == 0) return 0;
    if (!keys || !codes_out || !lens_out) return fail(ISX_EINVAL, "NULL argument");
    if (int rc0 = ensure_map(s)) return rc0;
    std::shared_lock<std::shared_mutex> g(s->rows_mu);
    std::lock_guard<std::mutex> gw(s->work_mu);
    int rc = set_device(s);
    if (rc) return rc;
    std::vector<uint64_t> loc(n, ~0ull);
    size_t found = 0;
    for (size_t i = 0; i < n; i++) {
        uint64_t l;
        if (s->map.find(load_key(s, keys, i), &l)) { loc[i] = l; lens_out[i] = (uint8_t)s->segs[(uint32_t)(l >> 32)].len_bytes; found++; }
        else lens_out[i] = 0;
    }
    if (!found) { memset(codes_out, 0, n * 32); return 0; }
    if ((rc = upload_segs(s))) return rc;
    if (s->d_stage_dest.ensure(n * 8) || s->d_stage_codes.ensure(n * 32)) return ISX_ENOMEM;
    CU(cudaMemcpyAsync(s->d_stage_dest.p, loc.data(), n * 8, cudaMemcpyHostToDevice, s->stream));
    k_gather_rows<<<(unsigned)((n * 8 + 255) / 256), 256, 0, s->stream>>>(s->d_segs.as<SegDesc>(), s->d_stage_dest.as<uint64_t>(),
                                                                          s->d_stage_codes.as<uint8_t>(), n);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(codes_out, s->d_stage_codes.p, n * 32, cudaMemcpyDeviceToHost, s->stream));
    CU(cudaStreamSynchronize(s->stream));
    return 0;
}

int isx_search(isx_store_t* s, const uint8_t* queries, const uint8_t* qlens, size_t q, uint32_t k, uint32_t thr_num,
               uint32_t thr_den, void* keys_out, uint16_t* hamming_out, uint16_t* nbits_out, uint32_t* counts_out,
               uint8_t* codes_out, uint8_t* first_of_asset_out) {
    if (!s) return fail(ISX_EINVAL, "store is NULL");
    if (k < 1) return fail(ISX_EINVAL, "`count` must be >= 1");
    if (q == 0) return 0;
    if (!queries || !qlens || !keys_out || !hamming_out || !nbits_out || !counts_out) return fail(ISX_EINVAL, "NULL argument");
    std::shared_lock<std::shared_mutex> g(s->rows_mu);
    std::lock_guard<std::mutex> gw(s->work_mu);
    int rc = set_device(s);
    if (rc) return rc;
    size_t qk = q * (size_t)k;
    if (s->d_out_khi.ensure(qk * 8) || s->d_out_klo.ensure(qk * 8) || s->d_out_h.ensure(qk * 2) || s->d_out_n.ensure(qk * 2) ||
        s->d_out_cnt.ensure(q * 4) || (codes_out && s->d_out_codes.ensure(qk * 32)))
        return ISX_ENOMEM;
    SearchOut out{s->d_out_khi.as<uint64_t>(), s->d_out_klo.as<uint64_t>(), s->d_out_h.as<uint16_t>(), s->d_out_n.as<uint16_t>(),
                  s->d_out_cnt.as<uint32_t>(), codes_out ? s->d_out_codes.as<uint8_t>() : nullptr};
    // pinned result block; the small-batch path lets the device write into it directly
    const size_t out_bytes = qk * (8 + 8 + 2 + 2) + q * 4;
    if (s->h_out.ensure(out_bytes)) return ISX_ENOMEM;
    {
        uint8_t* hb = s->h_out.as<uint8_t>();
        s->small_host_khi = reinterpret_cast<uint64_t*>(hb);
        s->small_host_klo = s->small_host_khi + qk;
        s->small_host_h = reinterpret_cast<uint16_t*>(s->small_host_klo + qk);
        s->small_host_n = s->small_host_h + qk;
        s->small_host_cnt = reinterpret_cast<uint32_t*>(s->small_host_n + qk);
        s->small_host_valid = !first_of_asset_out;   // the grouping kernel reads the device copy
        s->small_host_used = false;
    }
    rc = search_core(s, queries, false, qlens, q, k, thr_num, thr_den, out);
    s->small_host_valid = false;
    if (rc) return rc;
    const bool direct = s->small_host_used;
    if (first_of_asset_out) {
        // device-side grouping of simprint matches: flag the best record of every asset per query
        uint32_t H = 2;
        while (H < 2 * k) H <<= 1;
        const size_t smem = (size_t)H * 12 + 16;
        if (smem + 2048 > (size_t)s->max_smem_optin) {
            uint32_t H_max = 2;   // largest table that fits: every count with 2 * count <= H_max is accepted
            while ((size_t)H_max * 2 * 12 + 16 + 2048 <= (size_t)s->max_smem_optin) H_max <<= 1;
            return fail(ISX_ELIMIT, "first_of_asset_out supports count <= %u", H_max / 2);
        }
        if (s->d_stage_codes.ensure(qk)) return ISX_ENOMEM;
        {
            cudaFuncAttributes fa;
            CU(cudaFuncGetAttributes(&fa, k_first_per_asset));
            CU(cudaFuncSetAttribute(k_first_per_asset, cudaFuncAttributeMaxDynamicSharedMemorySize, s->max_smem_optin - (int)fa.sharedSizeBytes));
        }
        k_first_per_asset<<<(unsigned)q, 512, smem, s->stream>>>(out.khi, out.cnt, k, H, s->d_stage_codes.as<uint8_t>());
        CU(cudaGetLastError());
        s->stats.kernel_launches++;
        CU(cudaMemcpyAsync(first_of_asset_out, s->d_stage_codes.p, qk, cudaMemcpyDeviceToHost, s->stream));
    }
    // results -> pinned staging -> caller
    uint8_t* h = s->h_out.as<uint8_t>();
    uint64_t* h_khi = reinterpret_cast<uint64_t*>(h);
    uint64_t* h_klo = h_khi + qk;
    uint16_t* h_h = reinterpret_cast<uint16_t*>(h_klo + qk);
    uint16_t* h_n = h_h + qk;
    uint32_t* h_cnt = reinterpret_cast<uint32_t*>(h_n + qk);
    if (!direct) {
        CU(cudaMemcpyAsync(h_khi, out.khi, qk * 8, cudaMemcpyDeviceToHost, s->stream));
        if (s->key_bytes == 16) CU(cudaMemcpyAsync(h_klo, out.klo, qk * 8, cudaMemcpyDeviceToHost, s->stream));
        CU(cudaMemcpyAsync(h_h, out.h, qk * 2, cudaMemcpyDeviceToHost, s->stream));
        CU(cudaMemcpyAsync(h_n, out.n, qk * 2, cudaMemcpyDeviceToHost, s->stream));
        CU(cudaMemcpyAsync(h_cnt, out.cnt, q * 4, cudaMemcpyDeviceToHost, s->stream));
    }
    if (codes_out) CU(cudaMemcpyAsync(codes_out, out.codes, qk * 32, cudaMemcpyDeviceToHost, s->stream));
    CU(cudaStreamSynchronize(s->stream));
    memcpy(hamming_out, h_h, qk * 2);
    memcpy(nbits_out, h_n, qk * 2);
    memcpy(counts_out, h_cnt, q * 4);
    if (s->key_bytes == 8) memcpy(keys_out, h_khi, qk * 8);
    else for (size_t i = 0; i < qk; i++) store_key(s, keys_out, i, h_khi[i], h_klo[i]);
    return 0;
}

int isx_search_device(isx_store_t* s, const uint8_t* queries, int queries_on_device, const uint8_t* qlens, size_t q,
                      uint32_t k, uint32_t thr_num, uint32_t thr_den, uint64_t* d_keys_hi, uint64_t* d_keys_lo,
                      uint16_t* d_hamming, uint16_t* d_nbits, uint32_t* d_counts, int sync) {
    if (!s) return fail(ISX_EINVAL, "store is NULL");
    if (k < 1) return fail(ISX_EINVAL, "`count` must be >= 1");
    if (q == 0) return 0;
    if (!queries || !qlens || !d_keys_hi || !d_keys_lo || !d_hamming || !d_nbits || !d_counts) return fail(ISX_EINVAL, "NULL argument");
    std::shared_lock<std::shared_mutex> g(s->rows_mu);
    std::lock_guard<std::mutex> gw(s->work_mu);
    int rc = set_device(s);
    if (rc) return rc;
    SearchOut out{d_keys_hi, d_keys_lo, d_hamming, d_nbits, d_counts, nullptr};
    if ((rc = search_core(s, queries, queries_on_device != 0, qlens, q, k, thr_num, thr_den, out))) return rc;
    if (sync) CU(cudaStreamSynchronize(s->stream));
    return 0;
}

int isx_merge_device(isx_store_t* s, uint32_t n_shards, size_t q, uint32_t k, size_t shard_stride_bytes, const uint64_t* d_keys_hi,
                     const uint64_t* d_keys_lo, const uint16_t* d_hamming, const uint16_t* d_nbits,
                     const uint32_t* d_counts, uint64_t* d_out_keys_hi, uint64_t* d_out_keys_lo,
                     uint16_t* d_out_hamming, uint16_t* d_out_nbits, uint32_t* d_out_counts, int sync) {
    if (!s) return fail(ISX_EINVAL, "store is NULL");
    if (q == 0) return 0;
    if (n_shards < 1 || k < 1) return fail(ISX_EINVAL, "n_shards and k must be >= 1");
    std::lock_guard<std::mutex> gw(s->work_mu);
    int rc = set_device(s);
    if (rc) return rc;
    k_merge<<<(unsigned)q, 256, 0, s->stream>>>(n_shards, (uint32_t)q, k, shard_stride_bytes, d_keys_hi, d_keys_lo, d_hamming, d_nbits, d_counts,
                                               d_out_keys_hi, d_out_keys_lo, d_out_hamming, d_out_nbits, d_out_counts);
    CU(cudaGetLastError());
    s->stats.kernel_launches++;
    if (sync) CU(cudaStreamSynchronize(s->stream));
    return 0;
}

int isx_match_all(isx_store_t* s, const uint8_t* query, uint32_t qlen, uint32_t thr_num, uint32_t thr_den, size_t max_out,
                  void* keys_out, uint16_t* hamming_out, uint16_t* nbits_out, uint64_t* total_out) {
    if (!s) return fail(ISX_EINVAL, "store is NULL");
    if (!query || !total_out || (max_out && (!keys_out || !hamming_out || !nbits_out))) return fail(ISX_EINVAL, "NULL argument");
    if (thr_den == 0) return fail(ISX_EINVAL, "match_all needs a threshold (thr_den != 0)");
    if (qlen < 1 || qlen > s->max_bytes || (s->fixed_len && qlen != s->fixed_len)) return fail(ISX_EINVAL, "query length %u bytes not accepted by this index", qlen);
    if (max_out > 0xfffffff0u) return fail(ISX_ELIMIT, "max_out too large");
    std::shared_lock<std::shared_mutex> g(s->rows_mu);
    std::lock_guard<std::mutex> gw(s->work_mu);
    int rc = set_device(s);
    if (rc) return rc;
    isx_stats_t& st = s->stats;
    st = isx_stats_t{};
    s->join_valid = false;
    *total_out = 0;
    if ((rc = upload_segs(s)) || (rc = upload_blocks(s))) return rc;
    const uint32_t n_blocks_total = (uint32_t)s->h_blocks.size();
    if (n_blocks_total == 0) return 0;
    uint32_t cmask = 1u << (qlen - 1);
    for (uint32_t b = 1; b <= kMaxBytes; b++) if (s->bucket_rows[b]) cmask |= 1u << (std::min(qlen, b) - 1);
    if ((rc = build_tables(s, cmask))) return rc;
    const RankTables& tb = s->tables;
    const uint32_t R = tb.R;
    uint32_t tau = 0;
    while (tau + 1 < R && (uint64_t)tb.frac_h[tau + 1] * thr_den <= (uint64_t)thr_num * tb.frac_n[tau + 1]) tau++;
    const size_t C = std::max<size_t>(max_out, 1);
    if (s->d_queries.ensure(32) || s->d_tau.ensure(4) || s->d_hist.ensure((size_t)R * 4) || s->d_cnt.ensure(4) || s->d_ovf.ensure(4) ||
        s->d_fb_cand.ensure(C * 8) || s->h_flags.ensure(16) || s->d_out_khi.ensure(C * 8) || s->d_out_klo.ensure(C * 8) ||
        s->d_out_h.ensure(C * 2) || s->d_out_n.ensure(C * 2) || s->h_queries.ensure(32))
        return ISX_ENOMEM;
    uint8_t* hq = s->h_queries.as<uint8_t>();
    memset(hq, 0, 32);
    memcpy(hq, query, qlen);
    CU(cudaMemcpyAsync(s->d_queries.p, hq, 32, cudaMemcpyHostToDevice, s->stream));
    ScanParams p{};
    p.segs = s->d_segs.as<SegDesc>();
    p.blocks = s->d_blocks.as<uint2>();
    p.queries = s->d_queries.as<uint32_t>();
    p.T = 1;
    p.qlen_bytes = qlen;
    p.tau = s->d_tau.as<uint32_t>();
    p.hist = s->d_hist.as<uint32_t>();
    p.cand_cnt = s->d_cnt.as<uint32_t>();
    p.cand = s->d_fb_cand.as<uint64_t>();
    p.overflow = s->d_ovf.as<uint32_t>();
    p.C = (uint32_t)C; p.R = R; p.k = 1;
    p.rank_tab = tb.d_rank.as<uint16_t>();
    p.hmax_tab = tb.d_hmax.as<uint16_t>();
    p.update_tau = 0;  // fixed threshold: every row within it is emitted
    k_init_queries<<<std::max<uint32_t>(1, (R + 255) / 256), 256, 0, s->stream>>>(p.tau, p.hist, nullptr, p.cand_cnt, p.overflow, 1, R, tau);
    CU(cudaGetLastError());
    st.kernel_launches++;
    if ((rc = scan_range(s, p, 0, n_blocks_total, 16))) return rc;
    uint32_t* hf = s->h_flags.as<uint32_t>();
    CU(cudaMemcpyAsync(hf, p.cand_cnt, 4, cudaMemcpyDeviceToHost, s->stream));
    CU(cudaStreamSynchronize(s->stream));
    const uint32_t total = hf[0];
    *total_out = total;
    st.candidates = total;
    const uint32_t n = (uint32_t)std::min<size_t>(total, max_out);
    if (n == 0) return 0;
    k_gather_cands<<<(n + 255) / 256, 256, 0, s->stream>>>(p.segs, p.cand, n, qlen, s->d_out_khi.as<uint64_t>(), s->d_out_klo.as<uint64_t>(),
                                                          s->d_out_h.as<uint16_t>(), s->d_out_n.as<uint16_t>());
    CU(cudaGetLastError());
    st.kernel_launches++;
    std::vector<uint64_t> khi(n), klo(n);
    CU(cudaMemcpyAsync(khi.data(), s->d_out_khi.p, (size_t)n * 8, cudaMemcpyDeviceToHost, s->stream));
    if (s->key_bytes == 16) CU(cudaMemcpyAsync(klo.data(), s->d_out_klo.p, (size_t)n * 8, cudaMemcpyDeviceToHost, s->stream));
    CU(cudaMemcpyAsync(hamming_out, s->d_out_h.p, (size_t)n * 2, cudaMemcpyDeviceToHost, s->stream));
    CU(cudaMemcpyAsync(nbits_out, s->d_out_n.p, (size_t)n * 2, cudaMemcpyDeviceToHost, s->stream));
    CU(cudaStreamSynchronize(s->stream));
    if (s->key_bytes == 8) memcpy(keys_out, khi.data(), (size_t)n * 8);
    else for (uint32_t i = 0; i < n; i++) store_key(s, keys_out, i, khi[i], klo[i]);
    return 0;
}

int isx_self_join(isx_store_t* s, uint32_t thr_num, uint32_t thr_den, uint64_t* total_out) {
    if (!s || !total_out) return fail(ISX_EINVAL, "NULL argument");
    *total_out = 0;
    if (thr_den == 0) return fail(ISX_EINVAL, "isx_self_join needs a threshold (thr_den != 0)");
    std::shared_lock<std::shared_mutex> g(s->rows_mu);
    std::lock_guard<std::mutex> gw(s->work_mu);
    int rc = set_device(s);
    if (rc) return rc;
    if (s->profiling) CU(cudaEventRecord(s->ev[0], s->stream));
    if ((rc = self_join_core(s, thr_num, thr_den, total_out))) return rc;
    if (s->profiling) {
        CU(cudaEventRecord(s->ev[3], s->stream));
        CU(cudaStreamSynchronize(s->stream));
        float t = 0;
        CU(cudaEventElapsedTime(&t, s->ev[0], s->ev[3]));
        s->stats.total_ms = t;
    }
    return 0;
}

int isx_join_fetch(isx_store_t* s, uint64_t first, size_t n, void* keys_a_out, void* keys_b_out, uint16_t* hamming_out, uint16_t* nbits_out) {
    if (!s) return fail(ISX_EINVAL, "store is NULL");
    if (n && (!keys_a_out || !keys_b_out || !hamming_out || !nbits_out)) return fail(ISX_EINVAL, "NULL argument");
    std::shared_lock<std::shared_mutex> g(s->rows_mu);
    std::lock_guard<std::mutex> gw(s->work_mu);
    if (!s->join_valid || s->join_version != s->version)
        return fail(ISX_EINVAL, "isx_join_fetch: no self-join result (a search, match, mutation or isx_release_scratch since the last "
                                "isx_self_join ended it; run the join again)");
    if (first > s->join_total || n > s->join_total - first)
        return fail(ISX_EINVAL, "isx_join_fetch: records [%llu, %llu) are outside the %llu pairs of the join", (unsigned long long)first,
                    (unsigned long long)(first + n), (unsigned long long)s->join_total);
    if (n == 0) return 0;
    int rc = set_device(s);
    if (rc) return rc;
    const bool wide = s->key_bytes == 16;
    const size_t kb = wide ? sizeof(JoinKey16) : sizeof(JoinKey8);
    if (s->h_out.ensure(n * (kb + 4))) return ISX_ENOMEM;
    uint8_t* hk = s->h_out.as<uint8_t>();
    uint32_t* hv = reinterpret_cast<uint32_t*>(hk + n * kb);
    CU(cudaMemcpyAsync(hk, s->d_join_keys[s->join_cur].as<uint8_t>() + first * kb, n * kb, cudaMemcpyDeviceToHost, s->stream));
    CU(cudaMemcpyAsync(hv, s->d_join_vals[s->join_cur].as<uint32_t>() + first, n * 4, cudaMemcpyDeviceToHost, s->stream));
    CU(cudaStreamSynchronize(s->stream));
    if (wide) {
        const JoinKey16* k = reinterpret_cast<const JoinKey16*>(hk);
        for (size_t i = 0; i < n; i++) {
            store_key(s, keys_a_out, i, k[i].a_hi, k[i].a_lo);
            store_key(s, keys_b_out, i, k[i].b_hi, k[i].b_lo);
        }
    } else {
        const JoinKey8* k = reinterpret_cast<const JoinKey8*>(hk);
        uint64_t* a = reinterpret_cast<uint64_t*>(keys_a_out);
        uint64_t* b = reinterpret_cast<uint64_t*>(keys_b_out);
        for (size_t i = 0; i < n; i++) { a[i] = k[i].a; b[i] = k[i].b; }
    }
    for (size_t i = 0; i < n; i++) { hamming_out[i] = (uint16_t)(hv[i] & 0xffffu); nbits_out[i] = (uint16_t)(hv[i] >> 16); }
    return 0;
}

int isx_score_segments(isx_store_t* s, const uint32_t* seg, size_t n_assets, const uint32_t* rec_qi, const double* rec_sim,
                       const double* rec_idf, size_t n_rec, const double* q_idf, uint32_t n_queries, double* score_out) {
    if (!s) return fail(ISX_EINVAL, "store is NULL");
    if (n_assets == 0) return 0;
    if (!seg || !rec_qi || !rec_sim || !rec_idf || !q_idf || !score_out) return fail(ISX_EINVAL, "NULL argument");
    if (n_assets > 0xfffffff0u || n_rec > 0xfffffff0u) return fail(ISX_ELIMIT, "too many records");
    std::lock_guard<std::mutex> gw(s->work_mu);
    int rc = set_device(s);
    if (rc) return rc;
    // one staging block: seg | qi | sim | idf | q_idf | score
    const size_t b_seg = (n_assets + 1) * 4, b_qi = n_rec * 4, b_d = n_rec * 8, b_q = (size_t)n_queries * 8, b_out = n_assets * 8;
    auto al = [](size_t x) { return (x + 15) / 16 * 16; };
    const size_t o_qi = al(b_seg), o_sim = o_qi + al(b_qi), o_idf = o_sim + al(b_d), o_q = o_idf + al(b_d), o_out = o_q + al(b_q);
    if (s->d_stage_codes.ensure(o_out + b_out)) return ISX_ENOMEM;
    uint8_t* d = s->d_stage_codes.as<uint8_t>();
    CU(cudaMemcpyAsync(d, seg, b_seg, cudaMemcpyHostToDevice, s->stream));
    CU(cudaMemcpyAsync(d + o_qi, rec_qi, b_qi, cudaMemcpyHostToDevice, s->stream));
    CU(cudaMemcpyAsync(d + o_sim, rec_sim, b_d, cudaMemcpyHostToDevice, s->stream));
    CU(cudaMemcpyAsync(d + o_idf, rec_idf, b_d, cudaMemcpyHostToDevice, s->stream));
    CU(cudaMemcpyAsync(d + o_q, q_idf, b_q, cudaMemcpyHostToDevice, s->stream));
    k_score_segments<<<(unsigned)((n_assets + 127) / 128), 128, 0, s->stream>>>(
        reinterpret_cast<const uint32_t*>(d), reinterpret_cast<const uint32_t*>(d + o_qi), reinterpret_cast<const double*>(d + o_sim),
        reinterpret_cast<const double*>(d + o_idf), reinterpret_cast<const double*>(d + o_q), (uint32_t)n_assets, n_queries,
        reinterpret_cast<double*>(d + o_out));
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(score_out, d + o_out, b_out, cudaMemcpyDeviceToHost, s->stream));
    CU(cudaStreamSynchronize(s->stream));
    return 0;
}

// ---- cross-rank threshold sharing over NVLink peer memory (CUDA IPC) -------------------------------------
int isx_share_init(isx_store_t* s, uint32_t world, uint32_t rank, uint32_t max_queries, void* handle_out) {
    if (!s || !handle_out) return fail(ISX_EINVAL, "NULL argument");
    if (world < 2 || world > (uint32_t)kMaxRanks || rank >= world) return fail(ISX_EINVAL, "world must be 2..%d and rank < world", kMaxRanks);
    if (max_queries == 0) return fail(ISX_EINVAL, "max_queries must be > 0");
    std::lock_guard<std::mutex> gw(s->work_mu);
    int rc = set_device(s);
    if (rc) return rc;
    if (s->share_local) return fail(ISX_EINVAL, "sharing is already initialised for this store");
    const size_t slots = (max_queries + world - 1) / world;
    s->share_bytes = slots * isx_store::kShareRcap * sizeof(uint32_t);
    CU(cudaMalloc(&s->share_local, s->share_bytes));
    CU(cudaMemset(s->share_local, 0, s->share_bytes));
    cudaIpcMemHandle_t h;
    CU(cudaIpcGetMemHandle(&h, s->share_local));
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    memcpy(handle_out, &h, sizeof h);
    s->share_world = world;
    s->share_rank = rank;
    s->share_maxq = max_queries;
    s->share_ptrs[rank] = s->share_local;
    return 0;
}

int isx_share_attach(isx_store_t* s, uint32_t peer_rank, const void* handle) {
    if (!s || !handle) return fail(ISX_EINVAL, "NULL argument");
    std::lock_guard<std::mutex> gw(s->work_mu);
    if (!s->share_local) return fail(ISX_EINVAL, "call isx_share_init first");
    if (peer_rank >= s->share_world || peer_rank == s->share_rank) return fail(ISX_EINVAL, "bad peer rank %u", peer_rank);
    int rc = set_device(s);
    if (rc) return rc;
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof h);
    void* p = nullptr;
    CU(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    s->share_ptrs[peer_rank] = reinterpret_cast<uint32_t*>(p);
    return 0;
}

int isx_share_reset(isx_store_t* s) {
    if (!s) return fail(ISX_EINVAL, "store is NULL");
    std::lock_guard<std::mutex> gw(s->work_mu);
    if (!s->share_local) return 0;
    int rc = set_device(s);
    if (rc) return rc;
    for (uint32_t r = 0; r < s->share_world; r++)
        if (!s->share_ptrs[r]) return fail(ISX_EINVAL, "peer %u is not attached", r);
    CU(cudaMemsetAsync(s->share_local, 0, s->share_bytes, s->stream));
    s->share_armed = true;
    return 0;
}

int isx_share_set_lengths(isx_store_t* s, uint32_t global_length_mask) {
    if (!s) return fail(ISX_EINVAL, "store is NULL");
    std::lock_guard<std::mutex> gw(s->work_mu);
    s->share_len_mask = global_length_mask;
    return 0;
}

// ---- host-only self tests (no device needed): used by the CPU test-suite ------------------------------------
int isx_selftest_rank_table(uint32_t class_mask, uint16_t* rank_out, uint16_t* hmax_out, uint32_t hmax_stride, uint32_t* R_out) {
    if (!rank_out || !R_out) return fail(ISX_EINVAL, "NULL argument");
    RankTables t;
    int rc = compute_tables(class_mask, t);
    if (rc) return rc;
    memcpy(rank_out, t.rank.data(), t.rank.size() * 2);
    *R_out = t.R;
    if (hmax_out) {
        if (hmax_stride < t.R) return fail(ISX_EINVAL, "hmax_stride %u < R %u", hmax_stride, t.R);
        for (uint32_t m = 0; m <= kMaxBytes; m++) memcpy(hmax_out + (size_t)m * hmax_stride, t.hmax.data() + (size_t)m * t.R, t.R * 2);
    }
    return 0;
}

}  // extern "C" (templates cannot have C linkage)

// Host build of the device arithmetic helpers (kernels.cuh: pair_distance, LowerBound::eval) against a naive popcount.
template <int WE>
static int selftest_distance_we(uint64_t n, uint64_t& x) {
    auto next = [&]() { x ^= x << 13; x ^= x >> 7; x ^= x << 17; return x; };
    static const uint32_t masks[4] = {0xffffffffu, 0x000000ffu, 0x0000ffffu, 0x00ffffffu};
    for (uint64_t it = 0; it < n; it++) {
        uint4 a[WE];
        uint32_t qv[WE];
        const uint32_t sparse = (uint32_t)(it % 3);  // dense random words, near-identical rows, identical rows
        for (int w = 0; w < WE; w++) {
            qv[w] = (uint32_t)next();
            uint32_t r[4];
            for (int k = 0; k < 4; k++) {
                uint64_t v = next();
                r[k] = sparse == 0 ? (uint32_t)v : sparse == 1 ? (qv[w] ^ (uint32_t)(v & (v >> 16) & (v >> 32))) : qv[w];
            }
            a[w] = make_uint4(r[0], r[1], r[2], r[3]);
        }
        const uint32_t mask_last = masks[it & 3];
        for (int r = 0; r < 4; r++) {
            uint32_t xw[WE], exact = 0, fold2 = 0, fold3 = 0;
            for (int w = 0; w < WE; w++) {
                xw[w] = (comp(a[w], r) ^ qv[w]) & (w == WE - 1 ? mask_last : 0xffffffffu);
                exact += (uint32_t)__builtin_popcount(xw[w]);
            }
            for (int w = 0; w < WE; w += 2) fold2 += (uint32_t)__builtin_popcount(xw[w] | (w + 1 < WE ? xw[w + 1] : 0u));
            for (int w = 0; w < WE; w += 3) fold3 += (uint32_t)__builtin_popcount(xw[w] | (w + 1 < WE ? xw[w + 1] : 0u) | (w + 2 < WE ? xw[w + 2] : 0u));
            if (pair_distance<WE>(xw) != exact) return fail(ISX_EINVAL, "pair_distance<%d> differs from the naive popcount", WE);
            const uint32_t b2 = LowerBound<WE>::template eval<2>(a, qv, r, mask_last), b3 = LowerBound<WE>::template eval<3>(a, qv, r, mask_last);
            if (b2 != fold2 || b3 != fold3) return fail(ISX_EINVAL, "LowerBound<%d>::eval differs from the naive OR fold", WE);
            if (b2 > exact || b3 > exact) return fail(ISX_EINVAL, "LowerBound<%d> is not a lower bound", WE);
        }
    }
    return 0;
}

// Host build of the tensor-core scan's encoding (tc.cuh): rows as 0/1 bytes, queries as +-1 bytes zeroed past 8m bits, the
// byte dot product acc over the K-major layout, h = acc + popc(q[:m]) against a naive popcount, for every length m 1..32.
static int selftest_tc_encoding(uint64_t n, uint64_t& x) {
    auto next = [&]() { x ^= x << 13; x ^= x >> 7; x ^= x << 17; return x; };
    for (uint64_t it = 0; it < n; it++) {
        for (uint32_t m = 1; m <= kMaxBytes; m++) {
            const uint32_t WE = (m + 3) / 4, KB = 32 * WE;
            uint32_t a[8], q[8];
            const uint32_t sparse = (uint32_t)(it % 3);   // random rows, near-identical rows, identical rows
            for (uint32_t w = 0; w < WE; w++) {
                q[w] = (uint32_t)next();
                const uint64_t v = next();
                a[w] = sparse == 0 ? (uint32_t)v : sparse == 1 ? (q[w] ^ (uint32_t)(v & (v >> 16) & (v >> 32))) : q[w];
            }
            // row r = 1 and query row 9 of a 16-row tile: the second core matrix row group exercises the layout
            std::vector<int8_t> A(16 * KB, 0), B(16 * KB, 0);
            uint32_t popc_q = 0, exact = 0;
            for (uint32_t w = 0; w < WE; w++) {
                const uint32_t nb = tc_word_bits(m, w), mk = nb >= 32 ? 0xffffffffu : (1u << nb) - 1u;
                popc_q += popc32(q[w] & mk);
                exact += popc32((a[w] ^ q[w]) & mk);
                for (int j = 0; j < 8; j++) {
                    const uint32_t ra = tc_row_bytes(a[w], j), qb = tc_query_bytes(q[w], j, nb);
                    memcpy(&A[tc_off(1, 32 * w + 4 * j, KB)], &ra, 4);
                    memcpy(&B[tc_off(9, 32 * w + 4 * j, KB)], &qb, 4);
                }
            }
            int32_t acc = 0;
            for (uint32_t kb = 0; kb < KB; kb++) acc += (int32_t)A[tc_off(1, kb, KB)] * (int32_t)B[tc_off(9, kb, KB)];
            if (tc_hamming(acc, popc_q) != exact) return fail(ISX_EINVAL, "tensor-core encoding differs from the naive popcount at m = %u", m);
        }
    }
    return 0;
}

extern "C" {

int isx_selftest_distance(uint64_t n, uint64_t seed) {
    uint64_t x = seed * 0x9E3779B97F4A7C15ull + 1;
    int rc = 0;
    if ((rc = selftest_tc_encoding(n, x))) return rc;
    if ((rc = selftest_distance_we<1>(n, x)) || (rc = selftest_distance_we<2>(n, x)) || (rc = selftest_distance_we<3>(n, x)) ||
        (rc = selftest_distance_we<4>(n, x)) || (rc = selftest_distance_we<5>(n, x)) || (rc = selftest_distance_we<6>(n, x)) ||
        (rc = selftest_distance_we<7>(n, x)) || (rc = selftest_distance_we<8>(n, x)))
        return rc;
    return 0;
}

int isx_selftest_keymap(uint64_t n_ops, uint64_t seed, uint32_t key_space) {
    // random insert / update / erase / find against a std::vector reference over a small key space (many collisions
    // of home slots and long probe chains: exercises the backward-shift deletion)
    KeyMap map;
    std::vector<uint64_t> ref(key_space, ~0ull);
    uint64_t x = seed * 0x9E3779B97F4A7C15ull + 1;
    auto next = [&]() { x ^= x << 13; x ^= x >> 7; x ^= x << 17; return x; };
    size_t live = 0;
    for (uint64_t i = 0; i < n_ops; i++) {
        uint64_t r = next();
        uint32_t kidx = (uint32_t)(r % key_space);
        Key128 key{mix64(kidx) | 1, mix64(kidx * 31ull + 5)};  // one fixed 128-bit key per kidx
        uint32_t op = (uint32_t)((r >> 32) % 4);
        uint64_t loc;
        bool present = ref[kidx] != ~0ull;
        if (op == 0) {
            bool ok = map.insert(key, r >> 8 & 0xffffffffffull);
            if (ok == present) return fail(ISX_EINVAL, "keymap: insert result mismatch at op %llu", (unsigned long long)i);
            if (ok) { ref[kidx] = r >> 8 & 0xffffffffffull; live++; }
        } else if (op == 1) {
            bool ok = map.erase(key);
            if (ok != present) return fail(ISX_EINVAL, "keymap: erase result mismatch at op %llu", (unsigned long long)i);
            if (ok) { ref[kidx] = ~0ull; live--; }
        } else if (op == 2) {
            bool ok = map.update(key, i);
            if (ok != present) return fail(ISX_EINVAL, "keymap: update result mismatch at op %llu", (unsigned long long)i);
            if (ok) ref[kidx] = i;
        } else {
            bool ok = map.find(key, &loc);
            if (ok != present || (ok && loc != ref[kidx])) return fail(ISX_EINVAL, "keymap: find mismatch at op %llu", (unsigned long long)i);
        }
        if (map.size() != live) return fail(ISX_EINVAL, "keymap: size mismatch at op %llu", (unsigned long long)i);
    }
    for (uint32_t kidx = 0; kidx < key_space; kidx++) {  // final sweep: every key answers like the reference
        Key128 key{mix64(kidx) | 1, mix64(kidx * 31ull + 5)};
        uint64_t loc;
        bool ok = map.find(key, &loc);
        if (ok != (ref[kidx] != ~0ull) || (ok && loc != ref[kidx])) return fail(ISX_EINVAL, "keymap: final sweep mismatch at key %u", kidx);
    }
    return 0;
}

// ---- snapshot ----------------------------------------------------------------------------------
// magic | key_bytes, max_bytes, fixed_len, 0 | total rows | per bucket: [u32 L][u64 rows] then chunks
// [u32 n][keys hi n*8][keys lo n*8 if 16-byte keys][codes n*L] ... [u32 0] | [u32 0] end marker
static const char kMagic[8] = {'I', 'S', 'X', 'B', '2', '0', '0', '1'};

int isx_save(isx_store_t* s, const char* path) {
    if (!s || !path) return fail(ISX_EINVAL, "NULL argument");
    if (int rc0 = ensure_map(s)) return rc0;
    std::shared_lock<std::shared_mutex> g(s->rows_mu);
    std::lock_guard<std::mutex> gw(s->work_mu);
    int rc = set_device(s);
    if (rc) return rc;
    std::string tmp = std::string(path) + ".tmp";
    FILE* f = fopen(tmp.c_str(), "wb");
    if (!f) return fail(ISX_EIO, "cannot open %s for writing", tmp.c_str());
    bool ok = true;
    auto W = [&](const void* p, size_t n) { if (ok && n && fwrite(p, 1, n, f) != n) ok = false; };
    uint32_t hdr[4] = {s->key_bytes, s->max_bytes, s->fixed_len, 0};
    uint64_t total = s->n_rows;
    W(kMagic, 8); W(hdr, sizeof hdr); W(&total, 8);
    std::vector<uint32_t> plane;
    std::vector<uint8_t> rows;
    const uint32_t zero = 0;
    for (uint32_t L = 1; L <= kMaxBytes && ok; L++) {
        uint64_t n = s->bucket_rows[L];
        if (!n) continue;
        uint32_t L32 = L;
        W(&L32, 4); W(&n, 8);
        uint32_t words = (L + 3) / 4;
        for (uint32_t sid : s->bucket_segs[L]) {
            Segment& sg = s->segs[sid];
            uint32_t sn = sg.desc.n;
            if (!sn) continue;
            W(&sn, 4);
            W(sg.h_khi.data(), (size_t)sn * 8);
            if (s->key_bytes == 16) W(sg.h_klo.data(), (size_t)sn * 8);
            plane.resize((size_t)words * sn);
            for (uint32_t w = 0; w < words; w++) {
                cudaError_t e = cudaMemcpyAsync(plane.data() + (size_t)w * sn, sg.desc.planes + (size_t)w * sg.desc.cap, (size_t)sn * 4,
                                                cudaMemcpyDeviceToHost, s->stream);
                if (e != cudaSuccess) { fclose(f); remove(tmp.c_str()); return fail(ISX_ECUDA, "snapshot copy failed: %s", cudaGetErrorString(e)); }
            }
            if (cudaStreamSynchronize(s->stream) != cudaSuccess) { fclose(f); remove(tmp.c_str()); return fail(ISX_ECUDA, "snapshot copy failed"); }
            rows.resize((size_t)sn * L);
            for (uint32_t r = 0; r < sn; r++) {
                uint8_t tmpb[32];
                for (uint32_t w = 0; w < words; w++) memcpy(tmpb + 4 * w, &plane[(size_t)w * sn + r], 4);
                memcpy(&rows[(size_t)r * L], tmpb, L);
            }
            W(rows.data(), rows.size());
        }
        W(&zero, 4);
    }
    W(&zero, 4);
    if (fclose(f) != 0) ok = false;
    if (!ok) { remove(tmp.c_str()); return fail(ISX_EIO, "write to %s failed", tmp.c_str()); }
    if (rename(tmp.c_str(), path) != 0) { remove(tmp.c_str()); return fail(ISX_EIO, "rename to %s failed", path); }
    return 0;
}

int isx_load(isx_store_t* s, const char* path) {
    if (!s || !path) return fail(ISX_EINVAL, "NULL argument");
    FILE* f = fopen(path, "rb");
    if (!f) return fail(ISX_EIO, "cannot open %s", path);
    char magic[8];
    uint32_t hdr[4];
    uint64_t total;
    if (fread(magic, 1, 8, f) != 8 || memcmp(magic, kMagic, 8) != 0 || fread(hdr, 1, sizeof hdr, f) != sizeof hdr || fread(&total, 1, 8, f) != 8) {
        fclose(f);
        return fail(ISX_EIO, "%s is not an isx snapshot", path);
    }
    if (hdr[0] != s->key_bytes || hdr[1] > s->max_bytes || hdr[2] != s->fixed_len) {
        fclose(f);
        return fail(ISX_EINVAL, "snapshot %s was written for key_bytes=%u max_bytes=%u fixed_len=%u", path, hdr[0], hdr[1], hdr[2]);
    }
    int rc = isx_clear(s);
    if (rc) { fclose(f); return rc; }
    std::vector<uint64_t> khi, klo;
    std::vector<uint8_t> keys, rows, codes, lens;
    auto bad = [&](const char* why) { fclose(f); isx_clear(s); return fail(ISX_EIO, "%s snapshot %s", why, path); };
    for (;;) {
        uint32_t L;
        uint64_t n;
        if (fread(&L, 1, 4, f) != 4) return bad("truncated");
        if (L == 0) break;
        if (L > kMaxBytes || fread(&n, 1, 8, f) != 8) return bad("corrupt");
        for (;;) {
            uint32_t sn;
            if (fread(&sn, 1, 4, f) != 4) return bad("truncated");
            if (sn == 0) break;
            if (sn > kMaxSegRows) return bad("corrupt");
            khi.resize(sn);
            if (fread(khi.data(), 8, sn, f) != sn) return bad("truncated");
            if (s->key_bytes == 16) { klo.resize(sn); if (fread(klo.data(), 8, sn, f) != sn) return bad("truncated"); }
            rows.resize((size_t)sn * L);
            if (fread(rows.data(), 1, rows.size(), f) != rows.size()) return bad("truncated");
            codes.assign((size_t)sn * 32, 0);
            lens.assign(sn, (uint8_t)L);
            for (uint32_t r = 0; r < sn; r++) memcpy(&codes[(size_t)r * 32], &rows[(size_t)r * L], L);
            const void* kp = khi.data();
            if (s->key_bytes == 16) {
                keys.resize((size_t)sn * 16);
                for (uint32_t r = 0; r < sn; r++) store_key(s, keys.data(), r, khi[r], klo[r]);
                kp = keys.data();
            }
            if ((rc = isx_add(s, kp, codes.data(), lens.data(), sn, nullptr))) { fclose(f); return rc; }
        }
    }
    fclose(f);
    uint64_t have = 0;
    isx_size(s, &have);
    if (have != total) return fail(ISX_EIO, "snapshot %s: expected %llu rows, loaded %llu", path, (unsigned long long)total, (unsigned long long)have);
    return 0;
}

}  // extern "C"
