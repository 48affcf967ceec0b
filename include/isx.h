/*
 * isx.h - C ABI of libisx_b200.so: an HBM-resident, exact NPHD / Hamming top-k store for ISCC codes
 * on NVIDIA B200 (sm_100a). One store lives on ONE device of ONE process (one process per GPU;
 * multi-GPU = row shards + top-k merge, see isx_search_device / isx_merge_device).
 *
 * This is the drop-in boundary for the two vector-index classes iscc-search reaches through the
 * un-vendored `iscc-usearch` package (citations relative to /root/reference/):
 *
 *   ShardedNphdIndex  (variable-length codes, uint64 keys, NPHD metric)
 *       ctor            iscc_search/indexes/usearch/index.py:1617-1625, 1732-1740
 *       .search         iscc_search/indexes/usearch/index.py:2037
 *       .add / .remove  iscc_search/indexes/usearch/index.py:440, 436
 *       key in / .get   iscc_search/indexes/usearch/index.py:560, tests/test_indexes_usearch_persistence.py:704-706
 *       .size / .save   iscc_search/indexes/usearch/index.py:444, 474-475
 *   ShardedIndex128   (fixed ndim, 128-bit composite keys, Hamming metric)
 *       ctor            iscc_search/indexes/simprint/usearch_core.py:73-83
 *       .search         iscc_search/indexes/simprint/usearch_core.py:165
 *       .add/.remove    iscc_search/indexes/simprint/usearch_core.py:108, 119
 *       in / .get / len iscc_search/indexes/simprint/usearch_core.py:135, 221, 157
 *   and the LMDB equality join it replaces (h == 0 mode, ascending 16-byte key order, cap):
 *       search_simprints_exact  iscc_search/indexes/simprint/lmdb_ops.py:169-250
 *
 * Conventions
 *   - every function returns 0 on success or a negative ISX_E* code; isx_last_error() returns a
 *     thread-local message for the last failure on the calling thread.
 *   - the caller owns every buffer; pointers are plain host pointers unless the name says device.
 *   - codes cross the ABI as rows of ISX_MAX_BYTES (32) bytes, zero padded, plus one length byte
 *     per row (1..32 bytes; ISCC bodies are 8/16/24/32).
 *   - keys: key_bytes == 8  -> native-endian uint64 array;
 *           key_bytes == 16 -> rows of 16 raw bytes ordered bytewise (big-endian, the order LMDB
 *                              dupsort gives chunk pointers, lmdb_ops.py:30-49).
 *   - result order per query: (hamming/nbits ascending as an exact rational, key ascending).
 *     nbits = 8 * min(query_len, stored_len): NPHD prefix normalisation
 *     (docs/explanation/similarity-search.md:24-32). The float the reference sees is rebuilt by
 *     the host wrapper as float32(h)/float32(nbits) (NPHD) or float32(h) (Hamming).
 *   - thread safety: searches take a shared lock on the rows (and serialise on the store's
 *     scratch space); add/remove/clear/load take it exclusively.
 *   - there is NO CPU fallback: without a CUDA device every call fails with ISX_ECUDA.
 */
#ifndef ISX_H
#define ISX_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ISX_MAX_BYTES 32
#define ISX_ABI_VERSION 1

#define ISX_EINVAL (-1)   /* bad argument (maps to ValueError in the Python host) */
#define ISX_ECUDA (-2)    /* CUDA runtime failure / no device */
#define ISX_ENOMEM (-3)   /* host or device allocation failed */
#define ISX_EIO (-4)      /* snapshot file problem */
#define ISX_ELIMIT (-5)   /* k beyond the supported maximum */

typedef struct isx_store isx_store_t;

/* timing / launch accounting of the most recent isx_search* call on a store */
typedef struct isx_stats {
    uint64_t kernel_launches;   /* all kernels launched by the call */
    uint64_t scan_launches;     /* launches of the scan kernel family */
    float scan_ms;              /* CUDA-event time over all scan launches (0 unless profiling on) */
    float select_ms;            /* CUDA-event time of init + final select (0 unless profiling on) */
    float total_ms;             /* CUDA-event time first launch .. last launch */
    uint64_t pairs;             /* (query, code) pairs scored */
    uint64_t algo_bytes;        /* sum over passes of N_b * min(Lq, L_b): the algorithmic HBM bytes */
    uint64_t algo_popc;         /* 32-bit popcounts the pairs need (ceil(min(Lq,L_b)/4) each) */
    uint64_t candidates;        /* rows that passed the running threshold (all queries) */
    uint64_t fallback_queries;  /* queries answered by the exact re-scan path (candidate overflow) */
    uint64_t passes;            /* passes over the store (query tiles) */
    uint64_t issued_popc;       /* POPC (per lane) the scan issues in steady state: lower-bound filter for 2,4,5,6
                                   words, carry-save otherwise: 1,1,2,2,3,3,4,5 for 1..8 words (estimate: while a
                                   query's threshold is still loose the exact path adds its carry-save count) */
} isx_stats_t;

const char* isx_last_error(void);
int isx_abi_version(void);
int isx_device_count(int* n_out);

/* key_bytes: 8 | 16.  max_bytes: longest code accepted (1..32).  fixed_len: 0 = variable length
 * (NPHD store), else every code and query must be exactly this many bytes (Hamming store). */
int isx_open(isx_store_t** out, int device, uint32_t key_bytes, uint32_t max_bytes, uint32_t fixed_len);
int isx_close(isx_store_t* s);

/* Use an existing CUDA stream (e.g. torch's current stream handle) for all work of this store.
 * NULL restores the store's own stream. */
int isx_set_stream(isx_store_t* s, void* cuda_stream);
/* Record CUDA events around the kernels of each search so isx_get_stats reports device times. */
int isx_set_profiling(isx_store_t* s, int enabled);
int isx_get_stats(isx_store_t* s, isx_stats_t* out);

/* added[i] = 1 if row i was stored, 0 if its key was already present (first wins, also inside the
 * batch) - tests/test_usearch_add.py:53-63.  added may be NULL. */
int isx_add(isx_store_t* s, const void* keys, const uint8_t* codes, const uint8_t* lens, size_t n, uint8_t* added);
/*
 * Bulk append straight from DEVICE memory (warm start from a snapshot already in HBM, a partition produced by another
 * GPU job, the synthetic 1 B-row data sets of SURVEY 8d): d_keys (n x key_bytes, same form as isx_add), d_codes
 * (n x 32 bytes), d_lens (n length bytes, or NULL = every code has uniform_len bytes). The caller PROMISES that the
 * keys are unique and not stored yet - no per-row host work happens here; the host key map is completed lazily by the
 * first keyed call (add / remove / contains / get / save), which fails with ISX_EINVAL if the promise was broken.
 * Replaces the add loop of a rebuild (iscc_search/indexes/usearch/index.py:1650-1726, lmdb_ops.py:304-343) for
 * data that is already on the device. Row placement inside a bucket is unspecified (results never depend on it).
 */
int isx_add_device(isx_store_t* s, const void* d_keys, const uint8_t* d_codes, const uint8_t* d_lens, uint32_t uniform_len, size_t n);
/*
 * Bench / test facility, not part of the reference boundary: rows [start, start+n) of the synthetic data set of
 * SURVEY.md 8d (definition: iscc_search_b200/synth.py) generated on the device, on the store's stream, into
 * caller-owned device buffers in the form isx_add_device takes. key_mode 0: uint64 keys; 1: 16-byte simprint chunk
 * pointers (chunks_per_asset chunks per asset). lengths: n_lengths (<= 8) code lengths, picked per row by a hash.
 * dup_every > 0: every dup_every-th row repeats the code of the row dup_back before it. d_lens may be NULL.
 */
int isx_synth_rows_device(isx_store_t* s, uint64_t seed, uint64_t start, size_t n, const uint8_t* lengths, uint32_t n_lengths,
                          uint32_t key_mode, uint32_t chunks_per_asset, uint32_t dup_every, uint32_t dup_back, void* d_keys,
                          uint8_t* d_codes, uint8_t* d_lens);
/* removed[i] = 1 if the key was present - tests/test_usearch_remove.py:19-48.  May be NULL. */
int isx_remove(isx_store_t* s, const void* keys, size_t n, uint8_t* removed, uint64_t* n_removed);
int isx_contains(isx_store_t* s, const void* keys, size_t n, uint8_t* present);
/* codes_out: n rows of 32 bytes (zero padded); lens_out[i] = 0 when the key is missing. */
int isx_get(isx_store_t* s, const void* keys, size_t n, uint8_t* codes_out, uint8_t* lens_out);
int isx_size(isx_store_t* s, uint64_t* n_out);
int isx_clear(isx_store_t* s);
/* Free the per-search working memory of a store (candidate lists, histograms, result / staging buffers: up to a few GB
 * after a large batch); it re-grows on demand. Rows and keys are untouched. A process that keeps many stores open
 * (one per unit type and simprint type of every index, iscc_search/indexes/usearch/manager.py:258-279) calls this after
 * batch work so that idle stores do not pin HBM next to the data. */
int isx_release_scratch(isx_store_t* s, uint64_t* bytes_freed);
/* bytes of device memory currently allocated for rows (planes + keys) */
int isx_device_bytes(isx_store_t* s, uint64_t* n_out);
/* bit L-1 set when at least one stored code has L bytes */
int isx_length_mask(isx_store_t* s, uint32_t* mask_out);

/* snapshot of (keys, lens, codes) per length bucket; load replaces the store's content */
int isx_save(isx_store_t* s, const char* path);
int isx_load(isx_store_t* s, const char* path);

/*
 * Exact top-k.  queries: q rows of 32 bytes; qlens: q length bytes.
 * thr_den == 0: no threshold; else only rows with h/nbits <= thr_num/thr_den are returned
 * (simprint threshold, usearch_core.py:182-184; thr_num = 0 gives the equality join).
 * Outputs, row major q x k, first counts_out[i] entries of row i valid:
 *   keys_out (q*k*key_bytes), hamming_out, nbits_out, counts_out (q),
 *   codes_out (optional, q*k*32: the matched stored codes - replaces the per-match .get() round
 *   trips at usearch_core.py:221,243),
 *   first_of_asset_out (optional, q*k flags, 128-bit keys: 1 where a record is the best one of its asset
 *   = high 8 key bytes within its query - the grouping loop of usearch_core.py:187-196 done on the device).
 */
int isx_search(isx_store_t* s, const uint8_t* queries, const uint8_t* qlens, size_t q, uint32_t k,
               uint32_t thr_num, uint32_t thr_den, void* keys_out, uint16_t* hamming_out, uint16_t* nbits_out,
               uint32_t* counts_out, uint8_t* codes_out, uint8_t* first_of_asset_out);

/*
 * Same search, results left in DEVICE memory as q x k records (for the multi-GPU merge):
 *   d_keys_hi, d_keys_lo (uint64, lo is 0 for 8-byte keys), d_hamming, d_nbits (uint16), d_counts (uint32[q]).
 * Unused record slots are filled with key = UINT64_MAX, h = 0xFFFF, nbits = 1 (sorts last).
 * queries/qlens are HOST pointers unless queries_on_device != 0 (then `queries` is a device
 * pointer to q x 32 bytes; qlens stays on the host - it drives the launch plan).
 * The call is synchronous with respect to the store's stream only if `sync` != 0.
 */
int isx_search_device(isx_store_t* s, const uint8_t* queries, int queries_on_device, const uint8_t* qlens, size_t q,
                      uint32_t k, uint32_t thr_num, uint32_t thr_den, uint64_t* d_keys_hi, uint64_t* d_keys_lo,
                      uint16_t* d_hamming, uint16_t* d_nbits, uint32_t* d_counts, int sync);

/*
 * Merge G per-shard result sets (device, as written by isx_search_device and delivered by an NCCL
 * all-gather) into the global top-k per query, same order rule. Input layout:
 *   shard_stride_bytes == 0: each field is one dense array [g][q][k] (counts: [g][q]);
 *   shard_stride_bytes != 0: the pointers address shard 0 and shard g's arrays start g*stride bytes
 *                            later (every rank packed its fields into one buffer of `stride` bytes).
 * Output device arrays are q x k.  Runs on the store's stream.
 */
int isx_merge_device(isx_store_t* s, uint32_t n_shards, size_t q, uint32_t k, size_t shard_stride_bytes, const uint64_t* d_keys_hi,
                     const uint64_t* d_keys_lo, const uint16_t* d_hamming, const uint16_t* d_nbits,
                     const uint32_t* d_counts, uint64_t* d_out_keys_hi, uint64_t* d_out_keys_lo,
                     uint16_t* d_out_hamming, uint16_t* d_out_nbits, uint32_t* d_out_counts, int sync);

/*
 * Unbounded threshold match of ONE query: every row with h/nbits <= thr_num/thr_den (thr_den != 0), in no
 * particular order. thr = 0/1 is the bidirectional prefix match of INSTANCE codes
 * (iscc_search/indexes/usearch/index.py:1957-2022: stored code starts with the query, or is a prefix of it).
 * At most max_out records are written; *total_out is the number of matching rows - if it exceeds max_out
 * call again with a larger buffer.
 */
int isx_match_all(isx_store_t* s, const uint8_t* query, uint32_t qlen, uint32_t thr_num, uint32_t thr_den, size_t max_out,
                  void* keys_out, uint16_t* hamming_out, uint16_t* nbits_out, uint64_t* total_out);

/*
 * Self-join: every unordered pair {a, b} of two distinct stored rows with h * thr_den <= thr_num * nbits (thr_den != 0),
 * h = popc(a[:m] ^ b[:m]), m = min(len a, len b) bytes, nbits = 8m - the threshold rule of isx_search (thr_num = 0: exact
 * duplicates plus prefix-equal rows of different lengths, the INSTANCE semantics). Which codes of the store are
 * near-duplicates of each other, without k and without a round trip of the codes through the host.
 * Each pair is scored once on the device and kept there as one record (key_a, key_b, h, nbits) with key_a < key_b
 * (8-byte keys: uint64 order; 16-byte keys: bytewise), all records in ascending (key_a, key_b) order; *total_out = pairs.
 * The result does not depend on row placement. It lives in the store's working memory until the next search or match,
 * add / remove / clear / load, isx_release_scratch or isx_close. Nothing is truncated: when the records do not fit in
 * device memory the call fails with ISX_ENOMEM, *total_out still set to the number of pairs found.
 * Takes the same locks as a search; isx_get_stats reports it like a search (scan launches, pairs scored, candidates).
 */
int isx_self_join(isx_store_t* s, uint32_t thr_num, uint32_t thr_den, uint64_t* total_out);
/*
 * Records [first, first + n) of the last isx_self_join, in (key_a, key_b) order, into host buffers: keys_a_out and
 * keys_b_out (n x key_bytes, the key form of isx_search), hamming_out, nbits_out. Fetch a large result in pages.
 * ISX_EINVAL when the result has ended (see above) or the range lies past the join's total.
 */
int isx_join_fetch(isx_store_t* s, uint64_t first, size_t n, void* keys_a_out, void* keys_b_out, uint16_t* hamming_out,
                   uint16_t* nbits_out);

/*
 * Simprint asset scoring on the device (the per-asset loop of iscc_search/indexes/simprint/usearch_core.py:199-269):
 * the best record of every (asset, query simprint) pair, grouped by asset (segment a = records [seg[a], seg[a+1])),
 * ascending query index inside a segment: rec_qi (query index), rec_sim (1 - h/ndim), rec_idf (IDF of the matched
 * simprint); q_idf[q] = IDF of query simprint q (added for every query the asset did not match).
 * score_out[a] = sum(idf * sim) / (sum(idf of matched) + sum(idf of unmatched queries)), every double operation in the
 * reference's order and rounding (no FMA), so the result is bit-identical to the reference's Python floats.
 * All pointers are host pointers.
 */
int isx_score_segments(isx_store_t* s, const uint32_t* seg, size_t n_assets, const uint32_t* rec_qi, const double* rec_sim,
                       const double* rec_idf, size_t n_rec, const double* q_idf, uint32_t n_queries, double* score_out);

/*
 * Cross-rank threshold sharing for row-sharded search (one process per GPU, all GPUs on one NVLink box).
 * Every rank owns "home" rank-histograms for a slice of the queries of a batch; peers map them through
 * CUDA IPC and (a) count every candidate they emit there with remote atomics, (b) tighten their thresholds
 * from those GLOBAL counts. A shard then stops emitting rows that cannot reach the merged top-k, which keeps
 * the per-shard work proportional to its rows. Results are unchanged (the merged top-k is exact either way).
 *   isx_share_init   allocate + export this rank's histograms (handle_out: 64 bytes, cudaIpcMemHandle_t)
 *   isx_share_attach map a peer's histograms (handle from its isx_share_init)
 *   isx_share_reset  enqueue zeroing of the home histograms on the store's stream and ARM the next search.
 *                    Protocol per batch, same on every rank: isx_share_reset -> a collective on the same stream
 *                    (barrier; the host layer all-reduces the stored-length masks there) -> isx_share_set_lengths ->
 *                    isx_search_device (identical queries, qlens, k on all ranks) -> all-gather + isx_merge_device.
 *                    A search that was not armed by a reset (isx_search, match_all, ...) never touches the shared state.
 *   isx_share_set_lengths  union over ALL ranks of isx_length_mask. The shared histograms are indexed by the dense
 *                    rank of h/nbits among the compared-length classes, so every rank must derive its rank table
 *                    from the same classes even when its own shard lacks a length bucket.
 * Sharing is used only when all of world > 1, q <= max_queries and the distance classes fit (<= 512 ranks).
 */
int isx_share_init(isx_store_t* s, uint32_t world, uint32_t rank, uint32_t max_queries, void* handle_out);
int isx_share_attach(isx_store_t* s, uint32_t peer_rank, const void* handle);
int isx_share_reset(isx_store_t* s);
int isx_share_set_lengths(isx_store_t* s, uint32_t global_length_mask);

/*
 * Host-only self tests (no CUDA device needed; used by the CPU test-suite):
 *   isx_selftest_rank_table  the dense rank of every h/(8m) for the compared-length classes in class_mask
 *                            (bit m-1), rank_out[33][257] (0xFFFF = unused), optional hmax_out[33][hmax_stride]
 *   isx_selftest_keymap      randomized insert/update/erase/find of the key -> row map against a reference
 */
int isx_selftest_rank_table(uint32_t class_mask, uint16_t* rank_out, uint16_t* hmax_out, uint32_t hmax_stride, uint32_t* R_out);
int isx_selftest_keymap(uint64_t n_ops, uint64_t seed, uint32_t key_space);
/*   isx_selftest_distance    the scan kernels' arithmetic helpers (carry-save distance, OR-fold lower bounds), built for the
 *                            host from the same template code, against a naive popcount on n random rows per word count */
int isx_selftest_distance(uint64_t n, uint64_t seed);

/* largest k isx_search accepts for this store (shared-memory bound of the final selection) */
int isx_max_k(isx_store_t* s, uint32_t* k_out);

#ifdef __cplusplus
}
#endif
#endif /* ISX_H */
