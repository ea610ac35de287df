/*
 * yams_oracle.h -- CPU ORACLE for the yams-b200 hot path.  TEST INFRASTRUCTURE ONLY.
 *
 * This is a plain-C restatement of the reference's (trvon/yams @ 8ab82c1c) algorithms for the
 * path BASELINE.json:north_star names.  It exists so tests/, __graft_entry__.smoke() and the
 * cpu_baseline / --impl reference legs of bench.py have something to check the CUDA path against.
 * Nothing in the product (yams_b200/, include/) links, imports or calls it.
 *
 * Parity pinning: every function here is checked (tests/test_oracle_*.py) against
 *   - the reference's own KATs (SHA-256: tests/unit/crypto/crypto_test.cpp:92-99; distances:
 *     third_party/sqlite-vec-cpp/tests/test_distances.cpp:20-53, distance_metrics_test.cpp:98-120,
 *     254-292, test_batch_distance.cpp:19-104, sqlite_vec_c_api_smoke_catch2_test.cpp:19-75), and
 *   - oracle/_ref (the reference's own rabin_chunker.cpp / streaming_chunker.cpp /
 *     sha256_hasher.cpp / sqlite-vec-cpp distance headers compiled from /root/reference by
 *     oracle/Makefile), and the golden fixtures that build generated (tests/golden/).
 *
 * All path:line citations are relative to /root/reference.
 */
#ifndef YAMS_ORACLE_H
#define YAMS_ORACLE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- CDC (src/chunking) ------------------------------------------------------------------ */

enum { YO_CDC_STREAMING = 0, YO_CDC_RABIN = 1 };

typedef struct yo_cdc_config {
    uint64_t window_size; /* chunker.h:45  (ring is a fixed 48-byte array: chunker.h:151)       */
    uint64_t min_chunk;   /* chunker.h:46                                                        */
    uint64_t max_chunk;   /* chunker.h:48                                                        */
    uint64_t polynomial;  /* chunker.h:49                                                        */
    uint64_t mask;        /* chunker.h:50                                                        */
    int32_t variant;      /* YO_CDC_STREAMING = StreamingChunker, YO_CDC_RABIN = RabinChunker    */
} yo_cdc_config;

void yo_cdc_default_config(yo_cdc_config* cfg);

/* rabin_fingerprint_table.h:14-27 */
void yo_rabin_table(uint64_t polynomial, uint64_t out_table[256]);

/* Full rolling state (rabin_chunker.cpp:45-61 / streaming_chunker.cpp:37-69) evaluated at every
 * position of the stream; writes positions p with (h_p & mask) == mask.  Returns the count
 * (may exceed cap; only the first cap are written). */
size_t yo_cdc_candidates_full(const uint8_t* data, size_t n, const yo_cdc_config* cfg,
                              uint64_t* out_pos, size_t cap);

/* Closed-form predicate (SURVEY.md headline fact 3): bits < 8*s of h_p depend only on the s newest
 * and s oldest-leaving bytes.  Evaluated independently per position. */
size_t yo_cdc_candidates_local(const uint8_t* data, size_t n, const yo_cdc_config* cfg,
                               uint64_t* out_pos, size_t cap);

/* Sequential chunking, restating StreamingChunker::processBuffer (streaming_chunker.h:146-181,
 * remainder :115-118) or RabinChunker::chunkDataImpl/findChunkBoundary
 * (rabin_chunker.cpp:63-152).  Returns chunk count (may exceed cap). */
size_t yo_cdc_chunk(const uint8_t* data, size_t n, const yo_cdc_config* cfg, uint64_t* out_offsets,
                    uint64_t* out_sizes, size_t cap);

/* Chunk + SHA-256 per chunk (rabin_chunker.cpp:140, streaming_chunker.h:190). digests: cap*32 B */
size_t yo_cdc_chunk_and_hash(const uint8_t* data, size_t n, const yo_cdc_config* cfg,
                             uint64_t* out_offsets, uint64_t* out_sizes, uint8_t* out_digests,
                             size_t cap);

/* ---- SHA-256 (src/crypto -> OpenSSL EVP_sha256 == FIPS 180-4) --------------------------- */

typedef struct yo_sha256_ctx {
    uint32_t h[8];
    uint64_t nbytes;
    uint8_t buf[64];
    uint32_t buflen;
} yo_sha256_ctx;

void yo_sha256_init(yo_sha256_ctx* c);                                /* sha256_hasher.cpp:81  */
void yo_sha256_update(yo_sha256_ctx* c, const uint8_t* d, size_t n);  /* sha256_hasher.cpp:87  */
void yo_sha256_final(yo_sha256_ctx* c, uint8_t out[32]);              /* sha256_hasher.cpp:93  */
void yo_sha256(const uint8_t* d, size_t n, uint8_t out[32]);          /* sha256_hasher.cpp:167 */
void yo_sha256_batch(const uint8_t* base, const uint64_t* offsets, const uint64_t* sizes, size_t n,
                     uint8_t* out_digests);
void yo_bytes_to_hex(const uint8_t* d, size_t n, char* out /* 2n+1 */); /* sha256_hasher.cpp:19 */

/* ---- fp16 (sqlite-vec-cpp utils/float16.hpp:20-66) ---------------------------------------- */
uint16_t yo_f16_from_float(float f); /* truncating */
float yo_f16_to_float(uint16_t h);

/* ---- distances (sqlite-vec-cpp distances/{cosine,l2}.hpp scalar paths) -------------------- */
float yo_cosine_distance_f32(const float* a, const float* b, size_t d); /* cosine.hpp:48-69  */
float yo_l2_distance_f32(const float* a, const float* b, size_t d);     /* l2.hpp:108-118    */
/* l2_distance<float> in the operation order of the reference BUILD (sqlite-vec-cpp compiled with AVX, see
 * yams_b200/csrc/ref_order.cuh): d >= 16 && d % 16 == 0 -> eight lane-strided float partial sums (multiply and add
 * rounded separately), lanes summed left to right, sqrtf; otherwise the scalar loop of yo_l2_distance_f32. */
float yo_l2_distance_build_f32(const float* a, const float* b, size_t d);
/* vector_database.cpp:1786-1810 */
double yo_cosine_similarity_f64(const float* a, const float* b, size_t d);
/* sqlite_vec_c_api.cpp:57-105: returns 0 ok / 1 error, sizes in BYTES */
int yo_vec_distance_l2(const void* a, size_t abytes, const void* b, size_t bbytes, float* out);
int yo_vec_distance_cosine(const void* a, size_t abytes, const void* b, size_t bbytes, float* out);

/* ---- exact scan (src/vector/sqlite_vec_backend.cpp:4203-4331) ----------------------------- */

enum { YO_DTYPE_F32 = 0, YO_DTYPE_F16 = 1 };
enum { YO_METRIC_COSINE = 0, YO_METRIC_L2 = 1 };

/* status: 0 ok, 1 invalid argument (non-finite / zero-norm query, :4127-4130) */
/* rows: n x d row-major (fp32 or fp16 bit patterns, upcast with yo_f16_to_float).
 * rowids: nullable (then rowid = index).  tie_rank: nullable; when given, equal-similarity rows are
 * ordered by tie_rank asc (stands in for the chunk_id string order, :4218-4223), else by rowid asc.
 * allowed: nullable sorted rowid list (candidate set, CandidateFilterMode::Exact).
 * k == 0 -> AllMatching is NOT implied; k==0 returns 0 rows (:4123-4126).
 * all_matching != 0 -> every passing row, sorted (:4283-4288,4315-4316); out arrays must hold n.
 * Returns number of rows written through *out_count. */
int yo_exact_scan_cosine(const void* rows, int dtype, size_t n, size_t d, const int64_t* rowids,
                         const int64_t* tie_rank, const float* query, size_t k, float threshold,
                         const int64_t* allowed, size_t n_allowed, int all_matching,
                         int64_t* out_rowids, float* out_scores, size_t* out_count);

/* Q independent queries, OpenMP over queries; out arrays are Q x k, counts Q. */
int yo_exact_scan_cosine_batch(const void* rows, int dtype, size_t n, size_t d,
                               const float* queries, size_t nq, size_t k, float threshold,
                               int64_t* out_rowids, float* out_scores, uint32_t* out_counts);

/* vec0_run_exact_query (sqlite/vec0_module.hpp:376-430): float L2 + sqrt per row, sort asc by
 * distance (ties: rowid asc -- a legal refinement of the unstable std::sort), truncate to k if
 * k > 0 (k == 0 means "no k": all rows).  rowid filter: [rowid_lo, rowid_hi] inclusive when
 * use_range != 0. fp32 rows only. */
int yo_vec0_exact(const float* rows, size_t n, size_t d, const int64_t* rowids, const float* query,
                  size_t k, int use_range, int64_t rowid_lo, int64_t rowid_hi, int64_t* out_rowids,
                  float* out_dist, size_t* out_count);

/* Exact L2 top-k of Q queries (OpenMP over queries) with yo_l2_distance_build_f32(query, row): the library's L2 search
 * contract.  rows: n x d, fp32 or fp16 bit patterns (upcast exactly).  Order: distance asc, ties by row index asc; rows
 * whose distance is NaN are left out.  out arrays are Q x k: count = min(k, rows kept), the rest padded with rowid -1
 * and distance +inf. */
void yo_exact_scan_l2_batch(const void* rows, int dtype, size_t n, size_t d, const float* queries, size_t nq,
                            size_t k, int64_t* out_rowids, float* out_dist, uint32_t* out_counts);

/* distances/batch.hpp:74-92 batch_top_k: indices of the k smallest distances (ties: index asc).
 * metric: YO_METRIC_COSINE uses cosine *distance*, YO_METRIC_L2 uses l2_distance. */
size_t yo_batch_top_k(const float* query, const float* rows, size_t n, size_t d, int metric,
                      size_t k, uint64_t* out_idx, float* out_dist);

/* ---- synthetic inputs (SURVEY.md §8d) ------------------------------------------------------ */
uint64_t yo_splitmix64(uint64_t x);
/* byte[i] = (splitmix64(seed ^ (i>>3)) >> (8*(i&7))) & 0xFF for i in [start, start+n) */
void yo_gen_bytes(uint64_t seed, uint64_t start, size_t n, uint8_t* out);
/* row-major n x d: u = splitmix64(seed ^ (row*d + col)), x = (u>>40)*2^-23 - 1, L2-normalised in
 * fp32 (sum in double, scale in float); first_row lets callers generate slices. */
void yo_gen_rows_f32(uint64_t seed, uint64_t first_row, size_t n, size_t d, float* out);

/* ManifestManager::calculateChecksum (src/manifest/manifest_manager.cpp:705-730) over raw digests + (offset, size) */
uint32_t yo_manifest_checksum(const uint8_t* file_digest32, uint64_t file_size, const uint8_t* digests,
                              const uint64_t* offsets, const uint64_t* sizes, size_t n);

#ifdef __cplusplus
}
#endif
#endif
