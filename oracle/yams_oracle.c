/*
 * yams_oracle.c -- CPU ORACLE (test infrastructure only; see yams_oracle.h).
 * Restates the reference algorithms; citations are file:line under /root/reference.
 */
#include "yams_oracle.h"

#include <math.h>
#include <stdlib.h>
#include <stdio.h>
#include <string.h>

/* ============================== CDC ====================================================== */

void yo_cdc_default_config(yo_cdc_config* cfg) {
    /* include/yams/chunking/chunker.h:44-51, include/yams/core/types.h:280-285 */
    cfg->window_size = 48;
    cfg->min_chunk = 16 * 1024;
    cfg->max_chunk = 1024 * 1024;
    cfg->polynomial = 0x3DA3358B4DC173ULL;
    cfg->mask = 0x1FFF;
    cfg->variant = YO_CDC_STREAMING; /* `yams add` uses StreamingChunker:
                                        src/api/content_store_builder.cpp:152-165 */
}

void yo_rabin_table(uint64_t polynomial, uint64_t out_table[256]) {
    /* src/chunking/rabin_fingerprint_table.h:16-26 */
    for (int byte = 0; byte < 256; ++byte) {
        uint64_t hash = 0;
        for (int bit = 0; bit < 8; ++bit) {
            if ((byte & (1 << bit)) != 0) {
                hash ^= polynomial << bit;
            }
        }
        out_table[byte] = hash;
    }
}

/* Effective ring length.  StreamingChunker clamps to [1,48] (streaming_chunker.cpp:44-49);
 * RabinChunker wraps at config.windowSize over a 48-byte array (rabin_chunker.cpp:51-55), which is
 * only defined for 1..48.  The oracle therefore requires 1 <= window <= 48 and clamps like the
 * streaming variant. */
static size_t eff_window(const yo_cdc_config* cfg) {
    size_t w = (size_t)cfg->window_size;
    if (w == 0) w = 1;
    if (w > 48) w = 48;
    return w;
}

static uint64_t eff_poly(const yo_cdc_config* cfg) {
    /* rabin_chunker.cpp:30-36 / streaming_chunker.cpp:21-27: zero polynomial -> default */
    return cfg->polynomial != 0 ? cfg->polynomial : 0x3DA3358B4DC173ULL;
}

typedef struct {
    uint8_t ring[48];
    size_t pos;
    uint64_t hash;
} roll_state;

static inline void roll(roll_state* s, const uint64_t* T, size_t w, uint8_t b) {
    /* rabin_chunker.cpp:80-87 == streaming_chunker.cpp:55-68 */
    uint8_t old = s->ring[s->pos];
    s->ring[s->pos] = b;
    ++s->pos;
    if (s->pos >= w) s->pos = 0;
    s->hash = ((s->hash - T[old]) << 8) ^ T[b];
}

size_t yo_cdc_candidates_full(const uint8_t* data, size_t n, const yo_cdc_config* cfg,
                              uint64_t* out_pos, size_t cap) {
    uint64_t T[256];
    yo_rabin_table(eff_poly(cfg), T);
    const size_t w = eff_window(cfg);
    roll_state s;
    memset(&s, 0, sizeof s);
    size_t cnt = 0;
    for (size_t p = 0; p < n; ++p) {
        roll(&s, T, w, data[p]);
        if ((s.hash & cfg->mask) == cfg->mask) {
            if (cnt < cap) out_pos[cnt] = p;
            ++cnt;
        }
    }
    return cnt;
}

/* number of rolling steps whose bytes can influence bits selected by mask */
static int mask_steps(uint64_t mask) {
    if (mask == 0) return 0;
    int hi = 63;
    while (!((mask >> hi) & 1)) --hi;
    return hi / 8 + 1; /* 1..8 */
}

size_t yo_cdc_candidates_local(const uint8_t* data, size_t n, const yo_cdc_config* cfg,
                               uint64_t* out_pos, size_t cap) {
    uint64_t T[256];
    yo_rabin_table(eff_poly(cfg), T);
    const size_t w = eff_window(cfg);
    const int steps = mask_steps(cfg->mask);
    size_t cnt = 0;
    for (size_t p = 0; p < n; ++p) {
        /* h restarted from 0 at position p-steps+1: bits below 8*steps are identical to the
         * full-state value because '<< 8' only moves information upward and '-' only borrows
         * upward (SURVEY.md fact 3). Bytes before the stream start read as 0 (zero ring). */
        uint64_t h = 0;
        for (int j = steps - 1; j >= 0; --j) {
            if ((size_t)j > p) continue; /* before the stream start: state is still 0 */
            size_t q = p - (size_t)j;
            uint8_t nb = data[q];
            uint8_t ob = q >= w ? data[q - w] : 0;
            h = ((h - T[ob]) << 8) ^ T[nb];
        }
        if ((h & cfg->mask) == cfg->mask) {
            if (cnt < cap) out_pos[cnt] = p;
            ++cnt;
        }
    }
    return cnt;
}

static size_t chunk_streaming(const uint8_t* data, size_t n, const yo_cdc_config* cfg,
                              uint64_t* out_offsets, uint64_t* out_sizes, size_t cap) {
    /* streaming_chunker.h:146-181 (processBuffer), :184-204 (emitChunk), chunkData tail
     * streaming_chunker.cpp:124-134.  The 64 KiB buffering (streaming_chunker.cpp:99-121) does not
     * affect results: all state lives in the StreamingContext. */
    uint64_t T[256];
    yo_rabin_table(eff_poly(cfg), T);
    const size_t w = eff_window(cfg);
    roll_state s;
    memset(&s, 0, sizeof s);
    size_t cnt = 0;
    size_t acc = 0;          /* ctx.accumulator.size() */
    size_t chunk_start = 0;  /* ctx.currentChunkStart */
    for (size_t off = 0; off < n; ++off) {
        ++acc; /* accumulator.push_back */
        roll(&s, T, w, data[off]);
        int emit = 0;
        if (acc >= cfg->min_chunk) {
            if ((s.hash & cfg->mask) == cfg->mask) {
                emit = 1;
            } else if (acc >= cfg->max_chunk) {
                emit = 1;
            }
        }
        if (emit) {
            if (cnt < cap) {
                out_offsets[cnt] = chunk_start;
                out_sizes[cnt] = acc;
            }
            ++cnt;
            chunk_start = off + 1;
            acc = 0;
        }
    }
    if (acc != 0) { /* finalizeChunk */
        if (cnt < cap) {
            out_offsets[cnt] = chunk_start;
            out_sizes[cnt] = acc;
        }
        ++cnt;
    }
    return cnt;
}

static size_t chunk_rabin(const uint8_t* data, size_t n, const yo_cdc_config* cfg,
                          uint64_t* out_offsets, uint64_t* out_sizes, size_t cap) {
    /* rabin_chunker.cpp:120-152 (chunkDataImpl) + :63-110 (findChunkBoundary).  The window is
     * created once per call and never reset at a cut (:126-129). */
    uint64_t T[256];
    yo_rabin_table(eff_poly(cfg), T);
    const size_t w = eff_window(cfg);
    roll_state s;
    memset(&s, 0, sizeof s);
    size_t cnt = 0;
    size_t start = 0;
    while (start < n) {
        size_t min_b = start + cfg->min_chunk;
        if (min_b > n || min_b < start) min_b = n;
        size_t max_b = start + cfg->max_chunk;
        if (max_b > n || max_b < start) max_b = n;
        size_t pos = start;
        size_t end;
        int found = 0;
        while (pos < min_b) {
            roll(&s, T, w, data[pos++]);
        }
        end = pos;
        while (pos < max_b) {
            roll(&s, T, w, data[pos]);
            if ((s.hash & cfg->mask) == cfg->mask) {
                end = pos + 1;
                found = 1;
                break;
            }
            ++pos;
        }
        if (!found) end = pos;
        if (end == start) { /* max_chunk == 0 && min_chunk == 0: reference would spin forever */
            return cnt;
        }
        if (cnt < cap) {
            out_offsets[cnt] = start;
            out_sizes[cnt] = end - start;
        }
        ++cnt;
        start = end;
    }
    return cnt;
}

size_t yo_cdc_chunk(const uint8_t* data, size_t n, const yo_cdc_config* cfg, uint64_t* out_offsets,
                    uint64_t* out_sizes, size_t cap) {
    if (cfg->variant == YO_CDC_RABIN) return chunk_rabin(data, n, cfg, out_offsets, out_sizes, cap);
    return chunk_streaming(data, n, cfg, out_offsets, out_sizes, cap);
}

size_t yo_cdc_chunk_and_hash(const uint8_t* data, size_t n, const yo_cdc_config* cfg,
                             uint64_t* out_offsets, uint64_t* out_sizes, uint8_t* out_digests,
                             size_t cap) {
    size_t cnt = yo_cdc_chunk(data, n, cfg, out_offsets, out_sizes, cap);
    size_t m = cnt < cap ? cnt : cap;
    yo_sha256_batch(data, out_offsets, out_sizes, m, out_digests);
    return cnt;
}

/* ============================== SHA-256 (FIPS 180-4) ===================================== */
/* The reference delegates to OpenSSL libcrypto EVP_sha256 (src/crypto/sha256_hasher.cpp:71-109,
 * conanfile.py:95 pins openssl/3.2.0; not vendored).  Restated from the published standard. */

static const uint32_t K256[64] = {
    0x428a2f98, 0x71374491, 0xb5c0fbcf, 0xe9b5dba5, 0x3956c25b, 0x59f111f1, 0x923f82a4, 0xab1c5ed5,
    0xd807aa98, 0x12835b01, 0x243185be, 0x550c7dc3, 0x72be5d74, 0x80deb1fe, 0x9bdc06a7, 0xc19bf174,
    0xe49b69c1, 0xefbe4786, 0x0fc19dc6, 0x240ca1cc, 0x2de92c6f, 0x4a7484aa, 0x5cb0a9dc, 0x76f988da,
    0x983e5152, 0xa831c66d, 0xb00327c8, 0xbf597fc7, 0xc6e00bf3, 0xd5a79147, 0x06ca6351, 0x14292967,
    0x27b70a85, 0x2e1b2138, 0x4d2c6dfc, 0x53380d13, 0x650a7354, 0x766a0abb, 0x81c2c92e, 0x92722c85,
    0xa2bfe8a1, 0xa81a664b, 0xc24b8b70, 0xc76c51a3, 0xd192e819, 0xd6990624, 0xf40e3585, 0x106aa070,
    0x19a4c116, 0x1e376c08, 0x2748774c, 0x34b0bcb5, 0x391c0cb3, 0x4ed8aa4a, 0x5b9cca4f, 0x682e6ff3,
    0x748f82ee, 0x78a5636f, 0x84c87814, 0x8cc70208, 0x90befffa, 0xa4506ceb, 0xbef9a3f7, 0xc67178f2};

static inline uint32_t rotr32(uint32_t x, int r) { return (x >> r) | (x << (32 - r)); }

static void sha256_block(uint32_t st[8], const uint8_t* p) {
    uint32_t w[64];
    for (int i = 0; i < 16; ++i) {
        w[i] = ((uint32_t)p[4 * i] << 24) | ((uint32_t)p[4 * i + 1] << 16) |
               ((uint32_t)p[4 * i + 2] << 8) | (uint32_t)p[4 * i + 3];
    }
    for (int i = 16; i < 64; ++i) {
        uint32_t s0 = rotr32(w[i - 15], 7) ^ rotr32(w[i - 15], 18) ^ (w[i - 15] >> 3);
        uint32_t s1 = rotr32(w[i - 2], 17) ^ rotr32(w[i - 2], 19) ^ (w[i - 2] >> 10);
        w[i] = w[i - 16] + s0 + w[i - 7] + s1;
    }
    uint32_t a = st[0], b = st[1], c = st[2], d = st[3], e = st[4], f = st[5], g = st[6], h = st[7];
    for (int i = 0; i < 64; ++i) {
        uint32_t S1 = rotr32(e, 6) ^ rotr32(e, 11) ^ rotr32(e, 25);
        uint32_t ch = (e & f) ^ (~e & g);
        uint32_t t1 = h + S1 + ch + K256[i] + w[i];
        uint32_t S0 = rotr32(a, 2) ^ rotr32(a, 13) ^ rotr32(a, 22);
        uint32_t mj = (a & b) ^ (a & c) ^ (b & c);
        uint32_t t2 = S0 + mj;
        h = g; g = f; f = e; e = d + t1; d = c; c = b; b = a; a = t1 + t2;
    }
    st[0] += a; st[1] += b; st[2] += c; st[3] += d; st[4] += e; st[5] += f; st[6] += g; st[7] += h;
}

void yo_sha256_init(yo_sha256_ctx* c) {
    static const uint32_t iv[8] = {0x6a09e667, 0xbb67ae85, 0x3c6ef372, 0xa54ff53a,
                                   0x510e527f, 0x9b05688c, 0x1f83d9ab, 0x5be0cd19};
    memcpy(c->h, iv, sizeof iv);
    c->nbytes = 0;
    c->buflen = 0;
}

void yo_sha256_update(yo_sha256_ctx* c, const uint8_t* d, size_t n) {
    c->nbytes += n;
    if (c->buflen) {
        size_t take = 64 - c->buflen;
        if (take > n) take = n;
        memcpy(c->buf + c->buflen, d, take);
        c->buflen += (uint32_t)take;
        d += take;
        n -= take;
        if (c->buflen == 64) {
            sha256_block(c->h, c->buf);
            c->buflen = 0;
        }
    }
    while (n >= 64) {
        sha256_block(c->h, d);
        d += 64;
        n -= 64;
    }
    if (n) {
        memcpy(c->buf, d, n);
        c->buflen = (uint32_t)n;
    }
}

void yo_sha256_final(yo_sha256_ctx* c, uint8_t out[32]) {
    uint64_t bits = c->nbytes * 8;
    uint8_t pad[72];
    size_t padlen = (c->buflen < 56) ? (56 - c->buflen) : (120 - c->buflen);
    memset(pad, 0, sizeof pad);
    pad[0] = 0x80;
    for (int i = 0; i < 8; ++i) pad[padlen + i] = (uint8_t)(bits >> (56 - 8 * i));
    uint64_t keep = c->nbytes;
    yo_sha256_update(c, pad, padlen + 8);
    c->nbytes = keep;
    for (int i = 0; i < 8; ++i) {
        out[4 * i] = (uint8_t)(c->h[i] >> 24);
        out[4 * i + 1] = (uint8_t)(c->h[i] >> 16);
        out[4 * i + 2] = (uint8_t)(c->h[i] >> 8);
        out[4 * i + 3] = (uint8_t)(c->h[i]);
    }
    yo_sha256_init(c); /* sha256_hasher.cpp:104: finalize re-inits */
}

void yo_sha256(const uint8_t* d, size_t n, uint8_t out[32]) {
    yo_sha256_ctx c;
    yo_sha256_init(&c);
    if (n) yo_sha256_update(&c, d, n);
    yo_sha256_final(&c, out);
}

void yo_sha256_batch(const uint8_t* base, const uint64_t* offsets, const uint64_t* sizes, size_t n,
                     uint8_t* out_digests) {
    long i;
#pragma omp parallel for schedule(dynamic, 16)
    for (i = 0; i < (long)n; ++i) {
        yo_sha256(base + offsets[i], (size_t)sizes[i], out_digests + 32 * (size_t)i);
    }
}

void yo_bytes_to_hex(const uint8_t* d, size_t n, char* out) {
    static const char hex[] = "0123456789abcdef"; /* sha256_hasher.cpp:21 */
    for (size_t i = 0; i < n; ++i) {
        out[2 * i] = hex[(d[i] >> 4) & 0xF];
        out[2 * i + 1] = hex[d[i] & 0xF];
    }
    out[2 * n] = '\0';
}

/* ============================== fp16 ====================================================== */

uint16_t yo_f16_from_float(float f) {
    /* utils/float16.hpp:20-40 -- truncating mantissa, flush exp < -10, overflow -> inf.
     * NOTE (restated faithfully): NaN inputs have exp >= 31 and therefore map to +-inf. */
    uint32_t x;
    memcpy(&x, &f, 4);
    uint32_t sign = (x >> 16) & 0x8000;
    int32_t exp = (int32_t)((x >> 23) & 0xFF) - 127 + 15;
    uint32_t mant = x & 0x7FFFFF;
    uint16_t r;
    if (exp <= 0) {
        if (exp < -10) {
            r = (uint16_t)sign;
        } else {
            mant = (mant | 0x800000) >> (1 - exp);
            r = (uint16_t)(sign | (mant >> 13));
        }
    } else if (exp >= 31) {
        r = (uint16_t)(sign | 0x7C00);
    } else {
        r = (uint16_t)(sign | ((uint32_t)exp << 10) | (mant >> 13));
    }
    return r;
}

float yo_f16_to_float(uint16_t bits) {
    /* utils/float16.hpp:42-66 */
    uint32_t sign = ((uint32_t)bits & 0x8000) << 16;
    uint32_t exp = (bits >> 10) & 0x1F;
    uint32_t mant = bits & 0x3FF;
    uint32_t r;
    if (exp == 0) {
        if (mant == 0) {
            r = sign;
        } else {
            exp = 1;
            while ((mant & 0x400) == 0) {
                mant <<= 1;
                exp--;
            }
            mant &= 0x3FF;
            r = sign | ((exp + 127 - 15) << 23) | (mant << 13);
        }
    } else if (exp == 31) {
        r = sign | 0x7F800000 | (mant << 13);
    } else {
        r = sign | ((exp + 127 - 15) << 23) | (mant << 13);
    }
    float f;
    memcpy(&f, &r, 4);
    return f;
}

/* ============================== distances ================================================= */

float yo_cosine_distance_f32(const float* a, const float* b, size_t d) {
    /* distances/cosine.hpp:48-69 (scalar float path; the AVX path :99-107 differs only in
     * summation order) */
    float dot = 0.0f, am = 0.0f, bm = 0.0f;
    for (size_t i = 0; i < d; ++i) {
        dot += a[i] * b[i];
        am += a[i] * a[i];
        bm += b[i] * b[i];
    }
    float denom = sqrtf(am) * sqrtf(bm);
    if (denom < 1e-8f) return 1.0f;
    return 1.0f - (dot / denom);
}

float yo_l2_distance_f32(const float* a, const float* b, size_t d) {
    /* distances/l2.hpp:108-118 */
    float sum = 0.0f;
    for (size_t i = 0; i < d; ++i) {
        float diff = a[i] - b[i];
        sum += diff * diff;
    }
    return sqrtf(sum);
}

float yo_l2_distance_build_f32(const float* a, const float* b, size_t d) {
    /* The build compiles distances/simd/avx.hpp (SQLITE_VEC_ENABLE_AVX, no FMA macro): one 8-float accumulator, so lane l
     * sums the elements c + l, c = 0, 8, 16, ...; each (a - b)^2 is a rounded product added with its own rounding; the
     * 8 lanes are then added left to right.  The vector path runs for d >= 16 && d % 16 == 0 only. */
    if (d >= 16 && d % 16 == 0) {
        float p[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        for (size_t c = 0; c < d; c += 8) {
            for (int l = 0; l < 8; ++l) {
                float diff = a[c + l] - b[c + l];
                float sq = diff * diff;
                p[l] = p[l] + sq;
            }
        }
        float sum = p[0];
        for (int l = 1; l < 8; ++l) sum = sum + p[l];
        return sqrtf(sum);
    }
    return yo_l2_distance_f32(a, b, d);
}

double yo_cosine_similarity_f64(const float* a, const float* b, size_t d) {
    /* src/vector/vector_database.cpp:1786-1810 */
    double dp = 0.0, na = 0.0, nb = 0.0;
    for (size_t i = 0; i < d; ++i) {
        dp += (double)a[i] * (double)b[i];
        na += (double)a[i] * (double)a[i];
        nb += (double)b[i] * (double)b[i];
    }
    na = sqrt(na);
    nb = sqrt(nb);
    if (na == 0.0 || nb == 0.0) return 0.0;
    return dp / (na * nb);
}

int yo_vec_distance_l2(const void* a, size_t abytes, const void* b, size_t bbytes, float* out) {
    /* third_party/sqlite-vec-cpp/src/sqlite_vec_c_api.cpp:57-80 */
    if (!a || !b || !out) return 1;
    size_t d1 = abytes / sizeof(float), d2 = bbytes / sizeof(float);
    if (d1 != d2) return 1;
    *out = yo_l2_distance_f32((const float*)a, (const float*)b, d1);
    return 0;
}

int yo_vec_distance_cosine(const void* a, size_t abytes, const void* b, size_t bbytes, float* out) {
    /* sqlite_vec_c_api.cpp:82-105 */
    if (!a || !b || !out) return 1;
    size_t d1 = abytes / sizeof(float), d2 = bbytes / sizeof(float);
    if (d1 != d2) return 1;
    *out = yo_cosine_distance_f32((const float*)a, (const float*)b, d1);
    return 0;
}

/* ============================== exact scan ================================================ */

typedef struct {
    float sim;
    int64_t tie;
    int64_t rowid;
} scored;

/* "better" comparator: sqlite_vec_backend.cpp:4218-4223 */
static inline int better(const scored* a, const scored* b) {
    if (a->sim != b->sim) return a->sim > b->sim;
    return a->tie < b->tie;
}

static int cmp_better(const void* pa, const void* pb) {
    const scored* a = (const scored*)pa;
    const scored* b = (const scored*)pb;
    if (better(a, b)) return -1;
    if (better(b, a)) return 1;
    return 0;
}

/* binary heap with the WORST retained row at the front (std::push_heap with `better`) */
static void heap_sift_up(scored* h, size_t i) {
    while (i > 0) {
        size_t p = (i - 1) / 2;
        /* std heap w/ comparator better: parent must not be "better-less" than child, i.e.
         * front = element for which better(front, x) is false for all x = the worst. */
        if (better(&h[p], &h[i])) {
            scored t = h[p]; h[p] = h[i]; h[i] = t;
            i = p;
        } else {
            break;
        }
    }
}

static void heap_sift_down(scored* h, size_t n, size_t i) {
    for (;;) {
        size_t l = 2 * i + 1, r = l + 1, m = i;
        if (l < n && better(&h[m], &h[l])) m = l;
        if (r < n && better(&h[m], &h[r])) m = r;
        if (m == i) break;
        scored t = h[m]; h[m] = h[i]; h[i] = t;
        i = m;
    }
}

static int in_sorted(const int64_t* a, size_t n, int64_t v) {
    size_t lo = 0, hi = n;
    while (lo < hi) {
        size_t mid = lo + (hi - lo) / 2;
        if (a[mid] < v) lo = mid + 1; else hi = mid;
    }
    return lo < n && a[lo] == v;
}

int yo_exact_scan_cosine(const void* rows, int dtype, size_t n, size_t d, const int64_t* rowids,
                         const int64_t* tie_rank, const float* query, size_t k, float threshold,
                         const int64_t* allowed, size_t n_allowed, int all_matching,
                         int64_t* out_rowids, float* out_scores, size_t* out_count) {
    *out_count = 0;
    if (d == 0 || (!all_matching && k == 0)) return 0; /* :4123-4126 */
    /* :4127-4130 -> isFiniteEmbedding (:228-235), isZeroNormEmbedding (:204-211, < 1e-10) */
    double qn2 = 0.0;
    for (size_t i = 0; i < d; ++i) {
        if (!isfinite(query[i])) return 1;
        qn2 += (double)query[i] * (double)query[i];
    }
    if (qn2 < 1e-10) return 1;
    const double query_norm = sqrt(qn2); /* :4204-4209 */

    size_t cap = all_matching ? n : k;
    scored* sc = (scored*)malloc((cap ? cap : 1) * sizeof(scored));
    size_t cnt = 0;
    const float* r32 = (const float*)rows;
    const uint16_t* r16 = (const uint16_t*)rows;
    for (size_t r = 0; r < n; ++r) {
        int64_t rid = rowids ? rowids[r] : (int64_t)r;
        if (allowed && !in_sorted(allowed, n_allowed, rid)) continue;
        double norm_sq = 0.0, dot = 0.0;
        int finite = 1;
        for (size_t i = 0; i < d; ++i) { /* :4253-4266 */
            float v = dtype == YO_DTYPE_F16 ? yo_f16_to_float(r16[r * d + i]) : r32[r * d + i];
            if (!isfinite(v)) { finite = 0; break; }
            double sv = (double)v, qv = (double)query[i];
            norm_sq += sv * sv;
            dot += sv * qv;
        }
        if (!finite || norm_sq <= 1e-12) continue; /* :4267-4269 */
        double denom = sqrt(norm_sq) * query_norm;
        double simd = denom > 0.0 ? dot / denom : 0.0; /* :4271-4272 */
        if (!isfinite(simd)) continue;
        float sim = (float)simd; /* :4276 */
        if (sim < threshold) continue; /* :4277 */
        scored s;
        s.sim = sim;
        s.rowid = rid;
        s.tie = tie_rank ? tie_rank[r] : rid;
        if (all_matching) {
            sc[cnt++] = s;
        } else if (cnt < k) { /* :4289-4295 */
            sc[cnt++] = s;
            heap_sift_up(sc, cnt - 1);
        } else if (better(&s, &sc[0])) { /* :4296-4305 */
            sc[0] = s;
            heap_sift_down(sc, cnt, 0);
        }
    }
    qsort(sc, cnt, sizeof(scored), cmp_better); /* :4315-4318 (total order -> same result) */
    for (size_t i = 0; i < cnt; ++i) {
        out_rowids[i] = sc[i].rowid;
        out_scores[i] = sc[i].sim;
    }
    *out_count = cnt;
    free(sc);
    return 0;
}

typedef struct {
    float dist;
    int64_t rowid;
} distrow;

static int cmp_dist(const void* pa, const void* pb) {
    const distrow* a = (const distrow*)pa;
    const distrow* b = (const distrow*)pb;
    if (a->dist < b->dist) return -1;
    if (a->dist > b->dist) return 1;
    return (a->rowid > b->rowid) - (a->rowid < b->rowid);
}

int yo_vec0_exact(const float* rows, size_t n, size_t d, const int64_t* rowids, const float* query,
                  size_t k, int use_range, int64_t rowid_lo, int64_t rowid_hi, int64_t* out_rowids,
                  float* out_dist, size_t* out_count) {
    /* sqlite/vec0_module.hpp:393-428 */
    distrow* res = (distrow*)malloc((n ? n : 1) * sizeof(distrow));
    size_t cnt = 0;
    for (size_t r = 0; r < n; ++r) {
        int64_t rid = rowids ? rowids[r] : (int64_t)r;
        if (use_range && (rid < rowid_lo || rid > rowid_hi)) continue; /* :399-401 */
        res[cnt].dist = yo_l2_distance_f32(query, rows + r * d, d);    /* :411-413 */
        res[cnt].rowid = rid;
        ++cnt;
    }
    qsort(res, cnt, sizeof(distrow), cmp_dist); /* :424-425 */
    if (k && cnt > k) cnt = k;                  /* :426-428 */
    for (size_t i = 0; i < cnt; ++i) {
        out_rowids[i] = res[i].rowid;
        out_dist[i] = res[i].dist;
    }
    *out_count = cnt;
    free(res);
    return 0;
}

void yo_exact_scan_l2_batch(const void* rows, int dtype, size_t n, size_t d, const float* queries, size_t nq,
                            size_t k, int64_t* out_rowids, float* out_dist, uint32_t* out_counts) {
    static float f16_table[65536];
    static int f16_table_ready = 0;
    if (dtype == YO_DTYPE_F16 && !f16_table_ready) {
        for (uint32_t h = 0; h < 65536; ++h) f16_table[h] = yo_f16_to_float((uint16_t)h);
        f16_table_ready = 1;
    }
    const float* r32 = (const float*)rows;
    const uint16_t* r16 = (const uint16_t*)rows;
    long q;
#pragma omp parallel for schedule(dynamic, 1)
    for (q = 0; q < (long)nq; ++q) {
        const float* qv = queries + (size_t)q * d;
        distrow* res = (distrow*)malloc((n ? n : 1) * sizeof(distrow));
        float* row = (float*)malloc((d ? d : 1) * sizeof(float));
        size_t cnt = 0;
        for (size_t r = 0; r < n; ++r) {
            const float* rv = r32 + r * d;
            if (dtype == YO_DTYPE_F16) {
                for (size_t c = 0; c < d; ++c) row[c] = f16_table[r16[r * d + c]];
                rv = row;
            }
            float dist = yo_l2_distance_build_f32(qv, rv, d);
            if (dist != dist) continue;
            res[cnt].dist = dist;
            res[cnt].rowid = (int64_t)r;
            ++cnt;
        }
        qsort(res, cnt, sizeof(distrow), cmp_dist);
        size_t m = cnt < k ? cnt : k;
        for (size_t i = 0; i < k; ++i) {
            out_rowids[(size_t)q * k + i] = i < m ? res[i].rowid : -1;
            out_dist[(size_t)q * k + i] = i < m ? res[i].dist : INFINITY;
        }
        out_counts[q] = (uint32_t)m;
        free(row);
        free(res);
    }
}

size_t yo_batch_top_k(const float* query, const float* rows, size_t n, size_t d, int metric,
                      size_t k, uint64_t* out_idx, float* out_dist) {
    /* distances/batch.hpp:74-92 */
    distrow* res = (distrow*)malloc((n ? n : 1) * sizeof(distrow));
    for (size_t r = 0; r < n; ++r) {
        res[r].dist = metric == YO_METRIC_COSINE ? yo_cosine_distance_f32(query, rows + r * d, d)
                                                 : yo_l2_distance_f32(query, rows + r * d, d);
        res[r].rowid = (int64_t)r;
    }
    qsort(res, n, sizeof(distrow), cmp_dist);
    size_t m = k < n ? k : n;
    for (size_t i = 0; i < m; ++i) {
        out_idx[i] = (uint64_t)res[i].rowid;
        if (out_dist) out_dist[i] = res[i].dist;
    }
    free(res);
    return m;
}

/* ============================== manifest checksum ========================================= */

static uint32_t crc_text(uint32_t crc, const char* s, size_t n) {
    /* src/manifest/manifest_manager.cpp:711-718 (hash_string): bit-serial reflected CRC-32 step per character */
    for (size_t i = 0; i < n; ++i) {
        crc ^= (uint32_t)(int)s[i];
        for (int b = 0; b < 8; ++b) crc = (crc >> 1) ^ (0xEDB88320u * (crc & 1u));
    }
    return crc;
}

uint32_t yo_manifest_checksum(const uint8_t* file_digest32, uint64_t file_size, const uint8_t* digests,
                              const uint64_t* offsets, const uint64_t* sizes, size_t n) {
    /* ManifestManager::calculateChecksum, src/manifest/manifest_manager.cpp:705-730:
     * fileHash, to_string(fileSize), then per chunk hash, to_string(offset), to_string(size) (ChunkRef::size is uint32) */
    static const char* hexd = "0123456789abcdef";
    char hex[64], num[32];
    uint32_t crc = 0xFFFFFFFFu;
    for (int i = 0; i < 32; ++i) { hex[2 * i] = hexd[file_digest32[i] >> 4]; hex[2 * i + 1] = hexd[file_digest32[i] & 15]; }
    crc = crc_text(crc, hex, 64);
    crc = crc_text(crc, num, (size_t)snprintf(num, sizeof num, "%llu", (unsigned long long)file_size));
    for (size_t c = 0; c < n; ++c) {
        const uint8_t* d = digests + 32 * c;
        for (int i = 0; i < 32; ++i) { hex[2 * i] = hexd[d[i] >> 4]; hex[2 * i + 1] = hexd[d[i] & 15]; }
        crc = crc_text(crc, hex, 64);
        crc = crc_text(crc, num, (size_t)snprintf(num, sizeof num, "%llu", (unsigned long long)offsets[c]));
        crc = crc_text(crc, num, (size_t)snprintf(num, sizeof num, "%u", (unsigned)(uint32_t)sizes[c]));
    }
    return ~crc;
}

/* ============================== synthetic inputs ========================================== */

uint64_t yo_splitmix64(uint64_t x) {
    x += 0x9E3779B97F4A7C15ULL;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ULL;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBULL;
    return x ^ (x >> 31);
}

void yo_gen_bytes(uint64_t seed, uint64_t start, size_t n, uint8_t* out) {
    for (size_t j = 0; j < n; ++j) {
        uint64_t i = start + j;
        out[j] = (uint8_t)((yo_splitmix64(seed ^ (i >> 3)) >> (8 * (i & 7))) & 0xFF);
    }
}

void yo_gen_rows_f32(uint64_t seed, uint64_t first_row, size_t n, size_t d, float* out) {
    long r;
#pragma omp parallel for schedule(static)
    for (r = 0; r < (long)n; ++r) {
        uint64_t row = first_row + (uint64_t)r;
        float* o = out + (size_t)r * d;
        double ss = 0.0;
        for (size_t c = 0; c < d; ++c) {
            uint64_t u = yo_splitmix64(seed ^ (row * (uint64_t)d + (uint64_t)c));
            float x = (float)(u >> 40) * 1.1920928955078125e-07f - 1.0f; /* 2^-23 */
            o[c] = x;
            ss += (double)x * (double)x;
        }
        float inv = ss > 0.0 ? (float)(1.0 / sqrt(ss)) : 0.0f;
        for (size_t c = 0; c < d; ++c) o[c] = o[c] * inv;
    }
}

/* Batch form used by bench.py's cpu_baseline / --impl reference legs: Q independent queries,
 * OpenMP over queries (the reference runs a sequential for-loop over queries,
 * sqlite_vec_backend.cpp:4531-4546; threads here model `num_threads` of searchSimilarBatch). */
int yo_exact_scan_cosine_batch(const void* rows, int dtype, size_t n, size_t d,
                               const float* queries, size_t nq, size_t k, float threshold,
                               int64_t* out_rowids, float* out_scores, uint32_t* out_counts) {
    int rc_any = 0;
    long q;
#pragma omp parallel for schedule(dynamic, 1)
    for (q = 0; q < (long)nq; ++q) {
        size_t cnt = 0;
        int rc = yo_exact_scan_cosine(rows, dtype, n, d, NULL, NULL, queries + (size_t)q * d, k,
                                      threshold, NULL, 0, 0, out_rowids + (size_t)q * k,
                                      out_scores + (size_t)q * k, &cnt);
        out_counts[q] = (uint32_t)cnt;
        if (rc) {
#pragma omp atomic write
            rc_any = rc;
        }
    }
    return rc_any;
}
