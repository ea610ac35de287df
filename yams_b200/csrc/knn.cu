// knn.cu -- exact brute-force vector scan: CUDA-core stage-1 engine, top-K' selection, fp64
// rescoring, final ordering, L2 / vec0 surface, corpus mirror and the vector_scan_v1 entry points.
//
// Reference semantics matched (paths under /root/reference):
//   bruteForceSearchUnlocked fast path   src/vector/sqlite_vec_backend.cpp:4203-4331
//   isFinite / isZeroNorm query checks   src/vector/sqlite_vec_backend.cpp:204-235, 4127-4130
//   vec0_run_exact_query                 third_party/sqlite-vec-cpp/.../sqlite/vec0_module.hpp:376-430
//   float16_t::from_float (truncating)   third_party/sqlite-vec-cpp/.../utils/float16.hpp:20-40
//
// Pipeline (DESIGN.md §scan):
//   stage 1  approximate fp32/fp16 scores of every row against every query (GEMM-shaped; this file
//            holds the CUDA-core engine, knn_umma.cu the tcgen05 engine) with a fused per-query
//            threshold filter -> short candidate lists; thresholds come from a strided row sample;
//   select   exact top-K' (K' = k + slack) of each candidate list (radix select + bitonic sort);
//   stage 2  the K' survivors are re-scored exactly like the reference (sequential double
//            accumulation, skip rules, float cast) -> scores are bit-identical to the CPU path;
//   final    order by (similarity desc, rowid asc), apply the threshold, keep k, flag ties at k.
#include <cuda_fp16.h>
#include <math.h>

#include <algorithm>
#include <new>
#include <vector>

#include "knn.cuh"
#include "ref_order.cuh"

namespace yb {

// ---------------------------------------------------------------------------------------------------
// element helpers
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ float load_elem(const void* rows, int dtype, uint64_t idx) {
    if (dtype == YAMS_B200_F16) return __half2float(reinterpret_cast<const __half*>(rows)[idx]);
    return reinterpret_cast<const float*>(rows)[idx];
}

// reference truncating fp32 -> fp16 (utils/float16.hpp:20-40), restated on integer bits
__host__ __device__ __forceinline__ uint16_t f16_from_float_trunc(float f) {
    uint32_t x;
#if defined(__CUDA_ARCH__)
    x = __float_as_uint(f);
#else
    memcpy(&x, &f, 4);
#endif
    uint32_t sign = (x >> 16) & 0x8000u;
    int32_t e = (int32_t)((x >> 23) & 0xFFu) - 127 + 15;
    uint32_t m = x & 0x7FFFFFu;
    if (e <= 0) {
        if (e < -10) return (uint16_t)sign;
        m = (m | 0x800000u) >> (1 - e);
        return (uint16_t)(sign | (m >> 13));
    }
    if (e >= 31) return (uint16_t)(sign | 0x7C00u);
    return (uint16_t)(sign | ((uint32_t)e << 10) | (m >> 13));
}

__global__ void convert_f32_to_f16_trunc_kernel(const float* __restrict__ in, uint16_t* __restrict__ out, uint64_t n) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
        out[i] = f16_from_float_trunc(in[i]);
}

// SURVEY.md §8d generator: x = (splitmix64(seed ^ (row*d + c)) >> 40) * 2^-23 - 1
__device__ __forceinline__ float synth_value(uint64_t seed, uint64_t row, uint32_t d, uint32_t c) {
    uint64_t u = splitmix64(seed ^ (row * (uint64_t)d + (uint64_t)c));
    return (float)(u >> 40) * 1.1920928955078125e-07f - 1.0f;
}

// one thread per row: sequential double sum of squares (bit-identical to oracle yo_gen_rows_f32)
__global__ void synth_rownorm_kernel(uint64_t seed, uint64_t first_row, uint64_t n, uint32_t d, float* __restrict__ inv) {
    uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    double ss = 0.0;
    for (uint32_t c = 0; c < d; ++c) {
        float x = synth_value(seed, first_row + r, d, c);
        ss += (double)x * (double)x;
    }
    inv[r] = ss > 0.0 ? (float)(1.0 / sqrt(ss)) : 0.0f;
}

__global__ void synth_fill_kernel(uint64_t seed, uint64_t first_row, uint64_t n, uint32_t d, const float* __restrict__ inv,
                                  void* __restrict__ out, int dtype) {
    uint64_t total = n * (uint64_t)d;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t r = i / d;
        uint32_t c = (uint32_t)(i - r * d);
        float v = synth_value(seed, first_row + r, d, c) * inv[r];
        if (dtype == YAMS_B200_F16) reinterpret_cast<uint16_t*>(out)[i] = f16_from_float_trunc(v);
        else reinterpret_cast<float*>(out)[i] = v;
    }
}

// nonnegative floats order like their bit patterns: atomic max through the integer view
__device__ __forceinline__ void atomic_max_nonneg(float* addr, float v) {
    if (v == v) atomicMax(reinterpret_cast<unsigned int*>(addr), __float_as_uint(v));
}

// per-row validity + 1/|row| exactly as the reference evaluates it (sqlite_vec_backend.cpp:4253-4269):
// sequential double accumulation; rows with a non-finite element or |row|^2 <= 1e-12 get 0.
// L2 corpora (vec0 surface, no skip rules) keep |row|^2 in the same slot instead: stage 1 ranks by 2 q.r - |row|^2.
// stats[0] = max |row|, stats[1] = max |row - tf32(row)| (fp32 corpora read by the tf32 tensor-core engine),
// stats[2] = max of that residual relative to |row|: the inputs of the stage-1 error bound (DESIGN.md §4.2)
__global__ void row_stats_kernel(const void* __restrict__ rows, int dtype, uint32_t d, uint64_t first, uint64_t n,
                                 float* __restrict__ inv_norm, int metric, float* __restrict__ stats) {
    uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    uint64_t base = (first + r) * (uint64_t)d;
    double ss = 0.0, res = 0.0;
    bool finite = true;
    for (uint32_t c = 0; c < d; ++c) {
        float v = load_elem(rows, dtype, base + c);
        if (!isfinite(v)) { finite = false; break; }
        ss += (double)v * (double)v;
        if (dtype == YAMS_B200_F32) {
            float t = v - __uint_as_float(__float_as_uint(v) & 0xFFFFE000u);
            res += (double)t * (double)t;
        }
    }
    if (metric == YAMS_B200_L2) inv_norm[first + r] = finite ? (float)ss : INFINITY;
    else inv_norm[first + r] = (finite && ss > 1e-12) ? (float)(1.0 / sqrt(ss)) : 0.0f;
    if (finite && ss > 0.0) {
        float nrm = (float)sqrt(ss), rs = (float)sqrt(res);
        atomic_max_nonneg(&stats[0], nrm * 1.0000002f);
        atomic_max_nonneg(&stats[1], rs * 1.0000002f);
        if (ss > 1e-12) atomic_max_nonneg(&stats[2], (rs / nrm) * 1.0000002f);
    }
}

// Device-side status of one search call (read by the host once, after everything is enqueued)
struct ScanStatus {
    uint32_t n_invalid;   // queries the reference rejects (non-finite or zero norm, sqlite_vec_backend.cpp:4127-4130)
    uint32_t n_bad;       // queries whose fast-path result could not be certified exact -> resolved by the exhaustive levels
    uint32_t n_bad2;      // ... of which level 1 could not certify either -> full exact pass
    uint32_t pad;
    // followed by uint32_t bad[nq], bad2[nq]
};

// queries: invalid if non-finite or (cosine) |q|^2 < 1e-10 (sqlite_vec_backend.cpp:204-235,4127);
// qnorm[q] = sqrt(sum (double)q^2) (:4204-4209), qinv[q] = 1/qnorm as float (1 for L2: queries stay unscaled)
constexpr int QP_THREADS = 32;
__global__ void __launch_bounds__(QP_THREADS) query_prep_kernel(const float* __restrict__ q, uint32_t nq, uint32_t d, double* __restrict__ qnorm,
                                                                float* __restrict__ qinv, int metric, ScanStatus* __restrict__ status) {
    // thread = query, the reference's sequential double sum (sqlite_vec_backend.cpp:4140-4150).  The row is read with 16-byte
    // loads, four in flight (one 4-byte load per dependent trip cost 64 us for 1024 x 768 queries).
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nq) return;
    const float* row = q + (uint64_t)i * d;
    double ss = 0.0;
    bool finite = true;
    auto add = [&](float v) {
        if (!isfinite(v)) finite = false;
        ss += (double)v * (double)v;
    };
    uint32_t c = 0;
    if ((reinterpret_cast<uintptr_t>(row) & 15u) == 0) {
        const float4* r4 = reinterpret_cast<const float4*>(row);
        const uint32_t n4 = d / 4;
        uint32_t j = 0;
        for (; j + 4 <= n4; j += 4) {
            const float4 a0 = r4[j], a1 = r4[j + 1], a2 = r4[j + 2], a3 = r4[j + 3];
            add(a0.x); add(a0.y); add(a0.z); add(a0.w);
            add(a1.x); add(a1.y); add(a1.z); add(a1.w);
            add(a2.x); add(a2.y); add(a2.z); add(a2.w);
            add(a3.x); add(a3.y); add(a3.z); add(a3.w);
        }
        for (; j < n4; ++j) {
            const float4 a0 = r4[j];
            add(a0.x); add(a0.y); add(a0.z); add(a0.w);
        }
        c = n4 * 4;
    }
    for (; c < d; ++c) add(row[c]);
    bool bad = !finite || (metric == YAMS_B200_COSINE && ss < 1e-10);
    if (bad) atomicAdd(&status->n_invalid, 1u);
    double nrm = sqrt(ss);
    qnorm[i] = nrm;
    qinv[i] = metric == YAMS_B200_L2 ? 1.0f : (bad ? 0.0f : (float)(1.0 / nrm));
}

// error bound of the CUDA-core engine's stage-1 score (fp32 FMA chain over d products, Cauchy-Schwarz on sum |q_i r_i|;
// the float roundings of 1/|row|, 1/|q| or |row|^2 are covered by the +4):
//   cosine: |s~ - s| <= 2^-24 (d + 4);   L2 (s = 2 q.r - |r|^2): <= 2^-23 (d + 4) |q| Rmax + 2^-22 Rmax^2
__global__ void eps_cc_kernel(const double* __restrict__ qnorm, uint32_t nq, uint32_t d, int metric, float r_max,
                              float* __restrict__ eps, int keep_larger) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nq) return;
    const float u = 5.9604645e-08f;   // 2^-24
    float e;
    if (metric == YAMS_B200_L2) e = 2.f * u * (float)(d + 4) * (float)qnorm[i] * r_max + 4.f * u * r_max * r_max + 1e-30f;
    else e = u * (float)(d + 4) + 1e-7f;
    eps[i] = keep_larger ? fmaxf(eps[i], e) : e;
}

// ---------------------------------------------------------------------------------------------------
// stage 1, CUDA-core engine: tiled fp32 GEMM [rows x dim] x [dim x queries] with fused epilogue
// ---------------------------------------------------------------------------------------------------
constexpr int CC_BM = 128, CC_BN = 64, CC_BK = 32, CC_THREADS = 256;
constexpr int CC_AS = CC_BM + 1;  // padded k-major A tile: conflict-free transposed stores

template <bool FILTER>
__global__ void __launch_bounds__(CC_THREADS, 2) stage1_cc_kernel(Stage1Args a, uint32_t nqt) {
    __shared__ float As[CC_BK][CC_AS];
    __shared__ __align__(16) float Bs[CC_BK][CC_BN];
    const uint32_t qt = blockIdx.x % nqt;
    const uint64_t rt = blockIdx.x / nqt;
    const uint64_t row0 = rt * CC_BM;   // tile-local row index base (within this launch)
    const uint32_t q0 = qt * CC_BN;
    const int tid = threadIdx.x;
    const int ty = tid >> 4, tx = tid & 15;
    float acc[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

    const bool vec_ok = a.dtype == YAMS_B200_F16 ? (a.dim % 8 == 0) : (a.dim % 4 == 0);
    for (uint32_t k0 = 0; k0 < a.dim; k0 += CC_BK) {
        // ---- A tile: CC_BM rows x CC_BK k, transposed into As[k][m] ----
        if (a.dtype == YAMS_B200_F16) {
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                int idx = tid + CC_THREADS * j;  // 512 segments of 8 halves
                int m = idx >> 2, seg = idx & 3;
                uint64_t li = row0 + m;
                uint32_t kk = k0 + seg * 8;
                float v[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) v[e] = 0.f;
                if (li < a.nrows) {
                    uint64_t grow = a.row_start + li * a.row_stride;
                    const __half* src = reinterpret_cast<const __half*>(a.rows) + grow * a.dim + kk;
                    if (vec_ok && kk + 8 <= a.dim) {
                        uint4 raw = *reinterpret_cast<const uint4*>(src);
                        const __half2* h2 = reinterpret_cast<const __half2*>(&raw);
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            float2 f = __half22float2(h2[e]);
                            v[2 * e] = f.x;
                            v[2 * e + 1] = f.y;
                        }
                    } else {
#pragma unroll
                        for (int e = 0; e < 8; ++e)
                            if (kk + e < a.dim) v[e] = __half2float(src[e]);
                    }
                }
#pragma unroll
                for (int e = 0; e < 8; ++e) As[seg * 8 + e][m] = v[e];
            }
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                int idx = tid + CC_THREADS * j;  // 1024 segments of 4 floats
                int m = idx >> 3, seg = idx & 7;
                uint64_t li = row0 + m;
                uint32_t kk = k0 + seg * 4;
                float v[4] = {0.f, 0.f, 0.f, 0.f};
                if (li < a.nrows) {
                    uint64_t grow = a.row_start + li * a.row_stride;
                    const float* src = reinterpret_cast<const float*>(a.rows) + grow * a.dim + kk;
                    if (vec_ok && kk + 4 <= a.dim) {
                        float4 f = *reinterpret_cast<const float4*>(src);
                        v[0] = f.x; v[1] = f.y; v[2] = f.z; v[3] = f.w;
                    } else {
#pragma unroll
                        for (int e = 0; e < 4; ++e)
                            if (kk + e < a.dim) v[e] = src[e];
                    }
                }
#pragma unroll
                for (int e = 0; e < 4; ++e) As[seg * 4 + e][m] = v[e];
            }
        }
        // ---- B tile: CC_BK k x CC_BN queries (queries are row-major [q][dim]) ----
#pragma unroll
        for (int j = 0; j < (CC_BK * CC_BN) / CC_THREADS; ++j) {
            int idx = tid + CC_THREADS * j;
            int kk = idx & (CC_BK - 1), qn = idx / CC_BK;
            uint32_t q = q0 + qn, k = k0 + kk;
            Bs[kk][qn] = (q < a.nq && k < a.dim) ? a.q32[(uint64_t)q * a.dim + k] : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < CC_BK; ++kk) {
            float av[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) av[i] = As[kk][ty * 8 + i];
            float4 b4 = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
            float bv[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        __syncthreads();
    }
    // ---- epilogue ----
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        uint64_t li = row0 + ty * 8 + i;
        if (li >= a.nrows) continue;
        uint64_t grow = a.row_start + li * a.row_stride;
        float inr = a.inv_norm[grow];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            uint32_t q = q0 + tx * 4 + j;
            if (q >= a.nq) continue;
            float s;
            if (a.metric == YAMS_B200_L2) s = fmaf(2.f, acc[i][j], -inr);           // 2 q.r - |r|^2 (slot holds |r|^2)
            else s = inr > 0.f ? acc[i][j] * inr * a.qinv[q] : -INFINITY;
            if (FILTER) {
                bool pass = s > a.tau[q];
                if (pass && a.mask) pass = (a.mask[(uint64_t)q * a.mask_ld + (grow >> 5)] >> (grow & 31)) & 1u;
                if (pass) {
                    uint32_t pos = atomicAdd(&a.counts[q], 1u);
                    if (pos < a.cap) {
                        Cand c;
                        c.score = s;
                        c.row = (uint32_t)grow;
                        a.cands[(uint64_t)q * a.cap + pos] = c;
                    }
                }
            } else {
                a.out_scores[(uint64_t)q * a.ld + li] = s;
            }
        }
    }
}

yams_status_t stage1_cuda_core(const Stage1Args& a, bool filter, cudaStream_t st) {
    if (a.nrows == 0 || a.nq == 0) return YAMS_OK;
    uint32_t nqt = (a.nq + CC_BN - 1) / CC_BN;
    uint64_t nrt = (a.nrows + CC_BM - 1) / CC_BM;
    uint64_t grid = nrt * nqt;
    YB_ARG(grid < (1ull << 31), "scan too large for one launch");
    if (filter) stage1_cc_kernel<true><<<(unsigned)grid, CC_THREADS, 0, st>>>(a, nqt);
    else stage1_cc_kernel<false><<<(unsigned)grid, CC_THREADS, 0, st>>>(a, nqt);
    YB_CUDA(cudaGetLastError());
    return YAMS_OK;
}

// ---------------------------------------------------------------------------------------------------
// top-K selection (one CTA per query): radix select on monotone keys, gather, bitonic sort
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t fkey(float f) {
    if (f != f) return 0u;  // NaN ranks last
    uint32_t b = __float_as_uint(f);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float fkey_inv(uint32_t k) {
    uint32_t b = (k & 0x80000000u) ? (k & 0x7FFFFFFFu) : ~k;
    return __uint_as_float(b);
}

constexpr int SEL_THREADS = 256;
constexpr int SEL_MAXK = 4096;       // survivors per query the select / final kernels can order in shared memory

struct SelectIn {
    const float* dense;     // mode dense: scores[q * ld + i], row = row_start + i * row_stride
    uint64_t ld;
    uint64_t row_start, row_stride;
    uint64_t dense_len;
    const Cand* cands;      // mode list: cands[q * cap + i], length min(counts[q], cap)
    const uint32_t* counts;
    uint32_t cap;
    const uint32_t* qmap;   // nullable: CTA b handles query qmap[b] for the list/out side
    const float* tau;       // nullable (list mode): rows that never reached the list scored <= tau[q]
    float tau_margin;       // tau_only: subtracted from the selected score
    int fast_tau;           // tau_only, K <= 16: one pass, the K-th largest of the per-thread maxima (a lower bound of the K-th
                            // largest score: a threshold need not be exact, only close -- the certificate covers what it lets go)
};

__device__ __forceinline__ uint64_t sel_key(const SelectIn& in, uint32_t qsrc, uint64_t i) {
    float s;
    uint32_t row;
    if (in.dense) {
        s = in.dense[(uint64_t)qsrc * in.ld + i];
        row = (uint32_t)(in.row_start + i * in.row_stride);
    } else {
        Cand c = in.cands[(uint64_t)qsrc * in.cap + i];
        s = c.score;
        row = c.row;
    }
    return ((uint64_t)fkey(s) << 32) | (uint64_t)(0xFFFFFFFFu - row);
}

// tau_only: writes the K-th largest score to out_tau[q] (-inf when fewer than K items)
// else    : writes the top-K (sorted desc; ties -> smaller row first) to out_sel[b*K ..], count to out_n[b], and
//           out_bound[b] = an upper bound of the stage-1 score of every row that was NOT selected (the input of the
//           exactness certificate in final_kernel): the K-th selected score when the list was longer than K, else the
//           list threshold tau (rows that never reached the list), -inf when no other row exists, +inf when the list
//           overflowed its capacity (unknown rows were dropped)
__global__ void __launch_bounds__(SEL_THREADS) topk_select_kernel(SelectIn in, uint32_t K, int tau_only, float* __restrict__ out_tau,
                                                                  Cand* __restrict__ out_sel, uint32_t* __restrict__ out_n,
                                                                  float* __restrict__ out_bound) {
    __shared__ uint32_t hist[256];
    __shared__ uint64_t s_prefix;
    __shared__ uint32_t s_want;
    __shared__ uint32_t s_cnt;
    __shared__ uint64_t buf[SEL_MAXK];
    const uint32_t b = blockIdx.x;
    const uint32_t qdst = in.qmap ? in.qmap[b] : b;   // tau_only output slot / list-side query
    const uint32_t qsrc = in.dense ? b : qdst;
    uint64_t L = in.dense ? in.dense_len : (uint64_t)min(in.counts[qsrc], in.cap);
    // radix select of the K-th largest key among L > K items; result in s_prefix
    auto radix_select = [&](int npass) {
        if (threadIdx.x == 0) { s_prefix = 0; s_want = K; }
        __syncthreads();
        for (int p = 0; p < npass; ++p) {
            const int shift = 56 - 8 * p;
            for (int i = threadIdx.x; i < 256; i += SEL_THREADS) hist[i] = 0;
            __syncthreads();
            const uint64_t prefix = s_prefix;
            for (uint64_t i = threadIdx.x; i < L; i += SEL_THREADS) {
                uint64_t key = sel_key(in, qsrc, i);
                if (p == 0 || (key >> (shift + 8)) == prefix) atomicAdd(&hist[(key >> shift) & 255u], 1u);
            }
            __syncthreads();
            if (threadIdx.x == 0) {
                uint32_t want = s_want, cum = 0;
                int bsel = 0;
                for (int bk = 255; bk >= 0; --bk) {
                    uint32_t h = hist[bk];
                    if (cum + h >= want) { bsel = bk; break; }
                    cum += h;
                }
                s_want = want - cum;
                s_prefix = (prefix << 8) | (uint64_t)bsel;
            }
            __syncthreads();
        }
    };
    if (tau_only) {
        if (L < K || K == 0) {
            if (threadIdx.x == 0) out_tau[qdst] = -INFINITY;
        } else if (L == K) {
            if (threadIdx.x == 0) s_want = 0xFFFFFFFFu;
            __syncthreads();
            uint32_t mn = 0xFFFFFFFFu;
            for (uint64_t i = threadIdx.x; i < L; i += SEL_THREADS) mn = min(mn, (uint32_t)(sel_key(in, qsrc, i) >> 32));
            atomicMin(&s_want, mn);
            __syncthreads();
            if (threadIdx.x == 0) out_tau[qdst] = fkey_inv(s_want) - in.tau_margin;
        } else if (in.fast_tau && K <= 16 && L >= 16 * SEL_THREADS) {
            // One pass, no atomics: every thread keeps the best key of its strided share, the 256 maxima are sorted, the K-th of
            // them is the threshold.  It equals the K-th best score unless two of the top K fall into one thread's share (11 % for
            // K = 8), in which case it is the next one down: a slightly lower threshold, a few more survivors.
            uint32_t* arr = reinterpret_cast<uint32_t*>(buf);
            uint32_t mx = 0;
            const float* base = in.dense ? in.dense + (uint64_t)qsrc * in.ld : nullptr;
            if (base && (reinterpret_cast<uintptr_t>(base) & 15u) == 0) {
                // dense scores: 16-byte loads, four of them in flight per thread (one 4-byte load per trip was latency-bound:
                // 1.2 TB/s over the Q x S score matrix)
                const float4* b4 = reinterpret_cast<const float4*>(base);
                const uint64_t n4 = L / 4;
                uint64_t i = threadIdx.x;
                for (; i + 3 * SEL_THREADS < n4; i += 4 * SEL_THREADS) {
                    const float4 v0 = b4[i], v1 = b4[i + SEL_THREADS], v2 = b4[i + 2 * SEL_THREADS], v3 = b4[i + 3 * SEL_THREADS];
                    mx = max(mx, max(max(fkey(v0.x), fkey(v0.y)), max(fkey(v0.z), fkey(v0.w))));
                    mx = max(mx, max(max(fkey(v1.x), fkey(v1.y)), max(fkey(v1.z), fkey(v1.w))));
                    mx = max(mx, max(max(fkey(v2.x), fkey(v2.y)), max(fkey(v2.z), fkey(v2.w))));
                    mx = max(mx, max(max(fkey(v3.x), fkey(v3.y)), max(fkey(v3.z), fkey(v3.w))));
                }
                for (; i < n4; i += SEL_THREADS) {
                    const float4 v = b4[i];
                    mx = max(mx, max(max(fkey(v.x), fkey(v.y)), max(fkey(v.z), fkey(v.w))));
                }
                for (uint64_t j = n4 * 4 + threadIdx.x; j < L; j += SEL_THREADS) mx = max(mx, fkey(base[j]));
            } else {
                for (uint64_t i = threadIdx.x; i < L; i += SEL_THREADS) mx = max(mx, (uint32_t)(sel_key(in, qsrc, i) >> 32));
            }
            arr[threadIdx.x] = mx;
            __syncthreads();
            for (uint32_t size = 2; size <= SEL_THREADS; size <<= 1) {
                for (uint32_t stride = size >> 1; stride > 0; stride >>= 1) {
                    const uint32_t t = threadIdx.x;
                    if (t < SEL_THREADS / 2) {
                        uint32_t lo = (t / stride) * (stride * 2) + (t % stride), hi = lo + stride;
                        bool desc = ((lo & size) == 0);
                        uint32_t x = arr[lo], y = arr[hi];
                        if ((x < y) == desc) { arr[lo] = y; arr[hi] = x; }
                    }
                    __syncthreads();
                }
            }
            if (threadIdx.x == 0) out_tau[qdst] = fkey_inv(arr[K - 1]) - in.tau_margin;
        } else {
            // Two passes instead of four: a 4096-bin histogram of the top 12 key bits locates the bin that holds the K-th
            // best score; its (few) members are collected and sorted in shared memory.  A crowded bin (> 2048 members,
            // e.g. constant scores) falls back to the plain 4-pass radix select.
            uint32_t* h12 = reinterpret_cast<uint32_t*>(buf);            // [4096] counters
            uint32_t* members = h12 + 4096;                               // [4096] score keys of the boundary bin
            for (int i = threadIdx.x; i < 4096; i += SEL_THREADS) h12[i] = 0;
            __syncthreads();
            for (uint64_t i = threadIdx.x; i < L; i += SEL_THREADS) atomicAdd(&h12[(uint32_t)(sel_key(in, qsrc, i) >> 52)], 1u);
            __syncthreads();
            if (threadIdx.x == 0) {
                uint32_t cum = 0;
                int bsel = 0;
                for (int bk = 4095; bk >= 0; --bk) {
                    uint32_t h = h12[bk];
                    if (cum + h >= K) { bsel = bk; break; }
                    cum += h;
                }
                s_want = K - cum;               // rank inside the boundary bin (1-based)
                s_prefix = (uint64_t)bsel;
                s_cnt = 0;
            }
            __syncthreads();
            const uint32_t bsel = (uint32_t)s_prefix, pop = h12[bsel];
            if (pop <= 2048) {
                uint32_t np2 = 1;
                while (np2 < pop) np2 <<= 1;
                __syncthreads();
                for (uint32_t i = threadIdx.x; i < np2; i += SEL_THREADS) members[i] = 0;
                __syncthreads();
                for (uint64_t i = threadIdx.x; i < L; i += SEL_THREADS) {
                    uint32_t fk = (uint32_t)(sel_key(in, qsrc, i) >> 32);
                    if ((fk >> 20) == bsel) members[atomicAdd(&s_cnt, 1u)] = fk;
                }
                __syncthreads();
                for (uint32_t size = 2; size <= np2; size <<= 1) {
                    for (uint32_t stride = size >> 1; stride > 0; stride >>= 1) {
                        for (uint32_t t = threadIdx.x; t < np2 / 2; t += SEL_THREADS) {
                            uint32_t lo = (t / stride) * (stride * 2) + (t % stride), hi = lo + stride;
                            bool desc = ((lo & size) == 0);
                            uint32_t x = members[lo], y = members[hi];
                            if ((x < y) == desc) { members[lo] = y; members[hi] = x; }
                        }
                        __syncthreads();
                    }
                }
                if (threadIdx.x == 0) out_tau[qdst] = fkey_inv(members[s_want - 1]) - in.tau_margin;
            } else {
                __syncthreads();
                radix_select(4);
                if (threadIdx.x == 0) out_tau[qdst] = fkey_inv((uint32_t)s_prefix) - in.tau_margin;
            }
        }
        return;
    }
    uint64_t kth = 0;  // keys >= kth are selected
    constexpr int KPT = SEL_MAXK / SEL_THREADS;   // 16 keys per thread
    if (L <= SEL_MAXK) {
        // The normal case (a candidate list of 1-3 k entries): the keys are read ONCE into registers and the K-th largest is found
        // bit by bit from the top -- 64 block-wide counts (compare, warp reduce, one barrier each), ~8 k cycles, where eight
        // histogram passes over the list or a 4096-key sorting network cost 150-300 us per 1024 queries.
        uint64_t kreg[KPT];
#pragma unroll
        for (int j = 0; j < KPT; ++j) {
            const uint64_t i = (uint64_t)threadIdx.x + (uint64_t)j * SEL_THREADS;
            kreg[j] = i < L ? sel_key(in, qsrc, i) : 0ull;          // 0 is no key (a real key carries 0xFFFFFFFF - row != 0 below)
        }
        if (L > K && K > 0) {
            // Block-wide helpers over 8 warps: one barrier per call, partials double-buffered by `slot`.
            uint32_t* part = reinterpret_cast<uint32_t*>(hist);      // [4][8]
            int slot = 0;
            auto block_sum = [&](uint32_t v) {
                const uint32_t w = __reduce_add_sync(0xffffffffu, v);
                uint32_t* pb = part + (slot & 3) * 8;
                ++slot;
                if ((threadIdx.x & 31) == 0) pb[threadIdx.x >> 5] = w;
                __syncthreads();
                uint32_t t = 0;
#pragma unroll
                for (int x = 0; x < SEL_THREADS / 32; ++x) t += pb[x];
                return t;
            };
            // score words first (32-bit compares); the bits every valid key shares are skipped
            uint32_t a_and = 0xFFFFFFFFu, a_or = 0u;
#pragma unroll
            for (int j = 0; j < KPT; ++j)
                if (kreg[j] != 0ull) { a_and &= (uint32_t)(kreg[j] >> 32); a_or |= (uint32_t)(kreg[j] >> 32); }
            {
                const uint32_t wa = __reduce_and_sync(0xffffffffu, a_and), wo = __reduce_or_sync(0xffffffffu, a_or);
                uint32_t* pb = part + 16;                              // slots 2,3 of the table: [8] ands, [8] ors
                if ((threadIdx.x & 31) == 0) { pb[threadIdx.x >> 5] = wa; pb[8 + (threadIdx.x >> 5)] = wo; }
                __syncthreads();
                a_and = 0xFFFFFFFFu; a_or = 0u;
#pragma unroll
                for (int x = 0; x < SEL_THREADS / 32; ++x) { a_and &= pb[x]; a_or |= pb[8 + x]; }
                __syncthreads();                                       // the table is reused by block_sum below
            }
            const uint32_t diff = a_and ^ a_or;
            uint32_t want = K;
            uint32_t shi = a_or;                                       // all scores equal: that score
            if (diff) {
                const int top = 31 - __clz(diff);
                shi = top == 31 ? 0u : (a_or & ~((2u << top) - 1u));   // the shared leading bits
                for (int bit = top; bit >= 0; --bit) {
                    const uint32_t cand = shi | (1u << bit);
                    const uint32_t himask = ~((1u << bit) - 1u);
                    uint32_t c = 0;
#pragma unroll
                    for (int j = 0; j < KPT; ++j) c += (kreg[j] != 0ull && ((uint32_t)(kreg[j] >> 32) & himask) == cand) ? 1u : 0u;
                    const uint32_t tot = block_sum(c);
                    if (tot >= want) shi = cand; else want -= tot;    // block-uniform
                }
            }
            // `want` of the keys whose score word equals shi are needed (those with the largest low words, i.e. the smallest rows)
            uint32_t g = 0;
#pragma unroll
            for (int j = 0; j < KPT; ++j) g += (kreg[j] != 0ull && (uint32_t)(kreg[j] >> 32) == shi) ? 1u : 0u;
            const uint32_t group = block_sum(g);
            uint32_t slo = 0;                                          // group == want: the whole group is selected
            if (group > want) {                                        // equal scores straddle the K-th place: resolve by the low words
                for (int bit = 31; bit >= 0; --bit) {
                    const uint32_t cand = slo | (1u << bit);
                    const uint32_t lomask = ~((1u << bit) - 1u);
                    uint32_t c = 0;
#pragma unroll
                    for (int j = 0; j < KPT; ++j)
                        c += (kreg[j] != 0ull && (uint32_t)(kreg[j] >> 32) == shi && ((uint32_t)kreg[j] & lomask) == cand) ? 1u : 0u;
                    const uint32_t tot = block_sum(c);
                    if (tot >= want) slo = cand; else want -= tot;
                }
            }
            kth = ((uint64_t)shi << 32) | (uint64_t)slo;
        }
        if (threadIdx.x == 0) s_cnt = 0;
        for (int i = threadIdx.x; i < SEL_MAXK; i += SEL_THREADS) buf[i] = 0;
        __syncthreads();
#pragma unroll
        for (int j = 0; j < KPT; ++j) {
            if (kreg[j] != 0ull && kreg[j] >= kth) {
                uint32_t pos = atomicAdd(&s_cnt, 1u);
                if (pos < SEL_MAXK) buf[pos] = kreg[j];
            }
        }
        __syncthreads();
    } else {
    if (L > K) {
        radix_select(8);
        kth = s_prefix;
    }
    if (threadIdx.x == 0) s_cnt = 0;
    for (int i = threadIdx.x; i < SEL_MAXK; i += SEL_THREADS) buf[i] = 0;
    __syncthreads();
    for (uint64_t i = threadIdx.x; i < L; i += SEL_THREADS) {
        uint64_t key = sel_key(in, qsrc, i);
        if (key >= kth) {
            uint32_t pos = atomicAdd(&s_cnt, 1u);
            if (pos < SEL_MAXK) buf[pos] = key;
        }
    }
    __syncthreads();
    }
    uint32_t cnt = min(s_cnt, (uint32_t)SEL_MAXK);
    uint32_t np2 = 1;
    while (np2 < cnt) np2 <<= 1;
    // bitonic sort descending on buf[0..np2)
    for (uint32_t size = 2; size <= np2; size <<= 1) {
        for (uint32_t stride = size >> 1; stride > 0; stride >>= 1) {
            for (uint32_t t = threadIdx.x; t < np2 / 2; t += SEL_THREADS) {
                uint32_t lo = (t / stride) * (stride * 2) + (t % stride);
                uint32_t hi = lo + stride;
                bool desc = ((lo & size) == 0);
                uint64_t x = buf[lo], y = buf[hi];
                if ((x < y) == desc) { buf[lo] = y; buf[hi] = x; }
            }
            __syncthreads();
        }
    }
    uint32_t nout = min(cnt, K);
    for (uint32_t i = threadIdx.x; i < nout; i += SEL_THREADS) {
        uint64_t key = buf[i];
        Cand c;
        c.score = fkey_inv((uint32_t)(key >> 32));
        c.row = 0xFFFFFFFFu - (uint32_t)key;
        out_sel[(uint64_t)b * K + i] = c;
    }
    if (threadIdx.x == 0) {
        out_n[b] = nout;
        if (out_bound) {
            float bd;
            if (!in.dense && in.counts[qsrc] > in.cap) bd = INFINITY;
            else if (L > K && K > 0) bd = fkey_inv((uint32_t)(buf[K - 1] >> 32));
            else if (L > K) bd = INFINITY;
            else bd = (!in.dense && in.tau) ? in.tau[qsrc] : -INFINITY;
            out_bound[b] = bd;
        }
    }
}

// ---------------------------------------------------------------------------------------------------
// stage 2: exact re-scoring + final ordering
// ---------------------------------------------------------------------------------------------------
struct Exact {
    float sim;       // reference similarity (float cast of the double quotient); NaN marks "skipped"
    uint32_t row;
};

// one thread per (query, survivor).
// cosine: sqlite_vec_backend.cpp:4253-4279 evaluated in the same order (sequential double accumulation, skip rules, float cast)
// L2    : distances::l2_distance<float> as the reference BUILD evaluates it (YAMS compiles sqlite-vec-cpp with AVX,
//         src/vector/meson.build:79-87): dim >= 16 && dim % 16 == 0 -> simd/avx.hpp:20-66 (eight lane-strided float partial
//         sums, separate multiply and add, lanes summed left to right), else the scalar loop l2.hpp:108-118; sim = -dist.
// Entry b of sel/out belongs to query qmap[b] (or b).
__global__ void rescore_kernel(const void* __restrict__ rows, int dtype, uint32_t d, const float* __restrict__ q32,
                               const double* __restrict__ qnorm, const Cand* __restrict__ sel, const uint32_t* __restrict__ sel_n,
                               uint32_t Kp, uint32_t nq, float threshold, Exact* __restrict__ out, int metric,
                               const uint32_t* __restrict__ qmap, const uint32_t* __restrict__ mask, uint64_t mask_ld) {
    uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (uint64_t)nq * Kp) return;
    uint32_t b = (uint32_t)(t / Kp), j = (uint32_t)(t % Kp);
    const uint32_t q = qmap ? qmap[b] : b;
    Exact e;
    e.sim = __int_as_float(0x7FC00000);
    e.row = 0xFFFFFFFFu;
    bool take = j < sel_n[b] && sel[(uint64_t)b * Kp + j].row != 0xFFFFFFFFu;
    if (take && mask) {   // candidate-set mode: a row outside the allowed set is never a result
        uint32_t row = sel[(uint64_t)b * Kp + j].row;
        take = (mask[(uint64_t)q * mask_ld + (row >> 5)] >> (row & 31)) & 1u;
    }
    if (take) {
        uint32_t row = sel[(uint64_t)b * Kp + j].row;
        uint64_t base = (uint64_t)row * d;
        const float* qv = q32 + (uint64_t)q * d;
        if (metric == YAMS_B200_L2) {
            auto row_at = [&](uint32_t c) { return load_elem(rows, dtype, base + c); };
            auto q_at = [&](uint32_t c) { return qv[c]; };
            float dist = ref_l2_distance(q_at, row_at, d);
            if (dist == dist) {
                e.sim = -dist;
                e.row = row;
            }
        } else {
            double norm_sq = 0.0, dot = 0.0;
            bool finite = true;
            // same element order as the reference's loop; only the loads are widened (16-byte row and query chunks)
            uint32_t c = 0;
            if (dtype == YAMS_B200_F16 && d % 8 == 0) {
                const uint4* rp = reinterpret_cast<const uint4*>(static_cast<const __half*>(rows) + base);
                const float4* qp = reinterpret_cast<const float4*>(qv);
                for (; c < d; c += 8) {
                    const uint4 raw = __ldg(rp + (c >> 3));
                    const float4 q0 = __ldg(qp + (c >> 2)), q1 = __ldg(qp + (c >> 2) + 1);
                    const __half2* h2 = reinterpret_cast<const __half2*>(&raw);
                    const float2 f0 = __half22float2(h2[0]), f1 = __half22float2(h2[1]), f2 = __half22float2(h2[2]), f3 = __half22float2(h2[3]);
                    const float rv[8] = {f0.x, f0.y, f1.x, f1.y, f2.x, f2.y, f3.x, f3.y};
                    const float qq[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
#pragma unroll
                    for (int e = 0; e < 8; ++e) {
                        if (!isfinite(rv[e])) finite = false;
                        const double sv = (double)rv[e];
                        norm_sq += sv * sv;
                        dot += sv * (double)qq[e];
                    }
                }
            } else if (dtype == YAMS_B200_F32 && d % 4 == 0) {
                const float4* rp = reinterpret_cast<const float4*>(static_cast<const float*>(rows) + base);
                const float4* qp = reinterpret_cast<const float4*>(qv);
                for (; c < d; c += 4) {
                    const float4 r4 = __ldg(rp + (c >> 2)), q4 = __ldg(qp + (c >> 2));
                    const float rv[4] = {r4.x, r4.y, r4.z, r4.w};
                    const float qq[4] = {q4.x, q4.y, q4.z, q4.w};
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        if (!isfinite(rv[e])) finite = false;
                        const double sv = (double)rv[e];
                        norm_sq += sv * sv;
                        dot += sv * (double)qq[e];
                    }
                }
            }
            for (; c < d; ++c) {
                float v = load_elem(rows, dtype, base + c);
                if (!isfinite(v)) { finite = false; break; }
                double sv = (double)v, qd = (double)qv[c];
                norm_sq += sv * sv;
                dot += sv * qd;
            }
            if (finite && norm_sq > 1e-12) {
                double denom = sqrt(norm_sq) * qnorm[q];
                double simd = denom > 0.0 ? dot / denom : 0.0;
                if (isfinite(simd)) {
                    float sim = (float)simd;
                    if (!(sim < threshold)) {
                        e.sim = sim;
                        e.row = row;
                    }
                }
            }
        }
    }
    out[(uint64_t)b * Kp + j] = e;
}

// The exactness certificate (DESIGN.md §4.2).  Stage 1 ranks rows by an approximate score s~ with |s~ - s| <= eps[q];
// only the top-K' by s~ are re-scored exactly.  Every row that was NOT re-scored has s~ <= bound (topk_select_kernel), hence
// a true score <= bound + eps.  The emitted top-k is provably the reference's top-k iff no such row can reach the k-th exact
// score (or, with fewer than k valid survivors, the caller's threshold):
//   cosine:  bound + eps <  (valid >= k ? sim_k : threshold)
//   L2    :  (|q|^2 - bound - eps) (1 - g) > dist_k^2   (s~ = 2 q.r - |r|^2, so d^2 = |q|^2 - s; g: l2_rounding_slack)
// Only bound == -inf (no row was left out) skips the test; a NaN bound or eps (stage-1 scores that overflowed) fails it.
// Otherwise the query is queued for the exhaustive levels (status->bad / bad2) and flagged.
struct CertArgs {
    const float* bound;       // per CTA
    const float* eps;         // per query
    const double* qnorm;      // per query (L2)
    float threshold;
    int metric;
    ScanStatus* status;       // nullable: no certificate (results already exhaustive)
    int level;                // 0: failures go to bad[], 1: to bad2[]
    uint32_t nq_total;        // capacity of each list
    uint32_t dim;             // L2: rounding of |q|^2 in double
    double l2_slack;          // L2: relative rounding error of the reference's float distance^2 (l2_rounding_slack)
};

// The reference's float L2 distance (ref_order.cuh) is dist~ = sqrtf(S~), S~ a float sum of the terms fl(fl(a - b)^2).
// With u = 2^-24 and D the exact distance of the stored values: every term carries three roundings (the difference, counted
// twice once squared, and the product), each term passes at most m rounded additions (scalar loop: m = d; AVX lanes: d/8
// per lane plus 7 across the lanes, m = d/8 + 8 covers both), sqrtf rounds once more, counted twice in dist~^2.  So
//   dist~^2 >= D^2 (1 - u)^(m + 5) >= D^2 (1 - (m + 5) u).
// A row with D^2 >= L cannot reach dist_k (strictly) when L (1 - (m + 5) u) > dist_k^2.  For the scalar loop at d = 3000
// g = 1.8e-4: the former flat 1e-4 was too small beyond d ~ 1650.
static double l2_rounding_slack(uint32_t d) {
    const double m = (d >= 16 && d % 16 == 0) ? d / 8.0 + 8.0 : (double)d;
    return (m + 5.0) * 0x1p-24;
}

// one CTA per query: order survivors by (sim desc, row asc), emit k, certify.  CTA b serves query qmap[b] (or b).
__global__ void __launch_bounds__(SEL_THREADS) final_kernel(const Exact* __restrict__ ex, const uint32_t* __restrict__ ex_n,
                                                            uint32_t Kp, uint32_t k,
                                                            const int64_t* __restrict__ rowids, int negate,
                                                            int64_t* __restrict__ out_rowids, float* __restrict__ out_scores,
                                                            uint32_t* __restrict__ out_counts, uint64_t* __restrict__ out_flags,
                                                            float pad_score, const uint32_t* __restrict__ qmap, CertArgs cert) {
    __shared__ uint64_t buf[SEL_MAXK];
    const uint32_t b = blockIdx.x;
    const uint32_t q = qmap ? qmap[b] : b;
    uint32_t np2 = 1;
    while (np2 < Kp) np2 <<= 1;
    for (uint32_t i = threadIdx.x; i < np2; i += SEL_THREADS) {
        uint64_t key = 0;
        if (i < Kp && (!ex_n || i < ex_n[b])) {
            Exact e = ex[(uint64_t)b * Kp + i];
            if (e.sim == e.sim) key = ((uint64_t)fkey(e.sim) << 32) | (uint64_t)(0xFFFFFFFFu - e.row);
        }
        buf[i] = key;
    }
    __syncthreads();
    for (uint32_t size = 2; size <= np2; size <<= 1) {
        for (uint32_t stride = size >> 1; stride > 0; stride >>= 1) {
            for (uint32_t t = threadIdx.x; t < np2 / 2; t += SEL_THREADS) {
                uint32_t lo = (t / stride) * (stride * 2) + (t % stride);
                uint32_t hi = lo + stride;
                bool desc = ((lo & size) == 0);
                uint64_t x = buf[lo], y = buf[hi];
                if ((x < y) == desc) { buf[lo] = y; buf[hi] = x; }
            }
            __syncthreads();
        }
    }
    // valid entries are the non-zero keys at the front
    __shared__ uint32_t s_valid;
    if (threadIdx.x == 0) s_valid = 0;
    __syncthreads();
    uint32_t local = 0;
    for (uint32_t i = threadIdx.x; i < np2; i += SEL_THREADS) local += buf[i] != 0 ? 1u : 0u;
    atomicAdd(&s_valid, local);
    __syncthreads();
    uint32_t valid = s_valid;
    uint32_t nout = min(valid, k);
    for (uint32_t i = threadIdx.x; i < k; i += SEL_THREADS) {
        if (i < nout) {
            uint64_t key = buf[i];
            uint32_t row = 0xFFFFFFFFu - (uint32_t)key;
            float s = fkey_inv((uint32_t)(key >> 32));
            out_rowids[(uint64_t)q * k + i] = rowids[row];
            out_scores[(uint64_t)q * k + i] = negate ? -s : s;
        } else {
            out_rowids[(uint64_t)q * k + i] = -1;
            out_scores[(uint64_t)q * k + i] = pad_score;
        }
    }
    if (threadIdx.x == 0) {
        if (out_counts) out_counts[q] = nout;
        uint64_t f = 0;
        if (valid > k && k > 0 && (buf[k - 1] >> 32) == (buf[k] >> 32)) f |= YAMS_B200_FLAG_TIE_AT_K;
        if (cert.status && k > 0) {
            const float bd = cert.bound[b];
            bool certified = true;
            if (bd != -INFINITY) {   // NaN included: the comparisons below are then false
                const float e = cert.eps[q];
                if (cert.metric == YAMS_B200_L2) {
                    certified = false;
                    if (valid >= k) {
                        const float dk = -fkey_inv((uint32_t)(buf[k - 1] >> 32));
                        const double qq = cert.qnorm[q] * cert.qnorm[q];
                        // lower bound of D^2 of every row not re-scored, less the double rounding of |q|^2 and of the difference
                        const double lo = qq - (double)bd - (double)e;
                        const double rnd = (double)(cert.dim + 4) * 0x1p-52 * (qq + fabs((double)bd) + (double)e);
                        certified = (lo - rnd) * (1.0 - cert.l2_slack) > (double)dk * (double)dk;
                    }
                } else {
                    const float lvl = valid >= k ? fkey_inv((uint32_t)(buf[k - 1] >> 32)) : cert.threshold;
                    certified = bd + e < lvl;
                }
            }
            if (!certified) {
                f |= YAMS_B200_FLAG_FALLBACK_PATH;
                uint32_t* cnt = cert.level == 0 ? &cert.status->n_bad : &cert.status->n_bad2;
                uint32_t* list = reinterpret_cast<uint32_t*>(cert.status + 1) + (cert.level == 0 ? 0u : cert.nq_total);
                uint32_t pos = atomicAdd(cnt, 1u);
                if (pos < cert.nq_total) list[pos] = q;
            }
        }
        if (cert.level >= 1) f |= YAMS_B200_FLAG_FALLBACK_PATH;   // answered by an exhaustive level
        if (out_flags) out_flags[q] = f;
    }
}

// level 2 (full exact pass): keys sorted descending -> the k best of ONE query
__global__ void emit_sorted_kernel(const uint64_t* __restrict__ keys, uint64_t nkeys, uint32_t k, uint32_t q,
                                   const int64_t* __restrict__ rowids, int negate, float pad_score, int64_t* __restrict__ out_rowids,
                                   float* __restrict__ out_scores, uint32_t* __restrict__ out_counts, uint64_t* __restrict__ out_flags) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < k) {
        uint64_t key = i < nkeys ? keys[i] : 0;
        if (key) {
            float s = fkey_inv((uint32_t)(key >> 32));
            out_rowids[(uint64_t)q * k + i] = rowids[0xFFFFFFFFu - (uint32_t)key];
            out_scores[(uint64_t)q * k + i] = negate ? -s : s;
        } else {
            out_rowids[(uint64_t)q * k + i] = -1;
            out_scores[(uint64_t)q * k + i] = pad_score;
        }
    }
    if (i == 0) {
        uint32_t cnt = 0;
        while (cnt < k && cnt < nkeys && keys[cnt]) ++cnt;
        if (out_counts) out_counts[q] = cnt;
        uint64_t f = YAMS_B200_FLAG_FALLBACK_PATH;
        if (cnt == k && k < nkeys && keys[k] && (keys[k - 1] >> 32) == (keys[k] >> 32)) f |= YAMS_B200_FLAG_TIE_AT_K;
        if (out_flags) out_flags[q] = f;
    }
}

// ---------------------------------------------------------------------------------------------------
// candidate-set mask: bit (q, row) set when rowids[row] is in query q's allowed list
// ---------------------------------------------------------------------------------------------------
__global__ void build_mask_kernel(const int64_t* __restrict__ allowed, const uint64_t* __restrict__ offsets, uint32_t nq,
                                  const int64_t* __restrict__ rowids, uint64_t n, uint32_t* __restrict__ mask, uint64_t mask_ld) {
    uint32_t q = blockIdx.y;
    uint64_t lo = offsets[q], hi = offsets[q + 1];
    for (uint64_t i = lo + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += (uint64_t)gridDim.x * blockDim.x) {
        int64_t want = allowed[i];
        uint64_t a = 0, b = n;
        while (a < b) {
            uint64_t m = a + ((b - a) >> 1);
            if (rowids[m] < want) a = m + 1; else b = m;
        }
        if (a < n && rowids[a] == want) atomicOr(&mask[(uint64_t)q * mask_ld + (a >> 5)], 1u << (a & 31));
    }
}

// scores of rows outside query q's allowed set become -inf (threshold calibration sample / exhaustive fallback).
// scores[b * ld + i] belongs to query (qmap ? qmap[b] : b) and row row_start + i * row_stride.
__global__ void mask_scores_kernel(float* __restrict__ scores, uint64_t ld, uint64_t len, uint64_t row_stride,
                                   const uint32_t* __restrict__ mask, uint64_t mask_ld, const uint32_t* __restrict__ qmap) {
    const uint32_t b = blockIdx.y;
    const uint32_t q = qmap ? qmap[b] : b;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < len; i += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t row = i * row_stride;
        if (!((mask[(uint64_t)q * mask_ld + (row >> 5)] >> (row & 31)) & 1u)) scores[(uint64_t)b * ld + i] = -INFINITY;
    }
}

// Small candidate sets: no corpus pass at all.  One warp per (query, allowed rowid) pair: rowid -> row by binary
// search, stage-1 score by a coalesced fp32 dot product of that one row, Cand written at the pair's list position
// (unknown or repeated rowids become (-inf, 0xFFFFFFFF) and are skipped downstream).  Lists must be ascending.
template <int VEC>   // 8: fp16 rows, dim % 8 == 0; 4: fp32 rows, dim % 4 == 0; 0: scalar
__global__ void gather_score_kernel(const void* __restrict__ rows, int dtype, uint32_t d, const float* __restrict__ inv_norm,
                                    const int64_t* __restrict__ rowids, uint64_t n, const float* __restrict__ q32,
                                    const float* __restrict__ qinv, const int64_t* __restrict__ allowed,
                                    const uint64_t* __restrict__ offsets, uint32_t nq, uint64_t total, Cand* __restrict__ cands,
                                    uint32_t cap) {
    const uint64_t pair = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t lane = threadIdx.x & 31;
    if (pair >= total) return;
    uint32_t qa = 0, qb = nq;   // last q with offsets[q] <= pair
    while (qb - qa > 1) {
        uint32_t m = (qa + qb) >> 1;
        if (offsets[m] <= pair) qa = m; else qb = m;
    }
    const uint32_t q = qa;
    const uint64_t j = pair - offsets[q];
    const int64_t want = allowed[pair];
    bool valid = !(j > 0 && allowed[pair - 1] == want);
    uint64_t a = 0, b = n;
    while (a < b) {
        uint64_t m = a + ((b - a) >> 1);
        if (rowids[m] < want) a = m + 1; else b = m;
    }
    valid = valid && a < n && rowids[a] == want;
    Cand out;
    out.score = -INFINITY;
    out.row = 0xFFFFFFFFu;
    if (valid) {
        const float* qv = q32 + (uint64_t)q * d;
        float s = 0.f;
        if (VEC == 8) {
            const uint4* r = reinterpret_cast<const uint4*>(static_cast<const __half*>(rows) + a * d);
            for (uint32_t u = lane; u < d / 8; u += 32) {
                uint4 v = __ldg(r + u);
                const __half2* h = reinterpret_cast<const __half2*>(&v);
                const float4 q0 = *reinterpret_cast<const float4*>(qv + u * 8), q1 = *reinterpret_cast<const float4*>(qv + u * 8 + 4);
                float2 f0 = __half22float2(h[0]), f1 = __half22float2(h[1]), f2 = __half22float2(h[2]), f3 = __half22float2(h[3]);
                s = fmaf(f0.x, q0.x, s); s = fmaf(f0.y, q0.y, s); s = fmaf(f1.x, q0.z, s); s = fmaf(f1.y, q0.w, s);
                s = fmaf(f2.x, q1.x, s); s = fmaf(f2.y, q1.y, s); s = fmaf(f3.x, q1.z, s); s = fmaf(f3.y, q1.w, s);
            }
        } else if (VEC == 4) {
            const float4* r = reinterpret_cast<const float4*>(static_cast<const float*>(rows) + a * d);
            for (uint32_t u = lane; u < d / 4; u += 32) {
                float4 v = __ldg(r + u);
                const float4 qq = *reinterpret_cast<const float4*>(qv + u * 4);
                s = fmaf(v.x, qq.x, s); s = fmaf(v.y, qq.y, s); s = fmaf(v.z, qq.z, s); s = fmaf(v.w, qq.w, s);
            }
        } else {
            for (uint32_t cidx = lane; cidx < d; cidx += 32) s = fmaf(load_elem(rows, dtype, a * d + cidx), qv[cidx], s);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        out.score = s * inv_norm[a] * qinv[q];
        out.row = (uint32_t)a;
    }
    if (lane == 0) cands[(uint64_t)q * cap + j] = out;
}
__global__ void list_lengths_kernel(const uint64_t* __restrict__ offsets, uint32_t nq, uint32_t* __restrict__ counts) {
    uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q < nq) counts[q] = (uint32_t)(offsets[q + 1] - offsets[q]);
}

// ---------------------------------------------------------------------------------------------------
// sqlite-vec-cpp operator surface (vec0_run_exact_query, distances/batch.hpp): one thread per row evaluates the float
// distance in the reference build's own operation order (ref_order.cuh) -> bit-identical results.  NEGATED distance out so
// that the descending key sort used everywhere else yields ascending distances.
// ---------------------------------------------------------------------------------------------------
__global__ void batch_dist_kernel(const float* __restrict__ rows, uint32_t d, uint64_t n, const float* __restrict__ q, int metric,
                                  float* __restrict__ out_neg) {
    uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    F32At qa{q}, ra{rows + r * d};
    out_neg[r] = -(metric == YAMS_B200_L2 ? ref_l2_distance(qa, ra, d) : ref_cosine_distance(qa, ra, d));
}
// keys for the FILTERED mode: rows failing dist < threshold get key 0 (sort last)
__global__ void make_keys_filtered_kernel(const float* __restrict__ neg_dist, uint64_t n, uint64_t np2, float threshold,
                                          uint64_t* __restrict__ keys) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < np2; i += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t key = 0;
        if (i < n && (-neg_dist[i]) < threshold) key = ((uint64_t)fkey(neg_dist[i]) << 32) | (uint64_t)(0xFFFFFFFFu - (uint32_t)i);
        keys[i] = key;
    }
}
__global__ void unpack_idx_keys_kernel(const uint64_t* __restrict__ keys, uint64_t m, uint64_t* __restrict__ out_idx,
                                       float* __restrict__ out_dist) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t key = keys[i];
        out_idx[i] = 0xFFFFFFFFu - (uint32_t)key;
        out_dist[i] = -fkey_inv((uint32_t)(key >> 32));
    }
}
__global__ void negate_kernel(float* p, uint64_t n) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) p[i] = -p[i];
}
// computeCosineSimilarity (vector_database.cpp:1786-1810): one thread, the reference's accumulation order
__global__ void cosine_similarity_f64_kernel(const float* __restrict__ a_all, const float* __restrict__ b_all, uint64_t n, uint64_t d,
                                             double* __restrict__ out_all) {
    const uint64_t p = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const float* a = a_all + p * d;
    const float* b = b_all + p * d;
    double* out = out_all + p;
    double dp = 0.0, na = 0.0, nb = 0.0;
    for (uint64_t i = 0; i < d; ++i) {
        double x = (double)a[i], y = (double)b[i];
        dp += x * y;
        na += x * x;
        nb += y * y;
    }
    na = sqrt(na);
    nb = sqrt(nb);
    *out = (na == 0.0 || nb == 0.0) ? 0.0 : dp / (na * nb);
}

// global-memory bitonic sort (descending) of 64-bit keys, n a power of two
__global__ void bitonic_step_kernel(uint64_t* __restrict__ keys, uint64_t n, uint64_t size, uint64_t stride) {
    for (uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n / 2; t += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t lo = (t / stride) * (stride * 2) + (t % stride);
        uint64_t hi = lo + stride;
        bool desc = ((lo & size) == 0);
        uint64_t x = keys[lo], y = keys[hi];
        if ((x < y) == desc) { keys[lo] = y; keys[hi] = x; }
    }
}
__global__ void make_keys_kernel(const float* __restrict__ neg_dist, uint64_t n, uint64_t np2, uint64_t* __restrict__ keys) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < np2; i += (uint64_t)gridDim.x * blockDim.x)
        keys[i] = i < n ? (((uint64_t)fkey(neg_dist[i]) << 32) | (uint64_t)(0xFFFFFFFFu - (uint32_t)i)) : 0ull;
}
__global__ void unpack_keys_kernel(const uint64_t* __restrict__ keys, uint64_t m, const int64_t* __restrict__ rowids,
                                   int64_t* __restrict__ out_rowids, float* __restrict__ out_dist) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t key = keys[i];
        uint32_t row = 0xFFFFFFFFu - (uint32_t)key;
        out_rowids[i] = rowids ? rowids[row] : (int64_t)row;
        out_dist[i] = -fkey_inv((uint32_t)(key >> 32));
    }
}

// ---------------------------------------------------------------------------------------------------
// multi-GPU: merge R partial top-k lists per query
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(SEL_THREADS) merge_partials_kernel(const int64_t* __restrict__ rowids, const float* __restrict__ scores,
                                                                     uint64_t rank_stride_r, uint64_t rank_stride_s,
                                                                     uint32_t R, uint32_t nq, uint32_t k, int l2,
                                                                     int64_t* __restrict__ out_rowids, float* __restrict__ out_scores,
                                                                     uint32_t* __restrict__ out_counts) {
    extern __shared__ unsigned char smraw[];
    float* ks = reinterpret_cast<float*>(smraw);                 // np2 scores (as "bigger is better")
    int64_t* kr = reinterpret_cast<int64_t*>(smraw + 0);         // placed after scores, see below
    const uint32_t q = blockIdx.x;
    uint32_t total = R * k, np2 = 1;
    while (np2 < total) np2 <<= 1;
    kr = reinterpret_cast<int64_t*>(smraw + (((size_t)np2 * 4 + 7) & ~(size_t)7));
    for (uint32_t i = threadIdx.x; i < np2; i += SEL_THREADS) {
        float s = -INFINITY;
        int64_t r = INT64_MAX;
        if (i < total) {
            uint32_t rk = i / k, j = i % k;
            size_t idx = (size_t)q * k + j;
            r = rowids[(size_t)rk * rank_stride_r + idx];
            s = scores[(size_t)rk * rank_stride_s + idx];
            if (l2) s = -s;
            if (r < 0) { s = -INFINITY; r = INT64_MAX; }
        }
        ks[i] = s;
        kr[i] = r;
    }
    __syncthreads();
    for (uint32_t size = 2; size <= np2; size <<= 1) {
        for (uint32_t stride = size >> 1; stride > 0; stride >>= 1) {
            for (uint32_t t = threadIdx.x; t < np2 / 2; t += SEL_THREADS) {
                uint32_t lo = (t / stride) * (stride * 2) + (t % stride);
                uint32_t hi = lo + stride;
                bool desc = ((lo & size) == 0);
                float xs = ks[lo], ys = ks[hi];
                int64_t xr = kr[lo], yr = kr[hi];
                // "x is worse than y": lower score, or equal score and larger rowid
                bool x_worse = (xs < ys) || (xs == ys && xr > yr);
                if (x_worse == desc) { ks[lo] = ys; ks[hi] = xs; kr[lo] = yr; kr[hi] = xr; }
            }
            __syncthreads();
        }
    }
    __shared__ uint32_t s_valid;
    if (threadIdx.x == 0) s_valid = 0;
    __syncthreads();
    uint32_t local = 0;
    for (uint32_t i = threadIdx.x; i < np2; i += SEL_THREADS) local += (kr[i] != INT64_MAX) ? 1u : 0u;
    atomicAdd(&s_valid, local);
    __syncthreads();
    uint32_t nout = min(s_valid, k);
    for (uint32_t i = threadIdx.x; i < k; i += SEL_THREADS) {
        if (i < nout) {
            out_rowids[(size_t)q * k + i] = kr[i];
            out_scores[(size_t)q * k + i] = l2 ? -ks[i] : ks[i];
        } else {
            out_rowids[(size_t)q * k + i] = -1;
            out_scores[(size_t)q * k + i] = l2 ? INFINITY : -INFINITY;
        }
    }
    if (threadIdx.x == 0 && out_counts) out_counts[q] = nout;
}

// candidate rowids -> row indices (binary search in the ascending device rowid table); misses get 0xFFFFFFFF
__global__ void map_rowids_kernel(const int64_t* __restrict__ allowed, uint64_t na, const int64_t* __restrict__ rowids, uint64_t n,
                                  Cand* __restrict__ sel) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < na; i += (uint64_t)gridDim.x * blockDim.x) {
        int64_t want = allowed[i];
        uint64_t a = 0, b = n;
        while (a < b) {
            uint64_t m = a + ((b - a) >> 1);
            if (rowids[m] < want) a = m + 1; else b = m;
        }
        Cand c;
        c.score = 0.f;
        c.row = (a < n && rowids[a] == want) ? (uint32_t)a : 0xFFFFFFFFu;
        sel[i] = c;
    }
}
__global__ void iota_sel_kernel(Cand* sel, uint64_t n) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        Cand c;
        c.score = 0.f;
        c.row = (uint32_t)i;
        sel[i] = c;
    }
}
// Exact results -> sortable keys (skipped entries sort last as 0)
__global__ void exact_keys_kernel(const Exact* __restrict__ ex, uint64_t n, uint64_t np2, uint64_t* __restrict__ keys) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < np2; i += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t key = 0;
        if (i < n) {
            Exact e = ex[i];
            if (e.sim == e.sim) key = ((uint64_t)fkey(e.sim) << 32) | (uint64_t)(0xFFFFFFFFu - e.row);
        }
        keys[i] = key;
    }
}
__global__ void count_nonzero_kernel(const uint64_t* __restrict__ keys, uint64_t n, unsigned long long* __restrict__ out) {
    unsigned long long c = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) c += keys[i] != 0;
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(out, c);
}
__global__ void unpack_sim_keys_kernel(const uint64_t* __restrict__ keys, uint64_t m, const int64_t* __restrict__ rowids,
                                       int64_t* __restrict__ out_rowids, float* __restrict__ out_scores) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t key = keys[i];
        uint32_t row = 0xFFFFFFFFu - (uint32_t)key;
        out_rowids[i] = rowids[row];
        out_scores[i] = fkey_inv((uint32_t)(key >> 32));
    }
}

// ---- corpus_remove: stable compaction ------------------------------------------------------------------
__global__ void fill_u32_kernel(uint32_t* p, uint64_t n, uint32_t v) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) p[i] = v;
}
__global__ void mark_removed_kernel(const int64_t* __restrict__ gone, uint64_t ng, const int64_t* __restrict__ rowids, uint64_t n,
                                    uint32_t* __restrict__ keep) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < ng; i += (uint64_t)gridDim.x * blockDim.x) {
        int64_t want = gone[i];
        uint64_t a = 0, b = n;
        while (a < b) {
            uint64_t m = a + ((b - a) >> 1);
            if (rowids[m] < want) a = m + 1; else b = m;
        }
        if (a < n && rowids[a] == want) keep[a] = 0u;
    }
}
// kept rows of [b0, b1) -> tmp[dst[row] - dst[b0]]; one warp per row, UNIT-byte elements
template <typename UNIT>
__global__ void compact_gather_kernel(const UNIT* __restrict__ src, uint64_t units_per_row, uint64_t b0, uint64_t b1,
                                      const uint32_t* __restrict__ keep, const uint32_t* __restrict__ dst, UNIT* __restrict__ tmp) {
    uint64_t row = b0 + (((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    uint32_t lane = threadIdx.x & 31;
    if (row >= b1 || !keep[row] || dst[row] == row) return;
    const UNIT* s = src + row * units_per_row;
    UNIT* t = tmp + (uint64_t)(dst[row] - dst[b0]) * units_per_row;
    for (uint64_t u = lane; u < units_per_row; u += 32) t[u] = s[u];
}
template <typename UNIT>
__global__ void compact_scatter_kernel(UNIT* __restrict__ rows, uint64_t units_per_row, uint64_t b0, uint64_t b1,
                                       const uint32_t* __restrict__ keep, const uint32_t* __restrict__ dst, const UNIT* __restrict__ tmp) {
    uint64_t row = b0 + (((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    uint32_t lane = threadIdx.x & 31;
    if (row >= b1 || !keep[row] || dst[row] == row) return;
    UNIT* d = rows + (uint64_t)dst[row] * units_per_row;
    const UNIT* t = tmp + (uint64_t)(dst[row] - dst[b0]) * units_per_row;
    for (uint64_t u = lane; u < units_per_row; u += 32) d[u] = t[u];
}

// per-query state of one scan: survivor counts, certificate bounds, candidate-list counters
__global__ void scan_init_kernel(uint32_t nq, uint32_t* __restrict__ sel_n, float* __restrict__ bound, uint32_t* __restrict__ counts) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nq) {
        sel_n[i] = 0;
        bound[i] = -INFINITY;
        counts[i] = 0;
    }
}
__global__ void fill_f32_kernel(float* p, uint64_t n, float v) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) p[i] = v;
}
__global__ void iota_rowids_kernel(int64_t* p, uint64_t n, int64_t first) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
        p[i] = first + (int64_t)i;
}

}  // namespace yb

// ===================================================================================================
// host side: corpus mirror + search orchestration
// ===================================================================================================

namespace yb {

// tcgen05 engine (knn_umma.cu); returns YAMS_ERR_UNSUPPORTED when the shape is not covered
yams_status_t stage1_tcgen05(Corpus* c, const Stage1Args& a, bool filter, cudaStream_t st);
bool tcgen05_supported(const Corpus* c, uint32_t nq);

constexpr uint32_t kMaxK = 3072;          // K' = k + max(16, k/4) rounded to 32 must fit SEL_MAXK
constexpr uint32_t kSampleRows = 32768;   // strided sample that calibrates the per-query thresholds (dense fp32 scores: Q x 128 KiB)
constexpr uint32_t kSampleRank = 8;       // threshold = 8th best score of the sample
constexpr float kTauMargin = 2e-3f;       // cosine: keeps the candidate lists comfortably longer than K' (not needed for
                                          // exactness -- the certificate covers rows below the threshold)
constexpr uint32_t kCandCap = 8192;       // candidate list capacity per query
constexpr uint32_t kDenseLimit = 65536;   // corpora up to this many rows are scored densely
constexpr uint32_t kLevel1K = SEL_MAXK;   // survivors re-scored per query by exhaustive level 1
constexpr uint32_t kLevel1Group = 8;      // queries per level-1 group: group * n floats of scratch

static uint32_t survivors_for(uint32_t k) {
    uint32_t slack = std::max<uint32_t>(16, k / 4);
    uint32_t kp = ((k + slack + 31) / 32) * 32;
    return std::min<uint32_t>(kp, SEL_MAXK);
}

static yams_status_t corpus_reserve(Corpus* c, uint64_t n_total) {
    yams_status_t rc;
    if ((rc = c->rows.reserve((size_t)n_total * c->dim * c->elem() + 256, true, c->st)) != YAMS_OK) return rc;
    if ((rc = c->rowids.reserve((size_t)n_total * 8 + 256, true, c->st)) != YAMS_OK) return rc;
    if ((rc = c->inv_norm.reserve((size_t)n_total * 4 + 256, true, c->st)) != YAMS_OK) return rc;
    if (!c->stats.p) {
        if ((rc = c->stats.reserve(16)) != YAMS_OK) return rc;
        YB_CUDA(cudaMemsetAsync(c->stats.p, 0, 16, c->st));
    }
    return YAMS_OK;
}

// row statistics of the n_new rows already copied behind the current end + commit of the append.
// Nothing of the corpus state changes unless every check passed (a rejected batch leaves the corpus as it was).
static yams_status_t corpus_finish_append(Corpus* c, uint64_t n_new, const int64_t* rowids_host, int64_t first_synthetic = -1) {
    int64_t* d_rid = c->rowids.as<int64_t>() + c->n;
    int64_t last = c->last_rowid;
    bool dense = c->rowids_dense;
    if (rowids_host) {
        for (uint64_t i = 0; i < n_new; ++i) {
            YB_ARG(rowids_host[i] >= 0, "rowids must be non-negative (-1 marks an unused result slot)");
            YB_ARG(rowids_host[i] > last, "rowids must be appended in strictly ascending order");
            if (c->n + i > 0 && rowids_host[i] != last + 1) dense = false;
            last = rowids_host[i];
        }
        YB_CUDA(cudaMemcpyAsync(d_rid, rowids_host, (size_t)n_new * 8, cudaMemcpyHostToDevice, c->st));
    } else {
        int64_t first = first_synthetic >= 0 ? first_synthetic : (c->n == 0 ? 0 : last + 1);
        YB_ARG(first > last || c->n == 0, "rowids must be appended in strictly ascending order");
        if (c->n > 0 && first != last + 1) dense = false;
        iota_rowids_kernel<<<(unsigned)std::min<uint64_t>((n_new + 255) / 256, 4096), 256, 0, c->st>>>(d_rid, n_new, first);
        last = first + (int64_t)n_new - 1;
    }
    row_stats_kernel<<<(unsigned)((n_new + 127) / 128), 128, 0, c->st>>>(c->rows.p, c->dtype, c->dim, c->n, n_new,
                                                                       c->inv_norm.as<float>(), c->metric, c->stats.as<float>());
    YB_CUDA(cudaGetLastError());
    float h_stats[4] = {0, 0, 0, 0};
    YB_CUDA(cudaMemcpyAsync(h_stats, c->stats.p, 12, cudaMemcpyDeviceToHost, c->st));
    YB_CUDA(cudaStreamSynchronize(c->st));
    c->r_max = h_stats[0];
    c->dr_abs_max = h_stats[1];
    c->dr_rel_max = h_stats[2];
    c->last_rowid = last;
    c->rowids_dense = dense;
    c->n += n_new;
    ++c->generation;
    return YAMS_OK;
}

// Small candidate sets (CandidateFilterMode::Exact): device lists (ascending rowids, d_offsets[nq+1]) short enough that
// scoring the listed rows one by one is cheaper than a corpus pass -> gather_score_kernel
struct DirectLists {
    const int64_t* d_allowed = nullptr;
    const uint64_t* d_offsets = nullptr;
    uint64_t total = 0;
    uint32_t max_len = 0;
};

struct ScanPlan {
    uint32_t nq = 0, k = 0;
    float threshold = -1.f;
    const uint32_t* d_mask = nullptr;   // bit matrix [nq][mask_ld*32] of allowed rows -> masked corpus pass
    uint64_t mask_ld = 0;
    const DirectLists* direct = nullptr;
    bool use_tensor = false;
};

static ScanStatus* status_of(Corpus* c) { return c->status.as<ScanStatus>(); }

static void fill_stage1_common(Corpus* c, Stage1Args& a, uint32_t nq) {
    a.rows = c->rows.p;
    a.inv_norm = c->inv_norm.as<float>();
    a.dim = c->dim;
    a.dtype = c->dtype;
    a.q32 = c->q32.as<float>();
    a.qinv = c->qinv.as<float>();
    a.nq = nq;
    a.metric = c->metric;
    a.eps = c->eps.as<float>();
    a.r_max = c->r_max;
    a.dr_abs_max = c->dr_abs_max;
    a.dr_rel_max = c->dr_rel_max;
}

// Enqueues the whole pipeline for the nq queries already prepared on the device (prepare_queries) and writes the padded
// [nq][k] result into device buffers.  NO host synchronisation: list overflow, short lists and stage-1 rounding are all
// caught by the certificate in final_kernel, which queues such queries in the ScanStatus block for resolve_uncertain().
static yams_status_t scan_enqueue(Corpus* c, const ScanPlan& p, int64_t* d_out_rowids, float* d_out_scores, uint32_t* d_out_counts,
                                  uint64_t* d_out_flags) {
    yams_status_t rc;
    cudaStream_t st = c->st;
    const uint32_t nq = p.nq, k = p.k;
    const uint32_t Kp = survivors_for(k);
    const uint64_t n = c->n;
    const bool l2 = c->metric == YAMS_B200_L2;
    c->scan_timed = false;
    double* d_qnorm = reinterpret_cast<double*>(c->misc.as<uint8_t>());           // nq doubles
    uint32_t* d_counts = c->counts.as<uint32_t>();
    Stage1Args a{};
    fill_stage1_common(c, a, nq);
    bool qprep_done = false, tensor_used = false, cc_used = false;
    auto run_stage1 = [&](Stage1Args args, bool filter) -> yams_status_t {
        if (p.use_tensor) {
            args.skip_qprep = qprep_done;
            yams_status_t r = stage1_tcgen05(c, args, filter, st);
            if (r == YAMS_OK) { qprep_done = true; tensor_used = true; }
            if (r != YAMS_ERR_UNSUPPORTED) return r;
        }
        cc_used = true;
        return stage1_cuda_core(args, filter, st);
    };
    if ((rc = c->sel.reserve((size_t)nq * Kp * sizeof(Cand) + (size_t)nq * 4)) != YAMS_OK) return rc;
    if ((rc = c->bound.reserve((size_t)nq * 4)) != YAMS_OK) return rc;
    if ((rc = c->eps.reserve((size_t)nq * 4)) != YAMS_OK) return rc;
    a.eps = c->eps.as<float>();
    Cand* d_sel = c->sel.as<Cand>();
    uint32_t* d_sel_n = reinterpret_cast<uint32_t*>(d_sel + (size_t)nq * Kp);
    float* d_bound = c->bound.as<float>();
    scan_init_kernel<<<(nq + 255) / 256, 256, 0, st>>>(nq, d_sel_n, d_bound, d_counts);

    if (n == 0) {
        // nothing to score: every list is empty, bound = -inf
    } else if (p.direct) {
        // ---- small candidate sets: score the listed rows only ----
        const DirectLists* direct = p.direct;
        const uint32_t cap = std::max<uint32_t>(direct->max_len, 1);
        if ((rc = c->cands.reserve((size_t)nq * cap * sizeof(Cand))) != YAMS_OK) return rc;
        list_lengths_kernel<<<(nq + 255) / 256, 256, 0, st>>>(direct->d_offsets, nq, d_counts);
        if (direct->total) {
            const unsigned grid = (unsigned)((direct->total * 32 + 255) / 256);
            const bool v8 = c->dtype == YAMS_B200_F16 && c->dim % 8 == 0, v4 = c->dtype == YAMS_B200_F32 && c->dim % 4 == 0;
#define YB_GATHER(V)                                                                                                              \
    gather_score_kernel<V><<<grid, 256, 0, st>>>(c->rows.p, c->dtype, c->dim, c->inv_norm.as<float>(), c->rowids.as<int64_t>(), n, \
                                                 a.q32, a.qinv, direct->d_allowed, direct->d_offsets, nq, direct->total,           \
                                                 c->cands.as<Cand>(), cap)
            YB_CUDA(cudaEventRecord(c->ev_scan[0], st));
            if (v8) YB_GATHER(8); else if (v4) YB_GATHER(4); else YB_GATHER(0);
#undef YB_GATHER
            YB_CUDA(cudaEventRecord(c->ev_scan[1], st));
            c->scan_timed = true;
        }
        cc_used = true;   // fp32 CUDA-core dot products: same error bound as the CUDA-core engine
        SelectIn in{};
        in.cands = c->cands.as<Cand>(); in.counts = d_counts; in.cap = cap;
        topk_select_kernel<<<nq, SEL_THREADS, 0, st>>>(in, Kp, 0, nullptr, d_sel, d_sel_n, d_bound);
    } else if (!p.d_mask && n <= kDenseLimit) {
        // ---- dense: every score materialised, exact top-K' straight from the matrix ----
        if ((rc = c->dense.reserve((size_t)nq * n * 4)) != YAMS_OK) return rc;
        a.row_start = 0; a.row_stride = 1; a.nrows = n;
        a.out_scores = c->dense.as<float>(); a.ld = n;
        if ((rc = run_stage1(a, false)) != YAMS_OK) return rc;
        SelectIn in{};
        in.dense = c->dense.as<float>(); in.ld = n; in.row_start = 0; in.row_stride = 1; in.dense_len = n;
        topk_select_kernel<<<nq, SEL_THREADS, 0, st>>>(in, Kp, 0, nullptr, d_sel, d_sel_n, d_bound);
    } else {
        uint32_t cap;
        if ((rc = c->tau.reserve((size_t)nq * 4)) != YAMS_OK) return rc;
        float* d_tau = c->tau.as<float>();
        {
            // ---- thresholds from a strided sample (candidate-set mode: of the ALLOWED sample rows, so that ~4*K'
            //      allowed rows are expected above it; -inf when the sample holds fewer than m allowed rows) ----
            uint64_t S = std::min<uint64_t>(n, kSampleRows);
            uint64_t stride = n / S;
            // the sample rank is chosen so that ~4*K' rows are expected above the threshold
            uint32_t m = (uint32_t)std::max<uint64_t>(kSampleRank, (4ull * Kp + stride - 1) / stride);
            uint64_t expected = (uint64_t)m * stride;
            cap = (uint32_t)std::max<uint64_t>(kCandCap, ((3 * expected + 1023) / 1024) * 1024);
            if ((rc = c->sample_scores.reserve((size_t)nq * S * 4)) != YAMS_OK) return rc;
            Stage1Args s1 = a;
            s1.row_start = 0; s1.row_stride = stride; s1.nrows = S;
            s1.out_scores = c->sample_scores.as<float>(); s1.ld = S;
            if ((rc = run_stage1(s1, false)) != YAMS_OK) return rc;
            if (p.d_mask)
                mask_scores_kernel<<<dim3((unsigned)((S + 255) / 256), nq), 256, 0, st>>>(c->sample_scores.as<float>(), S, S, stride,
                                                                                         p.d_mask, p.mask_ld, nullptr);
            SelectIn in{};
            in.dense = c->sample_scores.as<float>(); in.ld = S; in.row_start = 0; in.row_stride = stride; in.dense_len = S;
            in.tau_margin = l2 ? 0.f : kTauMargin;
            in.fast_tau = p.d_mask ? 0 : 1;   // candidate sets: masked sample rows are -inf, the exact rank matters there
            topk_select_kernel<<<nq, SEL_THREADS, 0, st>>>(in, m, 1, d_tau, nullptr, nullptr, nullptr);
        }
        if ((rc = c->cands.reserve((size_t)nq * cap * sizeof(Cand))) != YAMS_OK) return rc;
        Stage1Args f = a;
        f.row_start = 0; f.row_stride = 1; f.nrows = n;
        f.tau = d_tau; f.cands = c->cands.as<Cand>(); f.cap = cap; f.counts = d_counts;
        f.mask = p.d_mask; f.mask_ld = p.mask_ld;
        YB_CUDA(cudaEventRecord(c->ev_scan[0], st));
        if ((rc = run_stage1(f, true)) != YAMS_OK) return rc;
        YB_CUDA(cudaEventRecord(c->ev_scan[1], st));
        c->scan_timed = true;
        SelectIn in{};
        in.cands = c->cands.as<Cand>(); in.counts = d_counts; in.cap = cap; in.tau = d_tau;
        topk_select_kernel<<<nq, SEL_THREADS, 0, st>>>(in, Kp, 0, nullptr, d_sel, d_sel_n, d_bound);
    }
    // error bound of the engine(s) that produced the ranking
    if (cc_used || !tensor_used)
        eps_cc_kernel<<<(nq + 255) / 256, 256, 0, st>>>(d_qnorm, nq, c->dim, c->metric, c->r_max, c->eps.as<float>(), tensor_used ? 1 : 0);
    YB_CUDA(cudaEventRecord(c->ev[1], st));
    // ---- stage 2: exact re-scoring, ordering, certificate ----
    if ((rc = c->outbuf.reserve((size_t)nq * Kp * sizeof(Exact))) != YAMS_OK) return rc;
    Exact* d_ex = c->outbuf.as<Exact>();
    uint64_t tot = (uint64_t)nq * Kp;
    rescore_kernel<<<(unsigned)((tot + 127) / 128), 128, 0, st>>>(c->rows.p, c->dtype, c->dim, a.q32, d_qnorm, d_sel, d_sel_n, Kp, nq,
                                                                  p.threshold, d_ex, c->metric, nullptr, p.d_mask, p.mask_ld);
    CertArgs cert{};
    cert.bound = d_bound; cert.eps = c->eps.as<float>(); cert.qnorm = d_qnorm; cert.threshold = p.threshold;
    cert.metric = c->metric; cert.status = status_of(c); cert.level = 0; cert.nq_total = nq;
    cert.dim = c->dim; cert.l2_slack = l2_rounding_slack(c->dim);
    final_kernel<<<nq, SEL_THREADS, 0, st>>>(d_ex, nullptr, Kp, k, c->rowids.as<int64_t>(), l2 ? 1 : 0, d_out_rowids, d_out_scores,
                                             d_out_counts, d_out_flags, l2 ? INFINITY : -INFINITY, nullptr, cert);
    YB_CUDA(cudaGetLastError());
    return YAMS_OK;
}

// entry points for the other engines (pq.cu): exact top-K of per-query candidate lists, and the plain final ordering
void launch_topk_lists(const Cand* lists, const uint32_t* counts, uint32_t cap, uint32_t nq, uint32_t K, Cand* out_sel, uint32_t* out_n,
                       cudaStream_t st) {
    SelectIn in{};
    in.cands = lists; in.counts = counts; in.cap = cap;
    topk_select_kernel<<<nq, SEL_THREADS, 0, st>>>(in, K, 0, nullptr, out_sel, out_n, nullptr);
}
void launch_final_plain(const void* exact, uint32_t Kp, uint32_t k, uint32_t nq, const int64_t* rowids, int64_t* out_rowids, float* out_scores,
                        uint32_t* out_counts, uint64_t* out_flags, cudaStream_t st) {
    CertArgs cert{};   // status == nullptr: no certificate (the caller's survivors are what the reference re-ranks, too)
    final_kernel<<<nq, SEL_THREADS, 0, st>>>(static_cast<const Exact*>(exact), nullptr, Kp, k, rowids, 0, out_rowids, out_scores, out_counts,
                                             out_flags, -INFINITY, nullptr, cert);
}

// Level 2: exact score of EVERY row for one query (the reference's own loop, row-parallel) + a global sort.
static yams_status_t exact_all_rows(Corpus* c, const ScanPlan& p, uint32_t q, int64_t* d_out_rowids, float* d_out_scores,
                                    uint32_t* d_out_counts, uint64_t* d_out_flags) {
    yams_status_t rc;
    cudaStream_t st = c->st;
    const uint64_t m = c->n;
    const bool l2 = c->metric == YAMS_B200_L2;
    uint64_t np2 = 1;
    while (np2 < std::max<uint64_t>(m, 1)) np2 <<= 1;
    if ((rc = c->sel.reserve((size_t)m * sizeof(Cand) + 64)) != YAMS_OK) return rc;
    if ((rc = c->outbuf.reserve((size_t)m * sizeof(Exact) + 64)) != YAMS_OK) return rc;
    if ((rc = c->dense.reserve((size_t)np2 * 8 + 64)) != YAMS_OK) return rc;
    if ((rc = c->lvl.reserve(64)) != YAMS_OK) return rc;
    Cand* d_sel = c->sel.as<Cand>();
    uint64_t* d_keys = c->dense.as<uint64_t>();
    uint32_t* d_small = c->lvl.as<uint32_t>();     // [0] = survivors (m), [1] = query index
    uint32_t h_small[2] = {(uint32_t)m, q};
    YB_CUDA(cudaMemcpyAsync(d_small, h_small, 8, cudaMemcpyHostToDevice, st));
    unsigned g = (unsigned)std::min<uint64_t>((np2 + 255) / 256, 65535);
    double* d_qnorm = reinterpret_cast<double*>(c->misc.as<uint8_t>());
    if (m) {
        iota_sel_kernel<<<g, 256, 0, st>>>(d_sel, m);
        rescore_kernel<<<(unsigned)((m + 127) / 128), 128, 0, st>>>(c->rows.p, c->dtype, c->dim, c->q32.as<float>(), d_qnorm, d_sel, d_small,
                                                                   (uint32_t)m, 1, p.threshold, c->outbuf.as<Exact>(), c->metric, d_small + 1,
                                                                   p.d_mask, p.mask_ld);
    }
    exact_keys_kernel<<<g, 256, 0, st>>>(c->outbuf.as<Exact>(), m, np2, d_keys);
    for (uint64_t size = 2; size <= np2; size <<= 1)
        for (uint64_t stride = size >> 1; stride > 0; stride >>= 1) bitonic_step_kernel<<<g, 256, 0, st>>>(d_keys, np2, size, stride);
    emit_sorted_kernel<<<(p.k + 255) / 256, 256, 0, st>>>(d_keys, np2, p.k, q, c->rowids.as<int64_t>(), l2 ? 1 : 0, l2 ? INFINITY : -INFINITY,
                                                          d_out_rowids, d_out_scores, d_out_counts, d_out_flags);
    YB_CUDA(cudaGetLastError());
    YB_CUDA(cudaStreamSynchronize(st));   // h_small / scratch reuse
    return YAMS_OK;
}

// Blocking: answers the queries the certificate rejected.
//   level 1: dense stage-1 scores of ALL rows with the CUDA-core engine (error bound eps_cc, ~1e-5), exact re-scoring of the
//            best kLevel1K (4096) rows instead of K', same certificate;
//   level 2: whatever level 1 cannot certify either (more than ~4000 rows within eps of the k-th score: a corpus of
//            duplicates) is answered by the exact score of every row.
static yams_status_t resolve_uncertain(Corpus* c, const ScanPlan& p, const uint32_t* bad, uint32_t n_bad, int64_t* d_out_rowids,
                                       float* d_out_scores, uint32_t* d_out_counts, uint64_t* d_out_flags) {
    yams_status_t rc;
    cudaStream_t st = c->st;
    const uint64_t n = c->n;
    const uint32_t k = p.k, G = kLevel1Group, K1 = kLevel1K;
    const bool l2 = c->metric == YAMS_B200_L2;
    if (n_bad == 0) return YAMS_OK;
    if ((rc = c->dense.reserve((size_t)G * n * 4 + (size_t)G * c->dim * 4 + (size_t)G * 8 + 64)) != YAMS_OK) return rc;
    if ((rc = c->lvl.reserve((size_t)G * K1 * (sizeof(Cand) + sizeof(Exact)) + (size_t)G * 16 + 64)) != YAMS_OK) return rc;
    if ((rc = c->eps2.reserve((size_t)p.nq * 4)) != YAMS_OK) return rc;
    float* d_scores = c->dense.as<float>();
    float* d_qg = d_scores + (size_t)G * n;
    float* d_qinv_g = d_qg + (size_t)G * c->dim;
    uint32_t* d_qmap = reinterpret_cast<uint32_t*>(d_qinv_g + G);
    Cand* d_sel1 = c->lvl.as<Cand>();
    Exact* d_ex1 = reinterpret_cast<Exact*>(d_sel1 + (size_t)G * K1);
    uint32_t* d_sel1_n = reinterpret_cast<uint32_t*>(d_ex1 + (size_t)G * K1);
    float* d_bound1 = reinterpret_cast<float*>(d_sel1_n + G);
    double* d_qnorm = reinterpret_cast<double*>(c->misc.as<uint8_t>());
    eps_cc_kernel<<<(p.nq + 255) / 256, 256, 0, st>>>(d_qnorm, p.nq, c->dim, c->metric, c->r_max, c->eps2.as<float>(), 0);
    Stage1Args a{};
    fill_stage1_common(c, a, p.nq);
    for (uint32_t g0 = 0; g0 < n_bad; g0 += G) {
        uint32_t g = std::min<uint32_t>(G, n_bad - g0);
        for (uint32_t i = 0; i < g; ++i) {
            YB_CUDA(cudaMemcpyAsync(d_qg + (size_t)i * c->dim, a.q32 + (size_t)bad[g0 + i] * c->dim, (size_t)c->dim * 4,
                                    cudaMemcpyDeviceToDevice, st));
            YB_CUDA(cudaMemcpyAsync(d_qinv_g + i, a.qinv + bad[g0 + i], 4, cudaMemcpyDeviceToDevice, st));
        }
        YB_CUDA(cudaMemcpyAsync(d_qmap, bad + g0, (size_t)g * 4, cudaMemcpyHostToDevice, st));
        Stage1Args e = a;
        e.q32 = d_qg; e.qinv = d_qinv_g; e.nq = g;
        e.row_start = 0; e.row_stride = 1; e.nrows = n; e.out_scores = d_scores; e.ld = n;
        if ((rc = stage1_cuda_core(e, false, st)) != YAMS_OK) return rc;
        if (p.d_mask)
            mask_scores_kernel<<<dim3((unsigned)std::min<uint64_t>((n + 255) / 256, 65535), g), 256, 0, st>>>(d_scores, n, n, 1, p.d_mask,
                                                                                                             p.mask_ld, d_qmap);
        SelectIn in{};
        in.dense = d_scores; in.ld = n; in.row_start = 0; in.row_stride = 1; in.dense_len = n;
        topk_select_kernel<<<g, SEL_THREADS, 0, st>>>(in, K1, 0, nullptr, d_sel1, d_sel1_n, d_bound1);
        uint64_t tot = (uint64_t)g * K1;
        rescore_kernel<<<(unsigned)((tot + 127) / 128), 128, 0, st>>>(c->rows.p, c->dtype, c->dim, a.q32, d_qnorm, d_sel1, d_sel1_n, K1, g,
                                                                      p.threshold, d_ex1, c->metric, d_qmap, p.d_mask, p.mask_ld);
        CertArgs cert{};
        cert.bound = d_bound1; cert.eps = c->eps2.as<float>(); cert.qnorm = d_qnorm; cert.threshold = p.threshold;
        cert.metric = c->metric; cert.status = status_of(c); cert.level = 1; cert.nq_total = p.nq;
        cert.dim = c->dim; cert.l2_slack = l2_rounding_slack(c->dim);
        final_kernel<<<g, SEL_THREADS, 0, st>>>(d_ex1, d_sel1_n, K1, k, c->rowids.as<int64_t>(), l2 ? 1 : 0, d_out_rowids, d_out_scores,
                                                d_out_counts, d_out_flags, l2 ? INFINITY : -INFINITY, d_qmap, cert);
        YB_CUDA(cudaGetLastError());
        YB_CUDA(cudaStreamSynchronize(st));  // d_qmap / bad reuse
    }
    // level 2 for what is left
    uint32_t n_bad2 = 0;
    YB_CUDA(cudaMemcpyAsync(&n_bad2, &status_of(c)->n_bad2, 4, cudaMemcpyDeviceToHost, st));
    YB_CUDA(cudaStreamSynchronize(st));
    if (n_bad2) {
        n_bad2 = std::min(n_bad2, p.nq);
        std::vector<uint32_t> bad2(n_bad2);
        const uint32_t* d_list2 = reinterpret_cast<const uint32_t*>(status_of(c) + 1) + p.nq;
        YB_CUDA(cudaMemcpyAsync(bad2.data(), d_list2, (size_t)n_bad2 * 4, cudaMemcpyDeviceToHost, st));
        YB_CUDA(cudaStreamSynchronize(st));
        for (uint32_t q : bad2)
            if ((rc = exact_all_rows(c, p, q, d_out_rowids, d_out_scores, d_out_counts, d_out_flags)) != YAMS_OK) return rc;
    }
    return YAMS_OK;
}

}  // namespace yb

using namespace yb;

template <typename UNIT>
static yams_status_t compact_array(Corpus* c, void* base, uint64_t row_bytes, const uint32_t* d_keep, const uint32_t* d_dst,
                                   DevBuf& tmp) {
    const uint64_t units = row_bytes / sizeof(UNIT);
    // batches of <= 256 MiB: destinations never pass sources, so batch i only overwrites rows that batches <= i
    // have already moved (or staged in tmp)
    uint64_t batch = std::max<uint64_t>(1, (256ull << 20) / row_bytes);
    yams_status_t rc = tmp.reserve((size_t)std::min<uint64_t>(batch, c->n) * row_bytes);
    if (rc != YAMS_OK) return rc;
    for (uint64_t b0 = 0; b0 < c->n; b0 += batch) {
        uint64_t b1 = std::min<uint64_t>(c->n, b0 + batch);
        unsigned grid = (unsigned)(((b1 - b0) * 32 + 255) / 256);
        compact_gather_kernel<UNIT><<<grid, 256, 0, c->st>>>(static_cast<const UNIT*>(base), units, b0, b1, d_keep, d_dst, tmp.as<UNIT>());
        compact_scatter_kernel<UNIT><<<grid, 256, 0, c->st>>>(static_cast<UNIT*>(base), units, b0, b1, d_keep, d_dst, tmp.as<UNIT>());
    }
    YB_CUDA(cudaGetLastError());
    return YAMS_OK;
}

extern "C" {

yams_status_t yams_b200_corpus_create(void* self, uint32_t dim, int dtype, int metric, uint64_t capacity_hint,
                                      yams_b200_corpus** out) {
    YB_TRY
    (void)self;
    YB_ARG(out, "out is null");
    *out = nullptr;
    YB_ARG(dim > 0 && dim <= 65536, "dim must be in 1..65536");  // vec0_module.hpp:109
    YB_ARG(dtype == YAMS_B200_F32 || dtype == YAMS_B200_F16, "unknown dtype");
    YB_ARG(metric == YAMS_B200_COSINE || metric == YAMS_B200_L2, "unknown metric");
    DeviceCtx* dev = nullptr;
    yams_status_t rc = ensure_device(&dev);
    if (rc != YAMS_OK) return rc;
    yams_b200_corpus* c = new (std::nothrow) yams_b200_corpus();
    if (!c) return YAMS_ERR_INTERNAL;
    c->dev = dev;
    c->dim = dim;
    c->dtype = dtype;
    c->metric = metric;
    if (cudaStreamCreateWithFlags(&c->st, cudaStreamNonBlocking) != cudaSuccess) {
        delete c;
        set_last_error("cudaStreamCreate failed");
        return YAMS_ERR_INTERNAL;
    }
    for (auto& e : c->ev) cudaEventCreate(&e);
    for (auto& e : c->ev_scan) cudaEventCreate(&e);
    if (capacity_hint) {
        rc = corpus_reserve(c, capacity_hint);
        if (rc != YAMS_OK) {
            yams_b200_corpus_destroy(c);
            return rc;
        }
    }
    *out = c;
    return YAMS_OK;
    YB_CATCH
}

void yams_b200_corpus_destroy(yams_b200_corpus* c) {
    if (!c) return;
    if (c->st) cudaStreamSynchronize(c->st);
    for (DevBuf* b : {&c->rows, &c->rowids, &c->inv_norm, &c->q32, &c->q16, &c->qinv, &c->tau, &c->counts, &c->cands,
                      &c->sample_scores, &c->sel, &c->outbuf, &c->dense, &c->mask, &c->misc, &c->dout, &c->stats, &c->status,
                      &c->bound, &c->eps, &c->eps2, &c->lvl})
        b->release();
    c->h_pin.release();
    for (auto& e : c->ev)
        if (e) cudaEventDestroy(e);
    for (auto& e : c->ev_scan)
        if (e) cudaEventDestroy(e);
    if (c->st) cudaStreamDestroy(c->st);
    delete c;
}

yams_status_t yams_b200_corpus_append(yams_b200_corpus* c, const void* rows, uint64_t n, const int64_t* rowids) {
    YB_TRY
    YB_ARG(c, "corpus is null");
    std::lock_guard<std::mutex> corpus_lock(c->mu);
    YB_BIND(c);
    if (n == 0) return YAMS_OK;
    YB_ARG(rows, "rows is null");
    YB_ARG(c->n + n < 0xFFFFFFFFull, "corpus is limited to 2^32-1 rows per GPU");
    yams_status_t rc = corpus_reserve(c, c->n + n);
    if (rc != YAMS_OK) return rc;
    size_t rb = (size_t)c->dim * c->elem();
    YB_CUDA(cudaMemcpyAsync(c->rows.as<uint8_t>() + (size_t)c->n * rb, rows, (size_t)n * rb, cudaMemcpyHostToDevice, c->st));
    return corpus_finish_append(c, n, rowids);
    YB_CATCH
}

yams_status_t yams_b200_corpus_append_f32_as_f16(yams_b200_corpus* c, const float* rows, uint64_t n, const int64_t* rowids) {
    YB_TRY
    YB_ARG(c, "corpus is null");
    std::lock_guard<std::mutex> corpus_lock(c->mu);
    YB_BIND(c);
    YB_ARG(c->dtype == YAMS_B200_F16, "corpus is not fp16");
    if (n == 0) return YAMS_OK;
    YB_ARG(rows, "rows is null");
    YB_ARG(c->n + n < 0xFFFFFFFFull, "corpus is limited to 2^32-1 rows per GPU");
    yams_status_t rc = corpus_reserve(c, c->n + n);
    if (rc != YAMS_OK) return rc;
    size_t cnt = (size_t)n * c->dim;
    if ((rc = c->dense.reserve(cnt * 4)) != YAMS_OK) return rc;
    YB_CUDA(cudaMemcpyAsync(c->dense.p, rows, cnt * 4, cudaMemcpyHostToDevice, c->st));
    convert_f32_to_f16_trunc_kernel<<<(unsigned)std::min<size_t>((cnt + 255) / 256, 65535), 256, 0, c->st>>>(
        c->dense.as<float>(), c->rows.as<uint16_t>() + (size_t)c->n * c->dim, cnt);
    return corpus_finish_append(c, n, rowids);
    YB_CATCH
}

yams_status_t yams_b200_corpus_append_synthetic(yams_b200_corpus* c, uint64_t seed, uint64_t first_row, uint64_t n) {
    YB_TRY
    YB_ARG(c, "corpus is null");
    std::lock_guard<std::mutex> corpus_lock(c->mu);
    YB_BIND(c);
    if (n == 0) return YAMS_OK;
    YB_ARG(c->n + n < 0xFFFFFFFFull, "corpus is limited to 2^32-1 rows per GPU");
    yams_status_t rc = corpus_reserve(c, c->n + n);
    if (rc != YAMS_OK) return rc;
    if ((rc = c->misc.reserve((size_t)n * 4)) != YAMS_OK) return rc;
    float* d_inv = c->misc.as<float>();
    synth_rownorm_kernel<<<(unsigned)((n + 127) / 128), 128, 0, c->st>>>(seed, first_row, n, c->dim, d_inv);
    size_t rb = (size_t)c->dim * c->elem();
    synth_fill_kernel<<<c->dev->sm_count * 16, 256, 0, c->st>>>(seed, first_row, n, c->dim, d_inv,
                                                               c->rows.as<uint8_t>() + (size_t)c->n * rb, c->dtype);
    YB_CUDA(cudaGetLastError());
    // rowid = first_row + i
    return corpus_finish_append(c, n, nullptr, (int64_t)first_row);
    YB_CATCH
}

yams_status_t yams_b200_corpus_remove(yams_b200_corpus* c, const int64_t* rowids, uint64_t n, uint64_t* out_removed) {
    YB_TRY
    YB_ARG(c, "corpus is null");
    std::lock_guard<std::mutex> corpus_lock(c->mu);
    YB_BIND(c);
    if (out_removed) *out_removed = 0;
    if (n == 0 || c->n == 0) return YAMS_OK;
    YB_ARG(rowids, "rowids is null");
    yams_status_t rc;
    cudaStream_t st = c->st;
    if ((rc = c->mask.reserve((size_t)n * 8)) != YAMS_OK) return rc;
    if ((rc = c->sel.reserve((size_t)c->n * 4 + 16)) != YAMS_OK) return rc;
    if ((rc = c->outbuf.reserve((size_t)c->n * 4 + 16)) != YAMS_OK) return rc;
    if ((rc = c->tau.reserve(8)) != YAMS_OK) return rc;
    uint32_t* d_keep = c->sel.as<uint32_t>();
    uint32_t* d_dst = c->outbuf.as<uint32_t>();
    uint64_t* d_total = reinterpret_cast<uint64_t*>(c->tau.p);
    YB_CUDA(cudaMemcpyAsync(c->mask.p, rowids, (size_t)n * 8, cudaMemcpyHostToDevice, st));
    unsigned g = (unsigned)std::min<uint64_t>((c->n + 255) / 256, 65535);
    fill_u32_kernel<<<g, 256, 0, st>>>(d_keep, c->n, 1u);
    mark_removed_kernel<<<(unsigned)std::min<uint64_t>((n + 255) / 256, 65535), 256, 0, st>>>(c->mask.as<int64_t>(), n, c->rowids.as<int64_t>(),
                                                                                              c->n, d_keep);
    if ((rc = exclusive_scan_u32(d_keep, d_dst, c->n, d_total, c->misc, st)) != YAMS_OK) return rc;
    uint64_t kept = 0;
    YB_CUDA(cudaMemcpyAsync(&kept, d_total, 8, cudaMemcpyDeviceToHost, st));
    YB_CUDA(cudaStreamSynchronize(st));
    if (kept == c->n) return YAMS_OK;
    const uint64_t row_bytes = (uint64_t)c->dim * c->elem();
    if (row_bytes % 16 == 0) rc = compact_array<uint4>(c, c->rows.p, row_bytes, d_keep, d_dst, c->dense);
    else if (row_bytes % 4 == 0) rc = compact_array<uint32_t>(c, c->rows.p, row_bytes, d_keep, d_dst, c->dense);
    else rc = compact_array<uint16_t>(c, c->rows.p, row_bytes, d_keep, d_dst, c->dense);
    if (rc == YAMS_OK) rc = compact_array<uint64_t>(c, c->rowids.p, 8, d_keep, d_dst, c->dense);
    if (rc == YAMS_OK) rc = compact_array<uint32_t>(c, c->inv_norm.p, 4, d_keep, d_dst, c->dense);
    if (rc != YAMS_OK) return rc;
    int64_t last = INT64_MIN;
    if (kept) YB_CUDA(cudaMemcpyAsync(&last, c->rowids.as<int64_t>() + (kept - 1), 8, cudaMemcpyDeviceToHost, st));
    YB_CUDA(cudaStreamSynchronize(st));
    if (out_removed) *out_removed = c->n - kept;
    c->n = kept;
    ++c->generation;
    c->last_rowid = last;
    c->rowids_dense = false;
    return YAMS_OK;
    YB_CATCH
}

yams_status_t yams_b200_corpus_clear(yams_b200_corpus* c) {
    YB_ARG(c, "corpus is null");
    std::lock_guard<std::mutex> corpus_lock(c->mu);
    YB_BIND(c);
    c->n = 0;
    ++c->generation;
    c->last_rowid = INT64_MIN;
    c->rowids_dense = true;
    c->pending.active = false;
    c->r_max = c->dr_abs_max = c->dr_rel_max = 0.f;
    if (c->stats.p) YB_CUDA(cudaMemsetAsync(c->stats.p, 0, 16, c->st));
    return YAMS_OK;
}

yams_status_t yams_b200_corpus_size(const yams_b200_corpus* c, uint64_t* out_n) {
    YB_ARG(c && out_n, "null argument");
    *out_n = c->n;
    return YAMS_OK;
}

yams_status_t yams_b200_corpus_sync(yams_b200_corpus* c) {
    YB_ARG(c, "corpus is null");
    std::lock_guard<std::mutex> corpus_lock(c->mu);
    YB_BIND(c);
    YB_CUDA(cudaStreamSynchronize(c->st));
    return YAMS_OK;
}

void* yams_b200_corpus_stream(yams_b200_corpus* c) { return c ? (void*)c->st : nullptr; }

// uploads the queries and enqueues their preparation: q32, qinv, qnorm (misc) on the device, status block zeroed,
// invalid queries counted in status->n_invalid (read by the host together with the results -- no synchronisation here)
static yams_status_t prepare_queries(yams_b200_corpus* c, const float* q_src, bool src_is_device, uint32_t nq) {
    yams_status_t rc;
    size_t qb = (size_t)nq * c->dim * 4;
    if ((rc = c->q32.reserve(qb)) != YAMS_OK) return rc;
    if ((rc = c->qinv.reserve((size_t)nq * 4)) != YAMS_OK) return rc;
    if ((rc = c->misc.reserve((size_t)nq * 8 + (size_t)nq * 4)) != YAMS_OK) return rc;
    if ((rc = c->counts.reserve((size_t)nq * 4)) != YAMS_OK) return rc;
    if ((rc = c->status.reserve(sizeof(ScanStatus) + (size_t)nq * 8)) != YAMS_OK) return rc;
    if ((rc = c->h_pin.reserve(sizeof(ScanStatus) + (size_t)nq * 8 + 64)) != YAMS_OK) return rc;
    YB_CUDA(cudaMemsetAsync(c->status.p, 0, sizeof(ScanStatus), c->st));
    YB_CUDA(cudaMemcpyAsync(c->q32.p, q_src, qb, src_is_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, c->st));
    double* d_qnorm = reinterpret_cast<double*>(c->misc.as<uint8_t>());
    query_prep_kernel<<<(nq + QP_THREADS - 1) / QP_THREADS, QP_THREADS, 0, c->st>>>(c->q32.as<float>(), nq, c->dim, d_qnorm, c->qinv.as<float>(), c->metric,
                                                        status_of(c));
    YB_CUDA(cudaGetLastError());
    return YAMS_OK;
}

// After the stream has been synchronised: the status block of the call (pinned copy) -> invalid queries are an error,
// uncertain queries are resolved by the exhaustive levels (results patched in the device output buffers).
static yams_status_t finish_scan(yams_b200_corpus* c, const ScanPlan& p, int64_t* d_or, float* d_os, uint32_t* d_oc, uint64_t* d_of,
                                 uint32_t* out_resolved) {
    const ScanStatus* hs = c->h_pin.as<ScanStatus>();
    if (out_resolved) *out_resolved = 0;
    YB_ARG(hs->n_invalid == 0, "exact vector search requires a finite, non-zero query embedding");
    uint32_t n_bad = std::min(hs->n_bad, p.nq);
    if (n_bad == 0) return YAMS_OK;
    std::vector<uint32_t> bad(reinterpret_cast<const uint32_t*>(hs + 1), reinterpret_cast<const uint32_t*>(hs + 1) + n_bad);
    std::sort(bad.begin(), bad.end());
    if (out_resolved) *out_resolved = n_bad;
    return resolve_uncertain(c, p, bad.data(), n_bad, d_or, d_os, d_oc, d_of);
}
static yams_status_t enqueue_status_readback(yams_b200_corpus* c, uint32_t nq) {
    YB_CUDA(cudaMemcpyAsync(c->h_pin.p, c->status.p, sizeof(ScanStatus) + (size_t)nq * 4, cudaMemcpyDeviceToHost, c->st));
    return YAMS_OK;
}

yams_status_t yams_b200_search(yams_b200_corpus* c, const float* queries, uint32_t nq, uint32_t k, float threshold,
                               const int64_t* allowed_rowids, const uint64_t* allowed_offsets, int64_t* out_rowids,
                               float* out_scores, uint32_t* out_counts, uint64_t* out_flags) {
    YB_TRY
    YB_ARG(c, "corpus is null");
    std::lock_guard<std::mutex> corpus_lock(c->mu);
    YB_BIND(c);
    if (nq == 0) return YAMS_OK;
    YB_ARG(queries && out_counts, "null argument");
    YB_ARG(!allowed_rowids || allowed_offsets, "allowed_offsets missing");
    YB_ARG(!allowed_offsets || allowed_rowids || allowed_offsets[nq] == 0, "allowed_rowids missing");
    for (uint32_t q = 0; q < nq; ++q) out_counts[q] = 0;
    if (out_flags) for (uint32_t q = 0; q < nq; ++q) out_flags[q] = 0;
    yams_status_t rc;
    cudaEvent_t w0 = c->ev[3];
    YB_CUDA(cudaEventRecord(w0, c->st));
    // the reference looks at k before it validates the query (sqlite_vec_backend.cpp:4123-4130: k == 0 returns
    // empty first): mirror that order
    if (k == 0) return YAMS_OK;
    YB_ARG(out_rowids && out_scores, "null output");
    YB_ARG(k <= kMaxK, "k > 3072 is not supported by the fused top-k path (page larger requests)");
    YB_ARG(nq <= 65535, "at most 65535 queries per call (split larger batches)");   // per-query grid dimensions
    YB_ARG(!allowed_offsets || c->metric == YAMS_B200_COSINE, "candidate sets are only supported for the cosine metric");
    c->pending.active = false;
    if ((rc = prepare_queries(c, queries, false, nq)) != YAMS_OK) return rc;
    YB_CUDA(cudaEventRecord(c->ev[0], c->st));
    // device outputs
    size_t ob = (size_t)nq * k * 12 + (size_t)nq * 4 + (size_t)nq * 8 + 64;
    DevBuf& dout = c->dout;
    if ((rc = dout.reserve(ob)) != YAMS_OK) return rc;
    int64_t* d_or = dout.as<int64_t>();
    uint64_t* d_of = reinterpret_cast<uint64_t*>(d_or + (size_t)nq * k);
    float* d_os = reinterpret_cast<float*>(d_of + nq);
    uint32_t* d_oc = reinterpret_cast<uint32_t*>(d_os + (size_t)nq * k);
    ScanPlan plan;
    plan.nq = nq; plan.k = k; plan.threshold = threshold;
    plan.use_tensor = tcgen05_supported(c, nq);
    DirectLists lists;
    bool direct = false;
    if (allowed_offsets && c->n) {
        // small ascending lists: score the listed rows directly instead of passing over the corpus.  Break-even
        // (DESIGN.md §4.4): a corpus pass costs ~max(1, nq/400) row reads per row, a gathered row about two.
        const uint64_t total = allowed_offsets[nq];
        direct = total <= std::max<uint64_t>(c->n / 2, c->n / 400 * nq) && total < (1ull << 31);
        for (uint32_t q = 0; q < nq && direct; ++q) {
            uint64_t lo = allowed_offsets[q], hi = allowed_offsets[q + 1];
            direct = hi >= lo && hi - lo < 0xFFFFFFFFull;
            for (uint64_t i = lo + 1; i < hi && direct; ++i) direct = allowed_rowids[i - 1] <= allowed_rowids[i];
            if (direct) lists.max_len = std::max<uint32_t>(lists.max_len, (uint32_t)(hi - lo));
        }
    }
    if (direct) {
        const uint64_t total = allowed_offsets[nq];
        if ((rc = c->mask.reserve((size_t)total * 8 + (size_t)(nq + 1) * 8 + 64)) != YAMS_OK) return rc;
        int64_t* d_allowed = c->mask.as<int64_t>();
        uint64_t* d_offs = reinterpret_cast<uint64_t*>(d_allowed + total);
        if (total) YB_CUDA(cudaMemcpyAsync(d_allowed, allowed_rowids, (size_t)total * 8, cudaMemcpyHostToDevice, c->st));
        YB_CUDA(cudaMemcpyAsync(d_offs, allowed_offsets, (size_t)(nq + 1) * 8, cudaMemcpyHostToDevice, c->st));
        lists.d_allowed = d_allowed;
        lists.d_offsets = d_offs;
        lists.total = total;
        plan.direct = &lists;
    } else if (allowed_offsets && c->n) {
        uint64_t total = allowed_offsets[nq];
        uint64_t mask_ld = (c->n + 31) / 32;
        size_t mb = (size_t)nq * mask_ld * 4;
        if ((rc = c->mask.reserve(mb + (size_t)total * 8 + (size_t)(nq + 1) * 8 + 64)) != YAMS_OK) return rc;
        uint32_t* dm = c->mask.as<uint32_t>();
        int64_t* d_allowed = reinterpret_cast<int64_t*>(c->mask.as<uint8_t>() + ((mb + 7) & ~(size_t)7));
        uint64_t* d_offs = reinterpret_cast<uint64_t*>(d_allowed + total);
        YB_CUDA(cudaMemsetAsync(dm, 0, mb, c->st));
        if (total) YB_CUDA(cudaMemcpyAsync(d_allowed, allowed_rowids, (size_t)total * 8, cudaMemcpyHostToDevice, c->st));
        YB_CUDA(cudaMemcpyAsync(d_offs, allowed_offsets, (size_t)(nq + 1) * 8, cudaMemcpyHostToDevice, c->st));
        dim3 grid(64, nq);
        build_mask_kernel<<<grid, 256, 0, c->st>>>(d_allowed, d_offs, nq, c->rowids.as<int64_t>(), c->n, dm, mask_ld);
        plan.d_mask = dm;
        plan.mask_ld = mask_ld;
    }
    if ((rc = scan_enqueue(c, plan, d_or, d_os, d_oc, d_of)) != YAMS_OK) return rc;
    cudaEventRecord(c->ev[2], c->st);
    if ((rc = enqueue_status_readback(c, nq)) != YAMS_OK) return rc;
    auto copy_out = [&]() -> cudaError_t {
        cudaError_t e = cudaMemcpyAsync(out_rowids, d_or, (size_t)nq * k * 8, cudaMemcpyDeviceToHost, c->st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(out_scores, d_os, (size_t)nq * k * 4, cudaMemcpyDeviceToHost, c->st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(out_counts, d_oc, (size_t)nq * 4, cudaMemcpyDeviceToHost, c->st);
        if (e == cudaSuccess && out_flags) e = cudaMemcpyAsync(out_flags, d_of, (size_t)nq * 8, cudaMemcpyDeviceToHost, c->st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->st);
        return e;
    };
    cudaError_t e = copy_out();
    if (e != cudaSuccess) {
        set_last_error("search failed: %s", cudaGetErrorString(e));
        return YAMS_ERR_INTERNAL;
    }
    cudaEventElapsedTime(&c->last_ms[0], c->ev[0], c->ev[1]);
    cudaEventElapsedTime(&c->last_ms[1], c->ev[1], c->ev[2]);
    cudaEventElapsedTime(&c->last_ms[2], c->ev[0], c->ev[2]);
    c->last_ms[4] = plan.use_tensor ? 1.f : 0.f;
    uint32_t resolved = 0;
    rc = finish_scan(c, plan, d_or, d_os, d_oc, d_of, &resolved);
    c->last_ms[6] = (float)resolved;
    if (rc != YAMS_OK) {
        for (uint32_t q = 0; q < nq; ++q) out_counts[q] = 0;
        return rc;
    }
    if (resolved && (e = copy_out()) != cudaSuccess) {
        set_last_error("search failed: %s", cudaGetErrorString(e));
        return YAMS_ERR_INTERNAL;
    }
    return YAMS_OK;
    YB_CATCH
}

// The full exact pass (level 2 of the fallback chain) for EVERY query: the reference's own loop evaluated for all rows,
// no stage 1, no thresholds, no certificate needed.  It is what bench.py and the tests check the fast path against at
// sizes the CPU oracle cannot reach; ~3 ms per query per 10 M rows.
yams_status_t yams_b200_search_exhaustive(yams_b200_corpus* c, const float* queries, uint32_t nq, uint32_t k, float threshold,
                                          int64_t* out_rowids, float* out_scores, uint32_t* out_counts, uint64_t* out_flags) {
    YB_TRY
    YB_ARG(c, "corpus is null");
    std::lock_guard<std::mutex> corpus_lock(c->mu);
    YB_BIND(c);
    if (nq == 0) return YAMS_OK;
    YB_ARG(queries && out_counts && out_rowids && out_scores, "null argument");
    YB_ARG(k > 0 && k <= kMaxK, "k must be in 1..3072");
    YB_ARG(nq <= 65535, "at most 65535 queries per call");
    yams_status_t rc;
    c->pending.active = false;
    if ((rc = prepare_queries(c, queries, false, nq)) != YAMS_OK) return rc;
    size_t ob = (size_t)nq * k * 12 + (size_t)nq * 4 + (size_t)nq * 8 + 64;
    if ((rc = c->dout.reserve(ob)) != YAMS_OK) return rc;
    int64_t* d_or = c->dout.as<int64_t>();
    uint64_t* d_of = reinterpret_cast<uint64_t*>(d_or + (size_t)nq * k);
    float* d_os = reinterpret_cast<float*>(d_of + nq);
    uint32_t* d_oc = reinterpret_cast<uint32_t*>(d_os + (size_t)nq * k);
    if ((rc = enqueue_status_readback(c, 0)) != YAMS_OK) return rc;
    YB_CUDA(cudaStreamSynchronize(c->st));
    YB_ARG(c->h_pin.as<ScanStatus>()->n_invalid == 0, "exact vector search requires a finite, non-zero query embedding");
    ScanPlan plan;
    plan.nq = nq; plan.k = k; plan.threshold = threshold;
    for (uint32_t q = 0; q < nq; ++q)
        if ((rc = exact_all_rows(c, plan, q, d_or, d_os, d_oc, d_of)) != YAMS_OK) return rc;
    YB_CUDA(cudaMemcpyAsync(out_rowids, d_or, (size_t)nq * k * 8, cudaMemcpyDeviceToHost, c->st));
    YB_CUDA(cudaMemcpyAsync(out_scores, d_os, (size_t)nq * k * 4, cudaMemcpyDeviceToHost, c->st));
    YB_CUDA(cudaMemcpyAsync(out_counts, d_oc, (size_t)nq * 4, cudaMemcpyDeviceToHost, c->st));
    if (out_flags) YB_CUDA(cudaMemcpyAsync(out_flags, d_of, (size_t)nq * 8, cudaMemcpyDeviceToHost, c->st));
    YB_CUDA(cudaStreamSynchronize(c->st));
    return YAMS_OK;
    YB_CATCH
}

yams_status_t yams_b200_search_all_matching(yams_b200_corpus* c, const float* query, float threshold,
                                            const int64_t* allowed_rowids, uint64_t n_allowed, int64_t* out_rowids,
                                            float* out_scores, uint64_t* out_count) {
    YB_TRY
    YB_ARG(c && query && out_count, "null argument");
    std::lock_guard<std::mutex> corpus_lock(c->mu);
    YB_BIND(c);
    *out_count = 0;
    c->pending.active = false;
    YB_ARG(c->metric == YAMS_B200_COSINE, "all-matching selection is defined for the cosine scan");
    // the reference gathers the candidate rowids into a set (:4412-4448): duplicates count once
    std::vector<int64_t> uniq;
    if (allowed_rowids) {
        bool ascending = true;
        for (uint64_t i = 1; i < n_allowed && ascending; ++i) ascending = allowed_rowids[i - 1] < allowed_rowids[i];
        if (!ascending) {
            uniq.assign(allowed_rowids, allowed_rowids + n_allowed);
            std::sort(uniq.begin(), uniq.end());
            uniq.erase(std::unique(uniq.begin(), uniq.end()), uniq.end());
            allowed_rowids = uniq.data();
            n_allowed = uniq.size();
        }
    }
    const uint64_t m = allowed_rowids ? n_allowed : c->n;
    yams_status_t rc;
    if ((rc = prepare_queries(c, query, false, 1)) != YAMS_OK) return rc;
    if ((rc = enqueue_status_readback(c, 0)) != YAMS_OK) return rc;
    YB_CUDA(cudaStreamSynchronize(c->st));
    YB_ARG(c->h_pin.as<ScanStatus>()->n_invalid == 0,
           "exact vector search requires a finite, non-zero query embedding");   // InvalidArgument for a bad query (:4127)
    if (m == 0 || c->n == 0) return YAMS_OK;
    YB_ARG(out_rowids && out_scores, "null output");
    YB_ARG(m < (1ull << 31), "candidate set too large");
    cudaStream_t st = c->st;
    uint64_t np2 = 1;
    while (np2 < m) np2 <<= 1;
    if ((rc = c->sel.reserve((size_t)m * sizeof(Cand) + 16)) != YAMS_OK) return rc;
    if ((rc = c->outbuf.reserve((size_t)m * sizeof(Exact))) != YAMS_OK) return rc;
    if ((rc = c->dense.reserve((size_t)np2 * 8 + (size_t)m * 12 + 64)) != YAMS_OK) return rc;
    if ((rc = c->mask.reserve((size_t)m * 8 + 64)) != YAMS_OK) return rc;
    Cand* d_sel = c->sel.as<Cand>();
    uint64_t* d_keys = c->dense.as<uint64_t>();
    int64_t* d_or = reinterpret_cast<int64_t*>(d_keys + np2);
    float* d_os = reinterpret_cast<float*>(d_or + m);
    unsigned g = (unsigned)std::min<uint64_t>((np2 + 255) / 256, 65535);
    if (allowed_rowids) {
        int64_t* d_allowed = c->mask.as<int64_t>();
        YB_CUDA(cudaMemcpyAsync(d_allowed, allowed_rowids, (size_t)m * 8, cudaMemcpyHostToDevice, st));
        map_rowids_kernel<<<g, 256, 0, st>>>(d_allowed, m, c->rowids.as<int64_t>(), c->n, d_sel);
    } else {
        iota_sel_kernel<<<g, 256, 0, st>>>(d_sel, m);
    }
    // one "query" with Kp = m survivors: exact re-scoring of every candidate
    uint32_t* d_seln = c->counts.as<uint32_t>();
    uint32_t mm = (uint32_t)m;
    YB_CUDA(cudaMemcpyAsync(d_seln, &mm, 4, cudaMemcpyHostToDevice, st));
    double* d_qnorm = reinterpret_cast<double*>(c->misc.as<uint8_t>());
    rescore_kernel<<<(unsigned)((m + 127) / 128), 128, 0, st>>>(c->rows.p, c->dtype, c->dim, c->q32.as<float>(), d_qnorm, d_sel, d_seln,
                                                               (uint32_t)m, 1, threshold, c->outbuf.as<Exact>(), YAMS_B200_COSINE, nullptr,
                                                               nullptr, 0);
    exact_keys_kernel<<<g, 256, 0, st>>>(c->outbuf.as<Exact>(), m, np2, d_keys);
    for (uint64_t size = 2; size <= np2; size <<= 1)
        for (uint64_t stride = size >> 1; stride > 0; stride >>= 1) bitonic_step_kernel<<<g, 256, 0, st>>>(d_keys, np2, size, stride);
    if ((rc = c->tau.reserve(8)) != YAMS_OK) return rc;
    unsigned long long* d_cnt = reinterpret_cast<unsigned long long*>(c->tau.p);
    YB_CUDA(cudaMemsetAsync(d_cnt, 0, 8, st));
    count_nonzero_kernel<<<g, 256, 0, st>>>(d_keys, np2, d_cnt);
    unsigned long long h_cnt = 0;
    YB_CUDA(cudaMemcpyAsync(&h_cnt, d_cnt, 8, cudaMemcpyDeviceToHost, st));
    YB_CUDA(cudaStreamSynchronize(st));
    if (h_cnt) {
        unpack_sim_keys_kernel<<<g, 256, 0, st>>>(d_keys, h_cnt, c->rowids.as<int64_t>(), d_or, d_os);
        YB_CUDA(cudaMemcpyAsync(out_rowids, d_or, (size_t)h_cnt * 8, cudaMemcpyDeviceToHost, st));
        YB_CUDA(cudaMemcpyAsync(out_scores, d_os, (size_t)h_cnt * 4, cudaMemcpyDeviceToHost, st));
        YB_CUDA(cudaStreamSynchronize(st));
    }
    *out_count = h_cnt;
    return YAMS_OK;
    YB_CATCH
}

yams_status_t yams_b200_search_device(yams_b200_corpus* c, const float* d_queries, uint32_t nq, uint32_t k, float threshold,
                                      int64_t* d_out_rowids, float* d_out_scores) {
    YB_TRY
    YB_ARG(c && d_queries && d_out_rowids && d_out_scores, "null argument");
    std::lock_guard<std::mutex> corpus_lock(c->mu);
    YB_BIND(c);
    YB_ARG(k > 0 && k <= 768, "k must be in 1..768");
    YB_ARG(nq <= 65535, "at most 65535 queries per call (split larger batches)");
    if (nq == 0) return YAMS_OK;
    yams_status_t rc;
    c->pending.active = false;
    if ((rc = prepare_queries(c, d_queries, true, nq)) != YAMS_OK) return rc;
    YB_CUDA(cudaEventRecord(c->ev[0], c->st));
    ScanPlan plan;
    plan.nq = nq; plan.k = k; plan.threshold = threshold;
    plan.use_tensor = tcgen05_supported(c, nq);
    if ((rc = scan_enqueue(c, plan, d_out_rowids, d_out_scores, nullptr, nullptr)) != YAMS_OK) return rc;
    YB_CUDA(cudaEventRecord(c->ev[2], c->st));
    if ((rc = enqueue_status_readback(c, nq)) != YAMS_OK) return rc;
    c->last_ms[4] = plan.use_tensor ? 1.f : 0.f;
    c->pending.active = true;
    c->pending.nq = nq;
    c->pending.k = k;
    c->pending.threshold = threshold;
    c->pending.d_out_rowids = d_out_rowids;
    c->pending.d_out_scores = d_out_scores;
    return YAMS_OK;
    YB_CATCH
}

yams_status_t yams_b200_search_device_finish(yams_b200_corpus* c, uint32_t* out_resolved) {
    YB_TRY
    YB_ARG(c, "corpus is null");
    std::lock_guard<std::mutex> corpus_lock(c->mu);
    YB_BIND(c);
    if (out_resolved) *out_resolved = 0;
    if (!c->pending.active) return YAMS_OK;
    YB_CUDA(cudaStreamSynchronize(c->st));
    c->pending.active = false;
    ScanPlan plan;
    plan.nq = c->pending.nq; plan.k = c->pending.k; plan.threshold = c->pending.threshold;
    return finish_scan(c, plan, c->pending.d_out_rowids, c->pending.d_out_scores, nullptr, nullptr, out_resolved);
    YB_CATCH
}

static yams_status_t merge_launch(yams_b200_corpus* c, const int64_t* d_rowids, const float* d_scores, uint64_t rank_stride_r,
                                  uint64_t rank_stride_s, uint32_t nranks, uint32_t nq, uint32_t k, int64_t* d_out_rowids,
                                  float* d_out_scores, uint32_t* d_out_counts, cudaStream_t st) {
    YB_ARG(nranks >= 1 && k >= 1, "bad shape");
    uint32_t total = nranks * k, np2 = 1;
    while (np2 < total) np2 <<= 1;
    YB_ARG(np2 <= 4096, "nranks * k too large to merge in one CTA");
    size_t smem = (((size_t)np2 * 4 + 7) & ~(size_t)7) + (size_t)np2 * 8;
    merge_partials_kernel<<<nq, SEL_THREADS, smem, st>>>(d_rowids, d_scores, rank_stride_r, rank_stride_s, nranks, nq, k,
                                                         c->metric == YAMS_B200_L2, d_out_rowids, d_out_scores, d_out_counts);
    YB_CUDA(cudaGetLastError());
    return YAMS_OK;
}

yams_status_t yams_b200_merge_partials_device(yams_b200_corpus* c, const int64_t* d_rowids, const float* d_scores,
                                              uint32_t nranks, uint32_t nq, uint32_t k, int64_t* d_out_rowids,
                                              float* d_out_scores, uint32_t* d_out_counts) {
    YB_ARG(c && d_rowids && d_scores && d_out_rowids && d_out_scores, "null argument");
    std::lock_guard<std::mutex> corpus_lock(c->mu);
    YB_BIND(c);
    return merge_launch(c, d_rowids, d_scores, (uint64_t)nq * k, (uint64_t)nq * k, nranks, nq, k, d_out_rowids, d_out_scores,
                        d_out_counts, c->st);
}

yams_status_t yams_b200_merge_packed_device(yams_b200_corpus* c, const void* d_packed, uint32_t nranks, uint32_t nq, uint32_t k,
                                            int64_t* d_out_rowids, float* d_out_scores, uint32_t* d_out_counts, void* stream) {
    YB_ARG(c && d_packed && d_out_rowids && d_out_scores, "null argument");
    YB_BIND(c);
    // one rank's record: [nq*k int64 rowids][nq*k float scores] = 12 * nq * k bytes
    const uint8_t* base = static_cast<const uint8_t*>(d_packed);
    const uint64_t rec = (uint64_t)nq * k * 12;
    YB_ARG(rec % 8 == 0, "nq * k must be even for the packed layout");
    return merge_launch(c, reinterpret_cast<const int64_t*>(base), reinterpret_cast<const float*>(base + (uint64_t)nq * k * 8),
                        rec / 8, rec / 4, nranks, nq, k, d_out_rowids, d_out_scores, d_out_counts,
                        stream ? static_cast<cudaStream_t>(stream) : c->st);
}

yams_status_t yams_b200_search_last_timings(yams_b200_corpus* c, float out_ms[8]) {
    YB_ARG(c && out_ms, "null argument");
    if (cudaEventQuery(c->ev[2]) == cudaSuccess) {
        cudaEventElapsedTime(&c->last_ms[0], c->ev[0], c->ev[1]);
        cudaEventElapsedTime(&c->last_ms[1], c->ev[1], c->ev[2]);
        cudaEventElapsedTime(&c->last_ms[2], c->ev[0], c->ev[2]);
        c->last_ms[5] = 0.f;
        if (c->scan_timed) cudaEventElapsedTime(&c->last_ms[5], c->ev_scan[0], c->ev_scan[1]);
    }
    for (int i = 0; i < 8; ++i) out_ms[i] = c->last_ms[i];
    return YAMS_OK;
}

// diagnostics: dense stage-1 scores of rows [row_start + i*row_stride, i < nrows) against the queries with the
// chosen engine (0 cuda-core, 1 tcgen05) -> out[q * nrows + i] (HOST). Used by the tests to compare engines.
yams_status_t yams_b200_debug_stage1_scores(yams_b200_corpus* c, const float* queries, uint32_t nq, int engine,
                                            uint64_t row_start, uint64_t row_stride, uint64_t nrows, float* out) {
    YB_ARG(c && queries && out && nq > 0 && nrows > 0 && row_stride > 0, "bad argument");
    std::lock_guard<std::mutex> corpus_lock(c->mu);
    YB_ARG(row_start + (nrows - 1) * row_stride < c->n, "rows out of range");
    yams_status_t rc;
    YB_BIND(c);
    c->pending.active = false;
    if ((rc = prepare_queries(c, queries, false, nq)) != YAMS_OK) return rc;
    if ((rc = c->dense.reserve((size_t)nq * nrows * 4)) != YAMS_OK) return rc;
    if ((rc = c->eps.reserve((size_t)nq * 4)) != YAMS_OK) return rc;
    YB_CUDA(cudaMemsetAsync(c->dense.p, 0xFF, (size_t)nq * nrows * 4, c->st));
    Stage1Args a{};
    fill_stage1_common(c, a, nq);
    a.row_start = row_start; a.row_stride = row_stride; a.nrows = nrows;
    a.out_scores = c->dense.as<float>(); a.ld = nrows;
    if (engine == 1) {
        rc = stage1_tcgen05(c, a, false, c->st);
    } else {
        rc = stage1_cuda_core(a, false, c->st);
        eps_cc_kernel<<<(nq + 255) / 256, 256, 0, c->st>>>(reinterpret_cast<double*>(c->misc.as<uint8_t>()), nq, c->dim, c->metric, c->r_max,
                                                           c->eps.as<float>(), 0);
    }
    if (rc != YAMS_OK) return rc;
    YB_CUDA(cudaMemcpyAsync(out, c->dense.p, (size_t)nq * nrows * 4, cudaMemcpyDeviceToHost, c->st));
    YB_CUDA(cudaStreamSynchronize(c->st));
    return YAMS_OK;
}

// bench / test utility: n synthetic rows of the SURVEY.md §8d generator (bit-identical to oracle yo_gen_rows_f32) as fp32
// into a DEVICE buffer -- the query batches of bench.py are produced by the library itself, not by the checker
yams_status_t yams_b200_synth_rows_device(uint64_t seed, uint64_t first_row, uint64_t n, uint32_t dim, float* d_out) {
    YB_TRY
    YB_ARG(d_out && dim > 0, "bad argument");
    if (n == 0) return YAMS_OK;
    DeviceCtx* dev = nullptr;
    yams_status_t rc = ensure_device(&dev);
    if (rc != YAMS_OK) return rc;
    float* d_inv = nullptr;
    YB_CUDA(cudaMalloc(&d_inv, (size_t)n * 4));
    synth_rownorm_kernel<<<(unsigned)((n + 127) / 128), 128>>>(seed, first_row, n, dim, d_inv);
    synth_fill_kernel<<<dev->sm_count * 16, 256>>>(seed, first_row, n, dim, d_inv, d_out, YAMS_B200_F32);
    cudaError_t e = cudaDeviceSynchronize();
    cudaFree(d_inv);
    if (e != cudaSuccess) {
        set_last_error("synth_rows_device failed: %s", cudaGetErrorString(e));
        return YAMS_ERR_INTERNAL;
    }
    return YAMS_OK;
    YB_CATCH
}

// diagnostics: the per-query stage-1 error bound eps[q] (certificate input) computed by the last search /
// debug_stage1_scores call on this corpus
yams_status_t yams_b200_debug_last_eps(yams_b200_corpus* c, uint32_t nq, float* out) {
    YB_ARG(c && out && nq > 0, "bad argument");
    std::lock_guard<std::mutex> corpus_lock(c->mu);
    YB_BIND(c);
    YB_ARG(c->eps.cap >= (size_t)nq * 4, "no search with that many queries has run");
    YB_CUDA(cudaMemcpyAsync(out, c->eps.p, (size_t)nq * 4, cudaMemcpyDeviceToHost, c->st));
    YB_CUDA(cudaStreamSynchronize(c->st));
    return YAMS_OK;
}

yams_status_t yams_b200_vec0_exact(void* self, const float* query, uint32_t dim, const float* rows, const int64_t* rowids,
                                   uint64_t n, uint64_t k, int use_range, int64_t rowid_lo, int64_t rowid_hi,
                                   int64_t* out_rowids, float* out_dist, uint64_t* out_count) {
    YB_TRY
    (void)self;
    YB_ARG(out_count, "out_count is null");
    *out_count = 0;
    YB_ARG(query && dim > 0, "bad query");
    if (n == 0) return YAMS_OK;
    YB_ARG(rows && out_rowids && out_dist, "null argument");
    YB_ARG(n < 0xFFFFFFFFull, "too many rows");
    yams_status_t rc = YAMS_OK;
    // rowid range filter (vec0_module.hpp:399-401) is applied on the host side of the copy: only rows in
    // range are uploaded (pure data movement, no arithmetic)
    std::vector<uint32_t> keep;
    if (use_range) {
        keep.reserve((size_t)n);
        for (uint64_t i = 0; i < n; ++i) {
            int64_t rid = rowids ? rowids[i] : (int64_t)i;
            if (rid >= rowid_lo && rid <= rowid_hi) keep.push_back((uint32_t)i);
        }
        if (keep.empty()) return YAMS_OK;
    }
    uint64_t m = use_range ? keep.size() : n;
    OpWsLease lease;
    if (!lease.w) return YAMS_ERR_INTERNAL;
    cudaStream_t st = lease.w->st;
    uint64_t np2 = 1;
    while (np2 < m) np2 <<= 1;
    DevBuf &d_rows = lease.w->d[0], &d_q = lease.w->d[1], &d_dist = lease.w->d[2], &d_keys = lease.w->d[3], &d_rid = lease.w->d[4],
           &d_or = lease.w->d[5], &d_od = lease.w->d[6];
    rc = d_rows.reserve((size_t)m * dim * 4);
    if (rc == YAMS_OK) rc = d_q.reserve((size_t)dim * 4);
    if (rc == YAMS_OK) rc = d_dist.reserve((size_t)m * 4);
    if (rc == YAMS_OK) rc = d_keys.reserve((size_t)np2 * 8);
    if (rc == YAMS_OK) rc = d_rid.reserve((size_t)m * 8);
    if (rc == YAMS_OK) rc = d_or.reserve((size_t)m * 8);
    if (rc == YAMS_OK) rc = d_od.reserve((size_t)m * 4);
    if (rc == YAMS_OK) {
        std::vector<int64_t> rid_h((size_t)m);
        std::vector<float> packed;   // rows passing the rowid range, packed on the host: one copy instead of one per row
        if (use_range) {
            packed.resize((size_t)m * dim);
            for (uint64_t j = 0; j < m; ++j) {
                memcpy(packed.data() + (size_t)j * dim, rows + (size_t)keep[j] * dim, (size_t)dim * 4);
                rid_h[j] = rowids ? rowids[keep[j]] : (int64_t)keep[j];
            }
            cudaMemcpyAsync(d_rows.p, packed.data(), (size_t)m * dim * 4, cudaMemcpyHostToDevice, st);
        } else {
            cudaMemcpyAsync(d_rows.p, rows, (size_t)m * dim * 4, cudaMemcpyHostToDevice, st);
            for (uint64_t j = 0; j < m; ++j) rid_h[j] = rowids ? rowids[j] : (int64_t)j;
        }
        cudaMemcpyAsync(d_rid.p, rid_h.data(), (size_t)m * 8, cudaMemcpyHostToDevice, st);
        cudaMemcpyAsync(d_q.p, query, (size_t)dim * 4, cudaMemcpyHostToDevice, st);
        batch_dist_kernel<<<(unsigned)((m + 127) / 128), 128, 0, st>>>(d_rows.as<float>(), dim, m, d_q.as<float>(), YAMS_B200_L2, d_dist.as<float>());
        unsigned g = (unsigned)std::min<uint64_t>((np2 + 255) / 256, 65535);
        make_keys_kernel<<<g, 256, 0, st>>>(d_dist.as<float>(), m, np2, d_keys.as<uint64_t>());
        for (uint64_t size = 2; size <= np2; size <<= 1)
            for (uint64_t stride = size >> 1; stride > 0; stride >>= 1)
                bitonic_step_kernel<<<g, 256, 0, st>>>(d_keys.as<uint64_t>(), np2, size, stride);
        uint64_t outn = (k && k < m) ? k : m;
        unpack_keys_kernel<<<g, 256, 0, st>>>(d_keys.as<uint64_t>(), outn, d_rid.as<int64_t>(), d_or.as<int64_t>(), d_od.as<float>());
        cudaError_t e = cudaMemcpyAsync(out_rowids, d_or.p, (size_t)outn * 8, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(out_dist, d_od.p, (size_t)outn * 4, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) {
            set_last_error("vec0_exact failed: %s", cudaGetErrorString(e));
            rc = YAMS_ERR_INTERNAL;
        } else {
            *out_count = outn;
        }
    }
    return rc;
    YB_CATCH
}

yams_status_t yams_b200_batch_distance(void* self, int metric, const float* query, uint32_t dim, const float* database,
                                       uint64_t n, int mode, uint64_t k, float threshold, uint64_t* out_idx, float* out_dist,
                                       uint64_t* out_count) {
    YB_TRY
    (void)self;
    YB_ARG(out_count, "out_count is null");
    *out_count = 0;
    YB_ARG(metric == YAMS_B200_COSINE || metric == YAMS_B200_L2, "unknown metric");
    YB_ARG(mode >= YAMS_B200_BATCH_ALL && mode <= YAMS_B200_BATCH_FILTERED, "unknown mode");
    YB_ARG(query && dim > 0, "bad query");
    if (n == 0 || (mode == YAMS_B200_BATCH_TOP_K && k == 0)) return YAMS_OK;
    YB_ARG(database, "database is null");
    YB_ARG(n < 0xFFFFFFFFull, "too many rows");
    YB_ARG(mode == YAMS_B200_BATCH_ALL ? out_dist != nullptr : out_idx != nullptr, "null output");
    YB_ARG(mode != YAMS_B200_BATCH_FILTERED || out_dist, "null output");
    OpWsLease lease;
    if (!lease.w) return YAMS_ERR_INTERNAL;
    cudaStream_t st = lease.w->st;
    yams_status_t rc;
    uint64_t np2 = 1;
    while (np2 < n) np2 <<= 1;
    DevBuf &d_rows = lease.w->d[0], &d_q = lease.w->d[1], &d_dist = lease.w->d[2], &d_keys = lease.w->d[3], &d_oi = lease.w->d[4],
           &d_od = lease.w->d[5], &d_cnt = lease.w->d[6];
    rc = d_rows.reserve((size_t)n * dim * 4);
    if (rc == YAMS_OK) rc = d_q.reserve((size_t)dim * 4);
    if (rc == YAMS_OK) rc = d_dist.reserve((size_t)n * 4);
    if (rc == YAMS_OK && mode != YAMS_B200_BATCH_ALL) {
        rc = d_keys.reserve((size_t)np2 * 8);
        if (rc == YAMS_OK) rc = d_oi.reserve((size_t)n * 8);
        if (rc == YAMS_OK) rc = d_od.reserve((size_t)n * 4);
        if (rc == YAMS_OK) rc = d_cnt.reserve(8);
    }
    if (rc == YAMS_OK) {
        cudaError_t e = cudaMemcpyAsync(d_rows.p, database, (size_t)n * dim * 4, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_q.p, query, (size_t)dim * 4, cudaMemcpyHostToDevice, st);
        batch_dist_kernel<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(d_rows.as<float>(), dim, n, d_q.as<float>(), metric, d_dist.as<float>());
        unsigned g = (unsigned)std::min<uint64_t>((np2 + 255) / 256, 65535);
        uint64_t outn = n;
        if (mode == YAMS_B200_BATCH_ALL) {
            negate_kernel<<<g, 256, 0, st>>>(d_dist.as<float>(), n);
            if (e == cudaSuccess) e = cudaMemcpyAsync(out_dist, d_dist.p, (size_t)n * 4, cudaMemcpyDeviceToHost, st);
            if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        } else {
            if (mode == YAMS_B200_BATCH_TOP_K)
                make_keys_kernel<<<g, 256, 0, st>>>(d_dist.as<float>(), n, np2, d_keys.as<uint64_t>());
            else
                make_keys_filtered_kernel<<<g, 256, 0, st>>>(d_dist.as<float>(), n, np2, threshold, d_keys.as<uint64_t>());
            for (uint64_t size = 2; size <= np2; size <<= 1)
                for (uint64_t stride = size >> 1; stride > 0; stride >>= 1)
                    bitonic_step_kernel<<<g, 256, 0, st>>>(d_keys.as<uint64_t>(), np2, size, stride);
            if (mode == YAMS_B200_BATCH_TOP_K) {
                outn = std::min<uint64_t>(k, n);
            } else {
                unsigned long long h_cnt = 0;
                if (e == cudaSuccess) e = cudaMemsetAsync(d_cnt.p, 0, 8, st);
                count_nonzero_kernel<<<g, 256, 0, st>>>(d_keys.as<uint64_t>(), np2, d_cnt.as<unsigned long long>());
                if (e == cudaSuccess) e = cudaMemcpyAsync(&h_cnt, d_cnt.p, 8, cudaMemcpyDeviceToHost, st);
                if (e == cudaSuccess) e = cudaStreamSynchronize(st);
                outn = h_cnt;
            }
            if (outn && e == cudaSuccess) {
                unpack_idx_keys_kernel<<<g, 256, 0, st>>>(d_keys.as<uint64_t>(), outn, d_oi.as<uint64_t>(), d_od.as<float>());
                e = cudaMemcpyAsync(out_idx, d_oi.p, (size_t)outn * 8, cudaMemcpyDeviceToHost, st);
                if (e == cudaSuccess && out_dist) e = cudaMemcpyAsync(out_dist, d_od.p, (size_t)outn * 4, cudaMemcpyDeviceToHost, st);
                if (e == cudaSuccess) e = cudaStreamSynchronize(st);
            }
        }
        if (e == cudaSuccess) e = cudaGetLastError();
        if (e != cudaSuccess) {
            set_last_error("batch_distance failed: %s", cudaGetErrorString(e));
            rc = YAMS_ERR_INTERNAL;
        } else {
            *out_count = outn;
        }
    }
    return rc;
    YB_CATCH
}

// n pairs (a_i, b_i) of d floats each -> n doubles; one thread per pair, the reference's accumulation order
static yams_status_t cosine_similarity_pairs(const float* a, const float* b, size_t n, size_t d, double* out) {
    OpWsLease lease;
    OpWs* w = lease.w;
    if (!w) return YAMS_ERR_INTERNAL;
    yams_status_t rc;
    const size_t vb = n * d * 4;
    if ((rc = w->d[0].reserve(2 * vb + n * 8 + 64)) != YAMS_OK) return rc;
    if ((rc = w->h.reserve(n * 8 + 64)) != YAMS_OK) return rc;
    float* da = w->d[0].as<float>();
    float* db = da + n * d;
    double* dout = reinterpret_cast<double*>(w->d[0].as<uint8_t>() + ((2 * vb + 7) & ~(size_t)7));
    YB_CUDA(cudaMemcpyAsync(da, a, vb, cudaMemcpyHostToDevice, w->st));
    YB_CUDA(cudaMemcpyAsync(db, b, vb, cudaMemcpyHostToDevice, w->st));
    cosine_similarity_f64_kernel<<<(unsigned)((n + 63) / 64), 64, 0, w->st>>>(da, db, n, d, dout);
    YB_CUDA(cudaMemcpyAsync(w->h.p, dout, n * 8, cudaMemcpyDeviceToHost, w->st));
    YB_CUDA(cudaStreamSynchronize(w->st));
    memcpy(out, w->h.p, n * 8);
    return YAMS_OK;
}

yams_status_t yams_b200_compute_cosine_similarity(void* self, const float* a, size_t na, const float* b, size_t nb, double* out) {
    YB_TRY
    (void)self;
    YB_ARG(out, "out is null");
    *out = 0.0;
    if (na != nb || na == 0) return YAMS_OK;   // vector_database.cpp:1788-1790
    YB_ARG(a && b, "null vector");
    return cosine_similarity_pairs(a, b, 1, na, out);
    YB_CATCH
}

// The rerank loops that call computeCosineSimilarity once per candidate (sqlite_vec_backend.cpp:4025,4374,4507) as ONE device
// pass: n pairs, row-major a[n][dim] / b[n][dim] (pass the same query n times, or n different pairs).
yams_status_t yams_b200_compute_cosine_similarity_many(void* self, const float* a, const float* b, size_t n, size_t dim, double* out) {
    YB_TRY
    (void)self;
    YB_ARG(out || n == 0, "out is null");
    if (n == 0) return YAMS_OK;
    if (dim == 0) {
        for (size_t i = 0; i < n; ++i) out[i] = 0.0;
        return YAMS_OK;
    }
    YB_ARG(a && b, "null vector");
    return cosine_similarity_pairs(a, b, n, dim, out);
    YB_CATCH
}

}  // extern "C"
