"""ctypes door onto the CPU oracle.  TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
import this module.  The product package (yams_b200/) never does.

Two libraries:
  * ``libyams_oracle.so``  -- oracle/yams_oracle.c, the plain-C restatement (always available;
    built on demand with gcc).
  * ``_ref/libyams_ref.so`` -- the reference's own sources compiled by oracle/Makefile where
    /root/reference exists (prebuilt file travels to the GPU box); optional.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from typing import Optional

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
_ORACLE_SO = os.path.join(HERE, "libyams_oracle.so")
_REF_SO = os.path.join(HERE, "_ref", "libyams_ref.so")

u8p = C.POINTER(C.c_uint8)
u64p = C.POINTER(C.c_uint64)
i64p = C.POINTER(C.c_int64)
f32p = C.POINTER(C.c_float)
u32p = C.POINTER(C.c_uint32)


class CdcConfig(C.Structure):
    _fields_ = [
        ("window_size", C.c_uint64),
        ("min_chunk", C.c_uint64),
        ("max_chunk", C.c_uint64),
        ("polynomial", C.c_uint64),
        ("mask", C.c_uint64),
        ("variant", C.c_int32),
    ]


STREAMING, RABIN = 0, 1
DTYPE_F32, DTYPE_F16 = 0, 1
METRIC_COSINE, METRIC_L2 = 0, 1


def default_config(variant: int = STREAMING, **kw) -> CdcConfig:
    cfg = CdcConfig(48, 16 * 1024, 1024 * 1024, 0x3DA3358B4DC173, 0x1FFF, variant)
    for k, v in kw.items():
        setattr(cfg, k, v)
    return cfg


def build(force: bool = False) -> None:
    """Compile the C restatement (and _ref when the reference tree is present)."""
    src = os.path.join(HERE, "yams_oracle.c")
    stale = (not os.path.exists(_ORACLE_SO)) or os.path.getmtime(_ORACLE_SO) < max(
        os.path.getmtime(src), os.path.getmtime(os.path.join(HERE, "yams_oracle.h")))
    if force or stale:
        subprocess.check_call(["make", "-s", "-C", HERE, "oracle"])
    if os.path.isdir("/root/reference/src/chunking"):
        shim = os.path.join(HERE, "ref_shim.cpp")
        if force or not os.path.exists(_REF_SO) or os.path.getmtime(_REF_SO) < os.path.getmtime(shim):
            subprocess.check_call(["make", "-s", "-C", HERE, "ref"])


_lib = None
_ref = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_ORACLE_SO)
        L.yo_cdc_candidates_full.restype = C.c_size_t
        L.yo_cdc_candidates_full.argtypes = [u8p, C.c_size_t, C.POINTER(CdcConfig), u64p, C.c_size_t]
        L.yo_cdc_candidates_local.restype = C.c_size_t
        L.yo_cdc_candidates_local.argtypes = L.yo_cdc_candidates_full.argtypes
        L.yo_cdc_chunk.restype = C.c_size_t
        L.yo_cdc_chunk.argtypes = [u8p, C.c_size_t, C.POINTER(CdcConfig), u64p, u64p, C.c_size_t]
        L.yo_cdc_chunk_and_hash.restype = C.c_size_t
        L.yo_cdc_chunk_and_hash.argtypes = [u8p, C.c_size_t, C.POINTER(CdcConfig), u64p, u64p, u8p,
                                            C.c_size_t]
        L.yo_rabin_table.argtypes = [C.c_uint64, u64p]
        L.yo_sha256.argtypes = [u8p, C.c_size_t, u8p]
        L.yo_sha256_batch.argtypes = [u8p, u64p, u64p, C.c_size_t, u8p]
        L.yo_f16_from_float.restype = C.c_uint16
        L.yo_f16_from_float.argtypes = [C.c_float]
        L.yo_f16_to_float.restype = C.c_float
        L.yo_f16_to_float.argtypes = [C.c_uint16]
        L.yo_cosine_distance_f32.restype = C.c_float
        L.yo_cosine_distance_f32.argtypes = [f32p, f32p, C.c_size_t]
        L.yo_l2_distance_f32.restype = C.c_float
        L.yo_l2_distance_f32.argtypes = [f32p, f32p, C.c_size_t]
        L.yo_l2_distance_build_f32.restype = C.c_float
        L.yo_l2_distance_build_f32.argtypes = [f32p, f32p, C.c_size_t]
        L.yo_exact_scan_l2_batch.restype = None
        L.yo_exact_scan_l2_batch.argtypes = [C.c_void_p, C.c_int, C.c_size_t, C.c_size_t, f32p, C.c_size_t, C.c_size_t,
                                             i64p, f32p, u32p]
        L.yo_cosine_similarity_f64.restype = C.c_double
        L.yo_cosine_similarity_f64.argtypes = [f32p, f32p, C.c_size_t]
        L.yo_vec_distance_l2.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, f32p]
        L.yo_vec_distance_cosine.argtypes = L.yo_vec_distance_l2.argtypes
        L.yo_exact_scan_cosine.argtypes = [C.c_void_p, C.c_int, C.c_size_t, C.c_size_t, i64p, i64p,
                                           f32p, C.c_size_t, C.c_float, i64p, C.c_size_t, C.c_int,
                                           i64p, f32p, C.POINTER(C.c_size_t)]
        L.yo_exact_scan_cosine_batch.argtypes = [C.c_void_p, C.c_int, C.c_size_t, C.c_size_t, f32p,
                                                 C.c_size_t, C.c_size_t, C.c_float, i64p, f32p, u32p]
        L.yo_vec0_exact.argtypes = [f32p, C.c_size_t, C.c_size_t, i64p, f32p, C.c_size_t, C.c_int,
                                    C.c_int64, C.c_int64, i64p, f32p, C.POINTER(C.c_size_t)]
        L.yo_batch_top_k.restype = C.c_size_t
        L.yo_batch_top_k.argtypes = [f32p, f32p, C.c_size_t, C.c_size_t, C.c_int, C.c_size_t, u64p,
                                     f32p]
        L.yo_splitmix64.restype = C.c_uint64
        L.yo_splitmix64.argtypes = [C.c_uint64]
        L.yo_gen_bytes.argtypes = [C.c_uint64, C.c_uint64, C.c_size_t, u8p]
        L.yo_gen_rows_f32.argtypes = [C.c_uint64, C.c_uint64, C.c_size_t, C.c_size_t, f32p]
        _lib = L
    return _lib


def ref_available() -> bool:
    return os.path.exists(_REF_SO)


def ref():
    """The reference-compiled library, or None when it was never built (no /root/reference)."""
    global _ref
    if _ref is None and ref_available():
        R = C.CDLL(_REF_SO)
        R.ref_chunk.restype = C.c_size_t
        R.ref_chunk.argtypes = [u8p, C.c_size_t, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64,
                                C.c_uint64, C.c_int, u64p, u64p, u8p, C.c_size_t]
        R.ref_sha256_hex.argtypes = [u8p, C.c_size_t, C.c_char_p]
        R.ref_sha256_stream_hex.argtypes = [u8p, C.c_size_t, C.c_size_t, C.c_char_p]
        R.ref_sha256_batch.argtypes = [u8p, u64p, u64p, C.c_size_t, u8p]
        R.ref_l2_distance.restype = C.c_float
        R.ref_l2_distance.argtypes = [f32p, f32p, C.c_size_t]
        R.ref_cosine_distance.restype = C.c_float
        R.ref_cosine_distance.argtypes = [f32p, f32p, C.c_size_t]
        R.ref_batch_top_k.restype = C.c_size_t
        R.ref_batch_top_k.argtypes = [f32p, f32p, C.c_size_t, C.c_size_t, C.c_int, C.c_size_t, u64p,
                                      f32p]
        R.ref_batch_top_k_queries.argtypes = [f32p, C.c_size_t, f32p, C.c_size_t, C.c_size_t,
                                              C.c_int, C.c_size_t, u64p, f32p]
        R.ref_f16_from_float.restype = C.c_uint16
        R.ref_f16_from_float.argtypes = [C.c_float]
        R.ref_f16_to_float.restype = C.c_float
        R.ref_f16_to_float.argtypes = [C.c_uint16]
        _ref = R
    return _ref


# ------------------------------------------------------------------------------------------
# numpy helpers
# ------------------------------------------------------------------------------------------

def _p(a: np.ndarray, t):
    return a.ctypes.data_as(t)


def _bytes_arr(data) -> np.ndarray:
    if isinstance(data, np.ndarray):
        a = np.ascontiguousarray(data, dtype=np.uint8)
    else:
        a = np.frombuffer(bytes(data), dtype=np.uint8)
    if a.size == 0:
        a = np.zeros(1, dtype=np.uint8)[:0]
    return a


def _data_ptr(a: np.ndarray):
    if a.size == 0:
        return C.cast(C.c_void_p(0), u8p)
    return _p(a, u8p)


def gen_bytes(seed: int, start: int, n: int) -> np.ndarray:
    out = np.empty(n, dtype=np.uint8)
    if n:
        lib().yo_gen_bytes(seed, start, n, _p(out, u8p))
    return out


def gen_rows_f32(seed: int, first_row: int, n: int, d: int) -> np.ndarray:
    out = np.empty((n, d), dtype=np.float32)
    if n:
        lib().yo_gen_rows_f32(seed, first_row, n, d, _p(out, f32p))
    return out


def f16_from_float(x: np.ndarray) -> np.ndarray:
    """Reference truncating conversion (utils/float16.hpp:20-40), vectorised in numpy; checked
    element-by-element against yo_f16_from_float / ref_f16_from_float in tests."""
    b = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32)
    sign = (b >> 16) & 0x8000
    exp = ((b >> 23) & 0xFF).astype(np.int32) - 127 + 15
    mant = b & 0x7FFFFF
    sub_shift = np.clip(1 - exp, 0, 31).astype(np.uint32)
    sub = (sign | (((mant | 0x800000) >> sub_shift) >> 13))
    norm = sign | (np.clip(exp, 0, 31).astype(np.uint32) << 10) | (mant >> 13)
    out = np.where(exp <= 0, np.where(exp < -10, sign, sub), np.where(exp >= 31, sign | 0x7C00, norm))
    return out.astype(np.uint16)


def f16_to_float(h: np.ndarray) -> np.ndarray:
    return np.ascontiguousarray(h, dtype=np.uint16).view(np.float16).astype(np.float32)


def sha256(data) -> bytes:
    a = _bytes_arr(data)
    out = np.empty(32, dtype=np.uint8)
    lib().yo_sha256(_data_ptr(a), a.size, _p(out, u8p))
    return out.tobytes()


def sha256_batch(base: np.ndarray, offsets: np.ndarray, sizes: np.ndarray) -> np.ndarray:
    base = _bytes_arr(base)
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
    sizes = np.ascontiguousarray(sizes, dtype=np.uint64)
    out = np.empty((len(offsets), 32), dtype=np.uint8)
    if len(offsets):
        lib().yo_sha256_batch(_data_ptr(base), _p(offsets, u64p), _p(sizes, u64p), len(offsets),
                              _p(out, u8p))
    return out


def cdc_candidates(data, cfg: CdcConfig, local: bool = False) -> np.ndarray:
    a = _bytes_arr(data)
    cap = max(16, a.size // 64 + 16)
    fn = lib().yo_cdc_candidates_local if local else lib().yo_cdc_candidates_full
    while True:
        out = np.empty(cap, dtype=np.uint64)
        n = fn(_data_ptr(a), a.size, C.byref(cfg), _p(out, u64p), cap)
        if n <= cap:
            return out[:n].copy()
        cap = n


def cdc_chunk(data, cfg: CdcConfig, hash: bool = True):
    """-> (offsets u64[n], sizes u64[n], digests u8[n,32] or None)"""
    a = _bytes_arr(data)
    cap = max(16, a.size // max(1, int(cfg.min_chunk)) + 16)
    cap = min(cap, a.size + 16)
    while True:
        offs = np.empty(cap, dtype=np.uint64)
        sizes = np.empty(cap, dtype=np.uint64)
        if hash:
            dig = np.empty((cap, 32), dtype=np.uint8)
            n = lib().yo_cdc_chunk_and_hash(_data_ptr(a), a.size, C.byref(cfg), _p(offs, u64p),
                                            _p(sizes, u64p), _p(dig, u8p), cap)
        else:
            dig = None
            n = lib().yo_cdc_chunk(_data_ptr(a), a.size, C.byref(cfg), _p(offs, u64p),
                                   _p(sizes, u64p), cap)
        if n <= cap:
            return offs[:n].copy(), sizes[:n].copy(), (dig[:n].copy() if dig is not None else None)
        cap = n


def ref_dedup_stats(data, cfg: CdcConfig, variant: Optional[int] = None) -> dict:
    """The reference's own calculateDeduplication over the reference chunker's output (oracle/_ref)."""
    a = _bytes_arr(data)
    out = (C.c_uint64 * 4)()
    v = cfg.variant if variant is None else variant
    R = ref()
    R.ref_dedup_stats.argtypes = [u8p, C.c_size_t, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, C.c_int,
                                  C.POINTER(C.c_uint64)]
    R.ref_dedup_stats.restype = None
    R.ref_dedup_stats(_data_ptr(a), a.size, cfg.window_size, cfg.min_chunk, cfg.max_chunk, cfg.polynomial, cfg.mask, v, out)
    return {"totalSize": int(out[0]), "uniqueSize": int(out[1]), "chunkCount": int(out[2]), "uniqueChunks": int(out[3])}


def ref_chunk(data, cfg: CdcConfig, variant: Optional[int] = None, hash: bool = True):
    """Reference StreamingChunker (variant 0) / RabinChunker lazy (1) / RabinChunker full (2)."""
    R = ref()
    assert R is not None, "oracle/_ref not built"
    a = _bytes_arr(data)
    v = cfg.variant if variant is None else variant
    cap = max(16, a.size // max(1, int(cfg.min_chunk)) + 16)
    cap = min(cap, a.size + 16)
    while True:
        offs = np.empty(cap, dtype=np.uint64)
        sizes = np.empty(cap, dtype=np.uint64)
        dig = np.empty((cap, 32), dtype=np.uint8)
        n = R.ref_chunk(_data_ptr(a), a.size, cfg.window_size, cfg.min_chunk, cfg.max_chunk,
                        cfg.polynomial, cfg.mask, v, _p(offs, u64p), _p(sizes, u64p),
                        _p(dig, u8p) if hash else C.cast(C.c_void_p(0), u8p), cap)
        if n <= cap:
            return offs[:n].copy(), sizes[:n].copy(), (dig[:n].copy() if hash else None)
        cap = n


def manifest_checksum(file_digest, file_size: int, digests: np.ndarray, offsets, sizes, use_ref: bool = False):
    """ManifestManager::calculateChecksum; use_ref -> the reference's own createManifest (returns (checksum, valid))."""
    fd = np.ascontiguousarray(np.frombuffer(bytes(file_digest), dtype=np.uint8))
    dg = np.ascontiguousarray(digests, dtype=np.uint8).reshape(-1, 32)
    of = np.ascontiguousarray(offsets, dtype=np.uint64)
    sz = np.ascontiguousarray(sizes, dtype=np.uint64)
    n = len(of)
    if use_ref:
        R = ref()
        R.ref_manifest_checksum.restype = C.c_uint32
        R.ref_manifest_checksum.argtypes = [u8p, C.c_uint64, u8p, u64p, u64p, C.c_size_t, C.POINTER(C.c_int)]
        valid = C.c_int(0)
        crc = R.ref_manifest_checksum(_p(fd, u8p), file_size, _p(dg, u8p) if n else C.cast(C.c_void_p(0), u8p), _p(of, u64p), _p(sz, u64p), n,
                                      C.byref(valid))
        return int(crc), int(valid.value)
    L = lib()
    L.yo_manifest_checksum.restype = C.c_uint32
    L.yo_manifest_checksum.argtypes = [u8p, C.c_uint64, u8p, u64p, u64p, C.c_size_t]
    return int(L.yo_manifest_checksum(_p(fd, u8p), file_size, _p(dg, u8p) if n else C.cast(C.c_void_p(0), u8p), _p(of, u64p), _p(sz, u64p), n))


def simeon_encode_ref(texts, ngram_min=3, ngram_max=5, sketch_dim=4096, output_dim=384, hash_seed=0xA5A5A5A5A5A5A5A5,
                      projection_seed=0xDEADBEEFCAFEBABE, l2_normalize=1) -> np.ndarray:
    """simeon::Encoder::encode (third_party/simeon compiled in place) over a list of byte strings."""
    R = ref()
    R.ref_simeon_encode.argtypes = [C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint64, C.c_uint64, C.c_int,
                                    C.POINTER(C.c_char_p), C.POINTER(C.c_size_t), C.c_size_t, f32p]
    raw = [t.encode("utf-8") if isinstance(t, str) else bytes(t) for t in texts]
    n = len(raw)
    out = np.zeros((n, output_dim), dtype=np.float32)
    if n:
        ptrs = (C.c_char_p * n)(*raw)
        lens = (C.c_size_t * n)(*[len(r) for r in raw])
        R.ref_simeon_encode(ngram_min, ngram_max, sketch_dim, output_dim, hash_seed, projection_seed, l2_normalize, ptrs, lens, n, _p(out, f32p))
    return out


def simeon_encode_modes_ref(texts, ngram_mode="CharAndWord", projection="Fwht", ngram_min=3, ngram_max=5, sketch_dim=4096, output_dim=1024,
                            hash_seed=0xA5A5A5A5A5A5A5A5, projection_seed=0xDEADBEEFCAFEBABE, l2_normalize=1) -> np.ndarray:
    """simeon::Encoder with an explicit n-gram mode and projection (the configurable profile of YAMS's Simeon backend)."""
    R = ref()
    R.ref_simeon_enum.argtypes = [C.c_char_p]
    R.ref_simeon_enum.restype = C.c_int
    R.ref_simeon_encode_modes.argtypes = [C.c_int, C.c_int, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint64, C.c_uint64, C.c_int,
                                          C.POINTER(C.c_char_p), C.POINTER(C.c_size_t), C.c_size_t, f32p]
    nm, pm = R.ref_simeon_enum(ngram_mode.encode()), R.ref_simeon_enum(projection.encode())
    assert nm >= 0 and pm >= 0
    raw = [t.encode("utf-8") if isinstance(t, str) else bytes(t) for t in texts]
    n = len(raw)
    out = np.zeros((n, output_dim), dtype=np.float32)
    if n:
        ptrs = (C.c_char_p * n)(*raw)
        lens = (C.c_size_t * n)(*[len(r) for r in raw])
        R.ref_simeon_encode_modes(nm, pm, ngram_min, ngram_max, sketch_dim, output_dim, hash_seed, projection_seed, l2_normalize, ptrs, lens, n,
                                  _p(out, f32p))
    return out


def _pq_fns():
    R = ref()
    R.ref_pq_encode.argtypes = [f32p, C.c_uint32, C.c_uint32, C.c_uint32, f32p, C.c_uint32, u8p]
    R.ref_pq_scores.argtypes = [f32p, C.c_uint32, C.c_uint32, C.c_uint32, f32p, u8p, C.c_size_t, f32p, f32p]
    R.ref_pq_train.argtypes = [C.c_uint32, C.c_uint32, C.c_uint32, f32p, C.c_uint32, f32p]
    return R


def normalize_like_reference(rows: np.ndarray):
    """normalizeEmbeddingInPlace (src/vector/sqlite_vec_backend.cpp:213-226): sequential double sum of squares, rows with
    norm_sq <= 1e-20 rejected, inv = 1.0f / sqrt(float(norm_sq)), float scale.  -> (normalised rows of the accepted, accepted mask)"""
    r = np.ascontiguousarray(rows, dtype=np.float32)
    sq = np.cumsum(r.astype(np.float64) ** 2, axis=1)[:, -1]            # cumsum adds left to right, like the reference loop
    ok = sq > 1e-20
    inv = (np.float32(1.0) / np.sqrt(sq[ok].astype(np.float32))).astype(np.float32)
    return (r[ok] * inv[:, None]).astype(np.float32), ok


def pq_encode_ref(codebooks, dim, m, k, normalised_rows):
    """simeon::ProductQuantizer::encode_batch (third_party/simeon/src/pq.cpp) compiled in place."""
    R = _pq_fns()
    v = np.ascontiguousarray(normalised_rows, dtype=np.float32)
    cb = np.ascontiguousarray(codebooks, dtype=np.float32)
    codes = np.zeros((len(v), m), dtype=np.uint8)
    R.ref_pq_encode(_p(cb, f32p), dim, m, k, _p(v, f32p), len(v), _p(codes, u8p))
    return codes


def pq_scores_ref(codebooks, dim, m, k, normalised_query, codes):
    """simeon::PQInnerProductQuery: (ADC inner products of every code row, the lookup table)."""
    R = _pq_fns()
    cb = np.ascontiguousarray(codebooks, dtype=np.float32)
    q = np.ascontiguousarray(normalised_query, dtype=np.float32)
    cd = np.ascontiguousarray(codes, dtype=np.uint8)
    out = np.zeros(len(cd), dtype=np.float32)
    lut = np.zeros(m * k, dtype=np.float32)
    R.ref_pq_scores(_p(cb, f32p), dim, m, k, _p(q, f32p), _p(cd, u8p), len(cd), _p(out, f32p), _p(lut, f32p))
    return out, lut


def pq_train_ref(dim, m, k, training):
    R = _pq_fns()
    t = np.ascontiguousarray(training, dtype=np.float32)
    cb = np.zeros(m * k * (dim // m), dtype=np.float32)
    R.ref_pq_train(dim, m, k, _p(t, f32p), len(t), _p(cb, f32p))
    return cb


def exact_scan_cosine(rows: np.ndarray, query: np.ndarray, k: int, threshold: float = -1.0,
                      rowids: Optional[np.ndarray] = None, tie_rank: Optional[np.ndarray] = None,
                      allowed: Optional[np.ndarray] = None, all_matching: bool = False):
    """-> (status, rowids i64[m], scores f32[m]); rows fp32 [n,d] or uint16 (fp16 bits) [n,d]."""
    rows = np.ascontiguousarray(rows)
    dtype = DTYPE_F16 if rows.dtype == np.uint16 else DTYPE_F32
    if dtype == DTYPE_F32:
        rows = rows.astype(np.float32, copy=False)
    n, d = rows.shape
    q = np.ascontiguousarray(query, dtype=np.float32)
    cap = n if all_matching else k
    out_r = np.empty(max(cap, 1), dtype=np.int64)
    out_s = np.empty(max(cap, 1), dtype=np.float32)
    cnt = C.c_size_t(0)
    nul = C.cast(C.c_void_p(0), i64p)
    rid = np.ascontiguousarray(rowids, dtype=np.int64) if rowids is not None else None
    tr = np.ascontiguousarray(tie_rank, dtype=np.int64) if tie_rank is not None else None
    al = np.ascontiguousarray(allowed, dtype=np.int64) if allowed is not None else None
    rc = lib().yo_exact_scan_cosine(rows.ctypes.data_as(C.c_void_p), dtype, n, d,
                                    _p(rid, i64p) if rid is not None else nul,
                                    _p(tr, i64p) if tr is not None else nul, _p(q, f32p), k,
                                    threshold, _p(al, i64p) if al is not None else nul,
                                    len(al) if al is not None else 0, int(all_matching),
                                    _p(out_r, i64p), _p(out_s, f32p), C.byref(cnt))
    return rc, out_r[:cnt.value].copy(), out_s[:cnt.value].copy()


def exact_scan_cosine_batch(rows: np.ndarray, queries: np.ndarray, k: int, threshold: float = -1.0):
    rows = np.ascontiguousarray(rows)
    dtype = DTYPE_F16 if rows.dtype == np.uint16 else DTYPE_F32
    n, d = rows.shape
    q = np.ascontiguousarray(queries, dtype=np.float32)
    nq = q.shape[0]
    out_r = np.full((nq, k), -1, dtype=np.int64)
    out_s = np.zeros((nq, k), dtype=np.float32)
    cnt = np.zeros(nq, dtype=np.uint32)
    rc = lib().yo_exact_scan_cosine_batch(rows.ctypes.data_as(C.c_void_p), dtype, n, d, _p(q, f32p),
                                          nq, k, threshold, _p(out_r, i64p), _p(out_s, f32p),
                                          _p(cnt, u32p))
    return rc, out_r, out_s, cnt


def l2_distance_build(a: np.ndarray, b: np.ndarray) -> float:
    """l2_distance<float> in the reference build's operation order (AVX lanes when d % 16 == 0, else the scalar loop)."""
    a = np.ascontiguousarray(a, dtype=np.float32)
    b = np.ascontiguousarray(b, dtype=np.float32)
    assert a.shape == b.shape and a.ndim == 1
    return lib().yo_l2_distance_build_f32(_p(a, f32p), _p(b, f32p), a.size)


def exact_scan_l2_batch(rows: np.ndarray, queries: np.ndarray, k: int):
    """Exact L2 top-k of every query, distances in the reference build's order -> (rowids i64[Q,k], dist f32[Q,k],
    counts u32[Q]); ties by row index, padding rowid -1 / +inf.  rows fp32 [n,d] or uint16 (fp16 bits) [n,d]."""
    rows = np.ascontiguousarray(rows)
    dtype = DTYPE_F16 if rows.dtype == np.uint16 else DTYPE_F32
    if dtype == DTYPE_F32:
        rows = rows.astype(np.float32, copy=False)
    n, d = rows.shape
    q = np.ascontiguousarray(queries, dtype=np.float32).reshape(-1, d)
    nq = q.shape[0]
    out_r = np.full((nq, k), -1, dtype=np.int64)
    out_d = np.full((nq, k), np.inf, dtype=np.float32)
    cnt = np.zeros(nq, dtype=np.uint32)
    if nq and k:
        lib().yo_exact_scan_l2_batch(rows.ctypes.data_as(C.c_void_p), dtype, n, d, _p(q, f32p), nq, k, _p(out_r, i64p),
                                     _p(out_d, f32p), _p(cnt, u32p))
    return out_r, out_d, cnt


def vec0_exact(rows: np.ndarray, query: np.ndarray, k: int = 0, rowids=None, rowid_range=None):
    rows = np.ascontiguousarray(rows, dtype=np.float32)
    n, d = rows.shape
    q = np.ascontiguousarray(query, dtype=np.float32)
    out_r = np.empty(max(n, 1), dtype=np.int64)
    out_d = np.empty(max(n, 1), dtype=np.float32)
    cnt = C.c_size_t(0)
    rid = np.ascontiguousarray(rowids, dtype=np.int64) if rowids is not None else None
    lo, hi = rowid_range if rowid_range is not None else (0, 0)
    lib().yo_vec0_exact(_p(rows, f32p), n, d,
                        _p(rid, i64p) if rid is not None else C.cast(C.c_void_p(0), i64p),
                        _p(q, f32p), k, int(rowid_range is not None), lo, hi, _p(out_r, i64p),
                        _p(out_d, f32p), C.byref(cnt))
    return out_r[:cnt.value].copy(), out_d[:cnt.value].copy()


def batch_top_k(query: np.ndarray, rows: np.ndarray, k: int, metric: int = METRIC_L2,
                use_ref: bool = False):
    rows = np.ascontiguousarray(rows, dtype=np.float32)
    n, d = rows.shape
    q = np.ascontiguousarray(query, dtype=np.float32)
    out_i = np.empty(max(k, 1), dtype=np.uint64)
    out_d = np.empty(max(k, 1), dtype=np.float32)
    fn = ref().ref_batch_top_k if use_ref else lib().yo_batch_top_k
    m = fn(_p(q, f32p), _p(rows, f32p), n, d, metric, k, _p(out_i, u64p), _p(out_d, f32p))
    return out_i[:m].copy(), out_d[:m].copy()
