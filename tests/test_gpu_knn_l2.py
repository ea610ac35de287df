"""GPU tests of the L2 metric (the vec0 surface, DESIGN.md §4.4) through every level of the exact scan: the stage-1 error
bound, the certificate's L2 branch, the exhaustive levels 1 and 2 behind it, the multi-GPU merge, and stage-1 scores that
overflow.  Every search result is compared, for every query, with the CPU oracle's exact L2 top-k in the reference
build's operation order (oracle.exact_scan_l2_batch, pinned bit for bit in tests/test_oracle_pin.py): ids, distances and
counts must be equal."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def Y():
    import yams_b200
    assert yams_b200.device_count() > 0
    assert yams_b200.plugin_init() == 0, yams_b200.health()
    return yams_b200


def stored(O, rows32, dt):
    """(what the corpus is given, the fp32 values it holds): fp16 rows go through the reference's truncating conversion."""
    if dt == "f16":
        h = O.f16_from_float(rows32).reshape(rows32.shape)
        return h, O.f16_to_float(h).reshape(rows32.shape)
    return rows32, rows32


def l2_corpus(Y, rows, d, rowids=None):
    if rows.dtype == np.uint16:
        c = Y.Corpus(d, Y.F16, Y.L2)
        if len(rows):
            c.append(rows.view(np.float16), rowids=rowids)
    else:
        c = Y.Corpus(d, Y.F32, Y.L2)
        if len(rows):
            c.append(rows, rowids=rowids)
    return c


def assert_exact(O, rows, queries, got, k):
    """ids, distances (bit for bit, padding included) and counts equal to the oracle's, for every query."""
    rid, dist, cnt = got[0], got[1], got[2]
    wr, wd, wc = O.exact_scan_l2_batch(rows, queries, k)
    for qi in range(len(queries)):
        assert cnt[qi] == wc[qi], (qi, cnt[qi], wc[qi])
        assert np.array_equal(rid[qi], wr[qi]), (qi, rid[qi], wr[qi])
        assert np.array_equal(dist[qi].view(np.uint32), wd[qi].view(np.uint32)), (qi, dist[qi], wd[qi])
    return wr, wd, wc


# ---- a. the stage-1 error bound -------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(60_000, 96, "f16"), (200_000, 768, "f16"), (120_000, 128, "f32"), (9_000, 100, "f32")])
def test_l2_stage1_error_stays_inside_the_certified_bound(Y, oracle, shape):
    """Measured |stage-1 score - (2 q.r - |r|^2 in fp64 over the stored values)| stays below eps[q] for both engines, on
    rows whose lengths span four decades and queries from tiny to far from the origin; the search is exact.  For three
    queries one row of the largest length points along the query's own operand rounding residual (fp16 round-to-nearest,
    or tf32 truncation for fp32 corpora): there the Cauchy-Schwarz term of eps is attained, the error is 2 dq Rmax against
    an eps of 2.5 dq Rmax + smaller terms."""
    O = oracle
    n, d, dt = shape
    rng = np.random.default_rng(d)
    rows32 = O.gen_rows_f32(42, 0, n, d) * np.exp(rng.uniform(np.log(1e-2), np.log(1e2), n)).astype(np.float32)[:, None]
    q = O.gen_rows_f32(43, 0, 24, d) * np.float32(1.7)
    q[5] *= np.float32(1e-4)                                        # tiny norm
    q[9] = q[9] * np.float32(300.0) + np.float32(20.0)              # far from the origin
    stride = max(1, n // 20_000)
    for qi in range(3):
        x = q[qi]
        y = (x.view(np.uint32) & np.uint32(0xFFFFE000)).view(np.float32) if dt == "f32" else x.astype(np.float16).astype(np.float32)
        res = (x - y).astype(np.float64)
        rows32[(qi + 1) * 97 * stride] = (100.0 * res / np.linalg.norm(res)).astype(np.float32)
    rows, up = stored(O, rows32, dt)
    c = l2_corpus(Y, rows, d)
    sub = up[::stride].astype(np.float64)
    qd = q.astype(np.float64)
    want = 2.0 * (qd @ sub.T) - np.sum(sub * sub, axis=1)[None, :]
    for engine in (1, 0):
        got = c.debug_stage1_scores(q, engine, row_start=0, row_stride=stride, nrows=len(sub))
        eps = c.debug_last_eps(len(q))
        err = np.abs(got.astype(np.float64) - want).max(axis=1)
        assert np.all(err <= eps), (engine, np.argmax(err - eps), err.max(), eps[np.argmax(err - eps)])
    assert_exact(O, rows, q, c.search(q, 10), 10)
    c.close()


# ---- b. near-tie shell: the certificate must reject ----------------------------------------------------------------
@pytest.mark.parametrize("dt", ["f16", "f32"])
@pytest.mark.parametrize("n", [5_000, 200_000])
def test_l2_near_tie_shell_is_rejected_and_resolved(Y, oracle, dt, n):
    """300 rows on a sphere of radius rho around the adversarial query: stage 1 cannot order them and K' = 32 survivors
    cannot hold them.  Only that query is rejected, resolved exhaustively and answered exactly."""
    O = oracle
    d, k, rho = 128, 10, 0.3
    rng = np.random.default_rng(12)
    rows32 = O.gen_rows_f32(42, 0, n, d)
    q_adv = O.gen_rows_f32(77, 0, 1, d)[0] * np.float32(0.5)
    pos = np.sort(rng.choice(n, size=300, replace=False))
    u = rng.standard_normal((300, d))
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    rows32[pos] = (q_adv.astype(np.float64) + rho * u).astype(np.float32)
    rows, up = stored(O, rows32, dt)
    c = l2_corpus(Y, rows, d)
    queries = np.concatenate([O.gen_rows_f32(43, 0, 7, d), q_adv[None, :]])
    got = c.search(queries, k)
    assert_exact(O, rows, queries, got, k)
    eps = c.debug_last_eps(len(queries))
    _, wd, _ = O.exact_scan_l2_batch(rows, q_adv[None, :], 400)
    d2 = wd[0].astype(np.float64) ** 2
    assert np.sum(d2 <= d2[k - 1] + eps[7] / 2) >= 200              # the input really is adversarial
    assert got[3][7] & Y.FLAG_FALLBACK_PATH
    assert not np.any(got[3][:7] & Y.FLAG_FALLBACK_PATH)
    assert c.last_timings()["resolved_exhaustively"] == 1
    c.close()


# ---- c. duplicates past exhaustive level 1 -------------------------------------------------------------------------
@pytest.mark.parametrize("n", [20_000, 150_000])
def test_l2_duplicates_take_the_full_exact_pass(Y, oracle, n):
    """6001 rows at distance 0 (more than level 1 re-scores): the full exact pass answers, ties in rowid order."""
    O = oracle
    d, k = 64, 10
    rows32 = O.gen_rows_f32(42, 0, n, d) * np.float32(2.0)
    rows32[3000:9000] = rows32[17]
    rows, up = stored(O, rows32, "f16")
    c = l2_corpus(Y, rows, d)
    queries = np.stack([up[17], O.gen_rows_f32(43, 0, 1, d)[0] * np.float32(2.0)])
    got = c.search(queries, k)
    wr, wd, wc = assert_exact(O, rows, queries, got, k)
    assert list(got[0][0]) == [17] + list(range(3000, 3009)) and not np.any(got[1][0])
    assert got[3][0] & Y.FLAG_FALLBACK_PATH and got[3][0] & Y.FLAG_TIE_AT_K
    assert not got[3][1] & Y.FLAG_FALLBACK_PATH
    ex = c.search_exhaustive(queries, k)
    assert np.array_equal(ex[0], wr) and np.array_equal(ex[1], wd) and np.array_equal(ex[2], wc)
    c.close()


# ---- d. rows far from the origin -----------------------------------------------------------------------------------
@pytest.mark.parametrize("dt", ["f16", "f32"])
def test_l2_cluster_far_from_the_origin(Y, oracle, dt):
    """A cluster at |c| ~ 1e3 with unit-scale spread: stage 1 subtracts numbers ~1e6 to resolve distances ~1."""
    O = oracle
    n, d, nq, k = 100_000, 128, 8, 10
    rng = np.random.default_rng(31)
    center = O.gen_rows_f32(5, 0, 1, d)[0] * np.float32(1000.0)
    rows32 = (center + rng.standard_normal((n, d)) / np.sqrt(d)).astype(np.float32)
    queries = (center + rng.standard_normal((nq, d)) / np.sqrt(d)).astype(np.float32)
    rows, up = stored(O, rows32, dt)
    c = l2_corpus(Y, rows, d)
    got = c.search(queries, k)
    assert_exact(O, rows, queries, got, k)
    resolved = c.last_timings()["resolved_exhaustively"]
    assert resolved == int(np.sum((got[3] & Y.FLAG_FALLBACK_PATH) != 0))
    print(f"\n[l2 far cluster {dt}] {resolved} of {nq} queries resolved exhaustively")
    c.close()


# ---- e. shapes and edges -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("d,dt", [(8, "f16"), (24, "f16"), (40, "f16"), (48, "f16"), (33, "f32"), (100, "f32"), (3000, "f32")])
def test_l2_shapes_and_k_edges(Y, oracle, d, dt):
    """fp16 shapes on the tensor engine whose re-scoring takes the scalar order (d % 16 != 0) or the lane order, fp32
    shapes on the CUDA-core (d = 33) and tf32 (d = 100, 3000) engines; d = 3000 re-scores in the scalar order, where the
    certificate's rounding slack is largest.  k = 1, 10, 3072, k > n, n = k and n = 0."""
    O = oracle
    n = 4_000 if d == 3000 else 8_000
    rows32 = O.gen_rows_f32(42, 0, n, d) * np.float32(3.0)
    rows32[n // 2] = rows32[7]                                      # an exact tie
    rows, up = stored(O, rows32, dt)
    c = l2_corpus(Y, rows, d)
    queries = O.gen_rows_f32(43, 0, 6, d) * np.float32(2.0)
    queries[1] = up[7]                                              # distance 0 twice
    for k in (1, 10, 3072):
        got = c.search(queries, k)
        if dt == "f16" or d % 4 == 0:
            assert c.last_timings()["engine"] == "tcgen05"
        assert_exact(O, rows, queries, got, k)
    assert list(got[0][1][:2]) == [7, n // 2]
    c.close()
    for m, k in ((50, 100), (10, 10), (0, 5)):                      # k > n, n = k, n = 0
        c = l2_corpus(Y, rows[:m], d)
        got = c.search(queries, k)
        assert_exact(O, rows[:m], queries, got, k)
        assert np.all(got[2] == m) and np.all(got[0][:, m:] == -1) and np.all(np.isposinf(got[1][:, m:]))
        c.close()


# ---- f. multi-GPU merge --------------------------------------------------------------------------------------------
def run_shards(Y, rows, bounds, d, queries, k, threshold, make):
    """search_device on every shard into one packed buffer ([nq*k int64 rowids][nq*k float scores] per rank), then
    search_device_finish; -> (packed, shards, queries resolved exhaustively)"""
    import torch
    nq, R = len(queries), len(bounds) - 1
    packed = torch.zeros((R, nq * k * 12), dtype=torch.uint8, device="cuda")
    dq = torch.from_numpy(np.ascontiguousarray(queries)).cuda()
    shards = []
    for r in range(R):
        a, b = bounds[r], bounds[r + 1]
        c = make(rows[a:b], np.arange(a, b))
        base = packed[r].data_ptr()
        c.search_device(dq.data_ptr(), nq, k, threshold, base, base + nq * k * 8)
        shards.append(c)
    resolved = sum(c.search_device_finish() for c in shards)
    return packed, shards, resolved


def merge_both(shards, packed, nq, k):
    """merge_partials_device on the unpacked partials and merge_packed_device on the packed buffer -> two (ids, scores,
    counts) triples"""
    import torch
    R = packed.shape[0]
    part_r = packed[:, :nq * k * 8].contiguous().view(torch.int64).reshape(R, nq, k).contiguous()
    part_s = packed[:, nq * k * 8:].contiguous().view(torch.float32).reshape(R, nq, k).contiguous()
    out = []
    for packed_mode in (False, True):
        mr = torch.full((nq, k), -7, dtype=torch.int64, device="cuda")
        ms = torch.zeros((nq, k), dtype=torch.float32, device="cuda")
        mc = torch.full((nq,), -7, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        if packed_mode:
            shards[0].merge_packed_device(packed.data_ptr(), R, nq, k, mr.data_ptr(), ms.data_ptr(), mc.data_ptr())
        else:
            shards[0].merge_partials_device(part_r.data_ptr(), part_s.data_ptr(), R, nq, k, mr.data_ptr(), ms.data_ptr(),
                                            mc.data_ptr())
        shards[0].sync()
        out.append((mr.cpu().numpy(), ms.cpu().numpy(), mc.cpu().numpy().astype(np.uint32)))
    return out, part_r.cpu().numpy(), part_s.cpu().numpy()


def test_l2_merge_of_shards(Y, oracle):
    """R = 4 L2 shards, the last shorter than k: identical rows in three shards tie across shards and must come back
    in rowid order, the short shard's padding must not displace real rows, and a near-tie query is resolved by
    search_device_finish before the merge.  Both merges equal the single-corpus search and the oracle."""
    O = oracle
    n, d, nq, k = 120_000, 64, 8, 10
    bounds = [0, 40_000, 80_000, n - 5, n]
    rng = np.random.default_rng(41)
    rows32 = O.gen_rows_f32(42, 0, n, d) * np.float32(2.0)
    copies = [40_010, 80_020, n - 3]
    for p in copies:
        rows32[p] = rows32[100]
    q_adv = O.gen_rows_f32(77, 0, 1, d)[0]
    pos = np.sort(rng.choice(np.setdiff1d(np.arange(bounds[3]), [100] + copies), size=300, replace=False))
    u = rng.standard_normal((300, d))
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    rows32[pos] = (q_adv.astype(np.float64) + 0.3 * u).astype(np.float32)
    rows, up = stored(O, rows32, "f16")
    queries = O.gen_rows_f32(43, 0, nq, d) * np.float32(2.0)
    queries[2] = up[100]                                            # distance 0 in shards 0, 1, 2 and 3
    queries[5] = q_adv
    packed, shards, resolved = run_shards(Y, rows, bounds, d, queries, k, -1.0, lambda r, ids: l2_corpus(Y, r, d, ids))
    assert resolved >= 1
    merged, part_r, part_s = merge_both(shards, packed, nq, k)
    wr, wd, wc = O.exact_scan_l2_batch(rows, queries, k)
    whole = l2_corpus(Y, rows, d)
    single = whole.search(queries, k)
    assert_exact(O, rows, queries, single, k)
    for mr, ms, mc in merged:
        assert np.array_equal(mr, wr) and np.array_equal(ms.view(np.uint32), wd.view(np.uint32)) and np.array_equal(mc, wc)
        assert np.array_equal(mr, single[0]) and np.array_equal(ms, single[1])
    assert list(wr[2][:4]) == [100, 40_010, 80_020, n - 3] and not np.any(wd[2][:4])
    # the short shard's own partial: its 5 rows, then padding
    sr, sd, sc = O.exact_scan_l2_batch(rows[bounds[3]:], queries, k)
    assert np.array_equal(part_r[3], np.where(sr >= 0, sr + bounds[3], -1)) and np.array_equal(part_s[3], sd)
    whole.close()
    for c in shards:
        c.close()


def test_cosine_merge_with_short_shards(Y, oracle):
    """Cosine shards whose threshold leaves fewer than k rows in every shard (and a shard of 5 rows): the merged counts
    are the oracle's and the -inf padding never displaces a real row."""
    import torch  # noqa: F401  (CUDA context for the device buffers)
    O = oracle
    n, d, nq, k = 120_005, 64, 8, 10
    bounds = [0, 40_000, 80_000, n - 5, n]
    rows32 = O.gen_rows_f32(42, 0, n, d)
    queries = O.gen_rows_f32(43, 0, nq, d)
    rows32[n - 2] = queries[0]                                      # the 5-row shard holds one result of query 0
    rows, _ = stored(O, rows32, "f16")
    threshold = 0.46

    def make(r, ids):
        c = Y.Corpus(d, Y.F16, Y.COSINE)
        c.append(r.view(np.float16), rowids=ids)
        return c
    packed, shards, _ = run_shards(Y, rows, bounds, d, queries, k, threshold, make)
    merged, part_r, _ = merge_both(shards, packed, nq, k)
    rc, wr, ws, wc = O.exact_scan_cosine_batch(rows, queries, k, threshold=threshold)
    assert rc == 0
    assert np.all(np.sum(part_r >= 0, axis=2) < k)                  # every shard is short for every query
    assert np.any(wc == k) and np.any(wc < k) and part_r[3, 0, 0] == n - 2
    for mr, ms, mc in merged:
        assert np.array_equal(mc, wc)
        for qi in range(nq):
            m = wc[qi]
            assert np.array_equal(mr[qi, :m], wr[qi, :m]) and np.array_equal(ms[qi, :m], ws[qi, :m]), qi
            assert np.all(mr[qi, m:] == -1) and np.all(np.isneginf(ms[qi, m:])), qi
    for c in shards:
        c.close()


# ---- g. non-finite stage-1 scores ----------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [20_000, 150_000])
def test_cosine_stage1_overflow_is_rejected(Y, oracle, n):
    """fp32 rows and queries with components ~1e20 (d = 37: the CUDA-core engine): q_i r_i overflows float.  The
    engine's FMA chain keeps the sign of the first overflowing product (inf + a finite product stays inf), so the stage-1
    scores are +-inf in no useful order and the selection bound (dense, n = 20k) or the list threshold (n = 150k) is +inf.
    The certificate must reject those queries at both levels and the full exact pass must return the reference's answer
    (its double accumulation does not overflow)."""
    O = oracle
    d, k = 37, 10
    rows = O.gen_rows_f32(42, 0, n, d) * np.float32(1e21)
    queries = O.gen_rows_f32(43, 0, 4, d)
    queries[:3] *= np.float32(1e21)                                 # query 3 stays at unit scale: no overflow
    c = Y.Corpus(d, Y.F32, Y.COSINE)
    c.append(rows)
    got = c.search(queries, k, threshold=-1.0)
    rc, wr, ws, wc = O.exact_scan_cosine_batch(rows, queries, k)
    assert rc == 0 and np.all(wc == k)
    assert np.array_equal(got[2], wc) and np.array_equal(got[0], wr) and np.array_equal(got[1], ws)
    assert np.all(got[3][:3] & Y.FLAG_FALLBACK_PATH)
    s1 = c.debug_stage1_scores(queries[:3], 0, nrows=1000)
    assert np.mean(~np.isfinite(s1)) > 0.99                         # the input really overflows stage 1
    c.close()


def test_l2_fp16_query_beyond_the_fp16_range(Y, oracle):
    """L2, fp16 rows, a column that is 0 in every row and a query component of 1e5: the tensor engine's fp16 copy of
    the query holds inf there and inf x 0 makes every stage-1 score NaN (observed on a B200).  NaN scores select last,
    so the list threshold and the selection bound are NaN: the certificate must reject the query (before the fix it
    returned an empty list as exact) and the exhaustive levels must answer it exactly."""
    O = oracle
    n, d, k = 100_000, 128, 10
    rows32 = O.gen_rows_f32(42, 0, n, d) * np.float32(2.0)
    rows32[:, 5] = 0.0
    rows, _ = stored(O, rows32, "f16")
    c = l2_corpus(Y, rows, d)
    queries = O.gen_rows_f32(43, 0, 4, d) * np.float32(2.0)
    queries[1, 5] = 1e5
    got = c.search(queries, k)
    assert c.last_timings()["engine"] == "tcgen05"
    assert_exact(O, rows, queries, got, k)
    assert got[3][1] & Y.FLAG_FALLBACK_PATH
    s1 = c.debug_stage1_scores(queries[1:2], 1, nrows=1000)
    print(f"\n[l2 fp16 query 1e5] tensor-engine stage-1 scores: {np.isnan(s1).mean():.3f} NaN, "
          f"{np.isinf(s1).mean():.3f} inf, eps = {c.debug_last_eps(1)[0]}")
    assert np.isnan(s1).all()
    c.close()
