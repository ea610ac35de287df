"""GPU tests of what makes the two-stage scan EXACT: the device-side certificate, the exhaustive levels behind it, the
headline shape checked query by query against the CPU oracle, and the L2 metric through the same tensor-core pipeline.

Reference semantics: bruteForceSearchUnlocked (src/vector/sqlite_vec_backend.cpp:4203-4331, comparator :4218-4223) and
vec0_run_exact_query (third_party/sqlite-vec-cpp/include/sqlite-vec-cpp/sqlite/vec0_module.hpp:376-430)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

TOL = 1e-4   # the reference tests' own epsilon (sqlite-vec-cpp/tests/test_distances.cpp:16-18)


@pytest.fixture(scope="module")
def Y():
    import yams_b200
    assert yams_b200.device_count() > 0
    assert yams_b200.plugin_init() == 0, yams_b200.health()
    return yams_b200


def oracle_rows_f16(O, seed, n, d, step=100_000):
    """The synthetic fp16 corpus exactly as corpus.append_synthetic builds it (generator + truncating conversion)."""
    out = np.empty((n, d), dtype=np.uint16)
    for r0 in range(0, n, step):
        m = min(step, n - r0)
        out[r0:r0 + m] = O.f16_from_float(O.gen_rows_f32(seed, r0, m, d)).reshape(m, d)
    return out


def test_headline_shape_every_query_vs_oracle(Y, oracle):
    """BASELINE config C2's own shape (768-d fp16 rows, a 1024-query batch = 4 query tiles x 12 K blocks, cosine top-10)
    on 1 M rows: EVERY query's ids and scores against the CPU oracle's double-precision scan -- ids equal, scores
    bit-equal -- and against the library's exhaustive pass."""
    O = oracle
    n, d, nq, k = 1_000_000, 768, 1024, 10
    c = Y.Corpus(d, Y.F16, Y.COSINE, capacity_hint=n)
    c.append_synthetic(42, 0, n)
    queries = O.gen_rows_f32(43, 0, nq, d)
    got = c.search(queries, k, threshold=-1.0)
    assert c.last_timings()["engine"] == "tcgen05"
    rows = oracle_rows_f16(O, 42, n, d)
    rc, wr, ws, wc = O.exact_scan_cosine_batch(rows, queries, k)
    assert rc == 0
    assert np.array_equal(got[2], wc)
    assert np.array_equal(got[0], wr)
    assert np.array_equal(got[1], ws)                               # fp64 re-scoring: bit-identical
    assert not np.any(got[3] & Y.FLAG_FALLBACK_PATH)                # ordinary data: every query certified on the fast path
    ex = c.search_exhaustive(queries[:8], k)
    assert np.array_equal(ex[0], wr[:8]) and np.array_equal(ex[1], ws[:8])
    c.close()


def near_tie_corpus(O, n, d, q, n_close, spread, seed, rng):
    """Random unit rows + n_close rows whose cosine with q lies within `spread` of 1."""
    rows = O.gen_rows_f32(seed, 0, n, d)
    pos = np.sort(rng.choice(n, size=n_close, replace=False))
    qn = q / np.linalg.norm(q)
    for p in pos:
        delta = rng.normal(size=d).astype(np.float32)
        delta -= qn * float(delta @ qn)                             # orthogonal to q
        delta *= np.float32(np.sqrt(2.0 * spread * rng.uniform(0.0, 1.0)) / np.linalg.norm(delta))
        rows[p] = (qn + delta) * np.float32(rng.uniform(0.5, 2.0))  # any length: cosine ignores it
    return rows, pos


@pytest.mark.parametrize("dtype", ["f16", "f32"])
@pytest.mark.parametrize("n", [5_000, 200_000])
def test_certificate_catches_near_ties(Y, oracle, dtype, n):
    """>= 200 rows within 1e-4 of the k-th score (near-duplicate chunks): stage 1 (fp16 / tf32 operands) cannot order
    them, K' = 32 survivors cannot hold them.  The certificate must notice and the exhaustive level must return the
    reference's answer, bit for bit; queries without the problem stay on the fast path."""
    O = oracle
    d, k = 128, 10
    rng = np.random.default_rng(11)
    q_adv = O.gen_rows_f32(77, 0, 1, d)[0]
    rows32, pos = near_tie_corpus(O, n, d, q_adv, 300, 1e-4, 42, rng)
    if dtype == "f16":
        rows = O.f16_from_float(rows32).reshape(n, d)
        c = Y.Corpus(d, Y.F16, Y.COSINE)
        c.append(rows.view(np.float16))
    else:
        rows = rows32
        c = Y.Corpus(d, Y.F32, Y.COSINE)
        c.append(rows)
    queries = np.concatenate([O.gen_rows_f32(43, 0, 7, d), q_adv[None, :]])
    got = c.search(queries, k, threshold=-1.0)
    rc, wr, ws, wc = O.exact_scan_cosine_batch(rows, queries, k)
    assert np.array_equal(got[2], wc) and np.array_equal(got[0], wr) and np.array_equal(got[1], ws)
    scores_all = O.exact_scan_cosine(rows, q_adv, 400)[2]
    assert np.sum(scores_all >= scores_all[k - 1] - 1e-4) >= 200     # the test really is adversarial
    assert got[3][7] & Y.FLAG_FALLBACK_PATH                          # the certificate rejected the fast-path answer
    assert not np.any(got[3][:7] & Y.FLAG_FALLBACK_PATH)
    assert c.last_timings()["resolved_exhaustively"] == 1
    # a threshold that only the near-duplicates pass, k larger than their number
    got = c.search(queries[7:], 400, threshold=0.99)
    rc, wr, ws, wc = O.exact_scan_cosine_batch(rows, queries[7:], 400, threshold=0.99)
    assert np.array_equal(got[2], wc) and np.array_equal(got[0][0, :wc[0]], wr[0, :wc[0]])
    assert np.array_equal(got[1][0, :wc[0]], ws[0, :wc[0]])
    c.close()


@pytest.mark.parametrize("n", [20_000, 150_000])
def test_corpus_of_duplicates_takes_the_full_exact_pass(Y, oracle, n):
    """More identical rows than exhaustive level 1 re-scores (4096): only the exact score of every row can answer.
    Equal scores are ordered by rowid and the tie is flagged for the host's chunk_id re-break (:4218-4223)."""
    O = oracle
    d, k = 64, 10
    rows32 = O.gen_rows_f32(42, 0, n, d)
    rows32[3000:9000] = rows32[17]
    rows = O.f16_from_float(rows32).reshape(n, d)
    c = Y.Corpus(d, Y.F16, Y.COSINE)
    c.append(rows.view(np.float16))
    queries = np.stack([rows32[17], O.gen_rows_f32(43, 0, 1, d)[0]])
    got = c.search(queries, k, threshold=-1.0)
    rc, wr, ws, wc = O.exact_scan_cosine_batch(rows, queries, k)
    assert np.array_equal(got[0], wr) and np.array_equal(got[1], ws) and np.array_equal(got[2], wc)
    assert list(got[0][0]) == [17] + list(range(3000, 3009))
    assert got[3][0] & Y.FLAG_FALLBACK_PATH and got[3][0] & Y.FLAG_TIE_AT_K
    assert not got[3][1] & Y.FLAG_FALLBACK_PATH
    ex = c.search_exhaustive(queries, k)
    assert np.array_equal(ex[0], wr) and np.array_equal(ex[1], ws)
    c.close()


@pytest.mark.parametrize("shape", [(60_000, 96, "f16"), (200_000, 768, "f16"), (120_000, 128, "f32"), (9_000, 100, "f32")])
def test_stage1_error_stays_inside_the_certified_bound(Y, oracle, shape):
    """The certificate is only as good as eps: measured |stage-1 score - exact score| must stay below eps[q] for the
    tensor engine (fp16 / tf32 operands) and the CUDA-core engine."""
    O = oracle
    n, d, dt = shape
    rows32 = O.gen_rows_f32(42, 0, n, d)
    if dt == "f16":
        rows = O.f16_from_float(rows32).reshape(n, d)
        up = O.f16_to_float(rows).reshape(n, d).astype(np.float64)
        c = Y.Corpus(d, Y.F16, Y.COSINE)
        c.append(rows.view(np.float16))
    else:
        up = rows32.astype(np.float64)
        c = Y.Corpus(d, Y.F32, Y.COSINE)
        c.append(rows32)
    q = O.gen_rows_f32(43, 0, 24, d) * np.float32(1.7)
    q[5] *= np.float32(1e-3)
    sub = np.arange(0, n, max(1, n // 20_000))
    want = (up[sub] @ q.astype(np.float64).T).T / (np.linalg.norm(up[sub], axis=1)[None, :] * np.linalg.norm(q.astype(np.float64), axis=1)[:, None])
    for engine in (1, 0):
        got = c.debug_stage1_scores(q, engine, row_start=0, row_stride=max(1, n // 20_000), nrows=len(sub))
        eps = c.debug_last_eps(len(q))
        err = np.abs(got - want).max(axis=1)
        assert np.all(err <= eps), (engine, err.max(), eps.min())
        assert eps.max() < (3e-3 if dt == "f32" and engine == 1 else 6e-4), eps.max()   # tight enough to certify ordinary data
    c.close()


def test_search_device_is_asynchronous_and_finish_resolves(Y, oracle):
    """search_device enqueues without synchronising; search_device_finish reports invalid queries and resolves the
    queries the certificate rejected, patching the device outputs in place.  Packed output + packed merge."""
    import torch
    O = oracle
    n, d, nq, k = 150_000, 64, 16, 10
    rng = np.random.default_rng(3)
    q_adv = O.gen_rows_f32(78, 0, 1, d)[0]
    rows32, _ = near_tie_corpus(O, n, d, q_adv, 250, 1e-4, 42, rng)
    rows = O.f16_from_float(rows32).reshape(n, d)
    queries = O.gen_rows_f32(43, 0, nq, d)
    queries[4] = q_adv
    R, per = 2, n // 2
    packed = torch.zeros((R, nq * k * 12), dtype=torch.uint8, device="cuda")
    dq = torch.from_numpy(queries).cuda()
    shards = []
    for r in range(R):
        c = Y.Corpus(d, Y.F16, Y.COSINE)
        c.append(rows[r * per:(r + 1) * per].view(np.float16), rowids=np.arange(r * per, (r + 1) * per))
        base = packed[r].data_ptr()
        c.search_device(dq.data_ptr(), nq, k, -1.0, base, base + nq * k * 8)
        shards.append(c)
    resolved = [c.search_device_finish() for c in shards]
    assert sum(resolved) >= 1                                        # the near-tie query went through the exhaustive level
    out_r = torch.empty((nq, k), dtype=torch.int64, device="cuda")
    out_s = torch.empty((nq, k), dtype=torch.float32, device="cuda")
    cnt = torch.empty((nq,), dtype=torch.int32, device="cuda")
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    shards[0].merge_packed_device(packed.data_ptr(), R, nq, k, out_r.data_ptr(), out_s.data_ptr(), cnt.data_ptr(), stream=side.cuda_stream)
    side.synchronize()
    rc, wr, ws, wc = O.exact_scan_cosine_batch(rows, queries, k)
    assert np.array_equal(out_r.cpu().numpy(), wr) and np.array_equal(out_s.cpu().numpy(), ws)
    assert np.array_equal(cnt.cpu().numpy().astype(np.uint32), wc)
    # an invalid query surfaces at finish, not at enqueue
    bad = queries.copy()
    bad[2] = 0
    dq2 = torch.from_numpy(bad).cuda()
    shards[0].search_device(dq2.data_ptr(), nq, k, -1.0, packed[0].data_ptr(), packed[0].data_ptr() + nq * k * 8)
    with pytest.raises(Y.YamsB200Error) as e:
        shards[0].search_device_finish()
    assert e.value.status == 1
    for c in shards:
        c.close()


@pytest.mark.parametrize("cfg", [(1_000_000, 128, "f32", 16), (300_000, 64, "f16", 40), (70_001, 100, "f32", 5), (3_000, 48, "f32", 3)])
def test_l2_corpus_through_the_tensor_engine(Y, oracle, cfg):
    """L2 corpora (the vec0 surface, vec0_module.hpp:376-430) take the same pipeline: tensor-core ranking by
    2 q.r - |r|^2, float re-scoring in the reference's order, certificate, exhaustive levels.  No dense Q x N scratch."""
    O = oracle
    n, d, dt, nq = cfg
    rows32 = O.gen_rows_f32(42, 0, n, d) * np.float32(3.0)
    rows32[n // 2] = rows32[7]                                      # an exact tie
    if dt == "f16":
        rows16 = O.f16_from_float(rows32).reshape(n, d)
        rows = O.f16_to_float(rows16).reshape(n, d)                 # the values the corpus holds
        c = Y.Corpus(d, Y.F16, Y.L2)
        c.append(rows16.view(np.float16))
    else:
        rows = rows32
        c = Y.Corpus(d, Y.F32, Y.L2)
        c.append(rows)
    queries = O.gen_rows_f32(43, 0, nq, d) * np.float32(2.0)
    queries[1] = rows[7]                                            # distance 0 twice
    k = 10
    rid, dist, cnt, flags = c.search(queries, k)
    if d % 8 == 0:
        assert c.last_timings()["engine"] == "tcgen05"
    # every query against the exact L2 top-k in the reference build's own operation order (AVX lanes when d % 16 == 0,
    # pinned bit for bit in tests/test_oracle_pin.py): ids, distances and counts equal
    wr, wd, wc = O.exact_scan_l2_batch(rows, queries, k)
    assert np.all(wc == k)
    for qi in range(nq):
        assert cnt[qi] == wc[qi], qi
        assert np.array_equal(rid[qi], wr[qi]), (qi, rid[qi], wr[qi])
        assert np.array_equal(dist[qi].view(np.uint32), wd[qi].view(np.uint32)), (qi, dist[qi], wd[qi])
    assert list(rid[1][:2]) == [7, n // 2] and dist[1][0] == 0.0
    assert np.all(np.diff(dist, axis=1) >= 0)
    ex = c.search_exhaustive(queries[:3], k)
    assert np.array_equal(ex[0], rid[:3]) and np.array_equal(ex[1], dist[:3])
    c.close()
