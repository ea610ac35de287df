"""GPU parity of the SimeonPqAdc engine (SURVEY.md §8f N3): index build (normalise + encode) and search (lookup table, ADC scan,
best approxK, exact rerank) against simeon's own ProductQuantizer / PQInnerProductQuery compiled in place and a restatement of
simeonPqSearchUnlocked (src/vector/sqlite_vec_backend.cpp:3868-4056) around them."""
import numpy as np
import pytest

from tests.refdata import digest, expect

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def Y():
    import yams_b200
    assert yams_b200.device_count() > 0
    assert yams_b200.plugin_init() == 0, yams_b200.health()
    return yams_b200


def reference_pq_search(O, key, rows, rowids, tie_keys, codebooks, m, kc, query, k, rerank, threshold):
    """simeonPqSearchUnlocked's answer -> (rowids, scores), as recorded from simeon's own PQ code (tests/refdata.py)."""
    got = expect(key, lambda: np.array(_reference_pq_search(O, rows, rowids, tie_keys, codebooks, m, kc, query, k, rerank, threshold),
                                       dtype=np.float64).reshape(2, -1))
    return [int(r) for r in got[0]], [np.float32(x) for x in got[1]]


def _reference_pq_search(O, rows, rowids, tie_keys, codebooks, m, kc, query, k, rerank, threshold):
    """simeonPqSearchUnlocked, line by line, over simeon's own PQ code (oracle/_ref)."""
    n, d = rows.shape
    normed, ok = O.normalize_like_reference(rows)
    idx = np.nonzero(ok)[0]
    codes = O.pq_encode_ref(codebooks, d, m, kc, normed)                        # :3650-3660
    qn, qok = O.normalize_like_reference(query[None, :])                        # :3895-3898
    if not qok[0] or len(idx) == 0 or k == 0:
        return [], []
    scores, _ = O.pq_scores_ref(codebooks, d, m, kc, qn[0], codes)              # :3963-3975
    approx = min(len(idx), max(k, k * max(1, rerank)))                          # :3952-3959
    order = np.lexsort((tie_keys[idx], -scores.astype(np.float64)))[:approx]   # :3984-3996: (score desc, tie-break key asc)
    recs = []
    for j in order:
        row = idx[j]
        sim = np.float32(O.lib().yo_cosine_similarity_f64(O._p(np.ascontiguousarray(query), O.f32p),
                                                          O._p(np.ascontiguousarray(rows[row]), O.f32p), d))   # :4024-4026
        if sim < np.float32(threshold):                                         # :4036
            continue
        recs.append((sim, int(rowids[row])))
    recs.sort(key=lambda t: (-float(t[0]), t[1]))                               # :4042-4047 (chunk_id order == rowid order here)
    recs = recs[:k]
    return [r for _, r in recs], [s for s, _ in recs]


@pytest.mark.parametrize("cfg", [(12_000, 768, 32, 256), (9_000, 384, 32, 256), (20_000, 128, 8, 64), (5_000, 96, 4, 16)])
def test_pq_index_and_search_match_the_reference_engine(Y, oracle, cfg):
    O = oracle
    n, d, m, kc = cfg
    rng = np.random.default_rng(n)
    rows = O.gen_rows_f32(42, 0, n, d) * rng.uniform(0.5, 3.0, size=(n, 1)).astype(np.float32)   # not unit length: the index normalises
    rows[17] = 0                                                                    # cannot be normalised: left out of the index
    rows[n // 3] = rows[n // 3 + 1]                                                 # identical codes -> equal ADC scores -> tie keys decide
    rowids = (np.arange(n, dtype=np.int64) * 2 + 5)
    tie_keys = rng.integers(0, 1 << 62, size=n).astype(np.uint64)
    normed, ok = O.normalize_like_reference(rows)
    if (n, d) == (20_000, 128):
        codebooks = expect(f"pq.train.{n}.{d}.{m}.{kc}", lambda: O.pq_train_ref(d, m, kc, normed[:4096]))   # the reference's own Lloyd training
    else:
        codebooks = (rng.normal(size=(m, kc, d // m)) / np.sqrt(d)).astype(np.float32).reshape(-1)
    c = Y.Corpus(d, Y.F32, Y.COSINE)
    c.append(rows, rowids=rowids)
    pq = Y.PqIndex(c, m, kc, codebooks, tie_break_keys=tie_keys)
    codes, code_rowids = pq.codes()
    assert np.array_equal(code_rowids, rowids[ok]) and len(codes) == n - 1
    assert np.array_equal(digest(codes), expect(f"pq.codes.{n}.{d}.{m}.{kc}",       # every code byte equals simeon's encode
                                                lambda: digest(O.pq_encode_ref(codebooks, d, m, kc, normed))))
    queries = O.gen_rows_f32(43, 0, 6, d) * np.float32(2.0)
    queries[2] = rows[n // 3] * np.float32(0.5)                                     # hits the duplicated row pair
    for k, rerank, thr in ((10, 2, 0.0), (5, 4, -1.0), (25, 1, 0.1)):
        rid, sc, cnt, flags = pq.search(queries, k, rerank_factor=rerank, threshold=thr)
        for qi in range(len(queries)):
            wr, ws = reference_pq_search(O, f"pq.search.{n}.{d}.{m}.{kc}.{k}.{rerank}.{thr}.{qi}", rows, rowids, tie_keys, codebooks, m, kc,
                                         queries[qi], k, rerank, thr)
            assert cnt[qi] == len(wr), (qi, k)
            assert list(rid[qi, :len(wr)]) == wr, (qi, k)
            assert np.array_equal(sc[qi, :len(wr)], np.array(ws, dtype=np.float32)), (qi, k)
    # a query that cannot be normalised returns nothing (:3896-3898); k == 0 returns nothing
    rid, sc, cnt, flags = pq.search(np.zeros((1, d), dtype=np.float32), 5)
    assert cnt[0] == 0
    assert pq.search(queries[:1], 0)[2][0] == 0
    # a mutated corpus invalidates the index (the reference marks it dirty and rebuilds)
    c.append(rows[:1], rowids=[int(rowids[-1]) + 1])
    with pytest.raises(Y.YamsB200Error):
        pq.search(queries[:1], 5)
    pq.close()
    c.close()


def test_pq_over_an_fp16_corpus_and_row_order_ties(Y, oracle):
    """fp16 corpus (the C2 layout): the index is built from the stored (fp16) values; without tie keys equal approximate
    scores are ordered by row."""
    O = oracle
    n, d, m, kc = 12_000, 256, 16, 256
    rng = np.random.default_rng(3)
    rows16 = O.f16_from_float(O.gen_rows_f32(42, 0, n, d)).reshape(n, d)
    rows = O.f16_to_float(rows16).reshape(n, d)
    rows[100] = rows[50]
    rows16[100] = rows16[50]
    codebooks = (rng.normal(size=(m, kc, d // m)) / np.sqrt(d)).astype(np.float32).reshape(-1)
    c = Y.Corpus(d, Y.F16, Y.COSINE)
    c.append(rows16.view(np.float16))
    pq = Y.PqIndex(c, m, kc, codebooks)
    queries = O.gen_rows_f32(43, 0, 4, d)
    queries[1] = rows[50]
    rid, sc, cnt, flags = pq.search(queries, 10, rerank_factor=2, threshold=-1.0)
    tie = np.arange(n, dtype=np.uint64)
    for qi in range(4):
        wr, ws = reference_pq_search(O, f"pq.fp16.{qi}", rows, np.arange(n), tie, codebooks, m, kc, queries[qi], 10, 2, -1.0)
        assert list(rid[qi, :len(wr)]) == wr and np.array_equal(sc[qi, :len(wr)], np.array(ws, dtype=np.float32))
    assert list(rid[1, :2]) == [50, 100] and flags[1] & Y.FLAG_TIE_AT_K == 0
    pq.close()
    c.close()


def _check_against_reference(O, key, pq, rows, rowids, tie_keys, codebooks, m, kc, queries, k, rerank, thr):
    rid, sc, cnt, flags = pq.search(queries, k, rerank_factor=rerank, threshold=thr)
    for qi in range(len(queries)):
        wr, ws = reference_pq_search(O, f"{key}.{k}.{rerank}.{thr}.{qi}", rows, rowids, tie_keys, codebooks, m, kc, queries[qi], k, rerank, thr)
        assert cnt[qi] == len(wr), (qi, k)
        assert list(rid[qi, :len(wr)]) == wr, (qi, k)
        assert np.array_equal(sc[qi, :len(wr)], np.array(ws, dtype=np.float32)), (qi, k)


def test_pq_filtered_scan_large_index(Y, oracle):
    """>= 64 tiles: the sampled-threshold (filtered) ADC pass replaces the per-tile sorting network; 1, 2 and 5 queries walk the
    1-, 2- and 4-table CTA variants.  Small k (16 centroids) makes equal approximate scores common: tie keys decide."""
    O = oracle
    n, d, m, kc = 300_000, 64, 8, 16
    rng = np.random.default_rng(11)
    rows = O.gen_rows_f32(42, 0, n, d)
    rows[1000:1064] = rows[2000]                                                    # a run of identical rows across the list boundary
    rowids = np.arange(n, dtype=np.int64) + 3
    tie_keys = rng.permutation(n).astype(np.uint64)
    codebooks = (rng.normal(size=(m, kc, d // m)) / np.sqrt(d)).astype(np.float32).reshape(-1)
    c = Y.Corpus(d, Y.F32, Y.COSINE)
    c.append(rows, rowids=rowids)
    pq = Y.PqIndex(c, m, kc, codebooks, tie_break_keys=tie_keys)
    queries = O.gen_rows_f32(43, 0, 5, d)
    queries[1] = rows[2000]
    for nq in (1, 2, 5):
        for k, rerank, thr in ((10, 2, -1.0), (40, 3, 0.0)):
            _check_against_reference(O, f"pq.filtered.{nq}", pq, rows, rowids, tie_keys, codebooks, m, kc, queries[:nq], k, rerank, thr)
    pq.close()
    c.close()


def test_pq_filtered_scan_overflow_falls_back(Y, oracle):
    """The sampled tiles (every 4th of 74) hold only rows pointing away from the query, every other tile rows pointing at it:
    the sample's threshold admits ~237 k rows into a 32 k list; the engine must notice and redo the selection unfiltered."""
    O = oracle
    n, d, m, kc = 300_000, 64, 8, 16
    rng = np.random.default_rng(12)
    query = O.gen_rows_f32(43, 0, 1, d)
    noise = O.gen_rows_f32(42, 0, n, d)
    tile = np.arange(n) // 4096
    sign = np.where((tile % 4 == 0) & (tile < 64), -1.0, 1.0).astype(np.float32)[:, None]
    rows = (noise * np.float32(0.7) + sign * query).astype(np.float32)
    rowids = np.arange(n, dtype=np.int64)
    tie_keys = np.arange(n, dtype=np.uint64)
    codebooks = (rng.normal(size=(m, kc, d // m)) / np.sqrt(d)).astype(np.float32).reshape(-1)
    c = Y.Corpus(d, Y.F32, Y.COSINE)
    c.append(rows, rowids=rowids)
    pq = Y.PqIndex(c, m, kc, codebooks, tie_break_keys=tie_keys)
    _check_against_reference(O, "pq.overflow", pq, rows, rowids, tie_keys, codebooks, m, kc, query, 10, 2, -1.0)
    pq.close()
    c.close()
