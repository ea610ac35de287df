"""GPU parity tests of the vector scan through the C ABI, against the CPU oracle's restatement of
bruteForceSearchUnlocked / vec0_run_exact_query and the reference golden vectors."""
import numpy as np
import pytest

from tests.refdata import expect

pytestmark = pytest.mark.gpu

TOL = 1e-4   # the reference tests' own epsilon (sqlite-vec-cpp/tests/test_distances.cpp:16-18)


@pytest.fixture(scope="module")
def Y():
    import yams_b200
    assert yams_b200.device_count() > 0
    assert yams_b200.plugin_init() == 0, yams_b200.health()
    return yams_b200


def check_against_oracle(O, rows, queries, got, k, threshold=-1.0, allowed=None, exact_scores=True):
    rid, sc, cnt, flags = got
    for qi, q in enumerate(queries):
        al = None if allowed is None else allowed[qi]
        rc, wr, ws = O.exact_scan_cosine(rows, q, k, threshold=threshold, allowed=al)
        assert rc == 0
        assert cnt[qi] == len(wr), (qi, cnt[qi], len(wr))
        assert list(rid[qi, :len(wr)]) == list(wr), qi
        if exact_scores:
            assert np.array_equal(sc[qi, :len(wr)], ws), qi      # fp64 rescoring: bit-identical
        else:
            assert np.allclose(sc[qi, :len(wr)], ws, atol=TOL)
        assert (rid[qi, len(wr):] == -1).all()


def test_c1_config_exact(Y, oracle, golden):
    """BASELINE config 1: 1k x 128 fp32, 16 queries, cosine top-10."""
    O = oracle
    rows = O.gen_rows_f32(42, 0, 1000, 128)
    queries = O.gen_rows_f32(43, 0, 16, 128)
    c = Y.Corpus(128, Y.F32, Y.COSINE)
    c.append(rows)
    got = c.search(queries, 10, threshold=-1.0)
    check_against_oracle(O, rows, queries, got, 10)
    for qi, g in enumerate(golden["c1_cosine_top10"]):           # ids the reference itself returns
        assert [int(x) for x in got[0][qi]] == g["idx"]
        assert np.allclose(1.0 - got[1][qi], g["dist"], atol=1e-5)
    assert len(c) == 1000
    c.close()


def test_exact_scan_contract(Y, oracle):
    # /root/reference/tests/unit/vector/vector_smoke_catch2_test.cpp:188-340
    rows = np.zeros((6, 4), dtype=np.float32)
    rows[0] = [1, 0, 0, 0]; rows[1] = [0.9, 0.1, 0, 0]; rows[2] = 0
    rows[3] = [np.nan, 1, 0, 0]; rows[4] = [1e19, 0, 0, 0]; rows[5] = [-1, 0, 0, 0]
    q = np.array([[1, 0, 0, 0]], dtype=np.float32)
    c = Y.Corpus(4, Y.F32, Y.COSINE)
    c.append(rows, rowids=[10, 11, 12, 13, 14, 15])
    rid, sc, cnt, flags = c.search(q, 10, threshold=-1.0)
    assert cnt[0] == 4 and list(rid[0, :4]) == [10, 14, 11, 15]
    assert sc[0, 0] == 1.0 and sc[0, 1] == 1.0 and sc[0, 3] == -1.0
    rid, sc, cnt, flags = c.search(q, 1, threshold=-1.0)
    assert list(rid[0]) == [10] and (flags[0] & 1) == 1          # tie straddles k -> host re-breaks by chunk_id
    rid, sc, cnt, flags = c.search(q, 10, threshold=0.5)
    assert cnt[0] == 3 and list(rid[0, :3]) == [10, 14, 11]
    assert c.search(q, 0)[2][0] == 0                              # k == 0 -> empty (:4123)
    for bad in ([0, 0, 0, 0], [np.nan, 0, 0, 0], [np.inf, 0, 0, 0], [1e-6, 0, 0, 0]):
        with pytest.raises(Y.YamsB200Error) as e:
            c.search(np.array([bad], dtype=np.float32), 3)
        assert e.value.status == 1                                # InvalidArgument (:4127)
    # candidate set (CandidateFilterMode::Exact)
    rid, sc, cnt, flags = c.search(q, 5, threshold=-1.0, allowed=[[11, 15, 99]])
    assert cnt[0] == 2 and list(rid[0, :2]) == [11, 15]
    c.clear()
    assert len(c) == 0 and c.search(q, 3)[2][0] == 0
    c.close()


@pytest.mark.parametrize("dtype", ["f16", "f32"])
def test_sampled_threshold_path_vs_oracle(Y, oracle, dtype):
    """n > 65536 rows: thresholds from a strided sample + filtered scan + exact rescoring."""
    O = oracle
    n, d, nq, k = 150_000, 96, 24, 10
    rows32 = O.gen_rows_f32(42, 0, n, d)
    queries = O.gen_rows_f32(43, 0, nq, d)
    if dtype == "f16":
        rows = O.f16_from_float(rows32).reshape(n, d)             # reference truncating conversion
        c = Y.Corpus(d, Y.F16, Y.COSINE)
        c.append(rows32)                                          # device-side truncating conversion
    else:
        rows = rows32
        c = Y.Corpus(d, Y.F32, Y.COSINE)
        c.append(rows)
    got = c.search(queries, k, threshold=-1.0)
    check_against_oracle(O, rows, queries, got, k)
    got = c.search(queries[:3], 100, threshold=0.1)
    check_against_oracle(O, rows, queries[:3], got, 100, threshold=0.1)
    c.close()


def test_odd_dim_duplicates_and_ties(Y, oracle):
    O = oracle
    n, d = 3000, 37                                               # dim % 8 != 0 -> scalar load path
    rows = O.gen_rows_f32(7, 0, n, d)
    rows[100:140] = rows[5]                                       # 41 identical rows -> equal scores
    rows[2000] = 0
    c = Y.Corpus(d, Y.F32, Y.COSINE)
    c.append(rows)
    queries = np.stack([rows[5], rows[17] + 0.01, -rows[9]])
    for k in (1, 10, 50):
        got = c.search(queries, k, threshold=-1.0)
        check_against_oracle(O, rows, queries, got, k)
    assert c.search(queries[:1], 10)[3][0] & 1                    # ties at the k boundary flagged
    c.close()


def test_candidate_sets_vs_oracle(Y, oracle):
    """BASELINE config 5 shape, scaled down: per-query allowed rowid lists."""
    O = oracle
    n, d, nq, k = 90_000, 64, 12, 10
    rows32 = O.gen_rows_f32(42, 0, n, d)
    rows = O.f16_from_float(rows32).reshape(n, d)
    rowids = np.arange(n, dtype=np.int64) * 3 + 1000              # sparse, non-dense rowids
    c = Y.Corpus(d, Y.F16, Y.COSINE)
    c.append(rows.view(np.float16), rowids=rowids)
    queries = O.gen_rows_f32(43, 0, nq, d)
    rng = np.random.default_rng(5)
    allowed = []
    for qi in range(nq):
        frac = [0.001, 0.01, 0.1][qi % 3]
        sel = np.sort(rng.choice(n, size=max(1, int(n * frac)), replace=False))
        allowed.append(rowids[sel])
    allowed[3] = np.zeros(0, dtype=np.int64)                      # empty candidate list
    rid, sc, cnt, flags = c.search(queries, k, threshold=-1.0, allowed=allowed)
    for qi in range(nq):
        rc, wr, ws = O.exact_scan_cosine(rows, queries[qi], k, threshold=-1.0, rowids=rowids, allowed=allowed[qi])
        assert cnt[qi] == len(wr) and list(rid[qi, :len(wr)]) == list(wr), qi
        assert np.array_equal(sc[qi, :len(wr)], ws)
    c.close()


def test_synthetic_corpus_bits_match_oracle(Y, oracle):
    """Device generator == oracle generator (SURVEY §8d), incl. truncating fp16: identical scores."""
    O = oracle
    n, d = 70_000, 128
    rows = O.f16_from_float(O.gen_rows_f32(42, 1000, n, d)).reshape(n, d)
    c = Y.Corpus(d, Y.F16, Y.COSINE)
    c.append_synthetic(42, 1000, n)
    queries = O.gen_rows_f32(43, 0, 8, d)
    got = c.search(queries, 10, threshold=-1.0)
    rid, sc, cnt, _ = got
    for qi, q in enumerate(queries):
        rc, wr, ws = O.exact_scan_cosine(rows, q, 10, threshold=-1.0, rowids=np.arange(1000, 1000 + n))
        assert list(rid[qi]) == list(wr) and np.array_equal(sc[qi], ws)
    c.close()


def test_vec0_exact_and_l2_surface(Y, oracle):
    O = oracle
    # third_party/sqlite-vec-cpp/tests/test_sqlite_functions.cpp:1261-1399 (exact plans)
    rows = np.array([[0, 0], [3, 4], [1, 0], [0, 2]], dtype=np.float32)
    rid, dist = Y.vec0_exact(np.zeros(2, dtype=np.float32), rows, k=0, rowids=[10, 11, 12, 13])
    assert list(rid) == [10, 12, 13, 11] and np.allclose(dist, [0, 1, 2, 5])
    rid, dist = Y.vec0_exact(np.zeros(2, dtype=np.float32), rows, k=2, rowids=[10, 11, 12, 13])
    assert list(rid) == [10, 12]
    rid, dist = Y.vec0_exact(np.zeros(2, dtype=np.float32), rows, k=0, rowids=[10, 11, 12, 13], rowid_range=(11, 12))
    assert list(rid) == [12, 11]
    # larger random case incl. ties
    big = O.gen_rows_f32(3, 0, 5000, 48)
    big[77] = big[5]
    q = O.gen_rows_f32(4, 0, 1, 48)[0]
    # both against the exact L2 order of the reference build's own float distances (AVX lanes for d = 48): equal ids and
    # bit-equal distances
    for k in (0, 25):
        wr, wd, wc = O.exact_scan_l2_batch(big, q[None, :], k or len(big))
        rid, dist = Y.vec0_exact(q, big, k=k)
        assert len(rid) == wc[0] and np.array_equal(rid, wr[0]) and np.array_equal(dist.view(np.uint32), wd[0].view(np.uint32))
    # corpus with the L2 metric (top-k ascending by distance)
    c = Y.Corpus(48, Y.F32, Y.L2)
    c.append(big)
    rid, sc, cnt, _ = c.search(q[None, :], 10)
    wr, wd, wc = O.exact_scan_l2_batch(big, q[None, :], 10)
    assert np.array_equal(cnt, wc) and np.array_equal(rid, wr) and np.array_equal(sc.view(np.uint32), wd.view(np.uint32))
    c.close()
    # test_batch_distance.cpp:19-104 KATs through the same surface
    rows = np.array([[1, 2, 3], [2, 3, 4], [0, 0, 0], [4, 5, 6]], dtype=np.float32)
    rid, dist = Y.vec0_exact(np.array([1, 2, 3], dtype=np.float32), rows, k=2)
    assert list(rid) == [0, 1] and np.allclose(dist, [0, np.sqrt(3.0)], atol=TOL)


def test_pairwise_c_api(Y):
    # /root/reference/tests/unit/vector/sqlite_vec_c_api_smoke_catch2_test.cpp:19-75
    rc, v = Y.vec_distance_l2(np.ones(16), np.ones(16))
    assert rc == 0 and abs(v) < 1e-6
    a = np.array([1, 2, 3, 4, 5, 6, 7, 8] * 2, dtype=np.float32)
    b = np.array([1, 2, 3, 4, 5, 6, 7, 8, 2, 3, 4, 5, 6, 7, 8, 9], dtype=np.float32)
    rc, v = Y.vec_distance_l2(a, b)
    assert rc == 0 and abs(v - np.sqrt(8.0)) < 1e-5
    rc, v = Y.vec_distance_cosine(np.full(16, 0.5), np.full(16, 0.5))
    assert rc == 0 and abs(v) < 1e-5
    assert Y.vec_distance_l2(np.ones(8), np.ones(16))[0] != 0
    assert Y.vec_distance_cosine(np.ones(8), np.ones(16))[0] != 0
    # test_distances.cpp:20-53 / distance_metrics_test.cpp:254-292 KATs
    assert abs(Y.vec_distance_l2([1, 2, 3, 4], [2, 3, 4, 5])[1] - 2.0) < TOL
    assert abs(Y.vec_distance_cosine([1, 2, 3], [-1, -2, -3])[1] - 2.0) < 1e-5
    assert abs(Y.vec_distance_cosine([0.6, 0.8], [0.8, 0.6])[1] - 0.04) < 1e-5
    assert Y.vec_distance_cosine([0, 0, 0], [1, 2, 3])[1] == 1.0


def test_partial_topk_merge_like_allgather(Y, oracle):
    """Row-sharded scan on one GPU: R shard corpora -> search_device partials laid out [R][Q][k] (what an
    all-gather produces) -> merge_partials_device == single-corpus answer."""
    import torch
    O = oracle
    n, d, nq, k, R = 80_000, 64, 16, 10, 4
    rows = O.f16_from_float(O.gen_rows_f32(42, 0, n, d)).reshape(n, d)
    queries = O.gen_rows_f32(43, 0, nq, d)
    dq = torch.from_numpy(queries).cuda()
    part_r = torch.empty((R, nq, k), dtype=torch.int64, device="cuda")
    part_s = torch.empty((R, nq, k), dtype=torch.float32, device="cuda")
    shards = []
    per = n // R
    for r in range(R):
        c = Y.Corpus(d, Y.F16, Y.COSINE)
        c.append(rows[r * per:(r + 1) * per].view(np.float16), rowids=np.arange(r * per, (r + 1) * per))
        c.search_device(dq.data_ptr(), nq, k, -1.0, part_r[r].data_ptr(), part_s[r].data_ptr())
        c.sync()
        shards.append(c)
    out_r = torch.empty((nq, k), dtype=torch.int64, device="cuda")
    out_s = torch.empty((nq, k), dtype=torch.float32, device="cuda")
    shards[0].merge_partials_device(part_r.data_ptr(), part_s.data_ptr(), R, nq, k, out_r.data_ptr(), out_s.data_ptr())
    shards[0].sync()
    for qi in range(nq):
        rc, wr, ws = O.exact_scan_cosine(rows, queries[qi], k, threshold=-1.0)
        assert list(out_r[qi].cpu().numpy()) == list(wr)
        assert np.array_equal(out_s[qi].cpu().numpy(), ws)
    for c in shards:
        c.close()


@pytest.mark.parametrize("shape", [(1000, 128, 16), (5000, 768, 300), (777, 72, 5), (40000, 64, 257)])
def test_tcgen05_engine_matches_cuda_core_engine(Y, oracle, shape):
    """Dense stage-1 scores: tensor-core engine vs CUDA-core engine vs the oracle's double-precision cosine."""
    O = oracle
    n, d, nq = shape
    rows32 = O.gen_rows_f32(42, 0, n, d)
    rows16 = O.f16_from_float(rows32).reshape(n, d)
    c = Y.Corpus(d, Y.F16, Y.COSINE)
    c.append(rows16.view(np.float16))
    q = O.gen_rows_f32(43, 0, nq, d) * np.float32(3.0)            # non-unit queries: 1/|q| folding
    cc = c.debug_stage1_scores(q, 0)
    tc = c.debug_stage1_scores(q, 1)
    assert np.isfinite(tc).all()
    assert np.abs(cc - tc).max() < 1e-3, np.abs(cc - tc).max()
    up = O.f16_to_float(rows16).reshape(n, d).astype(np.float64)
    qn = q.astype(np.float64)
    want = (up @ qn.T).T / (np.linalg.norm(up, axis=1)[None, :] * np.linalg.norm(qn, axis=1)[:, None])
    assert np.abs(tc - want).max() < 1e-3
    # strided rows (the sampling pass)
    ts = c.debug_stage1_scores(q[:3], 1, row_start=0, row_stride=7, nrows=n // 7)
    assert np.abs(ts - want[:3, 0:7 * (n // 7):7]).max() < 1e-3
    c.close()


@pytest.mark.parametrize("nq", [1, 3, 17, 40, 100])
def test_small_query_batches_through_tensor_engine(Y, oracle, nq):
    """Query tiles that are not a multiple of the 32-column TMEM chunk: stale accumulator columns must never
    reach the candidate lists (Q=1 once wrote past the per-query counters)."""
    O = oracle
    n, d = 100_000, 64
    rows = O.f16_from_float(O.gen_rows_f32(42, 0, n, d)).reshape(n, d)
    c = Y.Corpus(d, Y.F16, Y.COSINE)
    c.append_synthetic(42, 0, n)
    queries = O.gen_rows_f32(43, 0, nq, d)
    for _ in range(3):      # repeated searches reuse TMEM columns with stale contents
        got = c.search(queries, 10, threshold=-1.0)
    assert c.last_timings()["engine"] == "tcgen05"
    check_against_oracle(O, rows, queries, got, 10)
    c.close()


def test_large_k_and_many_queries_through_tensor_engine(Y, oracle):
    O = oracle
    n, d, nq = 120_000, 128, 300
    rows = O.f16_from_float(O.gen_rows_f32(42, 0, n, d)).reshape(n, d)
    c = Y.Corpus(d, Y.F16, Y.COSINE)
    c.append_synthetic(42, 0, n)
    queries = O.gen_rows_f32(43, 0, nq, d)
    got = c.search(queries, 10, threshold=-1.0)
    assert c.last_timings()["engine"] == "tcgen05"
    sub = list(range(0, nq, 37))
    check_against_oracle(O, rows, queries[sub], tuple(x[sub] for x in got), 10)
    c.close()


def test_cpp_host_adapters(Y, tmp_path):
    """yams_b200/host/b200_host.hpp (IChunker / IContentHasher / IVectorStore shaped C++ adapters) over the C ABI."""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "test_host_adapters")
    subprocess.check_call(["/usr/bin/g++", "-std=c++20", "-O1", os.path.join(root, "tests", "host_cpp", "test_host_adapters.cpp"),
                           "-o", exe, "-L" + os.path.join(root, "yams_b200"), "-lyams_b200",
                           "-Wl,-rpath," + os.path.join(root, "yams_b200")])
    out = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0 and "ALL OK" in out.stdout, out.stdout + out.stderr


def test_plugin_loader_walks_the_vtables(Y, tmp_path):
    """dlopen(RTLD_LAZY | RTLD_LOCAL) + dlsym of the 8 envelope symbols + get_interface + a chunk and a search through the
    returned vtables, exactly as the daemon's AbiPluginLoader reaches a plugin (abi_plugin_loader.cpp:303-341,657-680)."""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "test_plugin_loader")
    subprocess.check_call(["/usr/bin/g++", "-std=c++20", "-O1", os.path.join(root, "tests", "host_cpp", "test_plugin_loader.cpp"),
                           "-o", exe, "-ldl"])
    out = subprocess.run([exe, os.path.join(root, "yams_b200", "libyams_b200.so")], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0 and "LOADER OK" in out.stdout, out.stdout + out.stderr


def test_sqlite_glue_through_a_stand_in_sqlite(Y, tmp_path):
    """csrc/sqlite_glue.cpp (sqlite3_vec_init + vec_distance_l2/cosine/l1 SQL scalars; reference: sqlite_vec_c_api.cpp:15-55,
    sqlite/functions.hpp:76-278) compiled against the stand-in sqlite3.h of tests/host_cpp/mock_sqlite3 and driven like SQL would."""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "test_sqlite_glue")
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-O1", "-I" + os.path.join(root, "tests", "host_cpp", "mock_sqlite3"),
                           os.path.join(root, "yams_b200", "csrc", "sqlite_glue.cpp"), os.path.join(root, "tests", "host_cpp", "test_sqlite_glue.cpp"),
                           "-o", exe, "-L" + os.path.join(root, "yams_b200"), "-lyams_b200", "-Wl,-rpath," + os.path.join(root, "yams_b200")])
    out = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0 and "GLUE OK" in out.stdout, out.stdout + out.stderr


def test_pairwise_and_batch_operators_are_bit_identical_to_the_reference_build(Y, oracle):
    """R5/R6/R7: distances::{l2,cosine}_distance<float> in the operation order of the reference build (AVX lanes, FMA contraction
    where the compiler applies it) -- compared bit for bit with the reference compiled in place, at dims that take every path."""
    O = oracle

    def ref_dist(fn, q, rows):
        R = O.ref()
        return [getattr(R, fn)(O._p(q, O.f32p), O._p(np.ascontiguousarray(r), O.f32p), len(q)) for r in rows]
    rng = np.random.default_rng(9)
    for d in (1, 5, 7, 8, 13, 16, 31, 32, 100, 384, 768, 1536):
        for t in range(6):
            a = rng.normal(size=d).astype(np.float32)
            b = rng.normal(size=d).astype(np.float32)
            want_l2, want_cos = expect(f"knn.pairwise.{d}.{t}", lambda: np.array(
                ref_dist("ref_l2_distance", a, [b]) + ref_dist("ref_cosine_distance", a, [b]), dtype=np.float32))
            rc, got = Y.vec_distance_l2(a, b)
            assert rc == 0 and np.float32(got) == want_l2, ("l2", d)
            rc, got = Y.vec_distance_cosine(a, b)
            assert rc == 0 and np.float32(got) == want_cos, ("cos", d)
    for d, n in ((768, 4000), (100, 3000), (16, 500)):
        rows = rng.normal(size=(n, d)).astype(np.float32)
        q = rng.normal(size=d).astype(np.float32)
        for metric, om, fn in ((Y.COSINE, O.METRIC_COSINE, "ref_cosine_distance"), (Y.L2, O.METRIC_L2, "ref_l2_distance")):
            got = Y.batch_distance(q, rows, metric=metric, mode=Y.BATCH_ALL)
            want = expect(f"knn.batch_all.{d}.{metric}", lambda: np.array(ref_dist(fn, q, rows), dtype=np.float32))
            assert np.array_equal(got, want), (metric, d)
            idx, dist = Y.batch_distance(q, rows, metric=metric, mode=Y.BATCH_TOP_K, k=10)
            ri = expect(f"knn.batch_top_k.{d}.{metric}.idx", lambda: O.batch_top_k(q, rows, 10, metric=om, use_ref=True)[0])
            rd = expect(f"knn.batch_top_k.{d}.{metric}.dist", lambda: O.batch_top_k(q, rows, 10, metric=om, use_ref=True)[1])
            assert np.array_equal(dist, rd) and (list(idx) == list(ri) or len(set(rd)) < 10)
    # L1 (the SQL scalar vec_distance_l1): both paths of distances/l1.hpp against a float64 evaluation
    for d in (3, 7, 8, 100):
        a = rng.normal(size=d).astype(np.float32)
        b = rng.normal(size=d).astype(np.float32)
        rc, got = Y.vec_distance_l1(a, b)
        assert rc == 0 and abs(got - np.abs(a.astype(np.float64) - b.astype(np.float64)).sum()) < 1e-4 * d
    # computeCosineSimilarity for many pairs in one pass == one call per pair
    A = rng.normal(size=(50, 384)).astype(np.float32)
    B = rng.normal(size=(50, 384)).astype(np.float32)
    many = Y.compute_cosine_similarity_many(A, B)
    assert all(many[i] == Y.compute_cosine_similarity(A[i], B[i]) == O.lib().yo_cosine_similarity_f64(O._p(A[i], O.f32p), O._p(B[i], O.f32p), 384)
               for i in range(50))


def test_all_matching_candidate_rows(Y, oracle):
    """ExactRowSelection::AllMatching (sqlite_vec_backend.cpp:4283-4288,4315-4316): every passing candidate row."""
    O = oracle
    n, d = 20_000, 48
    rows = O.gen_rows_f32(42, 0, n, d)
    rows[123] = 0                      # zero norm -> skipped
    rows[77] = rows[5]                 # tie
    rowids = np.arange(n, dtype=np.int64) * 2 + 7
    c = Y.Corpus(d, Y.F32, Y.COSINE)
    c.append(rows, rowids=rowids)
    q = O.gen_rows_f32(43, 0, 1, d)[0]
    rng = np.random.default_rng(3)
    sel = np.sort(rng.choice(n, size=3000, replace=False))
    sel = np.unique(np.concatenate([sel, [5, 77, 123]]))
    allowed = np.concatenate([rowids[sel], [10**9]])           # one rowid that does not exist
    for thr in (-1.0, 0.05):
        rid, sc = c.search_all_matching(q, threshold=thr, allowed=np.concatenate([allowed[::-1], allowed[:5]]))
        rc, wr, ws = O.exact_scan_cosine(rows, q, 1, threshold=thr, rowids=rowids, allowed=np.sort(allowed), all_matching=True)
        assert rc == 0 and list(rid) == list(wr) and np.array_equal(sc, ws), thr
    rid, sc = c.search_all_matching(q, threshold=0.2)           # whole corpus
    rc, wr, ws = O.exact_scan_cosine(rows, q, 1, threshold=0.2, rowids=rowids, all_matching=True)
    assert list(rid) == list(wr) and np.array_equal(sc, ws)
    with pytest.raises(Y.YamsB200Error):
        c.search_all_matching(np.zeros(d, dtype=np.float32))
    c.close()


def test_batch_distance_surface(Y, oracle):
    """distances/batch.hpp:24-146 (batch_distance, batch_top_k, batch_distance_filtered), both metrics; the reference
    tests' epsilon 1e-4 (test_batch_distance.cpp:19-104)."""
    import ctypes as C
    O = oracle
    n, d = 5000, 96
    rows = O.gen_rows_f32(7, 0, n, d)
    rows[17] = 0                                            # zero norm: cosine distance 1.0 (cosine.hpp:64-68)
    rows[40] = rows[3]
    q = O.gen_rows_f32(8, 0, 1, d)[0]
    f32p = C.POINTER(C.c_float)
    for metric, om, fn in ((Y.COSINE, O.METRIC_COSINE, O.lib().yo_cosine_distance_f32), (Y.L2, O.METRIC_L2, O.lib().yo_l2_distance_f32)):
        want = np.array([fn(q.ctypes.data_as(f32p), rows[i].ctypes.data_as(f32p), d) for i in range(n)], dtype=np.float32)
        got = Y.batch_distance(q, rows, metric=metric, mode=Y.BATCH_ALL)
        assert got.shape == (n,) and np.max(np.abs(got - want)) <= 1e-4
        if metric == Y.COSINE:
            assert got[17] == 1.0
        # top-k: ascending, ids equal up to near-ties
        for k in (1, 10, 257, n + 5):
            idx, dist = Y.batch_distance(q, rows, metric=metric, mode=Y.BATCH_TOP_K, k=k)
            wi, wd = O.batch_top_k(q, rows, k, metric=om)
            m = min(k, n)
            assert len(idx) == m == len(wi)
            assert np.all(np.diff(dist) >= 0)
            assert np.max(np.abs(dist - wd)) <= 1e-4
            assert np.max(np.abs(want[idx.astype(np.int64)] - dist)) <= 1e-4
            differ = idx != wi
            assert np.all(np.abs(want[idx[differ].astype(np.int64)] - want[wi[differ].astype(np.int64)]) <= 1e-4)
        # filtered: strictly below the threshold, sorted
        thr = float(np.sort(want)[300]) + 1e-3
        idx, dist = Y.batch_distance(q, rows, metric=metric, mode=Y.BATCH_FILTERED, threshold=thr)
        sure = np.nonzero(want < thr - 1e-4)[0]
        maybe = np.nonzero(want < thr + 1e-4)[0]
        assert set(sure) <= set(idx.astype(np.int64)) <= set(maybe)
        assert np.all(np.diff(dist) >= 0) and np.all(dist < thr)
    assert len(Y.batch_distance(q, np.zeros((0, d), np.float32))) == 0
    idx, _ = Y.batch_distance(q, rows, mode=Y.BATCH_TOP_K, k=0)
    assert len(idx) == 0


def test_compute_cosine_similarity_is_bit_identical(Y, oracle):
    """VectorDatabase::computeCosineSimilarity (vector_database.cpp:1786-1810)."""
    import ctypes as C
    O = oracle
    f32p = C.POINTER(C.c_float)
    for d in (1, 3, 128, 769, 4096):
        ab = O.gen_rows_f32(100 + d, 0, 2, d) * np.float32(3.7)
        want = O.lib().yo_cosine_similarity_f64(ab[0].ctypes.data_as(f32p), ab[1].ctypes.data_as(f32p), d)
        assert Y.compute_cosine_similarity(ab[0], ab[1]) == want
    assert Y.compute_cosine_similarity(np.ones(4), np.ones(5)) == 0.0          # size mismatch
    assert Y.compute_cosine_similarity(np.zeros(8), np.ones(8)) == 0.0         # zero norm
    assert Y.compute_cosine_similarity(np.ones(8), np.ones(8)) == pytest.approx(1.0, abs=1e-15)


def test_corpus_remove_keeps_scan_order(Y, oracle):
    """deleteVector / deleteVectorsByDocument mirror: after removing rows the scan equals a scan of the remaining table."""
    O = oracle
    for dtype, d in ((Y.F32, 40), (Y.F16, 64), (Y.F32, 33)):
        n = 30_000
        rows = O.gen_rows_f32(11, 0, n, d)
        rowids = np.arange(n, dtype=np.int64) * 3 + 1
        c = Y.Corpus(d, dtype, Y.COSINE)
        c.append(rows, rowids=rowids)                        # F16 corpora convert with the truncating from_float
        stored = O.f16_from_float(rows) if dtype == Y.F16 else rows
        rng = np.random.default_rng(5)
        gone = np.sort(rng.choice(n, size=7000, replace=False))
        gone = np.unique(np.concatenate([gone, [0, n - 1]]))
        ask = np.concatenate([rowids[gone][::-1], [2, 10**12], rowids[gone][:10]])   # unknown ids and duplicates are ignored
        assert c.remove(ask) == len(gone)
        keep = np.setdiff1d(np.arange(n), gone)
        assert len(c) == len(keep)
        qs = O.gen_rows_f32(12, 0, 4, d)
        rid, sc, cnt, _ = c.search(qs, k=10)
        rc, wr, ws, wc = O.exact_scan_cosine_batch(stored[keep], qs, 10)
        assert rc == 0
        assert np.array_equal(rid, rowids[keep][wr]) and np.array_equal(sc, ws)
        # appending after a removal continues above the last remaining rowid
        extra = O.gen_rows_f32(13, 0, 5, d)
        with pytest.raises(Y.YamsB200Error):
            c.append(extra, rowids=np.arange(5, dtype=np.int64))
        new_ids = rowids[keep][-1] + 1 + np.arange(5, dtype=np.int64)
        c.append(extra, rowids=new_ids)
        assert len(c) == len(keep) + 5
        assert c.remove(rowids[keep]) == len(keep) and len(c) == 5
        assert c.remove(new_ids) == 5 and len(c) == 0
        c.close()


@pytest.mark.parametrize("dtype_name,d", [("f16", 64), ("f32", 36), ("f32", 30), ("f16", 20)])
def test_candidate_sets_direct_and_masked_paths(Y, oracle, dtype_name, d):
    """Candidate sets take one of two device paths (DESIGN.md §4.4): small ascending lists are scored row by row
    (gather_score_kernel), everything else by a masked corpus pass with thresholds calibrated on the allowed sample
    rows.  Both must equal the reference scan restricted to the candidate set (sqlite_vec_backend.cpp:4138-4175)."""
    O = oracle
    n, nq, k = 150_000, 6, 10
    rows32 = O.gen_rows_f32(21, 0, n, d)
    rows32[500] = 0
    if dtype_name == "f16":
        stored = O.f16_from_float(rows32).reshape(n, d)
        c = Y.Corpus(d, Y.F16, Y.COSINE)
        c.append(stored.view(np.float16), rowids=None)
    else:
        stored = rows32
        c = Y.Corpus(d, Y.F32, Y.COSINE)
        c.append(stored)
    rowids = np.arange(n, dtype=np.int64)
    queries = O.gen_rows_f32(22, 0, nq, d)
    rng = np.random.default_rng(17)

    def check(allowed, what):
        rid, sc, cnt, flags = c.search(queries, k, threshold=-1.0, allowed=allowed)
        for qi in range(nq):
            al = np.unique(np.asarray(allowed[qi], dtype=np.int64))
            rc, wr, ws = O.exact_scan_cosine(stored, queries[qi], k, threshold=-1.0, rowids=rowids, allowed=al)
            assert cnt[qi] == len(wr) and list(rid[qi, :len(wr)]) == list(wr), (what, qi)
            assert np.array_equal(sc[qi, :len(wr)], ws), (what, qi)

    # direct: ascending lists with repeats, ids that do not exist, a list shorter than k, an empty list, the zero row
    small = []
    for qi in range(nq):
        sel = np.sort(rng.choice(n, size=[3, 40, 700, 5000, 1, 2500][qi], replace=False))
        small.append(np.sort(np.concatenate([sel, sel[:2], [500], [n + 5, n + 9]])).astype(np.int64))
    small[4] = np.zeros(0, dtype=np.int64)
    check(small, "direct")
    # masked pass, few allowed rows (unsorted lists cannot take the direct path): thresholds fall back to -inf
    check([a[::-1].copy() for a in small], "masked-small")
    # masked pass, large lists: thresholds come from the allowed rows of the sample
    big = [np.sort(rng.choice(n, size=int(n * f), replace=False)).astype(np.int64) for f in (0.6, 0.3, 0.9, 0.05, 0.5, 0.7)]
    check(big, "masked-big")
    c.close()


def test_fp32_corpus_tf32_engine_vs_oracle(Y, oracle):
    """fp32 rows (the reference's BLOB layout, sqlite_vec_backend.cpp:343-363) take the kind::tf32 tensor-core engine for
    stage 1; the returned ids and scores must still equal the reference's double-precision scan."""
    O = oracle
    n, d, nq, k = 300_000, 128, 40, 10
    rows = O.gen_rows_f32(42, 0, n, d)
    rows[1234] = 0
    rows[777] = rows[5]
    c = Y.Corpus(d, Y.F32, Y.COSINE)
    c.append(rows)
    queries = O.gen_rows_f32(43, 0, nq, d)
    queries[3] = rows[5] * np.float32(2.5)                      # exact duplicates score 1.0 and tie
    got = c.search(queries, k, threshold=-1.0)
    assert c.last_timings()["engine"] == "tcgen05"
    rc, wr, ws, wc = O.exact_scan_cosine_batch(rows, queries, k)
    assert rc == 0 and np.array_equal(got[2], wc)
    assert np.array_equal(got[0], wr) and np.array_equal(got[1], ws)
    assert not np.any(got[3] & 2)                               # no query needed the exhaustive fallback
    # a dimension that is not a multiple of the 32-element K block (TMA zero-fills the tail), small batch
    d2 = 100
    rows2 = O.gen_rows_f32(44, 0, 120_000, d2)
    c2 = Y.Corpus(d2, Y.F32, Y.COSINE)
    c2.append(rows2)
    q2 = O.gen_rows_f32(45, 0, 3, d2)
    got2 = c2.search(q2, 7, threshold=0.1)
    rc, wr, ws, wc = O.exact_scan_cosine_batch(rows2, q2, 7, threshold=0.1)
    assert np.array_equal(got2[2], wc)
    for qi in range(3):
        assert list(got2[0][qi][:wc[qi]]) == list(wr[qi][:wc[qi]]) and np.array_equal(got2[1][qi][:wc[qi]], ws[qi][:wc[qi]])
    c.close()
    c2.close()


def test_concurrent_searches_on_one_corpus(Y, oracle):
    """The reference backend is shared by daemon worker threads (shared_mutex around the scan,
    sqlite_vec_backend.cpp:1433-1568): concurrent callers on one corpus must each get their own answer."""
    import threading
    O = oracle
    n, d = 120_000, 64
    c = Y.Corpus(d, Y.F16, Y.COSINE)
    c.append_synthetic(42, 0, n)
    batches = [O.gen_rows_f32(50 + t, 0, 5 + t, d) for t in range(6)]
    want = [c.search(b, 10) for b in batches]
    got = [None] * len(batches)
    errs = []

    def work(i):
        try:
            for _ in range(20):
                got[i] = c.search(batches[i], 10)
        except Exception as e:   # noqa: BLE001
            errs.append(e)

    ts = [threading.Thread(target=work, args=(i,)) for i in range(len(batches))]
    for th in ts:
        th.start()
    for th in ts:
        th.join()
    assert not errs
    for i in range(len(batches)):
        assert np.array_equal(got[i][0], want[i][0]) and np.array_equal(got[i][1], want[i][1])
    c.close()


def test_worker_threads_bind_the_plugin_device(Y):
    """A fresh host thread starts on CUDA device 0 whatever the plugin was initialised with: every handle-based entry must bind
    the handle's device itself (model_provider_v1.h:45 "thread-safe unless documented").  Needs a second GPU."""
    if Y.device_count() < 2:
        pytest.skip("needs two GPUs")
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = """
import threading, sys
import numpy as np
sys.path.insert(0, %r)
import yams_b200 as Y
assert Y.plugin_init({"device": 1}) == 0, Y.health()
assert Y.health()["device"] == 1
c = Y.Corpus(64, Y.F16, Y.COSINE)
c.append_synthetic(42, 0, 120000)
q = np.random.default_rng(0).normal(size=(5, 64)).astype(np.float32)
data = (np.arange(3 << 20, dtype=np.uint64) * 2654435761 >> 7).astype(np.uint8)
want = c.search(q, 7)
want_chunks = Y.chunk_and_hash(data)
got = {}
def work():
    got["s"] = c.search(q, 7)                       # corpus handle created on device 1, called from a device-0 thread
    got["c"] = Y.chunk_and_hash(data)               # pooled ingest workspace
    got["a"] = c.search_all_matching(q[0], 0.2)
    c.append_synthetic(42, 120000, 1000)
    got["n"] = len(c)
t = threading.Thread(target=work); t.start(); t.join()
assert np.array_equal(got["s"][0], want[0]) and np.array_equal(got["s"][1], want[1])
assert np.array_equal(got["c"], want_chunks) and got["n"] == 121000 and len(got["a"][0]) > 0
print("THREADS OK")
""" % root
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "THREADS OK" in out.stdout, out.stdout + out.stderr


def test_large_k(Y, oracle):
    """k in the thousands (rerank windows): K' = k + k/4 survivors are ordered in shared memory (limit k <= 3072)."""
    O = oracle
    n, d = 90_000, 32
    rows = O.f16_from_float(O.gen_rows_f32(42, 0, n, d)).reshape(n, d)
    c = Y.Corpus(d, Y.F16, Y.COSINE)
    c.append(rows.view(np.float16))
    queries = O.gen_rows_f32(43, 0, 3, d)
    for k in (769, 2000, 3072):
        rid, sc, cnt, _ = c.search(queries, k, threshold=-1.0)
        rc, wr, ws, wc = O.exact_scan_cosine_batch(rows, queries, k)
        assert np.array_equal(cnt, wc) and np.array_equal(rid, wr) and np.array_equal(sc, ws), k
    with pytest.raises(Y.YamsB200Error):
        c.search(queries, 3073)
    c.close()
