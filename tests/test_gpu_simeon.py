"""GPU parity of the Simeon text encoder's default profile (SURVEY.md §8f N4) against simeon's own Encoder compiled in place
(third_party/simeon/src/{simeon,projection,hasher,tokenizer,...}.cpp): bit-identical embeddings."""
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


def corpus_of_texts(rng, n):
    words = ["yams", "content", "addressed", "storage", "chunk", "hash", "vector", "search", "naïve", "日本語", "emoji🙂", "x", "_", "42"]
    texts = [b"", b"a", b"ab", b"abc", b"abcd", "The quick brown fox jumps over the lazy dog".encode()]
    for _ in range(n):
        kind = rng.integers(0, 3)
        if kind == 0:
            L = int(rng.integers(1, 60))
            texts.append(" ".join(words[int(i)] for i in rng.integers(0, len(words), size=L)).encode("utf-8"))
        elif kind == 1:
            texts.append(bytes(rng.integers(0, 256, size=int(rng.integers(1, 3000)), dtype=np.uint8)))   # arbitrary bytes, NULs included
        else:
            texts.append(bytes(rng.integers(97, 123, size=int(rng.integers(5, 20000)), dtype=np.uint8)))
    return texts


@pytest.mark.parametrize("cfg", [
    dict(),                                                         # simeon-v1-384: what YAMS runs
    dict(sketch_dim=8192, output_dim=768),                          # the 768-d variant of BASELINE config C2
    dict(ngram_min=1, ngram_max=8),                                 # 8-byte grams take the whole-word hash path
    dict(ngram_min=7, ngram_max=12, sketch_dim=5000, output_dim=100),   # > 8 bytes: word + tail; non-power-of-two sketch (modulo bucket)
    dict(l2_normalize=0, output_dim=33),                            # raw projection, odd dimension (scalar tail of the normaliser unused)
    dict(output_dim=40),                                            # 40 = 2 x 16 + 8: the normaliser's fused tail
])
def test_simeon_encoder_is_bit_identical(Y, oracle, cfg):
    O = oracle
    rng = np.random.default_rng(len(cfg) + 1)
    texts = corpus_of_texts(rng, 300)
    enc = Y.SimeonEncoder(**cfg)
    got = enc.encode(texts)
    key = "simeon.v1." + ".".join(f"{k}={v}" for k, v in sorted(cfg.items()))
    shape = expect(key + ".shape", lambda: O.simeon_encode_ref(texts, **cfg).shape)
    assert got.shape == tuple(shape)
    assert np.array_equal(digest(got.view(np.uint32)), expect(key + ".digest", lambda: digest(O.simeon_encode_ref(texts, **cfg).view(np.uint32))))
    if cfg.get("l2_normalize", 1):
        norms = np.linalg.norm(got.astype(np.float64), axis=1)
        assert np.all((np.abs(norms - 1) < 1e-5) | (norms == 0))    # texts shorter than ngram_min embed to zero
    # one text at a time == the batch (generateEmbedding vs generateEmbeddings, simeon_embedding_backend.cpp:183-209)
    for i in (0, 5, 17):
        assert np.array_equal(enc.encode([texts[i]])[0], got[i])
    enc.close()


def test_simeon_embeddings_feed_the_scan(Y, oracle):
    """End of the pipeline the encoder exists for: encode -> corpus -> exact search finds the text itself first."""
    rng = np.random.default_rng(9)
    texts = corpus_of_texts(rng, 2000)[6:]
    enc = Y.SimeonEncoder()
    emb = enc.encode(texts)
    c = Y.Corpus(384, Y.F32, Y.COSINE)
    c.append(emb)
    rid, sc, cnt, _ = c.search(emb[:50], 3, threshold=-1.0)
    assert all(rid[i, 0] == i or sc[i, 0] == sc[i, 1] for i in range(50)) and np.all(sc[:, 0] > 0.9999)
    c.close()
    enc.close()


@pytest.mark.parametrize("cfg", [
    dict(profile="yams-default"),                                                     # unconfigured YAMS: CharAndWord + Fwht, 4096 -> 1024
    dict(profile="yams-default", embedding_dim=384),
    dict(profile="yams-default", embedding_dim=768, sketch_dim=8192),
    dict(profile="yams-default", embedding_dim=100, sketch_dim=5000),                 # sketch padded 5000 -> 8192, modulo buckets
    dict(profile="yams-default", embedding_dim=4096),                                 # output_dim == pad_n: every coordinate sampled
    dict(flags=1),                                                                    # word tokens with the Achlioptas projection
    dict(flags=2, output_dim=40, l2_normalize=0),                                     # Fwht without word tokens, raw output
])
def test_simeon_yams_default_profile_is_bit_identical(Y, oracle, cfg):
    """The encoder an unconfigured YAMS builds (simeon_embedding_backend.cpp:18-47,118-135): byte n-grams + word tokens, count
    sketch, FWHT projection, L2 -- against simeon's own Encoder with ngram_mode / projection set the same way."""
    O = oracle
    rng = np.random.default_rng(123)
    texts = corpus_of_texts(rng, 300) + [b"_", b"a_b c-d e.f 0x1F", b"word" * 3000, b"  leading and trailing  ", "Größe_42 naïve".encode()]
    enc = Y.SimeonEncoder(**cfg)
    got = enc.encode(texts)
    c = enc.cfg

    def want():
        return O.simeon_encode_modes_ref(texts, ngram_mode="CharAndWord" if c.flags & Y.SIMEON_WORD_TOKENS else "CharOnly",
                                         projection="Fwht" if c.flags & Y.SIMEON_PROJECTION_FWHT else "AchlioptasSparse",
                                         ngram_min=c.ngram_min, ngram_max=c.ngram_max, sketch_dim=c.sketch_dim, output_dim=c.output_dim,
                                         hash_seed=c.hash_seed, projection_seed=c.projection_seed, l2_normalize=c.l2_normalize)
    key = "simeon.modes." + ".".join(f"{k}={v}" for k, v in sorted(cfg.items()))
    assert got.shape == tuple(expect(key + ".shape", lambda: want().shape))
    assert np.array_equal(digest(got.view(np.uint32)), expect(key + ".digest", lambda: digest(want().view(np.uint32))))
    assert np.array_equal(enc.encode([texts[7]])[0], got[7])
    enc.close()
    # the constraint of the reference constructor (projection.cpp:167-170)
    with pytest.raises(Y.YamsB200Error):
        Y.SimeonEncoder(profile="yams-default", embedding_dim=4096, sketch_dim=2048)


def test_simeon_matches_the_committed_golden_embeddings(Y):
    """tests/golden/simeon_golden.json: simeon's own Encoder run in the build container (make_simeon_golden.py); needs no reference."""
    import json
    import os
    g = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "simeon_golden.json")))
    texts = g["texts"]
    for key, kw in (("simeon_v1_384", dict()), ("yams_default_1024", dict(profile="yams-default")),
                    ("yams_default_384", dict(profile="yams-default", embedding_dim=384))):
        enc = Y.SimeonEncoder(**kw)
        got = enc.encode(texts).view(np.uint32)
        assert np.array_equal(got, np.array(g[key], dtype=np.uint32)), key
        enc.close()
