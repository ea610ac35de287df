"""GPU parity of the manifest step (SURVEY.md §8f N2): ChunkRef table + ManifestManager::calculateChecksum
(src/manifest/manifest_manager.cpp:411-436,705-730) computed on the device from the chunk table of chunk_and_hash."""
import hashlib

import numpy as np
import pytest

from tests.refdata import expect, key_of

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def Y():
    import yams_b200
    assert yams_b200.device_count() > 0
    assert yams_b200.plugin_init() == 0, yams_b200.health()
    return yams_b200


def check(Y, O, chunks, file_digest, file_size):
    refs, summ = Y.manifest_build(chunks, file_digest, file_size)
    want = O.manifest_checksum(file_digest, file_size, chunks["digest"], chunks["offset"], chunks["size"])
    assert summ["checksum"] == want
    dg, of, sz = (np.ascontiguousarray(chunks[f]) for f in ("digest", "offset", "size"))
    crc, valid = expect("manifest." + key_of(file_digest, file_size, dg, of, sz),
                        lambda: O.manifest_checksum(file_digest, file_size, dg, of, sz, use_ref=True))
    assert crc == summ["checksum"] and valid == summ["valid"]
    assert summ["chunk_count"] == len(chunks)
    for i in range(0, len(chunks), max(1, len(chunks) // 50)):
        assert refs[i]["hash"].decode() == bytes(chunks[i]["digest"]).hex()
        assert refs[i]["offset"] == chunks[i]["offset"] and refs[i]["size"] == chunks[i]["size"] and refs[i]["flags"] == 0
    return summ


def test_manifest_of_a_chunked_stream(Y, oracle):
    O = oracle
    data = O.gen_bytes(12345, 0, 96 << 20)
    chunks = Y.chunk_and_hash(data, Y.default_config())
    fd = hashlib.sha256(data.tobytes()).digest()
    summ = check(Y, O, chunks, fd, len(data))
    assert summ["valid"] == 1 and summ["offsets_sequential"] == 1 and summ["total_size"] == len(data)
    # small-chunk config: many records, every fold level exercised (64 per thread, tree, final chain)
    cfg = Y.default_config(min_chunk=64, max_chunk=1024, mask=0x3F)
    small = Y.chunk_and_hash(data[: 48 << 20], cfg)
    assert len(small) > 200_000
    check(Y, O, small, fd, 48 << 20)


@pytest.mark.parametrize("n", [0, 1, 2, 63, 64, 65, 4097])
def test_manifest_record_counts_and_invalid_tables(Y, oracle, n):
    O = oracle
    rng = np.random.default_rng(n)
    chunks = np.zeros(n, dtype=Y.lib_chunk_dtype())
    chunks["digest"] = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    chunks["size"] = rng.integers(1, 1 << 20, size=n)
    chunks["offset"] = np.concatenate([[0], np.cumsum(chunks["size"])[:-1]]) if n else []
    fd = bytes(rng.integers(0, 256, size=32, dtype=np.uint8))
    fs = int(chunks["size"].sum()) if n else 5
    summ = check(Y, O, chunks, fd, fs)
    assert summ["valid"] == (1 if n else 0)
    if n >= 2:
        bad = chunks.copy()
        bad["offset"][n // 2] += 1                       # validateManifest :452-461
        s2 = check(Y, O, bad, fd, fs)
        assert s2["valid"] == 0 and s2["offsets_sequential"] == 0
        s3 = check(Y, O, chunks, fd, fs + 1)             # total size mismatch :463-468
        assert s3["valid"] == 0 and s3["offsets_sequential"] == 1
