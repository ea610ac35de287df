"""Outputs of the reference implementation that tests compare against, stored in tests/golden/reference_outputs.npz.

The values were produced by running the reference's own sources, compiled by oracle/Makefile into oracle/_ref, on the
same seeded inputs the tests build.  To regenerate them, build oracle/_ref and run the tests that use this module with
YAMS_B200_RECORD_REFERENCE=<output .npz>: each value is then computed by the reference library and written there (merged
with the values already stored), and the tests compare against the freshly computed value.  Everywhere else the stored
value is used, so these comparisons need nothing outside the repository."""
import hashlib
import os

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_outputs.npz")
RECORD = os.environ.get("YAMS_B200_RECORD_REFERENCE")
_store = None


def _load() -> dict:
    global _store
    if _store is None:
        _store = {}
        for p in (PATH, RECORD):
            if p and os.path.exists(p):
                with np.load(p) as z:
                    _store.update({k: z[k] for k in z.files})
    return _store


def expect(key: str, compute) -> np.ndarray:
    """The reference's output stored under `key`; in record mode `compute()` (which calls the reference library) is run
    and its result stored first."""
    store = _load()
    if RECORD:
        from oracle import oracle as O
        assert O.ref_available(), "recording reference outputs needs oracle/_ref (make -C oracle ref)"
        store[key] = np.asarray(compute())
        np.savez_compressed(RECORD, **store)
    assert key in store, f"no stored reference output {key!r} in {PATH}"
    return store[key]


def digest(a) -> np.ndarray:
    """SHA-256 of an array's bytes: stands for an output too large to store; equal digests mean bit-equal arrays."""
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest(), dtype=np.uint8)


def key_of(*parts) -> str:
    """A short stable key for a value whose inputs are arrays (hex of the SHA-256 of their bytes)."""
    h = hashlib.sha256()
    for p in parts:
        h.update(np.ascontiguousarray(p).tobytes() if isinstance(p, np.ndarray) else repr(p).encode())
    return h.hexdigest()[:24]
