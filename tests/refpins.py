"""What the reference's own code returned on the tests' seeded inputs, stored in tests/golden/reference_pins.json so that the
tests pinned to the reference run where the reference is not available.

pin(key, ours, reference) asserts that `ours` equals the stored output of the reference for `key`. Arrays and byte strings
are stored as the first 128 bits of the SHA-256 digest of their bytes (the comparisons are bit for bit), everything else
(counts, return codes, result records) as the value itself.

To re-record, build oracle/_ref/ from the reference (oracle/build_ref.sh) and run the pinned tests with
DYNSLAM_RECORD_PINS=1: every pin then calls `reference()`, asserts that `ours` equals what it returned, and stores that
value; the file is rewritten when the test process exits."""
import atexit
import hashlib
import json
import os

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_pins.json")
RECORD = os.environ.get("DYNSLAM_RECORD_PINS") == "1"

_store = None


def _load():
    global _store
    if _store is None:
        _store = {}
        if os.path.exists(PATH):
            with open(PATH) as f:
                _store = json.load(f)
        if RECORD:
            atexit.register(_save)
    return _store


def _save():
    with open(PATH, "w") as f:
        json.dump(dict(sorted(_store.items())), f, indent=0, sort_keys=True)
        f.write("\n")


def _norm(v):
    if isinstance(v, np.ndarray):
        v = np.ascontiguousarray(v).tobytes()
    if isinstance(v, (bytes, bytearray)):
        return f"sha256:{hashlib.sha256(bytes(v)).hexdigest()[:32]}:{len(v)}"
    if isinstance(v, (list, tuple)):
        return [_norm(x) for x in v]
    if isinstance(v, dict):
        return {str(k): _norm(x) for k, x in v.items()}
    if isinstance(v, np.generic):
        return v.item()
    return v


def pin(key, ours, reference):
    """Asserts that `ours` equals what `reference()` (a call into the reference's code) returns for `key`."""
    store = _load()
    got = _norm(ours)
    if RECORD:
        want = _norm(reference())
        assert got == want, key
        store[key] = want
        return
    assert key in store, f"{key}: no stored reference output in {os.path.relpath(PATH)}"
    assert got == store[key], key
