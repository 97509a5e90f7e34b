"""Outputs of the reference's own code, frozen under tests/golden/ so that the tests pinned to them run without the reference
tree (tools/make_reference_golden.py writes them from oracle/_ref). An array is stored as the SHA-256 of its bytes plus a
fixed, seeded sample of its rows: the sample names the first rows that differ, the hash checks every byte."""
import hashlib
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
SAMPLE_ROWS = 256


def _rows(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint8).reshape(len(a), -1)


def pin(a):
    """What is stored of array `a` (one row per element of its first axis)."""
    r = _rows(a)
    n = len(r)
    idx = np.arange(n) if n <= SAMPLE_ROWS else np.sort(np.random.default_rng(n).choice(n, SAMPLE_ROWS, replace=False))
    return {"n": np.array(n), "index": idx, "rows": r[idx], "sha256": np.array(hashlib.sha256(r.tobytes()).hexdigest())}


def save(name, outputs):
    """outputs: key -> plain array (stored whole) or pin(array)."""
    flat = {}
    for key, v in outputs.items():
        if isinstance(v, dict):
            flat.update({key + "." + k: a for k, a in v.items()})
        else:
            flat[key] = np.asarray(v)
    np.savez_compressed(os.path.join(GOLDEN, name), **flat)


class Golden:
    def __init__(self, name):
        with np.load(os.path.join(GOLDEN, name), allow_pickle=False) as z:
            self.z = dict(z)

    def __getitem__(self, key):
        return self.z[key]

    def check(self, key, got):
        """Asserts that `got` is byte for byte the pinned array `key`."""
        r = _rows(got)
        n = int(self.z[key + ".n"])
        assert len(r) == n, "%s: %d rows, the reference has %d" % (key, len(r), n)
        idx = self.z[key + ".index"]
        bad = idx[(r[idx] != self.z[key + ".rows"]).any(axis=1)]
        assert bad.size == 0, "%s: %d of %d sampled rows differ from the reference, first ones %s" % (
            key, bad.size, idx.size, bad[:8].tolist())
        assert hashlib.sha256(r.tobytes()).hexdigest() == str(self.z[key + ".sha256"]), \
            "%s differs from the reference outside the sampled rows" % key
