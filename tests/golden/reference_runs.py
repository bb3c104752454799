"""Stored outputs of the unmodified reference programs (oracle/_ref, built by oracle/Makefile from the reference sources) for
the cases of the tests that compare with them, so that those tests run on a machine without the reference.

* Bit-exact comparisons keep one blake2b digest per block of 32 rows of every output raster (reference_runs.json): equal
  digests are equal rasters, and a mismatch is located to its block of rows.
* Comparisons with a tolerance keep the full NaN pattern of every output and its values on a fixed, seeded sample of
  pixels (reference_samples.npz).

A test asks for a case by key and passes the callable that runs the reference on that case.  The callable only runs when
S2PB_RECORD_REFERENCE=1, which (re)records the case; tests/golden/make_golden_reference_runs.py records every case.
"""
import hashlib
import json
import os
import zlib

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
DIGESTS = os.path.join(HERE, "reference_runs.json")
SAMPLES = os.path.join(HERE, "reference_samples.npz")
BLOCK = 32


def recording():
    return os.environ.get("S2PB_RECORD_REFERENCE") == "1"


def digests(a):
    """-> one hex digest per block of BLOCK rows (NaN payloads and the sign of zero normalised, as util.same ignores them)"""
    a = np.ascontiguousarray(a)
    if a.dtype.kind == "f":
        a = np.where(np.isnan(a), np.nan, a + 0.0).astype(a.dtype)
    return [hashlib.blake2b(a[r:r + BLOCK].tobytes(), digest_size=8).hexdigest() for r in range(0, a.shape[0], BLOCK)]


def _load_json():
    if not os.path.exists(DIGESTS):
        return {}
    with open(DIGESTS) as f:
        return json.load(f)


def reference_digests(key, run):
    """-> {output name: digests} of the reference run `key`; run() -> {output name: array}, or None when the reference
    program refuses the case (then None is returned)."""
    table = _load_json()
    if recording():
        out = run()
        table[key] = None if out is None else {k: digests(v) for k, v in out.items()}
        with open(DIGESTS, "w") as f:
            json.dump(table, f, indent=0, sort_keys=True)
            f.write("\n")
    assert key in table, "no stored reference output for %s (record it: tests/golden/make_golden_reference_runs.py)" % key
    return table[key]


def mismatches(got, want):
    """got: {name: array}; want: {name: digests}.  -> descriptions of the outputs that differ (empty when all are equal)"""
    bad = []
    for name, d in want.items():
        g = digests(got[name])
        blocks = [k for k, (a, b) in enumerate(zip(g, d)) if a != b]
        if len(g) != len(d) or blocks:
            bad.append("%s differs in %d of %d blocks of %d rows (first: rows %d..)" % (
                name, len(blocks), len(d), BLOCK, (blocks[0] if blocks else 0) * BLOCK))
    return bad


class Sample:
    """An output raster kept as its NaN pattern (full) and its values at `idx` (flat pixel indices, seeded sample)."""

    def __init__(self, shape, isnan, idx, val):
        self.shape, self.isnan, self.idx, self.val = shape, isnan, idx, val

    def at(self, a):
        """the values of `a` (same shape as the stored raster) at the sampled pixels"""
        a = np.asarray(a)
        assert a.shape == self.shape, (a.shape, self.shape)
        return a.reshape(self.shape[0] * self.shape[1], -1)[self.idx].reshape(self.val.shape)


def reference_samples(key, run, n=2048):
    """-> {output name: Sample} of the reference run `key`; run() -> {output name: array of shape (h, w, ...)}."""
    store = dict(np.load(SAMPLES)) if os.path.exists(SAMPLES) else {}
    if recording():
        for k in [k for k in store if k.startswith(key + "/")]:
            del store[k]
        for name, a in run().items():
            a = np.asarray(a)
            npx = a.shape[0] * a.shape[1]
            rng = np.random.default_rng(zlib.crc32(key.encode()))        # the same pixels for every output of the case
            idx = np.sort(rng.choice(npx, size=min(n, npx), replace=False)).astype(np.int32)
            p = "%s/%s/" % (key, name)
            store[p + "shape"] = np.array(a.shape, np.int64)
            store[p + "nan"] = np.packbits(np.isnan(a).ravel())
            store[p + "idx"] = idx
            store[p + "val"] = a.reshape(npx, -1)[idx].reshape((len(idx),) + a.shape[2:])
        np.savez_compressed(SAMPLES, **store)
    out = {}
    for k in store:
        if k.startswith(key + "/") and k.endswith("/shape"):
            name = k[len(key) + 1:-len("/shape")]
            p = "%s/%s/" % (key, name)
            shape = tuple(int(x) for x in store[p + "shape"])
            isnan = np.unpackbits(store[p + "nan"], count=int(np.prod(shape))).astype(bool).reshape(shape)
            out[name] = Sample(shape, isnan, store[p + "idx"], store[p + "val"])
    assert out, "no stored reference output for %s (record it: tests/golden/make_golden_reference_runs.py)" % key
    return out
