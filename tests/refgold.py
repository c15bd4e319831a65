"""What the reference kernels returned, for the parity tests on machines without a reference build.

The GPU parity tests run this library and the reference's own kernels (oracle/_ref, built by the oracle recipe from a
reference checkout) on identical inputs.  Every reference result a test compares with goes through reference(): with
oracle/_ref present the reference runs as before; without it the result is read back from
tests/golden/reference_outputs.json.  There each array is kept as its shape, dtype and a digest of its bytes (SHA-256
cut to 96 bits) plus a digest of its NaN pattern, so bit-exact comparisons keep their full strength; tolerance
comparisons ask for a fixed, seeded sample of rows to be kept as values as well.  Scalars are kept as they are.

Regenerate after a deliberate change of what the reference computes, on a GPU with oracle/_ref built:
    VOLDOR_GOLDEN_RECORD=/tmp/reference_outputs.json python -m pytest tests
and copy the file to tests/golden/.

The per-pixel random streams of the depth step continue from window to window and are re-seeded when the image size
changes (reference optimize_depth.cu:357-361).  reseed_depth_rng() starts every test from freshly seeded streams, so
what a test computes does not depend on which tests ran before it in the same process."""
import base64
import hashlib
import json
import os

import numpy as np

import ffi

LIVE = os.path.exists(ffi.REF)
PATH = os.path.join(ffi.ROOT, "tests", "golden", "reference_outputs.json")
RECORD = os.environ.get("VOLDOR_GOLDEN_RECORD")
SKIP_KEYS = ("stats_ms",)  # timings
_golden = None
_recorded = {}
_calls = {}


def _sha(b):
    return hashlib.sha256(b).hexdigest()[:24]  # 96 bits


class Digest:
    """a reference array known by its digest (and, where asked for, a seeded sample of its rows)"""

    def __init__(self, d):
        self.shape = tuple(d["shape"])
        self.dtype = np.dtype(d["dtype"])
        self.size = int(np.prod(self.shape))
        self.sha256 = d["sha256"]
        self.nan_sha256 = d.get("nan_sha256")
        self.row_dims = d.get("row_dims")
        self.sample_rows = None if d.get("sample_rows") is None else np.asarray(d["sample_rows"], np.int64)
        self.sample = None
        if d.get("sample") is not None:
            rows = np.frombuffer(base64.b64decode(d["sample"]), self.dtype)
            self.sample = rows.reshape((len(self.sample_rows),) + self.shape[self.row_dims:])

    def __len__(self):
        return self.shape[0]

    def matches(self, a):
        a = np.ascontiguousarray(a)
        return a.shape == self.shape and a.dtype == self.dtype and _sha(a.tobytes()) == self.sha256

    def nan_matches(self, a):
        a = np.asarray(a)
        return a.shape == self.shape and _sha(np.packbits(np.isnan(a)).tobytes()) == self.nan_sha256


def _rows(a, row_dims):
    return a.reshape((int(np.prod(a.shape[:row_dims])),) + a.shape[row_dims:])


def _encode(v, sample):
    if isinstance(v, np.ndarray):
        a = np.ascontiguousarray(v)
        d = {"shape": list(a.shape), "dtype": a.dtype.str, "sha256": _sha(a.tobytes())}
        if a.dtype.kind == "f":
            d["nan_sha256"] = _sha(np.packbits(np.isnan(a)).tobytes())
        if sample and a.dtype.kind == "f":
            n_rows, row_dims = sample
            rows = _rows(a, row_dims)
            idx = np.sort(np.random.default_rng(0).choice(rows.shape[0], min(n_rows, rows.shape[0]), replace=False))
            d.update(row_dims=row_dims, sample_rows=idx.tolist(),
                     sample=base64.b64encode(np.ascontiguousarray(rows[idx]).tobytes()).decode())
        return {"__array__": d}
    if isinstance(v, dict):
        return {k: _encode(x, sample) for k, x in v.items() if k not in SKIP_KEYS}
    if isinstance(v, (list, tuple)):
        return [_encode(x, sample) for x in v]
    if isinstance(v, str):
        return v
    if isinstance(v, (bool, np.bool_)):
        return bool(v)
    if isinstance(v, (int, np.integer)):
        return int(v)
    if isinstance(v, (float, np.floating)):
        return float(v)
    if v is None:
        return None
    raise TypeError(f"cannot keep a {type(v)} as golden data")


def _decode(v):
    if isinstance(v, dict):
        if "__array__" in v:
            return Digest(v["__array__"])
        return {k: _decode(x) for k, x in v.items()}
    if isinstance(v, list):
        return tuple(_decode(x) for x in v)
    return v


def _key():
    """<test file>::<test name and parameters>#<n-th reference result of that test>"""
    path, _, test = os.environ.get("PYTEST_CURRENT_TEST", "").rsplit(" (", 1)[0].partition("::")
    test = f"{os.path.basename(path)}::{test}"  # independent of the directory pytest was started from
    n = _calls.get(test, 0)
    _calls[test] = n + 1
    return f"{test}#{n}"


def reference(compute, sample=None, live=None, key=None):
    """compute() with the reference build present, else what it returned when the golden file was recorded.
    sample=(n_rows, row_dims) keeps n_rows seeded rows of each float array (rows = the first row_dims axes).
    live: whether the part of the reference build that compute() needs is there (default: the reference kernels).
    key: the name of the result outside a test (default: the calling test and the number of results it took before)."""
    key = key or _key()
    if LIVE if live is None else live:
        value = compute()
        if RECORD:
            _recorded[key] = _encode(value, sample)
            with open(RECORD, "w") as f:
                json.dump(_recorded, f, sort_keys=True)
        return value
    global _golden
    if _golden is None:
        with open(PATH) as f:
            _golden = json.load(f)
    assert key in _golden, f"{key}: no reference result recorded in {PATH}"
    return _decode(_golden[key])


def sampled(a, b):
    """(a, b) restricted to the rows b keeps as values when b is a Digest; unchanged when b is the live array"""
    if not isinstance(b, Digest):
        return np.asarray(a), np.asarray(b)
    assert b.sample is not None, "golden entry was recorded without a sample"
    return _rows(np.asarray(a), b.row_dims)[b.sample_rows], b.sample


def isfinite(b):
    """np.isfinite of a live array, or of the kept sample of a Digest"""
    return np.isfinite(b.sample if isinstance(b, Digest) else b)


def reseed_depth_rng():
    """one depth step at a size no test uses, on this library and (when present) on the reference: the next window at
    any test size starts from freshly seeded per-pixel streams on both"""
    import synth

    win = synth.make_window(24, 8, 1, seed=0)
    kw = dict(flows=list(win["flows"]), rig=[np.ones((8, 24), np.float32)], depth=win["depth_gt"], K=win["K"],
              Rs=list(win["Rs"]), ts=list(win["ts"]))
    libs = [ffi.ours()] + ([ffi.reference()] if LIVE else [])
    for lib in libs:
        assert lib.optimize_depth(24, 8, 1, **kw)[0] == 0
