"""Stored traces of the compiled reference, so that the bit-for-bit pins of the plain-C oracle against the reference run
everywhere, not only where the reference sources are at hand.

A pinned test hands `check` a function run(kind) that drives one library ("port" or "reference") through the test's
scenario and yields (label, value) pairs. The port's values are compared with the reference's in order, bit for bit,
with the semantics of np.array_equal(equal_nan=True) on arrays of the same dtype and shape. The reference's side is
kept in tests/golden/reference_traces.npz, one record per value: a 128-bit BLAKE2b digest (the full outputs run to
hundreds of MB), the number of elements, and the values at SAMPLES evenly spaced flat positions, so that a failure
says where and by how much the port left the reference. Where oracle/_ref/libmaxiref.so exists the reference also
runs live, and the stored records must still be its.

With MXB_RECORD_REFERENCE_TRACES=1 and the compiled reference present, the records of the tests that ran are
(re)written into the file instead of being checked against it; records of pinned tests that no longer exist are dropped:

    MXB_RECORD_REFERENCE_TRACES=1 python -m pytest tests -m "not gpu" -k "reference or fuzz or oracle_patch"
"""
import hashlib
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
PATH = os.path.join(HERE, "golden", "reference_traces.npz")
RECORD = os.environ.get("MXB_RECORD_REFERENCE_TRACES", "") == "1"
SAMPLES = 8
RECORD_DTYPE = np.dtype([("digest", np.uint8, 16), ("size", np.int64), ("samples", np.float64, SAMPLES)])
COLLECTED = set()       # keys of every pinned test collected in this session (tests/conftest.py)


def key(item):
    """'<test file name without .py>::<test name with parameters>': the same under every pytest import mode."""
    return f"{os.path.splitext(os.path.basename(str(item.path)))[0]}::{item.name}"


def _canonical(x):
    a = np.array(x)
    if a.dtype.kind in "fc":
        a[np.isnan(a)] = np.nan
        a[a == 0] = 0
    return a


def _positions(size):
    return np.unique(np.linspace(0, size - 1, SAMPLES).round().astype(np.int64)) if size else np.zeros(0, np.int64)


def record(x):
    """dtype, shape and values of x as one RECORD_DTYPE record; every NaN alike and -0.0 like 0.0 (np.array_equal(equal_nan=True))."""
    a = _canonical(x)
    h = hashlib.blake2b(digest_size=16)
    h.update(f"{a.dtype.str}{a.shape}".encode())
    h.update(np.ascontiguousarray(a).tobytes())
    r = np.zeros((), RECORD_DTYPE)
    r["digest"] = np.frombuffer(h.digest(), dtype=np.uint8)
    r["size"] = a.size
    r["samples"][:] = np.nan
    pos = _positions(a.size)
    r["samples"][:pos.size] = a.reshape(-1)[pos].astype(np.float64)
    return r


def explain(x, ref):
    """Where the port's value x leaves the reference's record `ref`, as far as the stored samples tell."""
    a = _canonical(x)
    if a.size != ref["size"]:
        return f"{a.size} elements (shape {a.shape}), the reference has {int(ref['size'])}"
    pos = _positions(a.size)
    got = a.reshape(-1)[pos].astype(np.float64)
    for p, g, r in zip(pos, got, ref["samples"][:pos.size]):
        if not (g == r or (np.isnan(g) and np.isnan(r))):
            return f"flat index {p} of shape {a.shape}: port {float(g)!r}, reference {float(r)!r}"
    return f"the {pos.size} sampled elements agree; the difference is elsewhere or in dtype / shape (port: {a.dtype} {a.shape})"


class Store:
    def __init__(self):
        self.traces = dict(np.load(PATH)) if os.path.exists(PATH) else {}
        self.recorded = {}

    def save(self):
        if not self.recorded:
            return
        collected_files = {k.split("::")[0] for k in COLLECTED}

        def alive(k):
            f = k.split("::")[0]
            return os.path.exists(os.path.join(HERE, f + ".py")) and (f not in collected_files or k in COLLECTED)
        traces = {k: v for k, v in self.traces.items() if alive(k)}
        traces.update(self.recorded)
        np.savez_compressed(PATH, **dict(sorted(traces.items())))


class Trace:
    def __init__(self, key, store, live):
        self.key, self.store, self.live = key, store, live

    def check(self, run):
        got = [(label, x, record(x)) for label, x in run("port")]
        if self.live is not None:
            ref = np.array([record(y) for _, y in run("reference")], dtype=RECORD_DTYPE)
            assert len(ref) == len(got), (self.key, len(ref), len(got))
            for (label, x, g), r in zip(got, ref):
                assert np.array_equal(g["digest"], r["digest"]), \
                    f"{self.key}: {label}: the port differs from the compiled reference: {explain(x, r)}"
            if RECORD:
                self.store.recorded[self.key] = ref
                return
        stored = self.store.traces.get(self.key)
        assert stored is not None, f"{self.key}: no stored reference trace in {os.path.basename(PATH)}"
        assert len(stored) == len(got), (self.key, len(stored), len(got))
        for (label, x, g), r in zip(got, stored):
            assert np.array_equal(g["digest"], r["digest"]), \
                f"{self.key}: {label}: differs from the stored trace of the compiled reference: {explain(x, r)}"
