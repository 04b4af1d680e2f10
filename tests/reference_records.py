"""Stored results of the reference build for the tests that compare with it (tests/golden/reference/<module>.npz).

The reference build (oracle/_ref: Flan's own sources compiled by oracle/Makefile) exists only where those sources are
at hand. Where it is absent, the tests compare with what it returned, as stored here; where it is present, they compare
with the live build and also check every stored record against it.

An array is stored as its shape, its dtype, the SHA-256 of its bytes (the whole comparison, bit for bit) and a seeded
sample of its elements that shows where a mismatch lies; small arrays, and those a test reads back, whole.

    FLAN_RECORD_REFERENCE=1 python -m pytest tests/test_oracle.py tests/test_oracle_io.py tests/test_oracle_modify.py \
        tests/test_gpu_io.py

rewrites the records: from the live reference build where it exists, otherwise from the checker's results (allowed
only where the checker passed these tests bit for bit against the build); each file names its source. The files
here were recorded without the build: from the checker (pv_oracle.c), unchanged since it last passed these tests
against the build, and, for the .flan files, from the device codec, which then wrote and read the same bytes.
"""
import hashlib
import os

import numpy as np

DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference")
SAMPLE = 64
WHOLE = 64
RECORD = os.environ.get("FLAN_RECORD_REFERENCE") == "1"


def _index(size, whole):
    if whole or size <= WHOLE:
        return np.arange(size)
    return np.sort(np.random.default_rng(0).choice(size, SAMPLE, replace=False))


def _record(a, whole):
    a = np.ascontiguousarray(a)
    return {"shape": np.array(a.shape, np.int64), "dtype": np.array(a.dtype.str),
            "sample": a.reshape(-1)[_index(a.size, whole)],
            "sha256": np.frombuffer(hashlib.sha256(a.tobytes()).digest(), np.uint8)}


class Records:
    def __init__(self, name):
        self.path = os.path.join(DIR, name + ".npz")
        self.stored = {} if RECORD else dict(np.load(self.path))
        self.sources = set()

    def check(self, key, mine, theirs=None, whole=False):
        """`mine` equals, bit for bit, what the reference build returned for `key`: `theirs` when the live build gave it,
        else the stored record. whole: store every element, for stored_array()."""
        mine = np.ascontiguousarray(mine)
        if theirs is not None:
            theirs = np.ascontiguousarray(theirs)
            assert mine.shape == theirs.shape and mine.dtype == theirs.dtype, (key, mine.shape, theirs.shape)
            assert mine.tobytes() == theirs.tobytes(), key
        if RECORD:
            self.sources.add(_STAND_IN or "reference build" if theirs is not None else "checker (oracle/pv_oracle.c)")
            for k, v in _record(theirs if theirs is not None else mine, whole).items():
                self.stored[key + "." + k] = v
            return
        self._compare(key, theirs if theirs is not None else mine)

    def _compare(self, key, a):
        g = self.stored
        assert key + ".sha256" in g, "no stored reference result for %s in %s" % (key, self.path)
        assert a.shape == tuple(g[key + ".shape"]) and a.dtype.str == str(g[key + ".dtype"]), (key, a.shape, a.dtype)
        want = g[key + ".sample"]
        idx = np.arange(a.size) if want.size == a.size else _index(a.size, False)
        got = a.reshape(-1)[idx]
        row = lambda v: np.frombuffer(v.tobytes(), np.uint8).reshape(len(idx), -1)  # noqa: E731
        bad = np.flatnonzero((row(got) != row(want)).any(axis=1)) if len(idx) else []
        assert len(bad) == 0, "%s: element %d is %r, the reference gave %r" % (key, idx[bad[0]], got[bad[0]], want[bad[0]])
        assert hashlib.sha256(a.tobytes()).digest() == g[key + ".sha256"].tobytes(), "%s differs from the reference" % key

    def stored_array(self, key):
        """The whole array stored for `key` (recorded with whole=True)."""
        g = self.stored
        a = g[key + ".sample"].reshape(tuple(g[key + ".shape"]))
        self._compare(key, a)
        return a

    def save(self):
        if RECORD and self.stored:
            os.makedirs(DIR, exist_ok=True)
            np.savez_compressed(self.path, source=np.array(" + ".join(sorted(self.sources))), **self.stored)


def live_reference():
    """The reference build (FFT backend 0, the parity stand-in) where oracle/_ref exists, else None."""
    from oracle_lib import RefLib
    return RefLib(0) if RefLib.available() else None


def live_reference_modify():
    from oracle_lib import RefModifyLib
    return RefModifyLib() if RefModifyLib.available() else None


_STAND_IN = None


class _DeviceFileCodec:
    def __init__(self):
        from flan_b200.engine import Engine
        self.eng = Engine(0)

    def save_flan(self, path, pv, sr, ar, W):
        import torch
        self.eng.save_flan(path, torch.from_numpy(np.ascontiguousarray(pv)).to(self.eng.device), sr, float(ar), W)

    def load_flan(self, path):
        pv, sr, rate, W = self.eng.load_flan(path)
        return pv.cpu().numpy(), sr, rate, W


def file_codec_reference():
    """The reference's PVBuffer::save / load: the live build where it exists. When recording without it, this project's
    device codec stands in for it: it wrote and read the same bytes as the build whenever the two ran side by side
    (tests/test_gpu_io.py). Else None: the tests read the stored records."""
    global _STAND_IN
    ref = live_reference()
    if ref is not None or not RECORD:
        return ref
    _STAND_IN = "device file codec (flan_b200_save_flan / flan_b200_load_flan)"
    return _DeviceFileCodec()
