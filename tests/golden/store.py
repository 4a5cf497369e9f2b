"""Stored outputs of the original InfiniTensor kernels, for the tests that compare with them.

The suite does not need the original project: its outputs were recorded once and are kept here as compressed .npz
files.  A test names each output and passes the function that computes it with the original
(`gold(key, lambda: ...)`).  With ITB_RECORD_GOLDEN=1 that function runs (the original built into oracle/_ref by
`make -C oracle ref ref_cuda REF=<InfiniTensor checkout>`) and its result is stored; otherwise the stored result is
read back.  Outputs larger than SAMPLE elements are kept as a fixed sample of SAMPLE flat positions, and the tests
compare the same positions of their own result (`pick`); smaller ones are kept whole."""
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
RECORD = os.environ.get("ITB_RECORD_GOLDEN") == "1"
SAMPLE = 1024
_STEP = 7919  # prime: the SAMPLE positions are distinct and spread over every axis


def pick(a):
    """The compared positions of `a`: all of it up to SAMPLE elements, else a fixed spread-out sample, flattened."""
    a = np.ascontiguousarray(a)
    if a.size <= SAMPLE:
        return a
    assert a.size % _STEP, a.size
    return a.ravel()[np.arange(SAMPLE, dtype=np.int64) * _STEP % a.size]


def _widen(a):
    return a.astype(np.float32) if a.dtype == np.float16 else a


class Golden:
    """The outputs stored in tests/golden/<name>.npz (half-precision outputs are stored as float16, read as float32)."""

    def __init__(self, name):
        self.path = os.path.join(HERE, name + ".npz")
        self.data = {}
        if os.path.exists(self.path):
            with np.load(self.path) as z:
                self.data = {k: z[k] for k in z.files}
        self.recorded = {}

    def __call__(self, key, fn):
        """pick() of the original's output `key` (a tuple of them when `fn` returns a tuple)."""
        if RECORD:
            out = fn()
            if isinstance(out, tuple):
                for i, o in enumerate(out):
                    self.recorded[f"{key}.{i}"] = pick(o)
            else:
                self.recorded[key] = pick(out)
            np.savez_compressed(self.path, **{**self.data, **self.recorded})
        stored = {**self.data, **self.recorded}
        if key in stored:
            return _widen(stored[key])
        n = sum(k.startswith(key + ".") for k in stored)
        assert n, f"{key}: no stored output in {self.path}"
        return tuple(_widen(stored[f"{key}.{i}"]) for i in range(n))
