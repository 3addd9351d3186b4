"""Recorded outputs of the unmodified reference, so that the tests that compare with it run where
oracle/_ref/libpffft_ref.so was not built.

Every result a test receives from the reference (through the `ref` fixture of tests/conftest.py) is
recorded per test and call: integers exactly; arrays by their size, their largest magnitude and K values at
seeded positions, for at most CAP evenly spaced arrays of a test.  Where the reference library is absent, the
plain-C restatement (oracle/liboracle.so) answers the same calls instead, and each of its results is first
checked against the reference's recorded one; a test then compares the CUDA path with that checked result,
under its own tolerance.

    PFFFT_B200_RECORD_REFERENCE=DIR python -m pytest tests ...   # with oracle/_ref built: writes DIR/*.npz
    python -m oracle.golden merge tests/golden/reference_samples.npz DIR/*.npz
"""
import os
import sys
import zlib

import numpy as np

from . import ref as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PATH = os.path.join(ROOT, "tests", "golden", "reference_samples.npz")
K = 4
CAP = 128                # keeps the file small: one test chains ~2000 small transforms through the reference
NONE = -(1 << 62)
# restatement vs reference, relative to the largest magnitude of the reference's output: the reference's double
# path keeps float-precision radix-3/5 constants (pffft_priv_impl.h:154, :259-262), hence 1e-6 for doubles.
# Values are stored as float32: exact for float outputs, within 6e-8 of double ones.
TOL = {np.dtype(np.float32): 1e-5, np.dtype(np.float64): 1e-6}


def _flatten(v, ints, arrays):
    """a result as the integers and arrays it is made of, in order; an array also puts its size among the integers"""
    if isinstance(v, tuple):
        for e in v:
            _flatten(e, ints, arrays)
    elif isinstance(v, np.ndarray):
        ints.append(int(v.size))
        arrays.append(v)
    elif v is None:
        ints.append(NONE)
    else:
        ints.append(int(v))


def positions(key, index, size):
    return np.random.default_rng([zlib.crc32(key.encode()), index]).integers(0, size, K)


def sample(key, index, a):
    """(largest magnitude, K values at seeded positions) of array `a`, the `index`-th array of test `key`"""
    a = np.asarray(a).ravel()
    if not a.size:
        return 0.0, np.zeros(K)
    return float(np.max(np.abs(a))), a[positions(key, index, a.size)].astype(np.float64)


def mismatch(key, index, a, peak, samp):
    """None when array `a` agrees with the recorded (peak, samples) of the reference, else why not"""
    got_peak, got = sample(key, index, a)
    err = max(abs(got_peak - peak), float(np.max(np.abs(got - samp))))
    tol = TOL.get(np.asarray(a).dtype, 0.0) * peak
    if not err <= tol:
        return "array %d differs from the reference's by %.3g (allowed %.3g)" % (index, err, tol)
    return None


class Recording:
    """the reference's results, by test: `record` adds to them, `check` walks them in call order"""

    def __init__(self):
        self.tests = {}          # key -> [ints, [(peak, samples)] of every stride-th array, stride]
        self.cursor = {}

    @classmethod
    def load(cls, path=PATH):
        g = np.load(path)
        rec = cls()
        keys = str(g["tests"]).split("\n")
        for k, stride in zip(keys, g["stride"]):
            rec.tests[k] = [[], [], int(stride)]
        for t, v in zip(g["int_test"], g["int_val"]):
            rec.tests[keys[t]][0].append(int(v))
        for t, m, s in zip(g["arr_test"], g["arr_peak"], g["arr_samples"]):
            rec.tests[keys[t]][1].append((float(m), s.astype(np.float64)))
        return rec

    def save(self, path):
        keys = sorted(self.tests)
        it, iv, at, am, asamp, strides = [], [], [], [], [], []
        for t, k in enumerate(keys):
            ints, arrays, stride = self.tests[k]
            step = -(-len(arrays) // CAP) or 1
            arrays = arrays[::step]
            strides.append(stride * step)
            it += [t] * len(ints); iv += ints
            at += [t] * len(arrays); am += [m for m, _ in arrays]; asamp += [s for _, s in arrays]
        np.savez_compressed(path, tests=np.array("\n".join(keys)), stride=np.array(strides, np.int32),
                            int_test=np.array(it, np.int32), int_val=np.array(iv, np.int64),
                            arr_test=np.array(at, np.int32), arr_peak=np.array(am, np.float32),
                            arr_samples=np.array(asamp, np.float32).reshape(-1, K))

    def record(self, key, result):
        ints, arrays = [], []
        _flatten(result, ints, arrays)
        t = self.tests.setdefault(key, [[], [], 1])
        for a in arrays:
            t[1].append(sample(key, len(t[1]), a))
        t[0].extend(ints)

    def check(self, key, result):
        """raises AssertionError unless `result` is what the reference returned at this point of test `key`"""
        if key not in self.tests:
            raise AssertionError("no recorded reference results for %s: record them with oracle/golden.py" % key)
        ni, na = self.cursor.get(key, (0, 0))
        ints, arrays = [], []
        _flatten(result, ints, arrays)
        want_i, want_a, stride = self.tests[key]
        assert ints == want_i[ni:ni + len(ints)], \
            "%s: the restatement returned %s where the reference returned %s" % (key, ints, want_i[ni:ni + len(ints)])
        for j, a in enumerate(arrays):
            if (na + j) % stride == 0:
                peak, samp = want_a[(na + j) // stride]
                why = mismatch(key, na + j, a, peak, samp)
                assert why is None, "%s: %s" % (key, why)
        self.cursor[key] = (ni + len(ints), na + len(arrays))


class _Lib:
    """attribute access to a library's C functions whose integer results pass through `observe`"""

    def __init__(self, lib, observe):
        self._lib, self._observe = lib, observe

    def __getattr__(self, name):
        f = getattr(self._lib, name)

        def call(*args):
            r = f(*args)
            self._observe(r)
            return r
        return call


class Observed:
    """a PffftLib (oracle/ref.py) whose results pass through `observe`; setups count by whether they exist"""

    def __init__(self, impl, observe):
        self._impl, self._observe = impl, observe
        self.lib = _Lib(impl.lib, observe)
        self.has_double = impl.has_double

    def new_setup(self, *args, **kw):
        s = self._impl.new_setup(*args, **kw)
        self._observe(int(bool(s)))
        return s

    def destroy_setup(self, *args, **kw):
        return self._impl.destroy_setup(*args, **kw)

    def __getattr__(self, name):              # transform, transform_batch, zreorder, zconvolve, fastconv
        f = getattr(self._impl, name)

        def call(*args, **kw):
            r = f(*args, **kw)
            self._observe(r)
            return r
        return call


class _Precise:
    """the restatement with its float transforms evaluated by its double path and rounded to float, so that a test's
    tolerance meets an answer at least as accurate as the reference's own float path (the restatement's float path
    is up to 2x further from the exact transform).  zreorder, zconvolve and fastconv stay in float: tests compare
    those bit for bit."""

    def __init__(self, impl):
        self._impl = impl
        self.lib, self.has_double = impl.lib, impl.has_double

    def transform(self, N, transform, x, direction, ordered=True, dtype=np.float32):
        return self._via_double("transform", N, transform, x, direction, ordered, dtype)

    def transform_batch(self, N, transform, x, direction, ordered=True, dtype=np.float32):
        return self._via_double("transform_batch", N, transform, x, direction, ordered, dtype)

    def _via_double(self, name, N, transform, x, direction, ordered, dtype):
        f = getattr(self._impl, name)
        if np.dtype(dtype) != np.float32:
            return f(N, transform, x, direction, ordered, dtype)
        return f(N, transform, np.asarray(x, np.float64), direction, ordered, np.float64).astype(np.float32)

    def __getattr__(self, name):
        return getattr(self._impl, name)


_recording = None


def checked_restatement(key):
    """the restatement, every result checked against the reference's recorded one for test `key`"""
    global _recording
    if _recording is None:
        _recording = Recording.load()
    _recording.cursor.pop(key, None)
    return Observed(_Precise(R.oracle()), lambda r: _recording.check(key, r))


def recording_reference(key, recording):
    """the live reference, every result added to `recording` under test `key`"""
    return Observed(R.ref(), lambda r: recording.record(key, r))


def merge(out, paths):
    rec = Recording()
    for p in paths:
        part = Recording.load(p)
        for k, v in part.tests.items():
            assert k not in rec.tests, "recorded twice: " + k
            rec.tests[k] = v
    rec.save(out)
    print("%s: %d tests, %d integers, %d arrays" % (out, len(rec.tests), sum(len(v[0]) for v in rec.tests.values()),
                                                   sum(len(v[1]) for v in rec.tests.values())))


if __name__ == "__main__":
    if len(sys.argv) >= 3 and sys.argv[1] == "merge":
        merge(sys.argv[2], sys.argv[3:])
    else:
        sys.exit("usage: python -m oracle.golden merge OUT.npz RECORDED.npz ...")
