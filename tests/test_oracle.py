"""Pins the checkers (CPU only): the plain-C restatement oracle/liboracle.so against the UNMODIFIED reference
compiled into oracle/_ref and against the committed golden vectors; and the reference against independent
second opinions (numpy float64 FFT), SURVEY 8(c)."""
import os

import numpy as np
import pytest

from conftest import ROOT, uniform

SIZES = [16, 32, 64, 96, 128, 160, 192, 256, 288, 384, 480, 512, 576, 640, 800, 864, 1024, 2048, 2592, 4000, 4096]


@pytest.fixture(scope="module")
def orc(R):
    if not R.have_oracle():
        pytest.skip("oracle/liboracle.so not built (make -C oracle)")
    return R.oracle()


def test_oracle_size_algebra_matches_reference(orc, ref):
    for tr in (0, 1):
        for N in range(0, 2000):
            assert orc.lib.pffft_is_valid_size(N, tr) == ref.lib.pffft_is_valid_size(N, tr)
            so = orc.new_setup(N, tr); sr = ref.new_setup(N, tr)
            assert bool(so) == bool(sr), (N, tr)              # is_valid_size <=> new_setup != NULL (test_fft_factors.c:36-61)
            assert bool(sr) == bool(ref.lib.pffft_is_valid_size(N, tr)) or N == 0
            if so: orc.destroy_setup(so)
            if sr: ref.destroy_setup(sr)
        for N in (1, 17, 100, 1000, 5000):
            for hi in (0, 1):
                assert orc.lib.pffft_nearest_transform_size(N, tr, hi) == ref.lib.pffft_nearest_transform_size(N, tr, hi)


@pytest.mark.parametrize("dtype,tol", [(np.float32, 2e-6), (np.float64, 1e-13)])
def test_oracle_transforms_match_reference(orc, ref, R, dtype, tol):
    rng = np.random.default_rng(0)
    for N in SIZES:
        for tr in (0, 1):
            if not ref.lib.pffft_is_valid_size(N, tr):
                continue
            per = N if tr == 0 else 2 * N
            x = uniform(rng, per, dtype)
            pow2 = (N & (N - 1)) == 0
            # the reference's double path has float-precision radix-3/5 constants (pffft_priv_impl.h:154,259-262)
            t = tol if (pow2 or dtype == np.float32) else 2e-7
            for ordered in (True, False):
                fr = ref.transform(N, tr, x, 0, ordered, dtype)
                fo = orc.transform(N, tr, x, 0, ordered, dtype)
                assert R.relmax(fo, fr) <= t, (N, tr, ordered, "fwd")
                br = ref.transform(N, tr, fr, 1, ordered, dtype)
                bo = orc.transform(N, tr, fr, 1, ordered, dtype)
                assert R.relmax(bo, br) <= t, (N, tr, ordered, "bwd")


def test_oracle_zreorder_bit_exact(orc, ref):
    for N in SIZES + [12000]:
        for tr in (0, 1):
            if not ref.lib.pffft_is_valid_size(N, tr):
                continue
            per = N if tr == 0 else 2 * N
            ramp = np.arange(per, dtype=np.float32)
            for d in (0, 1):
                assert np.array_equal(orc.zreorder(N, tr, ramp, d), ref.zreorder(N, tr, ramp, d)), (N, tr, d)


def test_oracle_zconvolve_bit_exact(orc, ref):
    rng = np.random.default_rng(1)
    for N, dt in ((256, np.float32), (96, np.float32), (1024, np.float64)):
        for tr in (0, 1):
            per = N if tr == 0 else 2 * N
            a, b, c = [uniform(rng, per, dt) for _ in range(3)]
            for acc in (True, False):
                assert np.array_equal(orc.zconvolve(N, tr, a, b, c, 0.37, acc, dt), ref.zconvolve(N, tr, a, b, c, 0.37, acc, dt))


def test_oracle_fastconv_matches_reference(orc, ref):
    x = (np.arange(9000) % 4093).astype(np.float32)
    for taps in (31, 124, 131, 144):
        h = np.array([(-1.0, 1.0, 0.5)[j % 3] for j in range(taps)], np.float32)
        for flags in (0, 1, 17, 64):
            for bl in (0, 512, 2048):
                for flush in (0, 1):
                    yr, nr, blr = ref.fastconv(h, x, bl, flags, flush)
                    yo, no, blo = orc.fastconv(h, x, bl, flags, flush)
                    assert (no, blo) == (nr, blr), (taps, flags, bl, flush)
                    if nr:
                        assert np.max(np.abs(yo - yr)) <= (yr.max() - yr.min()) / 1e5
    assert orc.fastconv(np.ones(8, np.float32), x, 0, 2, 1)[0] is None      # CPLX_FILTER -> NULL


def test_checkers_against_golden_and_numpy(orc, ref, R):
    g = np.load(os.path.join(ROOT, "tests", "golden", "pffft_golden.npz"))
    for key in sorted(k[:-2] for k in g.files if k.endswith("_x") and k.startswith("N")):
        N = int(key[1:].split("_")[0]); tr = 0 if "_r_" in key else 1
        dtype = np.dtype(np.float32 if key.endswith("f4") else np.float64)
        x = g[key + "_x"]
        fo, fz = ref.transform(N, tr, x, 0, True, dtype), ref.transform(N, tr, x, 0, False, dtype)
        if R.have_ref():
            # the golden file IS the reference's output: the reference built into oracle/_ref reproduces it bit-exactly
            assert np.array_equal(fo, g[key + "_fwd_ordered"]), key
            assert np.array_equal(fz, g[key + "_fwd_z"]), key
        tol = (2e-6 if dtype == np.float32 else (1e-13 if (N & (N - 1)) == 0 else 2e-7))
        assert R.relmax(orc.transform(N, tr, x, 0, True, dtype), g[key + "_fwd_ordered"]) <= tol, key
        # second opinion: numpy float64 (SURVEY App. D: 1.3e-7 .. 2.8e-7 for float)
        xd = x.astype(np.float64)
        if tr == 1:
            W = np.fft.fft(xd[0::2] + 1j * xd[1::2]); want = np.stack([W.real, W.imag], -1).ravel()
        else:
            W = np.fft.rfft(xd); want = np.stack([W.real[:-1], W.imag[:-1]], -1).ravel(); want[1] = W.real[-1]
        assert R.relmax(g[key + "_fwd_ordered"], want) <= (1e-6 if dtype == np.float32 else 1e-7), key
