"""Acceptance (SURVEY 8f N3): the reference's OWN test programs and examples -- sources unmodified, compiled by
`make -C oracle acceptance` against this repo's headers and libpffft_b200.so -- must pass on the GPU.
They exercise the classic host-pointer API one transform per call (tests/test_pffft.c, test_pffft.cpp through
pffft.hpp, test_fft_factors.c, test_pffastconv.c, examples/*.c of marton78/pffft)."""
import os
import subprocess

import pytest

from conftest import ROOT

ACC = os.path.join(ROOT, "oracle", "_ref", "acceptance")
pytestmark = pytest.mark.gpu

CASES = [
    ("test_pffft_float", [], 600),
    ("test_pffft_double", [], 600),
    ("test_pffft_float", ["--test-simd"], 120),
    ("test_pffft_cpp", [], 900),
    ("test_fft_factors", [], 300),
    ("test_pffastconv", ["--no-bench", "--quick"], 1500),
    ("test_pffastconv", ["--no-bench", "--quick", "--sym"], 1500),
    # the FULL sweep of tests/test_pffastconv.c:915-936: filter lengths 124 .. 256, real / complex 2x / complex single FFT,
    # block sizes 64 .. 64 K, output lengths with and without flush
    ("test_pffastconv", ["--no-bench"], 1500),
    ("example_c_real_flt_fwd", [], 60),
    ("example_c_cplx_dbl_fwd", [], 60),
]


@pytest.mark.parametrize("exe,args,timeout", CASES)
def test_reference_program_passes_against_drop_in_library(exe, args, timeout):
    path = os.path.join(ACC, exe)
    if not os.path.exists(path):
        pytest.skip("oracle/_ref/acceptance/%s not built: `make -C oracle acceptance REF=<pffft source tree>` builds the "
                    "reference's own test programs, which are not part of this repository" % exe)
    r = subprocess.run([path] + args, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=timeout)
    assert r.returncode == 0, "%s %s failed (rc=%d):\n%s" % (exe, " ".join(args), r.returncode, r.stdout[-3000:])
