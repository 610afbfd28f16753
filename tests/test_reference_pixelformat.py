"""The one reference translation unit that compiles without libjxl (N/Encoder/PixelFormatConversion.cpp:16-121) — the bit-exact oracle for
the encoder's BGRA repack (SURVEY.md §8c). Its outputs on the seeded surfaces are stored in tests/golden/bgra_repacks.json (provenance in
bgra_repack_cases.py), and the numpy restatement must reproduce them everywhere. Where the reference itself is built into oracle/_ref
(oracle/Makefile, from the reference's sources at REF; they are not part of this repository), it is compared live as well, and with the
stored outputs."""
import os

import numpy as np
import pytest

import bgra_repack_cases as R
import oracle_py


@pytest.fixture(scope="module")
def ref():
    if not os.path.exists(R.REF_LIB_PATH):
        oracle_py.build()
    if not os.path.exists(R.REF_LIB_PATH):
        pytest.skip("oracle/_ref not built: reference sources absent (REF in oracle/Makefile)")
    return R.REF_LIB_PATH


@pytest.mark.parametrize("w,h,pad", R.PIXELFORMAT_CASES)
def test_bgra_repacks_match_numpy_restatement(ref, w, h, pad):
    buf = R.pixelformat_surface(w, h, pad)
    golden = R.load_golden()
    for fn in R.REPACKS:
        out = R.reference(buf, w, fn)
        assert np.array_equal(out, R.restated(buf, w, fn)), fn
        assert R.matches_golden(golden[R.pixelformat_key(w, h, pad, fn)], out), fn


@pytest.mark.parametrize("w,h,pad", R.PIXELFORMAT_CASES)
def test_numpy_restatement_reproduces_the_stored_repack_outputs(w, h, pad):
    buf = R.pixelformat_surface(w, h, pad)
    golden = R.load_golden()
    for fn in R.REPACKS:
        assert R.matches_golden(golden[R.pixelformat_key(w, h, pad, fn)], R.restated(buf, w, fn)), fn
