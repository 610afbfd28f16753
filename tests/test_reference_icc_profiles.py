"""CPU tests with the two ICC profiles the reference ships (S/ColorProfiles/*.icc, used by I/DecoderImage.cs:166-184) as real-world vectors:
the oracle's ICC-stream codec must round-trip them byte for byte, and the product's host-side reader of matrix/TRC profiles (what a lossy
SaveImage with metadata->iccProfile uses, N/Encoder/JxlEncoder.cpp:258-262) must recover the published primaries and tone curves.
The profiles are stored in tests/golden/: written by LittleCMS 2 with the recipe the reference's files were made with (Rec.709 with the
BT.709 curve, Rec.2020 linear), not by this project's own ICC writers; tests/golden/make_icc_profiles.py says how."""
import os

import numpy as np
import pytest

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
NAMES = ["Rec2020-V4-g10.icc", "Rec709-V4-rec709.icc"]


def _profile(name):
    return open(os.path.join(GOLDEN, name), "rb").read()


@pytest.mark.parametrize("name", NAMES)
def test_icc_stream_codec_round_trips_the_reference_profiles(oracle, name):
    # the stored stand-ins for the reference's two profiles: LittleCMS output made with their recipe, not the shipped files (module docstring)
    icc = _profile(name)
    assert icc[36:40] == b"acsp" and int.from_bytes(icc[0:4], "big") == len(icc)
    stream = oracle.icc_stream_write(icc)
    assert len(stream) < len(icc)                      # the predicted-ICC coding must actually compress a real profile
    assert oracle.icc_stream_read(stream) == icc


def test_matrix_trc_reader_on_the_reference_profiles(pkg):
    # on the stored stand-ins for the reference's two profiles (LittleCMS output made with their recipe, not the shipped files)
    # Rec.709 primaries and curve: same primaries as sRGB -> identity matrix to linear sRGB; the curve is the BT.709 inverse OETF
    m, lut = pkg.debug_parse_icc(_profile("Rec709-V4-rec709.icc"))
    assert np.allclose(np.asarray(m).reshape(3, 3), np.eye(3), atol=2e-3)
    v = np.arange(256) / 255.0
    bt709 = np.where(v < 0.081, v / 4.5, ((v + 0.099) / 1.099) ** (1 / 0.45))
    assert np.allclose(np.asarray(lut).reshape(3, 256), bt709[None, :], atol=2e-3)
    # Rec.2020 primaries, linear curve: the published BT.2020 -> BT.709 matrix
    m, lut = pkg.debug_parse_icc(_profile("Rec2020-V4-g10.icc"))
    want = np.array([[1.6605, -0.5876, -0.0728], [-0.1246, 1.1329, -0.0083], [-0.0182, -0.1006, 1.1187]])
    assert np.allclose(np.asarray(m).reshape(3, 3), want, atol=3e-3)
    assert np.allclose(np.asarray(lut).reshape(3, 256), v[None, :], atol=1e-4)
