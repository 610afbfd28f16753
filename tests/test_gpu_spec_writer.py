"""GPU tests: files hand-assembled by the independent bit-level writer (tests/jxl_spec_writer.py) decoded through the C ABI
LoadImage. Lossless Modular files must come back bit-exact; the DC-only VarDCT frame within half an LSB of the float64 value
computed from the published XYB constants. The same files are checked against the oracle on CPU (test_spec_writer_cpu.py)."""
import numpy as np
import pytest

import jxl_spec_writer as W
import spec_cases
from test_spec_writer_cpu import expected_pixels

pytestmark = pytest.mark.gpu

CASES = spec_cases.cases()


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_load_image_decodes_spec_writer_files(gpu, case):
    name, data, px, info = case
    image = gpu.DecoderImage()
    gpu.JpegXLNative.LoadImage(data, image)
    got = image.layer_data.interleaved
    want, tol = expected_pixels(px)
    assert got.shape == want.shape, (got.shape, want.shape)
    err = np.abs(got.astype(np.float64) - want.astype(np.float64)).max()
    assert err <= tol + (0.5 if tol else 0), "%s: max error %g" % (name, err)
    assert image.format == info["format"] and image.has_transparency == info.get("has_transparency", False)
    if "name" in info:
        assert image.layer_data.name == info["name"].decode() + "\0"   # length passed includes the NUL (Appendix C-3)


def test_container_variants_through_load_image(gpu):
    for name, data, px, exif, xmps in spec_cases.containerised():
        image = gpu.DecoderImage()
        gpu.JpegXLNative.LoadImage(data, image)
        assert np.array_equal(image.layer_data.interleaved, px), name
        assert image.exif == exif and image.xmp == xmps[0], name
        assert image.callback_log.count("setXmp") == len(xmps) and image.callback_log.count("setExif") == 1


def test_dc_only_vardct_frame_matches_published_constants(gpu):
    data, want = spec_cases.vardct_dc_case()
    image = gpu.DecoderImage()
    gpu.JpegXLNative.LoadImage(data, image)
    err = np.abs(image.layer_data.interleaved.astype(np.float64) - want).max()
    assert err <= 0.5 + 1e-2, "DC-only VarDCT frame: max |decoded - expected| = %g" % err


def _refused(gpu, data, message):
    with pytest.raises(gpu.FormatException, match=message) as e:
        gpu.JpegXLNative.LoadImage(data, gpu.DecoderImage())
    assert e.value.status == "DecodeError"


def test_rct_over_channels_of_different_sizes_is_refused(gpu):
    # R, G, B and an extra channel at half resolution (dim_shift 1); the RCT on channels 1..3 takes B and the extra channel together.
    # The header is refused before any sample is read, so the extra channel's plane is written at full size.
    a = spec_cases._img(16, 24, 4, seed=41)
    data = W.modular_image(spec_cases._planes(a), extra=[dict(type=W.EC_DEPTH, bits=8, dim_shift=1)], rct=(1, 6))
    _refused(gpu, data, "RCT channel sizes")


def test_delta_palette_with_the_weighted_predictor_is_refused(gpu):
    colors = [(10, 20, 30), (200, 100, 50), (90, 90, 90)]
    a = np.array(colors)[np.random.default_rng(42).integers(0, 3, size=(16, 24))]
    data = W.modular_image(spec_cases._planes(a), palette=dict(begin=0, num_c=3, colors=colors, deltas=[(1, 2, 3)], predictor=6))
    _refused(gpu, data, "delta palettes with the weighted predictor are not supported")
