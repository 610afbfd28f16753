"""-m gpu parity tests for paths that exist in the engine but had no test (VERDICT r01 item 1c): CMYK + K merge, premultiplied
alpha, two-pass files, jxlp / brob boxes, BitmapData.stride > 4*w on SaveImage against the reference's BGRA repack (stored outputs, tests/bgra_repack_cases.py)."""
import ctypes as C
import io
import struct

import numpy as np
import pytest

import bgra_repack_cases as R

pytestmark = pytest.mark.gpu


def _decode_gpu(P, data):
    image = P.DecoderImage()
    P.JpegXLNative.LoadImage(data, image)
    return image


@pytest.mark.parametrize("alpha", [False, True])
def test_cmyk_black_channel_merge(gpu, oracle, alpha):
    """N/Decoder/JxlDecoder.cpp:159-215: the K extra channel is merged after the colour channels and C, M, Y, K are inverted."""
    img = oracle.synthetic_image(300, 260, seed=5, channels=4)
    src = np.concatenate([img, img[..., :1][:, ::-1]], axis=2) if alpha else img      # colour(3) + black [+ alpha]
    data = oracle.encode(src, num_color=3, has_alpha=alpha, lossless=1, black_channel=1)
    ref = oracle.decode(data)
    assert ref.format == 2 and ref.pixels.shape[2] == (5 if alpha else 4)
    want = np.concatenate([255 - src[..., :4]] + ([src[..., 4:5]] if alpha else []), axis=2)
    assert np.array_equal(ref.pixels, want)                                           # the oracle itself follows the reference lines
    image = _decode_gpu(gpu, data)
    assert image.format == "Cmyk" and image.has_transparency == alpha
    assert np.array_equal(image.layer_data.interleaved, want)


@pytest.mark.parametrize("kw,dtype", [(dict(lossless=1), np.uint8), (dict(effort=5), np.uint8), (dict(effort=5, bits=32, exp_bits=8), np.float32)])
def test_premultiplied_alpha_is_unpremultiplied(gpu, oracle, kw, dtype):
    """JxlDecoderSetUnpremultiplyAlpha(TRUE), N/Decoder/JxlDecoder.cpp:233: alpha_associated files come back with straight alpha."""
    img = oracle.synthetic_image(200, 136, seed=8, channels=4)
    img[..., 3] = np.maximum(img[..., 3], 40)
    img[..., :3] = (img[..., :3].astype(np.float32) * img[..., 3:4] / 255.0).astype(np.uint8)   # colour <= alpha: a premultiplied source
    src = img if dtype == np.uint8 else img.astype(np.float32) / 255.0
    data = oracle.encode(src, premultiplied=1, **kw)
    ref = oracle.decode(data).pixels
    got = _decode_gpu(gpu, data).layer_data.interleaved
    assert got.shape == ref.shape and got.dtype == ref.dtype
    if dtype == np.uint8:
        assert int(np.abs(got.astype(np.int32) - ref.astype(np.int32)).max()) <= 1
    else:
        assert float(np.abs(got - ref).max()) <= 1e-4 * max(1.0, float(np.abs(ref).max()))
    assert np.array_equal(got[..., 3], ref[..., 3])
    # straight alpha really was restored: where alpha is small the colour is scaled up past the stored value
    if kw.get("lossless"):
        a = img[..., 3:4].astype(np.float32) / 255.0
        want = np.clip(np.rint(img[..., :3] / 255.0 / a * 255.0), 0, 255)
        assert int(np.abs(got[..., :3].astype(np.int32) - want.astype(np.int32)).max()) <= 1


@pytest.mark.parametrize("w,h,shift,kw", [(520, 392, 1, dict(effort=7)), (300, 200, 2, dict(effort=3)), (600, 300, 1, dict(effort=5, use_prefix=1))])
def test_two_pass_vardct_files(gpu, oracle, w, h, shift, kw):
    """Progressive files: pass 0 carries the coefficients >> shift, pass 1 the remainder; each pass has its own contexts and code."""
    img = oracle.synthetic_image(w, h, seed=w + shift)
    data = oracle.encode(img, num_passes=2, pass_shift=shift, **kw)
    ref = oracle.decode(data, threads=4).pixels
    assert np.array_equal(ref, oracle.decode(oracle.encode(img, **kw), threads=4).pixels)    # same pixels as the single-pass file
    got = _decode_gpu(gpu, data).layer_data.color
    assert int(np.abs(got.astype(np.int32) - ref.astype(np.int32)).max()) <= 1 and oracle.psnr(got, ref) >= 60.0


def test_two_pass_file_with_alpha_in_the_last_pass(gpu, oracle):
    img = oracle.synthetic_image(300, 260, seed=4, channels=4)
    data = oracle.encode(img, effort=5, num_passes=2)
    ref = oracle.decode(data).pixels
    layer = _decode_gpu(gpu, data).layer_data
    assert int(np.abs(layer.color.astype(np.int32) - ref[..., :3].astype(np.int32)).max()) <= 1
    assert np.array_equal(layer.transparency, img[..., 3])


def _box(t, payload):
    return struct.pack(">I", 8 + len(payload)) + t + payload


def _brotli(data):
    lib = C.CDLL("libbrotlienc.so.1")
    cap = C.c_size_t(len(data) + 1024)
    out = C.create_string_buffer(cap.value)
    lib.BrotliEncoderCompress.argtypes = [C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_char_p, C.POINTER(C.c_size_t), C.c_char_p]
    assert lib.BrotliEncoderCompress(5, 22, 0, len(data), data, C.byref(cap), out) == 1
    return out.raw[:cap.value]


def test_brob_boxes_and_jxlp_parts(gpu, oracle):
    """N/Decoder/JxlDecoder.cpp:433-440,687-784: brob boxes are decompressed (JxlDecoderSetDecompressBoxes), the first Exif box and
    every xml box are reported in file order; a codestream split over jxlp boxes decodes like the contiguous one."""
    img = oracle.synthetic_image(120, 90, seed=2)
    cs = oracle.encode(img, effort=3, container=0)
    exif = b"\x00\x00\x00\x00MM\x00*\x00\x00\x00\x08\x00\x00" + bytes(range(200))
    xmp = b"<x:xmpmeta xmlns:x='adobe:ns:meta/'>" + b"a" * 500 + b"</x:xmpmeta>"
    head = b"\x00\x00\x00\x0cJXL \x0d\x0a\x87\x0a" + _box(b"ftyp", b"jxl \x00\x00\x00\x00jxl ")
    cut1, cut2 = len(cs) // 4, len(cs) // 2
    try:
        packed_exif, packed_xmp = _brotli(exif), _brotli(xmp)
    except OSError:
        pytest.skip("libbrotlienc.so.1 not available to build the brob boxes")
    data = (head + _box(b"jxlp", struct.pack(">I", 0) + cs[:cut1]) + _box(b"brob", b"Exif" + packed_exif) + _box(b"jxlp", struct.pack(">I", 1) + cs[cut1:cut2]) +
            _box(b"brob", b"xml " + packed_xmp) + _box(b"Exif", b"\x00\x00\x00\x00second") + _box(b"xml ", b"<second/>") + _box(b"jxlp", struct.pack(">I", 0x80000002) + cs[cut2:]))
    ref = oracle.decode(data)
    assert ref.exif == exif and ref.xmp == [xmp, b"<second/>"]
    image = _decode_gpu(gpu, data)
    assert image.exif == exif and image.xmp == xmp
    assert image.callback_log == ["setBasicInfo", "setKnownColorProfile", "setExif", "setXmp", "setXmp", "setLayerData"]
    assert int(np.abs(image.layer_data.color.astype(np.int32) - ref.pixels.astype(np.int32)).max()) <= 1
    plain = _decode_gpu(gpu, head + _box(b"jxlc", cs))
    assert np.array_equal(plain.layer_data.color, image.layer_data.color)


@pytest.mark.parametrize("w,h,pad,kind", R.STRIDE_CASES)
def test_save_image_with_padded_stride_matches_the_reference_repack(gpu, oracle, w, h, pad, kind):
    """BitmapData.stride may exceed 4*w (N/Common.h:17-23). Lossless SaveImage must store exactly the samples that the reference's own
    PixelFormatConversion.cpp hands to libjxl for the same padded surface: its output stored in tests/golden/bgra_repacks.json, and the
    compiled reference itself where oracle/_ref is built."""
    buf = R.stride_surface(w, h, pad, kind)
    fn = R.KIND_TO_REPACK[kind]
    want = R.restated(buf, w, fn)
    assert R.matches_golden(R.load_golden()[R.stride_key(w, h, pad, kind)], want), kind
    live = R.reference(buf, w, fn)
    assert live is None or np.array_equal(live, want), kind
    data = gpu.encode_to_memory(None, gpu.EncoderOptions(lossless=True), host_array=buf, width=w, height=h, stride=4 * w + pad)
    d = oracle.decode(data)
    assert d.pixels.shape == want.shape and np.array_equal(d.pixels, want), kind
    assert np.array_equal(_decode_gpu(gpu, data).layer_data.interleaved, want)


@pytest.mark.parametrize("colors,alpha", [(1, False), (1, True), (3, False), (3, True)])
@pytest.mark.parametrize("kw,dtype", [(dict(lossless=1), np.uint8), (dict(lossless=1, bits=16), np.uint16), (dict(effort=3, bits=16, exp_bits=5), np.float16), (dict(lossless=1, bits=16, exp_bits=5), np.float16),
                                      (dict(lossless=1, bits=32, exp_bits=8), np.float32), (dict(effort=5, bits=32, exp_bits=8), np.float32)])
def test_layer_bitmaps_on_the_gpu_match_the_managed_repack(gpu, oracle, colors, alpha, kw, dtype):
    """JxlB200LoadImageLayers == LoadImage + DecoderLayerData's Set{Gray,GrayAlpha,Rgb,Rgba}{UInt8,UInt16,Float16,Float32}ImageData
    (I/DecoderLayerData.cs:245-992): gray replicated into RGB, alpha through TransparencyMapping.ToEightBit — bit for bit."""
    img = oracle.synthetic_image(150, 90, seed=3 + colors, channels=4)
    src = np.concatenate([img[..., :colors]] + ([img[..., 3:4]] if alpha else []), axis=2)
    src = src if dtype == np.uint8 else src.astype(np.float32) / 255.0
    data = oracle.encode(src, num_color=colors, has_alpha=alpha, **kw)
    image = _decode_gpu(gpu, data)
    layer = image.layer_data
    color, transparency = gpu.load_image_layers(data)
    assert color.dtype == dtype and color.shape == (90, 150, 3)
    assert np.array_equal(color.view(np.uint8), layer.color.view(np.uint8))
    if alpha:
        assert transparency.dtype == np.uint8 and np.array_equal(transparency, layer.transparency)
        assert len(np.unique(transparency)) > 50
    else:
        assert transparency is None


@pytest.mark.parametrize("alpha", [False, True])
def test_cmyk_layer_bitmaps_on_the_gpu(gpu, oracle, alpha):
    """SetCmykUInt8ImageData / SetCmykAlphaUInt8ImageData (I/DecoderLayerData.cs:164-243) after the native K merge."""
    img = oracle.synthetic_image(120, 80, seed=15, channels=4)
    src = np.concatenate([img, img[..., :1][:, ::-1]], axis=2) if alpha else img
    data = oracle.encode(src, num_color=3, has_alpha=alpha, lossless=1, black_channel=1)
    layer = _decode_gpu(gpu, data).layer_data
    color, transparency = gpu.load_image_layers(data)
    assert color.shape == (80, 120, 4) and np.array_equal(color, layer.color)
    assert (transparency is None) == (not alpha) and (not alpha or np.array_equal(transparency, layer.transparency))
