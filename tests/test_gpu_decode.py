"""-m gpu parity tests: CUDA decode through the C ABI vs the CPU oracle on the same files.
Bars (BASELINE.json north_star): bit-exact for lossless / integer stages, <= 1 LSB max-abs for 8-bit lossy."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _decode_gpu(P, data):
    image = P.DecoderImage()
    P.JpegXLNative.LoadImage(data, image)
    return image


@pytest.mark.parametrize("w,h,kw", [
    (64, 48, dict(effort=3)),                       # single group, single TOC entry
    (300, 200, dict(effort=3)),                     # 2 groups
    (520, 392, dict(effort=7)),                     # gab + EPF + varblocks + CfL + adaptive quant
    (519, 387, dict(effort=7, distance=3.0)),       # ragged size, EPF 2 iterations
    (300, 200, dict(effort=7, distance=8.0)),       # EPF 3 iterations
    (2100, 300, dict(effort=5, use_prefix=1)),      # 2 LF groups, prefix codes
])
def test_vardct_rgb8_matches_oracle(gpu, oracle, w, h, kw):
    img = oracle.synthetic_image(w, h, seed=w + h)
    data = oracle.encode(img, **kw)
    ref = oracle.decode(data, threads=4).pixels
    got = _decode_gpu(gpu, data).layer_data.color
    assert got.shape == ref.shape
    err = np.abs(got.astype(np.int32) - ref.astype(np.int32))
    assert int(err.max()) <= 1, "max abs error %d LSB" % int(err.max())
    assert oracle.psnr(got, ref) >= 60.0


@pytest.mark.parametrize("strategy", [0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 18, 19, 20, 21, 22, 23, 24, 25, 26])
def test_every_supported_ac_strategy(gpu, oracle, strategy):
    img = oracle.synthetic_image(531, 277, seed=strategy)
    data = oracle.encode(img, effort=3, force_strategy=strategy)
    ref = oracle.decode(data, threads=4).pixels
    got = _decode_gpu(gpu, data).layer_data.color
    assert int(np.abs(got.astype(np.int32) - ref.astype(np.int32)).max()) <= 1


@pytest.mark.parametrize("w,h,channels,shift", [(200, 150, 3, 1), (300, 260, 4, 1), (100, 90, 1, 1), (700, 300, 3, 0), (1100, 600, 4, 2)])
def test_lossless_modular_bit_exact(gpu, oracle, w, h, channels, shift):
    img = oracle.synthetic_image(w, h, seed=11 * channels + w, channels=channels)
    data = oracle.encode(img, lossless=1, modular_group_shift=shift)
    image = _decode_gpu(gpu, data)
    layer = image.layer_data
    ref = oracle.decode(data).pixels
    assert np.array_equal(ref, img)
    if channels == 1:
        assert np.array_equal(layer.color[..., 0], img[..., 0])
    else:
        assert np.array_equal(layer.color, img[..., :3])
    if channels == 4:
        assert np.array_equal(layer.transparency, img[..., 3])


def test_lossy_with_alpha(gpu, oracle):
    img = oracle.synthetic_image(300, 260, seed=3, channels=4)
    data = oracle.encode(img, effort=7)
    ref = oracle.decode(data).pixels
    image = _decode_gpu(gpu, data)
    assert image.has_transparency and image.format == "Rgb"
    assert int(np.abs(image.layer_data.color.astype(np.int32) - ref[..., :3].astype(np.int32)).max()) <= 1
    assert np.array_equal(image.layer_data.transparency, img[..., 3])     # alpha is coded losslessly


def test_bgra_surface_matches_managed_repack(gpu, oracle):
    """JxlB200LoadImageBgra == LoadImage + DecoderLayerData + JpegXLLoad repack (I/DecoderLayerData.cs, S/JpegXLLoad.cs:219-249)."""
    for ch in (3, 4):
        img = oracle.synthetic_image(333, 222, seed=ch, channels=ch)
        data = oracle.encode(img, effort=5)
        doc = gpu.JpegXLLoad.Load(data)
        fused = gpu.load_image_bgra(data)
        assert np.array_equal(doc.surface, fused)


def test_callback_order_and_metadata(gpu, oracle):
    img = oracle.synthetic_image(64, 64, seed=1)
    exif = b"\x00\x00\x00\x00II*\x00\x08\x00\x00\x00\x00\x00"
    data = oracle.encode(img, effort=3, exif=exif, xmp=b"<x:xmpmeta/>")
    image = _decode_gpu(gpu, data)
    assert image.callback_log == ["setBasicInfo", "setKnownColorProfile", "setExif", "setXmp", "setLayerData"]
    assert image.known_color_profile == "Srgb" and image.exif == exif and image.xmp == b"<x:xmpmeta/>"
    assert (image.width, image.height, image.format, image.channel_representation) == (64, 64, "Rgb", 0)


def test_truncated_and_invalid_inputs(gpu, oracle):
    img = oracle.synthetic_image(300, 200, seed=2)
    data = oracle.encode(img, effort=3)
    with pytest.raises(gpu.FormatException) as e:
        _decode_gpu(gpu, data[: len(data) // 2])
    assert e.value.status == "DecodeError"
    with pytest.raises(gpu.FormatException) as e:
        _decode_gpu(gpu, b"not a jxl file at all")
    assert e.value.status == "InvalidFileSignature"
    corrupt = bytearray(data)
    corrupt[len(corrupt) * 3 // 4] ^= 0x5A
    try:
        _decode_gpu(gpu, bytes(corrupt))   # either decodes to something or reports DecodeError; it must not crash
    except gpu.FormatException as ex:
        assert ex.status == "DecodeError"


def test_golden_files(gpu, oracle):
    import json
    import os
    gdir = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    index = json.load(open(os.path.join(gdir, "index.json")))
    for name, meta in index.items():
        data = open(os.path.join(gdir, name + ".jxl"), "rb").read()
        want = np.load(os.path.join(gdir, name + ".npy"))
        image = _decode_gpu(gpu, data)
        layer = image.layer_data
        ncol = 1 if image.format == "Gray" else 3
        got = layer.color[..., :ncol]
        if meta["lossless"]:
            assert np.array_equal(got, want[..., :ncol]), name
        else:
            assert int(np.abs(got.astype(np.int32) - want[..., :ncol].astype(np.int32)).max()) <= 1, name
        if image.has_transparency:
            assert np.array_equal(layer.transparency, want[..., ncol]), name


@pytest.mark.parametrize("kw,dtype,tol", [
    (dict(bits=16), np.uint16, 1.0 / 255),                                   # u16 output
    (dict(bits=16, exp_bits=5), np.float16, 1e-3),                            # f16 output: one half-precision ulp (2^-10) — a rounding flip
    (dict(bits=32, exp_bits=8), np.float32, 1e-4),                            # f32 output: <= 1e-4 relative (north_star); measured 1.1e-5
    (dict(bits=32, exp_bits=8, primaries=9, tf=16, intensity_target=1000.0), np.float32, 5e-4),   # f32 PQ: measured 3.3e-4 with the PQ curve in double on
    # both sides, so the curve is not the cause: a 1e-7 absolute rounding difference of an fp32 XYB sample (IDCT summation order) is 7e-9 on the
    # cube at black, i.e. 7e-4 relative on a linear value of 1e-5, before the +11 / -9.9 opsin inverse. Two fp32-plane decoders agree to 1e-4 on dark
    # PQ samples only if they round identically at every step (DESIGN.md §6).
    (dict(bits=16, primaries=9, tf=16, intensity_target=1000.0), np.uint16, 1.0 / 255),   # Rec.2020 PQ HDR, gab + EPF
    (dict(bits=16, primaries=11), np.uint16, 1.0 / 255),                      # Display P3
    (dict(bits=16, primaries=9, tf=18, intensity_target=1000.0), np.uint16, 1.0 / 255),   # Rec.2100 HLG: samples come back HLG-encoded (no OOTF)
    (dict(bits=16, exp_bits=5, primaries=9, tf=18, intensity_target=1000.0), np.float16, 1e-3),   # HLG, half-float samples
    (dict(bits=32, exp_bits=8, tf=8), np.float32, 1e-4),                      # linear sRGB float
])
def test_hdr_and_high_bit_depth_outputs(gpu, oracle, kw, dtype, tol):
    img = oracle.synthetic_image(200, 136, seed=21).astype(np.float32) / 255.0
    data = oracle.encode(img, effort=7, **kw)
    ref = oracle.decode(data).pixels
    image = _decode_gpu(gpu, data)
    got = image.layer_data.color
    assert got.dtype == dtype and got.shape == ref.shape
    if dtype == np.uint16:
        assert int(np.abs(got.astype(np.int64) - ref.astype(np.int64)).max()) <= 257      # <= 1 LSB at 8-bit precision
    else:
        a, b = got.astype(np.float64), ref.astype(np.float64)
        worst = float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-3)))           # relative, with a floor of 1e-3 for samples near zero
        assert worst <= tol, "worst relative difference %.3g" % worst


@pytest.mark.parametrize("orientation", [2, 3, 4, 5, 6, 7, 8])
def test_orientation(gpu, oracle, orientation):
    img = oracle.synthetic_image(72, 40, seed=orientation)
    data = oracle.encode(img, lossless=1, orientation=orientation)
    ref = oracle.decode(data).pixels
    image = _decode_gpu(gpu, data)
    assert (image.width, image.height) == (ref.shape[1], ref.shape[0])
    assert np.array_equal(image.layer_data.color, ref)


def test_batch_matches_single_decodes(gpu, oracle):
    files = [oracle.encode(oracle.synthetic_image(300 + 8 * i, 200, seed=i), effort=7 if i % 2 else 3) for i in range(6)]
    outs = [np.zeros((200, 300 + 8 * i, 3), np.uint8) for i in range(6)]
    st = gpu.decode_batch(files, outs, max_in_flight=4)
    assert st == [0] * 6
    for f, o in zip(files, outs):
        assert np.array_equal(o, _decode_gpu(gpu, f).layer_data.color)


def test_batch_pipeline_mixed_content(gpu, oracle):
    """The three-phase batch pipeline with 8 sections per warp (count >= 8), on files that exercise its lazy paths: 64x64+ transforms
    (second plane set allocated only when the LF kernel reports them), multi-group frames, alpha, and a lossless Modular frame."""
    imgs, files = [], []
    for i, strat in enumerate([0, 21, 24, 26, 5, 18, 0, 22, 4, 25]):
        img = oracle.synthetic_image(600 + 16 * i, 520, seed=40 + i)
        files.append(oracle.encode(img, effort=3, force_strategy=strat))
    rgba = oracle.synthetic_image(520, 300, seed=77, channels=4)
    files.append(oracle.encode(rgba, effort=7))
    files.append(oracle.encode(oracle.synthetic_image(300, 280, seed=78), lossless=True))
    singles = []
    for f in files:   # the batch writes the interleaved buffer LoadImage hands to setLayerData: colour channels, then alpha
        ld = _decode_gpu(gpu, f).layer_data
        singles.append(ld.color if ld.transparency is None else np.concatenate([ld.color, ld.transparency[..., None]], axis=2))
    outs = [np.zeros_like(s) for s in singles]
    st = gpu.decode_batch(files, outs, max_in_flight=12)
    assert st == [0] * len(files)
    for o, s in zip(outs, singles):
        assert np.array_equal(o, s)
    # one broken file must not disturb its neighbours
    bad = list(files); bad[3] = files[3][: len(files[3]) // 2]
    outs2 = [np.zeros_like(s) for s in singles]
    st2 = gpu.decode_batch(bad, outs2, max_in_flight=12, raise_on_error=False) if "raise_on_error" in gpu.decode_batch.__code__.co_varnames else None
    if st2 is not None:
        assert st2[3] != 0 and all(s == 0 for i, s in enumerate(st2) if i != 3)
        for i, (o, s) in enumerate(zip(outs2, singles)):
            if i != 3:
                assert np.array_equal(o, s)


@pytest.mark.parametrize("kw", [dict(effort=7), dict(effort=7, distance=8.0), dict(effort=3, force_strategy=24), dict(lossless=True, channels=4), dict(effort=5, channels=4),
                                dict(effort=7, bgra=True)])
def test_band_decode_stitches_to_the_full_frame(gpu, oracle, kw):
    """Config-5 style sharding on one GPU: the frame decoded as three bands of group rows equals the full decode bit for bit (each band
    reconstructs one extra group row per side, so gaborish + 3 EPF iterations see the same neighbours as in the full frame). The BGRA32
    bands are compared with the BGRA32 surface of the whole file."""
    kw = dict(kw)
    ch = kw.pop("channels", 3)
    bgra = kw.pop("bgra", False)
    img = oracle.synthetic_image(700, 1500, seed=31, channels=ch)
    data = oracle.encode(img, **kw)
    if bgra:
        full = gpu.load_image_bgra(data)
    else:
        ld = _decode_gpu(gpu, data).layer_data
        full = ld.color if ld.transparency is None else np.concatenate([ld.color, ld.transparency[..., None]], axis=2)
    w, h, gdim, rows = gpu.band_layout(data)
    assert (w, h) == (700, 1500) and rows == -(-1500 // gdim)
    cuts = [0, 1, rows - 2, rows] if rows >= 4 else [0, 1, rows]
    parts = [gpu.decode_band(data, a, b, bgra=bgra) for a, b in zip(cuts[:-1], cuts[1:]) if b > a]
    assert np.array_equal(np.concatenate(parts, axis=0), full)
    with pytest.raises(gpu.FormatException):
        gpu.decode_band(data, 0, rows + 1)


def test_call_after_an_invalid_device_index_succeeds(gpu, oracle):
    """A call given a device index that does not exist fails with its own status. The runtime keeps that failure in the thread's error
    state; the next call on the same thread must not read it as a refused kernel launch of its own."""
    img = oracle.synthetic_image(300, 200, seed=4)
    data = oracle.encode(img, effort=7, distance=1.0)
    ref = _decode_gpu(gpu, data).layer_data.color
    bgra = np.concatenate([img[..., ::-1], np.full(img.shape[:2] + (1,), 255, np.uint8)], axis=2)
    bad = 4096
    with pytest.raises(gpu.FormatException) as e:
        gpu.decode_band(data, 0, 1, device=bad)
    assert e.value.status == "InvalidParameter"
    assert np.array_equal(_decode_gpu(gpu, data).layer_data.color, ref)
    with pytest.raises(gpu.FormatException, match="cudaSetDevice"):
        gpu.BandEncoder(bgra, 200, 0, 0, 0, gpu.EncoderOptions(quality=90, effort=3), device=bad)
    assert oracle.psnr(oracle.decode(gpu.encode_to_memory(bgra, gpu.EncoderOptions(quality=90, effort=3))).pixels, img) > 30.0


def test_large_batch_uses_bundles_and_wide_warps(gpu, oracle):
    """64+ files with 32+ streams is the configuration bench.py measures: two images per entropy launch and 16 AC sections per warp.
    Every output must equal the single-image decode of the same file."""
    distinct = [oracle.encode(oracle.synthetic_image(600 + 40 * i, 520, seed=90 + i), effort=7 if i % 2 else 3) for i in range(5)]
    singles = [_decode_gpu(gpu, f).layer_data.color for f in distinct]
    files = [distinct[i % 5] for i in range(70)]
    outs = [np.zeros_like(singles[i % 5]) for i in range(70)]
    st = gpu.decode_batch(files, outs, max_in_flight=40)
    assert st == [0] * 70
    for i, o in enumerate(outs):
        assert np.array_equal(o, singles[i % 5]), i


def test_two_batches_in_flight_through_submit_and_wait(gpu, oracle):
    """JxlB200DecodeBatchSubmit / Wait: a second batch submitted before the first is waited for; both deliver the single-image pixels,
    a corrupt file only fails its own status."""
    files = [oracle.encode(oracle.synthetic_image(320 + 16 * i, 240, seed=40 + i), effort=7 if i % 2 else 3) for i in range(4)]
    singles = [_decode_gpu(gpu, f).layer_data.color for f in files]
    a_files, b_files = [files[i % 4] for i in range(40)], [files[(i + 1) % 4] for i in range(36)]
    b_files[5] = b_files[5][: len(b_files[5]) // 2]                      # truncated: DecodeError for this one only
    a_out = [np.zeros_like(singles[i % 4]) for i in range(40)]
    b_out = [np.zeros_like(singles[(i + 1) % 4]) for i in range(36)]
    ha = gpu.decode_batch_submit(a_files, a_out, max_in_flight=32)
    hb = gpu.decode_batch_submit(b_files, b_out, max_in_flight=32)
    sb = hb.wait(raise_on_error=False)
    sa = ha.wait()
    assert sa == [0] * 40 and sb[5] == gpu.DECODER_STATUS.index("DecodeError") and all(s == 0 for k, s in enumerate(sb) if k != 5)
    for i in range(40):
        assert np.array_equal(a_out[i], singles[i % 4]), i
    for i in range(36):
        if i != 5:
            assert np.array_equal(b_out[i], singles[(i + 1) % 4]), i
