"""-m gpu tests of the SaveImage path: GPU-encoded files must decode with the CPU oracle (and with the GPU decoder)
to the source within lossy tolerance, bit-exactly for lossless, with the reference's pixel-format decisions."""
import io

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _bgra(img):
    h, w, c = img.shape
    out = np.empty((h, w, 4), np.uint8)
    if c == 1:
        out[..., 0] = out[..., 1] = out[..., 2] = img[..., 0]
        out[..., 3] = 255
    else:
        out[..., 0], out[..., 1], out[..., 2] = img[..., 2], img[..., 1], img[..., 0]
        out[..., 3] = img[..., 3] if c == 4 else 255
    return out


@pytest.mark.parametrize("w,h,ch,effort,quality", [(64, 48, 3, 3, 90), (300, 200, 3, 3, 90), (300, 200, 3, 1, 90), (519, 387, 4, 2, 75), (2100, 300, 1, 1, 90),   # efforts 1-2: prefix codes
                                                      (519, 387, 3, 7, 90), (300, 260, 4, 7, 75), (100, 90, 1, 7, 90), (2100, 300, 3, 5, 50)])
def test_lossy_save_roundtrip(gpu, oracle, w, h, ch, effort, quality):
    img = oracle.synthetic_image(w, h, seed=w, channels=ch)
    out = io.BytesIO()
    gpu.JpegXLSave.Save(_bgra(img), out, quality=quality, effort=effort)
    data = out.getvalue()
    d = oracle.decode(data, threads=4)
    assert d.is_container and (d.width, d.height) == (w, h)
    assert d.num_channels == ch and d.has_alpha == (ch == 4) and d.format == (0 if ch == 1 else 1)
    color = d.pixels[..., :3] if ch >= 3 else d.pixels[..., :1]
    src = img[..., :3] if ch >= 3 else img[..., :1]
    assert oracle.psnr(color, src) > (30.0 if quality >= 75 else 26.0)
    if ch == 4:
        assert np.array_equal(d.pixels[..., 3], img[..., 3])
    # the GPU decoder agrees with the oracle on the GPU-encoded file
    image = gpu.DecoderImage()
    gpu.JpegXLNative.LoadImage(data, image)
    got = image.layer_data.color[..., :color.shape[2]]
    assert int(np.abs(got.astype(np.int32) - color.astype(np.int32)).max()) <= 1


def test_gpu_encoder_close_to_oracle_encoder(gpu, oracle):
    """Same settings (DCT8-only, no gab/EPF): the two encoders quantise the same coefficients up to fp32 rounding."""
    img = oracle.synthetic_image(520, 392, seed=5)
    a = gpu.encode_to_memory(_bgra(img), gpu.EncoderOptions(quality=90, effort=3))
    b = oracle.encode(img, effort=3, distance=1.0, intent=0)
    da, db = oracle.decode(a).pixels, oracle.decode(b).pixels
    assert abs(oracle.psnr(da, img) - oracle.psnr(db, img)) < 0.05
    assert abs(len(a) - len(b)) < 0.02 * len(b)
    assert oracle.psnr(da, db) > 55.0


@pytest.mark.parametrize("w,h,ch", [(200, 150, 3), (300, 260, 4), (100, 90, 1), (700, 600, 3), (64, 64, 4)])
def test_lossless_save_bit_exact(gpu, oracle, w, h, ch):
    img = oracle.synthetic_image(w, h, seed=h, channels=ch)
    if ch == 1:
        pass
    data = gpu.encode_to_memory(_bgra(img), gpu.EncoderOptions(lossless=True, effort=7))
    d = oracle.decode(data)
    assert d.xyb == 0 and np.array_equal(d.pixels, img)
    surf = gpu.load_image_bgra(data)
    assert np.array_equal(surf, _bgra(img))


def test_progress_sequence_and_cancel(gpu, oracle):
    img = oracle.synthetic_image(300, 200, seed=1)
    seen = []
    out = io.BytesIO()
    gpu.JpegXLSave.Save(_bgra(img), out, progress_callback=lambda p: (seen.append(p), True)[1])
    # 0,5,15,20,25, then +5 per output buffer starting from 30 (capped at 90), 95 before the flush, buffers continue after it
    assert seen[:5] == [0, 5, 15, 20, 25] and seen[5] == 35 and 95 in seen and max(seen) == 95
    rest = [p for p in seen[5:] if p != 95]
    assert all(b >= a for a, b in zip(rest, rest[1:])) and max(rest) <= 90
    with pytest.raises(gpu.OperationCanceledException):
        gpu.JpegXLSave.Save(_bgra(img), io.BytesIO(), progress_callback=lambda p: p < 20)


def test_metadata_boxes_pass_through(gpu, oracle):
    img = oracle.synthetic_image(64, 64, seed=2)
    exif = b"\x00\x00\x00\x00II*\x00\x08\x00\x00\x00\x00\x00"
    out = io.BytesIO()
    gpu.JpegXLSave.Save(_bgra(img), out, exif=exif, xmp=b"<x:xmpmeta/>")
    d = oracle.decode(out.getvalue())
    assert d.exif == exif and d.xmp == [b"<x:xmpmeta/>"]


def test_write_error_is_sticky(gpu, oracle):
    class Broken(io.RawIOBase):
        def write(self, b):
            raise IOError("disk full")
    img = oracle.synthetic_image(64, 64, seed=3)
    with pytest.raises(IOError):
        gpu.JpegXLSave.Save(_bgra(img), Broken())


@pytest.mark.parametrize("ch,kw,bands", [(3, dict(quality=90, effort=3), 3), (4, dict(quality=90, effort=1), 3), (4, dict(lossless=True, effort=1), 2), (3, dict(quality=90, effort=7), 2), (4, dict(quality=75, effort=7), 3),
                                         (4, dict(lossless=True), 3), (1, dict(quality=90, effort=5), 8)])
def test_banded_encode_is_bit_identical_to_save_image(gpu, oracle, ch, kw, bands):
    """Sharded encode (SURVEY §8e): bands of whole LF-group rows, each through its own JxlB200BandEncoder session, flags OR-ed and histograms
    summed between the steps. The assembled file must be the file SaveImage writes for the whole frame — including with gaborish on
    (effort >= 5), where a band needs its neighbours' rows for the inverse-gaborish stencil — and must decode."""
    w, h = 520, 4500                                      # 3 LF-group rows: bands of 2048, 2048 and 404 rows
    img = oracle.synthetic_image(w, h, seed=31 + ch, channels=ch)
    surface = _bgra(img)
    opts = gpu.EncoderOptions(**kw)
    whole = gpu.encode_to_memory(surface, opts)
    banded = gpu.encode_in_bands(surface, opts, bands)
    assert banded == whole
    image = gpu.DecoderImage()
    gpu.JpegXLNative.LoadImage(banded, image)
    got = image.layer_data.color[..., :min(ch, 3)]
    src = img[..., :3] if ch >= 3 else img[..., :1]
    if kw.get("lossless"):
        assert np.array_equal(got, src) and np.array_equal(image.layer_data.transparency, img[..., 3])
    else:
        assert oracle.psnr(got[..., :src.shape[2]], src) > 26.0


def test_band_encoder_rejects_misaligned_bands(gpu, oracle):
    img = _bgra(oracle.synthetic_image(300, 2500, seed=2))
    opts = gpu.EncoderOptions(quality=90, effort=3)
    with pytest.raises(gpu.FormatException, match="multiple of 2048"):
        gpu.BandEncoder(img[1000:2500], 2500, 1000, 0, 0, opts)           # a band must start on an LF-group row
    with pytest.raises(gpu.FormatException, match="halo"):
        gpu.BandEncoder(img[2048:2500], 2500, 2048, 0, 0, opts)           # and bring the 8 rows above it


def test_refused_launch_fails_the_save(gpu):
    """A 64 x 65 536 bitmap is taller than the grid of the colour / alpha scan can reach (grid.y <= 65 535): the runtime refuses that
    launch before it reaches the device. SaveImage must fail with EncodeError rather than write the image as gray and opaque."""
    w, h = 64, 65536
    y, x = np.mgrid[0:h, 0:w]
    bgra = np.stack([(x * 4) % 256, y % 256, (x + y) % 256, 255 - y % 7], axis=-1).astype(np.uint8)
    out = io.BytesIO()
    try:
        gpu.JpegXLSave.Save(bgra, out, lossless=True)
    except gpu.FormatException as e:
        assert e.status == "EncodeError" and "CUDA" in str(e), (e.status, str(e))
        return
    image = gpu.DecoderImage()
    gpu.JpegXLNative.LoadImage(out.getvalue(), image)
    assert np.array_equal(image.layer_data.color, bgra[..., 2::-1]) and np.array_equal(image.layer_data.transparency, bgra[..., 3])
