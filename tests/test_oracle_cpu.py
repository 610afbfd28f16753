"""CPU tests of the oracle (the checker): known-answer material constructible offline (SURVEY.md §8c) and the committed goldens.
PARITY UNPINNED against libjxl — these pin the restatement against itself, closed forms and the reference's own constants."""
import json
import math
import os

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden")
INDEX = json.load(open(os.path.join(GOLDEN, "index.json")))


@pytest.mark.parametrize("name", sorted(INDEX))
def test_golden_files_decode_to_committed_pixels(oracle, name):
    data = open(os.path.join(GOLDEN, name + ".jxl"), "rb").read()
    want = np.load(os.path.join(GOLDEN, name + ".npy"))
    got = oracle.decode(data, threads=2).pixels
    assert got.shape == want.shape and np.array_equal(got, want)
    meta = INDEX[name]
    if meta["lossless"]:
        src = oracle.synthetic_image(meta["image"]["w"], meta["image"]["h"], seed=meta["image"]["seed"], channels=meta["image"]["ch"])
        assert np.array_equal(got, src)


def test_golden_files_are_what_the_encoder_still_produces(oracle):
    for name in ("lossy_e3_64x48", "lossless_gray_40x30"):
        m = INDEX[name]
        img = oracle.synthetic_image(m["image"]["w"], m["image"]["h"], seed=m["image"]["seed"], channels=m["image"]["ch"])
        assert oracle.encode(img, **m["encode"]) == open(os.path.join(GOLDEN, name + ".jxl"), "rb").read()


# covered 8x8 cells (rows, columns) per AC strategy; 14-17 (AFV) are not supported
COVERED_Y = [1, 1, 1, 1, 2, 4, 2, 1, 4, 1, 4, 2, 1, 1, 1, 1, 1, 1, 8, 8, 4, 16, 16, 8, 32, 32, 16]
COVERED_X = [1, 1, 1, 1, 2, 4, 1, 2, 1, 4, 2, 4, 1, 1, 1, 1, 1, 1, 8, 4, 8, 16, 8, 16, 32, 16, 32]
PLAIN_DCTS = [0, 4, 5, 6, 7, 8, 9, 10, 11, 18, 19, 20, 21, 22, 23, 24, 25, 26]


@pytest.mark.parametrize("strategy", [0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 18, 19, 20, 21, 22, 23, 24, 25, 26])
def test_transforms_invert_and_match_fp64_dct(oracle, strategy):
    L = oracle.lib()
    H, W = COVERED_Y[strategy] * 8, COVERED_X[strategy] * 8
    rng = np.random.default_rng(strategy)
    px = rng.standard_normal((H, W)).astype(np.float32)
    coef = np.zeros(H * W, np.float32)
    back = np.zeros((H, W), np.float32)
    L.jxlo_transform_from_pixels(strategy, px.ctypes.data, W, coef.ctypes.data)
    L.jxlo_transform_to_pixels(strategy, coef.ctypes.data, back.ctypes.data, W)
    assert np.max(np.abs(back - px)) < 2e-5
    if strategy in PLAIN_DCTS:   # separable textbook fp64 DCT-II scaled by 1/N per dimension
        def dct_mat(n):
            k, i = np.meshgrid(np.arange(n), np.arange(n), indexing="ij")
            m = np.cos((2 * i + 1) * k * np.pi / (2 * n)) * np.where(k == 0, 1.0, np.sqrt(2.0))
            return m / n
        F = dct_mat(H) @ px.astype(np.float64) @ dct_mat(W).T      # F[vf][hf]
        # SURVEY A.9 storage: min(H, W) rows of max(H, W) coefficients, the longer side horizontal. A block at least as tall as wide
        # (square ones included) is stored transposed, S[hf][vf]; a wide one as it is, S[vf][hf].
        if H >= W:
            S = coef.reshape(W, H).T
        else:
            S = coef.reshape(H, W)
        assert np.max(np.abs(S - F)) < 2e-6 * max(1.0, np.abs(F).max())
        assert abs(S[0, 0] - px.mean()) < 1e-6                      # DC = block mean (A.9 scaling)
        # the inverse is the fp64 DCT-III of the same coefficients
        Fi = rng.standard_normal((H, W)) * np.exp(-np.add.outer(np.arange(H) / H, np.arange(W) / W) * 4)
        stored = (Fi.T if H >= W else Fi).astype(np.float32).reshape(-1)
        L.jxlo_transform_to_pixels(strategy, stored.ctypes.data, back.ctypes.data, W)
        want = np.linalg.solve(dct_mat(H), np.linalg.solve(dct_mat(W), Fi.astype(np.float32).astype(np.float64).T).T)
        assert np.max(np.abs(back - want)) < 1e-5 * max(1.0, np.abs(want).max())


def test_gaborish_stage_matches_fp64_convolution(oracle):
    """SURVEY A.10 gaborish in float64 (default weights w1 = 0.115169525, w2 = 0.061248592 for every channel, 3x3 kernel
    [w2 w1 w2; w1 1 w1; w2 w1 w2] / (1 + 4 w1 + 4 w2), edges mirrored at the image size, not at the padded size) on the oracle's
    reconstruction reproduces the oracle's gaborish stage inside the image."""
    w, h = 203, 141                                                  # neither a multiple of 8: the planes carry padding
    data = oracle.encode(oracle.synthetic_image(w, h, seed=4), effort=7, gab=1, epf=0)
    d = oracle.decode(data, keep_stages=True)
    idct = d.stages["idct"].reshape(3, d.ypad, d.xpad).astype(np.float64)[:, :h, :w]
    gab = d.stages["gab"].reshape(3, d.ypad, d.xpad)[:, :h, :w]
    w1, w2 = 0.115169525, 0.061248592
    norm = 1 + 4 * w1 + 4 * w2
    p = np.pad(idct, ((0, 0), (1, 1), (1, 1)), mode="symmetric")    # x[-1] = x[0], x[n] = x[n - 1]
    def at(dy, dx):
        return p[:, 1 + dy:1 + dy + h, 1 + dx:1 + dx + w]
    want = (at(0, 0) + w1 * (at(-1, 0) + at(1, 0) + at(0, -1) + at(0, 1)) + w2 * (at(-1, -1) + at(-1, 1) + at(1, -1) + at(1, 1))) / norm
    err = np.abs(gab - want).max(axis=(1, 2)) / np.abs(want).max(axis=(1, 2))
    assert np.all(err < 1e-6), err                                   # fp32 rounding of the weights and the sums
    assert np.abs(gab - idct).max() > 1e-3                           # the filter did something


def test_resample_scale_closed_form(oracle):
    def s(n, u):
        return 1.0 / np.prod([math.cos(u * math.pi * (1 << k) / (16.0 * n)) for k in range(3)])
    assert abs(s(2, 1) - 1.108937353592731823) < 1e-12
    for u, v in zip((1, 2, 3), (1.02576009678, 1.10893735359, 1.27055936877)):
        assert abs(s(4, u) - v) < 1e-9
    # LLF of a DCT16 block from a constant LF patch is the constant itself in position 0
    import ctypes as C
    L = oracle.lib()
    dc = np.full((2, 2), 0.37, np.float32)
    block = np.zeros(256, np.float32)
    L.jxlo_llf_from_dc(4, dc.ctypes.data, 2, block.ctypes.data)
    assert abs(block[0] - 0.37) < 1e-6 and abs(block[1]) < 1e-6 and abs(block[16]) < 1e-6


def test_opsin_matrices_are_inverse_and_colour_roundtrips(oracle):
    M = np.array([[0.30, 0.622, 0.078], [0.23, 0.692, 0.078], [0.24342268924547819, 0.20476744424496821, 0.55180986650955360]])
    Mi = np.array([[11.031566901960783, -9.866943921568629, -0.16462299647058826], [-3.254147380392157, 4.418770392156863, -0.16462299647058826],
                   [-3.6588512862745097, 2.7129230470588235, 1.9459282392156863]])
    assert np.max(np.abs(Mi @ M - np.eye(3))) < 1e-6
    L = oracle.lib()
    rng = np.random.default_rng(0)
    rgb = rng.integers(0, 256, (4096, 3), dtype=np.uint8)
    x, y, b = (np.zeros(4096, np.float32) for _ in range(3))
    L.jxlo_srgb8_to_xyb(rgb.ctypes.data, 4096, x.ctypes.data, y.ctypes.data, b.ctypes.data)
    out = np.zeros((4096, 3), np.uint8)
    L.jxlo_xyb_to_srgb8(x.ctypes.data, y.ctypes.data, b.ctypes.data, 4096, out.ctypes.data)
    assert np.array_equal(out, rgb)


def test_natural_order_is_a_permutation_with_llf_first(oracle):
    L = oracle.lib()
    sizes = [64, 64, 256, 1024, 128, 256, 512, 4096, 2048, 16384, 8192, 65536, 32768]
    for o, n in enumerate(sizes):
        buf = np.zeros(n, np.uint32)
        assert L.jxlo_natural_order(o, buf.ctypes.data) == n
        assert np.array_equal(np.sort(buf), np.arange(n, dtype=np.uint32))
    buf = np.zeros(64, np.uint32)
    L.jxlo_natural_order(0, buf.ctypes.data)
    assert list(buf[:4]) == [0, 1, 8, 16]


def test_dequant_tables_positive_and_dct8_values(oracle):
    L = oracle.lib()
    n = L.jxlo_dequant_table(0, None)
    t = np.zeros(n, np.float32)
    L.jxlo_dequant_table(0, t.ctypes.data)
    assert n == 192 and np.all(t > 0)
    assert abs(t[0] - 1 / 3150.0) < 1e-9 and abs(t[64] - 1 / 560.0) < 1e-9 and abs(t[128] - 1 / 512.0) < 1e-9   # A.8 DCT8 band 0
    for table in range(1, 17):
        if table == 10:
            continue   # AFV: not restated
        m = L.jxlo_dequant_table(table, None)
        tt = np.zeros(m, np.float32)
        L.jxlo_dequant_table(table, tt.ctypes.data)
        assert np.all(np.isfinite(tt)) and np.all(tt > 0)


@pytest.mark.parametrize("kw", [dict(effort=3), dict(effort=7), dict(effort=5, use_prefix=1), dict(effort=7, distance=6.0), dict(lossless=1), dict(lossless=1, use_prefix=1)])
def test_encode_decode_identities(oracle, kw):
    img = oracle.synthetic_image(141, 99, seed=9, channels=4)
    d = oracle.decode(oracle.encode(img, **kw))
    assert d.pixels.shape == img.shape and np.array_equal(d.pixels[..., 3], img[..., 3])
    if kw.get("lossless"):
        assert np.array_equal(d.pixels, img)
    else:
        assert oracle.psnr(d.pixels[..., :3], img[..., :3]) > 27.0


def test_oracle_rejects_bad_input(oracle):
    with pytest.raises(oracle.OracleError):
        oracle.decode(b"\x00\x01\x02\x03")
    data = oracle.encode(oracle.synthetic_image(300, 200, seed=1), effort=3)
    with pytest.raises(oracle.OracleError):
        oracle.decode(data[: len(data) // 2])
    assert oracle.lib().jxlo_signature_check(data, len(data)) == 2
    assert oracle.lib().jxlo_signature_check(b"\xff\x0a", 2) == 1


def test_orientation_and_16bit_float_outputs(oracle):
    img = oracle.synthetic_image(40, 24, seed=3)
    for orient in range(1, 9):
        d = oracle.decode(oracle.encode(img, lossless=1, orientation=orient))
        assert (d.width, d.height) == ((24, 40) if orient >= 5 else (40, 24))
    base = oracle.decode(oracle.encode(img, lossless=1)).pixels
    assert np.array_equal(oracle.decode(oracle.encode(img, lossless=1, orientation=2)).pixels, base[:, ::-1])
    assert np.array_equal(oracle.decode(oracle.encode(img, lossless=1, orientation=3)).pixels, base[::-1, ::-1])
    assert np.array_equal(oracle.decode(oracle.encode(img, lossless=1, orientation=4)).pixels, base[::-1])
    assert np.array_equal(oracle.decode(oracle.encode(img, lossless=1, orientation=5)).pixels, base.transpose(1, 0, 2))
    f = img.astype(np.float32) / 255.0
    d16 = oracle.decode(oracle.encode(f, bits=16, effort=3))
    assert d16.sample_type == 1 and d16.pixels.dtype == np.uint16 and oracle.psnr(d16.pixels / 257.0, img) > 30
    dh = oracle.decode(oracle.encode(f, bits=16, exp_bits=5, effort=3))
    assert dh.sample_type == 2 and dh.pixels.dtype == np.float16
    df = oracle.decode(oracle.encode(f, bits=32, exp_bits=8, effort=3))
    assert df.sample_type == 3 and df.pixels.dtype == np.float32 and oracle.psnr(df.pixels * 255.0, img) > 30


# ---------------------------------------------------------------- ICC profile stream (SURVEY A.3 "ICC stream")
def _varint(v):
    out = bytearray()
    while v > 127:
        out.append((v & 127) | 128)
        v >>= 7
    out.append(v)
    return bytes(out)


def test_icc_stream_round_trip(oracle):
    import icc_util
    rng = np.random.default_rng(5)
    profiles = [icc_util.make_matrix_icc(icc_util.P3_PRIMS, gamma=2.2), icc_util.make_matrix_icc(icc_util.ADOBE_PRIMS, gamma=2.19921875, curve="curv1"),
                icc_util.make_matrix_icc(icc_util.SRGB_PRIMS, gamma=2.4, curve="table"), bytes(rng.integers(0, 256, 1, dtype=np.uint8)),
                bytes(rng.integers(0, 256, 127, dtype=np.uint8)), bytes(rng.integers(0, 256, 128, dtype=np.uint8)), bytes(rng.integers(0, 256, 5000, dtype=np.uint8))]
    for icc in profiles:
        stream = oracle.icc_stream_write(icc)
        assert oracle.icc_stream_read(stream) == icc
    # the predicted header makes a real profile's first 128 bytes nearly free
    real = profiles[0]
    assert len(oracle.icc_stream_write(real)) < len(real)


def test_icc_predictor_commands(oracle):
    """Hand-written command streams through the predictor: tag-table shortcuts (TRC / XYZ triples, named tags, explicit offsets), type
    keywords, the XYZ command, shuffled and N-th order predicted runs. Expected bytes are computed here, independently of the C++."""
    import struct
    header = bytearray(128)
    header[8] = 4; header[12:16] = b"mntr"; header[16:20] = b"RGB "; header[20:24] = b"XYZ "; header[36:40] = b"acsp"
    header[68:80] = bytes([0, 0, 0xF6, 0xD6, 0, 1, 0, 0, 0, 0, 0xD3, 0x2D])
    # expected profile: header (with a few deviations from the prediction), tag table of 8 tags, then content
    # (the implicit offset of the first tag is 128 + 12 * numtags: the predictor does not count the 4-byte tag count)
    want_tags = [(b"desc", 128 + 8 * 12, 40), (b"rTRC", 264, 16), (b"gTRC", 264, 16), (b"bTRC", 264, 16), (b"rXYZ", 280, 20), (b"gXYZ", 300, 20), (b"bXYZ", 320, 20), (b"ABCD", 1000, 7)]
    content = b"mluc" + b"\0" * 4 + bytes(range(32))                                        # type keyword command + raw insert
    content += b"XYZ " + b"\0" * 4 + bytes(range(100, 112))                                  # XYZ command
    ramp16 = b"".join(struct.pack(">H", 1000 + 37 * i) for i in range(24))                   # order-1, width-2 predictable ramp
    content += ramp16
    shuf_src = bytes(range(200, 216))                                                        # shuffle-4 run
    content += shuf_src
    total = 128 + 4 + 12 * len(want_tags) + len(content)
    hdr = bytearray(header); hdr[0:4] = struct.pack(">I", total); hdr[4:8] = b"lcms"; hdr[40:44] = b"APPL"; hdr[80:84] = b"lcms"; hdr[100] = 9
    expected = bytes(hdr) + struct.pack(">I", len(want_tags)) + b"".join(s + struct.pack(">II", o, n) for s, o, n in want_tags) + content

    # --- encode by hand
    pred = bytearray(header); pred[0:4] = struct.pack(">I", total)
    data = bytearray()
    for i in range(128):
        if i == 8:
            pred[80:84] = hdr[4:8]
        if i == 41 and hdr[40] == ord("A"):
            pred[41:44] = b"PPL"
        data.append((hdr[i] - pred[i]) & 255)
    cmds = bytearray()
    cmds += _varint(len(want_tags) + 1)
    cmds += bytes([4 + 12 | 128]) + _varint(40)                     # 'desc' (string index 12), implicit offset, explicit size
    cmds += bytes([2 | 128]) + _varint(16)                          # TRC triple, implicit offset (= 224 + 40), explicit size
    cmds += bytes([3])                                              # XYZ triple: offset = prev start + prev size, size 20 implied
    cmds += bytes([1 | 64 | 128]) + _varint(1000) + _varint(7)      # unknown tag: keyword from the data stream, explicit offset + size
    data += b"ABCD"
    cmds += bytes([0])                                              # end of tag list
    cmds += bytes([16 + 3])                                         # type keyword 'mluc' + 4 zero bytes
    cmds += bytes([1]) + _varint(32); data += bytes(range(32))     # insert
    cmds += bytes([10]); data += bytes(range(100, 112))             # XYZ
    # predicted run: width 2 (flags bits 0-1 = 1), order 1 (bits 2-3 = 1), default stride = width; residuals then byte-plane split
    first = ramp16[:4]
    cmds += bytes([1]) + _varint(4); data += first
    resid = bytearray()
    vals = [1000 + 37 * i for i in range(24)]
    prevbytes = bytes(expected[: expected.index(ramp16) + 4])
    out_so_far = bytearray(prevbytes)
    for i in range(2, 24):
        p1 = (out_so_far[-2] << 8) | out_so_far[-1]; p2 = (out_so_far[-4] << 8) | out_so_far[-3]
        pr = (2 * p1 - p2) & 0xFFFF
        hi, lo = (vals[i] >> 8) & 255, vals[i] & 255
        resid += bytes([(hi - (pr >> 8)) & 255, (lo - (pr & 255)) & 255])
        out_so_far += bytes([hi, lo])
    n = len(resid); planes = bytes(resid[0::2]) + bytes(resid[1::2])   # encoder side of Shuffle(width 2)
    cmds += bytes([4, 1 | (1 << 2)]) + _varint(n); data += planes
    cmds += bytes([3]) + _varint(16); data += bytes(shuf_src[0::4]) + bytes(shuf_src[1::4]) + bytes(shuf_src[2::4]) + bytes(shuf_src[3::4])
    enc = _varint(total) + _varint(len(cmds)) + bytes(cmds) + bytes(data)
    got = oracle.icc_unpredict(enc)
    assert got == expected


def test_icc_profile_travels_through_the_codestream(oracle):
    import icc_util
    icc = icc_util.make_matrix_icc(icc_util.P3_PRIMS, gamma=2.2)
    img = oracle.synthetic_image(96, 64, seed=9)
    d = oracle.decode(oracle.encode(img, lossless=True, icc=icc))
    assert d.icc == icc and d.known_profile == -1 and np.array_equal(d.pixels, img)


@pytest.mark.parametrize("mode", ["replace", "add", "blend", "muladd", "mul"])
def test_layered_files_decode_to_the_blend_formulas(oracle, mode):
    """Multi-frame stills (layers): the oracle's compositing loop against a numpy statement of the blend modes, crops inside and across the
    canvas border, and a third layer that blends onto a reference slot other than the one the second layer wrote."""
    import layer_util as L
    W, H = 160, 120
    base = oracle.synthetic_image(W, H, seed=1, channels=4)
    base[..., 3] = np.maximum(base[..., 3], 100)
    over = oracle.synthetic_image(70, 50, seed=2, channels=4)
    for x0, y0 in ((30, 20), (-20, 90), (120, -10)):
        data = oracle.encode_layers(W, H, [(base, dict()), (over, dict(x0=x0, y0=y0, mode=mode))], lossless=1)
        got = oracle.decode(data).pixels
        want = L.to_u8(L.composite(base.astype(np.float32) / 255.0, over.astype(np.float32) / 255.0, x0, y0, mode))
        assert got.shape == (H, W, 4) and int(np.abs(got.astype(np.int32) - want.astype(np.int32)).max()) == 0
    other = oracle.synthetic_image(W, H, seed=3, channels=4)
    layers = [(base, dict(save=1)), (other, dict(source=2, save=2, mode="add")), (over, dict(x0=40, y0=30, source=1, mode=mode))]
    got = oracle.decode(oracle.encode_layers(W, H, layers, lossless=1)).pixels
    want = L.to_u8(L.composite(base.astype(np.float32) / 255.0, over.astype(np.float32) / 255.0, 40, 30, mode))
    assert int(np.abs(got.astype(np.int32) - want.astype(np.int32)).max()) == 0
