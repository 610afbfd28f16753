"""-m gpu stage tests of the VarDCT decoder: the GPU's intermediate planes against the oracle's, and the rendered samples against a float64
restatement of the colour conversion (SURVEY.md A.10).

The pixel-level parity tests allow 1 LSB of 8-bit output, which hides any systematic error of a stage that stays below about 0.4 % of full
scale. Here every stage is compared at the precision it is computed in:
  * quantised coefficients (JxlB200DebugDecodeStage which=4): exact integer equality;
  * LF planes after dequantisation, chroma-from-luma and adaptive smoothing (which=3): fp32 level, relative to each channel's range;
  * reconstruction after dequantisation, CfL, LLF and the inverse transforms (which=0): fp32 level, relative to each channel's range;
  * output samples: within half a code unit (+ a measured delta) of a float64 colour conversion of the oracle's filtered planes.
Each float bound sits at about 4x the worst value measured on a B200 and is checked against what one 8-bit LSB means in that stage."""
import numpy as np
import pytest
from spec_cases import OPSIN_BIAS, OPSIN_INV

pytestmark = pytest.mark.gpu

ALL_STRATEGIES = [0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 18, 19, 20, 21, 22, 23, 24, 25, 26]
MIXED = dict(effort=7, distance=1.0, varblock_scale=4.0, varblock_pattern=1)   # the variable-block workload of bench.py

# Relative to the channel's range (max |value| of the oracle plane), about 4x the worst case measured on a B200 (1000 W). One 8-bit LSB
# is at least 1.3e-3 of the range in these stages (lsb_in_xyb at the most sensitive sample), so each bound is checked to be 20x below it.
LF_REL_BOUND = 4e-6      # measured 9.3e-7 (X channel, 2100 x 300: smoothing across the LF-group border); 0 where the GPU skips smoothing
RECON_REL_BOUND = 7e-6   # measured 1.7e-6 (B channel, DCT256); 1.4e-6 for DCT16, under 8e-7 for DCT8 and the 8x8 special transforms

# Which reconstruction kernel handles a strategy (dev/recon_kernels.cu LaunchReconstruct): DCT8 has its own kernel, varblocks whose longer
# side is at most 16 px go to k_reconstruct<16>, 32-px ones to k_reconstruct<32>, and a side of 64 px or more to the large-block pass.
RECON_KERNEL = {0: "k_reconstruct_dct8", **{s: "k_reconstruct<16>" for s in (1, 2, 3, 4, 6, 7, 12, 13)},
                **{s: "k_reconstruct<32>" for s in (5, 8, 9, 10, 11)}, **{s: ">=64 pass" for s in range(18, 27)}}


def _geometry(w, h):
    xb, yb = -(-w // 8), -(-h // 8)
    xg, yg = -(-w // 256), -(-h // 256)
    return xb, yb, xg, yg


def _encode(oracle, w, h, seed=None, channels=3, **kw):
    img = oracle.synthetic_image(w, h, seed=w + h if seed is None else seed, channels=channels)
    if any(k in kw for k in ("bits", "exp_bits")):
        img = img.astype(np.float32) / 255.0
    data = oracle.encode(img, **kw)
    return data, oracle.last_encode_strategy_cells()


def _gpu_coeffs(gpu, data, w, h):
    """GPU coefficients [group][c][32 x 32 cells][64] -> the oracle's [c][cell][64] (cell = by * xb + bx); also the largest |value| the
    GPU holds in cells outside the image."""
    xb, yb, xg, yg = _geometry(w, h)
    raw, _ = gpu.debug_decode_stage(data, 4, xg * yg * 3 * 65536)
    assert raw.size == xg * yg * 3 * 65536
    q = raw.astype(np.int32).reshape(xg * yg, 3, 32, 32, 64)
    out = np.zeros((3, yb, xb, 64), np.int32)
    outside = 0
    for g in range(xg * yg):
        gy, gx = divmod(g, xg)
        ch, cw = min(32, yb - 32 * gy), min(32, xb - 32 * gx)
        out[:, 32 * gy:32 * gy + ch, 32 * gx:32 * gx + cw] = q[g, :, :ch, :cw]
        outside = max(outside, int(np.abs(q[g, :, ch:]).max(initial=0)), int(np.abs(q[g, :, :ch, cw:]).max(initial=0)))
    return out.reshape(3, -1), outside


def _gpu_planes(gpu, data, which, w, h):
    xb, yb, _, _ = _geometry(w, h)
    if which == 3:
        v, _ = gpu.debug_decode_stage(data, 3, 3 * xb * yb)
        return v.reshape(3, yb, xb)
    v, (xpad, ypad) = gpu.debug_decode_stage(data, 0, 3 * 64 * xb * yb)
    assert (xpad, ypad) == (8 * xb, 8 * yb)
    return v.reshape(3, ypad, xpad)


def _rel_err(got, ref):
    """Per channel: max |got - ref| over the plane / max |ref| over the plane."""
    got, ref = got.reshape(3, -1).astype(np.float64), ref.reshape(3, -1).astype(np.float64)
    return np.abs(got - ref).max(axis=1) / np.maximum(np.abs(ref).max(axis=1), 1e-30)


# ------------------------------------------------------------------------------------------------ float64 colour reference (SURVEY A.10)
# CIE xy of the codestream's primaries enums (the sRGB values are the spec's, not the rounded 0.64 / 0.33 ...), all with the D65 white point
PRIMARIES = {1: ((0.639998686, 0.330010138), (0.300003784, 0.600003357), (0.150002046, 0.059997204)),
             9: ((0.708, 0.292), (0.170, 0.797), (0.131, 0.046)),
             11: ((0.680, 0.320), (0.265, 0.690), (0.150, 0.060))}
D65 = (0.3127, 0.3290)
TF_709, TF_LINEAR, TF_SRGB, TF_PQ, TF_HLG = 1, 8, 13, 16, 18
PQ_M1, PQ_M2, PQ_C1, PQ_C2, PQ_C3 = 2610.0 / 16384, 2523.0 / 4096 * 128, 3424.0 / 4096, 2413.0 / 4096 * 32, 2392.0 / 4096 * 32


def _rgb_to_xyz(prims):
    P = np.array([[x / y, 1.0, (1 - x - y) / y] for x, y in prims]).T      # columns: XYZ of each primary at Y = 1
    wx, wy = D65
    S = np.linalg.solve(P, np.array([wx / wy, 1.0, (1 - wx - wy) / wy]))
    return P * S


def linear_srgb_to(primaries):
    return np.linalg.solve(_rgb_to_xyz(PRIMARIES[primaries]), _rgb_to_xyz(PRIMARIES[1]))


def transfer(v, tf, intensity_target):
    a = np.abs(v)
    if tf == TF_LINEAR:
        r = a
    elif tf == TF_SRGB:
        r = np.where(a <= 0.0031308, 12.92 * a, 1.055 * np.power(a, 1 / 2.4) - 0.055)
    elif tf == TF_709:
        r = np.where(a < 0.018, 4.5 * a, 1.099 * np.power(a, 0.45) - 0.099)
    elif tf == TF_PQ:
        p = np.power(np.minimum(a * intensity_target / 10000.0, 1.0), PQ_M1)
        r = np.power((PQ_C1 + PQ_C2 * p) / (1 + PQ_C3 * p), PQ_M2)
    elif tf == TF_HLG:
        r = np.where(a <= 1 / 12, np.sqrt(3 * a), 0.17883277 * np.log(np.maximum(12 * a - 0.28466892, 1e-300)) + 0.55991073)
    else:
        raise ValueError(tf)
    return np.sign(v) * r


def pq_to_linear(e):
    p = np.abs(e) ** (1 / PQ_M2)
    return np.sign(e) * (np.maximum(p - PQ_C1, 0) / (PQ_C2 - PQ_C3 * p)) ** (1 / PQ_M1)


def xyb_to_output(xyb, primaries=1, tf=TF_SRGB, intensity_target=255.0, opsin_inv=OPSIN_INV, opsin_bias=(OPSIN_BIAS,) * 3):
    """xyb: [3][h][w] float64 -> [h][w][3] colour samples in the output encoding (before the sample type). opsin_inv: the 3 x 3 inverse
    opsin matrix; opsin_bias: the three (positive) biases b of m = (g + cbrt(b))^3 - b."""
    X, Y, B = xyb
    bias = np.asarray(opsin_bias, np.float64)
    cb = np.cbrt(bias)
    mix = np.stack([(Y + X + cb[0]) ** 3 - bias[0], (Y - X + cb[1]) ** 3 - bias[1], (B + cb[2]) ** 3 - bias[2]], axis=-1)
    lin = mix @ (linear_srgb_to(primaries) @ np.asarray(opsin_inv, np.float64).reshape(3, 3)).T * (255.0 / intensity_target)
    return transfer(lin, tf, intensity_target)


def orient(a, orientation):
    return {1: lambda t: t, 2: lambda t: t[:, ::-1], 3: lambda t: t[::-1, ::-1], 4: lambda t: t[::-1], 5: lambda t: t.transpose(1, 0, 2),
            6: lambda t: t[::-1].transpose(1, 0, 2), 7: lambda t: t[::-1, ::-1].transpose(1, 0, 2), 8: lambda t: t[:, ::-1].transpose(1, 0, 2)}[orientation](a)


def lsb_in_xyb(xyb):
    """Per channel: the smallest XYB change that moves some 8-bit sRGB output of these samples by one code value (central differences of
    the float64 conversion at every sample, over the channel's range so that it compares with the relative bounds)."""
    h = 1e-6
    out = []
    for c in range(3):
        d = np.zeros((3, 1, 1))
        d[c] = h
        slope = np.abs(xyb_to_output(xyb + d) - xyb_to_output(xyb - d)).max() / (2 * h)
        out.append((1 / 255.0) / slope / max(np.abs(xyb[c]).max(), 1e-30))
    return np.array(out)


def _oracle_planes(d, name):
    return d.stages[name].reshape(3, d.ypad, d.xpad).astype(np.float64)


# ------------------------------------------------------------------------------------------------ 1. quantised coefficients: exact
COEFF_CASES = [("strategy%d" % s, 531, 277, dict(effort=3, force_strategy=s)) for s in ALL_STRATEGIES] + [
    ("mixed", 600, 456, MIXED),
    ("two_pass", 531, 277, dict(effort=7, num_passes=2)),        # the second pass adds into the int16 accumulator
    ("prefix_codes", 531, 277, dict(effort=5, use_prefix=1)),
    ("ragged_groups", 777, 555, dict(effort=7, distance=2.0)),   # 4 x 3 groups, the last column and row of groups partly outside
]


@pytest.mark.parametrize("name,w,h,kw", COEFF_CASES, ids=[c[0] for c in COEFF_CASES])
def test_quantised_coefficients_equal_the_oracle(gpu, oracle, name, w, h, kw):
    data, cells = _encode(oracle, w, h, **kw)
    if "force_strategy" in kw and kw["force_strategy"] != 0:
        assert cells[kw["force_strategy"]] > 0, "the encoder fell back to DCT8 for every block"
    ref = oracle.decode(data, threads=4, keep_stages=True).stages["coeffs"]
    got, outside = _gpu_coeffs(gpu, data, w, h)
    assert ref.shape == got.shape
    assert np.count_nonzero(ref) > 0
    assert outside == 0, "non-zero coefficients in cells outside the image"
    bad = np.argwhere(got != ref)
    assert bad.size == 0, "%d coefficients differ, first at (channel, index) %s: GPU %d, oracle %d" % (
        len(bad), tuple(bad[0]), got[tuple(bad[0])], ref[tuple(bad[0])])


# ------------------------------------------------------------------------------------------------ 1. LF planes: fp32 level
LF_CASES = [("w9", 9, 40, dict(effort=7)), ("w16", 16, 40, dict(effort=7)),                       # xb <= 2: neither side smooths
            ("h12", 60, 12, dict(effort=7)),                                                        # yb <= 2
            ("w17", 17, 40, dict(effort=7)), ("w24", 24, 33, dict(effort=7)),                       # exactly 3 blocks: one smoothed column
            ("skip_smoothing", 300, 200, dict(effort=7, skip_lf_smoothing=1)),
            ("two_lf_groups", 2100, 300, dict(effort=5)),                                           # smoothing across the 2048-px LF-group border
            ("aq_cfl", 531, 277, dict(effort=7, distance=2.0)),
            ("no_aq_cfl", 531, 277, dict(effort=7, cfl=0, adaptive_quant=0))]


@pytest.mark.parametrize("name,w,h,kw", LF_CASES, ids=[c[0] for c in LF_CASES])
def test_lf_planes_match_the_oracle(gpu, oracle, name, w, h, kw):
    data, _ = _encode(oracle, w, h, **kw)
    d = oracle.decode(data, threads=4, keep_stages=True)
    xb, yb, _, _ = _geometry(w, h)
    ref = d.stages["lf"].reshape(3, yb, xb).astype(np.float64)
    got = _gpu_planes(gpu, data, 3, w, h)
    err = _rel_err(got, ref)
    assert np.all(err <= LF_REL_BOUND), "LF planes differ by %s of the channel range" % err
    assert np.all(LF_REL_BOUND * 20 <= lsb_in_xyb(ref))


# ------------------------------------------------------------------------------------------------ 1. reconstruction: fp32 level
RECON_CASES = [("strategy%d" % s, 531, 277, dict(effort=3, force_strategy=s)) for s in ALL_STRATEGIES] + [
    ("mixed", 600, 456, MIXED),
    ("aq_cfl", 531, 277, dict(effort=7, distance=2.0)),
    ("no_aq_no_cfl", 531, 277, dict(effort=7, cfl=0, adaptive_quant=0)),
    ("cfl_only", 531, 277, dict(effort=7, adaptive_quant=0)),
    ("two_pass", 531, 277, dict(effort=7, num_passes=2)),
    ("edge_inside_last_cell", 509, 301, dict(effort=7, varblock_scale=4.0, varblock_pattern=1)),   # 509 = 63 cells + 5 px, 301 = 37 cells + 5 px
]


@pytest.mark.parametrize("name,w,h,kw", RECON_CASES, ids=[c[0] for c in RECON_CASES])
def test_reconstruction_matches_the_oracle(gpu, oracle, name, w, h, kw):
    data, cells = _encode(oracle, w, h, **kw)
    s = kw.get("force_strategy")
    if s is not None:
        assert cells[s] * 2 >= sum(cells), "strategy %d (%s) covers %d of %d cells" % (s, RECON_KERNEL[s], cells[s], sum(cells))
    d = oracle.decode(data, threads=4, keep_stages=True)
    ref = _oracle_planes(d, "idct")
    got = _gpu_planes(gpu, data, 0, w, h).astype(np.float64)
    err = _rel_err(got, ref)
    assert np.all(err <= RECON_REL_BOUND), "reconstruction differs by %s of the channel range" % err
    assert np.all(RECON_REL_BOUND * 20 <= lsb_in_xyb(ref[:, :h, :w]))


def test_every_reconstruction_kernel_is_exercised():
    assert set(RECON_KERNEL) == set(ALL_STRATEGIES)
    assert set(RECON_KERNEL.values()) == {"k_reconstruct_dct8", "k_reconstruct<16>", "k_reconstruct<32>", ">=64 pass"}


# ------------------------------------------------------------------------------------------------ 2. rendered samples vs float64 colour
def render_branch(gab, epf, w, h, sample="u8", alpha=False, orientation=1, bgra=False):
    """The kernel LaunchFusedRender / LaunchRenderT / LaunchOutput (dev/recon_kernels.cu) select for a VarDCT frame with these parameters
    (device buffers are always aligned, so the alignment conditions hold)."""
    if not gab and not epf:
        return "k_output"
    rgb8 = not bgra and sample == "u8" and not alpha and orientation == 1
    fast_bgra = bgra and not alpha and orientation == 1
    if (rgb8 or fast_bgra) and gab == 1 and epf == 1:
        return "k_render_wide_tma<1,%s>" % ("true" if bgra else "false")
    return "k_render<%d,%d,%s>" % (gab, epf, "true" if rgb8 and (w * 3) % 4 == 0 else "false")


# Output bounds, about 4x the worst case measured on a B200 (1000 W): |got - real| <= 0.5 + delta code units for integer samples.
U8_DELTA = 1e-3          # measured 2.3e-4 (k_render_wide_tma, 191 x 161)
U16_DELTA = 0.2          # measured 0.049 (Rec.709 transfer); the bound is 1/1285 of an 8-bit LSB
F32_REL = 3e-5           # relative, floor 1e-3; measured 6.8e-6 (linear sRGB)
F16_REL = 5e-6           # relative, over half a binary16 ulp; measured 1.2e-6
PQ_LIN_REL, PQ_LIN_ABS = 2e-4, 1.2e-7   # PQ in linear light (relative term as test_config4b_8k_hdr_pq); measured 2.7e-8 over the relative term


def _pq_dark_in_linear_light(got, real):
    """PQ has unbounded slope at black: a 1e-7 fp32 difference of a dark linear sample moves its code value by 1e-3. Every sample is
    compared in linear light (relative + absolute, the treatment of test_config4b_8k_hdr_pq); the code-value bound applies from 100 cd/m2
    (1e-2 of the PQ range) up. Returns the mask of those samples."""
    lin_g, lin_r = pq_to_linear(got), pq_to_linear(real)
    worst = float((np.abs(lin_g - lin_r) - PQ_LIN_REL * np.abs(lin_r)).max())
    assert worst <= PQ_LIN_ABS, "linear light differs by %.3g over %.0e relative" % (worst, PQ_LIN_REL)
    return lin_r >= 1e-2

GW = dict(gab=1, epf=1)
RENDER_CASES = [
    # wide 64x32 tiles, TMA loads: sizes at 64k +- 1 and 32k +- 1 (odd widths: 3 * w % 4 != 0, the byte-store fallback of the pack)
    ("wide_tma_127x95", 127, 95, GW, {}, "k_render_wide_tma<1,false>"),
    ("wide_tma_129x97", 129, 97, GW, {}, "k_render_wide_tma<1,false>"),
    ("wide_tma_191x161", 191, 161, GW, {}, "k_render_wide_tma<1,false>"),
    ("wide_tma_256x160", 256, 160, GW, {}, "k_render_wide_tma<1,false>"),   # 4-byte aligned rows
    ("wide_tma_bgra", 193, 65, GW, dict(bgra=True), "k_render_wide_tma<1,true>"),
    ("wide_narrow", 64, 150, GW, {}, "k_render_wide_tma<1,false>"),         # narrower than 132: no interior tile, no TMA copy
    ("wide_short", 200, 30, GW, {}, "k_render_wide_tma<1,false>"),          # shorter than 67: no interior tile, no TMA copy
    ("render_0_1", 200, 136, dict(gab=0, epf=1), {}, "k_render<0,1,true>"),
    ("render_0_2", 200, 136, dict(gab=0, epf=2), {}, "k_render<0,2,true>"),
    ("render_0_3", 200, 136, dict(gab=0, epf=3), {}, "k_render<0,3,true>"),
    ("render_1_0", 200, 136, dict(gab=1, epf=0), {}, "k_render<1,0,true>"),
    ("render_1_2", 200, 136, dict(gab=1, epf=2), {}, "k_render<1,2,true>"),
    ("render_1_3", 200, 136, dict(gab=1, epf=3), {}, "k_render<1,3,true>"),
    ("render_1_2_odd", 201, 136, dict(gab=1, epf=2), {}, "k_render<1,2,false>"),
    ("render_alpha", 200, 136, dict(gab=1, epf=1), dict(alpha=True), "k_render<1,1,false>"),
    ("render_orientation6", 200, 136, dict(gab=1, epf=2, orientation=6), dict(orientation=6), "k_render<1,2,false>"),
    ("output_e3", 200, 136, dict(effort=3), {}, "k_output"),
    ("output_no_filters_orientation3", 150, 100, dict(gab=0, epf=0, orientation=3), dict(orientation=3), "k_output"),
    # sample types and colour encodings of test_hdr_and_high_bit_depth_outputs
    ("u16_srgb", 200, 136, dict(effort=7, bits=16), dict(sample="u16"), "k_render<1,1,false>"),
    ("f16_srgb", 200, 136, dict(effort=7, bits=16, exp_bits=5), dict(sample="f16"), "k_render<1,1,false>"),
    ("f32_srgb", 200, 136, dict(effort=7, bits=32, exp_bits=8), dict(sample="f32"), "k_render<1,1,false>"),
    ("f32_linear", 200, 136, dict(effort=7, bits=32, exp_bits=8, tf=8), dict(sample="f32"), "k_render<1,1,false>"),
    ("u16_709", 200, 136, dict(effort=7, bits=16, tf=1), dict(sample="u16"), "k_render<1,1,false>"),
    ("u16_p3", 200, 136, dict(effort=7, bits=16, primaries=11), dict(sample="u16"), "k_render<1,1,false>"),
    ("u16_pq", 200, 136, dict(effort=7, bits=16, primaries=9, tf=16, intensity_target=1000.0), dict(sample="u16"), "k_render<1,1,false>"),
    ("f32_pq", 200, 136, dict(effort=7, bits=32, exp_bits=8, primaries=9, tf=16, intensity_target=1000.0), dict(sample="f32"), "k_render<1,1,false>"),
    ("u16_hlg", 200, 136, dict(effort=7, bits=16, primaries=9, tf=18, intensity_target=1000.0), dict(sample="u16"), "k_render<1,1,false>"),
    ("f16_hlg", 200, 136, dict(effort=7, bits=16, exp_bits=5, primaries=9, tf=18, intensity_target=1000.0), dict(sample="f16"), "k_render<1,1,false>"),
]


@pytest.mark.parametrize("name,w,h,kw,out,branch", RENDER_CASES, ids=[c[0] for c in RENDER_CASES])
def test_rendered_samples_match_float64_colour(gpu, oracle, name, w, h, kw, out, branch):
    kw = dict(kw)
    kw.setdefault("effort", 7)
    gab = kw.get("gab", 1 if kw["effort"] >= 5 else 0)
    epf = kw.get("epf", 1 if kw["effort"] >= 5 else 0)     # the encoder's default at distance 1
    orientation = kw.get("orientation", 1)
    assert render_branch(gab, epf, w, h, **out) == branch
    data, _ = _encode(oracle, w, h, channels=4 if out.get("alpha") else 3, **kw)
    d = oracle.decode(data, threads=4, keep_stages=True)
    idct, gabp, epfp = (_oracle_planes(d, n) for n in ("idct", "gab", "epf"))
    assert np.array_equal(gabp, idct) == (gab == 0) and np.array_equal(epfp, gabp) == (epf == 0)   # the file carries the filters under test
    real = xyb_to_output(epfp[:, :h, :w], kw.get("primaries", 1), kw.get("tf", TF_SRGB), kw.get("intensity_target", 255.0))
    real = orient(real, orientation)
    if out.get("bgra"):
        got = gpu.load_image_bgra(data)
        assert np.all(got[..., 3] == 255)
        got = got[..., 2::-1]
    else:
        image = gpu.DecoderImage()
        gpu.JpegXLNative.LoadImage(data, image)
        got = image.layer_data.color
    assert got.shape == real.shape
    sample = out.get("sample", "u8")
    g = got.astype(np.float64)
    if sample in ("u8", "u16"):
        scale = 255.0 if sample == "u8" else 65535.0
        ref = np.clip(real, 0, 1) * scale
        excess = np.abs(g - ref) - 0.5
        if kw.get("tf") == TF_PQ:
            excess = excess[_pq_dark_in_linear_light(g / scale, np.clip(real, 0, 1))]
        assert float(excess.max()) <= (U8_DELTA if sample == "u8" else U16_DELTA), "worst |got - real| = 0.5 + %.4g code units" % float(excess.max())
    else:
        if sample == "f16":
            half_ulp = 0.5 * np.spacing(np.abs(real).astype(np.float16)).astype(np.float64)
            rel = (np.abs(g - real) - half_ulp) / np.maximum(np.abs(real), 1e-3)
            bound = F16_REL
        else:
            rel = np.abs(g - real) / np.maximum(np.abs(real), 1e-3)
            bound = F32_REL
        if kw.get("tf") == TF_PQ:
            rel = rel[_pq_dark_in_linear_light(g, real)]
        assert float(rel.max()) <= bound, "worst relative difference %.4g" % float(rel.max())
