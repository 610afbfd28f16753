"""-m gpu stage tests of the VarDCT encoder (dev/encode_kernels.cu behind SaveImage): every device stage of a band session
(JxlB200BandEncoderDebugStage) against a float64 restatement (tests/enc_reference.py), and the written file against those stages.

A round trip through a decoder catches syntax errors but not an arithmetic error that still gives a valid file (a wrong opsin constant,
dead zone, bias or CfL factor costs a few percent of quality or size). Here each stage is compared with the GPU's own output of the stage
before it as input, so that a failure names one kernel:
  * XYB planes (k_enc_to_xyb, stage 0) and the inverse gaborish (stage 1): fp32 level, relative to each channel's range;
  * block statistics (k_enc_block_stats, stage 2): fp32 level; the hf_mul and CfL maps (k_enc_tile_params, stages 3-4): exact;
  * LF (stage 5): fp32 level; quantised LF and AC coefficients (stages 6-7): exact; non-zero counts (stage 8): exact;
  * the file: the oracle decodes exactly the coefficients, LF integers and HF maps the device produced;
  * the token histograms: exactly the device's tokens plus the HF metadata the host adds.
Integer decisions are exact except where the float64 value before rounding lies within an fp32 error bound (delta) of a decision
boundary; there one step of difference is allowed, and such ambiguous values must stay below 1e-3 of the values compared. Each float bound
sits at about 4x the worst value measured on a B200 (1000 W) and is checked against what it means: a fraction of the channel range for
planes, a fraction of the quantisation step for coefficients."""
import numpy as np
import pytest

import enc_reference as R
import icc_util

pytestmark = pytest.mark.gpu

EPS = R.FP32_EPS
NUM_AC_CTX = 495 * 15
ALPHABET = 128
AMBIGUOUS_MAX = 1e-3      # of the compared values

# Relative to each channel's range (max |reference|), about 4x the worst case measured on a B200 (1000 W). One 8-bit LSB is at least 1.3e-3
# of the range in the XYB planes (test_gpu_stages.py, lsb_in_xyb), more than 60x every bound here.
# XYB: X = (g0 - g1) / 2 and Y = (g0 + g1) / 2 come from the same two fp32 cube roots, so X is measured against the range of Y, the size of its
# terms (its own range is ~1/25 of that on the synthetic image and 0 on a gray one, where the device's X is a few 1e-8 of rounding).
XYB_REL_BOUND = 1e-6      # measured 2.5e-7 (Y and B of the gray 200 x 136 surface; X at most 6.2e-8 on that scale)
GAB_REL_BOUND = 6e-7      # measured 1.35e-7 (Y, 2100 x 300): two fp32 Van Cittert steps
STATS_REL_BOUND = 2.5e-6  # measured 6.4e-7 (sum X*Y, synthetic 531 x 277); relative to the largest value of the statistic over the frame
LF_REL_BOUND = 6e-7       # measured 1.56e-7 (Y, 777 x 555): LF is coefficient 0 of the fp32 DCT


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


def _geometry(w, h):
    xb, yb = -(-w // 8), -(-h // 8)
    return xb, yb, -(-xb // 8), -(-yb // 8), -(-xb // 32), -(-yb // 32)


class Run:
    """One whole-frame band session stopped between tokenize() and finish(): its stages, and on demand the file it writes."""

    def __init__(self, gpu, surface, opts, icc=None):
        self.gpu, self.surface, self.opts, self.icc = gpu, surface, opts, icc
        h, w, _ = surface.shape
        self.w, self.h = w, h
        meta = gpu.EncoderImageMetadata(icc=icc) if icc else None
        self.enc = gpu.BandEncoder(surface, h, 0, 0, 0, opts, metadata=meta)
        self.flags = self.enc.flags
        self.hist = self.enc.tokenize(self.flags)
        self._stages = {}

    def stage(self, which):
        if which not in self._stages:
            self._stages[which] = self.enc.debug_stage(which)
        return self._stages[which]

    def file(self):
        blob = self.enc.finish(self.hist)
        self.enc.close()
        meta = self.gpu.EncoderImageMetadata(icc=self.icc) if self.icc else None
        return self.gpu.assemble_bands(self.w, self.h, self.opts, self.flags, self.hist, [blob], meta)


def _cells(coeffs, w, h):
    """GPU coefficients [group][3][1024 cells][64] -> [3][yb][xb][64]; also the largest |value| in cells outside the image."""
    xb, yb, _, _, xg, yg = _geometry(w, h)
    q = coeffs.astype(np.int64).reshape(xg * yg, 3, 32, 32, 64)
    out = np.zeros((3, yb, xb, 64), np.int64)
    outside = 0
    for g in range(xg * yg):
        gy, gx = divmod(g, xg)
        ch, cw = min(32, yb - 32 * gy), min(32, xb - 32 * gx)
        out[:, 32 * gy:32 * gy + ch, 32 * gx:32 * gx + cw] = q[g, :, :ch, :cw]
        outside = max(outside, int(np.abs(q[g, :, ch:]).max(initial=0)), int(np.abs(q[g, :, :ch, cw:]).max(initial=0)))
    return out, outside


def _rel_err(got, ref, scale=None):
    """Per channel: max |got - ref| / max |ref| (or / scale[channel])."""
    got, ref = got.reshape(got.shape[0], -1).astype(np.float64), ref.reshape(ref.shape[0], -1)
    den = np.abs(ref).max(axis=1) if scale is None else np.asarray(scale, np.float64)
    return np.abs(got - ref).max(axis=1) / np.maximum(den, 1e-30)


def _check_decisions(name, got, ref, amb, step=1):
    """Exact except at ambiguous values, where got may differ from ref by one step; reports and bounds the ambiguous count."""
    got, ref, amb = np.asarray(got), np.asarray(ref), np.asarray(amb)
    bad = (got != ref) & ~amb
    idx = np.argwhere(bad)
    assert not bad.any(), "%s: %d of %d differ outside the ambiguous set, first at %s: GPU %s, reference %s" % (
        name, int(bad.sum()), got.size, tuple(idx[0]), got[tuple(idx[0])], ref[tuple(idx[0])])
    off = np.abs(got.astype(np.int64) - ref.astype(np.int64))
    assert int(off.max(initial=0)) <= step, "%s: an ambiguous value differs by %d" % (name, int(off.max()))
    n_amb = int(amb.sum())
    print("%s: %d compared, %d ambiguous, %d of them differ" % (name, got.size, n_amb, int((got != ref).sum())))
    assert n_amb <= AMBIGUOUS_MAX * got.size, "%s: %d of %d values are ambiguous" % (name, n_amb, got.size)


def _quantiser(run, d):
    """(inv_gs, quant_lf, xm, bm, base hf_mul) of the file the session writes; d: its oracle decode."""
    inv_gs = 65536.0 / d.global_scale
    q_ac = np.float32(0.79) / np.float32(max(run.opts.distance, 0.01))
    base = int(np.rint(np.float32(q_ac * np.float32(65536.0)) / np.float32(d.global_scale)))
    return inv_gs, d.quant_lf, 0.8 ** (d.x_qm_scale - 2), 0.8 ** (d.b_qm_scale - 2), max(1, min(255, base))


def _dequant_table(oracle):
    dq = np.zeros(3 * 64, np.float32)
    oracle.lib().jxlo_dequant_table(0, dq.ctypes.data)
    return dq.astype(np.float64)


def _stage1_blocks(run, channel):
    """Float64 DCT8 of the GPU's stage-1 plane (the frame's own rows) of one channel, and the bound on each coefficient's magnitude terms."""
    xb, yb = _geometry(run.w, run.h)[:2]
    p = run.stage(1)[channel, :8 * yb].astype(np.float64)
    return R.dct8_blocks(p), R.dct8_blocks(p, absolute=True)


# ------------------------------------------------------------------------------------------------ images
def _synthetic(oracle, w, h, seed=None, channels=3):
    return _bgra(oracle.synthetic_image(w, h, seed=w + h if seed is None else seed, channels=channels))


def _all_levels():
    """Every level of each channel alone and of gray, then 4096 random colours: 256 x 20 pixels."""
    rng = np.random.default_rng(7)
    rows = []
    for c in range(3):
        r = np.zeros((256, 3), np.uint8)
        r[:, c] = np.arange(256)
        rows.append(r)
    rows.append(np.repeat(np.arange(256, dtype=np.uint8)[:, None], 3, axis=1))
    rgb = np.concatenate(rows + [rng.integers(0, 256, (4096, 3), dtype=np.uint8)]).reshape(20, 256, 3)
    return _bgra(rgb)


def _flat(w, h):
    return _bgra(np.full((h, w, 3), (90, 160, 210), np.uint8))


def _noise(w, h):
    return _bgra(np.random.default_rng(9).integers(0, 256, (h, w, 3), dtype=np.uint8))


def _blue_texture(w, h):
    """Random blue on a mid-gray red / green: B varies about 2.3x as much as Y with it, so 84 * (sum BY / sum YY - 1) passes 127."""
    rgb = np.full((h, w, 3), 128, np.uint8)
    rgb[..., 2] = np.random.default_rng(11).integers(0, 256, (h, w), dtype=np.uint8)
    return _bgra(rgb)


# ------------------------------------------------------------------------------------------------ 1. XYB planes (stage 0)
XYB_CASES = [("531x277", lambda o: _synthetic(o, 531, 277), 7, None),
             ("531x277_e3", lambda o: _synthetic(o, 531, 277), 3, None),          # no gaborish: stage 0 is the buffer the DCT reads
             ("9x7", lambda o: _synthetic(o, 9, 7), 7, None),                     # a single partial block
             ("all_levels", lambda o: _all_levels(), 7, None),
             ("gray", lambda o: _synthetic(o, 200, 136, channels=1), 7, None),
             ("rgba", lambda o: _synthetic(o, 200, 136, channels=4), 7, None)] + [
             ("icc_" + c, lambda o: (_synthetic(o, 200, 136, seed=25).astype(np.float64) * 0.8 + 25).astype(np.uint8), 7, c)
             for c in ("para", "curv1", "table")]


@pytest.mark.parametrize("name,make,effort,curve", XYB_CASES, ids=[c[0] for c in XYB_CASES])
def test_xyb_planes_match_float64(gpu, oracle, name, make, effort, curve):
    surface = make(oracle)
    if name.startswith("icc"):
        surface[..., 3] = 255
    icc = icc_util.make_matrix_icc(icc_util.P3_PRIMS, gamma=2.2, curve=curve) if curve else None
    run = Run(gpu, surface, gpu.EncoderOptions(quality=90, effort=effort), icc=icc)
    h, w, _ = surface.shape
    got = run.stage(0)
    xb, yb = _geometry(w, h)[:2]
    assert got.shape == (3, 8 * yb, 8 * xb)
    gray = name == "gray"
    assert (run.flags & 1) == (0 if gray else 1)
    ref = R.bgra_to_xyb(R.extend(surface, 8 * yb, 8 * xb), gray=gray, icc=icc)
    yrange, brange = np.abs(ref[1]).max(), np.abs(ref[2]).max()
    err = _rel_err(got, ref, scale=(yrange, yrange, brange))
    print("%s: XYB relative error %s" % (name, err))
    assert np.all(err <= XYB_REL_BOUND), "XYB differs by %s of the channel range" % err
    if name == "rgba":   # alpha is coded losslessly next to the XYB planes
        d = oracle.decode(run.file())
        assert d.has_alpha and np.array_equal(d.pixels[..., 3], surface[..., 3])


# ------------------------------------------------------------------------------------------------ 2. inverse gaborish (stage 1)
@pytest.mark.parametrize("w,h", [(531, 277), (203, 141), (8, 8), (2100, 300)])
def test_inverse_gaborish_matches_float64(gpu, oracle, w, h):
    run = Run(gpu, _synthetic(oracle, w, h), gpu.EncoderOptions(quality=90, effort=7))
    s0, s1 = run.stage(0).astype(np.float64), run.stage(1)
    ref = R.inverse_gaborish(s0)             # mirrored at the extent of the planes (xpad x ext_rows), as the kernel does
    err = _rel_err(s1, ref)
    print("%dx%d: inverse gaborish relative error %s" % (w, h, err))
    assert np.all(err <= GAB_REL_BOUND), "inverse gaborish differs by %s of the channel range" % err
    assert np.abs(s1 - s0).max() > 1e-3                                    # it did something
    # what the decoder's filter makes of it, inside the image (recorded, not bounded tightly: the encoder's inverse is approximate)
    res = np.abs(R.gaborish(s1.astype(np.float64)) - s0)[:, :h, :w] / np.abs(s0).max(axis=(1, 2))[:, None, None]
    parts = {"interior": res[:, 1:-1, 1:-1], "first row": res[:, 0], "last row": res[:, -1], "first column": res[:, :, 0], "last column": res[:, :, -1]}
    print("%dx%d: |G(stage 1) - stage 0| / range: %s" % (w, h, ", ".join("%s %.3g" % (k, v.max()) for k, v in parts.items() if v.size)))
    assert res.max() < 0.25     # measured 0.05 (interior, 531 x 277); the inverse is approximate, this only catches a broken one


def test_band_planes_equal_the_whole_frame(gpu, oracle):
    """A band's stage 0 (with its 8 halo rows) is the whole frame's, bit for bit; stage 1 is too on the band's own rows (the halo rows are
    mirrored at the band's edge and discarded)."""
    w, h = 300, 2300
    surface = _synthetic(oracle, w, h, seed=3)
    opts = gpu.EncoderOptions(quality=90, effort=7)
    whole = Run(gpu, surface, opts)
    band = gpu.BandEncoder(surface[2040:], h, 2048, 8, 0, opts)
    band.tokenize(whole.flags | band.flags)
    b0, b1 = band.debug_stage(0), band.debug_stage(1)
    band.close()
    w0, w1 = whole.stage(0), whole.stage(1)
    assert b0.shape == (3, 8 + 256, 8 * 38) and np.array_equal(b0, w0[:, 2040:])
    assert np.array_equal(b1[:, 8:], w1[:, 2048:])


# ------------------------------------------------------------------------------------------------ 3. block statistics and tile parameters (stages 2-4)
QUALITIES = {0.5: 95, 1: 90, 3: 68, 10: 13}     # quality -> distance 0.55, 1.0, 2.98, 9.98
PARAM_CASES = [("synthetic_d%s" % d, lambda o: _synthetic(o, 531, 277), q) for d, q in QUALITIES.items()] + [
    ("flat", lambda o: _flat(200, 136), 90), ("noise", lambda o: _noise(200, 136), 90), ("blue_texture", lambda o: _blue_texture(200, 136), 90)]


@pytest.mark.parametrize("name,make,quality", PARAM_CASES, ids=[c[0] for c in PARAM_CASES])
def test_block_statistics_and_tile_parameters(gpu, oracle, name, make, quality):
    surface = make(oracle)
    h, w, _ = surface.shape
    xb, yb, xt, yt, _, _ = _geometry(w, h)
    run = Run(gpu, surface, gpu.EncoderOptions(quality=quality, effort=7))
    stats, hfm, cfl = run.stage(2).astype(np.float64), run.stage(3), run.stage(4)
    assert stats.shape == (yb, xb, 4) and hfm.shape == (yb, xb) and cfl.shape == (2, yt, xt)
    # statistics from a float64 DCT of the GPU's stage 1
    Sx, Sy, Sb = (_stage1_blocks(run, c)[0][..., 1:] for c in range(3))
    ref = np.stack([np.abs(Sy).sum(-1), (Sx * Sy).sum(-1), (Sb * Sy).sum(-1), (Sy * Sy).sum(-1)], axis=-1)
    if name != "flat":   # nothing to measure against on a flat surface; the maps below are exact there
        err = _rel_err(np.moveaxis(stats, -1, 0), np.moveaxis(ref, -1, 0))
        print("%s: block statistics relative error %s" % (name, err))
        assert np.all(err <= STATS_REL_BOUND), "block statistics differ by %s of their range" % err
    # hf_mul from the GPU's activity
    d = oracle.decode(run.file(), keep_stages=True)
    base = _quantiser(run, d)[4]
    want, mulq = R.aq_hf_mul(stats[..., 0], base)
    # __powf: a few ulp plus the exp2 error of y * log2(x); the activity is an fp32 sum of 63 magnitudes
    d_mulq = mulq * (64 * EPS * 0.2 + (4 + 1.173 * np.abs(0.2 * np.log2(R.AQ_REF / (stats[..., 0] + 1e-4)))) * 2 * EPS + 2 ** -22)
    amb = np.zeros(mulq.shape, bool)
    for t in R.AQ_THRESHOLDS:
        amb |= np.abs(mulq - t) < d_mulq
    _check_decisions(name + " hf_mul", hfm, want, amb, step=int(np.ceil(base * 0.2)) + 1)
    # ytox / ytob from the GPU's statistics, summed per tile
    fx, fb, rx, rb, syy = R.cfl_factors(stats, yt, xt)
    pad = np.zeros((yt * 8, xt * 8, 4))
    pad[:yb, :xb] = np.abs(stats)
    asum = pad.reshape(yt, 8, xt, 8, 4).sum(axis=(1, 3))
    den = np.where(syy > 0, syy, 1.0)
    dx = R.COLOR_FACTOR * 16 * EPS * (asum[..., 1] + np.abs(rx / R.COLOR_FACTOR) * asum[..., 3]) / den + np.abs(rx) * 4 * EPS
    db = R.COLOR_FACTOR * 16 * EPS * (asum[..., 2] + np.abs(rb / R.COLOR_FACTOR + 1) * asum[..., 3]) / den + np.abs(rb) * 4 * EPS
    edge = np.abs(syy - 1e-12) < 16 * EPS * asum[..., 3] + 1e-18
    _check_decisions(name + " ytox", cfl[0], fx, R.ambiguous_rounding(rx, dx) | edge)
    _check_decisions(name + " ytob", cfl[1], fb, R.ambiguous_rounding(rb, db) | edge)
    # the maps the file carries are the device's
    assert np.array_equal(d.stages["hf_mul"], hfm) and np.array_equal(d.stages["ytox"], cfl[0]) and np.array_equal(d.stages["ytob"], cfl[1])
    if name == "flat":
        assert np.all(hfm == min(255, int(np.rint(base * 1.35)))) and not cfl.any()
    if name == "noise":
        assert np.all(hfm == int(np.rint(base * 0.75)))
    if name == "blue_texture":
        assert np.all(cfl[1] == 127)


# ------------------------------------------------------------------------------------------------ 4. quantisation (stages 5-8)
QUANT_CASES = [("531x277_e7_d%s" % d, 531, 277, 7, q) for d, q in QUALITIES.items()] + [
    ("531x277_e3_d1", 531, 277, 3, 90), ("531x277_e3_d10", 531, 277, 3, 13),
    ("777x555_e7_d3", 777, 555, 7, 68), ("777x555_e3_d1", 777, 555, 3, 90),    # 4 x 3 groups, the last ones partial
    ("9x7_e7_d1", 9, 7, 7, 90), ("9x7_e3_d1", 9, 7, 3, 90)]


@pytest.mark.parametrize("name,w,h,effort,quality", QUANT_CASES, ids=[c[0] for c in QUANT_CASES])
def test_quantisation_matches_float64(gpu, oracle, dequant, name, w, h, effort, quality):
    xb, yb, xt, yt, _, _ = _geometry(w, h)
    run = Run(gpu, _synthetic(oracle, w, h), gpu.EncoderOptions(quality=quality, effort=effort))
    lf, lfq, coeffs, nz = run.stage(5).astype(np.float64), run.stage(6), run.stage(7), run.stage(8)
    q, outside = _cells(coeffs, w, h)
    if effort >= 5:
        hfm, cfl = run.stage(3), run.stage(4).astype(np.float64)
    S = [_stage1_blocks(run, c) for c in range(3)]
    d = oracle.decode(run.file(), keep_stages=True)
    inv_gs, quant_lf, xm, bm, base = _quantiser(run, d)
    if effort < 5:
        hfm, cfl = np.full((yb, xb), base), np.zeros((2, yt, xt))
    # LF: coefficient 0 of each block
    err = _rel_err(lf, np.stack([s[0][..., 0] for s in S]))
    print("%s: LF relative error %s" % (name, err))
    assert np.all(err <= LF_REL_BOUND), "LF differs by %s of the channel range" % err
    # quantised LF from the GPU's LF: Y, then X and B against the GPU's dequantised Y (LF chroma-from-luma: kx = 0, kb = 1)
    fac = [R.LF_DEQUANT[c] * inv_gs / quant_lf for c in range(3)]
    ydq = lfq[0] * fac[1]
    pre = [lf[1] / fac[1], lf[0] / fac[0], (lf[2] - ydq) / fac[2]]
    dl = [np.abs(pre[0]) * 8 * EPS, np.abs(pre[1]) * 8 * EPS, (np.abs(lf[2]) + np.abs(ydq)) / fac[2] * 8 * EPS]
    for k, nm in enumerate("YXB"):
        _check_decisions("%s LF %s" % (name, nm), lfq[k], np.rint(pre[k]).astype(np.int64), R.ambiguous_rounding(pre[k], dl[k]))
    # AC: Y first, X and B against the GPU's Y integers dequantised with the spec's bias rule and the GPU's per-tile factors
    step = R.ac_steps(dequant, inv_gs, hfm, xm, bm)
    tile = cfl[:, np.arange(yb) // 8][:, :, np.arange(xb) // 8]
    kc = {0: tile[0] / R.COLOR_FACTOR, 2: 1.0 + tile[1] / R.COLOR_FACTOR}
    ydq = R.dequant_bias(q[1], 1) * step[1]
    for c, nm in ((1, "Y"), (0, "X"), (2, "B")):
        coef, mag = S[c]
        v, vmag = coef, mag * 32 * EPS
        if c != 1:
            v = coef - kc[c][..., None] * ydq
            vmag = vmag + np.abs(kc[c][..., None] * ydq) * 4 * EPS
        qf = v / step[c]
        want = R.quantise(qf)
        amb = R.ambiguous_rounding(qf, vmag / step[c] + np.abs(qf) * 8 * EPS, dead_zone=True)
        want[..., 0], amb[..., 0] = 0, False          # position 0 is the LF, coded separately
        _check_decisions("%s AC %s" % (name, nm), q[c], want, amb)
    assert outside == 0, "non-zero coefficients in cells outside the image"
    assert np.array_equal(nz, np.count_nonzero(q[..., 1:], axis=-1).astype(np.uint8))
    assert np.count_nonzero(q) > 0


@pytest.fixture(scope="module")
def dequant(oracle):
    return _dequant_table(oracle)


# ------------------------------------------------------------------------------------------------ 5. the file carries the device's decisions
FILE_CASES = [("e1_prefix", 531, 277, 1), ("e3", 531, 277, 3), ("e5", 531, 277, 5), ("e7", 777, 555, 7)]


def _check_file(d, q, lfq, hfm, cfl):
    yb, xb = hfm.shape
    assert np.array_equal(d.stages["coeffs"].reshape(3, yb, xb, 64), q)
    assert np.array_equal(d.stages["lfq"], lfq[[1, 0, 2]])      # stream order Y, X, B -> channel order X, Y, B
    assert np.array_equal(d.stages["hf_mul"], hfm)
    assert np.array_equal(d.stages["ytox"], cfl[0]) and np.array_equal(d.stages["ytob"], cfl[1])


@pytest.mark.parametrize("name,w,h,effort", FILE_CASES, ids=[c[0] for c in FILE_CASES])
def test_file_carries_the_device_decisions(gpu, oracle, name, w, h, effort):
    xb, yb, xt, yt, _, _ = _geometry(w, h)
    run = Run(gpu, _synthetic(oracle, w, h), gpu.EncoderOptions(quality=90, effort=effort))
    q, _ = _cells(run.stage(7), w, h)
    lfq = run.stage(6)
    hfm, cfl = (run.stage(3), run.stage(4)) if effort >= 5 else (None, np.zeros((2, yt, xt), np.int8))
    d = oracle.decode(run.file(), keep_stages=True)
    if hfm is None:
        hfm = np.full((yb, xb), _quantiser(run, d)[4])
        assert np.all(d.stages["hf_mul"] == hfm[0, 0])          # a constant map below effort 5
    _check_file(d, q, lfq, hfm, cfl)


def test_two_band_file_carries_the_device_decisions(gpu, oracle):
    w, h = 300, 2300
    surface = _synthetic(oracle, w, h, seed=4)
    opts = gpu.EncoderOptions(quality=75, effort=7)
    bands = [gpu.BandEncoder(surface[:2056], h, 0, 0, 8, opts), gpu.BandEncoder(surface[2040:], h, 2048, 8, 0, opts)]
    flags = bands[0].flags | bands[1].flags
    hist = np.sum([b.tokenize(flags) for b in bands], axis=0, dtype=np.uint64)
    parts = []
    for b, rows in zip(bands, (2048, h - 2048)):
        q, _ = _cells(b.debug_stage(7), w, rows)
        parts.append((q, b.debug_stage(6), b.debug_stage(3), b.debug_stage(4)))
    blobs = [b.finish(hist) for b in bands]
    for b in bands:
        b.close()
    data = gpu.assemble_bands(w, h, opts, flags, hist, blobs)
    assert data == gpu.encode_to_memory(surface, opts)
    d = oracle.decode(data, keep_stages=True)
    _check_file(d, *(np.concatenate([p[k] for p in parts], axis=axis) for k, axis in enumerate((1, 1, 0, 1))))   # along the block / tile rows


# ------------------------------------------------------------------------------------------------ 6. histograms
@pytest.mark.parametrize("w,h,effort", [(531, 277, 1), (2100, 300, 7)])
def test_histograms_count_the_device_tokens(gpu, oracle, w, h, effort):
    run = Run(gpu, _synthetic(oracle, w, h), gpu.EncoderOptions(quality=90, effort=effort))
    counts, tokens, n_mod = run.stage(9)
    nleaves = run.hist.size // ALPHABET - NUM_AC_CTX
    assert run.hist.size == (nleaves + NUM_AC_CTX) * ALPHABET
    key = (tokens[:, 0] & 0xffff).astype(np.int64) * ALPHABET + ((tokens[:, 0] >> 16) & 0xff)
    n_mod_tokens = int(counts[:n_mod].sum())
    assert len(counts) == n_mod + _geometry(w, h)[4] * _geometry(w, h)[5]
    ac = np.bincount(key[n_mod_tokens:], minlength=NUM_AC_CTX * ALPHABET)
    assert ac.size == NUM_AC_CTX * ALPHABET, "an AC token has a context outside the AC contexts"
    assert np.array_equal(run.hist[nleaves * ALPHABET:], ac.astype(np.uint64))
    mod = np.bincount(key[:n_mod_tokens], minlength=nleaves * ALPHABET)
    assert mod.size == nleaves * ALPHABET, "a Modular token has a context outside the tree's leaves"
    extra = run.hist[:nleaves * ALPHABET].astype(np.int64) - mod
    assert extra.min() >= 0
    xb, yb = _geometry(w, h)[:2]
    samples = 0
    for gy in range(-(-yb // 256)):
        for gx in range(-(-xb // 256)):
            bw, bh = min(256, xb - 256 * gx), min(256, yb - 256 * gy)
            tw, th, nb = -(-bw // 8), -(-bh // 8), bw * bh
            samples += 2 * tw * th + 2 * nb + nb      # ytox, ytob; block info (strategy, hf_mul); EPF sharpness
    assert int(extra.sum()) == samples


def test_stage_dumps_exist_only_between_tokenize_and_finish(gpu, oracle):
    surface = _synthetic(oracle, 64, 48)
    enc = gpu.BandEncoder(surface, 48, 0, 0, 0, gpu.EncoderOptions(quality=90, effort=3))
    with pytest.raises(gpu.FormatException, match="between Tokenize and Finish"):
        enc.debug_stage(1)
    hist = enc.tokenize(enc.flags)
    assert enc.debug_stage(1).shape == (3, 48, 64)
    with pytest.raises(gpu.FormatException, match="effort 5"):
        enc.debug_stage(3)
    enc.finish(hist)
    with pytest.raises(gpu.FormatException, match="between Tokenize and Finish"):
        enc.debug_stage(9)
    enc.close()
