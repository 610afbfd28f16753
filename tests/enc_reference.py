"""Float64 restatement of the VarDCT encoder's arithmetic (dev/encode_kernels.cu), vectorised over all samples / blocks, for the encoder
stage tests. Nothing here imports the engine: the colour constants and quantiser rules come from the specification (SURVEY.md A.8 - A.10),
ICC curves and colorants are read with tests/icc_util.py, and the DCT8 dequantisation table and natural order are the oracle's.

Layouts follow JxlB200BandEncoderDebugStage: planes [3 (X, Y, B)][rows][columns], blocks [yb][xb], DCT coefficients of a block in the
storage layout of square blocks, S[hf * 8 + vf] (S[0] is the LF sample)."""
import struct

import numpy as np

import icc_util

# ---------------------------------------------------------------------------------------------------------------- colour (SURVEY A.10)
OPSIN_ABSORBANCE = np.array([[0.30, 0.622, 0.078],
                             [0.23, 0.692, 0.078],
                             [0.24342268924547819, 0.20476744424496821, 0.55180986650955360]])
OPSIN_BIAS = 0.0037930732552754493


def srgb_to_linear(v8):
    """IEC 61966-2-1 decoding of 8-bit samples, in float64."""
    v = np.asarray(v8, np.float64) / 255.0
    return np.where(v <= 0.04045, v / 12.92, ((v + 0.055) / 1.055) ** 2.4)


def linear_to_xyb(lin):
    """lin: [..., 3] linear sRGB -> [3][...] X, Y, B."""
    mix = lin @ OPSIN_ABSORBANCE.T + OPSIN_BIAS
    g = np.cbrt(np.maximum(mix, 0.0)) - np.cbrt(OPSIN_BIAS)
    g = np.moveaxis(g, -1, 0)
    return np.stack([0.5 * (g[0] - g[1]), 0.5 * (g[0] + g[1]), g[2]])


def icc_curve(tag):
    """A TRC tag ('para' types 0-4, 'curv' identity / gamma / table) as a float64 function on [0, 1]."""
    if tag[:4] == b"para":
        t, p = icc_util.para_of(tag)
        g = p[0]
        if t == 0:
            return lambda x: x ** g
        a, b = p[1], p[2]
        if t == 1:
            return lambda x: np.where(x >= -b / a, np.maximum(a * x + b, 0) ** g, 0.0)
        if t == 2:
            c = p[3]
            return lambda x: np.where(x >= -b / a, np.maximum(a * x + b, 0) ** g + c, c)
        c, d = p[3], p[4]
        e, f = (p[5], p[6]) if t == 4 else (0.0, 0.0)
        return lambda x: np.where(x >= d, np.maximum(a * x + b, 0) ** g + e, c * x + f)
    assert tag[:4] == b"curv"
    n = struct.unpack(">I", tag[8:12])[0]
    if n == 0:
        return lambda x: x
    if n == 1:
        g = struct.unpack(">H", tag[12:14])[0] / 256.0
        return lambda x: x ** g
    table = np.array(struct.unpack(">%dH" % n, tag[12:12 + 2 * n]), np.float64) / 65535.0
    return lambda x: np.interp(x * (n - 1), np.arange(n), table)


def icc_to_linear_srgb(icc):
    """(3 tone curves, 3x3 matrix profile RGB (linear) -> linear sRGB) of a matrix/TRC profile: the D50 colorants, adapted to sRGB's
    D65 white through Bradford."""
    tags = icc_util.parse_icc(icc)["tags"]
    curves = [icc_curve(tags[s]) for s in (b"rTRC", b"gTRC", b"bTRC")]
    colorants = np.stack([icc_util.xyz_of(tags[s]) for s in (b"rXYZ", b"gXYZ", b"bXYZ")], axis=1)
    srgb_d50 = icc_util.adapt_to_d50(0.3127, 0.3290) @ icc_util.rgb_to_xyz(icc_util.SRGB_PRIMS, 0.3127, 0.3290)
    return curves, np.linalg.solve(srgb_d50, colorants)


def bgra_to_xyb(bgra, gray=False, icc=None):
    """bgra: [rows][cols][4] u8 -> [3][rows][cols] float64 XYB. Gray frames take the B channel for all three; an ICC source maps its
    samples through its own curves and colorants."""
    b, g, r = (bgra[..., k] for k in range(3))
    if icc is not None:
        curves, m = icc_to_linear_srgb(icc)
        lin = np.stack([curves[k](v / 255.0) for k, v in enumerate((r, g, b))], axis=-1) @ m.T
    elif gray:
        lin = np.repeat(srgb_to_linear(b)[..., None], 3, axis=-1)
    else:
        lin = np.stack([srgb_to_linear(r), srgb_to_linear(g), srgb_to_linear(b)], axis=-1)
    return linear_to_xyb(lin)


def extend(a, rows, cols):
    """Repeats the last row and column of a [rows0][cols0][...] array out to [rows][cols][...] (the encoder's padding)."""
    return a[np.minimum(np.arange(rows), a.shape[0] - 1)][:, np.minimum(np.arange(cols), a.shape[1] - 1)]


# ---------------------------------------------------------------------------------------------------------------- gaborish (SURVEY A.10)
GAB_W1, GAB_W2 = 1.1 * 0.104699568, 1.1 * 0.055680538      # the default weights, the same for the three channels


def gaborish(planes):
    """The decoder's 3x3 gaborish over the whole extent of [3][h][w] planes, edges mirrored (x[-1] = x[0], x[n] = x[n - 1])."""
    _, h, w = planes.shape
    p = np.pad(planes, ((0, 0), (1, 1), (1, 1)), mode="symmetric")

    def at(dy, dx):
        return p[:, 1 + dy:1 + dy + h, 1 + dx:1 + dx + w]
    edge = at(-1, 0) + at(1, 0) + at(0, -1) + at(0, 1)
    corner = at(-1, -1) + at(-1, 1) + at(1, -1) + at(1, 1)
    return (at(0, 0) + GAB_W1 * edge + GAB_W2 * corner) / (1 + 4 * GAB_W1 + 4 * GAB_W2)


def inverse_gaborish(planes, steps=2):
    """Van Cittert iterations x <- x + (orig - G(x)), starting from x = orig: an approximate inverse of the decoder's gaborish."""
    cur = planes.copy()
    for _ in range(steps):
        cur = cur + (planes - gaborish(cur))
    return cur


# ---------------------------------------------------------------------------------------------------------------- DCT8 (SURVEY A.9)
def dct_matrix(n=8):
    """Textbook DCT-II scaled by 1/n (the DC coefficient is the mean): F = D @ x @ D.T."""
    k, i = np.meshgrid(np.arange(n), np.arange(n), indexing="ij")
    return np.cos((2 * i + 1) * k * np.pi / (2 * n)) * np.where(k == 0, 1.0, np.sqrt(2.0)) / n


def dct8_blocks(plane, absolute=False):
    """[8 yb][8 xb] -> [yb][xb][64] in the storage layout S[hf * 8 + vf]. absolute=True transforms |x| with |D|: the sum of the magnitudes of
    the terms of each coefficient, which bounds its fp32 rounding error."""
    h, w = plane.shape
    D = dct_matrix()
    if absolute:
        D, plane = np.abs(D), np.abs(plane)
    blocks = plane.reshape(h // 8, 8, w // 8, 8).transpose(0, 2, 1, 3)       # [yb][xb][y][x]
    F = np.einsum("vy,abyx,hx->abhv", D, blocks, D)                           # F[hf][vf]
    return F.reshape(h // 8, w // 8, 64)


# ---------------------------------------------------------------------------------------------------------------- quantiser (SURVEY A.8)
QUANT_BIAS = (1 - 0.05465007330715401, 1 - 0.07005449891748593, 1 - 0.049935103337343655, 0.145)
LF_DEQUANT = (1.0 / 4096, 1.0 / 512, 1.0 / 256)     # the default LfChannelDequantization, X, Y, B
COLOR_FACTOR = 84                                   # default colour_factor of the chroma-from-luma factors
DEAD_ZONE = 0.56                                    # |v / step| below this quantises to 0


def quantise(qf):
    """Nearest integer (ties to even), 0 inside the dead zone, clamped to int16."""
    q = np.where(np.abs(qf) >= DEAD_ZONE, np.rint(qf), 0.0)
    return np.clip(q, -32768, 32767).astype(np.int64)


def dequant_bias(q, c):
    """The decoder's biased reconstruction of a quantised AC coefficient of channel c, in units of the step."""
    qd = q.astype(np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        far = qd - QUANT_BIAS[3] / qd
    return np.where(q == 0, 0.0, np.where(np.abs(q) == 1, np.sign(qd) * QUANT_BIAS[c], far))


def ambiguous_rounding(x, delta, dead_zone=False):
    """True where rounding x to an integer could go either way given an error of up to delta: x lies within delta of k + 1/2 (or of the
    dead zone's edge)."""
    frac = np.abs(x - np.floor(x) - 0.5)
    amb = frac < delta
    if dead_zone:
        amb |= np.abs(np.abs(x) - DEAD_ZONE) < delta
    return amb


FP32_EPS = 2.0 ** -24


def ac_steps(dq, inv_gs, hf_mul, xm, bm):
    """Quantisation step [3][yb][xb][64] of every coefficient: dequant table x inv_global_scale / hf_mul x qm scale (X, B)."""
    base = inv_gs / hf_mul.astype(np.float64)                     # [yb][xb]
    qm = np.array([xm, 1.0, bm])
    return qm[:, None, None, None] * base[None, :, :, None] * dq.reshape(3, 1, 1, 64)


# ---------------------------------------------------------------------------------------------------------------- AQ and CfL (k_enc_tile_params)
AQ_REF = 0.05
AQ_THRESHOLDS = (0.81, 0.93, 1.08, 1.25)
AQ_LEVELS = (0.75, 0.87, 1.0, 1.16, 1.35)


def aq_multiplier(activity):
    """(aq_ref / activity)^0.2, limited to [0.75, 1.35]."""
    return np.clip((AQ_REF / (activity + 1e-4)) ** 0.2, 0.75, 1.35)


def aq_hf_mul(activity, base):
    """Per block: (hf_mul map, mulq). The product base x level is one fp32 multiplication of fp32 constants, restated exactly: several
    levels times a small base land on k + 1/2 (10 x 0.75), and rounding that tie to even is part of the rule."""
    mulq = aq_multiplier(activity)
    level = np.asarray(AQ_LEVELS, np.float32)[np.searchsorted(AQ_THRESHOLDS, mulq, side="right")]
    pre = np.float32(base) * level
    return np.clip(np.rint(pre), 1, 255).astype(np.int64), mulq


def cfl_factors(stats, yt, xt):
    """Per 64x64 tile from the block statistics [yb][xb][4]: (ytox, ytob, 84 * sum XY / sum YY, 84 * (sum BY / sum YY - 1), sum YY) with
    the int8 clamp, 0 where sum YY <= 1e-12."""
    yb, xb, _ = stats.shape
    pad = np.zeros((yt * 8, xt * 8, 4))
    pad[:yb, :xb] = stats
    t = pad.reshape(yt, 8, xt, 8, 4).sum(axis=(1, 3))
    syy = t[..., 3]
    ok = syy > 1e-12
    safe = np.where(ok, syy, 1.0)
    rx, rb = COLOR_FACTOR * t[..., 1] / safe, COLOR_FACTOR * (t[..., 2] / safe - 1.0)
    fx = np.where(ok, np.clip(np.rint(rx), -128, 127), 0).astype(np.int64)
    fb = np.where(ok, np.clip(np.rint(rb), -128, 127), 0).astype(np.int64)
    return fx, fb, rx, rb, syy
