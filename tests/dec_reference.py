"""Float64 restatements of the VarDCT decoder's arithmetic (SURVEY.md A.8, A.9), for files whose integers the tests know in advance
(tests/vardct_syntax_cases.py): LF dequantisation with its chroma-from-luma, dequantisation tables from mode-6 (DCT band) parameters,
AC dequantisation with the file's quant biases, hf_mul and qm scales followed by chroma from luma, and the inverse DCT8.

What these pin, and what they do not:
  * a single-band table is the same weight at every frequency, so a case that uses one pins the dequantiser without the interpolation;
  * a multi-band table is pinned only to the digest's formula: the band recurrence of A.8 and a geometric interpolation over the radial
    frequency normalised as (num_bands - 1) / (sqrt 2 + 1e-6) per unit of the table's diagonal, which the digest does not spell out;
  * the storage layout of square blocks (row index = horizontal frequency) is the decoders' convention, checked here against the oracle's
    transform (test_vardct_syntax_cpu.py), not against the digest, which only fixes it for rectangular blocks.

The restoration stages (A.8 adaptive LF smoothing, A.10 gaborish and EPF) follow the digest and the header defaults of A.3. Where the digest
is silent or only approximate, this module makes a choice, and each choice that a decoder could make otherwise has a switch (SWITCHES) that
only the CPU sensitivity test turns on:
  * LF smoothing weights: the digest's centre / edge / corner weights (0.052262735, 0.203343183, 0.033497792) are marked low-confidence and do
    not sum to 1, so a flat LF image would not stay flat. This module uses edge 0.20345139757231578, corner 0.0334829185968739 and the centre
    1 - 4 (edge + corner) = 0.05226273532, which match the digest's centre and sum to 1. "Within half a quant step" is read as a blend:
    gap = max(0.5, max_c |smoothed - LF| / step_c), step_c = lf_dequant[c] * (65536 / global_scale) / quant_lf (no extra_precision),
    out = LF + (smoothed - LF) * max(0, 3 - 4 gap); the outermost LF row and column and LF images under 3 x 3 are left as they are;
  * sigma: per 8x8 cell, from the cell's own sharpness and its varblock's hf_mul (switch first_cell_sharpness: the varblock's first cell's
    sharpness for the whole block): sigma = quant_mul * sharp_lut[sharpness] / (global_scale / 65536 * hf_mul), inv_sigma = -1.1715728752538099
    / max(sigma, 1e-4 * 1.1715728752538099), so a sharpness whose LUT entry is 0 gives a huge negative inv_sigma;
  * skip threshold: "no filtering when sigma < ~0.3" is the comparison inv_sigma < -3.90524291751269967 (sigma < 0.29999), and a skipped pixel
    keeps its value in every pass (switch no_skip);
  * the SAD scale: the weight is max(0, 1 + SAD * inv_sigma * 1.65 * sigma_scale), the factor 1.65 with sigma_scale = pass0_sigma_scale, 1 and
    pass2_sigma_scale for passes 0, 1, 2 (switch sigma_scales_swapped), times border_sad_mul on border pixels;
  * border rule: a pixel whose image position is 0 or 7 mod 8 in x or y is a border pixel (switch no_border_rule);
  * SAD: sum over channels of channel_scale[c] times |differences| over the 5-pixel plus in passes 0 and 1, one pixel in pass 2 (switches
    channel_scale_reversed, single_pixel_sad_pass1);
  * image edges: every filter reads the image mirrored at its own size (x -> -x - 1 and 2 n - 1 - x, repeated while outside), never the padded
    planes (switch clamp: edge samples repeated instead);
  * gaborish weights: channel c uses gab_w[2 c], gab_w[2 c + 1] (switch gab_y_weights: Y's weights for every channel); the sharpness LUT is
    the file's (switch default_sharp_lut)."""
import numpy as np

import jxl_spec_writer as jw

DEFAULT_QUANT_BIAS = (1 - 0.05465007330715401, 1 - 0.07005449891748593, 1 - 0.049935103337343655, 0.145)
DEFAULT_LF_DEQUANT = (1.0 / 4096, 1.0 / 512, 1.0 / 256)
DEFAULT_CFL = (84, 0.0, 1.0, 128, 128)


def lf_planes(lfq, lf_dequant_f16=None, global_scale=32768, quant_lf=64, extra_precision=0, cfl=None):
    """[3 (X, Y, B)][yb][xb] LF samples: q * lf_dequant[c] * (65536 / global_scale) / quant_lf / 2^extra_precision, then X and B gain
    (base + (factor_lf - 128) / colour_factor) * Y."""
    mul = DEFAULT_LF_DEQUANT if lf_dequant_f16 is None else [v / 128.0 for v in lf_dequant_f16]
    cf, base_x, base_b, xlf, blf = cfl or DEFAULT_CFL
    fac = [m * (65536.0 / global_scale) / quant_lf / 2.0 ** extra_precision for m in mul]
    X, Y, B = (np.asarray(q, np.float64) * f for q, f in zip(lfq, fac))
    return np.stack([X + (base_x + (xlf - 128) / cf) * Y, Y, B + (base_b + (blf - 128) / cf) * Y])


def band_weights(params):
    """A.8: band[0] = p0; band[i] = band[i-1] * (p_i > 0 ? 1 + p_i : 1 / (1 - p_i))."""
    bands = [float(params[0])]
    for p in params[1:]:
        bands.append(bands[-1] * (1 + p if p > 0 else 1 / (1 - p)))
    return bands


def dequant_table(rows, cols, params3):
    """[3][rows * cols] dequantisation multipliers (1 / weight) of a mode-6 table; params3: the band parameters of X, Y and B with the first
    band in the table's units (the file's value x 64)."""
    out = []
    for params in params3:
        bands = band_weights(params)
        nb = len(bands)
        if nb == 1:
            w = np.full((rows, cols), bands[0])
        else:
            scale = (nb - 1) / (np.sqrt(2.0) + 1e-6)
            y, x = np.mgrid[0:rows, 0:cols].astype(np.float64)
            d = np.hypot(x * scale / (cols - 1), y * scale / (rows - 1))
            idx = np.minimum(d.astype(np.int64), nb - 2)
            b = np.array(bands)
            w = b[idx] * (b[idx + 1] / b[idx]) ** (d - idx)
        out.append((1.0 / w).ravel())
    return np.stack(out)


def adjust(q, bias_c, bias_ac):
    """A.8 adj(q): 0 -> 0, +-1 -> +-quant_bias[c], otherwise q - quant_bias[3] / q."""
    q = np.asarray(q, np.float64)
    safe = np.where(q == 0, 1.0, q)
    return np.where(q == 0, 0.0, np.where(np.abs(q) == 1, np.sign(q) * bias_c, q - bias_ac / safe))


def idct8(F):
    """A.9 inverse DCT8 of [..., 8 (row index = horizontal frequency), 8 (vertical frequency)] -> pixels [..., 8 (y), 8 (x)]: the plain
    DCT-III sum with c0 = 1, ck = sqrt 2 (the forward transform divides by 8 per dimension, so coefficient 0 is the block mean)."""
    k, i = np.mgrid[0:8, 0:8]
    C = np.where(k == 0, 1.0, np.sqrt(2.0)) * np.cos((2 * i + 1) * k * np.pi / 16)      # C[k][i]
    return np.einsum("...hv,vy,hx->...yx", F, C, C)


def dct8_reconstruction(ints, table0, quant_bias=None):
    """[3][ypad][xpad] XYB samples of a DCT8-only case: AC dequantisation adj(q) * dq[c][k] * (65536 / global_scale) / hf_mul * qm[c]
    (qm[X] = 0.8^(x_qm_scale - 2), qm[B] = 0.8^(b_qm_scale - 2), qm[Y] = 1), chroma from luma per 64 x 64 tile (X += (base_x + ytox / colour_factor)
    * Y, B += (base_b + ytob / colour_factor) * Y), the LF sample as coefficient 0, then the inverse DCT8. table0: [3][64] multipliers of table 0."""
    kw = ints["kw"]
    xb, yb = ints["xb"], ints["yb"]
    qb = quant_bias or DEFAULT_QUANT_BIAS
    cf, base_x, base_b, _, _ = kw["cfl"] or DEFAULT_CFL
    inv_gs = 65536.0 / kw["global_scale"]
    qm = (0.8 ** (kw["x_qm_scale"] - 2), 1.0, 0.8 ** (kw["b_qm_scale"] - 2))
    hf_mul = np.zeros((yb, xb))
    for by, bx, s, hm in ints["blocks"]:
        assert s == 0
        hf_mul[by, bx] = hm
    q = np.asarray(ints["coeffs"], np.float64).reshape(3, yb, xb, 64)
    F = np.stack([adjust(q[c], qb[c], qb[3]) * np.asarray(table0[c]) * inv_gs / hf_mul[..., None] * qm[c] for c in range(3)])
    tiles = lambda a: np.repeat(np.repeat(np.asarray(a, np.float64), 8, 0), 8, 1)[:yb, :xb, None]
    F[0] += (base_x + tiles(ints["ytox"]) / cf) * F[1]
    F[2] += (base_b + tiles(ints["ytob"]) / cf) * F[1]
    F[:, :, :, 0] = lf_planes(ints["lfq"], kw["lf_dequant"], kw["global_scale"], kw["quant_lf"], kw["extra_precision"], kw["cfl"])
    px = idct8(F.reshape(3, yb, xb, 8, 8))                           # [3][yb][xb][8][8]
    return px.transpose(0, 1, 3, 2, 4).reshape(3, 8 * yb, 8 * xb)


def table0_of(ints):
    """[3][64] multipliers of table 0 a case's file carries: its mode-6 parameters, or None for the library table."""
    tables = ints["kw"]["tables"]
    return None if tables is None or 0 not in tables else dequant_table(*jw.QUANT_TABLE_SHAPE[0], tables[0])


# ------------------------------------------------------------------------------------------------ restoration (A.8 smoothing, A.10)
LF_SMOOTH_W1, LF_SMOOTH_W2 = 0.20345139757231578, 0.0334829185968739                 # edge, corner; centre = 1 - 4 (w1 + w2)
INV_SIGMA_NUM = -1.1715728752538099024
MIN_INV_SIGMA = -3.90524291751269967465540850526868                                  # inv_sigma below this: the pixel is not filtered
EPF_SAD_MUL = 1.65
DEFAULT_RESTORATION = dict(gab_w=(0.115169525, 0.061248592) * 3, sharp_lut=tuple(i / 7 for i in range(8)), channel_scale=(40.0, 5.0, 3.5),
                           quant_mul=0.46, pass0_sigma_scale=0.9, pass2_sigma_scale=6.5, border_sad_mul=2.0 / 3.0, sigma_for_modular=1.0)
SWITCHES = ("gab_y_weights", "channel_scale_reversed", "sigma_scales_swapped", "no_border_rule", "no_skip", "default_sharp_lut",
            "first_cell_sharpness", "single_pixel_sad_pass1", "clamp")
EPF_NEIGHBOURS = {0: [(-2, 0), (-1, -1), (-1, 0), (-1, 1), (0, -2), (0, -1), (0, 1), (0, 2), (1, -1), (1, 0), (1, 1), (2, 0)],     # (dy, dx)
                  1: [(-1, 0), (0, -1), (0, 1), (1, 0)], 2: [(-1, 0), (0, -1), (0, 1), (1, 0)]}
PLUS = [(0, 0), (-1, 0), (1, 0), (0, -1), (0, 1)]


def restoration_params(restoration=None):
    """The filter parameters a file with frame_header(restoration=...) carries: its own values, the defaults for the others."""
    p = dict(DEFAULT_RESTORATION)
    p.update({k: v for k, v in (restoration or {}).items() if k in DEFAULT_RESTORATION})
    return p


def lf_smoothing(lf, lf_dequant_f16=None, global_scale=32768, quant_lf=64):
    """A.8 adaptive LF smoothing of [3][yb][xb] LF samples (see the module docstring for the weights and the gate)."""
    lf = np.asarray(lf, np.float64)
    _, h, w = lf.shape
    if h <= 2 or w <= 2:
        return lf.copy()
    mul = DEFAULT_LF_DEQUANT if lf_dequant_f16 is None else [v / 128.0 for v in lf_dequant_f16]
    step = np.array([m * (65536.0 / global_scale) / quant_lf for m in mul])[:, None, None]
    m = lf[:, 1:-1, 1:-1]
    edge = lf[:, :-2, 1:-1] + lf[:, 2:, 1:-1] + lf[:, 1:-1, :-2] + lf[:, 1:-1, 2:]
    corner = lf[:, :-2, :-2] + lf[:, :-2, 2:] + lf[:, 2:, :-2] + lf[:, 2:, 2:]
    sm = m * (1 - 4 * (LF_SMOOTH_W1 + LF_SMOOTH_W2)) + edge * LF_SMOOTH_W1 + corner * LF_SMOOTH_W2
    gap = np.maximum(0.5, (np.abs(m - sm) / step).max(axis=0))
    out = lf.copy()
    out[:, 1:-1, 1:-1] = m + (sm - m) * np.maximum(0.0, 3 - 4 * gap)
    return out


def _edge_index(n, pad, clamp=False):
    """Source index of positions -pad .. n + pad - 1 of a line of n samples: mirrored at the line's ends (repeatedly), or clamped."""
    i = np.arange(-pad, n + pad)
    if clamp:
        return np.clip(i, 0, n - 1)
    i = np.mod(i, 2 * n)
    return np.where(i < n, i, 2 * n - 1 - i)


def _extend(planes, pad, clamp=False):
    _, h, w = planes.shape
    return planes[:, _edge_index(h, pad, clamp)][:, :, _edge_index(w, pad, clamp)]


def gaborish(planes, gab_w, switches=()):
    """A.10 gaborish of [3][h][w] planes (the image itself, not the padded planes)."""
    planes = np.asarray(planes, np.float64)
    _, h, w = planes.shape
    e = _extend(planes, 1, "clamp" in switches)
    out = np.empty_like(planes)
    for c in range(3):
        k = 1 if "gab_y_weights" in switches else c
        w1, w2 = gab_w[2 * k], gab_w[2 * k + 1]
        p = e[c]
        edge = p[:-2, 1:-1] + p[2:, 1:-1] + p[1:-1, :-2] + p[1:-1, 2:]
        corner = p[:-2, :-2] + p[:-2, 2:] + p[2:, :-2] + p[2:, 2:]
        out[c] = (p[1:-1, 1:-1] + w1 * edge + w2 * corner) / (1 + 4 * (w1 + w2))
    return out


def cell_map(blocks, xb, yb, value):
    """[yb][xb] per cell: value(block) of the varblock covering it; blocks = [(by, bx, strategy, hf_mul)]."""
    out = np.zeros((yb, xb))
    for blk in blocks:
        by, bx, s = blk[:3]
        cy, cx = jw.VARBLOCK[s]
        out[by:by + cy, bx:bx + cx] = value(blk)
    return out


def inv_sigma(sharp, blocks, global_scale, params, switches=()):
    """[yb][xb] EPF inv_sigma of a VarDCT frame: per cell, its sharpness and its varblock's hf_mul (module docstring)."""
    sharp = np.asarray(sharp, np.int64)
    yb, xb = sharp.shape
    hf_mul = cell_map(blocks, xb, yb, lambda b: b[3])
    if "first_cell_sharpness" in switches:
        sharp = cell_map(blocks, xb, yb, lambda b: sharp[b[0], b[1]]).astype(np.int64)
    lut = np.asarray(DEFAULT_RESTORATION["sharp_lut"] if "default_sharp_lut" in switches else params["sharp_lut"], np.float64)
    sigma = params["quant_mul"] * lut[sharp] / (global_scale / 65536.0 * hf_mul)
    return INV_SIGMA_NUM / np.maximum(sigma, 1e-4 * -INV_SIGMA_NUM)


def epf_pass(planes, inv_sig, pas, params, switches=()):
    """One A.10 EPF pass (0: 12 neighbours, plus SAD; 1: 4 neighbours, plus SAD; 2: 4 neighbours, one-pixel SAD) of [3][h][w] planes with
    [yb][xb] inv_sigma."""
    planes = np.asarray(planes, np.float64)
    _, h, w = planes.shape
    pad = 3
    e = _extend(planes, pad, "clamp" in switches)
    at = lambda dy, dx: e[:, pad + dy:pad + dy + h, pad + dx:pad + dx + w]
    isg = np.repeat(np.repeat(np.asarray(inv_sig, np.float64), 8, 0), 8, 1)[:h, :w]
    scales = {0: params["pass0_sigma_scale"], 1: 1.0, 2: params["pass2_sigma_scale"]}
    if "sigma_scales_swapped" in switches:
        scales[0], scales[2] = scales[2], scales[0]
    y, x = np.mgrid[0:h, 0:w]
    border = np.isin(y % 8, (0, 7)) | np.isin(x % 8, (0, 7))
    if "no_border_rule" in switches:
        border[:] = False
    inv = isg * EPF_SAD_MUL * scales[pas] * np.where(border, params["border_sad_mul"], 1.0)
    cs = np.asarray(params["channel_scale"], np.float64)[::-1 if "channel_scale_reversed" in switches else 1][:, None, None]
    one_pixel = pas == 2 or (pas == 1 and "single_pixel_sad_pass1" in switches)
    acc, wsum = planes.copy(), np.ones((h, w))
    for dy, dx in EPF_NEIGHBOURS[pas]:
        taps = [(0, 0)] if one_pixel else PLUS
        sad = sum((np.abs(at(dy + py, dx + px) - at(py, px)) * cs).sum(axis=0) for py, px in taps)
        wgt = np.maximum(0.0, 1 + sad * inv)
        acc += wgt * at(dy, dx)
        wsum += wgt
    out = acc / wsum
    if "no_skip" not in switches:
        out = np.where(isg < MIN_INV_SIGMA, planes, out)
    return out


def restore(planes, w, h, gab, epf_iters, restoration=None, sharp=None, blocks=None, global_scale=32768, switches=()):
    """[3][h][w] samples after gaborish (if gab) and epf_iters EPF passes (pass 0 with 3 iterations, pass 1 with >= 1, pass 2 with >= 2) of
    the image in planes[:, :h, :w]; restoration: the file's custom fields (frame_header), sharp / blocks: the frame's integers."""
    assert set(switches) <= set(SWITCHES)
    params = restoration_params(restoration)
    out = np.asarray(planes, np.float64)[:, :h, :w]
    if gab:
        out = gaborish(out, params["gab_w"], switches)
    if epf_iters:
        isg = inv_sigma(sharp, blocks, global_scale, params, switches)
        for pas in ((0,) if epf_iters == 3 else ()) + (1,) + ((2,) if epf_iters >= 2 else ()):
            out = epf_pass(out, isg, pas, params, switches)
    return out
