"""Float64 restatements of the VarDCT decoder's arithmetic (SURVEY.md A.8, A.9), for files whose integers the tests know in advance
(tests/vardct_syntax_cases.py): LF dequantisation with its chroma-from-luma, dequantisation tables from mode-6 (DCT band) parameters,
AC dequantisation with the file's quant biases, hf_mul and qm scales followed by chroma from luma, and the inverse DCT8.

What these pin, and what they do not:
  * a single-band table is the same weight at every frequency, so a case that uses one pins the dequantiser without the interpolation;
  * a multi-band table is pinned only to the digest's formula: the band recurrence of A.8 and a geometric interpolation over the radial
    frequency normalised as (num_bands - 1) / (sqrt 2 + 1e-6) per unit of the table's diagonal, which the digest does not spell out;
  * the storage layout of square blocks (row index = horizontal frequency) is the decoders' convention, checked here against the oracle's
    transform (test_vardct_syntax_cpu.py), not against the digest, which only fixes it for rectangular blocks."""
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
