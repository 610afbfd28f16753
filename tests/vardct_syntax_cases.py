"""VarDCT files from the independent writer (jxl_spec_writer.vardct_frame) that use the syntax the oracle's encoder never writes: custom LF
dequantisation, block-context maps, chroma-from-luma parameters, dequantisation tables, several HF presets, coefficient-order permutations,
two passes, prefix and LZ77 AC codes and a custom opsin matrix. Every integer a decoder must recover is drawn here from a seeded generator;
the writer turns it into a file, so the expected coefficients, LF and HF metadata are known without any encoder."""
import functools

import numpy as np

import jxl_spec_writer as jw
from spec_cases import OPSIN_INV

# F16-exact custom parameters
LF_DEQUANT_F16 = (0.0625, 0.1875, 0.25)                 # stored values; the multipliers are these / 128
CFL = (100, 0.125, 0.875, 140, 101)                     # colour_factor, base_x, base_b, x_factor_lf, b_factor_lf


def _f16(x):
    return float(np.float16(x))


OPSIN = (tuple(_f16(v * 1.03) for v in OPSIN_INV.ravel()), (-0.00390625, _f16(-0.0034), _f16(-0.0042)),
         (0.9375, 0.921875, 0.953125, 0.125))
TABLES = {0: [[48.0 * 64, -0.5, -0.25, 0.5], [12.0 * 64, -0.25, 0.25, -1.5], [8.0 * 64, 0.5, -1.0, -0.375]],     # DCT8, 4 bands
          4: [[40.0 * 64], [9.0 * 64], [6.5 * 64]],                                                            # DCT16, one band
          5: [[56.0 * 64, -0.75, -0.5], [14.0 * 64, -0.5, -0.25], [10.0 * 64, -1.25, 0.25]],                  # DCT32, 3 bands
          6: [[44.0 * 64, -1.0], [11.0 * 64, -0.5], [7.0 * 64, 0.75]]}                                        # DCT16X8 / DCT8X16, 2 bands
TABLES_DCT8_SINGLE = {0: [[40.0 * 64], [10.0 * 64], [6.0 * 64]]}
LF_THR = ([-20], [0, 60], [10])
QF_THR = [2, 5, 40, 121]
HF_MULS = [1, 2, 3, 5, 6, 40, 41, 121, 122, 200, 256]  # the thresholds themselves (a >= / > difference), both ends of the range
# Restoration parameters no encoder writes (F16-exact): distinct gaborish weights per channel, a non-monotone sharpness LUT with zeros,
# channel scales, sigma scales and border multiplier away from the defaults, non-zero bits in the two skipped 16-bit fields
RESTORATION = dict(gab_w=(0.125, 0.0625, 0.09375, 0.03125, 0.15625, 0.046875), sharp_lut=(0.0, 0.75, 0.25, 1.25, 0.0, 0.5, 1.0, 0.375),
                   channel_scale=(32.0, 6.5, 2.5), zero_flush=(0.4375, 0.625), quant_mul=0.53125, pass0_sigma_scale=0.75, pass2_sigma_scale=5.0,
                   border_sad_mul=0.5)
# Small coefficients and LF (XYB within about +-1): larger samples would leave the colour conversion's cube and opsin matrix to cancel
# values of 1e4 in linear light, and the rendered samples could no longer be held to fp32 level
FILTERED = dict(strategies=[0, 0, 4, 7], bctx=True, cfl=True, tables=TABLES, orders=True, opsin=True, amp=1, lf_amp=40, global_scale=3000,
                quant_lf=20, restoration=RESTORATION)


def block_ctx_map(rng, n=8):
    size = 3 * jw.NUM_ORDERS * (len(QF_THR) + 1) * 12
    m = list(rng.integers(0, n, size))
    m[:n] = range(n)
    return jw.BlockCtxMap(LF_THR, QF_THR, m)


def layout(rng, xb, yb, strategies):
    """Blocks in raster order of their first cell, chosen from `strategies` where they fit (inside the image, one group, uncovered cells)."""
    owner = np.zeros((yb, xb), bool)
    blocks = []
    for by in range(yb):
        for bx in range(xb):
            if owner[by, bx]:
                continue
            s = 0
            for cand in rng.permutation(strategies):
                cy, cx = jw.VARBLOCK[int(cand)]
                if by + cy <= yb and bx + cx <= xb and by // 32 == (by + cy - 1) // 32 and bx // 32 == (bx + cx - 1) // 32 \
                        and not owner[by:by + cy, bx:bx + cx].any():
                    s = int(cand)
                    break
            cy, cx = jw.VARBLOCK[s]
            owner[by:by + cy, bx:bx + cx] = True
            blocks.append((by, bx, s, int(rng.choice(HF_MULS))))
    return blocks


def coefficients(rng, xb, yb, blocks, amp, max_nz=None):
    """[3][cells][64] quantised coefficients: per block and channel a non-zero count drawn from 0, size/16 (the initial-prev boundary), a few,
    many or every AC position (dense DCT8 blocks give neighbours a predicted count of 63)."""
    q = np.zeros((3, yb * xb, 64), np.int64)
    for by, bx, s, _ in blocks:
        rows, cols = jw.storage_shape(s)
        size = rows * cols
        llf = set(jw.llf_positions(s))
        free = [p for p in range(size) if p not in llf]
        for c in range(3):
            kind = rng.integers(0, 6)
            nz = [0, size // 16, int(rng.integers(1, 6)), int(rng.integers(1, len(free) + 1)), len(free), size // 16 + 1][kind]
            if max_nz is not None:
                nz = min(nz, max_nz)
            for p in rng.choice(free, nz, replace=False):
                v = int(rng.integers(1, amp + 1)) * (1 if rng.integers(0, 2) else -1)
                cell, k = jw.coef_index(by, bx, s, int(p), xb)
                q[c, cell, k] = v
    return q


def permutations(rng, order_ids, npasses):
    out = {}
    for o in order_ids:
        n = {0: 64, 2: 256, 3: 1024, 4: 128}[o]
        skip = n // 64
        out[o] = [[list(range(skip)) + [skip + int(v) for v in rng.permutation(n - skip)] for _ in range(3)] for _ in range(npasses)]
    return out


# name -> (width, height, options); see build()
SPECS = {
    # 75 x 67 cells: 3 x 3 groups, the last column and row ragged; every LfGlobal / HfGlobal feature, three HF presets, permuted orders
    "multi_group_ans": (600, 530, dict(strategies=[0, 0, 4, 5, 6, 7], bctx=True, cfl=True, lf_dequant=True, tables=TABLES, presets=True,
                                       orders=True, opsin=True, extra_precision=1, global_scale=3000, quant_lf=20, amp=40)),
    # one group, one pass: all sections under one TOC entry; simple prefix codes (the generic AC reader)
    "single_group_prefix": (203, 150, dict(strategies=[0, 0, 4, 6, 7], bctx=True, cfl=True, tables=TABLES, orders=True, extra_precision=2,
                                           global_scale=5000, quant_lf=33, amp=1, max_nz=3, code="prefix")),
    # ANS with LZ77 runs (copies of distance 1) in the AC streams
    "lz77": (300, 270, dict(strategies=[0, 0, 4, 5], bctx=True, cfl=True, tables=TABLES, presets=True, orders=True, amp=2, code="lz77",
                            global_scale=1500, quant_lf=12, extra_precision=3)),
    # two passes with a shift of 2, different orders per pass
    "two_pass": (331, 200, dict(strategies=[0, 0, 4, 6, 7], bctx=True, cfl=True, tables=TABLES, orders=True, presets=True, pass_shift=2, amp=30,
                                global_scale=2500, quant_lf=24)),
    # 263 x 8 cells: two LF groups
    "two_lf_groups": (2100, 64, dict(strategies=[0, 0, 0, 4, 7], bctx=True, cfl=True, lf_dequant=True, tables=TABLES, presets=True, orders=True,
                                     global_scale=4000, quant_lf=18, amp=20)),
    # DCT8 only, for the float64 reconstruction: a single-band table (constant: pins the dequantiser alone), custom CfL, biases, qm scales
    "dct8_single_band": (131, 97, dict(strategies=[0], cfl=True, lf_dequant=True, tables=TABLES_DCT8_SINGLE, opsin=True, amp=25,
                                       x_qm_scale=5, b_qm_scale=0, global_scale=2048, quant_lf=16)),
    # DCT8 only with the 4-band table 0 and the custom block-context map
    "dct8_bands": (264, 136, dict(strategies=[0], bctx=True, cfl=True, tables=TABLES, orders=True, opsin=True, amp=25, x_qm_scale=1,
                                  b_qm_scale=4, global_scale=3500, quant_lf=40, extra_precision=1)),
    # adaptive LF smoothing on
    "smoothing": (264, 200, dict(strategies=[0, 0, 4, 7], bctx=True, cfl=True, lf_dequant=True, tables=TABLES, orders=True, opsin=True, amp=15,
                                 smoothing=True, global_scale=3000, quant_lf=20)),
    # gaborish + one EPF iteration: the wide TMA render kernel with a custom opsin matrix and the default filter parameters
    "gab_epf1": (256, 160, dict(strategies=[0, 0, 4, 7], bctx=True, cfl=True, tables=TABLES, orders=True, opsin=True, amp=15, gab=True, epf=1,
                                global_scale=3000, quant_lf=20)),
    # Restoration filters with the custom parameters (RESTORATION) unless noted; the render kernel each case selects is in
    # test_gpu_vardct_syntax.RENDER_KERNEL. Sizes at 32k +- 1 and 64k +- 1, widths of 4k (k_render<.., true>) and not.
    "epf1_260x97": (260, 97, dict(FILTERED, epf=1)),
    "epf1_95x63": (95, 63, dict(FILTERED, epf=1)),
    "epf2_128x65": (128, 65, dict(FILTERED, epf=2)),
    "epf2_161x33": (161, 33, dict(FILTERED, epf=2)),
    "epf3_132x67": (132, 67, dict(FILTERED, epf=3)),
    "gab_192x129": (192, 129, dict(FILTERED, gab=True)),
    "gab_127x95": (127, 95, dict(FILTERED, gab=True)),
    # the one-bit all_default form: gaborish and two EPF iterations with the default parameters, adaptive LF smoothing on
    "all_default_224x100": (224, 100, dict(FILTERED, gab=True, epf=2, restoration=dict(all_default=True), smoothing=True)),
    # 3 group rows (band decodes), the 7-px halo of gaborish + EPF 3 across the group and band borders
    "bands_300x530": (300, 530, dict(FILTERED, gab=True, epf=3)),
    # frames smaller than the 7-px (or 4-px) halo: it reflects more than once
    "tiny_1x1": (1, 1, dict(FILTERED, strategies=[0], epf=3)),
    "tiny_5x3": (5, 3, dict(FILTERED, strategies=[0], gab=True, epf=2)),
    "tiny_9x7": (9, 7, dict(FILTERED, strategies=[0], gab=True, epf=3, global_scale=500)),   # a coarser quantiser: one of its two cells is filtered
    # the wide kernel with custom parameters: interior (TMA) tiles, and a frame without one
    "wide_193x161": (193, 161, dict(FILTERED, gab=True, epf=1)),
    "wide_129x63": (129, 63, dict(FILTERED, gab=True, epf=1)),
    # other outputs of gaborish + EPF 1 (k_render<1,1,false>): 16-bit samples in orientation 6, and DCT8-only f32 linear samples
    # (the case the float64 chain runs from the writer's integers alone)
    "u16_orient6_200x136": (200, 136, dict(FILTERED, gab=True, epf=1, bits=16, orientation=6)),
    "dct8_f32_linear": (203, 150, dict(FILTERED, strategies=[0], gab=True, epf=1, bits=32, exp_bits=8, color=dict(tf=jw.TF_LINEAR))),
}


def raw_table_file():
    """A DCT8-only file whose table 0 is coded in mode 7 (RAW), which neither decoder supports."""
    c = _ints("dct8_single_band")
    kw = dict(c["kw"], tables={0: "raw"})
    return jw.vardct_frame(c["w"], c["h"], c["lfq"], c["blocks"], c["ytox"], c["ytob"], c["coeffs"], **kw)


def smooth_lf_field(rng, c, xb, yb):
    """Quantised LF of channel c for a case with adaptive LF smoothing: a smooth field plus 0 / +-1 noise in about half the cells, so that
    the smoothing gate takes all three of its branches (smoothed, blended, kept) in many cells; random LF would keep every sample."""
    y, x = np.mgrid[0:yb, 0:xb]
    noise = rng.integers(-1, 2, (yb, xb)) * (rng.random((yb, xb)) < 0.5)
    return np.round(30 * np.sin(x / 6.0 + c) + 20 * np.cos(y / 5.0 - c) + 0.5 * x).astype(np.int64) + noise


def _ints(name):
    """The integers of case `name` (seeded by its name): dict(w, h, xb, yb, lfq, blocks, ytox, ytob, sharp, coeffs, kwargs for vardct_frame)."""
    w, h, o = SPECS[name]
    rng = np.random.default_rng(sum(map(ord, name)))
    xb, yb = -(-w // 8), -(-h // 8)
    yt, xt = -(-yb // 8), -(-xb // 8)
    smooth_lf = o.get("smoothing")
    lf_amp = o.get("lf_amp", 300)
    lfq = [smooth_lf_field(rng, c, xb, yb) if smooth_lf else rng.integers(-lf_amp, lf_amp + 1, (yb, xb)) for c in range(3)]
    blocks = layout(rng, xb, yb, o["strategies"])
    ytox, ytob = rng.integers(-128, 128, (yt, xt)), rng.integers(-128, 128, (yt, xt))
    ytox.flat[0], ytob.flat[-1] = -128, 127
    ytox.flat[-1], ytob.flat[0] = 127, -128
    sharp = rng.integers(0, 8, (yb, xb))
    coeffs = coefficients(rng, xb, yb, blocks, o["amp"], o.get("max_nz"))
    ngroups = -(-xb // 32) * -(-yb // 32)
    npasses = 2 if o.get("pass_shift") else 1
    used_orders = sorted({jw.ORDER_ID[b[2]] for b in blocks})
    kw = dict(sharp=sharp, lf_dequant=LF_DEQUANT_F16 if o.get("lf_dequant") else None, global_scale=o.get("global_scale", 32768),
              quant_lf=o.get("quant_lf", 64), extra_precision=o.get("extra_precision", 0), bctx=block_ctx_map(rng) if o.get("bctx") else None,
              cfl=CFL if o.get("cfl") else None, tables=o.get("tables"),
              presets=[g % 3 for g in range(ngroups)] if o.get("presets") and ngroups > 1 else None,
              orders=permutations(rng, used_orders, npasses) if o.get("orders") else None, pass_shift=o.get("pass_shift"), code=o.get("code", "ans"),
              opsin=OPSIN if o.get("opsin") else None, skip_smoothing=not smooth_lf, gab=bool(o.get("gab")), epf_iters=o.get("epf", 0),
              restoration=o.get("restoration"), x_qm_scale=o.get("x_qm_scale", 3), b_qm_scale=o.get("b_qm_scale", 2), bits=o.get("bits", 8),
              exp_bits=o.get("exp_bits", 0), color=o.get("color"), orientation=o.get("orientation", 1))
    return dict(w=w, h=h, xb=xb, yb=yb, lfq=lfq, blocks=blocks, ytox=ytox, ytob=ytob, sharp=sharp, coeffs=coeffs, kw=kw)


@functools.lru_cache(maxsize=None)
def case(name, wrong=None):
    """(file, integers) of case `name`; wrong = one of jxl_spec_writer.WRONG_RULES writes it with that rule deliberately misapplied."""
    c = _ints(name)
    data = jw.vardct_frame(c["w"], c["h"], c["lfq"], c["blocks"], c["ytox"], c["ytob"], c["coeffs"], wrong=wrong, **c["kw"])
    return data, c


NAMES = list(SPECS)
FILTER_NAMES = [n for n in NAMES if SPECS[n][2].get("gab") or SPECS[n][2].get("epf")]
