"""An independent, bit-level JPEG XL writer for the tests — NOT derived from oracle/ or csrc/host/.

Why it exists: the product's host front-end (csrc/host/{bits,entropy,headers}.h) and the oracle's
(oracle/jxlo_{bits,entropy,headers}.h) began as the same text, so "GPU vs oracle" cannot catch a
misreading of the codestream syntax that both share. This module assembles files field by field,
straight from the syntax tables of ISO/IEC 18181-1 (SizeHeader, ImageMetadata, FrameHeader, TOC,
entropy-code headers, ANS / prefix streams, MA tree, Modular sub-bitstream, LfGlobal / HfGlobal of a
DC-only VarDCT frame) and 18181-2 (boxes), in pure Python with its own bit writer, its own alias
table construction and its own rANS encoder. The tests then require that BOTH readers decode these
files to the pixels the writer was given (tests/test_spec_writer_*.py).

Pure Python, sized for images of a few thousand samples.
"""
import math
import struct


# ----------------------------------------------------------------------------- bit level (18181-1 B.2)
class Bits:
    """LSB-first bit sink: u(n) appends the n low bits of v, least significant first."""

    def __init__(self):
        self.acc = 0
        self.n = 0

    def u(self, nbits, v):
        assert 0 <= v < (1 << nbits) or nbits == 0 and v == 0, (nbits, v)
        self.acc |= v << self.n
        self.n += nbits

    def bool(self, b):
        self.u(1, 1 if b else 0)

    def pad_to_byte(self):
        self.n = (self.n + 7) // 8 * 8

    def bytes(self):
        self.pad_to_byte()
        return self.acc.to_bytes(self.n // 8, "little")

    # U32(d0..d3): each distribution is ("val", c) | ("bits", n) | ("bo", n, offset)
    def u32(self, dists, v):
        for sel, d in enumerate(dists):
            if d[0] == "val" and d[1] == v:
                self.u(2, sel)
                return
            if d[0] == "bits" and 0 <= v < (1 << d[1]):
                self.u(2, sel)
                self.u(d[1], v)
                return
            if d[0] == "bo" and d[2] <= v < d[2] + (1 << d[1]):
                self.u(2, sel)
                self.u(d[1], v - d[2])
                return
        raise ValueError("U32 cannot represent %d with %r" % (v, dists))

    def u64(self, v):
        if v == 0:
            self.u(2, 0)
        elif v <= 16:
            self.u(2, 1)
            self.u(4, v - 1)
        elif v <= 272:
            self.u(2, 2)
            self.u(8, v - 17)
        else:
            self.u(2, 3)
            self.u(12, v & 0xFFF)
            v >>= 12
            shift = 12
            while v:
                self.u(1, 1)
                if shift == 60:
                    self.u(4, v & 0xF)
                    return
                self.u(8, v & 0xFF)
                v >>= 8
                shift += 8
            self.u(1, 0)

    def f16(self, x):
        self.u(16, struct.unpack("<H", struct.pack("<e", x))[0])

    def enum(self, v):
        self.u32((("val", 0), ("val", 1), ("bo", 4, 2), ("bo", 6, 18)), v)

    def u8(self, v):   # the 8-bit "U8" of the ANS distribution syntax
        if v == 0:
            self.u(1, 0)
        else:
            n = v.bit_length() - 1
            self.u(1, 1)
            self.u(3, n)
            self.u(n, v - (1 << n))


def f16_exact(x):
    """x itself, asserted to survive the trip through binary16 (a field the syntax stores as F16 must carry exactly the value meant)."""
    assert struct.unpack("<e", struct.pack("<e", x))[0] == x, "%r is not representable as F16" % x
    return x


def pack_signed(v):
    return 2 * v if v >= 0 else -2 * v - 1


def ceil_log2(x):
    return 0 if x <= 1 else (x - 1).bit_length()


# ----------------------------------------------------------------------------- headers (18181-1 Annex A)
def size_header(b, xsize, ysize, allow_small=True, allow_ratio=True):
    ratios = {1: (1, 1), 2: (12, 10), 3: (4, 3), 4: (3, 2), 5: (16, 9), 6: (5, 4), 7: (2, 1)}
    ratio = 0
    if allow_ratio:
        for r, (num, den) in ratios.items():
            if xsize == ysize * num // den:
                ratio = r
                break
    small = allow_small and ysize % 8 == 0 and ysize <= 256 and (ratio or (xsize % 8 == 0 and xsize <= 256))
    dist = (("bits", 9), ("bits", 13), ("bits", 18), ("bits", 30))
    b.bool(small)
    if small:
        b.u(5, ysize // 8 - 1)
    else:
        b.u32(dist, ysize - 1)
    b.u(3, ratio)
    if not ratio:
        if small:
            b.u(5, xsize // 8 - 1)
        else:
            b.u32(dist, xsize - 1)


def bit_depth(b, bits, exp_bits=0):
    b.bool(exp_bits > 0)
    if exp_bits == 0:
        b.u32((("val", 8), ("val", 10), ("val", 12), ("bo", 6, 1)), bits)
    else:
        b.u32((("val", 32), ("val", 16), ("val", 24), ("bo", 6, 1)), bits)
        b.u(4, exp_bits - 1)


EC_ALPHA, EC_DEPTH, EC_SPOT, EC_SELECTION, EC_BLACK = 0, 1, 2, 3, 4


def extra_channel_info(b, ec):
    """ec: dict(type, bits, exp_bits=0, dim_shift=0, name=b"", alpha_associated=False)"""
    default = ec["type"] == EC_ALPHA and ec["bits"] == 8 and not ec.get("exp_bits") and not ec.get("dim_shift") and not ec.get("name") and not ec.get("alpha_associated")
    b.bool(default)
    if default:
        return
    b.enum(ec["type"])
    bit_depth(b, ec["bits"], ec.get("exp_bits", 0))
    b.u32((("val", 0), ("val", 3), ("val", 4), ("bo", 3, 1)), ec.get("dim_shift", 0))
    name = ec.get("name", b"")
    b.u32((("val", 0), ("bits", 4), ("bo", 5, 16), ("bo", 10, 48)), len(name))
    for ch in name:
        b.u(8, ch)
    if ec["type"] == EC_ALPHA:
        b.bool(ec.get("alpha_associated", False))
    # (spot colour / CFA fields are not needed by the tests)


CS_RGB, CS_GRAY = 0, 1
WP_D65 = 1
PR_SRGB, PR_2100, PR_P3 = 1, 9, 11
TF_709, TF_LINEAR, TF_SRGB, TF_PQ = 1, 8, 13, 16


def color_encoding(b, color_space=CS_RGB, white_point=WP_D65, primaries=PR_SRGB, tf=TF_SRGB, intent=1, gamma=None):
    default = color_space == CS_RGB and white_point == WP_D65 and primaries == PR_SRGB and tf == TF_SRGB and intent == 1 and gamma is None
    b.bool(default)
    if default:
        return
    b.bool(False)                 # want_icc
    b.enum(color_space)
    b.enum(white_point)           # (colour space is never XYB here)
    if color_space != CS_GRAY:
        b.enum(primaries)
    b.bool(gamma is not None)
    if gamma is not None:
        b.u(24, gamma)
    else:
        b.enum(tf)
    b.enum(intent)


def image_metadata(b, bits=8, exp_bits=0, extra_channels=(), xyb_encoded=False, orientation=1, color=None, intensity_target=None, opsin=None):
    """opsin = (inverse matrix: 9 values, row-major; bias: 3 values; quant_bias: 4 values), all F16-exact: written as CustomTransformData with
    default_m = 0 (an XYB-encoded image only)."""
    color = color or {}
    all_default = bits == 8 and exp_bits == 0 and not extra_channels and xyb_encoded and orientation == 1 and not color and intensity_target is None
    b.bool(all_default)
    if not all_default:
        extra_fields = orientation != 1 or intensity_target is not None
        b.bool(extra_fields)
        if extra_fields:
            b.u(3, orientation - 1)
            b.bool(False)         # have_intrinsic_size
            b.bool(False)         # have_preview
            b.bool(False)         # have_animation
        bit_depth(b, bits, exp_bits)
        b.bool(True)              # modular_16_bit_buffer_sufficient
        b.u32((("val", 0), ("val", 1), ("bo", 4, 2), ("bo", 12, 1)), len(extra_channels))
        for ec in extra_channels:
            extra_channel_info(b, ec)
        b.bool(xyb_encoded)
        color_encoding(b, **color)
        if extra_fields:          # ToneMapping
            tm_default = intensity_target is None
            b.bool(tm_default)
            if not tm_default:
                b.f16(intensity_target)
                b.f16(0.0)        # min_nits
                b.bool(False)     # relative_to_max_display
                b.f16(0.0)        # linear_below
        b.u64(0)                  # extensions
    b.bool(opsin is None)         # default_m: default opsin inverse matrix and upsampling weights
    if opsin is not None:
        assert xyb_encoded
        b.bool(False)             # OpsinInverseMatrix.all_default
        for v in list(opsin[0]) + list(opsin[1]) + list(opsin[2]):
            b.f16(f16_exact(v))
        b.u(3, 0)                 # custom_weights_mask: default upsampling weights


def passes(b, num_passes=1, shifts=(), downsample=(), last_pass=()):
    b.u32((("val", 1), ("val", 2), ("val", 3), ("bo", 3, 4)), num_passes)
    if num_passes != 1:
        b.u32((("val", 0), ("val", 1), ("val", 2), ("bo", 1, 3)), len(downsample))
        assert len(shifts) == num_passes - 1
        for s in shifts:
            b.u(2, s)
        for d in downsample:
            b.u32((("val", 1), ("val", 2), ("val", 4), ("val", 8)), d)
        for p in last_pass:
            b.u32((("val", 0), ("val", 1), ("val", 2), ("bits", 3)), p)


FLAG_NOISE, FLAG_PATCHES, FLAG_SPLINES, FLAG_USE_LF_FRAME, FLAG_SKIP_LF_SMOOTHING = 1, 2, 16, 32, 128


RESTORATION_SIGMA = ("quant_mul", "pass0_sigma_scale", "pass2_sigma_scale", "border_sad_mul")


def frame_header(b, modular, num_extra=0, xyb_encoded=False, flags=0, group_size_shift=1, num_passes=1, pass_shifts=(), name=b"",
                 x_qm_scale=3, b_qm_scale=2, crop=None, canvas=None, blend=None, ec_blend=None, is_last=True, save_as_reference=0, gab=False, epf_iters=0,
                 restoration=None):
    """A regular frame, by default without restoration filters. Defaults: full size, last, blend mode Replace. crop = (x0, y0, width, height) with
    canvas = (image width, image height); blend / ec_blend[i] = dict(mode, alpha_channel, clamp, source) (F.2: BlendingInfo).
    restoration: the RestorationFilter fields written instead of the defaults, where the syntax has them (gaborish weights only with gab, the
    EPF fields only with epf_iters > 0), every value F16-exact:
      all_default=True: the one-bit form (gaborish on with default weights, two EPF iterations; gab and epf_iters must say so);
      gab_w: 6 values (x_w1, x_w2, y_w1, y_w2, b_w1, b_w2); sharp_lut: 8 values (VarDCT only);
      channel_scale: 3 values, with zero_flush: the two 16-bit fields after them, which decoders skip (non-zero bits by default);
      quant_mul (VarDCT only), pass0_sigma_scale, pass2_sigma_scale, border_sad_mul: all four together;
      sigma_for_modular (Modular only; 1.0 when absent)."""
    r = dict(restoration or {})
    assert not set(r) - {"all_default", "gab_w", "sharp_lut", "channel_scale", "zero_flush", "sigma_for_modular"} - set(RESTORATION_SIGMA), r
    b.bool(False)                 # all_default
    b.u(2, 0)                     # frame_type: regular
    b.u(1, 1 if modular else 0)   # encoding
    b.u64(flags)
    if not xyb_encoded:
        b.bool(False)             # do_YCbCr
    if not flags & FLAG_USE_LF_FRAME:
        up = (("val", 1), ("val", 2), ("val", 4), ("val", 8))
        b.u32(up, 1)              # upsampling
        for _ in range(num_extra):
            b.u32(up, 1)          # ec_upsampling
    if modular:
        b.u(2, group_size_shift)
    elif xyb_encoded:
        b.u(3, x_qm_scale)
        b.u(3, b_qm_scale)
    passes(b, num_passes, pass_shifts)
    b.bool(crop is not None)      # have_crop
    full_frame = True
    if crop is not None:
        dim = (("bits", 8), ("bo", 11, 256), ("bo", 14, 2304), ("bo", 30, 18688))
        x0, y0, cw, chh = crop
        b.u32(dim, pack_signed(x0))
        b.u32(dim, pack_signed(y0))
        b.u32(dim, cw)
        b.u32(dim, chh)
        full_frame = x0 <= 0 and y0 <= 0 and x0 + cw >= canvas[0] and y0 + chh >= canvas[1]
    mode = (("val", 0), ("val", 1), ("val", 2), ("bo", 2, 3))

    def blending_info(info):
        info = info or {}
        m = info.get("mode", 0)
        b.u32(mode, m)
        if num_extra and m in (2, 3):
            b.u32((("val", 0), ("val", 1), ("val", 2), ("bo", 3, 3)), info.get("alpha_channel", 0))
        if (num_extra and m in (2, 3)) or m == 4:
            b.bool(info.get("clamp", False))
        if m != 0 or not full_frame:
            b.u(2, info.get("source", 0))

    blending_info(blend)
    for i in range(num_extra):
        blending_info(ec_blend[i] if ec_blend else None)
    b.bool(is_last)               # (no animation: no duration field)
    if not is_last:
        b.u(2, save_as_reference)
        if (blend or {}).get("mode", 0) == 0 and full_frame:
            b.bool(False)         # save_before_color_transform
    b.u32((("val", 0), ("bits", 4), ("bo", 5, 16), ("bo", 10, 48)), len(name))
    for ch in name:
        b.u(8, ch)
    # RestorationFilter (all_default switches gaborish with its default weights and two EPF iterations on)
    def f16s(key, n):
        vals = list(r[key])
        assert len(vals) == n, (key, vals)
        for v in vals:
            b.f16(f16_exact(float(v)))

    b.bool(bool(r.get("all_default")))
    if r.get("all_default"):
        assert gab and epf_iters == 2 and set(r) == {"all_default"}
        b.u64(0)                  # frame header extensions
        return
    b.bool(gab)
    if gab:
        b.bool("gab_w" in r)      # gab_custom
        if "gab_w" in r:
            f16s("gab_w", 6)
    b.u(2, epf_iters)
    if epf_iters:
        if not modular:
            b.bool("sharp_lut" in r)            # epf_sharp_custom
            if "sharp_lut" in r:
                f16s("sharp_lut", 8)
        b.bool("channel_scale" in r)            # epf_weight_custom
        if "channel_scale" in r:
            f16s("channel_scale", 3)
            for v in r.get("zero_flush", (0.4375, 0.625)):
                b.f16(f16_exact(float(v)))      # two 16-bit fields no decoder uses
        sigma = [k for k in RESTORATION_SIGMA if k in r and not (modular and k == "quant_mul")]
        assert not sigma or len(sigma) == len(RESTORATION_SIGMA) - int(modular), "the sigma fields go together: %s" % sigma
        b.bool(bool(sigma))                     # epf_sigma_custom
        for k in sigma:
            b.f16(f16_exact(float(r[k])))
        if modular:
            b.f16(f16_exact(float(r.get("sigma_for_modular", 1.0))))
    b.u64(0)                      # restoration filter extensions
    b.u64(0)                      # frame header extensions


def toc(b, sizes, permutation=None):
    b.bool(permutation is not None)
    if permutation is not None:
        write_permutation_stream(b, permutation)
    b.pad_to_byte()
    dist = (("bits", 10), ("bo", 14, 1024), ("bo", 22, 17408), ("bo", 30, 4211712))
    for s in sizes:
        b.u32(dist, s)
    b.pad_to_byte()


# ----------------------------------------------------------------------------- entropy coding (18181-1 Annex C)
class Hybrid:
    def __init__(self, split_exp, msb, lsb):
        self.split_exp, self.msb, self.lsb = split_exp, msb, lsb

    def encode(self, v):
        """value -> (token, nbits, extra bits)"""
        split = 1 << self.split_exp
        if v < split:
            return v, 0, 0
        n = v.bit_length() - 1
        m = v - (1 << n)
        tok = split + ((n - self.split_exp) << (self.msb + self.lsb)) + ((m >> (n - self.msb)) << self.lsb) + (m & ((1 << self.lsb) - 1))
        nbits = n - self.msb - self.lsb
        return tok, nbits, (m >> self.lsb) & ((1 << nbits) - 1)

    def write(self, b, log_alpha):
        b.u(ceil_log2(log_alpha + 1), self.split_exp)
        if self.split_exp != log_alpha:
            b.u(ceil_log2(self.split_exp + 1), self.msb)
            b.u(ceil_log2(self.split_exp - self.msb + 1), self.lsb)


def alias_lookup_table(D, log_alpha):
    """C.2.6 alias mapping: returns for every 12-bit index the (symbol, offset) the decoder will produce."""
    log_bucket = 12 - log_alpha
    bucket, table = 1 << log_bucket, 1 << log_alpha
    D = list(D) + [0] * (table - len(D))
    symbols, offsets, cutoffs = [0] * table, [0] * table, [0] * table
    single = [i for i, d in enumerate(D) if d == 4096]
    if single:
        for j in range(table):
            symbols[j], offsets[j], cutoffs[j] = single[0], bucket * j, 0
    else:
        under, over = [], []
        for i in range(table):
            cutoffs[i] = D[i]
            if cutoffs[i] > bucket:
                over.append(i)
            elif cutoffs[i] < bucket:
                under.append(i)
        while over:
            o, u = over.pop(), under.pop()
            by = bucket - cutoffs[u]
            cutoffs[o] -= by
            symbols[u] = o
            offsets[u] = cutoffs[o]
            if cutoffs[o] < bucket:
                under.append(o)
            elif cutoffs[o] > bucket:
                over.append(o)
        for i in range(table):
            if cutoffs[i] == bucket:
                symbols[i], offsets[i], cutoffs[i] = i, 0, 0
            else:
                offsets[i] -= cutoffs[i]
    out = []
    for idx in range(4096):
        i, pos = idx >> log_bucket, idx & (bucket - 1)
        out.append((symbols[i], offsets[i] + pos) if pos >= cutoffs[i] else (i, pos))
    return out


def flat_distribution(n):
    return [4096 // n + (1 if i < 4096 % n else 0) for i in range(n)]


class TreeSelect(tuple):
    """Four symbols of a simple prefix code written with tree-select = 1: code lengths 1, 2, 3, 3 in the order listed."""


class EntropyCode:
    """One clustered entropy code. Each cluster is ("flat", n) | ("single", sym) | ("two", s0, s1, p0) for ANS, or a tuple of
    1..4 symbols for a simple prefix code (four symbols as a TreeSelect: code lengths 1, 2, 3, 3 in listed order instead of 2, 2, 2, 2).
    ctx_map maps context -> cluster."""

    def __init__(self, ctx_map, clusters, hybrids=None, use_prefix=False, log_alpha=None, lz77=None):
        """lz77: None or dict(min_symbol, min_length, len_hybrid=Hybrid(..)): ctx_map then carries one extra entry, the cluster of the
        distance context; stream items may be ("copy", length, distance_symbol) triples (C.2.5)."""
        self.ctx_map, self.clusters, self.use_prefix, self.lz77 = list(ctx_map), list(clusters), use_prefix, lz77
        self.log_alpha = 15 if use_prefix else (log_alpha if log_alpha is not None else 8)
        assert use_prefix or 5 <= self.log_alpha <= 8
        self.hybrids = hybrids or [Hybrid(4, 2, 0)] * len(clusters)   # the syntax's customary default configuration
        if use_prefix:
            self.codes = [self._simple_prefix(c) for c in clusters]
        else:
            self.dists = [self._dist(c) for c in clusters]
            self.inverse = []
            for D in self.dists:
                inv = {}
                for idx, (sym, off) in enumerate(alias_lookup_table(D, self.log_alpha)):
                    inv[(sym, off)] = idx
                self.inverse.append(inv)

    @staticmethod
    def _dist(c):
        if c[0] == "flat":
            return flat_distribution(c[1])
        if c[0] == "single":
            return [0] * c[1] + [4096]
        s0, s1, p0 = c[1], c[2], c[3]
        D = [0] * (max(s0, s1) + 1)
        D[s0], D[s1] = p0, 4096 - p0
        return D

    @staticmethod
    def _simple_prefix(syms):
        """symbol -> (code bits in reading order, length), Brotli simple-code canonical assignment."""
        n = len(syms)
        if n == 1:
            return {syms[0]: ((), 0)}
        if n == 2:
            lens = {syms[0]: 1, syms[1]: 1}
        elif n == 3:
            lens = {syms[0]: 1, syms[1]: 2, syms[2]: 2}
        elif isinstance(syms, TreeSelect):
            lens = {syms[0]: 1, syms[1]: 2, syms[2]: 3, syms[3]: 3}
        else:
            lens = {s: 2 for s in syms}
        code, codes, prev = 0, {}, 0
        for length, s in sorted((l, s) for s, l in lens.items()):
            code <<= length - prev
            prev = length
            codes[s] = (tuple((code >> (length - 1 - k)) & 1 for k in range(length)), length)
            code += 1
        return codes

    def write_header(self, b):
        b.bool(self.lz77 is not None)                   # lz77.enabled
        if self.lz77 is not None:
            b.u32((("val", 224), ("val", 512), ("val", 4096), ("bo", 15, 8)), self.lz77["min_symbol"])
            b.u32((("val", 3), ("val", 4), ("bo", 2, 5), ("bo", 8, 9)), self.lz77["min_length"])
            self.lz77["len_hybrid"].write(b, 8)         # the length configuration is always coded against log_alpha_size 8
        if len(self.ctx_map) > 1:
            nbits = ceil_log2(len(self.clusters))
            assert nbits <= 3
            b.bool(True)                                # simple context map
            b.u(2, nbits)
            for c in self.ctx_map:
                b.u(nbits, c)
        b.bool(self.use_prefix)
        if not self.use_prefix:
            b.u(2, self.log_alpha - 5)
        for h in self.hybrids:
            h.write(b, self.log_alpha)
        if self.use_prefix:
            counts = [max(c) + 1 for c in self.clusters]
            for cnt in counts:
                if cnt == 1:
                    b.bool(False)
                else:
                    n = (cnt - 1).bit_length() - 1
                    b.bool(True)
                    b.u(4, n)
                    b.u(n, cnt - 1 - (1 << n))
            for cnt, syms in zip(counts, self.clusters):
                if cnt == 1:
                    continue
                width = (cnt - 1).bit_length()
                b.u(2, 1)                               # hskip = 1: simple code
                b.u(2, len(syms) - 1)
                for s in syms:
                    b.u(width, s)
                if len(syms) == 4:
                    b.bool(isinstance(syms, TreeSelect))   # tree-select: lengths 1,2,3,3 or 2,2,2,2
        else:
            for c in self.clusters:
                if c[0] == "flat":
                    b.bool(False)
                    b.bool(True)
                    b.u8(c[1] - 1)
                elif c[0] == "single":
                    b.bool(True)
                    b.bool(False)
                    b.u8(c[1])
                else:
                    b.bool(True)
                    b.bool(True)
                    b.u8(c[1])
                    b.u8(c[2])
                    b.u(12, c[3])

    def write_stream(self, b, items):
        """items: list of (context, value). Writes the ANS state + symbols (or the prefix codes) with the hybrid-uint extra bits."""
        toks = []
        for it in items:
            if it[0] == "copy":                          # (copy, context of the symbol that would have been coded here, length, distance symbol)
                _, ctx, length, dist_sym = it
                cl = self.ctx_map[ctx]
                t, nb, ex = self.lz77["len_hybrid"].encode(length - self.lz77["min_length"])
                toks.append((cl, self.lz77["min_symbol"] + t, nb, ex))
                dcl = self.ctx_map[-1]                   # the distance context is the last one
                t, nb, ex = self.hybrids[dcl].encode(dist_sym)
                toks.append((dcl, t, nb, ex))
                continue
            ctx, v = it
            cl = self.ctx_map[ctx]
            t, nb, ex = self.hybrids[cl].encode(v)
            assert self.lz77 is None or t < self.lz77["min_symbol"]
            toks.append((cl, t, nb, ex))
        if self.use_prefix:
            for cl, t, nb, ex in toks:
                bits, length = self.codes[cl][t]
                for bit in bits:
                    b.u(1, bit)
                b.u(nb, ex)
            return
        state, refill = 0x130000, [None] * len(toks)
        for i in range(len(toks) - 1, -1, -1):
            cl, t, _, _ = toks[i]
            freq = self.dists[cl][t]
            assert freq > 0, "symbol %d has no probability in cluster %d" % (t, cl)
            if state >= freq << 20:
                refill[i] = state & 0xFFFF
                state >>= 16
            state = ((state // freq) << 12) + self.inverse[cl][(t, state % freq)]
        b.u(32, state)
        for i, (cl, t, nb, ex) in enumerate(toks):
            if refill[i] is not None:
                b.u(16, refill[i])
            b.u(nb, ex)


def permutation_items(perm, skip=0):
    """(context, value) items of a Lehmer-coded permutation (C.3.2; A.5): `end`, then the Lehmer codes of positions skip .. skip + end - 1
    (the first `skip` positions must be the identity; trailing zero codes are not written)."""
    n = len(perm)
    assert list(perm[:skip]) == list(range(skip))
    lehmer, rest = [], list(range(n))
    for p in perm:
        k = rest.index(p)
        lehmer.append(k)
        rest.pop(k)
    end = n
    while end > skip and lehmer[end - 1] == 0:
        end -= 1
    ctx_of = lambda x: min(7, ceil_log2(x + 1))
    items, prev = [(ctx_of(n), end - skip)], 0
    for v in lehmer[skip:end]:
        items.append((ctx_of(prev), v))
        prev = v
    return items


def write_permutation_stream(b, perm):
    """TOC permutation (C.3.2 Lehmer code) with its own 8-context entropy code (flat ANS over 64 symbols)."""
    code = EntropyCode([0] * 8, [("flat", 64)], log_alpha=6)
    code.write_header(b)
    code.write_stream(b, permutation_items(perm))


# ----------------------------------------------------------------------------- Modular (18181-1 Annex H)
class Leaf:
    def __init__(self, ctx, predictor, offset=0, multiplier=1):
        self.ctx, self.predictor, self.offset, self.multiplier = ctx, predictor, offset, multiplier


class Split:
    def __init__(self, prop, value, gt, le):   # property > value -> gt, else le
        self.prop, self.value, self.gt, self.le = prop, value, gt, le


def tree_nodes_bfs(root):
    order, queue = [], [root]
    while queue:
        n = queue.pop(0)
        order.append(n)
        if isinstance(n, Split):
            queue += [n.gt, n.le]
    return order


def write_tree(b, root):
    """MA tree in breadth-first order over its own 6-context code; returns the number of leaves (= contexts of the data code)."""
    items, nleaf = [], 0
    for n in tree_nodes_bfs(root):
        if isinstance(n, Split):
            items += [(1, n.prop + 1), (0, pack_signed(n.value))]
        else:
            assert n.ctx == nleaf, "leaf contexts are numbered in breadth-first order"
            nleaf += 1
            ml = 0
            while n.multiplier % (2 << ml) == 0:
                ml += 1
            items += [(1, 0), (2, n.predictor), (3, pack_signed(n.offset)), (4, ml), (5, (n.multiplier >> ml) - 1)]
    code = EntropyCode([0] * 6, [("flat", 64)], hybrids=[Hybrid(4, 1, 0)], log_alpha=6)
    code.write_header(b)
    code.write_stream(b, items)
    return nleaf


def predict(pred, W, N, NW, NE, NN, WW, NEE):
    if pred == 0:
        return 0
    if pred == 1:
        return W
    if pred == 2:
        return N
    if pred == 3:
        return (W + N) // 2 if W + N >= 0 else -((-(W + N)) // 2)   # C++ division truncates towards zero
    if pred == 4:
        p = W + N - NW
        return W if abs(p - W) < abs(p - N) else N
    if pred == 5:
        return max(min(W, N), min(max(W, N), W + N - NW))
    if pred == 7:
        return NE
    if pred == 8:
        return NW
    if pred == 9:
        return WW
    raise NotImplementedError(pred)


def modular_items(root, channels, stream_id=0, first_channel=0):
    """Residual tokens of `channels` (list of 2-D integer lists) under the MA tree: [(context, packed residual)]. first_channel: index of
    channels[0] in the image's channel list (property 0) when the list is a tail of it (group sections skip the meta channels)."""
    items = []
    for ci, ch in enumerate(channels):
        h, w = len(ch), len(ch[0]) if ch else 0
        for y in range(h):
            for x in range(w):
                W = ch[y][x - 1] if x else (ch[y - 1][x] if y else 0)
                N = ch[y - 1][x] if y else W
                NW = ch[y - 1][x - 1] if x and y else W
                NE = ch[y - 1][x + 1] if y and x + 1 < w else N
                NN = ch[y - 2][x] if y > 1 else N
                WW = ch[y][x - 2] if x > 1 else W
                NEE = ch[y - 1][x + 2] if y and x + 2 < w else NE
                props = {0: ci + first_channel, 1: stream_id, 2: y, 3: x, 4: abs(N), 5: abs(W), 6: N, 7: W, 9: W + N - NW, 10: W - NW, 11: NW - N, 12: N - NE, 13: N - NN, 14: W - WW}
                if x:   # property 8: W minus the gradient prediction error context of the pixel to the left
                    Wl = ch[y][x - 2] if x > 1 else (ch[y - 1][x - 1] if y else 0)
                    Nl = ch[y - 1][x - 1] if y else Wl
                    NWl = ch[y - 1][x - 2] if x > 1 and y else Wl
                    props[8] = W - (Wl + Nl - NWl)
                else:
                    props[8] = W
                # properties 16 + 4k .. 19 + 4k: the k-th previous channel of the same size (nearest first): |v|, v, |v - g|, v - g with g the
                # clamped gradient of that channel at the same position (H.4.1)
                k = 0
                for cj in range(ci - 1, -1, -1):
                    r = channels[cj]
                    if len(r) != h or len(r[0]) != w:
                        continue
                    v = r[y][x]
                    rW = r[y][x - 1] if x else 0
                    rN = r[y - 1][x] if y else rW
                    rNW = r[y - 1][x - 1] if x and y else rW
                    g = max(min(rW, rN), min(max(rW, rN), rW + rN - rNW))
                    props[16 + 4 * k], props[17 + 4 * k], props[18 + 4 * k], props[19 + 4 * k] = abs(v), v, abs(v - g), v - g
                    k += 1
                n = root
                while isinstance(n, Split):
                    n = n.gt if props.get(n.prop, 0) > n.value else n.le
                r = ch[y][x] - predict(n.predictor, W, N, NW, NE, NN, WW, NEE) - n.offset
                assert r % n.multiplier == 0, "sample not representable with this leaf's multiplier"
                items.append((n.ctx, pack_signed(r // n.multiplier)))
    return items


def rle_copies(items, min_length, dist_sym):
    """Replaces runs of equal (context, value) pairs by one literal plus a copy of distance 1 (`dist_sym` is the distance SYMBOL that means
    "one sample back": 1 in Modular streams, where symbols below 120 index the special-distance table and entry 1 is (dx, dy) = (1, 0))."""
    out, i = [], 0
    while i < len(items):
        j = i
        while j + 1 < len(items) and items[j + 1][1] == items[i][1]:
            j += 1
        run = j - i + 1
        out.append(items[i])
        if run - 1 >= min_length:
            out.append(("copy", items[i + 1][0], run - 1, dist_sym))
        else:
            out += items[i + 1:j + 1]
        i = j + 1
    return out


def lz77_copies(items, min_length, max_distance, dist_sym):
    """Greedy LZ77 over the values of (context, value) items: wherever the next >= min_length values repeat values 1 .. max_distance back,
    one ("copy", context, length, dist_sym(distance)) replaces them (the longest match, the nearest on a tie)."""
    vals = [it[1] for it in items]
    out, i, recent = [], 0, {}
    while i < len(items):
        best_len, best_d = 0, 0
        key = tuple(vals[i:i + min_length])
        if len(key) == min_length:
            for j in reversed(recent.get(key, [])):
                d = i - j
                if d > max_distance:
                    break
                n = 0
                while i + n < len(vals) and n < 1000 and vals[j + n] == vals[i + n]:   # may overlap the copy itself (j + n >= i), as a decoder allows
                    n += 1
                if n > best_len:
                    best_len, best_d = n, d
        take = best_len if best_len >= min_length else 1
        if best_len >= min_length:
            out.append(("copy", items[i][0], best_len, dist_sym(best_d)))
        else:
            out.append(items[i])
        for k in range(i, i + take):
            if k + min_length <= len(vals):
                recent.setdefault(tuple(vals[k:k + min_length]), []).append(k)
        i += take
    return out


def group_header(b, transforms=(), local=None):
    """Modular sub-bitstream header (H.2). local = (tree root, EntropyCode): the stream brings its own MA tree and code, written after the
    transforms (use_global_tree = 0)."""
    b.bool(local is None)   # use_global_tree
    b.bool(True)       # default weighted-predictor parameters
    b.u32((("val", 0), ("val", 1), ("bo", 4, 2), ("bo", 8, 18)), len(transforms))
    begin_c = (("bits", 3), ("bo", 6, 8), ("bo", 10, 72), ("bo", 13, 1096))
    for t in transforms:
        if t[0] == "rct":
            b.u(2, 0)
            b.u32(begin_c, t[1])
            b.u32((("val", 6), ("bits", 2), ("bo", 4, 2), ("bo", 6, 10)), t[2])                # rct_type
        elif t[0] == "squeeze":                                                                # ("squeeze", [(horizontal, in_place, begin_c, num_c), ...]); [] = default parameters
            b.u(2, 2)
            b.u32((("val", 0), ("bo", 4, 1), ("bo", 6, 9), ("bo", 8, 41)), len(t[1]))
            for horizontal, in_place, bc, nc in t[1]:
                b.bool(horizontal)
                b.bool(in_place)
                b.u32(begin_c, bc)
                b.u32((("val", 1), ("val", 2), ("val", 3), ("bo", 4, 4)), nc)
        else:
            assert t[0] == "palette"                                                           # ("palette", begin_c, num_c, nb_colours, nb_deltas, predictor)
            b.u(2, 1)
            b.u32(begin_c, t[1])
            b.u32((("val", 1), ("val", 3), ("val", 4), ("bo", 13, 1)), t[2])
            b.u32((("bo", 8, 0), ("bo", 10, 256), ("bo", 12, 1280), ("bo", 16, 5376)), t[3])
            b.u32((("val", 0), ("bo", 8, 1), ("bo", 10, 257), ("bo", 16, 1281)), t[4])
            b.u(4, t[5])
    if local is not None:
        write_tree(b, local[0])
        local[1].write_header(b)


def implicit_palette_index(pixel, bits=8):
    """Index offset (relative to the end of the explicit palette) of a colour of the implicit cubes (H.6.3), or None: first the 4x4x4 cube
    whose levels are ((k * max) >> 2) + 2^(bits-3), then the 5x5x5 cube with levels (k * max) >> 2."""
    maxv = (1 << bits) - 1
    small = [((k * maxv) >> 2) + (1 << max(0, bits - 3)) for k in range(4)]
    large = [(k * maxv) >> 2 for k in range(5)]
    if len(pixel) == 3 and all(v in small for v in pixel):
        return small.index(pixel[0]) + 4 * small.index(pixel[1]) + 16 * small.index(pixel[2])
    if len(pixel) == 3 and all(v in large for v in pixel):
        return 64 + large.index(pixel[0]) + 5 * large.index(pixel[1]) + 25 * large.index(pixel[2])
    return None


def forward_palette(planes, begin, num_c, colors, bits=8, deltas=(), predictor=0, delta_mask=None):
    """-> (palette plane: num_c rows of len(deltas) + len(colors) entries, index plane). A pixel takes the index of its colour among `colors`
    (offset by the delta entries, which come first), else an implicit-cube index. Where delta_mask[y][x] is an int d, the pixel is coded as
    delta entry d: it must equal prediction + deltas[d] in every channel (the caller builds the image that way)."""
    h, w = len(planes[begin]), len(planes[begin][0])
    nd = len(deltas)
    lut = {tuple(c): nd + i for i, c in enumerate(colors)}
    idx = [[0] * w for _ in range(h)]
    for y in range(h):
        for x in range(w):
            px = tuple(planes[begin + c][y][x] for c in range(num_c))
            if delta_mask is not None and delta_mask[y][x] is not None:
                idx[y][x] = delta_mask[y][x]
                continue
            if px in lut:
                idx[y][x] = lut[px]
            else:
                k = implicit_palette_index(px, bits)
                assert k is not None, "colour %r is neither in the palette nor in the implicit cubes" % (px,)
                idx[y][x] = nd + len(colors) + k
    pal = [[d[c] for d in deltas] + [col[c] for col in colors] for c in range(num_c)]
    return pal, idx


# ----------------------------------------------------------------------------- whole files
def container(codestream, boxes=(), split_at=None, level=None):
    """18181-2: signature box, ftyp, optional jxll, extra boxes, then jxlc (or two jxlp parts when split_at is given)."""
    def box(t, payload):
        return struct.pack(">I", 8 + len(payload)) + t + payload
    out = b"\x00\x00\x00\x0cJXL \x0d\x0a\x87\x0a" + box(b"ftyp", b"jxl \x00\x00\x00\x00jxl ")
    if level is not None:
        out += box(b"jxll", bytes([level]))
    if split_at is None:
        for t, p in boxes:
            out += box(t, p)
        return out + box(b"jxlc", codestream)
    out += box(b"jxlp", struct.pack(">I", 0) + codestream[:split_at])
    for t, p in boxes:     # metadata boxes between the two codestream parts
        out += box(t, p)
    return out + box(b"jxlp", struct.pack(">I", 0x80000001) + codestream[split_at:])


def modular_image(channels, bits=8, gray=False, alpha_bits=0, tree=None, data_code=None, rct=None, name=b"", orientation=1,
                  small_size=True, group_size_shift=1, toc_permutation=None, alpha_associated=False, extra=None, rle=None, palette=None,
                  local_global=False, group_local=None, group_rct=None):
    """A lossless Modular frame. channels: colour planes (1 or 3) + optional alpha + optional `extra` channels, each a list of rows.
    tree/data_code default to a single gradient-predictor leaf over a flat 256-symbol ANS code. Images larger than one group are
    written with a real multi-section TOC (each group its own section); toc_permutation reorders the sections in the file.
    palette = dict(begin, num_c, colors, deltas=(), predictor=0, delta_mask=None): a Palette transform (after the RCT, if any): the palette
    becomes meta channel 0, coded in the global section whatever its size; the index channel takes the place of the colour channels."""
    h, w = len(channels[0]), len(channels[0][0])
    ncolor = 1 if gray else 3
    ecs = []
    if alpha_bits:
        ecs.append(dict(type=EC_ALPHA, bits=alpha_bits, alpha_associated=alpha_associated))
    for e in (extra or []):
        ecs.append(e)
    assert len(channels) == ncolor + len(ecs)
    tree = tree or Leaf(0, 5)
    b = Bits()
    b.u(16, 0x0AFF)
    size_header(b, w, h, allow_small=small_size)
    image_metadata(b, bits=bits, extra_channels=ecs, xyb_encoded=False, orientation=orientation,
                   color=dict(color_space=CS_GRAY) if gray else None)
    b.pad_to_byte()
    return b.bytes() + modular_frame(channels, len(ecs), bits=bits, tree=tree, data_code=data_code, rct=rct, name=name, group_size_shift=group_size_shift,
                                     toc_permutation=toc_permutation, rle=rle, palette=palette, local_global=local_global, group_local=group_local, group_rct=group_rct)


def modular_frame(channels, num_extra, bits=8, tree=None, data_code=None, rct=None, name=b"", group_size_shift=1, toc_permutation=None, rle=None, palette=None,
                  local_global=False, group_local=None, group_rct=None, **header):
    """One Modular frame (frame header, TOC, sections) of `channels` (its own size); starts byte-aligned. **header: crop, canvas, blend, ec_blend,
    is_last, save_as_reference of frame_header(). local_global: the frame has NO global MA tree and the global stream brings its own (tree, data_code).
    group_local = (tree, code): every group section brings this tree and code of its own instead of using the global ones.
    group_rct = function(group index) -> list of (begin_c, rct_type) / ("palette", dict(begin, num_c, colors)): transforms listed in that group's own
    header (what libjxl's lossless encoder chooses per group), applied to the group's rectangles in the order listed."""
    h, w = len(channels[0]), len(channels[0][0])
    tree = tree or Leaf(0, 5)
    b = Bits()
    frame_header(b, modular=True, num_extra=num_extra, xyb_encoded=False, group_size_shift=group_size_shift, name=name, **header)
    gdim = 128 << group_size_shift
    gx, gy = -(-w // gdim), -(-h // gdim)
    ngroups, nlf = gx * gy, (-(-w // (gdim * 8))) * (-(-h // (gdim * 8)))
    # ---- LfGlobal: LF dequantisation (default), global tree + code, global Modular header (+ data when it fits one group)
    g = Bits()
    g.bool(True)                                         # LfChannelDequantization.all_default
    nleaf = len([n for n in tree_nodes_bfs(tree) if isinstance(n, Leaf)])
    code = data_code or EntropyCode([0] * nleaf, [("flat", 256)], log_alpha=8)
    g.bool(not local_global)                             # global tree present
    if not local_global:
        write_tree(g, tree)
        code.write_header(g)
    transforms = [("rct", rct[0], rct[1])] if rct else []
    for pl in ([palette] if isinstance(palette, dict) else (palette or [])):
        transforms.append(("palette", pl["begin"], pl["num_c"], len(pl["colors"]), len(pl.get("deltas", ())), pl.get("predictor", 0)))
    planes = [[list(r) for r in ch] for ch in channels]
    will_fit = w <= gdim and h <= gdim
    has_global_data = will_fit or bool(palette)
    assert not local_global or has_global_data or group_local, "a frame without a global tree needs local trees wherever data is coded"
    group_header(g, transforms, local=(tree, code) if (local_global and has_global_data) else None)
    if rct:
        planes = forward_rct(planes, rct[0], rct[1])
    nb_meta = 0
    for pl in ([palette] if isinstance(palette, dict) else (palette or [])):   # several palettes: each `begin` indexes the channel list as it is then
        pal, idx = forward_palette(planes, pl["begin"], pl["num_c"], pl["colors"], bits, pl.get("deltas", ()), pl.get("predictor", 0), pl.get("delta_mask"))
        planes = [pal] + planes[:pl["begin"]] + [idx] + planes[pl["begin"] + pl["num_c"]:]
        nb_meta += 1
    fits = w <= gdim and h <= gdim
    pack = (lambda it: rle_copies(it, rle[0], rle[1])) if rle else (lambda it: it)   # rle = (min run to replace, distance symbol)
    if fits:
        code.write_stream(g, pack(modular_items(tree, planes, 0)))
    elif nb_meta:
        code.write_stream(g, pack(modular_items(tree, planes[:nb_meta], 0)))         # meta channels live in the global section
    if ngroups == 1:
        sections = [g.bytes()]
    else:
        sections = [g.bytes()] + [b""] * nlf + [b""]      # LfGroups and HfGlobal are empty for Modular frames
        for gi in range(ngroups):
            x0, y0 = (gi % gx) * gdim, (gi // gx) * gdim
            s = Bits()
            if not fits:
                gtree, gcode = group_local if group_local else (tree, code)
                gts = group_rct(gi) if group_rct else []      # (begin_c, rct_type) or ("palette", dict(begin, num_c, colors)), in the order listed
                sub = [[row[x0:x0 + gdim] for row in ch[y0:y0 + gdim]] for ch in planes[nb_meta:]]
                listed = []
                for gt in gts:
                    if gt[0] == "palette":
                        pl = gt[1]
                        gpal, gidx = forward_palette(sub, pl["begin"], pl["num_c"], pl["colors"], bits)
                        sub = [gpal] + sub[:pl["begin"]] + [gidx] + sub[pl["begin"] + pl["num_c"]:]
                        listed.append(("palette", pl["begin"], pl["num_c"], len(pl["colors"]), 0, 0))
                    else:
                        sub = forward_rct(sub, gt[0], gt[1])
                        listed.append(("rct", gt[0], gt[1]))
                group_header(s, transforms=listed, local=group_local)
                gcode.write_stream(s, pack(modular_items(gtree, sub, 1 + 3 * nlf + 17 + gi)))   # channels are numbered from 0 inside a group section
            sections.append(s.bytes())
    # toc_permutation lists the logical section indices in the order they are stored in the file. The TOC codes the sizes in FILE
    # order plus the permutation that maps a logical section to its file slot.
    order = list(range(len(sections))) if toc_permutation is None else list(toc_permutation)
    assert sorted(order) == list(range(len(sections)))
    slot_of = [order.index(i) for i in range(len(sections))]
    toc(b, [len(sections[i]) for i in order], None if toc_permutation is None else slot_of)
    body = b"".join(sections[i] for i in order)
    return b.bytes() + body


def forward_rct(planes, begin, rct_type):
    perm, kind = rct_type // 7, rct_type % 7
    a, bb, c = planes[begin:begin + 3]
    h, w = len(a), len(a[0])
    # inverse permutation: output channel v[k] comes from the k-th decoded channel
    idx = [perm % 3, (perm + 1 + perm // 3) % 3, (perm + 2 - perm // 3) % 3]
    src = [None, None, None]
    for k in range(3):
        src[k] = planes[begin + idx[k]]
    out = [[[0] * w for _ in range(h)] for _ in range(3)]
    for y in range(h):
        for x in range(w):
            p, q, r = src[0][y][x], src[1][y][x], src[2][y][x]
            if kind == 6:                                  # YCgCo: decoder computes G, R, B from (Y, Co, Cg)
                co = p - r
                t = r + (co >> 1)
                cg = q - t
                yy = t + (cg >> 1)
                o = (yy, co, cg)
            else:
                first, second, third = p, q, r
                if kind & 1:
                    third -= first
                if kind >> 1 == 1:
                    second -= first
                elif kind >> 1 == 2:
                    second -= (first + r) >> 1
                o = (first, second, third)
            for k in range(3):
                out[k][y][x] = o[k]
    return planes[:begin] + out + planes[begin + 3:]


def modular_layers(canvas_w, canvas_h, layers, bits=8, alpha_bits=8, alpha_associated=False, group_size_shift=1):
    """A layered still: RGB + alpha image of canvas_w x canvas_h whose frames are `layers` = [dict(channels=[R, G, B, A planes], x0, y0,
    blend=dict(...), alpha_blend=dict(...), save=slot)], the last one is_last. Every frame carries its crop rectangle."""
    b = Bits()
    b.u(16, 0x0AFF)
    size_header(b, canvas_w, canvas_h)
    image_metadata(b, bits=bits, extra_channels=[dict(type=EC_ALPHA, bits=alpha_bits, alpha_associated=alpha_associated)], xyb_encoded=False)
    b.pad_to_byte()
    out = b.bytes()
    for i, ly in enumerate(layers):
        ch = ly["channels"]
        hh, ww = len(ch[0]), len(ch[0][0])
        out += modular_frame(ch, 1, bits=bits, group_size_shift=group_size_shift, crop=(ly.get("x0", 0), ly.get("y0", 0), ww, hh), canvas=(canvas_w, canvas_h),
                             blend=ly.get("blend"), ec_blend=[ly.get("alpha_blend", ly.get("blend"))], is_last=i + 1 == len(layers), save_as_reference=ly.get("save", 0))
    return out


# ----------------------------------------------------------------------------- Squeeze (H.6.2)
def _cdiv(v, d):
    """C division (truncation toward zero), as the smooth-tendency term is specified."""
    return -((-v) // d) if v < 0 else v // d


def smooth_tendency(B, a, n):
    diff = 0
    if B >= a >= n:
        diff = _cdiv(4 * B - 3 * n - a + 6, 12)
        if diff - (diff & 1) > 2 * (B - a):
            diff = 2 * (B - a) + 1
        if diff + (diff & 1) > 2 * (a - n):
            diff = 2 * (a - n)
    elif B <= a <= n:
        diff = _cdiv(4 * B - 3 * n - a - 6, 12)
        if diff + (diff & 1) < 2 * (B - a):
            diff = 2 * (B - a) - 1
        if diff - (diff & 1) < 2 * (a - n):
            diff = 2 * (a - n)
    return diff


def _squeeze_rows(rows):
    """Horizontal forward squeeze of a plane given as rows: -> (average rows, residual rows)."""
    avg_rows, res_rows = [], []
    for row in rows:
        w = len(row)
        aw = (w + 1) // 2
        avg = [(row[2 * x] + row[2 * x + 1] + (1 if row[2 * x] > row[2 * x + 1] else 0)) >> 1 if 2 * x + 1 < w else row[2 * x] for x in range(aw)]
        res = []
        for x in range(w - aw):
            a = avg[x]
            nxt = avg[x + 1] if x + 1 < aw else a
            left = row[2 * x - 1] if x else a
            res.append((row[2 * x] - row[2 * x + 1]) - smooth_tendency(left, a, nxt))
        avg_rows.append(avg)
        res_rows.append(res)
    return avg_rows, res_rows


def _transpose(rows):
    return [list(col) for col in zip(*rows)] if rows and rows[0] else []


def default_squeeze_params(chans, nb_meta):
    """chans: list of dicts with "rows"; the default parameter list a decoder derives when the transform lists none."""
    def dims(c):
        return (len(c["rows"][0]) if c["rows"] else 0, len(c["rows"]))
    nb = len(chans) - nb_meta
    w, h = dims(chans[nb_meta])
    out = []
    if nb > 2 and dims(chans[nb_meta + 1]) == (w, h):
        out += [(True, False, nb_meta + 1, 2), (False, False, nb_meta + 1, 2)]
    if not w > h:
        if h > 8:
            out.append((False, True, nb_meta, nb))
            h = (h + 1) // 2
    while w > 8 or h > 8:
        if w > 8:
            out.append((True, True, nb_meta, nb))
            w = (w + 1) // 2
        if h > 8:
            out.append((False, True, nb_meta, nb))
            h = (h + 1) // 2
    return out


def apply_squeeze(chans, params):
    """chans: list of dict(rows, hs, vs); applies the steps in order (the channel-list side and the samples)."""
    chans = [dict(c) for c in chans]
    for horizontal, in_place, bc, nc in params:
        end = bc + nc - 1
        offset = end + 1 if in_place else len(chans)
        for c in range(bc, end + 1):
            ch = chans[c]
            if horizontal:
                avg, res = _squeeze_rows(ch["rows"])
                new_hs, new_vs = ch["hs"] + 1, ch["vs"]
            else:
                at, rt = _squeeze_rows(_transpose(ch["rows"]))
                avg, res = _transpose(at), _transpose(rt)
                if not res:
                    res = []
                new_hs, new_vs = ch["hs"], ch["vs"] + 1
            chans[c] = dict(rows=avg, hs=new_hs, vs=new_vs)
            chans.insert(offset + (c - bc), dict(rows=res, hs=new_hs, vs=new_vs))
    return chans


def modular_squeeze_image(channels, bits=8, alpha_bits=0, params=None, group_size_shift=1, tree=None, data_code=None, section_local=None):
    """A lossless Modular frame whose global header lists one Squeeze transform (params = None: the default parameter list, written as an empty
    list). The residual channels are spread over the sections as H.4 prescribes: the global stream takes the channels up to the first one larger
    than a group, the LF-group sections those of shift >= 3, the pass-group sections the rest. section_local = (tree, code): every LF-group and
    pass-group section brings this MA tree and code of its own (use_global_tree = 0)."""
    h, w = len(channels[0]), len(channels[0][0])
    ecs = [dict(type=EC_ALPHA, bits=alpha_bits)] if alpha_bits else []
    assert len(channels) == 3 + len(ecs)
    tree = tree or Leaf(0, 5)
    nleaf = len([n for n in tree_nodes_bfs(tree) if isinstance(n, Leaf)])
    code = data_code or EntropyCode([0] * nleaf, [("flat", 256)], log_alpha=8)
    b = Bits()
    b.u(16, 0x0AFF)
    size_header(b, w, h)
    image_metadata(b, bits=bits, extra_channels=ecs, xyb_encoded=False)
    b.pad_to_byte()
    frame_header(b, modular=True, num_extra=len(ecs), xyb_encoded=False, group_size_shift=group_size_shift)
    gdim = 128 << group_size_shift
    gx, gy = -(-w // gdim), -(-h // gdim)
    lx, ly = -(-w // (gdim * 8)), -(-h // (gdim * 8))
    ngroups, nlf = gx * gy, lx * ly
    chans = [dict(rows=[list(r) for r in ch], hs=0, vs=0) for ch in channels]
    used = default_squeeze_params(chans, 0) if params is None else list(params)
    chans = apply_squeeze(chans, used)
    dims = lambda c: (len(c["rows"][0]) if c["rows"] else 0, len(c["rows"]))
    c0 = 0
    while c0 < len(chans) and not (dims(chans[c0])[0] > gdim or dims(chans[c0])[1] > gdim):
        c0 += 1
    g = Bits()
    g.bool(True)                                         # LfChannelDequantization.all_default
    g.bool(True)                                         # global tree present
    write_tree(g, tree)
    code.write_header(g)
    group_header(g, [("squeeze", [] if params is None else used)])
    # (every channel of the global stream is coded, empty ones included: they keep their channel index)
    glob = [c["rows"] for c in chans[:c0]]
    if any(dims(c)[0] and dims(c)[1] for c in chans[:c0]):
        code.write_stream(g, modular_items(tree, [r if r else [] for r in glob], 0))

    def section(x0, y0, dim, lo, hi, stream_id):
        sub = []
        for c in chans[c0:]:
            shift = min(c["hs"], c["vs"])
            cw, chh = dims(c)
            if shift < lo or shift > hi or not cw or not chh:
                continue
            rx0, ry0 = x0 >> c["hs"], y0 >> c["vs"]
            if rx0 >= cw or ry0 >= chh:
                continue
            rw, rh = min(dim >> c["hs"], cw - rx0), min(dim >> c["vs"], chh - ry0)
            if rw <= 0 or rh <= 0:
                continue
            sub.append([row[rx0:rx0 + rw] for row in c["rows"][ry0:ry0 + rh]])
        s = Bits()
        if sub:
            stree, scode = section_local if section_local else (tree, code)
            group_header(s, local=section_local)
            scode.write_stream(s, modular_items(stree, sub, stream_id))
        return s.bytes()

    if ngroups == 1:
        sections = [g.bytes()]
    else:
        sections = [g.bytes()]
        for li in range(nlf):
            sections.append(section((li % lx) * gdim * 8, (li // lx) * gdim * 8, gdim * 8, 3, 1000, 1 + nlf + li))
        sections.append(b"")                              # HfGlobal: empty for Modular frames
        for gi in range(ngroups):
            sections.append(section((gi % gx) * gdim, (gi // gx) * gdim, gdim, 0, 2, 1 + 3 * nlf + 17 + gi))
    toc(b, [len(sec) for sec in sections])
    return b.bytes() + b"".join(sections)


# ----------------------------------------------------------------------------- DC-only VarDCT frame
def vardct_dc_only(lf_xyb_quant, xsize, ysize, global_scale=32768, quant_lf=64, skip_smoothing=True):
    """A lossy frame whose every 8x8 block is DCT8 with all AC coefficients zero: pixels are the dequantised LF samples
    pushed through the inverse XYB transform. lf_xyb_quant: three planes (X, Y, B) of quantised LF ints, yb x xb each.
    Single group only (<= 256x256 px)."""
    xb, yb = -(-xsize // 8), -(-ysize // 8)
    assert xb <= 32 and yb <= 32
    b = Bits()
    b.u(16, 0x0AFF)
    size_header(b, xsize, ysize)
    image_metadata(b, xyb_encoded=True)                  # all_default: 8-bit sRGB, XYB-encoded
    b.pad_to_byte()
    frame_header(b, modular=False, xyb_encoded=True, flags=FLAG_SKIP_LF_SMOOTHING if skip_smoothing else 0)
    s = Bits()
    # ---- LfGlobal
    s.bool(True)                                         # LfChannelDequantization.all_default (1/4096, 1/512, 1/256)
    s.u32((("bo", 11, 1), ("bo", 11, 2049), ("bo", 12, 4097), ("bo", 16, 8193)), global_scale)
    s.u32((("val", 16), ("bo", 5, 1), ("bo", 8, 1), ("bo", 16, 1)), quant_lf)
    s.bool(True)                                         # default block context map
    s.bool(True)                                         # default chroma-from-luma parameters
    s.bool(True)                                         # global MA tree present
    tree = Leaf(0, 5)
    write_tree(s, tree)
    code = EntropyCode([0], [("flat", 256)], hybrids=[Hybrid(4, 2, 0)], log_alpha=8)
    code.write_header(s)
    # (the global Modular image has no channels here: no sub-bitstream header follows)
    # ---- LfGroup: LF coefficients (channel order Y, X, B), then HF metadata
    s.u(2, 0)                                            # extra_precision
    group_header(s)
    X, Y, B = lf_xyb_quant
    code.write_stream(s, modular_items(tree, [Y, X, B], 1))
    nb = xb * yb
    s.u(ceil_log2(nb), nb - 1)                           # nb_blocks - 1
    group_header(s)
    tw, th = -(-xb // 8), -(-yb // 8)
    zeros = lambda hh, ww: [[0] * ww for _ in range(hh)]
    block_info = [[0] * nb, [0] * nb]                    # row 0: strategy (DCT8 = 0), row 1: hf multiplier - 1
    sharp = zeros(yb, xb)
    code.write_stream(s, modular_items(tree, [zeros(th, tw), zeros(th, tw), block_info, sharp], 1 + 2 * 1 + 0))
    # ---- HfGlobal
    s.bool(True)                                         # default dequantisation matrices
    # num_hf_presets - 1 in ceil(log2(num_groups)) = 0 bits
    s.u32((("val", 0x5F), ("val", 0x13), ("val", 0), ("bits", 13)), 0)   # used_orders = 0: natural orders
    _write_ac_code_header(s, 495 * 15)                   # 495 contexts x 1 preset x 15 default block contexts
    # ---- PassGroup: every (block, channel) has zero non-zero coefficients: one token 0 each from a single-symbol distribution
    s.u(32, 0x130000)                                    # ANS state: never changes when every distribution is a single symbol
    body = s.bytes()
    toc(b, [len(body)])
    return b.bytes() + body


def _write_ac_code_header(b, num_ctx):
    """Entropy code with `num_ctx` contexts that all map to one cluster whose distribution is the single symbol 0."""
    b.bool(False)                  # lz77.enabled
    b.bool(True)                   # simple context map
    b.u(2, 0)                      # 0 bits per entry: every context -> cluster 0
    b.bool(False)                  # ANS
    b.u(2, 0)                      # log_alpha_size = 5
    Hybrid(4, 2, 0).write(b, 5)
    b.bool(True)                   # simple distribution
    b.bool(False)                  # one symbol
    b.u8(0)                        # symbol 0 with probability 4096


# ----------------------------------------------------------------------------- VarDCT frame with AC coefficients (A.8, A.9)
# Varblocks the writer places: strategy -> (cells down, cells across). A.8 names them; A.9: coefficients are stored with the longer side
# horizontal, so DCT16X8 (two cells down) is stored as one row of two cells, like DCT8X16.
VARBLOCK = {0: (1, 1), 4: (2, 2), 5: (4, 4), 6: (2, 1), 7: (1, 2)}
ORDER_ID = {0: 0, 4: 2, 5: 3, 6: 4, 7: 4}       # A.8 coefficient-order ids
# Dequantisation table of each strategy. The digest lists 17 tables but not their numbering; this is the standard's (DCT8, IDENTITY, DCT2X2,
# DCT4X4, DCT16, DCT32, DCT8X16, ...), unpinned by the digest.
QUANT_TABLE = {0: 0, 4: 4, 5: 5, 6: 6, 7: 6}
QUANT_TABLE_SHAPE = {0: (8, 8), 4: (16, 16), 5: (32, 32), 6: (8, 16)}    # (rows, columns) of coefficients in storage layout
NUM_ORDERS = 13
NUM_NZ_BUCKETS, NUM_ZDC = 37, 458
FREQ_CTX = [0] + list(range(15)) + [15 + i // 2 for i in range(16)] + [23 + i // 4 for i in range(32)]                # A.8 FreqCtx[64]
# A.8 NumNZCtx[64]; the digest writes "206 x 32", one more than the 64 entries leave room for: 206 fills the remaining 31
NUM_NZ_CTX = [0, 0, 31, 62, 62] + [93] * 4 + [123] * 4 + [152] * 8 + [180] * 12 + [206] * 31
assert len(FREQ_CTX) == 64 and len(NUM_NZ_CTX) == 64

# Deliberately wrong rules (vardct_frame(wrong=...)): each encodes the file as a reader with that one misreading would expect it.
WRONG_RULES = ("preset_offset", "qf_ge", "lf_idx_xyb", "block_ctx_c", "perm_inverted", "perm_no_skip", "nz_bucket_63", "prev_lt", "lz77_multiplier",
               "nz_floor")


def storage_shape(strategy):
    """(rows, columns) of a varblock's coefficients in storage layout: the shorter side vertical (A.9)."""
    cy, cx = VARBLOCK[strategy]
    return 8 * min(cy, cx), 8 * max(cy, cx)


def llf_positions(strategy):
    """Storage positions of the LLF entries (the cy x cx lowest frequencies, taken from the LF image, never coded)."""
    cy, cx = VARBLOCK[strategy]
    rows, cols = min(cy, cx), max(cy, cx)
    return [r * 8 * cols + c for r in range(rows) for c in range(cols)]


def coef_index(by, bx, strategy, p, xb):
    """(cell, k) of storage position p of the varblock whose first cell is (by, bx): position p lives in the (p // 64)-th covered cell in raster
    order of the block (the decoder's debug layout of quantised coefficients: [channel][cell][64])."""
    bw = VARBLOCK[strategy][1]
    j = p >> 6
    return (by + j // bw) * xb + bx + j % bw, p & 63


def nonzero_ctx(pred, wrong=None):
    """A.8 NonZeroCtx: n < 8 ? n : n < 64 ? 4 + n / 2 : 36."""
    limit = 63 if wrong == "nz_bucket_63" else 64
    return pred if pred < 8 else (4 + pred // 2 if pred < limit else 36)


def zero_density_ctx(nz, k, cells, log_cells):
    return (NUM_NZ_CTX[min(63, (nz + cells - 1) >> log_cells)] + FREQ_CTX[min(63, k >> log_cells)]) * 2


class BlockCtxMap:
    """LfGlobal's BlockCtxMap (A.8): thresholds on the quantised LF of X, Y and B, thresholds on hf_mul, and a map of
    3 x 13 x (#qf + 1) x n_lf entries to block contexts. lf_thr = (X, Y, B) lists; qf_thr values >= 1."""

    def __init__(self, lf_thr, qf_thr, ctx_map):
        self.lf_thr, self.qf_thr, self.ctx_map = [list(t) for t in lf_thr], list(qf_thr), [int(v) for v in ctx_map]
        self.n_lf = (len(self.lf_thr[0]) + 1) * (len(self.lf_thr[1]) + 1) * (len(self.lf_thr[2]) + 1)
        assert len(self.ctx_map) == 3 * NUM_ORDERS * (len(self.qf_thr) + 1) * self.n_lf
        self.num_ctx = max(self.ctx_map) + 1

    def lf_idx(self, qx, qy, qb, wrong=None):
        ix, iy, ib = (sum(1 for t in thr if q > t) for thr, q in zip(self.lf_thr, (qx, qy, qb)))
        ny, nb = len(self.lf_thr[1]) + 1, len(self.lf_thr[2]) + 1
        if wrong == "lf_idx_xyb":
            return (ix * ny + iy) * nb + ib
        return (ix * nb + ib) * ny + iy                 # nested X, B, Y

    def context(self, lf_idx, hf_mul, order, c, wrong=None):
        qf_idx = sum(1 for t in self.qf_thr if (hf_mul >= t if wrong == "qf_ge" else hf_mul > t))
        cc = c if wrong == "block_ctx_c" else (c ^ 1 if c < 2 else 2)     # the map lists Y, X, B
        return self.ctx_map[((cc * NUM_ORDERS + order) * (len(self.qf_thr) + 1) + qf_idx) * self.n_lf + lf_idx]

    def write(self, b):
        b.bool(False)                                   # not the default map
        for thr in self.lf_thr:
            b.u(4, len(thr))
            for t in thr:
                b.u32((("bits", 4), ("bo", 8, 16), ("bo", 16, 272), ("bo", 32, 65808)), pack_signed(t))
        b.u(4, len(self.qf_thr))
        for t in self.qf_thr:
            b.u32((("bits", 2), ("bo", 3, 4), ("bo", 5, 12), ("bo", 8, 44)), t - 1)
        nbits = ceil_log2(self.num_ctx)
        assert nbits <= 3, "the simple context map holds at most 8 block contexts"
        b.bool(True)                                    # simple context map
        b.u(2, nbits)
        for v in self.ctx_map:
            b.u(nbits, v)


def vardct_frame(xsize, ysize, lfq, blocks, ytox, ytob, coeffs, sharp=None, lf_dequant=None, global_scale=32768, quant_lf=64, extra_precision=0,
                 bctx=None, cfl=None, tables=None, presets=None, orders=None, pass_shift=None, code="ans", opsin=None, skip_smoothing=True,
                 gab=False, epf_iters=0, restoration=None, x_qm_scale=3, b_qm_scale=2, bits=8, exp_bits=0, color=None, orientation=1, wrong=None):
    """A complete XYB VarDCT image (codestream) whose every integer is the caller's:
      lfq: quantised LF, three (X, Y, B) integer arrays of yb x xb cells (row-major nested lists or numpy);
      blocks: [(by, bx, strategy, hf_mul)] covering every cell once, strategies from VARBLOCK, never across a 256-px group border;
      ytox, ytob: CfL factors per 64 x 64 tile (-128 .. 127); sharp: EPF sharpness per cell (default 0);
      coeffs: quantised coefficients [3 (X, Y, B)][yb * xb][64] in the layout of coef_index(); LLF positions must be 0. With two passes
        (pass_shift = s) the first pass carries coeffs >> s and the second the rest, so the decoded sum is `coeffs`.
    LfGlobal: lf_dequant = three F16 values (the stored F16, i.e. 128 x the multiplier) or None; global_scale, quant_lf; bctx = BlockCtxMap or None
      (default map); cfl = (colour_factor, base_x, base_b, x_factor_lf, b_factor_lf) or None.
    HfGlobal: tables = {table id: [3 lists of band parameters (X, Y, B), first band in the file's units x 64] | "raw"}: every listed table is
      written in mode 6 (DCT bands) or mode 7 (RAW, constant weights), the others as Library; None writes all_default. presets = per-group preset index list (num_hf_presets = max + 1);
      orders = {order id: [pass][3 channels] permutation of range(size) whose first size/64 entries are the identity}: coefficient order =
      natural[perm[k]].
    code: "ans" (clustered ANS, 8 clusters), "prefix" (simple prefix codes; every value must be <= 3) or "lz77" (ANS + LZ77 copies at
      distances 1 .. 160).
    opsin = (inverse matrix, bias, quant_bias) as image_metadata(); bits, exp_bits, color, orientation: the image's as image_metadata(), which
    set the output's sample type, transfer function and orientation. gab, epf_iters, restoration: the restoration filters as frame_header().
    wrong: one of WRONG_RULES."""
    import oracle_py                                    # natural coefficient orders only (jxlo_natural_order); everything else is this writer's
    import numpy as np
    assert wrong is None or wrong in WRONG_RULES
    xb, yb = -(-xsize // 8), -(-ysize // 8)
    xg, yg = -(-xb // 32), -(-yb // 32)
    xl, yl = -(-xb // 256), -(-yb // 256)
    ngroups, nlf = xg * yg, xl * yl
    npasses = 1 if pass_shift is None else 2
    lfq = [np.asarray(p, dtype=np.int64) for p in lfq]
    ytox, ytob = np.asarray(ytox, dtype=np.int64), np.asarray(ytob, dtype=np.int64)
    sharp = np.zeros((yb, xb), np.int64) if sharp is None else np.asarray(sharp, dtype=np.int64)
    coeffs = np.asarray(coeffs, dtype=np.int64).reshape(3, yb * xb, 64)
    presets = list(presets) if presets is not None else [0] * ngroups
    num_presets = max(presets) + 1
    assert len(presets) == ngroups and (num_presets == 1 or num_presets <= (1 << ceil_log2(ngroups)))
    # ---- cell map
    first = {}
    owner = np.full((yb, xb), -1, np.int64)
    for i, (by, bx, s, hm) in enumerate(blocks):
        cy, cx = VARBLOCK[s]
        assert 1 <= hm <= 256 and by + cy <= yb and bx + cx <= xb and by // 32 == (by + cy - 1) // 32 and bx // 32 == (bx + cx - 1) // 32, (by, bx, s)
        assert (owner[by:by + cy, bx:bx + cx] == -1).all(), "overlapping blocks"
        owner[by:by + cy, bx:bx + cx] = i
        first[(by, bx)] = i
    assert (owner >= 0).all(), "cells without a block"

    def natural(order_id):
        n = {0: 64, 2: 256, 3: 1024, 4: 128}[order_id]
        out = np.zeros(n, np.uint32)
        assert oracle_py.lib().jxlo_natural_order(order_id, out.ctypes.data) == n
        return [int(v) for v in out]

    orders = orders or {}
    used = [sorted(orders) if orders else [] for _ in range(npasses)]
    coding_order = {}                                   # (pass, order id, channel) -> storage positions in coding order
    for o in (0, 2, 3, 4):
        nat = natural(o)
        for p in range(npasses):
            for c in range(3):
                perm = orders[o][p][c] if o in orders else list(range(len(nat)))
                coding_order[(p, o, c)] = [nat[perm[k]] for k in range(len(nat))]

    # ---- entropy code of the AC coefficients: 8 clusters, each with its own hybrid-uint configuration and alphabet size
    nbctx = bctx.num_ctx if bctx is not None else 15
    num_ctx = 495 * num_presets * nbctx
    ctx_cluster = [((c * 5) ^ (c >> 3) ^ (c >> 6)) % 8 for c in range(num_ctx)]    # adjacent contexts fall into different clusters
    if code == "prefix":
        # values 0..3: the first two configurations give tokens 0, 1, 2 (+ 1 extra bit for 2, 3), the others code 0..3 as tokens 0..3
        hybrids = [Hybrid(0, 0, 0), Hybrid(1, 0, 0), Hybrid(2, 0, 0), Hybrid(1, 1, 0), Hybrid(1, 0, 1), Hybrid(2, 1, 0), Hybrid(2, 0, 1), Hybrid(3, 1, 1)]
    else:
        hybrids = [Hybrid(4, 2, 0), Hybrid(3, 1, 1), Hybrid(2, 0, 0), Hybrid(4, 1, 2), Hybrid(1, 0, 0), Hybrid(3, 2, 1), Hybrid(0, 0, 0), Hybrid(4, 0, 0)]
    lz = code == "lz77"

    def default_block_ctx(c, order_id):                 # A.8 default map: 15 block contexts
        d = [0, 1, 2, 2, 3, 3, 4, 5, 6, 6, 6, 6, 6, 7, 8, 9, 9, 10, 11, 12, 13, 14, 14, 14, 14, 14, 7, 8, 9, 9, 10, 11, 12, 13, 14, 14, 14, 14, 14]
        cc = c if wrong == "block_ctx_c" else (c ^ 1 if c < 2 else 2)
        return d[cc * NUM_ORDERS + order_id]

    def group_items(p, g):
        """(context, value) items of pass p of group g (A.8 PassGroup AC decode)."""
        gy, gx = divmod(g, xg)
        items = []
        nzc = np.zeros((3, 32, 32), np.int64)
        offset = 0 if wrong == "preset_offset" else 495 * nbctx * presets[g]
        for cy0 in range(32):
            for cx0 in range(32):
                by, bx = gy * 32 + cy0, gx * 32 + cx0
                if (by, bx) not in first:
                    continue
                _, _, s, hm = blocks[first[(by, bx)]]
                cy, cx = VARBLOCK[s]
                cells, size = cy * cx, cy * cx * 64
                log_cells = cells.bit_length() - 1
                o = ORDER_ID[s]
                for c in (1, 0, 2):
                    if bctx is not None:
                        li = bctx.lf_idx(lfq[0][by, bx], lfq[1][by, bx], lfq[2][by, bx], wrong)
                        bc = bctx.context(li, hm, o, c, wrong)
                    else:
                        bc = default_block_ctx(c, o)
                    if cx0 == 0:
                        pred = 32 if cy0 == 0 else nzc[c, cy0 - 1, cx0]
                    elif cy0 == 0:
                        pred = nzc[c, cy0, cx0 - 1]
                    else:
                        pred = (nzc[c, cy0 - 1, cx0] + nzc[c, cy0, cx0 - 1] + 1) // 2
                    order = coding_order[(p, o, c)]
                    vals = []
                    for k in range(size):
                        cell, kk = coef_index(by, bx, s, order[k], xb)
                        q = int(coeffs[c, cell, kk])
                        if k < cells:
                            assert q == 0, "LLF positions carry no coefficient"
                            continue
                        if npasses == 2:
                            q = q >> pass_shift if p == 0 else q - ((q >> pass_shift) << pass_shift)
                        vals.append(q)
                    nz = sum(1 for v in vals if v)
                    items.append((offset + nonzero_ctx(int(pred), wrong) * nbctx + bc, nz))
                    per_cell = nz // cells if wrong == "nz_floor" else -(-nz // cells)
                    nzc[c, cy0:cy0 + cy, cx0:cx0 + cx] = per_cell
                    prev = int(nz < size // 16) if wrong == "prev_lt" else int(nz <= size // 16)
                    left = nz
                    histo = offset + nbctx * NUM_NZ_BUCKETS + NUM_ZDC * bc
                    for i, v in enumerate(vals):
                        if left == 0:
                            break
                        items.append((histo + zero_density_ctx(left, cells + i, cells, log_cells) + prev, pack_signed(v)))
                        prev = int(v != 0)
                        left -= prev
        return items

    streams = {(p, g): group_items(p, g) for p in range(npasses) for g in range(ngroups)}
    if lz:
        # AC rule: distance = symbol + 1 (no multiplier, no special-distance table). Distances up to 160 give symbols on both sides of 120,
        # where a reader that sent AC distances through Modular's table (symbols < 120) or its offset (symbol - 119) would go astray.
        dist_sym = (lambda d: d + 119) if wrong == "lz77_multiplier" else (lambda d: d - 1)
        streams = {k: lz77_copies(v, 3, 160, dist_sym) for k, v in streams.items()}
    # alphabets: every cluster gets its own size, larger than any token it has to code
    tok_max = 0
    for items in streams.values():
        for it in items:
            if it[0] != "copy":
                tok_max = max(tok_max, hybrids[ctx_cluster[it[0]]].encode(it[1])[0])
    if code == "prefix":
        assert tok_max <= 3, "prefix-code case: values must stay <= 3"
        # clusters 0 and 1 (tokens 0..2): an unused fourth symbol sets the alphabet size; the rest code tokens 0..3. Lengths 1, 2, 3, 3 in listed
        # order, a different order per cluster, except cluster 2 (2, 2, 2, 2): no two clusters share a code
        clusters = [TreeSelect((0, 1, 2, 5)), TreeSelect((2, 0, 1, 7)), (0, 1, 2, 3), TreeSelect((3, 2, 1, 0)), TreeSelect((1, 3, 0, 2)),
                    TreeSelect((2, 0, 3, 1)), TreeSelect((0, 2, 1, 3)), TreeSelect((3, 0, 2, 1))]
        ac_code = EntropyCode(ctx_cluster, clusters, hybrids=hybrids, use_prefix=True)
    elif lz:
        assert tok_max < 224
        lzp = dict(min_symbol=224, min_length=3, len_hybrid=Hybrid(0, 0, 0))
        ac_code = EntropyCode(ctx_cluster + [5], [("flat", 240 + 2 * k) for k in range(8)], hybrids=hybrids, log_alpha=8, lz77=lzp)
    else:
        ac_code = EntropyCode(ctx_cluster, [("flat", tok_max + 1 + 3 * k) for k in range(8)], hybrids=hybrids, log_alpha=8)

    # ---- headers
    b = Bits()
    b.u(16, 0x0AFF)
    size_header(b, xsize, ysize)
    image_metadata(b, bits=bits, exp_bits=exp_bits, xyb_encoded=True, orientation=orientation, color=color, opsin=opsin)
    b.pad_to_byte()
    frame_header(b, modular=False, xyb_encoded=True, flags=FLAG_SKIP_LF_SMOOTHING if skip_smoothing else 0, num_passes=npasses,
                 pass_shifts=(pass_shift,) if npasses == 2 else (), x_qm_scale=x_qm_scale, b_qm_scale=b_qm_scale, gab=gab, epf_iters=epf_iters,
                 restoration=restoration)
    single = ngroups == 1 and npasses == 1
    sections = []
    s = Bits()
    # ---- LfGlobal
    s.bool(lf_dequant is None)                          # LfChannelDequantization.all_default
    if lf_dequant is not None:
        for v in lf_dequant:
            s.f16(f16_exact(v))
    s.u32((("bo", 11, 1), ("bo", 11, 2049), ("bo", 12, 4097), ("bo", 16, 8193)), global_scale)
    s.u32((("val", 16), ("bo", 5, 1), ("bo", 8, 1), ("bo", 16, 1)), quant_lf)
    if bctx is None:
        s.bool(True)
    else:
        bctx.write(s)
    s.bool(cfl is None)                                 # ColorCorrelation.all_default
    if cfl is not None:
        s.u32((("val", 84), ("val", 256), ("bo", 8, 2), ("bo", 16, 258)), cfl[0])
        s.f16(f16_exact(cfl[1]))
        s.f16(f16_exact(cfl[2]))
        s.u(8, cfl[3])
        s.u(8, cfl[4])
    s.bool(True)                                        # global MA tree
    tree = Leaf(0, 5)
    write_tree(s, tree)
    mcode = EntropyCode([0], [("flat", 256)], hybrids=[Hybrid(4, 2, 0)], log_alpha=8)
    mcode.write_header(s)

    def next_section():
        nonlocal s
        if not single:
            sections.append(s.bytes())
            s = Bits()

    next_section()
    # ---- LfGroups: LF coefficients (Y, X, B), HF metadata
    for li in range(nlf):
        ly, lx = divmod(li, xl)
        c0, r0 = lx * 256, ly * 256
        w, h = min(256, xb - c0), min(256, yb - r0)
        s.u(2, extra_precision)
        group_header(s)
        sub = lambda a: [[int(v) for v in row[c0:c0 + w]] for row in a[r0:r0 + h]]
        mcode.write_stream(s, modular_items(tree, [sub(lfq[1]), sub(lfq[0]), sub(lfq[2])], 1 + li))
        listed = []
        for y in range(r0, r0 + h):
            for x in range(c0, c0 + w):
                if (y, x) in first:
                    listed.append(blocks[first[(y, x)]])
        s.u(ceil_log2(w * h), len(listed) - 1)
        group_header(s)
        t0, tw, th = c0 // 8, -(-w // 8), -(-h // 8)
        tiles = lambda a: [[int(v) for v in row[t0:t0 + tw]] for row in a[r0 // 8:r0 // 8 + th]]
        info = [[bl[2] for bl in listed], [bl[3] - 1 for bl in listed]]
        mcode.write_stream(s, modular_items(tree, [tiles(ytox), tiles(ytob), info, sub(sharp)], 1 + 2 * nlf + li))
        next_section()
    # ---- HfGlobal
    s.bool(tables is None)                              # dequantisation matrices all_default
    if tables is not None:
        for t in range(17):
            if t not in tables:
                s.u(3, 0)                               # Library
                continue
            if tables[t] == "raw":                      # RAW: F16 denominator, then the weights as a 3-channel Modular image (A.8)
                rows, cols = QUANT_TABLE_SHAPE[t]
                s.u(3, 7)
                s.f16(1.0 / 64)
                group_header(s)
                mcode.write_stream(s, modular_items(tree, [[[100] * cols for _ in range(rows)]] * 3, 1 + 3 * nlf + t))
                continue
            s.u(3, 6)                                   # DCT bands
            nb = len(tables[t][0])
            s.u(4, nb - 1)
            for c in range(3):
                assert len(tables[t][c]) == nb
                for i, v in enumerate(tables[t][c]):
                    s.f16(f16_exact(v / 64.0 if i == 0 else v))
    s.u(ceil_log2(ngroups), num_presets - 1)
    for p in range(npasses):
        mask = sum(1 << o for o in used[p])
        s.u32((("val", 0x5F), ("val", 0x13), ("val", 0), ("bits", 13)), mask)
        if mask:
            items = []
            for o in used[p]:
                for c in range(3):
                    perm = list(orders[o][p][c])
                    n = len(perm)
                    if wrong == "perm_inverted":
                        inv = [0] * n
                        for k, v in enumerate(perm):
                            inv[v] = k
                        perm = inv
                    items += permutation_items(perm, 0 if wrong == "perm_no_skip" else n // 64)
            pcode = EntropyCode([0] * 8, [("flat", 64)], log_alpha=6)
            pcode.write_header(s)
            pcode.write_stream(s, items)
        ac_code.write_header(s)
    next_section()
    # ---- PassGroups, pass-major
    for p in range(npasses):
        for g in range(ngroups):
            s.u(ceil_log2(num_presets), presets[g])
            ac_code.write_stream(s, streams[(p, g)])
            next_section()
    if single:
        sections = [s.bytes()]
    toc(b, [len(x) for x in sections])
    return b.bytes() + b"".join(sections)
