"""ctypes door onto oracle/_build/liboracle.so — test infrastructure only.

The oracle is the CPU restatement of the JPEG XL work the reference reaches through libjxl
(N/Decoder/JxlDecoder.cpp:252, N/Encoder/JxlEncoder.cpp:128,367). PARITY UNPINNED: no libjxl,
no golden vectors exist offline (SURVEY.md §4, §8c). Only tests/, __graft_entry__.smoke() and
bench.py's cpu_baseline / --impl reference legs import this module.
"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
ORACLE_DIR = os.path.join(ROOT, "oracle")
LIB_PATH = os.path.join(ORACLE_DIR, "_build", "liboracle.so")
REF_LIB_PATH = os.path.join(ORACLE_DIR, "_ref", "libpixelformat_ref.so")


def build():
    subprocess.run(["make", "-s", "-C", ORACLE_DIR], check=True, stdout=subprocess.DEVNULL)


class EncodeParams(C.Structure):
    _fields_ = [("distance", C.c_float)] + [(n, C.c_int32) for n in (
        "effort", "lossless", "gab", "epf", "varblocks", "cfl", "adaptive_quant", "force_strategy", "use_prefix", "container",
        "modular_group_shift", "orientation", "skip_lf_smoothing", "threads", "bits", "exp_bits", "color_space", "white_point",
        "primaries", "tf", "intent")] + [("intensity_target", C.c_float), ("premultiplied", C.c_int32), ("black_channel", C.c_int32), ("num_passes", C.c_int32), ("pass_shift", C.c_int32), ("varblock_scale", C.c_float), ("varblock_pattern", C.c_int32)] + [
        (n, C.c_int32) for n in ("canvas_w", "canvas_h", "crop_x0", "crop_y0", "blend_mode", "alpha_blend_mode", "blend_source", "blend_clamp", "is_last", "save_as_reference", "frame_only")]


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            build()
        L = C.CDLL(LIB_PATH)
        L.jxlo_encode.argtypes = [C.c_void_p, C.c_int, C.c_uint32, C.c_uint32, C.c_int, C.c_int, C.POINTER(EncodeParams), C.c_void_p, C.c_size_t,
                                  C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.c_char_p, C.c_size_t]
        L.jxlo_decode.argtypes = [C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.POINTER(C.c_void_p), C.c_char_p, C.c_size_t]
        L.jxlo_image_free.argtypes = [C.c_void_p]
        L.jxlo_free.argtypes = [C.c_void_p]
        L.jxlo_image_info.argtypes = [C.c_void_p, C.POINTER(C.c_int32)]
        for n in ("jxlo_image_pixels", "jxlo_image_name", "jxlo_image_exif", "jxlo_image_icc"):
            getattr(L, n).argtypes = [C.c_void_p, C.POINTER(C.c_size_t)]
            getattr(L, n).restype = C.c_void_p
        L.jxlo_image_xmp.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_size_t)]
        L.jxlo_image_xmp.restype = C.c_void_p
        L.jxlo_image_stage_f32.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]
        L.jxlo_image_stage_f32.restype = C.c_size_t
        L.jxlo_image_stage_coeffs.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
        L.jxlo_image_stage_coeffs.restype = C.c_size_t
        L.jxlo_image_stage_i32.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]
        L.jxlo_image_stage_i32.restype = C.c_size_t
        L.jxlo_set_next_icc.argtypes = [C.c_char_p, C.c_size_t]
        for n in ("jxlo_icc_stream_write", "jxlo_icc_stream_read", "jxlo_icc_unpredict"):
            getattr(L, n).argtypes = [C.c_char_p, C.c_size_t, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.c_char_p, C.c_size_t]
        L.jxlo_signature_check.argtypes = [C.c_void_p, C.c_size_t]
        L.jxlo_transform_to_pixels.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_size_t]
        L.jxlo_transform_from_pixels.argtypes = [C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]
        L.jxlo_llf_from_dc.argtypes = [C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]
        L.jxlo_dequant_table.argtypes = [C.c_int, C.c_void_p]
        L.jxlo_dequant_table.restype = C.c_size_t
        L.jxlo_natural_order.argtypes = [C.c_int, C.c_void_p]
        L.jxlo_natural_order.restype = C.c_size_t
        L.jxlo_xyb_to_srgb8.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
        L.jxlo_srgb8_to_xyb.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


def default_params(**kw):
    p = EncodeParams()
    lib().jxlo_default_params(C.byref(p))
    for k, v in kw.items():
        if not hasattr(p, k):
            raise KeyError(k)
        setattr(p, k, v)
    return p


class OracleError(RuntimeError):
    pass


def encode(pixels, num_color=None, has_alpha=None, exif=b"", xmp=b"", icc=b"", **kw):
    """pixels: HxWxC uint8 or float32 array (C = colour [+black] [+alpha])."""
    a = np.ascontiguousarray(pixels)
    if a.ndim == 2:
        a = a[:, :, None]
    h, w, c = a.shape
    black = int(kw.get("black_channel", 0))
    if num_color is None:
        num_color = 1 if (c - black) <= 2 else 3
    if has_alpha is None:
        has_alpha = (c - black - num_color) == 1
    assert c == num_color + black + int(has_alpha)
    is_float = a.dtype != np.uint8
    if is_float:
        a = a.astype(np.float32)
    p = default_params(**kw)
    out = C.c_void_p()
    n = C.c_size_t()
    err = C.create_string_buffer(512)
    if icc:
        lib().jxlo_set_next_icc(bytes(icc), len(icc))
    rc = lib().jxlo_encode(a.ctypes.data, int(is_float), w, h, num_color, int(has_alpha), C.byref(p), exif, len(exif), xmp, len(xmp),
                           C.byref(out), C.byref(n), err, 512)
    if rc:
        raise OracleError(err.value.decode())
    data = C.string_at(out, n.value)
    lib().jxlo_free(out)
    return data


BLEND = dict(replace=0, add=1, blend=2, muladd=3, mul=4)


def encode_layers(canvas_w, canvas_h, layers, **common):
    """A multi-frame still: layers = [(pixels, dict(x0=, y0=, mode=, alpha_mode=, source=, save=, clamp=))...], every layer a regular frame
    of zero duration, the last one is_last. All layers share the source description in `common` (bit depth, colour, lossless / effort ...).
    Returns a bare codestream (no container)."""
    out = b""
    for i, (px, kw) in enumerate(layers):
        last = i + 1 == len(layers)
        out += encode(px, container=0, canvas_w=canvas_w, canvas_h=canvas_h, crop_x0=kw.get("x0", 0), crop_y0=kw.get("y0", 0),
                      blend_mode=BLEND[kw.get("mode", "replace")], alpha_blend_mode=BLEND[kw.get("alpha_mode", kw.get("mode", "replace"))],
                      blend_source=kw.get("source", 0), blend_clamp=int(kw.get("clamp", False)), is_last=int(last), save_as_reference=kw.get("save", 0),
                      frame_only=int(i > 0), **common)
    return out


def last_encode_strategy_cells():
    """Cells (8x8 units) covered per AC strategy in the last encode() of this thread."""
    out = (C.c_int64 * 27)()
    lib().jxlo_last_encode_strategy_cells(out)
    return list(out)


def _icc_call(fn, data):
    out, n, err = C.c_void_p(), C.c_size_t(), C.create_string_buffer(512)
    if fn(bytes(data), len(data), C.byref(out), C.byref(n), err, 512):
        raise OracleError(err.value.decode())
    r = C.string_at(out, n.value)
    lib().jxlo_free(out)
    return r


def icc_stream_write(icc):
    return _icc_call(lib().jxlo_icc_stream_write, icc)


def icc_stream_read(data):
    return _icc_call(lib().jxlo_icc_stream_read, data)


def icc_unpredict(enc):
    return _icc_call(lib().jxlo_icc_unpredict, enc)


_DT = {0: np.uint8, 1: np.uint16, 2: np.float16, 3: np.float32}


class Decoded:
    pass


def decode(data, threads=1, keep_stages=False):
    img = C.c_void_p()
    err = C.create_string_buffer(512)
    buf = bytes(data)
    rc = lib().jxlo_decode(buf, len(buf), threads, int(keep_stages), C.byref(img), err, 512)
    if rc:
        raise OracleError(err.value.decode())
    try:
        info = (C.c_int32 * 16)()
        lib().jxlo_image_info(img, info)
        d = Decoded()
        (d.width, d.height, d.format, d.sample_type, d.has_alpha, d.num_channels, d.xpad, d.ypad, d.known_profile, d.orientation,
         d.is_container, d.has_exif, d.num_xmp, d.bits, d.exp_bits, d.xyb) = list(info)
        n = C.c_size_t()
        p = lib().jxlo_image_pixels(img, C.byref(n))
        raw = np.frombuffer(C.string_at(p, n.value), dtype=_DT[d.sample_type])
        d.pixels = raw.reshape(d.height, d.width, -1).copy()
        p = lib().jxlo_image_name(img, C.byref(n))
        d.name = C.string_at(p, n.value) if n.value else b""
        p = lib().jxlo_image_icc(img, C.byref(n))
        d.icc = C.string_at(p, n.value) if n.value else None
        p = lib().jxlo_image_exif(img, C.byref(n))
        d.exif = C.string_at(p, n.value) if d.has_exif else None
        d.xmp = []
        for k in range(d.num_xmp):
            p = lib().jxlo_image_xmp(img, k, C.byref(n))
            d.xmp.append(C.string_at(p, n.value))
        if keep_stages and d.xpad:
            d.stages = {}
            for which, name in ((0, "idct"), (1, "gab"), (2, "epf"), (3, "lf")):
                ptr = C.c_void_p()
                cnt = lib().jxlo_image_stage_f32(img, which, C.byref(ptr))
                if cnt:
                    arr = np.frombuffer(C.string_at(ptr, cnt * 4), dtype=np.float32).copy()
                    d.stages[name] = arr.reshape(3, -1)
            ptr = C.c_void_p()
            cnt = lib().jxlo_image_stage_coeffs(img, C.byref(ptr))
            if cnt:
                d.stages["coeffs"] = np.frombuffer(C.string_at(ptr, cnt * 4), dtype=np.int32).copy().reshape(3, -1)
            # the integers the file carries: quantised LF [3 (X, Y, B)][yb][xb], hf_mul [yb][xb], ytox / ytob [yt][xt], and the quantiser
            xb, yb = d.xpad // 8, d.ypad // 8
            shapes = {"lfq": (3, yb, xb), "hf_mul": (yb, xb), "ytox": (-(-yb // 8), -(-xb // 8)), "ytob": (-(-yb // 8), -(-xb // 8)), "quant": (4,)}
            for which, name in enumerate(("lfq", "hf_mul", "ytox", "ytob", "quant")):
                cnt = lib().jxlo_image_stage_i32(img, which, C.byref(ptr))
                if cnt:
                    d.stages[name] = np.frombuffer(C.string_at(ptr, cnt * 4), dtype=np.int32).copy().reshape(shapes[name])
            if "quant" in d.stages:
                d.global_scale, d.quant_lf, d.x_qm_scale, d.b_qm_scale = (int(v) for v in d.stages.pop("quant"))
        return d
    finally:
        lib().jxlo_image_free(img)


from synth import synthetic_image  # noqa: E402,F401  (re-exported for the tests)


def psnr(a, b, peak=255.0):
    d = a.astype(np.float64) - b.astype(np.float64)
    mse = float(np.mean(d * d))
    return 99.0 if mse == 0 else 10 * np.log10(peak * peak / mse)
