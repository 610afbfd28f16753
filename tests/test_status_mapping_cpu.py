"""CPU test: the status and ErrorInfo text every exported entry point reports for each failure that is reachable without a device.

A C caller sees a failure only as a return value and the 255-character text in ErrorInfo, so these two are the whole contract of the error
paths. ErrorInfo is filled with a sentinel before each call: UNTOUCHED below means the call writes no text at all. CUDA stands for the
text JxlB200CudaAvailable reports (the cases that need it only run where no device is present).

The host-only entries (JxlB200PeekInfo, JxlB200BandLayout, JxlB200DebugSectionSizes) are also swept over a seeded set of mutated files and
compared with tests/golden/status_mapping.json (regenerate it with `python tests/test_status_mapping_cpu.py --write-golden`)."""
import ctypes as C
import functools
import hashlib
import json
import os
import random
import struct
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden", "status_mapping.json")
SENTINEL = b"<untouched>"
UNTOUCHED = object()
CUDA = object()

D_NULL, D_INVALID, D_DIMS, D_CHANNELS, D_DECODE, D_SIGNATURE = 1, 2, 6, 7, 10, 12
E_NULL, E_CANCELED, E_ENCODE = 1, 3, 4
LAYERED = "layered (multi-frame) files are decoded by LoadImage / JxlB200LoadImageBgra only, not by the batch and band calls"


class ErrorInfo(C.Structure):
    _fields_ = [("errorMessage", C.c_char * 256)]


class BitmapData(C.Structure):
    _fields_ = [("scan0", C.c_void_p), ("width", C.c_uint32), ("height", C.c_uint32), ("stride", C.c_uint32)]


class EncoderOptions(C.Structure):
    _fields_ = [("distance", C.c_float), ("effort", C.c_int32), ("lossless", C.c_bool)]


SetBasicInfo = C.CFUNCTYPE(None, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_bool)
SetMetadata = C.CFUNCTYPE(C.c_bool, C.c_void_p, C.c_size_t)
SetKnownProfile = C.CFUNCTYPE(C.c_bool, C.c_int32)
SetLayerData = C.CFUNCTYPE(C.c_bool, C.c_void_p, C.c_void_p, C.c_size_t)
Progress = C.CFUNCTYPE(C.c_bool, C.c_int32)
Write = C.CFUNCTYPE(C.c_int32, C.c_void_p, C.c_size_t)
Seek = C.CFUNCTYPE(C.c_int32, C.c_uint64)


class DecoderCallbacks(C.Structure):
    _fields_ = [("setBasicInfo", SetBasicInfo), ("setIccProfile", SetMetadata), ("setKnownColorProfile", SetKnownProfile),
                ("setExif", SetMetadata), ("setXmp", SetMetadata), ("setLayerData", SetLayerData)]


class IOCallbacks(C.Structure):
    _fields_ = [("Write", Write), ("Seek", Seek)]


P, S, I32, I64, U32 = C.c_void_p, C.c_size_t, C.c_int32, C.c_int64, C.c_uint32
SIGNATURES = {
    "LoadImage": (I32, [P, P, S, P]),
    "SaveImage": (I32, [P, P, P, P, P, P]),
    "JxlB200PeekInfo": (I32, [P, S, P, P]),
    "JxlB200LoadImageBgra": (I32, [P, S, P, S, P, P, P]),
    "JxlB200LoadImageLayers": (I32, [P, S, P, S, P, S, P, P]),
    "JxlB200BandLayout": (I32, [P, S, P, P]),
    "JxlB200DecodeBand": (I32, [I32, P, S, U32, U32, P, S, I32, P, P]),
    "JxlB200DecodeBatch": (I32, [I32, I32, P, P, P, P, I32, I32, I32, I32, P, P]),
    "JxlB200DecodeBatchSubmit": (P, [I32, I32, P, P, P, P, I32, I32, I32, I32, P]),
    "JxlB200DecodeBatchWait": (I32, [P, P, P]),
    "JxlB200EncodeToMemory": (I32, [P, P, P, I32, P, P, P]),
    "JxlB200DebugParseIcc": (I32, [P, S, P, P, P]),
    "JxlB200BandEncoderCreate": (P, [I32, P, U32, U32, U32, U32, P, P, I32, P, P]),
    "JxlB200BandEncoderTokenize": (I32, [P, U32, P, P, P]),
    "JxlB200BandEncoderFinish": (I32, [P, P, S, P, P, P, P]),
    "JxlB200BandEncoderDebugStage": (I64, [P, I32, P, I64, P, P]),
    "JxlB200AssembleBands": (I32, [U32, U32, P, P, U32, P, S, P, P, I32, P, P, P]),
    "JxlB200DebugDecodeStage": (I64, [P, S, I32, P, I64, P, P]),
    "JxlB200DebugSectionSizes": (I64, [P, S, P, I64, P, P]),
    "JxlB200CudaAvailable": (I32, [P]),
}


class Abi:
    """The library through its C signatures only; every call returns (return value, ErrorInfo text or UNTOUCHED)."""

    def __init__(self, path):
        self.lib = C.CDLL(path)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(self.lib, name)
            fn.restype, fn.argtypes = res, args

    def __call__(self, name, *args):
        ei = ErrorInfo()
        ei.errorMessage = SENTINEL
        r = getattr(self.lib, name)(*[C.byref(ei) if a is ErrorInfo else a for a in args])
        text = ei.errorMessage
        return r, (UNTOUCHED if text == SENTINEL else text.decode("latin-1"))


def _buf(data):
    return C.create_string_buffer(bytes(data), max(len(data), 1))


# ---- inputs
def _golden_files():
    d = os.path.join(HERE, "golden")
    return [open(os.path.join(d, f), "rb").read() for f in sorted(os.listdir(d)) if f.endswith(".jxl")]


def _header_only(xsize, ysize, **meta):
    """A bare codestream: signature, SizeHeader and ImageMetadata, then zero bytes."""
    import jxl_spec_writer as W
    b = W.Bits()
    b.u(16, 0x0AFF)
    W.size_header(b, xsize, ysize)
    W.image_metadata(b, **meta)
    return b.bytes() + bytes(64)


def _oversized():      # ysize 2^30 with the 2:1 ratio: xsize 2^31 does not fit an int32
    return _header_only(1 << 31, 1 << 30, xyb_encoded=True)


def _float_cmyk():
    import jxl_spec_writer as W
    return _header_only(64, 64, bits=16, exp_bits=5, extra_channels=[dict(type=W.EC_BLACK, bits=16, exp_bits=5)])


def _two_blacks():
    import jxl_spec_writer as W
    return _header_only(64, 64, extra_channels=[dict(type=W.EC_BLACK, bits=8), dict(type=W.EC_BLACK, bits=8)])


@functools.lru_cache(maxsize=None)
def _spec_cases():
    import spec_cases
    return [(name, bytes(data)) for name, data, *_ in spec_cases.cases()]


def _layered():
    return next(data for name, data in _spec_cases() if "layer" in name or "blend" in name)


def _valid():
    return _golden_files()[0]


def _truncated():
    return _valid()[:40]


@pytest.fixture(scope="module")
def abi(pkg):
    return Abi(pkg.LIB_PATH)


@pytest.fixture(scope="module")
def no_device(abi):
    ok, text = abi("JxlB200CudaAvailable", ErrorInfo)
    if ok:
        pytest.skip("a CUDA device is present")
    return text


def _expect(got, want, cuda_text=None):
    want = tuple(cuda_text if w is CUDA else w for w in want)
    assert got == want, (got, want)


# ---- decode entry points
def test_load_image(abi):
    cb = DecoderCallbacks(SetBasicInfo(lambda *a: None), SetMetadata(lambda p, n: True), SetKnownProfile(lambda p: True),
                          SetMetadata(lambda p, n: True), SetMetadata(lambda p, n: True), SetLayerData(lambda p, n, s: True))
    load = lambda data: abi("LoadImage", C.byref(cb), _buf(data), len(data), ErrorInfo)
    _expect(abi("LoadImage", None, None, 0, ErrorInfo), (D_NULL, UNTOUCHED))
    _expect(abi("LoadImage", C.byref(cb), None, 0, ErrorInfo), (D_NULL, UNTOUCHED))
    _expect(load(b"definitely not a jxl file"), (D_SIGNATURE, UNTOUCHED))
    _expect(load(_oversized()), (D_DIMS, UNTOUCHED))
    _expect(load(_two_blacks()), (D_CHANNELS, UNTOUCHED))
    _expect(load(_float_cmyk()), (D_DECODE, "Floating point CMYK images are not supported."))
    r, text = load(_truncated())
    assert r == D_DECODE and text is not UNTOUCHED and text


def test_host_only_queries(abi):
    peek = lambda d: abi("JxlB200PeekInfo", _buf(d) if d is not None else None, len(d or b""), (C.c_int32 * 8)(), ErrorInfo)
    layout = lambda d: abi("JxlB200BandLayout", _buf(d) if d is not None else None, len(d or b""), (C.c_int32 * 4)(), ErrorInfo)
    sections = lambda d, cap=4096: abi("JxlB200DebugSectionSizes", _buf(d) if d is not None else None, len(d or b""), (C.c_uint64 * 4096)(), cap, (C.c_int32 * 2)(), ErrorInfo)
    for fn, null, ok_ret in ((peek, D_NULL, 0), (layout, D_NULL, 0), (sections, 0, 4)):
        _expect(fn(None), (null, UNTOUCHED))
        _expect(fn(b"definitely not a jxl file"), (null if fn is sections else D_SIGNATURE, UNTOUCHED))
        _expect(fn(_oversized()), (0 if fn is sections else D_DIMS, UNTOUCHED))
        _expect(fn(_two_blacks()), (0 if fn is sections else D_CHANNELS, UNTOUCHED))
        _expect(fn(_float_cmyk()), (0 if fn is sections else D_DECODE, "Floating point CMYK images are not supported."))
    _expect(layout(_layered()), (D_DECODE, LAYERED))
    _expect(sections(_layered()), (0, LAYERED))
    assert peek(_layered()) == (0, UNTOUCHED)
    assert sections(_valid())[0] > 0 and sections(_valid(), cap=0) == (0, UNTOUCHED)


def test_image_decodes_before_the_device(abi):
    data = _valid()
    out = (C.c_uint8 * 64)()
    _expect(abi("JxlB200LoadImageBgra", None, 0, None, 0, None, None, ErrorInfo), (D_NULL, UNTOUCHED))
    _expect(abi("JxlB200LoadImageBgra", _buf(b"not a jxl"), 9, out, 64, None, None, ErrorInfo), (D_SIGNATURE, UNTOUCHED))
    _expect(abi("JxlB200LoadImageLayers", None, 0, None, 0, None, 0, None, ErrorInfo), (D_NULL, UNTOUCHED))
    _expect(abi("JxlB200LoadImageLayers", _buf(b"not a jxl"), 9, out, 64, None, 0, None, ErrorInfo), (D_SIGNATURE, UNTOUCHED))
    _expect(abi("JxlB200DecodeBand", -1, None, 0, 0, 1, None, 0, 0, None, ErrorInfo), (D_NULL, UNTOUCHED))
    _expect(abi("JxlB200DecodeBand", -1, _buf(b"not a jxl"), 9, 0, 1, out, 64, 0, None, ErrorInfo), (D_SIGNATURE, UNTOUCHED))
    _expect(abi("JxlB200DecodeBand", -1, _buf(data), len(data), 1, 1, out, 64, 0, None, ErrorInfo), (D_INVALID, "band decode: empty group-row range"))
    _expect(abi("JxlB200DebugDecodeStage", None, 0, 0, None, 0, None, ErrorInfo), (0, UNTOUCHED))
    _expect(abi("JxlB200DebugDecodeStage", _buf(b"not a jxl"), 9, 0, out, 16, None, ErrorInfo), (0, UNTOUCHED))


def test_batch_arguments(abi):
    arr = (C.c_void_p * 1)()
    sizes = (C.c_size_t * 1)()
    _expect(abi("JxlB200DecodeBatch", -1, 1, None, sizes, arr, sizes, 0, 1, 1, 0, None, ErrorInfo), (D_NULL, UNTOUCHED))
    _expect(abi("JxlB200DecodeBatch", -1, -1, arr, sizes, arr, sizes, 0, 1, 1, 0, None, ErrorInfo), (D_NULL, UNTOUCHED))
    _expect(abi("JxlB200DecodeBatchSubmit", -1, 1, arr, None, arr, sizes, 0, 1, 1, 0, ErrorInfo), (None, "null parameter"))
    _expect(abi("JxlB200DecodeBatchWait", None, None, ErrorInfo), (D_NULL, UNTOUCHED))


def test_decode_without_a_device(abi, no_device):
    data = _valid()
    out = (C.c_uint8 * 64)()
    cb = DecoderCallbacks(SetBasicInfo(lambda *a: None), SetMetadata(lambda p, n: True), SetKnownProfile(lambda p: True),
                          SetMetadata(lambda p, n: True), SetMetadata(lambda p, n: True), SetLayerData(lambda p, n, s: True))
    for d in (data, _truncated()):
        _expect(abi("JxlB200LoadImageBgra", _buf(d), len(d), out, 64, None, None, ErrorInfo), (D_DECODE, CUDA), no_device)
        _expect(abi("JxlB200LoadImageLayers", _buf(d), len(d), out, 64, None, 0, None, ErrorInfo), (D_DECODE, CUDA), no_device)
        _expect(abi("JxlB200DecodeBand", -1, _buf(d), len(d), 0, 1, out, 64, 0, None, ErrorInfo), (D_DECODE, CUDA), no_device)
        _expect(abi("JxlB200DebugDecodeStage", _buf(d), len(d), 0, (C.c_float * 16)(), 16, None, ErrorInfo), (0, CUDA), no_device)
    _expect(abi("LoadImage", C.byref(cb), _buf(data), len(data), ErrorInfo), (D_DECODE, CUDA), no_device)
    _expect(abi("JxlB200DecodeBand", 0, _buf(data), len(data), 0, 1, out, 64, 0, None, ErrorInfo), (D_INVALID, "cudaSetDevice failed"))
    datas, sizes = (C.c_void_p * 1)(C.cast(_buf(data), C.c_void_p)), (C.c_size_t * 1)(len(data))
    outs, out_sizes = (C.c_void_p * 1)(C.cast(out, C.c_void_p)), (C.c_size_t * 1)(64)
    for count in (0, 1):
        _expect(abi("JxlB200DecodeBatch", -1, count, datas, sizes, outs, out_sizes, 0, 1, 1, 0, None, ErrorInfo), (D_DECODE, CUDA), no_device)
        _expect(abi("JxlB200DecodeBatchSubmit", -1, count, datas, sizes, outs, out_sizes, 0, 1, 1, 0, ErrorInfo), (None, CUDA), no_device)


# ---- encode entry points
def _bitmap(pixels=None):
    px = pixels if pixels is not None else np.zeros((16, 16, 4), np.uint8)
    return BitmapData(px.ctypes.data, px.shape[1], px.shape[0], px.strides[0]), px


def test_encode_arguments(abi):
    bm, _hold = _bitmap()
    null_bm = BitmapData(None, 16, 16, 64)
    opts, meta = EncoderOptions(1.0, 3, False), (C.c_uint8 * 48)()
    io = IOCallbacks(Write(lambda p, n: 0), Seek(lambda p: 0))
    _expect(abi("SaveImage", None, None, None, None, ErrorInfo, None), (E_NULL, UNTOUCHED))
    _expect(abi("SaveImage", C.byref(bm), C.byref(opts), None, C.byref(io), ErrorInfo, None), (E_NULL, UNTOUCHED))
    _expect(abi("SaveImage", C.byref(null_bm), C.byref(opts), meta, C.byref(io), ErrorInfo, None), (E_NULL, ""))
    _expect(abi("SaveImage", C.byref(bm), C.byref(opts), meta, C.byref(io), ErrorInfo, Progress(lambda p: p < 15)), (E_CANCELED, ""))
    _expect(abi("JxlB200EncodeToMemory", None, C.byref(opts), None, 0, C.byref(C.c_void_p()), C.byref(C.c_size_t()), ErrorInfo), (E_NULL, UNTOUCHED))
    _expect(abi("JxlB200EncodeToMemory", C.byref(null_bm), C.byref(opts), None, 0, C.byref(C.c_void_p()), C.byref(C.c_size_t()), ErrorInfo), (E_NULL, UNTOUCHED))
    flags = C.c_uint32()
    _expect(abi("JxlB200BandEncoderCreate", -1, None, 16, 0, 0, 0, C.byref(opts), None, 0, C.byref(flags), ErrorInfo), (None, "null parameter"))
    _expect(abi("JxlB200BandEncoderCreate", -1, C.byref(null_bm), 16, 0, 0, 0, C.byref(opts), None, 0, C.byref(flags), ErrorInfo), (None, "null parameter"))
    _expect(abi("JxlB200BandEncoderTokenize", None, 0, C.byref(C.c_void_p()), C.byref(C.c_size_t()), ErrorInfo), (E_NULL, UNTOUCHED))
    _expect(abi("JxlB200BandEncoderFinish", None, (C.c_uint64 * 1)(), 1, C.byref(C.c_void_p()), C.byref(C.c_size_t()), None, ErrorInfo), (E_NULL, UNTOUCHED))
    _expect(abi("JxlB200BandEncoderDebugStage", None, 0, None, 0, None, ErrorInfo), (0, "null parameter"))
    abi.lib.JxlB200BandEncoderDestroy(None)


def test_assemble_bands_is_host_only(abi):
    opts = EncoderOptions(1.0, 3, False)
    hist = (C.c_uint64 * 8)()

    def assemble(blobs, count=None, h=hist, words=8):
        bufs = [_buf(b) for b in blobs]
        ptrs = (C.c_void_p * max(len(blobs), 1))(*[C.cast(b, C.c_void_p) for b in bufs])
        sizes = (C.c_size_t * max(len(blobs), 1))(*[len(b) for b in blobs])
        return abi("JxlB200AssembleBands", 64, 64, C.byref(opts), None, 0, h, words, ptrs, sizes, len(blobs) if count is None else count,
                   C.byref(C.c_void_p()), C.byref(C.c_size_t()), ErrorInfo)

    _expect(abi("JxlB200AssembleBands", 64, 64, None, None, 0, hist, 8, None, None, 1, None, None, ErrorInfo), (E_NULL, UNTOUCHED))
    _expect(assemble([b"x"], count=0), (E_NULL, UNTOUCHED))
    _expect(assemble([b"not a section blob"]), (E_ENCODE, "band sections: bad magic"))
    _expect(assemble([struct.pack("<I", 0x4253584a)]), (E_ENCODE, "band sections truncated"))
    _expect(assemble([struct.pack("<IIIIQQ", 0x4253584a, 1, 2, 0, 8, 100)]), (E_ENCODE, "band sections truncated"))
    _expect(assemble([struct.pack("<II", 0x4253584a, 0)]), (E_ENCODE, "histogram size"))


def test_refused_icc_profiles(abi):
    import icc_util
    m, lut = (C.c_float * 9)(), (C.c_float * 768)()
    parse = lambda icc: abi("JxlB200DebugParseIcc", _buf(icc), len(icc), m, lut, ErrorInfo)
    _expect(abi("JxlB200DebugParseIcc", None, 0, m, lut, ErrorInfo), (0, UNTOUCHED))
    assert parse(icc_util.make_matrix_icc(icc_util.P3_PRIMS))[0] == 1
    cmyk = bytearray(icc_util.make_matrix_icc(icc_util.P3_PRIMS)); cmyk[16:20] = b"CMYK"
    lab = bytearray(icc_util.make_matrix_icc(icc_util.P3_PRIMS)); lab[20:24] = b"Lab "
    for icc in (bytes(cmyk), bytes(lab), b"\0" * 64, b"\0" * 200):
        r, text = parse(icc)
        assert r == 0 and text is not UNTOUCHED and text, text


def test_encode_without_a_device(abi, no_device):
    bm, _hold = _bitmap()
    opts, meta = EncoderOptions(1.0, 3, False), (C.c_uint8 * 48)()
    io = IOCallbacks(Write(lambda p, n: 0), Seek(lambda p: 0))
    _expect(abi("SaveImage", C.byref(bm), C.byref(opts), meta, C.byref(io), ErrorInfo, None), (E_ENCODE, CUDA), no_device)
    _expect(abi("JxlB200EncodeToMemory", C.byref(bm), C.byref(opts), None, 0, C.byref(C.c_void_p()), C.byref(C.c_size_t()), ErrorInfo), (E_ENCODE, CUDA), no_device)
    flags = C.c_uint32()
    _expect(abi("JxlB200BandEncoderCreate", -1, C.byref(bm), 16, 0, 0, 0, C.byref(opts), None, 0, C.byref(flags), ErrorInfo), (None, CUDA), no_device)
    _expect(abi("JxlB200BandEncoderCreate", 0, C.byref(bm), 16, 0, 0, 0, C.byref(opts), None, 0, C.byref(flags), ErrorInfo), (None, "cudaSetDevice failed"))


# ---- the seeded sweep over the host-only entries
def _mutations(n=300, seed=20261021):
    seeds = _golden_files() + [_oversized(), _float_cmyk(), _two_blacks(), _layered()]
    seeds += [data for _, data in _spec_cases() if len(data) < 2000][:8]
    rng = random.Random(seed)
    for _ in range(n):
        s = bytearray(rng.choice(seeds))
        for _ in range(rng.randint(1, 4)):
            m = rng.random()
            if m < 0.6:
                s[rng.randrange(min(len(s), 256))] ^= 1 << rng.randrange(8)
            elif m < 0.8:
                s[rng.randrange(len(s))] = rng.randrange(256)
            elif m < 0.9:
                del s[rng.randrange(8, len(s)):]
            else:
                a = rng.randrange(len(s))
                s[a:a + 8] = bytes([0xff] * 8)
        yield bytes(s)


def _sweep(abi):
    rows = []
    for data in _mutations():
        row = [hashlib.sha1(data).hexdigest()[:12]]
        for name, out in (("JxlB200PeekInfo", (C.c_int32 * 8)()), ("JxlB200BandLayout", (C.c_int32 * 4)())):
            r, text = abi(name, _buf(data), len(data), out, ErrorInfo)
            row.append([r, None if text is UNTOUCHED else text])
        r, text = abi("JxlB200DebugSectionSizes", _buf(data), len(data), (C.c_uint64 * 65536)(), 65536, (C.c_int32 * 2)(), ErrorInfo)
        row.append([r, None if text is UNTOUCHED else text])
        rows.append(row)
    return rows


def test_host_only_entries_over_mutated_files(abi):
    want = json.load(open(GOLDEN))
    got = _sweep(abi)
    assert [r[0] for r in got] == [r[0] for r in want], "the mutated inputs changed: regenerate the golden file"
    diff = [(g, w) for g, w in zip(got, want) if g != w]
    assert not diff, diff[:5]
    statuses = {r[1][0] for r in want}
    assert {0, D_DECODE, D_SIGNATURE} <= statuses, statuses


if __name__ == "__main__" and "--write-golden" in sys.argv:
    sys.path.insert(0, os.path.dirname(HERE))
    sys.path.insert(0, HERE)
    import pkgload
    with open(GOLDEN, "w") as f:
        json.dump(_sweep(Abi(pkgload.load().LIB_PATH)), f, indent=0)
        f.write("\n")
