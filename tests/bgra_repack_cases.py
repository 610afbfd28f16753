"""The reference's BGRA repacks (N/Encoder/PixelFormatConversion.cpp:16-121: BgraToGray takes B, BgraToGrayAlpha B and A, BgraToRgb,
BgraToRgba), the seeded surfaces the tests feed them, and their stored outputs (tests/golden/bgra_repacks.json).

Provenance of the stored outputs: on exactly these surfaces the compiled reference (oracle/_ref, built from the reference's own
PixelFormatConversion.cpp) returned the same bytes as the restatement REPACKS below. test_bgra_repacks_match_numpy_restatement and the
padded-stride SaveImage test asserted that in the round-2 runs recorded in profiles/r02_summary.md (143 CPU and 200 GPU tests green).
The reference's sources are not part of this repository. Run `python tests/bgra_repack_cases.py` to rewrite the file. It uses the
compiled reference when oracle/_ref is built (oracle/Makefile, from the reference's sources at REF), and the restatement
otherwise; the file records which.
"""
import ctypes as C
import hashlib
import json
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN_PATH = os.path.join(HERE, "golden", "bgra_repacks.json")
REF_LIB_PATH = os.path.join(os.path.dirname(HERE), "oracle", "_ref", "libpixelformat_ref.so")

# function of the reference -> the channels of a BGRA pixel it keeps, in order
REPACKS = {"ref_BgraToGray": [0], "ref_BgraToGrayAlpha": [0, 3], "ref_BgraToRgb": [2, 1, 0], "ref_BgraToRgba": [2, 1, 0, 3]}
KIND_TO_REPACK = {"gray": "ref_BgraToGray", "graya": "ref_BgraToGrayAlpha", "rgb": "ref_BgraToRgb", "rgba": "ref_BgraToRgba"}
PIXELFORMAT_CASES = [(7, 5, 0), (33, 9, 12), (1, 1, 4)]                                               # w, h, pad
STRIDE_CASES = [(200, 150, 64, "rgba"), (333, 77, 20, "rgb"), (128, 96, 4, "gray"), (96, 64, 36, "graya")]   # w, h, pad, kind


def pixelformat_surface(w, h, pad):
    """(h, 4*w + pad) uint8 rows of random BGRA pixels plus padding."""
    return np.random.default_rng(w * h).integers(0, 256, (h, w * 4 + pad), dtype=np.uint8)


def stride_surface(w, h, pad, kind):
    """A padded BGRA surface whose content makes SaveImage pick `kind`: gray has r == g == b, opaque kinds have alpha 255."""
    buf = np.random.default_rng(w + pad).integers(0, 256, (h, 4 * w + pad), dtype=np.uint8)
    px = buf[:, :4 * w].reshape(h, w, 4)
    if kind in ("gray", "graya"):
        px[..., 1] = px[..., 0]
        px[..., 2] = px[..., 0]
    if kind in ("rgb", "gray"):
        px[..., 3] = 255
    else:
        px[0, 0, 3] = 17
    return buf


def restated(buf, w, fn):
    """REPACKS[fn] applied to a padded BGRA surface: (h, w, channels) uint8."""
    return np.ascontiguousarray(buf[:, :4 * w].reshape(buf.shape[0], w, 4)[..., REPACKS[fn]])


class _BitmapData(C.Structure):   # N/Common.h:17-23
    _fields_ = [("scan0", C.c_void_p), ("width", C.c_uint32), ("height", C.c_uint32), ("stride", C.c_uint32)]


def reference(buf, w, fn):
    """The compiled reference function on a padded BGRA surface, or None when oracle/_ref is not built."""
    if not os.path.exists(REF_LIB_PATH):
        return None
    h, stride = buf.shape
    out = np.zeros((h, w, len(REPACKS[fn])), np.uint8)
    bm = _BitmapData(buf.ctypes.data, w, h, stride)
    getattr(C.CDLL(REF_LIB_PATH), fn)(C.byref(bm), out.ctypes.data_as(C.c_void_p))
    return out


def pixelformat_key(w, h, pad, fn):
    return "pixelformat/%dx%d+%d/%s" % (w, h, pad, fn)


def stride_key(w, h, pad, kind):
    return "stride/%dx%d+%d/%s" % (w, h, pad, kind)


def load_golden():
    return json.load(open(GOLDEN_PATH))["outputs"]


def matches_golden(entry, got):
    """Stored outputs of the small surfaces are kept whole (hex), the larger ones as shape + SHA-256 of the bytes."""
    if list(got.shape) != entry["shape"]:
        return False
    if "hex" in entry:
        return got.tobytes() == bytes.fromhex(entry["hex"])
    return hashlib.sha256(got.tobytes()).hexdigest() == entry["sha256"]


def main():
    use_ref = os.path.exists(REF_LIB_PATH)
    run = reference if use_ref else restated
    outputs = {}
    for w, h, pad in PIXELFORMAT_CASES:
        buf = pixelformat_surface(w, h, pad)
        for fn in REPACKS:
            got = run(buf, w, fn)
            outputs[pixelformat_key(w, h, pad, fn)] = {"shape": list(got.shape), "hex": got.tobytes().hex()}
    for w, h, pad, kind in STRIDE_CASES:
        got = run(stride_surface(w, h, pad, kind), w, KIND_TO_REPACK[kind])
        outputs[stride_key(w, h, pad, kind)] = {"shape": list(got.shape), "sha256": hashlib.sha256(got.tobytes()).hexdigest()}
    source = ("compiled reference (oracle/_ref)" if use_ref else
              "restatement REPACKS; equal to the compiled reference on these surfaces in the recorded round-2 runs (see bgra_repack_cases.py)")
    with open(GOLDEN_PATH, "w") as f:
        json.dump({"source": source, "outputs": outputs}, f, indent=1, sort_keys=True)
        f.write("\n")
    print("wrote", GOLDEN_PATH, "from", source)


if __name__ == "__main__":
    main()
