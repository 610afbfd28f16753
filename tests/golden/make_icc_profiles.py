"""Regenerates the two ICC profiles in this directory that stand in for the ones the reference ships (S/ColorProfiles/
Rec709-elle-V4-rec709.icc, 1180 B, and Rec2020-elle-V4-g10.icc, 1232 B; used by I/DecoderImage.cs:166-184).

The reference's files are third-party data that this repository does not carry. They were written by LittleCMS 2 following Elle Stone's
make-elles-profiles.c. This script uses the same library and the same recipe, so the stored profiles are written by a tool independent
of this project: v4 matrix/TRC profiles of D65 white adapted to D50 by LittleCMS (chad), with the Rec.709 primaries and the BT.709 curve
as a parametric curve (LittleCMS type 4 = ICC 'para' type 3), and the Rec.2020 primaries with a linear curve. Texts and dates are not the
reference's, so the bytes differ from the reference's files.

Needs a LittleCMS 2 shared library (the one Pillow bundles is found automatically, or pass its path).
Run: python tests/golden/make_icc_profiles.py [path/to/liblcms2.so]
"""
import ctypes as C
import glob
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
D65 = (0.3127, 0.3290)
PROFILES = {
    "Rec709-V4-rec709.icc": dict(prims=((0.640, 0.330), (0.300, 0.600), (0.150, 0.060)), curve=(4, (1 / 0.45, 1 / 1.099, 0.099 / 1.099, 1 / 4.5, 0.081)),
                                 desc="Rec.709 primaries, BT.709 tone curve (ICC v4)"),
    "Rec2020-V4-g10.icc": dict(prims=((0.708, 0.292), (0.170, 0.797), (0.131, 0.046)), curve=(1, (1.0,)),
                               desc="Rec.2020 primaries, linear tone curve (ICC v4)"),
}


class xyY(C.Structure):
    _fields_ = [("x", C.c_double), ("y", C.c_double), ("Y", C.c_double)]


def find_lcms():
    if len(sys.argv) > 1:
        return sys.argv[1]
    import PIL
    hits = glob.glob(os.path.join(os.path.dirname(os.path.dirname(PIL.__file__)), "pillow.libs", "liblcms2*"))
    return hits[0] if hits else "liblcms2.so.2"


def main():
    L = C.CDLL(find_lcms())
    L.cmsBuildParametricToneCurve.restype = C.c_void_p
    L.cmsBuildParametricToneCurve.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_double)]
    L.cmsCreateRGBProfile.restype = C.c_void_p
    L.cmsCreateRGBProfile.argtypes = [C.POINTER(xyY), C.POINTER(xyY * 3), C.POINTER(C.c_void_p * 3)]
    L.cmsSetProfileVersion.argtypes = [C.c_void_p, C.c_double]
    L.cmsMLUalloc.restype = C.c_void_p
    L.cmsMLUalloc.argtypes = [C.c_void_p, C.c_uint32]
    L.cmsMLUsetASCII.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p, C.c_char_p]
    L.cmsWriteTag.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p]
    L.cmsSaveProfileToMem.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_uint32)]
    L.cmsCloseProfile.argtypes = [C.c_void_p]
    L.cmsFreeToneCurve.argtypes = [C.c_void_p]
    L.cmsMLUfree.argtypes = [C.c_void_p]
    L.cmsSetHeaderFlags.argtypes = [C.c_void_p, C.c_uint32]
    sig = lambda s: int.from_bytes(s, "big")
    for name, p in PROFILES.items():
        ctype, params = p["curve"]
        curve = L.cmsBuildParametricToneCurve(None, ctype, (C.c_double * len(params))(*params))
        white = xyY(D65[0], D65[1], 1.0)
        prims = (xyY * 3)(*[xyY(x, y, 1.0) for x, y in p["prims"]])
        h = L.cmsCreateRGBProfile(C.byref(white), C.byref(prims), C.byref((C.c_void_p * 3)(curve, curve, curve)))
        L.cmsSetProfileVersion(h, C.c_double(4.3))
        for tag, text in ((b"desc", p["desc"]), (b"cprt", "No copyright, use freely")):
            mlu = L.cmsMLUalloc(None, 1)
            L.cmsMLUsetASCII(mlu, b"en", b"US", text.encode())
            L.cmsWriteTag(h, sig(tag), mlu)
            L.cmsMLUfree(mlu)
        n = C.c_uint32()
        L.cmsSaveProfileToMem(h, None, C.byref(n))
        buf = C.create_string_buffer(n.value)
        L.cmsSaveProfileToMem(h, buf, C.byref(n))
        L.cmsCloseProfile(h)
        L.cmsFreeToneCurve(curve)
        data = bytearray(buf.raw[:n.value])
        data[24:36] = bytes(12)   # creation date: zero, so the file depends only on the recipe and the library version
        open(os.path.join(HERE, name), "wb").write(bytes(data))
        print(name, len(data), "bytes")


if __name__ == "__main__":
    main()
