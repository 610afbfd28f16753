"""pdn-jpegxl_b200 — host-side mirror of the reference's managed interop layer, over ctypes.

`dotnet` is absent in this image, so the C# caller contract of the reference is restated here
in Python with the same names, argument meaning and error behaviour:

  JpegXLNative.LoadImage / SaveImage / GetLibJxlVersion   I/JpegXLNative.cs:23-126 (+ error mapping :128-239)
  DecoderImage (callback sink)                            I/DecoderImage.cs:41-263
  DecoderLayerData (pixel repack, alpha -> 8 bit)         I/DecoderLayerData.cs:26-105,164-992, I/TransparencyMapping.cs:19-55
  JpegXLLoad.Load (RGB24 (+A8) -> BGRA32 surface)         S/JpegXLLoad.cs:30-115,219-249
  EncoderOptions / QualityToDistanceLookupTable           I/EncoderOptions.cs:24-31, I/QualityToDistanceLookupTable.cs:26-65
  StreamIOCallbacks (HRESULT-returning Write/Seek)        I/StreamIOCallbacks.cs:52-114
  BitmapUtil2.EnumerateLockRects                          S/BitmapUtil2.cs:30-77

The native library (libJpegXLFileTypeIO_X64.so, built by build.py with nvcc for sm_100a) does all
codec work in CUDA kernels. It is loaded eagerly; if it is missing, importing this package fails
loudly — there is no Python or CPU fallback.
"""
import ctypes as C
import io
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_NAME = "libJpegXLFileTypeIO_X64.so"
LIB_PATH = os.path.join(_HERE, LIB_NAME)


class NativeLibraryMissing(ImportError):
    pass


if not os.path.exists(LIB_PATH):
    raise NativeLibraryMissing(
        "%s not found next to %s. Build it with `python pdn-jpegxl_b200/build.py` (nvcc, sm_100a). "
        "The engine has no CPU fallback." % (LIB_NAME, __file__))

os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")   # see abi.cu: one hardware queue per in-flight image stream
_lib = C.CDLL(LIB_PATH)


# ---- struct mirrors (I/BitmapData.cs, I/DecoderCallbacks.cs, I/ErrorInfo.cs, I/EncoderOptions.Marshaller.cs, I/IOCallbacks.cs) ----
class BitmapData(C.Structure):
    _fields_ = [("scan0", C.c_void_p), ("width", C.c_uint32), ("height", C.c_uint32), ("stride", C.c_uint32)]


class ErrorInfo(C.Structure):
    _fields_ = [("errorMessage", C.c_char * 256)]


class EncoderOptionsNative(C.Structure):
    _fields_ = [("distance", C.c_float), ("effort", C.c_int32), ("lossless", C.c_bool)]


class EncoderImageMetadataNative(C.Structure):
    _fields_ = [("exif", C.c_void_p), ("exifSize", C.c_size_t), ("iccProfile", C.c_void_p), ("iccProfileSize", C.c_size_t),
                ("xmp", C.c_void_p), ("xmpSize", C.c_size_t)]


SetBasicInfoFn = C.CFUNCTYPE(None, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_bool)
SetMetadataFn = C.CFUNCTYPE(C.c_bool, C.POINTER(C.c_uint8), C.c_size_t)
SetKnownColorProfileFn = C.CFUNCTYPE(C.c_bool, C.c_int32)
SetLayerDataFn = C.CFUNCTYPE(C.c_bool, C.POINTER(C.c_uint8), C.POINTER(C.c_char), C.c_size_t)
ProgressFn = C.CFUNCTYPE(C.c_bool, C.c_int32)
WriteFn = C.CFUNCTYPE(C.c_int32, C.POINTER(C.c_uint8), C.c_size_t)
SeekFn = C.CFUNCTYPE(C.c_int32, C.c_uint64)


class DecoderCallbacks(C.Structure):
    _fields_ = [("setBasicInfo", SetBasicInfoFn), ("setIccProfile", SetMetadataFn), ("setKnownColorProfile", SetKnownColorProfileFn),
                ("setExif", SetMetadataFn), ("setXmp", SetMetadataFn), ("setLayerData", SetLayerDataFn)]


class IOCallbacks(C.Structure):
    _fields_ = [("Write", WriteFn), ("Seek", SeekFn)]


EXPORTS = ["GetLibJxlVersion", "LoadImage", "SaveImage", "JxlB200LoadImageBgra", "JxlB200PeekInfo", "JxlB200DecodeBatch", "JxlB200EncodeToMemory",
           "JxlB200Free", "JxlB200LastStageTimes", "JxlB200KernelLaunchCount", "JxlB200DebugDecodeStage", "JxlB200CudaAvailable", "JxlB200BandLayout",
           "JxlB200DecodeBand", "JxlB200ReleaseMemory", "JxlB200DebugParseIcc", "JxlB200DecodeBatchSubmit", "JxlB200DecodeBatchWait", "JxlB200LoadImageLayers",
           "JxlB200BandEncoderCreate", "JxlB200BandEncoderTokenize", "JxlB200BandEncoderFinish", "JxlB200BandEncoderDestroy", "JxlB200AssembleBands", "JxlB200DebugSectionSizes",
           "JxlB200BandEncoderDebugStage"]

_lib.GetLibJxlVersion.restype = C.c_uint32
_lib.LoadImage.argtypes = [C.POINTER(DecoderCallbacks), C.c_void_p, C.c_size_t, C.POINTER(ErrorInfo)]
_lib.LoadImage.restype = C.c_int32
_lib.SaveImage.argtypes = [C.POINTER(BitmapData), C.POINTER(EncoderOptionsNative), C.POINTER(EncoderImageMetadataNative), C.POINTER(IOCallbacks),
                           C.POINTER(ErrorInfo), ProgressFn]
_lib.SaveImage.restype = C.c_int32
_lib.JxlB200LoadImageBgra.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(ErrorInfo)]
_lib.JxlB200LoadImageBgra.restype = C.c_int32
_lib.JxlB200PeekInfo.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(C.c_int32), C.POINTER(ErrorInfo)]
_lib.JxlB200LoadImageLayers.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.POINTER(C.c_int32), C.POINTER(ErrorInfo)]
_lib.JxlB200LoadImageLayers.restype = C.c_int32
_lib.JxlB200BandLayout.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(C.c_int32), C.POINTER(ErrorInfo)]
_lib.JxlB200BandLayout.restype = C.c_int32
_lib.JxlB200DecodeBand.argtypes = [C.c_int32, C.c_void_p, C.c_size_t, C.c_uint32, C.c_uint32, C.c_void_p, C.c_size_t, C.c_int32, C.POINTER(C.c_int32), C.POINTER(ErrorInfo)]
_lib.JxlB200DecodeBand.restype = C.c_int32
_lib.JxlB200PeekInfo.restype = C.c_int32
_lib.JxlB200DecodeBatch.argtypes = [C.c_int32, C.c_int32, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.POINTER(C.c_void_p), C.POINTER(C.c_size_t),
                                    C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_int32), C.POINTER(ErrorInfo)]
_lib.JxlB200DecodeBatch.restype = C.c_int32
_lib.JxlB200DecodeBatchSubmit.argtypes = [C.c_int32, C.c_int32, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.POINTER(C.c_void_p), C.POINTER(C.c_size_t),
                                          C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(ErrorInfo)]
_lib.JxlB200DecodeBatchSubmit.restype = C.c_void_p
_lib.JxlB200DecodeBatchWait.argtypes = [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(ErrorInfo)]
_lib.JxlB200DecodeBatchWait.restype = C.c_int32
_lib.JxlB200EncodeToMemory.argtypes = [C.POINTER(BitmapData), C.POINTER(EncoderOptionsNative), C.POINTER(EncoderImageMetadataNative), C.c_int32,
                                       C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.POINTER(ErrorInfo)]
_lib.JxlB200EncodeToMemory.restype = C.c_int32
_lib.JxlB200Free.argtypes = [C.c_void_p]
_lib.JxlB200LastStageTimes.argtypes = [C.POINTER(C.c_float)]
_lib.JxlB200KernelLaunchCount.restype = C.c_int64
_lib.JxlB200DebugDecodeStage.argtypes = [C.c_void_p, C.c_size_t, C.c_int32, C.c_void_p, C.c_int64, C.POINTER(C.c_int32), C.POINTER(ErrorInfo)]
_lib.JxlB200DebugDecodeStage.restype = C.c_int64
_lib.JxlB200CudaAvailable.argtypes = [C.POINTER(ErrorInfo)]
_lib.JxlB200CudaAvailable.restype = C.c_int32

# ---- enums (I/DecoderStatus.cs, I/EncoderStatus.cs, I/JpegXLImageChannelRepresentation.cs, I/KnownColorProfile.cs, I/HResult.cs) ----
DECODER_STATUS = ["Ok", "NullParameter", "InvalidParameter", "OutOfMemory", "HasAnimation", "HasMultipleFrames", "ImageDimensionExceedsInt32",
                  "UnsupportedChannelFormat", "CreateLayerError", "CreateMetadataError", "DecodeError", "MetadataError", "InvalidFileSignature"]
ENCODER_STATUS = ["Ok", "NullParameter", "OutOfMemory", "UserCancelled", "EncodeError", "WriteError"]
IMAGE_FORMAT = ["Gray", "Rgb", "Cmyk"]
CHANNEL_REPRESENTATION = ["Uint8", "Uint16", "Float16", "Float32"]
KNOWN_COLOR_PROFILE = ["Srgb", "LinearSrgb", "LinearGray", "GraySrgbTRC", "DisplayP3", "Rec709", "Rec2020Linear", "Rec2020PQ"]
S_OK, E_POINTER, E_ABORT, E_OUTOFMEMORY, SEEK_ERROR = 0, -2147467261, -2147467260, -2147024882, -2147024871
_DTYPES = [np.uint8, np.uint16, np.float16, np.float32]


class FormatException(Exception):
    """FormatException thrown by I/JpegXLNative.cs:128-239 for every non-Ok status."""

    def __init__(self, status, message):
        super().__init__(message)
        self.status = status


class OperationCanceledException(Exception):
    pass


class OutOfMemoryException(MemoryError):
    pass


# ---- QualityToDistanceLookupTable (I/QualityToDistanceLookupTable.cs:26-65) and EncoderOptions (I/EncoderOptions.cs:24-31) ----
def quality_to_distance(quality):
    q = int(quality)
    if q >= 30:
        return float(np.float32(0.1) + np.float32(100 - q) * np.float32(0.09))
    if q <= 8:
        return 15.0
    return float(np.float32(6.4) + np.float32(np.power(np.float32(2.5), np.float32(30 - q) / np.float32(5.0))) / np.float32(6.25))


class EncoderOptions:
    def __init__(self, quality=90, lossless=False, effort=7):
        self.distance = 0.0 if lossless else quality_to_distance(quality)
        self.lossless = bool(lossless)
        self.effort = int(effort)


class EncoderImageMetadata:
    def __init__(self, exif=None, icc=None, xmp=None):
        self.exif, self.icc, self.xmp = exif, icc, xmp


# ---- TransparencyMapping (I/TransparencyMapping.cs:19-55) ----
def alpha_to_eight_bit(alpha):
    a = np.asarray(alpha)
    if a.dtype == np.uint8:
        return a
    if a.dtype == np.uint16:
        return (a // 257).astype(np.uint8)
    if a.dtype == np.float16:   # evaluated in half precision, then truncated
        return (np.clip(a, np.float16(0), np.float16(1)) * np.float16(255)).astype(np.float16).astype(np.uint8)
    return (np.clip(a.astype(np.float32), np.float32(0), np.float32(1)) * np.float32(255)).astype(np.uint8)


def enumerate_lock_rects(width, height, bits_per_pixel):
    """BitmapUtil2.EnumerateLockRects (S/BitmapUtil2.cs:30-77): full-width strips under WIC's 4 GB lock limit."""
    stride = (width * bits_per_pixel + 7) >> 3
    copy_height = max(1, ((1 << 30) // 4) // stride)
    y = 0
    while y < height:
        yield (0, y, width, min(y + copy_height, height))
        y += copy_height


class DecoderLayerData:
    """I/DecoderLayerData.cs: splits the native interleaved buffer into a colour bitmap and an 8-bit alpha bitmap."""

    def __init__(self, pixels, name, width, height, fmt, representation, has_transparency):
        self.name = name
        ncolor = {"Gray": 1, "Rgb": 3, "Cmyk": 4}[fmt]
        nch = ncolor + (1 if has_transparency else 0)
        arr = np.frombuffer(pixels, dtype=_DTYPES[representation]).reshape(height, width, nch)
        self.interleaved = arr   # the native buffer as handed to setLayerData (tests compare it with the oracle's pixels)
        if fmt == "Cmyk" and representation != 0:
            raise FormatException("DecodeError", "unsupported CMYK channel representation")
        color = arr[..., :ncolor]
        if fmt == "Gray":
            color = np.repeat(color, 3, axis=2)   # gray is replicated to RGB (I/DecoderLayerData.cs:164-330)
        self.color = np.ascontiguousarray(color)
        self.transparency = alpha_to_eight_bit(np.ascontiguousarray(arr[..., ncolor])) if has_transparency else None
        self.format = fmt
        self.representation = representation


class DecoderImage:
    """I/DecoderImage.cs: the callback sink handed to the native LoadImage."""

    def __init__(self):
        self.width = self.height = 0
        self.format = None
        self.channel_representation = 0
        self.has_transparency = False
        self.icc_profile = None
        self.known_color_profile = None
        self.exif = None
        self.xmp = None
        self.layer_data = None
        self.exception = None
        self.callback_log = []
        self._cb = DecoderCallbacks(SetBasicInfoFn(self._set_basic_info), SetMetadataFn(self._set_icc), SetKnownColorProfileFn(self._set_known),
                                    SetMetadataFn(self._set_exif), SetMetadataFn(self._set_xmp), SetLayerDataFn(self._set_layer))

    def get_decoder_callbacks(self):
        return self._cb

    def _guard(self, fn):
        try:
            fn()
            return True
        except Exception as e:   # exceptions never cross the boundary (I/DecoderImage.cs:126-130)
            self.exception = e
            return False

    def _set_basic_info(self, w, h, fmt, rep, transparency):
        self.callback_log.append("setBasicInfo")
        self.width, self.height, self.format, self.channel_representation, self.has_transparency = w, h, IMAGE_FORMAT[fmt], rep, bool(transparency)

    def _set_icc(self, data, n):
        self.callback_log.append("setIccProfile")
        return self._guard(lambda: setattr(self, "icc_profile", C.string_at(data, n)))

    def _set_known(self, profile):
        self.callback_log.append("setKnownColorProfile")
        return self._guard(lambda: setattr(self, "known_color_profile", KNOWN_COLOR_PROFILE[profile]))

    def _set_exif(self, data, n):
        self.callback_log.append("setExif")
        return self._guard(lambda: setattr(self, "exif", C.string_at(data, n)))

    def _set_xmp(self, data, n):
        self.callback_log.append("setXmp")

        def keep_first():
            if self.xmp is None:   # managed side keeps the first packet (I/DecoderImage.cs:248)
                self.xmp = C.string_at(data, n)
        return self._guard(keep_first)

    def _set_layer(self, pixels, name, name_len):
        self.callback_log.append("setLayerData")

        def make():
            bps = [1, 2, 2, 4][self.channel_representation]
            ncolor = {"Gray": 1, "Rgb": 3, "Cmyk": 4}[self.format]
            nbytes = self.width * self.height * (ncolor + (1 if self.has_transparency else 0)) * bps
            layer_name = C.string_at(name, name_len).decode("utf-8") if name and name_len else None   # trailing NUL kept (Appendix C-3)
            self.layer_data = DecoderLayerData(C.string_at(pixels, nbytes), layer_name, self.width, self.height, self.format,
                                               self.channel_representation, self.has_transparency)
        return self._guard(make)


def _message(ei):
    return ei.errorMessage.decode("utf-8", "replace")


class JpegXLNative:
    """I/JpegXLNative.cs."""

    @staticmethod
    def GetLibJxlVersion():
        v = _lib.GetLibJxlVersion()
        return ((v >> 24) & 0xff, (v >> 16) & 0xff, (v >> 8) & 0xff)

    @staticmethod
    def LoadImage(data, decoder_image):
        buf = bytes(data)
        ei = ErrorInfo()
        cb = decoder_image.get_decoder_callbacks()
        status = _lib.LoadImage(C.byref(cb), buf, len(buf), C.byref(ei))
        if status != 0:
            JpegXLNative._handle_decoder_error(status, ei, decoder_image)

    @staticmethod
    def _handle_decoder_error(status, ei, decoder_image):
        name = DECODER_STATUS[status]
        if name in ("CreateLayerError", "CreateMetadataError") and decoder_image.exception is not None:
            raise decoder_image.exception
        if name == "OutOfMemory":
            raise OutOfMemoryException()
        msg = _message(ei)
        if name == "DecodeError" and msg:
            raise FormatException(name, msg)
        raise FormatException(name, {"InvalidFileSignature": "The file is not a valid JPEG XL image.", "DecodeError": "An error occurred when decoding the image.",
                                     "UnsupportedChannelFormat": "The image has an unsupported channel format.",
                                     "ImageDimensionExceedsInt32": "The image dimensions are too large."}.get(name, name))

    @staticmethod
    def SaveImage(surface_bgra, options, metadata, progress_callback, output_stream):
        surf = np.ascontiguousarray(surface_bgra, dtype=np.uint8)
        h, w, c = surf.shape
        assert c == 4
        bitmap = BitmapData(surf.ctypes.data, w, h, surf.strides[0])
        opts = EncoderOptionsNative(options.distance, options.effort, options.lossless)
        keep = []

        def blob(b):
            if not b:
                return None, 0
            arr = (C.c_uint8 * len(b)).from_buffer_copy(b)
            keep.append(arr)
            return C.cast(arr, C.c_void_p), len(b)

        meta = EncoderImageMetadataNative()
        meta.exif, meta.exifSize = blob(metadata.exif)
        meta.iccProfile, meta.iccProfileSize = blob(metadata.icc)
        meta.xmp, meta.xmpSize = blob(metadata.xmp)
        io_cb = StreamIOCallbacks(output_stream)
        native_io = io_cb.get_native()
        ei = ErrorInfo()
        ei.errorMessage = b"\xcc" * 255   # the managed caller passes it uninitialised (I/JpegXLNative.cs:102)
        prog = ProgressFn(progress_callback) if progress_callback else C.cast(None, ProgressFn)
        status = _lib.SaveImage(C.byref(bitmap), C.byref(opts), C.byref(meta), C.byref(native_io), C.byref(ei), prog)
        if status != 0:
            name = ENCODER_STATUS[status]
            if name == "UserCancelled":
                raise OperationCanceledException()
            if name == "OutOfMemory":
                raise OutOfMemoryException()
            if name == "WriteError" and io_cb.exception is not None:
                raise io_cb.exception
            msg = _message(ei) if name == "EncodeError" else ""
            raise FormatException(name, msg or name)


class StreamIOCallbacks:
    """I/StreamIOCallbacks.cs:52-114: Write/Seek over a stream, returning HRESULTs."""

    def __init__(self, stream):
        self.stream = stream
        self.exception = None
        self._w = WriteFn(self._write)
        self._s = SeekFn(self._seek)

    def get_native(self):
        return IOCallbacks(self._w, self._s)

    def _write(self, buf, n):
        if not buf:
            return E_POINTER
        try:
            self.stream.write(C.string_at(buf, n))
            return S_OK
        except Exception as e:
            self.exception = e
            return E_ABORT if isinstance(e, OperationCanceledException) else -2147467259

    def _seek(self, pos):
        try:
            self.stream.seek(pos)
            return S_OK
        except Exception as e:
            self.exception = e
            return SEEK_ERROR


class Document:
    def __init__(self, width, height):
        self.width, self.height = width, height
        self.surface = np.zeros((height, width, 4), np.uint8)   # BGRA32 (Paint.NET Surface)
        self.color_profile = None
        self.exif = None
        self.xmp = None
        self.layer_name = None


class JpegXLLoad:
    """S/JpegXLLoad.cs:30-115, 219-249 for the 8-bit Gray/RGB(A) path (the WIC / Direct2D branches are out of scope)."""

    @staticmethod
    def Load(data):
        image = DecoderImage()
        JpegXLNative.LoadImage(data, image)
        layer = image.layer_data
        doc = Document(image.width, image.height)
        doc.color_profile = image.known_color_profile or image.icc_profile
        doc.exif, doc.xmp, doc.layer_name = image.exif, image.xmp, layer.name
        if layer.format == "Cmyk" or layer.representation != 0:
            raise NotImplementedError("CMYK / >8-bit surfaces need the host's WIC colour conversion (S/JpegXLLoad.cs:146-172,312-319), out of scope")
        for (x0, y0, x1, y1) in enumerate_lock_rects(doc.width, doc.height, 24):
            src = layer.color[y0:y1, x0:x1]
            dst = doc.surface[y0:y1, x0:x1]
            dst[..., 0] = src[..., 2]   # SetLayerColorDataFromRgbImage: dst.B = src.B ... (S/JpegXLLoad.cs:219-241)
            dst[..., 1] = src[..., 1]
            dst[..., 2] = src[..., 0]
        doc.surface[..., 3] = layer.transparency if layer.transparency is not None else 255   # S/JpegXLLoad.cs:243-249,111
        return doc


class JpegXLSave:
    """S/JpegXLSave.cs:30-63."""

    @staticmethod
    def Save(surface_bgra, output_stream, quality=90, lossless=False, effort=7, progress_callback=None, exif=None, icc=None, xmp=None):
        JpegXLNative.SaveImage(surface_bgra, EncoderOptions(quality, lossless, effort), EncoderImageMetadata(exif, icc, xmp), progress_callback, output_stream)


# ---- extensions ----
def shard_indices(count, rank, world):
    """Multi-GPU partition of a batch (DESIGN.md §7): file i goes to rank i mod world; no collective on the data path."""
    return list(range(rank, count, world))



def cuda_available():
    ei = ErrorInfo()
    ok = _lib.JxlB200CudaAvailable(C.byref(ei))
    return bool(ok), _message(ei)


def peek_info(data):
    buf = bytes(data)
    info = (C.c_int32 * 8)()
    ei = ErrorInfo()
    st = _lib.JxlB200PeekInfo(buf, len(buf), info, C.byref(ei))
    if st != 0:
        raise FormatException(DECODER_STATUS[st], _message(ei) or DECODER_STATUS[st])
    return dict(width=info[0], height=info[1], format=IMAGE_FORMAT[info[2]], representation=info[3], has_transparency=bool(info[4]),
                num_channels=info[5], known_profile=(KNOWN_COLOR_PROFILE[info[6]] if info[6] >= 0 else None), is_container=bool(info[7]))


def load_image_bgra(data):
    info = peek_info(data)
    buf = bytes(data)
    out = np.empty((info["height"], info["width"], 4), np.uint8)
    w, h = C.c_int32(), C.c_int32()
    ei = ErrorInfo()
    st = _lib.JxlB200LoadImageBgra(buf, len(buf), out.ctypes.data, out.nbytes, C.byref(w), C.byref(h), C.byref(ei))
    if st != 0:
        raise FormatException(DECODER_STATUS[st], _message(ei) or DECODER_STATUS[st])
    return out


def load_image_layers(data):
    """JxlB200LoadImageLayers: the colour bitmap and the Alpha8 bitmap of I/DecoderLayerData.cs, split on the GPU. Returns (color, transparency | None)."""
    info = peek_info(data)
    buf = bytes(data)
    if info["format"] == "Cmyk" and info["representation"] != 0:
        raise FormatException("UnsupportedChannelFormat", "unsupported CMYK channel representation")
    ch = 4 if info["format"] == "Cmyk" else 3
    color = np.empty((info["height"], info["width"], ch), _DTYPES[info["representation"]])
    alpha = np.empty((info["height"], info["width"]), np.uint8) if info["has_transparency"] else None
    got = (C.c_int32 * 6)()
    ei = ErrorInfo()
    st = _lib.JxlB200LoadImageLayers(buf, len(buf), color.ctypes.data, color.nbytes, alpha.ctypes.data if alpha is not None else None,
                                     alpha.nbytes if alpha is not None else 0, got, C.byref(ei))
    if st != 0:
        raise FormatException(DECODER_STATUS[st], _message(ei) or DECODER_STATUS[st])
    assert (got[0], got[1], got[5]) == (info["width"], info["height"], ch)
    return color, alpha


def _native_metadata(metadata):
    """EncoderImageMetadata (N/Encoder/JxlEncoderTypes.h:35-42) from the Python-side metadata; returns it with the buffers to keep alive."""
    meta = EncoderImageMetadataNative()
    keep = []
    if metadata is not None:
        for field, size, b in (("exif", "exifSize", metadata.exif), ("iccProfile", "iccProfileSize", metadata.icc), ("xmp", "xmpSize", metadata.xmp)):
            if b:
                arr = (C.c_uint8 * len(b)).from_buffer_copy(b)
                keep.append(arr)
                setattr(meta, field, C.cast(arr, C.c_void_p))
                setattr(meta, size, len(b))
    return meta, keep


def encode_to_memory(surface_bgra, options, metadata=None, device_ptr=None, width=None, height=None, stride=None, host_array=None):
    """host_array: a 2-D uint8 array of `height` rows of `stride` bytes (BitmapData with stride > 4*width, N/Common.h:17-23)."""
    if host_array is not None:
        assert host_array.dtype == np.uint8 and host_array.flags.c_contiguous and host_array.shape == (height, stride)
        bitmap = BitmapData(host_array.ctypes.data, width, height, stride)
    elif device_ptr is None:
        surf = np.ascontiguousarray(surface_bgra, dtype=np.uint8)
        h, w, _ = surf.shape
        bitmap = BitmapData(surf.ctypes.data, w, h, surf.strides[0])
    else:
        bitmap = BitmapData(device_ptr, width, height, stride)
    opts = EncoderOptionsNative(options.distance, options.effort, options.lossless)
    meta, keep = _native_metadata(metadata)
    out = C.c_void_p()
    n = C.c_size_t()
    ei = ErrorInfo()
    st = _lib.JxlB200EncodeToMemory(C.byref(bitmap), C.byref(opts), C.byref(meta), 1 if device_ptr is not None else 0, C.byref(out), C.byref(n), C.byref(ei))
    if st != 0:
        raise FormatException(ENCODER_STATUS[st], _message(ei) or ENCODER_STATUS[st])
    data = C.string_at(out, n.value)
    _lib.JxlB200Free(out)
    return data


def debug_parse_icc(icc):
    """(3x3 matrix profile-RGB-linear -> linear sRGB, 3x256 tone curves) the encoder derives from a matrix/TRC ICC profile, or raises."""
    b = bytes(icc)
    m = (C.c_float * 9)()
    lut = (C.c_float * 768)()
    ei = ErrorInfo()
    _lib.JxlB200DebugParseIcc.restype = C.c_int32
    _lib.JxlB200DebugParseIcc.argtypes = [C.c_char_p, C.c_size_t, C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(ErrorInfo)]
    if not _lib.JxlB200DebugParseIcc(b, len(b), m, lut, C.byref(ei)):
        raise FormatException("EncodeError", _message(ei) or "unsupported ICC profile")
    return np.array(m, dtype=np.float64).reshape(3, 3), np.array(lut, dtype=np.float64).reshape(3, 256)


def release_memory():
    """Returns the engine's cached device / page-locked buffers to the driver."""
    _lib.JxlB200ReleaseMemory()


def band_layout(data):
    """(width, height, group size in pixels, number of group rows) of the first frame — what a caller shards over."""
    b = bytes(data)
    lay = (C.c_int32 * 4)()
    ei = ErrorInfo()
    st = _lib.JxlB200BandLayout(b, len(b), lay, C.byref(ei))
    if st != 0:
        raise FormatException(DECODER_STATUS[st], _message(ei) or DECODER_STATUS[st])
    return tuple(lay)


def band_partition(num_group_rows, world):
    """Contiguous group-row ranges per rank (SURVEY §8e): rank r decodes rows [begin, end); ranks beyond the row count get (0, 0)."""
    base, extra = divmod(num_group_rows, world)
    out, at = [], 0
    for r in range(world):
        n = base + (1 if r < extra else 0)
        out.append((at, at + n) if n else (0, 0))
        at += n
    return out


def decode_band(data, group_row_begin, group_row_end, bgra=False, device=-1):
    """Decodes group rows [begin, end) of the frame on `device`; returns the H_band x W x C array of those image rows."""
    b = bytes(data)
    info = peek_info(b)
    w, _, gdim, _ = band_layout(b)
    nch = 4 if bgra else info["num_channels"] + (1 if info["format"] == "Cmyk" else 0)
    dtype = np.uint8 if bgra else _DTYPES[info["representation"]]
    rows_cap = (group_row_end - group_row_begin) * gdim
    out = np.empty((rows_cap, w, nch), dtype)
    rows = C.c_int32()
    ei = ErrorInfo()
    st = _lib.JxlB200DecodeBand(device, b, len(b), group_row_begin, group_row_end, out.ctypes.data, out.nbytes, int(bgra), C.byref(rows), C.byref(ei))
    if st != 0:
        raise FormatException(DECODER_STATUS[st], _message(ei) or DECODER_STATUS[st])
    return out[: rows.value]


# ---- sharded encode (SURVEY §8e "Encode sharding"): bands of whole LF-group rows, one session per band / GPU
ENC_BAND_ROWS = 2048   # one LF-group row: 8 groups of 256 px


def encode_band_partition(height, world):
    """Contiguous bands of whole LF-group rows per rank: [(first_row, row_count)]; ranks beyond the LF-group rows get (0, 0)."""
    lf_rows = -(-height // ENC_BAND_ROWS)
    out = []
    for begin, end in band_partition(lf_rows, world):
        y0, y1 = begin * ENC_BAND_ROWS, min(end * ENC_BAND_ROWS, height)
        out.append((y0, y1 - y0) if end > begin else (0, 0))
    return out


def band_rows_with_halo(height, first_row, rows):
    """(first row to hand over, halo_top, halo_bottom) for a band: 8 rows of each neighbour (fewer at the end of the frame)."""
    halo_top = min(8, first_row)
    halo_bottom = min(8, height - (first_row + rows))
    return first_row - halo_top, halo_top, halo_bottom


_lib.JxlB200BandEncoderCreate.argtypes = [C.c_int32, C.POINTER(BitmapData), C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(EncoderOptionsNative),
                                          C.POINTER(EncoderImageMetadataNative), C.c_int32, C.POINTER(C.c_uint32), C.POINTER(ErrorInfo)]
_lib.JxlB200BandEncoderCreate.restype = C.c_void_p
_lib.JxlB200BandEncoderTokenize.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.POINTER(ErrorInfo)]
_lib.JxlB200BandEncoderTokenize.restype = C.c_int32
_lib.JxlB200BandEncoderFinish.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.POINTER(C.c_float), C.POINTER(ErrorInfo)]
_lib.JxlB200BandEncoderFinish.restype = C.c_int32
_lib.JxlB200BandEncoderDestroy.argtypes = [C.c_void_p]
_lib.JxlB200BandEncoderDestroy.restype = None
_lib.JxlB200BandEncoderDebugStage.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.POINTER(C.c_int64), C.POINTER(ErrorInfo)]
_lib.JxlB200BandEncoderDebugStage.restype = C.c_int64
_lib.JxlB200AssembleBands.argtypes = [C.c_uint32, C.c_uint32, C.POINTER(EncoderOptionsNative), C.POINTER(EncoderImageMetadataNative), C.c_uint32, C.c_void_p, C.c_size_t,
                                      C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.c_int32, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.POINTER(ErrorInfo)]
_lib.JxlB200AssembleBands.restype = C.c_int32


def _enc_check(st, ei):
    if st != 0:
        raise FormatException(ENCODER_STATUS[st], _message(ei) or ENCODER_STATUS[st])


class BandEncoder:
    """One band of a frame on one GPU (JxlB200BandEncoder*). `rows_bgra`: the rows handed over, halo rows included (H x W x 4 uint8)."""

    def __init__(self, rows_bgra, frame_height, first_row, halo_top, halo_bottom, options, device=-1, metadata=None):
        self._rows = np.ascontiguousarray(rows_bgra, dtype=np.uint8)
        h, w, _ = self._rows.shape
        bitmap = BitmapData(self._rows.ctypes.data, w, h - halo_top - halo_bottom, self._rows.strides[0])
        self._opts = EncoderOptionsNative(options.distance, options.effort, options.lossless)
        flags, ei = C.c_uint32(), ErrorInfo()
        meta, hold = _native_metadata(metadata) if metadata is not None else (None, None)   # the session keeps its own copy of the ICC profile
        self._h = _lib.JxlB200BandEncoderCreate(device, C.byref(bitmap), frame_height, first_row, halo_top, halo_bottom, C.byref(self._opts),
                                                C.byref(meta) if meta is not None else None, 0, C.byref(flags), C.byref(ei))
        del hold
        if not self._h:
            raise FormatException("EncodeError", _message(ei) or "band encoder")
        self.flags = int(flags.value)
        self.device_ms = 0.0

    def tokenize(self, frame_flags):
        p, n, ei = C.c_void_p(), C.c_size_t(), ErrorInfo()
        _enc_check(_lib.JxlB200BandEncoderTokenize(self._h, frame_flags, C.byref(p), C.byref(n), C.byref(ei)), ei)
        hist = np.frombuffer(C.string_at(p, n.value * 8), dtype=np.uint64).copy()
        _lib.JxlB200Free(p)
        return hist

    def finish(self, frame_hist):
        hist = np.ascontiguousarray(frame_hist, dtype=np.uint64)
        p, n, ms, ei = C.c_void_p(), C.c_size_t(), C.c_float(), ErrorInfo()
        _enc_check(_lib.JxlB200BandEncoderFinish(self._h, hist.ctypes.data, hist.size, C.byref(p), C.byref(n), C.byref(ms), C.byref(ei)), ei)
        blob = C.string_at(p, n.value)
        _lib.JxlB200Free(p)
        self.device_ms = float(ms.value)
        return blob

    # element type of each stage of JxlB200BandEncoderDebugStage (9, the tokens, is returned as (counts, tokens, Modular stream count))
    _STAGE_DTYPES = {0: np.float32, 1: np.float32, 2: np.float32, 3: np.uint8, 4: np.int8, 5: np.float32, 6: np.int32, 7: np.int16, 8: np.uint8}

    def debug_stage(self, which):
        """One device buffer of the session between tokenize() and finish(), shaped as the header documents."""
        dims, ei = (C.c_int64 * 4)(), ErrorInfo()
        _lib.JxlB200BandEncoderDebugStage(self._h, which, None, 0, dims, C.byref(ei))   # sizes the buffer (or fails with the reason)
        d = [int(v) for v in dims]
        if which == 9:
            nbytes = d[0] * 4 + d[1] * 8
        else:
            shape = tuple(v for v in d if v)
            if not shape:
                raise FormatException("EncodeError", _message(ei) or "debug stage unavailable")
            nbytes = int(np.prod(shape)) * np.dtype(self._STAGE_DTYPES[which]).itemsize
        buf = np.empty(max(nbytes, 1), np.uint8)
        n = _lib.JxlB200BandEncoderDebugStage(self._h, which, buf.ctypes.data, buf.size, dims, C.byref(ei))
        if n == 0 or n != nbytes:
            raise FormatException("EncodeError", _message(ei) or "debug stage unavailable")
        if which == 9:
            counts = buf[:d[0] * 4].view(np.uint32).copy()
            return counts, buf[d[0] * 4:nbytes].view(np.uint32).reshape(-1, 2).copy(), d[2]
        return buf[:nbytes].view(self._STAGE_DTYPES[which]).reshape(shape).copy()

    def close(self):
        if self._h:
            _lib.JxlB200BandEncoderDestroy(self._h)
            self._h = None

    def __del__(self):
        self.close()


def assemble_bands(width, height, options, frame_flags, frame_hist, blobs, metadata=None):
    opts = EncoderOptionsNative(options.distance, options.effort, options.lossless)
    hist = np.ascontiguousarray(frame_hist, dtype=np.uint64)
    keep = [bytes(b) for b in blobs]
    ptrs = (C.c_void_p * len(keep))(*[C.cast(C.c_char_p(b), C.c_void_p) for b in keep])
    sizes = (C.c_size_t * len(keep))(*[len(b) for b in keep])
    meta, hold = _native_metadata(metadata)
    out, n, ei = C.c_void_p(), C.c_size_t(), ErrorInfo()
    _enc_check(_lib.JxlB200AssembleBands(width, height, C.byref(opts), C.byref(meta), frame_flags, hist.ctypes.data, hist.size, ptrs, sizes, len(keep),
                                         C.byref(out), C.byref(n), C.byref(ei)), ei)
    data = C.string_at(out, n.value)
    _lib.JxlB200Free(out)
    del hold
    return data


def encode_in_bands(surface_bgra, options, num_bands, devices=None, metadata=None):
    """The sharded encoder driven from ONE process (tests; a single host that owns several GPUs): band i runs on devices[i % len]."""
    surf = np.ascontiguousarray(surface_bgra, dtype=np.uint8)
    h, w, _ = surf.shape
    encs = []
    for i, (y0, rows) in enumerate(encode_band_partition(h, num_bands)):
        if rows == 0:
            continue
        first, ht, hb = band_rows_with_halo(h, y0, rows)
        dev = -1 if not devices else devices[i % len(devices)]
        encs.append(BandEncoder(surf[first:y0 + rows + hb], h, y0, ht, hb, options, device=dev))
    flags = 0
    for e in encs:
        flags |= e.flags
    hists = [e.tokenize(flags) for e in encs]
    total = np.sum(np.stack(hists), axis=0, dtype=np.uint64)
    blobs = [e.finish(total) for e in encs]
    for e in encs:
        e.close()
    return assemble_bands(w, h, options, flags, total, blobs, metadata)


def encode_band_distributed(rows_bgra, width, height, first_row, rows, options, dist, device=-1, metadata=None, dst=0, group=None):
    """One rank's part of a sharded encode under torch.distributed (one process per GPU): this rank's band (rows handed over with their
    halo), two reductions (flags: MAX of bit fields via OR-able ints; histograms: SUM), a gather of the section blobs to `dst`, which
    returns the file (other ranks return None). Ranks with no rows (rows == 0) only take part in the reductions. The tensors are host
    tensors: `group` must be a group with a CPU backend (gloo) when the default group is NCCL-only."""
    import torch
    enc = None
    if rows:
        _, ht, hb = band_rows_with_halo(height, first_row, rows)
        enc = BandEncoder(rows_bgra, height, first_row, ht, hb, options, device=device)
    bits = torch.tensor([(enc.flags >> 0) & 1, (enc.flags >> 1) & 1] if enc else [0, 0], dtype=torch.int64)
    dist.all_reduce(bits, op=dist.ReduceOp.MAX, group=group)
    flags = int(bits[0].item()) | (int(bits[1].item()) << 1)
    words = torch.tensor([0], dtype=torch.int64)
    hist = enc.tokenize(flags) if enc else None
    if hist is not None:
        words[0] = hist.size
    dist.all_reduce(words, op=dist.ReduceOp.MAX, group=group)
    t = torch.zeros(int(words.item()), dtype=torch.int64)
    if hist is not None:
        t += torch.from_numpy(hist.astype(np.int64))
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    total = t.numpy().astype(np.uint64)
    blob = enc.finish(total) if enc else b""
    ms = enc.device_ms if enc else 0.0
    if enc:
        enc.close()
    gathered = [None] * dist.get_world_size() if dist.get_rank() == dst else None
    dist.gather_object(blob, gathered, dst=dst, group=group)
    if dist.get_rank() != dst:
        return None, ms
    return assemble_bands(width, height, options, flags, total, [b for b in gathered if b], metadata), ms


class BatchHandle:
    """A batch in flight (JxlB200DecodeBatchSubmit). Keeps the input bytes alive until wait()."""

    def __init__(self, handle, n, keep):
        self.handle, self.n, self.keep = handle, n, keep

    def wait(self, raise_on_error=True):
        statuses = (C.c_int32 * self.n)()
        ei = ErrorInfo()
        st = _lib.JxlB200DecodeBatchWait(self.handle, statuses, C.byref(ei))
        self.handle, self.keep = None, None
        if st != 0 and raise_on_error:
            raise FormatException(DECODER_STATUS[st], _message(ei) or DECODER_STATUS[st])
        return list(statuses)


def decode_batch_submit(datas, out_arrays=None, bgra=False, device=-1, max_in_flight=16, device_inputs=None, device_outputs=None, sizes=None, out_sizes=None):
    """Starts a batch and returns a BatchHandle at once. Host path: datas = list of bytes, out_arrays = list of writable numpy arrays.
    Device path: device_inputs/device_outputs = lists of int pointers. The buffers must stay valid until handle.wait() returns."""
    n = len(datas) if device_inputs is None else len(device_inputs)
    ptrs = (C.c_void_p * n)()
    lens = (C.c_size_t * n)()
    outs = (C.c_void_p * n)()
    olens = (C.c_size_t * n)()
    keep = []
    for i in range(n):
        if device_inputs is None:
            b = bytes(datas[i])
            keep.append(b)
            ptrs[i] = C.cast(C.c_char_p(b), C.c_void_p)
            lens[i] = len(b)
        else:
            ptrs[i] = device_inputs[i]
            lens[i] = sizes[i]
        if device_outputs is None:
            outs[i] = out_arrays[i].ctypes.data
            olens[i] = out_arrays[i].nbytes
        else:
            outs[i] = device_outputs[i]
            olens[i] = out_sizes[i]
    ei = ErrorInfo()
    h = _lib.JxlB200DecodeBatchSubmit(device, n, ptrs, lens, outs, olens, int(bgra), int(device_inputs is None), int(device_outputs is None), max_in_flight, C.byref(ei))
    if not h:
        raise FormatException("DecodeError", _message(ei) or "batch submit failed")
    return BatchHandle(h, n, keep)


def decode_batch(datas, out_arrays=None, bgra=False, device=-1, max_in_flight=16, device_inputs=None, device_outputs=None, sizes=None, out_sizes=None, raise_on_error=True):
    """Synchronous batch decode (submit + wait)."""
    return decode_batch_submit(datas, out_arrays, bgra, device, max_in_flight, device_inputs, device_outputs, sizes, out_sizes).wait(raise_on_error)


def section_sizes(data):
    """(sizes of the first frame's sections in logical TOC order, number of LF groups, number of groups) — host only."""
    b = bytes(data)
    out = (C.c_uint64 * 70000)()
    counts = (C.c_int32 * 2)()
    ei = ErrorInfo()
    _lib.JxlB200DebugSectionSizes.restype = C.c_int64
    _lib.JxlB200DebugSectionSizes.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_int64, C.POINTER(C.c_int32), C.POINTER(ErrorInfo)]
    n = _lib.JxlB200DebugSectionSizes(b, len(b), out, 70000, counts, C.byref(ei))
    if n == 0:
        raise FormatException("DecodeError", _message(ei) or "section sizes")
    return list(out[:n]), counts[0], counts[1]


def last_stage_times():
    t = (C.c_float * 8)()
    _lib.JxlB200LastStageTimes(t)
    return dict(zip(["h2d", "lf", "ac", "recon", "filters", "output", "d2h", "total"], list(t)))


def kernel_launch_count():
    return int(_lib.JxlB200KernelLaunchCount())


def debug_decode_stage(data, which, capacity):
    buf = bytes(data)
    out = np.empty(capacity, np.float32)
    dims = (C.c_int32 * 2)()
    ei = ErrorInfo()
    n = _lib.JxlB200DebugDecodeStage(buf, len(buf), which, out.ctypes.data, capacity, dims, C.byref(ei))
    if n == 0:
        raise FormatException("DecodeError", _message(ei) or "debug stage unavailable")
    return out[:n].copy(), (dims[0], dims[1])
