/* pdn-jpegxl_b200 — C ABI of the drop-in native library (libJpegXLFileTypeIO_X64.so).
 *
 * The first block restates, byte for byte, the boundary of the reference's native DLL
 * "JxlFileTypeIO" so that the unchanged C# P/Invoke declarations bind to it:
 *   exports ............ N/JxlFileTypeIO.h:29-43   (callers: I/JpegXL_X64.cs:21-39, I/JpegXL_Arm64.cs:21-39)
 *   BitmapData etc. .... N/Common.h:17-60
 *   decoder types ...... N/Decoder/JxlDecoderTypes.h:17-71
 *   encoder types ...... N/Encoder/JxlEncoderTypes.h:17-42
 * (N/ = /root/reference/src/JxlFileTypeIO/, I/ = /root/reference/src/Interop/.)
 * __stdcall is a no-op on x86-64 / AArch64 System V, so the plain C declarations below are
 * ABI-identical to the reference's stdcall exports. Struct sizes on LP64: BitmapData 24,
 * EncoderOptions 12, EncoderImageMetadata 48, DecoderCallbacks 48, IOCallbacks 16, ErrorInfo 256.
 *
 * The second block ("extensions") adds entry points that do not exist in the reference; the
 * frozen three keep their exact behaviour. Every function runs its codec work as sm_100a CUDA
 * kernels; there is no CPU fallback — without a usable GPU, LoadImage returns DecodeError and
 * SaveImage returns EncodeError with a message saying so.
 */
#ifndef JXL_FILETYPE_IO_H_
#define JXL_FILETYPE_IO_H_

#include <stdbool.h>
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define JXLFT_API __declspec(dllexport)
#define JXLFT_CALL __stdcall
#else
#define JXLFT_API __attribute__((visibility("default")))
#define JXLFT_CALL
#endif

/* ---- N/Common.h:17-60 ---------------------------------------------------------------- */
typedef struct BitmapData { uint8_t* scan0; uint32_t width; uint32_t height; uint32_t stride; } BitmapData;
typedef struct ColorBgra { uint8_t b, g, r, a; } ColorBgra;
typedef int32_t ImageChannelRepresentation;  /* Uint8 = 0, Uint16, Float16, Float32 */
enum { JXLFT_Uint8 = 0, JXLFT_Uint16 = 1, JXLFT_Float16 = 2, JXLFT_Float32 = 3 };
typedef bool(JXLFT_CALL* ProgressProc)(int32_t progressPercentage);                        /* false = cancel */
typedef int32_t(JXLFT_CALL* WriteCallback)(const uint8_t* buffer, size_t sizeInBytes);     /* Windows HRESULT */
typedef int32_t(JXLFT_CALL* SeekCallback)(uint64_t position);                              /* Windows HRESULT, absolute */
typedef struct IOCallbacks { WriteCallback Write; SeekCallback Seek; } IOCallbacks;
typedef struct ErrorInfo { char errorMessage[256]; } ErrorInfo;                             /* <= 255 chars + NUL */

/* ---- N/Decoder/JxlDecoderTypes.h:17-71 ------------------------------------------------ */
typedef int32_t DecoderStatus;
enum { DecoderStatus_Ok = 0, DecoderStatus_NullParameter, DecoderStatus_InvalidParameter, DecoderStatus_OutOfMemory, DecoderStatus_HasAnimation,
       DecoderStatus_HasMultipleFrames, DecoderStatus_ImageDimensionExceedsInt32, DecoderStatus_UnsupportedChannelFormat, DecoderStatus_CreateLayerError,
       DecoderStatus_CreateMetadataError, DecoderStatus_DecodeError, DecoderStatus_MetadataError, DecoderStatus_InvalidFileSignature };
typedef int32_t DecoderImageFormat;  /* Gray = 0, Rgb, Cmyk */
typedef int32_t KnownColorProfile;   /* Srgb = 0, LinearSrgb, LinearGray, GraySrgbTRC, DisplayP3, Rec709, Rec2020Linear, Rec2020PQ */
typedef void(JXLFT_CALL* DecoderSetBasicInfo)(int32_t width, int32_t height, DecoderImageFormat format, ImageChannelRepresentation channelFormat, bool hasTransparency);
typedef bool(JXLFT_CALL* DecoderSetMetadata)(uint8_t* data, size_t length);
typedef bool(JXLFT_CALL* DecoderSetKnownColorProfile)(KnownColorProfile profile);
typedef bool(JXLFT_CALL* DecoderSetLayerData)(uint8_t* pixels, char* name, size_t nameLength);
typedef struct DecoderCallbacks {
  DecoderSetBasicInfo setBasicInfo; DecoderSetMetadata setIccProfile; DecoderSetKnownColorProfile setKnownColorProfile;
  DecoderSetMetadata setExif; DecoderSetMetadata setXmp; DecoderSetLayerData setLayerData;
} DecoderCallbacks;

/* ---- N/Encoder/JxlEncoderTypes.h:17-42 ------------------------------------------------ */
typedef int32_t EncoderStatus;
enum { EncoderStatus_Ok = 0, EncoderStatus_NullParameter, EncoderStatus_OutOfMemory, EncoderStatus_UserCanceled, EncoderStatus_EncodeError, EncoderStatus_WriteError };
typedef struct EncoderOptions { float distance; int32_t effort; bool lossless; } EncoderOptions;
typedef struct EncoderImageMetadata { uint8_t* exif; size_t exifSize; uint8_t* iccProfile; size_t iccProfileSize; uint8_t* xmp; size_t xmpSize; } EncoderImageMetadata;

/* ---- N/JxlFileTypeIO.h:29-43: the three frozen exports --------------------------------- */
/* Replaces N/JxlFileTypeIO.cpp:18-21. Packed (major<<24)|(minor<<16)|(patch<<8) of the libjxl release whose bitstream
 * behaviour the engine follows (unpacked by I/JpegXLNative.cs:40-42). */
JXLFT_API uint32_t JXLFT_CALL GetLibJxlVersion(void);
/* Replaces N/JxlFileTypeIO.cpp:23-30 -> DecoderReadImage (N/Decoder/JxlDecoder.cpp:796-852). Callbacks run on the calling
 * thread in the order setBasicInfo, (setKnownColorProfile | setIccProfile)?, setExif?, setXmp*, setLayerData. */
JXLFT_API DecoderStatus JXLFT_CALL LoadImage(DecoderCallbacks* callbacks, const uint8_t* data, size_t dataSize, ErrorInfo* errorInfo);
/* Replaces N/JxlFileTypeIO.cpp:32-41 -> EncoderWriteImage (N/Encoder/JxlEncoder.cpp:147-392). */
JXLFT_API EncoderStatus JXLFT_CALL SaveImage(const BitmapData* bitmap, const EncoderOptions* options, const EncoderImageMetadata* metadata,
                                              IOCallbacks* callbacks, ErrorInfo* errorInfo, ProgressProc progressCallback);

/* ======================================================================================= *
 * Extensions (not in the reference). Plain pointers and sizes only.                        *
 * ======================================================================================= */

/* Decode straight into a BGRA32 surface (stride = 4*width), fusing the managed repack passes the reference performs after
 * LoadImage returns: I/DecoderLayerData.cs:667-744 (+ I/TransparencyMapping.cs:19-32) and S/JpegXLLoad.cs:219-249.
 * On success *width and *height receive the (post-orientation) size; `surface` must hold width*height*4 bytes, which the
 * caller learns from JxlB200PeekInfo. Returns a DecoderStatus. */
JXLFT_API DecoderStatus JXLFT_CALL JxlB200LoadImageBgra(const uint8_t* data, size_t dataSize, uint8_t* surface, size_t surfaceBytes,
                                                         int32_t* width, int32_t* height, ErrorInfo* errorInfo);
/* Decode into the two bitmaps a layer is made of, fusing the managed repack of I/DecoderLayerData.cs:26-125 (Set*ImageData, :127-992)
 * and I/TransparencyMapping.cs:18-32: `color` receives Rgb24 / Rgb48 / Rgb48Half / Rgb96Float pixels (gray replicated into R, G, B) or
 * Cmyk32, `transparency` (may be NULL for images without alpha) the Alpha8 bitmap; both tightly packed. info[6] receives width, height,
 * DecoderImageFormat, ImageChannelRepresentation, hasTransparency and the channel count of the colour bitmap. */
JXLFT_API DecoderStatus JXLFT_CALL JxlB200LoadImageLayers(const uint8_t* data, size_t dataSize, uint8_t* color, size_t colorBytes,
                                                           uint8_t* transparency, size_t transparencyBytes, int32_t* info, ErrorInfo* errorInfo);
/* Header-only pass (pass 1 of DecoderReadImage, N/Decoder/JxlDecoder.cpp:412-793) without callbacks. info[8] receives:
 * width, height, DecoderImageFormat, ImageChannelRepresentation, hasTransparency, numChannels, KnownColorProfile or -1, isContainer. */
JXLFT_API DecoderStatus JXLFT_CALL JxlB200PeekInfo(const uint8_t* data, size_t dataSize, int32_t* info, ErrorInfo* errorInfo);

/* Band decode (BASELINE config 5, SURVEY §8e "gigapixel"): one rank's share of a frame that is sharded by group rows. JxlB200BandLayout
 * reports layout[4] = {width, height, group size in pixels (256 for VarDCT), number of group rows}; JxlB200DecodeBand decodes group rows
 * [groupRowBegin, groupRowEnd) on device `device` (-1: current) and writes image rows [groupRowBegin*groupDim, min(groupRowEnd*groupDim,
 * height)) to `out`, interleaved and tightly packed as LoadImage hands them to setLayerData (BGRA32 when bgra != 0); *rows receives the
 * row count. No exchange between ranks: each reconstructs one extra group row on either side (the 7-pixel filter halo). The image must
 * not carry an orientation other than identity. */
JXLFT_API DecoderStatus JXLFT_CALL JxlB200BandLayout(const uint8_t* data, size_t dataSize, int32_t* layout, ErrorInfo* errorInfo);
JXLFT_API DecoderStatus JXLFT_CALL JxlB200DecodeBand(int32_t device, const uint8_t* data, size_t dataSize, uint32_t groupRowBegin, uint32_t groupRowEnd,
                                                      uint8_t* out, size_t outBytes, int32_t bgra, int32_t* rows, ErrorInfo* errorInfo);

/* The engine caches device and page-locked buffers between calls (cudaMalloc costs more than a decode). This returns them to the
 * driver; call it when a burst of work is over. */
JXLFT_API void JXLFT_CALL JxlB200ReleaseMemory(void);

/* Host-only diagnostic: the colorant matrix (profile RGB, linear -> linear sRGB, 9 floats) and the three tone curves sampled at v/255
 * (768 floats) that SaveImage derives from a matrix/TRC ICC profile for lossy encoding. Returns 1 on success, 0 (with a message) when the
 * profile is not a matrix/TRC RGB profile. */
JXLFT_API int32_t JXLFT_CALL JxlB200DebugParseIcc(const uint8_t* icc, size_t iccSize, float* matrix9, float* lut768, ErrorInfo* errorInfo);

/* Batch decode (BASELINE config 3): `count` independent files, each decoded by the full single-image pipeline on its own
 * CUDA stream of device `device`; outputs[i] (host memory, outputBytes[i] bytes, interleaved as LoadImage delivers, or
 * BGRA32 when bgra != 0) are filled on return. statuses[i] receives a DecoderStatus per file. Returns the first non-Ok
 * status or Ok. hostInputs/hostOutputs = 0 means the pointers are device pointers (inputs already resident in HBM and
 * outputs left there: the configuration bench.py reports as `value`). */
JXLFT_API DecoderStatus JXLFT_CALL JxlB200DecodeBatch(int32_t device, int32_t count, const uint8_t* const* datas, const size_t* dataSizes,
                                                       uint8_t* const* outputs, const size_t* outputBytes, int32_t bgra,
                                                       int32_t hostInputs, int32_t hostOutputs, int32_t maxInFlight,
                                                       DecoderStatus* statuses, ErrorInfo* errorInfo);

/* Asynchronous form of JxlB200DecodeBatch: Submit starts the batch on internal host threads and returns at once (NULL + message on an
 * immediate failure); Wait blocks until every file is done, fills statuses[count] (may be NULL), frees the handle and returns the first
 * non-Ok status. The data, output and size arrays are copied by Submit; the buffers they point to must stay valid until Wait returns.
 * Several batches may be in flight on one device: a caller that submits the next batch before waiting for the previous one keeps the
 * GPU busy across the fill / drain of each batch (bench.py pipelines half-batches this way). */
typedef struct JxlB200Batch JxlB200Batch;
JXLFT_API JxlB200Batch* JXLFT_CALL JxlB200DecodeBatchSubmit(int32_t device, int32_t count, const uint8_t* const* datas, const size_t* dataSizes,
                                                            uint8_t* const* outputs, const size_t* outputBytes, int32_t bgra,
                                                            int32_t hostInputs, int32_t hostOutputs, int32_t maxInFlight, ErrorInfo* errorInfo);
JXLFT_API DecoderStatus JXLFT_CALL JxlB200DecodeBatchWait(JxlB200Batch* batch, DecoderStatus* statuses, ErrorInfo* errorInfo);

/* Encode a BGRA32 surface to a .jxl file in memory (same pipeline as SaveImage, no callbacks). *out is malloc'ed; free it
 * with JxlB200Free. deviceInput != 0: scan0 is a device pointer. Returns an EncoderStatus. */
JXLFT_API EncoderStatus JXLFT_CALL JxlB200EncodeToMemory(const BitmapData* bitmap, const EncoderOptions* options, const EncoderImageMetadata* metadata,
                                                          int32_t deviceInput, uint8_t** out, size_t* outSize, ErrorInfo* errorInfo);
JXLFT_API void JXLFT_CALL JxlB200Free(void* p);

/* Sharded encode (BASELINE config 5, SURVEY §8e "Encode sharding"; the reference hands the whole frame to libjxl in one process,
 * N/Encoder/JxlEncoder.cpp:128,367). A frame is cut into bands of whole LF-group rows (2048 pixel rows; the last band takes the rest);
 * each band is encoded by its own session, normally one per GPU / process:
 *   Create    band = the band's rows of the frame (width = frame width, height = rows of the band, scan0 = first row HANDED OVER, which is
 *             haloTop rows before the band's first row; haloTop = min(8, firstRow), haloBottom = min(8, rows of the frame below the band):
 *             the neighbouring bands' pixels the inverse-gaborish stencil reaches). Uploads and scans -> *bandFlags.
 *   Tokenize  frameFlags = OR of all bands' flags (the GetOutputPixelFormat decision of N/Encoder/JxlEncoder.cpp:33-77 is per frame)
 *             -> this band's token histograms (malloc'ed, histWords 64-bit counters; free with JxlB200Free).
 *   Finish    frameHist = element-wise SUM of all bands' histograms -> this band's sections as one opaque blob (free with JxlB200Free).
 * JxlB200AssembleBands then builds the file from the blobs of all bands (any order) on one rank. Two reductions (4 bytes, a few MB) are
 * the only exchange between ranks; the file is bit-identical to SaveImage's for the same frame. Returns NULL / an EncoderStatus. */
typedef struct JxlB200BandEncoder JxlB200BandEncoder;
JXLFT_API JxlB200BandEncoder* JXLFT_CALL JxlB200BandEncoderCreate(int32_t device, const BitmapData* band, uint32_t frameHeight, uint32_t firstRow, uint32_t haloTop,
                                                                   uint32_t haloBottom, const EncoderOptions* options, const EncoderImageMetadata* metadata,
                                                                   int32_t deviceInput, uint32_t* bandFlags, ErrorInfo* errorInfo);
JXLFT_API EncoderStatus JXLFT_CALL JxlB200BandEncoderTokenize(JxlB200BandEncoder* enc, uint32_t frameFlags, uint64_t** hist, size_t* histWords, ErrorInfo* errorInfo);
JXLFT_API EncoderStatus JXLFT_CALL JxlB200BandEncoderFinish(JxlB200BandEncoder* enc, const uint64_t* frameHist, size_t histWords, uint8_t** sections,
                                                             size_t* sectionBytes, float* deviceMs, ErrorInfo* errorInfo);
JXLFT_API void JXLFT_CALL JxlB200BandEncoderDestroy(JxlB200BandEncoder* enc);
JXLFT_API EncoderStatus JXLFT_CALL JxlB200AssembleBands(uint32_t width, uint32_t height, const EncoderOptions* options, const EncoderImageMetadata* metadata,
                                                         uint32_t frameFlags, const uint64_t* frameHist, size_t histWords, const uint8_t* const* bandSections,
                                                         const size_t* bandSectionBytes, int32_t bandCount, uint8_t** out, size_t* outSize, ErrorInfo* errorInfo);

/* Instrumentation for bench.py / tests: per-stage device times (ms) of the last single-image decode on this thread
 * (h2d, lf, ac, recon, filters, output, d2h, total), number of kernels launched by this process, and raw stage dumps of
 * one VarDCT decode for parity tests. Each call decodes the whole file, then copies one buffer out as floats:
 *   which = 4: the quantised AC coefficients, [group][channel X, Y, B][65536] (int16 values), cell-chunked: coefficient k of the
 *              cell (by, bx) of a group at ((by * 32 + bx) * 64 + k), a varblock's storage position p in its (p / 64)-th covered cell
 *              in raster order; cells outside the image are zero. Two-pass files hold the sum of both passes.
 *   which = 3: the LF planes the reconstruction reads, [3][yblocks][xblocks], after dequantisation, chroma-from-luma and adaptive
 *              LF smoothing (unsmoothed when the frame skips it or has at most 2 block rows or columns).
 *   which = 0: the XYB buffer, [3][ypad][xpad] (padded to whole 8x8 blocks). It holds the reconstruction (dequantisation, CfL, LLF
 *              and inverse transforms, before gaborish and EPF).
 * dims2 receives (xpad, ypad) for which = 0. Returns the element count written (<= capacity), or 0 when the file is not
 * VarDCT, the decode failed or the buffer is too small. */
JXLFT_API void JXLFT_CALL JxlB200LastStageTimes(float* ms8);
JXLFT_API int64_t JXLFT_CALL JxlB200KernelLaunchCount(void);
JXLFT_API int64_t JXLFT_CALL JxlB200DebugDecodeStage(const uint8_t* data, size_t dataSize, int32_t which, float* out, int64_t capacity, int32_t* dims2, ErrorInfo* errorInfo);
JXLFT_API int32_t JXLFT_CALL JxlB200CudaAvailable(ErrorInfo* errorInfo);
/* Host-only instrumentation: byte sizes of the first frame's sections in logical TOC order (LfGlobal, LF groups, HfGlobal, pass groups);
 * counts[2] = {LF groups, groups}. Returns the number of entries written or 0. */
JXLFT_API int64_t JXLFT_CALL JxlB200DebugSectionSizes(const uint8_t* data, size_t dataSize, uint64_t* sizes, int64_t capacity, int32_t* counts, ErrorInfo* errorInfo);

#ifdef __cplusplus
}
#endif
#endif /* JXL_FILETYPE_IO_H_ */
