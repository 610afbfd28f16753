// pdn-jpegxl_b200 engine — internal C++ interface between the C-ABI layer (abi.cc) and the
// CUDA decode / encode pipelines. Nothing here is exported; the exported surface is
// include/JxlFileTypeIO.h (the reference's N/JxlFileTypeIO.h:29-43 plus documented extensions).
#pragma once
#include <cstdint>
#include <cstddef>
#include <string>
#include <vector>
#include <memory>
#include <cuda_runtime.h>

namespace jxlgpu {

enum class Status : int32_t { Ok = 0, NullParameter, InvalidParameter, OutOfMemory, HasAnimation, HasMultipleFrames, ImageDimensionExceedsInt32, UnsupportedChannelFormat,
                              CreateLayerError, CreateMetadataError, DecodeError, MetadataError, InvalidFileSignature };

struct ParsedInfo {
  uint32_t group_dim = 0, num_group_rows = 0;   // frame group size in pixels and number of group rows (band decode layout)   // what pass 1 of the reference reports (N/Decoder/JxlDecoder.cpp:412-793)
  uint32_t width = 0, height = 0; int format = 1; int sample_type = 0; bool has_alpha = false; int num_channels = 3;
  int known_profile = -1; std::vector<uint8_t> icc; bool is_container = false; bool has_exif = false; std::vector<uint8_t> exif; std::vector<std::vector<uint8_t>> xmp;
  std::string frame_name; double bpp = 0;
};

struct DecodeRequest {
  const uint8_t* data = nullptr; size_t size = 0;
  bool bgra = false;            // fused BGRA32 surface output (extension; replaces I/DecoderLayerData.cs + S/JpegXLLoad.cs:219-249 passes)
  bool device_output = false;   // leave pixels in device memory (bench `value`: inputs/outputs resident in HBM)
  const uint8_t* device_input = nullptr;   // optional: the same file bytes already resident in device memory
  int device = -1;              // -1: current device
  uint8_t* out_device = nullptr;    // optional: decode straight into this device buffer (out_capacity bytes)
  uint8_t* out_pinned = nullptr;    // optional: copy the pixels straight into this page-locked host buffer (out_capacity bytes)
  size_t out_capacity = 0;
  uint32_t band_begin = 0, band_end = 0;   // band decode: output only group rows [band_begin, band_end) of the frame (0,0 = whole frame); needs orientation 1
  // Layer of a multi-frame still (internal, set by DecodeOnGpu): decode the frame whose header starts at byte layer_pos of the codestream into float
  // samples of the output encoding (interleaved colour [+ alpha], the frame's own size, device memory): no orientation, no unpremultiply.
  bool layer = false; size_t layer_pos = 0;
  int ac_lanes = 0;                 // AC sections walked per warp (power of two, 1..32); 0: 1 (lowest latency). Batches raise it for throughput.
};

struct StageTimes { float h2d = 0, lf = 0, ac = 0, recon = 0, filters = 0, output = 0, d2h = 0, total = 0; };

class DecodeJob;   // opaque
struct DecodeResult {
  Status status = Status::Ok; std::string message; ParsedInfo info;
  uint8_t* pixels = nullptr; size_t pixel_bytes = 0;   // pinned host memory (or device memory when device_output), owned by the job
  uint32_t out_width = 0, out_height = 0; StageTimes times;
  bool layered = false;   // DecodeEnqueue only: the file is a layered (multi-frame) still, which the phased batch pipeline does not decode — use DecodeOnGpu
  std::shared_ptr<DecodeJob> job;                       // keeps `pixels` alive
};

// Parses headers + metadata only (pass 1 of the reference). Never touches the GPU.
DecodeResult ParseInfo(const uint8_t* data, size_t size);
// Full decode on the GPU. Fails loudly (DecodeError with a message) when no CUDA device is usable: there is no CPU fallback.
DecodeResult DecodeOnGpu(const DecodeRequest& req);
// Asynchronous variant for batches: enqueue everything on `stream`, return without synchronising. Finish() waits and reads the error word.
std::shared_ptr<DecodeJob> DecodeEnqueue(const DecodeRequest& req, cudaStream_t stream, DecodeResult* res, bool lf_phase_only = false, bool defer_entropy = false);
void DecodeBundleLaunch(const std::vector<std::shared_ptr<DecodeJob>>& jobs, int phase);   // phase 1: pending LF launches, 2: pending AC launches (jobs share one stream)
bool DecodeEnqueuePhase(std::shared_ptr<DecodeJob>& job, int phase, DecodeResult* res);   // phase 2: AC entropy kernels, 3: reconstruction + render; false: job failed (res filled, job released)
bool DecodeStreamIdle(const std::shared_ptr<DecodeJob>& job);
void DumpPoolStats();
void DecodeReservePools(const std::shared_ptr<DecodeJob>& job, size_t count);   // pre-populate the caching pools with `count` more sets of this job's buffers
void DecodeStreamSync(const std::shared_ptr<DecodeJob>& job);
Status DecodeBandLayout(const uint8_t* data, size_t size, ParsedInfo* info, std::string* message);
void DecodeFinish(const std::shared_ptr<DecodeJob>& job, DecodeResult* res);
Status DecodeSectionSizes(const uint8_t* data, size_t size, std::vector<uint64_t>* sizes, uint32_t* num_lf_groups, uint32_t* num_groups, std::string* message);
// stage dumps for parity tests (3 planes xpad*ypad floats or coefficient ints), copied to host
bool DecodeDebugPlanes(const std::shared_ptr<DecodeJob>& job, int which, std::vector<float>* out, int* xpad, int* ypad);
bool DecodeDebugCoeffs(const std::shared_ptr<DecodeJob>& job, std::vector<int16_t>* out);

bool CudaAvailable(std::string* why);
void TrimPools();
void DumpHostTrace();
void* PinnedGet(size_t bytes);            // cached page-locked host memory (cudaHostAlloc costs far more than a decode)
void PinnedPut(void* p, size_t bytes);
void* DeviceGet(size_t bytes, void** pool_token);   // cached device memory of the current device (the encoder allocates ~25 buffers per call)
void DevicePut(void* p, size_t bytes, void* pool_token);

// ---- encoder
struct EncodeRequest {
  const uint8_t* bgra = nullptr; uint32_t width = 0, height = 0, stride = 0;   // BitmapData (N/Common.h:17-23)
  float distance = 1.0f; int effort = 7; bool lossless = false;
  const uint8_t* exif = nullptr; size_t exif_size = 0; const uint8_t* icc = nullptr; size_t icc_size = 0; const uint8_t* xmp = nullptr; size_t xmp_size = 0;
  bool device_input = false;   // bgra points at device memory (bench)
  // Band of a larger frame (sharded encode, DESIGN.md §7): `height` rows starting at frame row band_y0 of a frame_height-row frame; `bgra` points at
  // the first of halo_top rows that precede the band's own rows, halo_bottom rows follow them. frame_height == 0: the bitmap is the whole frame.
  uint32_t frame_height = 0, band_y0 = 0, halo_top = 0, halo_bottom = 0;
};
enum class EncStatus : int32_t { Ok = 0, NullParameter, OutOfMemory, UserCanceled, EncodeError, WriteError };
struct EncodeResult { EncStatus status = EncStatus::Ok; std::string message; std::vector<uint8_t> file; StageTimes times; int pixel_format = 2; /* 0 Gray 1 GrayAlpha 2 Rgb 3 Rgba */ };
EncodeResult EncodeOnGpu(const EncodeRequest& req);
// Sharded encode: one session per band (one per GPU), three steps with two small reductions between them, then AssembleBands on one rank.
struct BandSession;
BandSession* BandEncoderCreate(const EncodeRequest& band, uint32_t* band_flags, EncStatus* status, std::string* message);
EncStatus BandEncoderTokenize(BandSession* s, uint32_t frame_flags, std::vector<uint64_t>* band_hist, std::string* message);
EncStatus BandEncoderFinish(BandSession* s, const uint64_t* frame_hist, size_t words, std::vector<uint8_t>* sections, float* device_ms, std::string* message);
void BandEncoderDestroy(BandSession* s);
// Stage dump of a session between Tokenize and Finish (JxlB200BandEncoderDebugStage): bytes written, or 0 with a message.
int64_t BandEncoderDebugStage(BandSession* s, int32_t which, void* out, int64_t capacity, int64_t* dims4, std::string* message);
EncStatus AssembleBands(const EncodeRequest& frame, uint32_t frame_flags, const uint64_t* frame_hist, size_t words, const uint8_t* const* blobs, const size_t* sizes, size_t count,
                        std::vector<uint8_t>* file, std::string* message);

}  // namespace jxlgpu
