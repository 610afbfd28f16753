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
#include "../../include/JxlFileTypeIO.h"
#include "dev/enc_frame.cuh"
#include "host/headers.h"
#include "host/modular_host.h"

// Failures are thrown: StatusError (host/bits.h) for those with their own DecoderStatus / EncoderStatus, any other std::exception for
// DecodeError / EncodeError with its text. abi.cu turns them into status codes.
namespace jxlgpu {

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
  ParsedInfo info;
  uint8_t* pixels = nullptr; size_t pixel_bytes = 0;   // pinned host memory (or device memory when device_output), owned by the job
  uint32_t out_width = 0, out_height = 0; StageTimes times;
  std::shared_ptr<DecodeJob> job;                       // keeps `pixels` alive
};
// Thrown for a layered (multi-frame) still where only a plain single frame can be decoded: the phased batch pipeline passes such a file
// to DecodeOnGpu, every other caller reports it as DecodeError.
struct LayeredStill : Error { LayeredStill(); };

// Parses headers + metadata only (pass 1 of the reference). Never touches the GPU.
ParsedInfo ParseInfo(const uint8_t* data, size_t size);
// Full decode on the GPU. Fails loudly (DecodeError with a message) when no CUDA device is usable: there is no CPU fallback.
DecodeResult DecodeOnGpu(const DecodeRequest& req);
// Asynchronous variant for batches: enqueue everything on `stream`, return without synchronising. DecodeFinish waits and reads the error word.
std::shared_ptr<DecodeJob> DecodeEnqueue(const DecodeRequest& req, cudaStream_t stream, bool lf_phase_only, bool defer_entropy);
void DecodeBundleLaunch(const std::vector<std::shared_ptr<DecodeJob>>& jobs, int phase);   // phase 1: pending LF launches, 2: pending AC launches (jobs share one stream)
void DecodeEnqueuePhase(const std::shared_ptr<DecodeJob>& job, int phase);   // phase 2: AC entropy kernels, 3: reconstruction + render; on failure the job's stream has drained
void DecodeReservePools(const std::shared_ptr<DecodeJob>& job, size_t count);   // pre-populate the caching pools with `count` more sets of this job's buffers
ParsedInfo DecodeBandLayout(const uint8_t* data, size_t size);
DecodeResult DecodeFinish(const std::shared_ptr<DecodeJob>& job);
struct SectionSizes { std::vector<uint64_t> sizes; uint32_t num_lf_groups = 0, num_groups = 0; };
SectionSizes DecodeSectionSizes(const uint8_t* data, size_t size);
// stage dumps for parity tests (3 planes xpad*ypad floats or coefficient ints), copied to host
bool DecodeDebugPlanes(const std::shared_ptr<DecodeJob>& job, int which, std::vector<float>* out, int* xpad, int* ypad);
bool DecodeDebugCoeffs(const std::shared_ptr<DecodeJob>& job, std::vector<int16_t>* out);

bool CudaAvailable(std::string* why);
void TrimPools();

// A buffer from the engine's caching pools: device memory of the device current at Alloc, or page-locked host memory with pinned = true
// (cudaMalloc / cudaHostAlloc cost more than a decode or most encoder kernels; cudaFree also synchronises). It goes back to the pool it
// came from, and only after the work that uses it has been synchronised (the jobs and sessions sync their stream before they let go).
class Pool;
struct Buf { void* p = nullptr; size_t n = 0; Pool* pool = nullptr; void Alloc(size_t bytes, bool pinned = false); void Free();   // Alloc throws std::bad_alloc when the pool cannot get the memory
  void Swap(Buf& o) { std::swap(p, o.p); std::swap(n, o.n); std::swap(pool, o.pool); } template <class T> T* as() const { return static_cast<T*>(p); }
  Buf() {} ~Buf() { Free(); } Buf(const Buf&) = delete; Buf& operator=(const Buf&) = delete; };

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
struct EncodeResult { std::vector<uint8_t> file; StageTimes times; };
EncodeResult EncodeOnGpu(const EncodeRequest& req);

// Everything that depends on the frame only (size, options, pixel format), never on pixels.
struct EncPlan {
  bool lossless = false, is_gray = false, has_alpha = false; int ncolor = 3, num_ec = 0, nplanes = 0;
  ImageMetadata m; FrameHeader fh;
  Tree tree; std::vector<Token> tree_tokens; EncCode tree_code; size_t nleaves = 0; std::vector<uint16_t> leaf_lut;
  EncOptions mopt, aopt; uint32_t global_scale = 1, quant_lf = 16; float q_ac = 1;
  bool groups_have_modular = false, global_has_modular = false, single = false, aq = false, cfl = false; GroupHeader plain, gheader;
  size_t HistWords() const;
};

// kind: 0 global Modular stream, 1 LF group, 2 pass group. The payload is either owned (`bytes`) or a view into a band's serialised blob.
struct BandSection { uint32_t kind = 0, index = 0; uint64_t bits = 0; std::vector<uint8_t> bytes; const uint8_t* view = nullptr; size_t view_n = 0;
  const uint8_t* data() const { return view ? view : bytes.data(); } size_t size() const { return view ? view_n : bytes.size(); } };

// The encoder as three steps over a band of the frame (encode_engine.cu); SaveImage runs it over a single band, the sharded encode
// (JxlB200BandEncoder*) over one band per GPU, with AssembleBands writing the file from the sections of all bands.
class BandEncoder {
 public:
  explicit BandEncoder(const EncodeRequest& r) : req(r) {}
  ~BandEncoder() { if (st) { cudaStreamSynchronize(st); cudaStreamDestroy(st); } }
  uint32_t Begin();                                         // -> flags of this band (bit 0: a non-gray pixel, bit 1: a non-opaque pixel)
  std::vector<uint64_t> Tokenize(uint32_t frame_flags);     // -> this band's histograms, [context][kEncAlphabet] (Modular contexts, then AC contexts)
  std::vector<BandSection> Finish(const std::vector<uint64_t>& frame_hist);
  std::vector<uint8_t> FinishBlob(const std::vector<uint64_t>& frame_hist);   // Finish, serialised for AssembleBands
  int64_t DebugStage(int32_t which, void* out, int64_t capacity, int64_t* dims4);   // JxlB200BandEncoderDebugStage
  const EncPlan& Plan() const { return plan; }
  float device_ms = 0;

 private:
  // device_ms only: its calls are not checked
  struct Timer { cudaEvent_t a, b; cudaStream_t s; float* acc; Timer(cudaStream_t st_, float* acc_) : s(st_), acc(acc_) { cudaEventCreate(&a); cudaEventCreate(&b); cudaEventRecord(a, s); }
    ~Timer() { cudaEventRecord(b, s); cudaEventSynchronize(b); float ms = 0; cudaEventElapsedTime(&ms, a, b); *acc += ms; cudaEventDestroy(a); cudaEventDestroy(b); } };
  EncodeRequest req; cudaStream_t st = nullptr; EncPlan plan; DEncFrame e; FrameHeader fb;   // fb: frame header of the band taken as an image of its own (group / LF-group layout)
  uint32_t frame_h = 0, lf_group0 = 0, group0 = 0;      // frame height; index of the band's first LF group / first group in the frame
  const uint8_t* d_bgra = nullptr;                       // first row of the band itself (halo rows lie before it)
  Buf d_in, d_flags, d_e, d_xyb, d_tmp1, d_tmp2, d_planes, d_lf, d_lfq, d_coeffs, d_nz, d_dq, d_order, d_tokens, d_account, d_lut, d_modstreams, d_streams, d_hist_m, d_hist_a, d_bytes, d_bits, d_gabframe, d_srclut, d_hfm, d_ytox, d_ytob, d_stats;
  std::vector<DEncModStream> mod_streams; std::vector<DEncStream> m_streams, a_streams; std::vector<uint32_t> ac_counts;
  uint32_t first_lf_stream = 0, first_group_stream = 0, max_mod_tokens = 0; uint64_t byte_cursor = 0;
  std::vector<std::vector<Token>> hfmeta_tokens; std::vector<uint32_t> hfmeta_nb;
  bool stages_valid = false;                             // between Tokenize and Finish: k_enc_ans overwrites the token words in place
};
// The file from the serialised sections of every band of a frame (any order).
std::vector<uint8_t> AssembleBands(const EncodeRequest& frame, uint32_t frame_flags, const uint64_t* frame_hist, size_t words, const uint8_t* const* blobs, const size_t* sizes, size_t count);

}  // namespace jxlgpu
