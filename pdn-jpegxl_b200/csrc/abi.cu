// pdn-jpegxl_b200 engine — the C-ABI layer: LoadImage / SaveImage / GetLibJxlVersion with the
// exact observable behaviour of the reference's native DLL, plus the documented extensions.
//   LoadImage  restates DecoderReadImage           N/Decoder/JxlDecoder.cpp:796-852 (callback order :461-784, :389-400)
//   SaveImage  restates EncoderWriteImage          N/Encoder/JxlEncoder.cpp:147-392 and OutputProcessor (N/Encoder/OutputProcessor.cpp:18-151)
//   error text restates SetErrorMessage            N/Common.cpp:18-53
// No exception crosses the boundary: Guard turns every failure into a status code (+ optional message).
#include "../../include/JxlFileTypeIO.h"
#include "engine.h"
#include "dev/kernels.h"
#include "host/icc.h"
#include <cstring>
#include <cstdlib>
#include <algorithm>
#include <deque>
#include <memory>
#include <thread>
#include <map>
#include <chrono>
#include <mutex>
#include <atomic>
#include <stdexcept>

using namespace jxlgpu;

namespace {

// More hardware work queues than the default 8, so that the per-image CUDA streams of a batch do not share (and serialise on) a queue.
// Only effective when set before the process creates its CUDA context; never overrides the user's own setting.
struct EnvInit { EnvInit() { setenv("CUDA_DEVICE_MAX_CONNECTIONS", "32", 0); } } g_env_init;

void SetErrorMessage(ErrorInfo* ei, const char* msg) {   // N/Common.cpp:18-30: dropped when empty or longer than 255 chars
  if (ei && msg) { size_t n = strlen(msg); if (n > 0 && n <= 255) { memcpy(ei->errorMessage, msg, n); ei->errorMessage[n] = 0; } }
}
void SetErrorMessage(ErrorInfo* ei, const std::string& s) { if (s.size() > 255) SetErrorMessage(ei, s.substr(0, 255).c_str()); else SetErrorMessage(ei, s.c_str()); }

thread_local StageTimes g_last_times;

// Runs one engine call and keeps its stage times for JxlB200LastStageTimes (zero when the call fails).
template <class Result, class Request> Result WithTimes(Result (*call)(const Request&), const Request& req) { g_last_times = StageTimes(); Result r = call(req); g_last_times = r.times; return r; }

// The one place where the engine's exceptions become what a C caller sees. `body` returns the status of a call that did not throw;
// a failure becomes StatusError's status, OutOfMemory, or DecodeError / EncodeError, with the exception's text in ErrorInfo.
// The thread's CUDA error state is cleared when a call enters and when it leaves: a runtime call that failed and was reported (an invalid
// device index) or was unchecked on purpose would otherwise be read by the launch check of a later call and fail that call instead.
struct Decoding { static const int32_t kOutOfMemory = DecoderStatus_OutOfMemory, kError = DecoderStatus_DecodeError; };
struct Encoding { static const int32_t kOutOfMemory = EncoderStatus_OutOfMemory, kError = EncoderStatus_EncodeError; };
template <class Codec, class F> int32_t Guard(ErrorInfo* ei, F&& body) {
  struct ClearCudaError { ClearCudaError() { cudaGetLastError(); } ~ClearCudaError() { cudaGetLastError(); } } clear;
  try { return body(); }
  catch (const StatusError& e) { SetErrorMessage(ei, std::string(e.what())); return e.status; }
  catch (const std::bad_alloc&) { return Codec::kOutOfMemory; }
  catch (const std::exception& e) { SetErrorMessage(ei, std::string(e.what())); return Codec::kError; }
  catch (...) { return Codec::kError; }
}

const int32_t kSOk = 0, kEPointer = int32_t(0x80004003), kEAbort = int32_t(0x80004004), kEOutOfMemory = int32_t(0x8007000E);

// N/Encoder/OutputProcessor.cpp: <= 64 KiB chunks, sticky first failure, progress tick per buffer request.
class OutputProcessor {
 public:
  explicit OutputProcessor(IOCallbacks* cb) : cb_(cb) {}
  void InitializeProgressReporting(ProgressProc p, int32_t initial, int32_t max, int32_t step) { progress_ = p; pct_ = initial; max_ = max; step_ = step; }
  EncoderStatus GetWriteStatus() const { return status_; }
  // mirrors GetBuffer/ReleaseBuffer pairs: returns false once a callback failed or the user cancelled
  bool Write(const uint8_t* data, size_t size) {
    size_t pos = 0;
    while (pos < size) {
      if (status_ != EncoderStatus_Ok || !ReportProgress()) return false;
      size_t n = std::min<size_t>(65536, size - pos); SetIfFailed(cb_->Write(data + pos, n)); pos += n;
    }
    return status_ == EncoderStatus_Ok;
  }
  void Seek(uint64_t p) { SetIfFailed(cb_->Seek(p)); }
 private:
  bool ReportProgress() { bool r = true; if (progress_) { if (pct_ < max_) pct_ += step_; r = progress_(pct_); if (!r) status_ = EncoderStatus_UserCanceled; } return r; }
  void SetIfFailed(int32_t hr) { if (hr < 0) { if (hr == kEAbort) status_ = EncoderStatus_UserCanceled; else if (hr == kEOutOfMemory) status_ = EncoderStatus_OutOfMemory; else status_ = EncoderStatus_WriteError; } }
  IOCallbacks* cb_; EncoderStatus status_ = EncoderStatus_Ok; ProgressProc progress_ = nullptr; int32_t pct_ = 0, max_ = 0, step_ = 0;
};

bool ReportProgress(ProgressProc p, int32_t pct) { return p ? p(pct) : true; }
// malloc'ed copies for the caller (freed with JxlB200Free)
void* CopyOut(const void* p, size_t n) { void* m = malloc(n ? n : 1); if (!m) throw std::bad_alloc(); if (n) memcpy(m, p, n); return m; }

}  // namespace

extern "C" {

uint32_t GetLibJxlVersion(void) { return (0u << 24) | (11u << 16) | (1u << 8); }   // bitstream behaviour follows libjxl 0.11.x (SURVEY.md §3.3)

DecoderStatus LoadImage(DecoderCallbacks* callbacks, const uint8_t* data, size_t dataSize, ErrorInfo* errorInfo) {
  if (!callbacks || !data) return DecoderStatus_NullParameter;
  return Guard<Decoding>(errorInfo, [&] {
    // pass 1: basic info, colour profile, metadata boxes (N/Decoder/JxlDecoder.cpp:412-793)
    const ParsedInfo pi = ParseInfo(data, dataSize);
    callbacks->setBasicInfo(int32_t(pi.width), int32_t(pi.height), pi.format, pi.sample_type, pi.has_alpha);
    if (pi.known_profile >= 0) { if (!callbacks->setKnownColorProfile(pi.known_profile)) return DecoderStatus_CreateMetadataError; }
    else if (!pi.icc.empty()) { std::vector<uint8_t> icc = pi.icc; if (!callbacks->setIccProfile(icc.data(), icc.size())) return DecoderStatus_CreateMetadataError; }
    if (pi.is_container) {
      if (pi.has_exif) { std::vector<uint8_t> e = pi.exif; if (!callbacks->setExif(e.data(), e.size())) return DecoderStatus_CreateMetadataError; }
      for (const auto& x : pi.xmp) { std::vector<uint8_t> b = x; if (!callbacks->setXmp(b.data(), b.size())) return DecoderStatus_CreateMetadataError; }
    }
    // pass 2: the frame (N/Decoder/JxlDecoder.cpp:217-410)
    DecodeRequest req; req.data = data; req.size = dataSize;
    const DecodeResult res = WithTimes(DecodeOnGpu, req);
    // layer name: length passed includes the NUL terminator (N/Decoder/JxlDecoder.cpp:274,366-370 — Appendix C-3)
    std::vector<char> name; if (!res.info.frame_name.empty()) { name.assign(res.info.frame_name.begin(), res.info.frame_name.end()); name.push_back(0); }
    if (!callbacks->setLayerData(res.pixels, name.empty() ? nullptr : name.data(), name.size())) return DecoderStatus_CreateLayerError;
    return DecoderStatus_Ok;
  });
}

EncoderStatus SaveImage(const BitmapData* bitmap, const EncoderOptions* options, const EncoderImageMetadata* metadata, IOCallbacks* callbacks, ErrorInfo* errorInfo, ProgressProc progressCallback) {
  if (!bitmap || !options || !callbacks || !metadata) return EncoderStatus_NullParameter;
  if (errorInfo) errorInfo->errorMessage[0] = 0;   // the managed caller passes it uninitialised (I/JpegXLNative.cs:102)
  return Guard<Encoding>(errorInfo, [&]() -> EncoderStatus {
    // progress sequence 0, 5, 15, 20, 25, then +5 per output buffer from 30 capped at 90, then 95 (N/Encoder/JxlEncoder.cpp:162-362)
    if (!ReportProgress(progressCallback, 0)) return EncoderStatus_UserCanceled;
    EncodeRequest req; req.bgra = bitmap->scan0; req.width = bitmap->width; req.height = bitmap->height; req.stride = bitmap->stride;
    req.distance = options->distance; req.effort = options->effort; req.lossless = options->lossless;
    req.exif = metadata->exif; req.exif_size = metadata->exifSize; req.icc = metadata->iccProfile; req.icc_size = metadata->iccProfileSize; req.xmp = metadata->xmp; req.xmp_size = metadata->xmpSize;
    if (!ReportProgress(progressCallback, 5)) return EncoderStatus_UserCanceled;
    if (!ReportProgress(progressCallback, 15)) return EncoderStatus_UserCanceled;
    if (!ReportProgress(progressCallback, 20)) return EncoderStatus_UserCanceled;
    if (!ReportProgress(progressCallback, 25)) return EncoderStatus_UserCanceled;
    OutputProcessor out(callbacks); out.InitializeProgressReporting(progressCallback, 30, 90, 5);
    const EncodeResult res = WithTimes(EncodeOnGpu, req);
    // libjxl streams output while encoding; the engine produces the file after the kernels finish and streams it the same way
    size_t half = res.file.size() / 2;
    bool ok = out.Write(res.file.data(), half);
    if (!ok) { EncoderStatus st = out.GetWriteStatus(); if (st == EncoderStatus_Ok) { SetErrorMessage(errorInfo, "JxlEncoderAddImageFrame failed."); st = EncoderStatus_EncodeError; } return st; }
    if (!ReportProgress(progressCallback, 95)) return EncoderStatus_UserCanceled;
    ok = out.Write(res.file.data() + half, res.file.size() - half);
    if (!ok) { EncoderStatus st = out.GetWriteStatus(); if (st != EncoderStatus_Ok) return st; SetErrorMessage(errorInfo, "JxlEncoderFlushInput failed."); return EncoderStatus_EncodeError; }
    return EncoderStatus_Ok;
  });
}

DecoderStatus JxlB200PeekInfo(const uint8_t* data, size_t dataSize, int32_t* info, ErrorInfo* errorInfo) {
  if (!data || !info) return DecoderStatus_NullParameter;
  return Guard<Decoding>(errorInfo, [&] {
    const ParsedInfo r = ParseInfo(data, dataSize);
    info[0] = int32_t(r.width); info[1] = int32_t(r.height); info[2] = r.format; info[3] = r.sample_type; info[4] = r.has_alpha; info[5] = r.num_channels; info[6] = r.known_profile; info[7] = r.is_container;
    return DecoderStatus_Ok;
  });
}

DecoderStatus JxlB200LoadImageBgra(const uint8_t* data, size_t dataSize, uint8_t* surface, size_t surfaceBytes, int32_t* width, int32_t* height, ErrorInfo* errorInfo) {
  if (!data || !surface) return DecoderStatus_NullParameter;
  return Guard<Decoding>(errorInfo, [&] {
    DecodeRequest req; req.data = data; req.size = dataSize; req.bgra = true; const DecodeResult res = WithTimes(DecodeOnGpu, req);
    if (surfaceBytes < res.pixel_bytes) { SetErrorMessage(errorInfo, "surface buffer too small"); return DecoderStatus_InvalidParameter; }
    memcpy(surface, res.pixels, res.pixel_bytes); if (width) *width = int32_t(res.out_width); if (height) *height = int32_t(res.out_height);
    return DecoderStatus_Ok;
  });
}

// The managed layer repack as a GPU epilogue (I/DecoderLayerData.cs:26-125 and its eighteen Set*ImageData variants): the decoder's
// interleaved output stays on the device, k_split_layers writes the colour bitmap (Rgb24 / Rgb48 / Rgb48Half / Rgb96Float with gray
// replicated, Cmyk32) and the Alpha8 transparency bitmap, and only those two cross PCIe.
DecoderStatus JxlB200LoadImageLayers(const uint8_t* data, size_t dataSize, uint8_t* color, size_t colorBytes, uint8_t* transparency, size_t transparencyBytes,
                                     int32_t* info6, ErrorInfo* errorInfo) {
  if (!data || !color) return DecoderStatus_NullParameter;
  Buf d_color, d_alpha;
  const DecoderStatus rc = Guard<Decoding>(errorInfo, [&] {
    DecodeRequest req; req.data = data; req.size = dataSize; req.device_output = true; const DecodeResult res = WithTimes(DecodeOnGpu, req);
    const ParsedInfo& pi = res.info; const size_t npix = size_t(res.out_width) * res.out_height; const size_t bps = pi.sample_type == 0 ? 1 : pi.sample_type == 3 ? 4 : 2;
    if (pi.format == 2 && pi.sample_type != 0) { SetErrorMessage(errorInfo, "unsupported CMYK channel representation"); return DecoderStatus_UnsupportedChannelFormat; }   // I/DecoderLayerData.cs:127-162
    const size_t dst_ch = pi.format == 2 ? 4 : 3, need_color = npix * dst_ch * bps, need_alpha = pi.has_alpha ? npix : 0;
    if (info6) { info6[0] = int32_t(res.out_width); info6[1] = int32_t(res.out_height); info6[2] = pi.format; info6[3] = pi.sample_type; info6[4] = pi.has_alpha ? 1 : 0; info6[5] = int32_t(dst_ch); }
    if (colorBytes < need_color || (pi.has_alpha && (!transparency || transparencyBytes < need_alpha))) { SetErrorMessage(errorInfo, "layer buffers too small"); return DecoderStatus_InvalidParameter; }
    d_color.Alloc(need_color); d_alpha.Alloc(need_alpha);
    {
      LaunchSplitLayers(res.pixels, d_color.p, d_alpha.as<uint8_t>(), npix, pi.format, pi.sample_type, pi.has_alpha, 0);
      cudaError_t e = cudaMemcpy(color, d_color.p, need_color, cudaMemcpyDeviceToHost);
      if (e == cudaSuccess && need_alpha) e = cudaMemcpy(transparency, d_alpha.p, need_alpha, cudaMemcpyDeviceToHost);
      JXLG_CHECK(e == cudaSuccess, std::string("CUDA: ") + cudaGetErrorString(e));
    }
    return DecoderStatus_Ok;
  });
  if (d_color.p || d_alpha.p) cudaDeviceSynchronize();   // the split kernel ran on the default stream (the copies above were synchronous): drained before the buffers go back to the pool
  return rc;
}

// Band decode: one rank's share of a frame sharded by group rows (SURVEY §8e "gigapixel": AC-group row ranges per GPU, no collective —
// each rank reconstructs one extra group row on either side instead of exchanging a halo). layout4 = {width, height, group size in
// pixels, number of group rows}. Rows [groupRowBegin*groupDim, min(groupRowEnd*groupDim, height)) are written to `out`, interleaved
// and tightly packed exactly as LoadImage would hand them to setLayerData.
DecoderStatus JxlB200BandLayout(const uint8_t* data, size_t dataSize, int32_t* layout4, ErrorInfo* errorInfo) {
  if (!data || !layout4) return DecoderStatus_NullParameter;
  return Guard<Decoding>(errorInfo, [&] {
    const ParsedInfo pi = DecodeBandLayout(data, dataSize);
    layout4[0] = int32_t(pi.width); layout4[1] = int32_t(pi.height); layout4[2] = int32_t(pi.group_dim); layout4[3] = int32_t(pi.num_group_rows); return DecoderStatus_Ok;
  });
}
DecoderStatus JxlB200DecodeBand(int32_t device, const uint8_t* data, size_t dataSize, uint32_t groupRowBegin, uint32_t groupRowEnd, uint8_t* out, size_t outBytes, int32_t bgra, int32_t* rows, ErrorInfo* errorInfo) {
  if (!data || !out) return DecoderStatus_NullParameter;
  return Guard<Decoding>(errorInfo, [&] {
    if (device >= 0 && cudaSetDevice(device) != cudaSuccess) { SetErrorMessage(errorInfo, "cudaSetDevice failed"); return DecoderStatus_InvalidParameter; }
    if (groupRowBegin >= groupRowEnd) { SetErrorMessage(errorInfo, "band decode: empty group-row range"); return DecoderStatus_InvalidParameter; }
    DecodeRequest req; req.data = data; req.size = dataSize; req.bgra = bgra != 0; req.band_begin = groupRowBegin; req.band_end = groupRowEnd; const DecodeResult res = WithTimes(DecodeOnGpu, req);
    if (outBytes < res.pixel_bytes) { SetErrorMessage(errorInfo, "band buffer too small"); return DecoderStatus_InvalidParameter; }
    memcpy(out, res.pixels, res.pixel_bytes); if (rows) *rows = int32_t(res.out_height);
    return DecoderStatus_Ok;
  });
}

// One shard of a batch: images [begin, end) of the caller's arrays, decoded by the three-phase pipeline below on `nstreams` streams owned
// by this shard. Runs on its own host thread (see JxlB200DecodeBatch): the enqueue work of an image (header parse, table building,
// ~40 CUDA calls) costs more host time than the image costs the GPU, so one enqueue thread caps a batch at about 1.2 images/ms.
struct BatchArgs {
  int32_t device, count; const uint8_t* const* datas; const size_t* dataSizes; uint8_t* const* outputs; const size_t* outputBytes;
  int32_t bgra, hostInputs, hostOutputs; DecoderStatus* statuses;
};
struct ShardResult { DecoderStatus first = DecoderStatus_Ok; std::string message; };
// Set once the caching pools of a device hold a full batch's buffer sets: until then only shard 0 enqueues (it reserves the sets when
// its first image is parsed); the other shards would otherwise race it with one cudaMalloc per buffer while the GPU is busy.
static std::atomic<int> g_pools_warm[64];

// Streams are created once per (device, shard slot) and reused by later batches (stream creation is not free).
static std::vector<cudaStream_t>& ShardStreams(int device, int slot, int want) {
  static std::mutex mu; static std::map<std::pair<int, int>, std::vector<cudaStream_t>> cache;
  std::lock_guard<std::mutex> lk(mu);
  std::vector<cudaStream_t>& v = cache[std::make_pair(device, slot)];
  while (int(v.size()) < want) {
    cudaStream_t st = nullptr;
    if (cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) != cudaSuccess) throw std::runtime_error("cudaStreamCreate failed");
    v.push_back(st);
  }
  return v;
}

// Pacing of batches whose pixels go to HOST memory. Such a batch is bound by the device-to-host copy (9.2 GB per 256 images of 12 MP: 166 ms at
// the 55.6 GB/s this box's PCIe link delivers, against 151 ms of decode), and started all at once its images move through LF / AC / tiles in
// lock-step, so every copy waits for the tiles phase at the end (r02: 267 ms per step = ~100 ms until the first image is rendered + 167 ms of
// copies). Starting the images at the rate the link can take them away turns the batch into a rolling pipeline: copies run from the first
// finished image on, beside the entropy phases of the images started later. One pacer per device, shared by every batch in flight on it.
// The rate images are started at: somewhat above the 55.6 GB/s the link was measured to deliver (the sweep in profiles/r02_e2e_pipeline.md);
// the in-flight cap gives the back-pressure.
static const double kPaceGBps = 80.0;
static std::atomic<int64_t> g_pace_next_ns[64];
static int64_t SteadyNs() { return std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
static int64_t PaceReserve(int dev, int64_t step_ns) {   // -> earliest start time of the caller's next bundle
  std::atomic<int64_t>& next = g_pace_next_ns[dev & 63]; const int64_t now = SteadyNs(); int64_t prev = next.load();
  for (;;) { const int64_t t = std::max(prev, now); if (next.compare_exchange_weak(prev, t + step_ns)) return t; }
}

static void RunBatchShard(const BatchArgs& a, int slot, int begin, int end, int nstreams, int batch_lanes, int bundle_size, size_t reserve_sets, ShardResult* out) {
  const int count = end - begin;
  if (count <= 0) return;
  Buf pin;   // outlives the catch blocks below, which wait for the copies into it
  std::vector<cudaEvent_t> in_ready;
  struct EventGuard { std::vector<cudaEvent_t>& v; ~EventGuard() { for (cudaEvent_t e : v) if (e) cudaEventDestroy(e); } } in_ready_guard{in_ready};
  std::vector<uint8_t> finished(size_t(count), 0);
  auto record = [&](int idx, DecoderStatus st, const std::string& msg) {
    if (a.statuses) a.statuses[idx] = st;
    finished[size_t(idx - begin)] = 1;
    if (st != DecoderStatus_Ok && out->first == DecoderStatus_Ok) { out->first = st; out->message = msg; }
  };
  try {
    if (a.device >= 0 && cudaSetDevice(a.device) != cudaSuccess) throw std::runtime_error("cudaSetDevice failed");
    int cur_dev = 0; cudaGetDevice(&cur_dev);
    std::vector<cudaStream_t>& all_streams = ShardStreams(cur_dev, slot, nstreams + 1);
    cudaStream_t copy_stream = all_streams[0];
    std::vector<cudaStream_t> free_streams(all_streams.rbegin(), all_streams.rbegin() + nstreams);
    struct InFlight { int idx; std::shared_ptr<DecodeJob> job; bool direct = false; };
    std::vector<size_t> in_off(size_t(count) + 1, 0); const uint8_t* host_in = nullptr;
    // Device-resident inputs: the headers are parsed on the host, so every file comes back once through one pinned buffer. The copies
    // are queued up front on their own stream, one event per file, and a file is only waited for when its turn to be parsed comes.
    if (!a.hostInputs) {
      for (int i = 0; i < count; i++) in_off[i + 1] = in_off[i] + ((a.dataSizes[begin + i] + 63) & ~size_t(63));
      pin.Alloc(in_off[count] + 64, true); in_ready.resize(size_t(count), nullptr);
      for (int i = 0; i < count; i++) {
        CUDA_OK(cudaMemcpyAsync(pin.as<uint8_t>() + in_off[i], a.datas[begin + i], a.dataSizes[begin + i], cudaMemcpyDeviceToHost, copy_stream));
        if (cudaEventCreateWithFlags(&in_ready[i], cudaEventDisableTiming) != cudaSuccess || cudaEventRecord(in_ready[i], copy_stream) != cudaSuccess)
          throw std::runtime_error("cannot read device inputs");
      }
      host_in = pin.as<uint8_t>();
    }
    // host outputs that are page-locked receive the pixels directly (no staging copy)
    std::vector<uint8_t> out_is_pinned(size_t(count), 0);
    if (a.hostOutputs) for (int i = 0; i < count; i++) {
      cudaPointerAttributes at;
      if (cudaPointerGetAttributes(&at, a.outputs[begin + i]) == cudaSuccess && at.type == cudaMemoryTypeHost) out_is_pinned[i] = 1; else cudaGetLastError();
    }
    // Three-phase pipeline per image (LF entropy | AC entropy | reconstruction + render): a phase is enqueued only once the image's
    // stream has drained, so a kernel waiting on a 40 ms predecessor never sits at the head of a hardware queue shared with other
    // streams (there are 32 queues). Images travel in bundles of `bundle_size` that share a stream and whose LF / AC entropy kernels
    // are one multi-image launch each: the device holds at most 128 resident grids, and an image keeps one for ~70 ms.
    // q1/q2/q3 hold the bundles whose phase 1/2/3 is running.
    struct Bundle { std::vector<std::unique_ptr<InFlight>> items; cudaStream_t stream = nullptr; };
    std::deque<std::unique_ptr<Bundle>> q1, q2, q3; int next = 0, done = 0;
    auto finish = [&](InFlight& f, const DecodeResult& res) {   // records a decoded image
      DecoderStatus st = DecoderStatus_Ok;
      if (res.pixel_bytes > a.outputBytes[f.idx]) st = DecoderStatus_InvalidParameter;
      else if (!f.direct) memcpy(a.outputs[f.idx], res.pixels, res.pixel_bytes);
      record(f.idx, st, std::string());
      f.job.reset(); done++;
    };
    // Runs one step of an image (enqueue, a later phase, finish). A failure is recorded for the image and drops it (false).
    auto step = [&](InFlight& f, auto&& fn) {
      ErrorInfo ei; ei.errorMessage[0] = 0;
      const DecoderStatus st = Guard<Decoding>(&ei, [&] { fn(); return DecoderStatus_Ok; });
      if (st != DecoderStatus_Ok) { record(f.idx, st, ei.errorMessage); f.job.reset(); done++; }
      return st == DecoderStatus_Ok;
    };
    // A busy stream answers cudaErrorNotReady, which is cleared so that the launch checks of this thread do not report it as a failure.
    auto idle = [](const Bundle& b) { const cudaError_t e = cudaStreamQuery(b.stream); if (e == cudaErrorNotReady) cudaGetLastError(); return e != cudaErrorNotReady; };
    auto jobs_of = [](Bundle& b) { std::vector<std::shared_ptr<DecodeJob>> v; for (auto& it : b.items) v.push_back(it->job); return v; };
    auto next_phase = [&](Bundle& b, int phase) {   // enqueue `phase` for every image of the bundle; images that fail are finished and dropped
      for (size_t k = 0; k < b.items.size();) {
        InFlight& f = *b.items[k];
        if (step(f, [&] { DecodeEnqueuePhase(f.job, phase); })) k++; else b.items.erase(b.items.begin() + k);
      }
      if (phase == 2) DecodeBundleLaunch(jobs_of(b), 2);
    };
    auto advance = [&]() {   // moves bundles whose current phase has drained to the next one (polling: a blocking wait on one stream would stall all others)
      bool progressed = false; const size_t kWindow = 24;   // bundles finish roughly in order; look a little past the front of each queue
      for (size_t k = 0; k < std::min(kWindow, q3.size());) {
        if (!idle(*q3[k])) { k++; continue; }
        Bundle& b = *q3[k];
        for (auto& f : b.items) step(*f, [&] { finish(*f, DecodeFinish(f->job)); });
        free_streams.push_back(b.stream); q3.erase(q3.begin() + k); progressed = true;
      }
      for (size_t k = 0; k < std::min(kWindow, q2.size());) {
        if (!idle(*q2[k])) { k++; continue; }
        std::unique_ptr<Bundle> b = std::move(q2[k]); q2.erase(q2.begin() + k); progressed = true;
        next_phase(*b, 3);
        if (b->items.empty()) free_streams.push_back(b->stream); else q3.push_back(std::move(b));
      }
      for (size_t k = 0; k < std::min(kWindow, q1.size());) {
        if (!idle(*q1[k])) { k++; continue; }
        std::unique_ptr<Bundle> b = std::move(q1[k]); q1.erase(q1.begin() + k); progressed = true;
        next_phase(*b, 2);
        if (b->items.empty()) free_streams.push_back(b->stream); else q2.push_back(std::move(b));
      }
      return progressed;
    };
    bool reserved = reserve_sets == 0;
    // pacing (host outputs only): ns per image = its output bytes over kPaceGBps
    int64_t pace_ns = 0, launch_at = 0;
    if (a.hostOutputs && a.count >= 64) pace_ns = int64_t(double(a.outputBytes[begin]) / kPaceGBps);
    while (done < count) {
      const bool progressed = advance();
      if (pace_ns && next < count && !free_streams.empty() && launch_at == 0) launch_at = PaceReserve(cur_dev, pace_ns * std::min(bundle_size, count - next));
      if (next < count && !free_streams.empty() && (launch_at == 0 || SteadyNs() >= launch_at)) {
        launch_at = 0;
        std::unique_ptr<Bundle> b(new Bundle); b->stream = free_streams.back(); free_streams.pop_back();
        for (int k = 0; k < bundle_size && next < count; k++) {
          const int li = next++, i = begin + li;
          std::unique_ptr<InFlight> f(new InFlight); f->idx = i;
          DecodeRequest req; req.bgra = a.bgra != 0; req.device_output = !a.hostOutputs; req.size = a.dataSizes[i]; req.out_capacity = a.outputBytes[i]; req.ac_lanes = batch_lanes;
          if (a.hostInputs) req.data = a.datas[i]; else { CUDA_OK(cudaEventSynchronize(in_ready[li])); req.data = host_in + in_off[li]; req.device_input = a.datas[i]; }
          if (!a.hostOutputs) { req.out_device = a.outputs[i]; f->direct = true; } else if (out_is_pinned[li]) { req.out_pinned = a.outputs[i]; f->direct = true; }
          if (reserve_sets == 0 && a.count >= 32) for (int spin = 0; spin < 40000 && !g_pools_warm[cur_dev & 63].load(); spin++) std::this_thread::sleep_for(std::chrono::microseconds(50));   // at most 2 s, first batch only
          bool layered = false;
          step(*f, [&] { try { f->job = DecodeEnqueue(req, b->stream, true, bundle_size > 1); } catch (const LayeredStill&) { layered = true; } });
          if (!reserved) { reserved = true; if (f->job) DecodeReservePools(f->job, reserve_sets); g_pools_warm[cur_dev & 63].store(1); }   // the first image tells the buffer sizes of the batch
          if (layered) {   // a layered still inside a batch: composited by the single-image path, on this shard's thread
            DecodeRequest lr = req; lr.ac_lanes = 0; step(*f, [&] { finish(*f, DecodeOnGpu(lr)); });
          }
          if (f->job) b->items.push_back(std::move(f));
        }
        if (bundle_size > 1) DecodeBundleLaunch(jobs_of(*b), 1);
        if (b->items.empty()) free_streams.push_back(b->stream); else q1.push_back(std::move(b));
      } else if (!progressed) std::this_thread::sleep_for(std::chrono::microseconds(20));
    }
  } catch (const std::exception& e) {   // a failure of the shard itself (streams, input copies): every image not finished yet fails with it
    // Work may still be running on this shard's streams and writing into caller-owned buffers: wait for it before returning them.
    cudaDeviceSynchronize(); cudaGetLastError();
    const DecoderStatus st = dynamic_cast<const std::bad_alloc*>(&e) ? DecoderStatus_OutOfMemory : DecoderStatus_DecodeError;
    for (int i = begin; i < end; i++) if (!finished[size_t(i - begin)]) record(i, st, e.what());
  } catch (...) {
    cudaDeviceSynchronize(); cudaGetLastError();
    for (int i = begin; i < end; i++) if (!finished[size_t(i - begin)]) record(i, DecoderStatus_DecodeError, "batch decode failed");
  }
}

// A batch in flight: owns copies of the caller's pointer arrays, the per-file statuses and the shard threads.
struct JxlB200Batch {
  std::vector<const uint8_t*> datas; std::vector<size_t> sizes; std::vector<uint8_t*> outputs; std::vector<size_t> out_bytes;
  std::vector<DecoderStatus> statuses; std::vector<ShardResult> results; std::vector<std::thread> threads; std::vector<int> slots; BatchArgs args;
};
// Stream sets are leased per shard so that two batches in flight on one device never share a stream.
static std::mutex g_slot_mu; static std::vector<uint8_t> g_slot_busy;
static int AcquireSlot() { std::lock_guard<std::mutex> lk(g_slot_mu); for (size_t i = 0; i < g_slot_busy.size(); i++) if (!g_slot_busy[i]) { g_slot_busy[i] = 1; return int(i); } g_slot_busy.push_back(1); return int(g_slot_busy.size()) - 1; }
static void ReleaseSlot(int slot) { std::lock_guard<std::mutex> lk(g_slot_mu); g_slot_busy[size_t(slot)] = 0; }

JxlB200Batch* JxlB200DecodeBatchSubmit(int32_t device, int32_t count, const uint8_t* const* datas, const size_t* dataSizes, uint8_t* const* outputs, const size_t* outputBytes, int32_t bgra,
                                       int32_t hostInputs, int32_t hostOutputs, int32_t maxInFlight, ErrorInfo* errorInfo) {
  if (!datas || !dataSizes || !outputs || !outputBytes || count < 0) { SetErrorMessage(errorInfo, "null parameter"); return nullptr; }
  JxlB200Batch* raw = nullptr;
  Guard<Decoding>(errorInfo, [&] {
    std::string why; JXLG_CHECK(CudaAvailable(&why), why);
    JXLG_CHECK(device < 0 || cudaSetDevice(device) == cudaSuccess, "cudaSetDevice failed");
    std::unique_ptr<JxlB200Batch> b(new JxlB200Batch);
    b->datas.assign(datas, datas + count); b->sizes.assign(dataSizes, dataSizes + count); b->outputs.assign(outputs, outputs + count); b->out_bytes.assign(outputBytes, outputBytes + count);
    b->statuses.assign(size_t(count), DecoderStatus_Ok);
    const int nstreams = std::max(1, std::min(maxInFlight > 0 ? maxInFlight : 16, 256));   // maxInFlight counts streams (bundles) in flight
    // AC sections per warp: more lanes = fewer resident warps and instructions per section, but a longer walk (16 / 24 / 31 / 41 ms for
    // 1 / 4 / 8 / 16 lanes on a 12 MP image). Large batches are bound by issue slots and take 16; small ones (a rank's share of a
    // sharded batch) are bound by the walk itself and take just enough lanes to keep every section resident at once.
    const int batch_lanes = nstreams < 8 ? 1 : count >= 192 ? 16 : count >= 96 ? 8 : count >= 48 ? 4 : count >= 24 ? 2 : 1;
    const int bundle_size = std::max(1, std::min((count > nstreams && nstreams >= 32) ? 2 : 1, kMaxBundle));   // images per stream / per entropy launch: only when the batch has more images than streams
    // Host threads: the per-image enqueue work is split over `shards` threads, each with its own share of the streams.
    int hw = int(std::thread::hardware_concurrency()); if (hw <= 0) hw = 4;
    int shards = std::min(4, std::max(1, hw / 2));
    shards = std::max(1, std::min(std::min(shards, nstreams / 8), count / 16));   // small batches keep a single enqueue thread
    b->args = BatchArgs{device, count, b->datas.data(), b->sizes.data(), b->outputs.data(), b->out_bytes.data(), bgra, hostInputs, hostOutputs, b->statuses.data()};
    b->results.resize(size_t(shards));
    const size_t reserve_sets = size_t(std::min(count, nstreams * bundle_size)) - (count > 0 ? 1 : 0);
    JxlB200Batch* self = b.get();
    for (int k = 0; k < shards; k++) {
      const int i0 = int(int64_t(count) * k / shards), i1 = int(int64_t(count) * (k + 1) / shards), ns = nstreams * (k + 1) / shards - nstreams * k / shards;
      const int slot = AcquireSlot(); b->slots.push_back(slot);
      b->threads.emplace_back([self, k, slot, i0, i1, ns, batch_lanes, bundle_size, reserve_sets]() {
        RunBatchShard(self->args, slot, i0, i1, std::max(1, ns), batch_lanes, bundle_size, k == 0 ? reserve_sets : 0, &self->results[size_t(k)]);
      });
    }
    raw = b.release(); return DecoderStatus_Ok;
  });
  return raw;
}

DecoderStatus JxlB200DecodeBatchWait(JxlB200Batch* batch, DecoderStatus* statuses, ErrorInfo* errorInfo) {
  if (!batch) return DecoderStatus_NullParameter;
  std::unique_ptr<JxlB200Batch> b(batch);
  for (auto& t : b->threads) if (t.joinable()) t.join();
  for (int slot : b->slots) ReleaseSlot(slot);
  if (statuses) for (size_t i = 0; i < b->statuses.size(); i++) statuses[i] = b->statuses[i];
  for (size_t k = 0; k < b->results.size(); k++) if (b->results[k].first != DecoderStatus_Ok) { SetErrorMessage(errorInfo, b->results[k].message); return b->results[k].first; }
  return DecoderStatus_Ok;
}

DecoderStatus JxlB200DecodeBatch(int32_t device, int32_t count, const uint8_t* const* datas, const size_t* dataSizes, uint8_t* const* outputs, const size_t* outputBytes, int32_t bgra,
                                 int32_t hostInputs, int32_t hostOutputs, int32_t maxInFlight, DecoderStatus* statuses, ErrorInfo* errorInfo) {
  if (!datas || !dataSizes || !outputs || !outputBytes || count < 0) return DecoderStatus_NullParameter;
  ErrorInfo local; local.errorMessage[0] = 0;
  JxlB200Batch* b = JxlB200DecodeBatchSubmit(device, count, datas, dataSizes, outputs, outputBytes, bgra, hostInputs, hostOutputs, maxInFlight, &local);
  if (!b) { SetErrorMessage(errorInfo, local.errorMessage); return std::string(local.errorMessage) == "cudaSetDevice failed" ? DecoderStatus_InvalidParameter : DecoderStatus_DecodeError; }
  return JxlB200DecodeBatchWait(b, statuses, errorInfo);
}

EncoderStatus JxlB200EncodeToMemory(const BitmapData* bitmap, const EncoderOptions* options, const EncoderImageMetadata* metadata, int32_t deviceInput, uint8_t** out, size_t* outSize, ErrorInfo* errorInfo) {
  if (!bitmap || !options || !out || !outSize) return EncoderStatus_NullParameter;
  return Guard<Encoding>(errorInfo, [&] {
    EncodeRequest req; req.bgra = bitmap->scan0; req.width = bitmap->width; req.height = bitmap->height; req.stride = bitmap->stride; req.distance = options->distance; req.effort = options->effort; req.lossless = options->lossless; req.device_input = deviceInput != 0;
    if (metadata) { req.exif = metadata->exif; req.exif_size = metadata->exifSize; req.icc = metadata->iccProfile; req.icc_size = metadata->iccProfileSize; req.xmp = metadata->xmp; req.xmp_size = metadata->xmpSize; }
    const EncodeResult res = WithTimes(EncodeOnGpu, req);
    *out = static_cast<uint8_t*>(CopyOut(res.file.data(), res.file.size())); *outSize = res.file.size();
    return EncoderStatus_Ok;
  });
}
void JxlB200Free(void* p) { free(p); }
// Host-only: what the encoder reads out of a matrix/TRC ICC profile (SaveImage with metadata->iccProfile, lossy): matrix9 = profile RGB
// (linear) -> linear sRGB, lut768 = the three tone curves sampled at v/255. Returns 0 and a message when the profile cannot be used.
int32_t JxlB200DebugParseIcc(const uint8_t* icc, size_t iccSize, float* matrix9, float* lut768, ErrorInfo* errorInfo) {
  if (!icc || !matrix9 || !lut768) return 0;
  return Guard<Encoding>(nullptr, [&] {
    IccMatrixTrc m; std::string why; if (!ParseMatrixTrcIcc(icc, iccSize, &m, &why)) { SetErrorMessage(errorInfo, why); return EncoderStatus_EncodeError; }
    for (int i = 0; i < 9; i++) matrix9[i] = float(m.to_linear_srgb[i]); memcpy(lut768, m.lut, sizeof(m.lut)); return EncoderStatus_Ok;
  }) == EncoderStatus_Ok ? 1 : 0;
}
// Returns the cached device and page-locked buffers of the calling thread's current device to the driver (after a large batch the
// pools hold one buffer set per image that was in flight).
// ---- sharded encode (BASELINE config 5, SURVEY §8e "Encode sharding"): one band session per GPU, see encode_engine.cu
// The session holds the band encoder, its device and its own copy of the ICC profile (the caller's metadata need not outlive Create).
struct JxlB200BandEncoder { std::unique_ptr<BandEncoder> enc; int device = -1; std::vector<uint8_t> icc; };
static EncodeRequest BandRequest(const BitmapData* b, const EncoderOptions* o, const EncoderImageMetadata* md) {
  EncodeRequest req; req.bgra = b->scan0; req.width = b->width; req.height = b->height; req.stride = b->stride; req.distance = o->distance; req.effort = o->effort; req.lossless = o->lossless;
  if (md) { req.exif = md->exif; req.exif_size = md->exifSize; req.icc = md->iccProfile; req.icc_size = md->iccProfileSize; req.xmp = md->xmp; req.xmp_size = md->xmpSize; }
  return req;
}
JxlB200BandEncoder* JxlB200BandEncoderCreate(int32_t device, const BitmapData* band, uint32_t frameHeight, uint32_t firstRow, uint32_t haloTop, uint32_t haloBottom,
                                             const EncoderOptions* options, const EncoderImageMetadata* metadata, int32_t deviceInput, uint32_t* bandFlags, ErrorInfo* errorInfo) {
  if (!band || !band->scan0 || !options || !bandFlags) { SetErrorMessage(errorInfo, "null parameter"); return nullptr; }
  std::unique_ptr<JxlB200BandEncoder> h;
  const EncoderStatus st = Guard<Encoding>(errorInfo, [&] {
    JXLG_CHECK(device < 0 || cudaSetDevice(device) == cudaSuccess, "cudaSetDevice failed");
    EncodeRequest req = BandRequest(band, options, metadata); req.device_input = deviceInput != 0;
    req.frame_height = frameHeight; req.band_y0 = firstRow; req.halo_top = haloTop; req.halo_bottom = haloBottom;
    h.reset(new JxlB200BandEncoder); h->device = device;
    if (req.icc_size) { h->icc.assign(req.icc, req.icc + req.icc_size); req.icc = h->icc.data(); }
    req.exif = nullptr; req.exif_size = 0; req.xmp = nullptr; req.xmp_size = 0;
    h->enc.reset(new BandEncoder(req)); *bandFlags = h->enc->Begin();
    return EncoderStatus_Ok;
  });
  if (st == EncoderStatus_OutOfMemory) SetErrorMessage(errorInfo, "band encoder: out of memory");
  return st == EncoderStatus_Ok ? h.release() : nullptr;
}
EncoderStatus JxlB200BandEncoderTokenize(JxlB200BandEncoder* enc, uint32_t frameFlags, uint64_t** hist, size_t* histWords, ErrorInfo* errorInfo) {
  if (!enc || !hist || !histWords) return EncoderStatus_NullParameter;
  return Guard<Encoding>(errorInfo, [&] {
    JXLG_CHECK(enc->device < 0 || cudaSetDevice(enc->device) == cudaSuccess, "cudaSetDevice failed");
    const std::vector<uint64_t> h = enc->enc->Tokenize(frameFlags);
    *hist = static_cast<uint64_t*>(CopyOut(h.data(), h.size() * 8)); *histWords = h.size(); return EncoderStatus_Ok;
  });
}
EncoderStatus JxlB200BandEncoderFinish(JxlB200BandEncoder* enc, const uint64_t* frameHist, size_t histWords, uint8_t** sections, size_t* sectionBytes, float* deviceMs, ErrorInfo* errorInfo) {
  if (!enc || !frameHist || !sections || !sectionBytes) return EncoderStatus_NullParameter;
  return Guard<Encoding>(errorInfo, [&] {
    JXLG_CHECK(enc->device < 0 || cudaSetDevice(enc->device) == cudaSuccess, "cudaSetDevice failed");
    const std::vector<uint8_t> blob = enc->enc->FinishBlob(std::vector<uint64_t>(frameHist, frameHist + histWords)); if (deviceMs) *deviceMs = enc->enc->device_ms;
    *sections = static_cast<uint8_t*>(CopyOut(blob.data(), blob.size())); *sectionBytes = blob.size(); return EncoderStatus_Ok;
  });
}
int64_t JxlB200BandEncoderDebugStage(JxlB200BandEncoder* enc, int32_t which, void* out, int64_t capacityBytes, int64_t* dims4, ErrorInfo* errorInfo) {
  if (!enc) { SetErrorMessage(errorInfo, "null parameter"); return 0; }
  int64_t n = 0;
  Guard<Encoding>(errorInfo, [&] { JXLG_CHECK(enc->device < 0 || cudaSetDevice(enc->device) == cudaSuccess, "cudaSetDevice failed"); n = enc->enc->DebugStage(which, out, capacityBytes, dims4); return EncoderStatus_Ok; });
  return n;
}
void JxlB200BandEncoderDestroy(JxlB200BandEncoder* enc) {
  if (!enc) return;
  Guard<Encoding>(nullptr, [&] { if (enc->device >= 0) cudaSetDevice(enc->device); enc->enc.reset(); return EncoderStatus_Ok; });   // the encoder waits for its stream
  delete enc;
}
EncoderStatus JxlB200AssembleBands(uint32_t width, uint32_t height, const EncoderOptions* options, const EncoderImageMetadata* metadata, uint32_t frameFlags, const uint64_t* frameHist, size_t histWords,
                                   const uint8_t* const* bandSections, const size_t* bandSectionBytes, int32_t bandCount, uint8_t** out, size_t* outSize, ErrorInfo* errorInfo) {
  if (!options || !frameHist || !bandSections || !bandSectionBytes || !out || !outSize || bandCount <= 0) return EncoderStatus_NullParameter;
  return Guard<Encoding>(errorInfo, [&] {
    BitmapData whole{nullptr, width, height, width * 4}; EncodeRequest req = BandRequest(&whole, options, metadata);
    const std::vector<uint8_t> file = AssembleBands(req, frameFlags, frameHist, histWords, bandSections, bandSectionBytes, size_t(bandCount));
    *out = static_cast<uint8_t*>(CopyOut(file.data(), file.size())); *outSize = file.size(); return EncoderStatus_Ok;
  });
}

int64_t JxlB200DebugSectionSizes(const uint8_t* data, size_t dataSize, uint64_t* sizes, int64_t capacity, int32_t* counts2, ErrorInfo* errorInfo) {
  if (!data || !sizes) return 0;
  int64_t n = 0;
  Guard<Decoding>(errorInfo, [&] {
    const SectionSizes s = DecodeSectionSizes(data, dataSize);
    if (int64_t(s.sizes.size()) > capacity) return DecoderStatus_Ok;
    for (size_t i = 0; i < s.sizes.size(); i++) sizes[i] = s.sizes[i]; if (counts2) { counts2[0] = int32_t(s.num_lf_groups); counts2[1] = int32_t(s.num_groups); } n = int64_t(s.sizes.size());
    return DecoderStatus_Ok;
  });
  return n;
}
void JxlB200ReleaseMemory(void) { Guard<Decoding>(nullptr, [] { cudaDeviceSynchronize(); TrimPools(); for (auto& w : g_pools_warm) w.store(0); return DecoderStatus_Ok; }); }

void JxlB200LastStageTimes(float* ms8) { if (!ms8) return; const StageTimes& t = g_last_times; ms8[0] = t.h2d; ms8[1] = t.lf; ms8[2] = t.ac; ms8[3] = t.recon; ms8[4] = t.filters; ms8[5] = t.output; ms8[6] = t.d2h; ms8[7] = t.total; }
int64_t JxlB200KernelLaunchCount(void) { return LaunchCount(); }
int32_t JxlB200CudaAvailable(ErrorInfo* errorInfo) { std::string why; bool ok = CudaAvailable(&why); if (!ok) SetErrorMessage(errorInfo, why); return ok ? 1 : 0; }

int64_t JxlB200DebugDecodeStage(const uint8_t* data, size_t dataSize, int32_t which, float* out, int64_t capacity, int32_t* dims2, ErrorInfo* errorInfo) {
  if (!data || !out) return 0;
  int64_t n = 0;
  Guard<Decoding>(errorInfo, [&] {
    DecodeRequest req; req.data = data; req.size = dataSize; const DecodeResult res = DecodeOnGpu(req);
    if (which == 4) { std::vector<int16_t> c; if (DecodeDebugCoeffs(res.job, &c) && int64_t(c.size()) <= capacity) { for (size_t i = 0; i < c.size(); i++) out[i] = float(c[i]); n = int64_t(c.size()); } return DecoderStatus_Ok; }
    std::vector<float> v; int xp = 0, yp = 0; if (!DecodeDebugPlanes(res.job, which, &v, &xp, &yp) || int64_t(v.size()) > capacity) return DecoderStatus_Ok;
    memcpy(out, v.data(), v.size() * 4); if (dims2) { dims2[0] = xp; dims2[1] = yp; } n = int64_t(v.size());
    return DecoderStatus_Ok;
  });
  return n;
}

}  // extern "C"
