// pdn-jpegxl_b200 engine — decode orchestration: host front-end parse -> flat device tables ->
// kernel pipeline -> pixel buffer. This is the engine behind LoadImage; it restates what
// DecoderReadImage drives through libjxl (N/Decoder/JxlDecoder.cpp:796-852): header/metadata
// pass (:412-793), format decisions (:461-561), first frame only (:398-400), interleaved
// tightly-packed output (:289-323), straight alpha (:233), CMYK merge (:159-215).
// There is no CPU decode path: without a CUDA device every call fails with DecodeError.
#include "engine.h"
#include "dev/kernels.h"
#include "host/headers.h"
#include "host/modular_host.h"
#include "host/vardct_tables.h"
#define JXLG_ICC_DEFINE_STREAM_FUNCS
#include "host/icc.h"
#include <dlfcn.h>
#include <map>
#include <mutex>
#include <atomic>
#include <memory>
#include <functional>

namespace jxlgpu {

// ---------------------------------------------------------------- small utilities
bool CudaAvailable(std::string* why) {
  int n = 0; cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) { if (why) *why = std::string("no usable CUDA device (") + (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0") + "); the engine has no CPU fallback"; cudaGetLastError(); return false; }
  return true;
}

// Caching allocators (device + pinned host). cudaMalloc / cudaHostAlloc cost milliseconds; a decode is a handful of ms.
// The shard threads of a batch take and return buffers concurrently: every access to the maps and the cached byte count holds mu_,
// and no allocation runs under it.
class Pool {
 public:
  explicit Pool(bool pinned) : pinned_(pinned) {}
  void* Get(size_t bytes) {
    size_t sz = Round(bytes); { std::lock_guard<std::mutex> lk(mu_); auto it = free_.find(sz); if (it != free_.end() && !it->second.empty()) { void* p = it->second.back(); it->second.pop_back(); cached_ -= sz; return p; } }
    void* p = nullptr; cudaError_t e = Malloc(&p, sz);
    if (e != cudaSuccess) { cudaGetLastError(); Trim(); e = Malloc(&p, sz); }
    if (e != cudaSuccess) { cudaGetLastError(); throw std::bad_alloc(); }
    { std::lock_guard<std::mutex> lk(mu_); total_[sz]++; }
    return p;
  }
  void Put(void* p, size_t bytes) { if (!p) return; size_t sz = Round(bytes); std::lock_guard<std::mutex> lk(mu_); free_[sz].push_back(p); cached_ += sz; if (cached_ > LimitLocked()) TrimLocked(); }
  void Trim() { std::lock_guard<std::mutex> lk(mu_); TrimLocked(); }
  // Makes sure `count` buffers of this size class are cached (batch start: the first image tells the sizes; allocating them one
  // by one while the GPU is busy stalls the enqueue thread for milliseconds each and takes many batches to converge).
  // `count` is the number of buffers of this class the pool must OWN (free or handed out): other threads take buffers while a
  // reservation runs, so counting only the free ones would allocate a fresh set on every batch.
  void Reserve(size_t bytes, size_t count) {
    const size_t sz = Round(bytes); size_t have; { std::lock_guard<std::mutex> lk(mu_); have = total_[sz]; }
    for (; have < count; have++) {
      { std::lock_guard<std::mutex> lk(mu_); if (cached_ + sz > LimitLocked()) return; }
      void* p = nullptr; if (Malloc(&p, sz) != cudaSuccess) { cudaGetLastError(); return; }
      std::lock_guard<std::mutex> lk(mu_); free_[sz].push_back(p); cached_ += sz; total_[sz]++; }
  }
  // size classes: powers of two from 4 KiB up to 16 MiB (files of different sizes then share every small bucket, so the first image of
  // a batch can reserve for all of them), eighths of a power of two above (the big planes, whose size depends on the dimensions only)
  static size_t Round(size_t b) { if (b <= 4096) return 4096; int k = 63 - __builtin_clzll(b - 1); if (b <= (size_t(16) << 20)) return size_t(2) << k; k = 63 - __builtin_clzll(b); size_t g = size_t(1) << (k - 3); return (b + g - 1) / g * g; }
 private:
  size_t LimitLocked() { if (!limit_) { size_t fr = 0, tot = 0; if (pinned_ || cudaMemGetInfo(&fr, &tot) != cudaSuccess) { cudaGetLastError(); limit_ = size_t(32) << 30; } else limit_ = tot / 4 * 3; } return limit_; }
  cudaError_t Malloc(void** p, size_t sz) { return pinned_ ? cudaHostAlloc(p, sz, cudaHostAllocDefault) : cudaMalloc(p, sz); }
  void TrimLocked() { for (auto& kv : free_) { for (void* p : kv.second) { if (pinned_) cudaFreeHost(p); else cudaFree(p); } total_[kv.first] -= std::min(total_[kv.first], kv.second.size()); } free_.clear(); cached_ = 0; }
  bool pinned_; std::mutex mu_; std::map<size_t, std::vector<void*>> free_; std::map<size_t, size_t> total_; size_t cached_ = 0, limit_ = 0;
};
static Pool& DevPool() {   // one pool per device: a cached buffer must never cross devices
  static std::mutex mu; static std::map<int, std::unique_ptr<Pool>> pools; int dev = 0; cudaGetDevice(&dev); std::lock_guard<std::mutex> lk(mu); auto& p = pools[dev]; if (!p) p.reset(new Pool(false)); return *p; }
static Pool& HostPool() { static Pool p(true); return p; }
void TrimPools() { DevPool().Trim(); HostPool().Trim(); }
void Buf::Alloc(size_t bytes, bool pinned) { Free(); n = bytes ? bytes : 1; pool = pinned ? &HostPool() : &DevPool(); p = pool->Get(n); }
void Buf::Free() { if (p) pool->Put(p, n); p = nullptr; n = 0; }

static const DTables* DeviceTables() {
  static std::mutex mu; static std::map<int, DTables*> per_dev; std::lock_guard<std::mutex> lk(mu); int dev = 0; CUDA_OK(cudaGetDevice(&dev));
  auto it = per_dev.find(dev); if (it != per_dev.end()) return it->second;
  std::unique_ptr<DTables> h(new DTables); FillDeviceTables(h.get()); DTables* d = nullptr; CUDA_OK(cudaMalloc(&d, sizeof(DTables))); CUDA_OK(cudaMemcpy(d, h.get(), sizeof(DTables), cudaMemcpyHostToDevice)); per_dev[dev] = d; return d;
}

// Per-device static blob: default dequantisation tables and natural coefficient orders (about 3 MB), uploaded once.
struct StaticBlob { const uint8_t* dev = nullptr; uint32_t dq_off[kNumQuantTables]; uint32_t nat_off[kNumOrders]; };
static const std::vector<float>& DefaultDequant(int t); static const std::vector<uint32_t>& NaturalOrderCached(int o);
static const StaticBlob& DeviceStaticBlob() {
  static std::mutex mu; static std::map<int, StaticBlob> per_dev; std::lock_guard<std::mutex> lk(mu); int dev = 0; CUDA_OK(cudaGetDevice(&dev));
  auto it = per_dev.find(dev); if (it != per_dev.end()) return it->second;
  StaticBlob sb; std::vector<uint8_t> b; auto add = [&](const void* p, size_t n) { size_t off = (b.size() + 15) & ~size_t(15); b.resize(off + n); memcpy(b.data() + off, p, n); return uint32_t(off) | kStaticBlobBit; };
  for (int t = 0; t < kNumQuantTables; t++) { const std::vector<float>& d = DefaultDequant(t); sb.dq_off[t] = add(d.data(), d.size() * 4); }
  for (int o = 0; o < kNumOrders; o++) { const std::vector<uint32_t>& n = NaturalOrderCached(o); sb.nat_off[o] = add(n.data(), n.size() * 4); }
  uint8_t* d = nullptr; CUDA_OK(cudaMalloc(&d, b.size())); CUDA_OK(cudaMemcpy(d, b.data(), b.size(), cudaMemcpyHostToDevice)); sb.dev = d; return per_dev[dev] = sb;
}

static std::vector<uint8_t> BrotliDecompress(const uint8_t* data, size_t size) {
  typedef int (*Fn)(size_t, const uint8_t*, size_t*, uint8_t*);
  static Fn fn = []() -> Fn { void* h = dlopen("libbrotlidec.so.1", RTLD_NOW); return h ? reinterpret_cast<Fn>(dlsym(h, "BrotliDecoderDecompress")) : nullptr; }();
  JXLG_CHECK(fn != nullptr, "brob box: libbrotlidec.so.1 not available");
  for (size_t cap = std::max<size_t>(size * 8, 1 << 16); cap <= (size_t(1) << 31); cap *= 4) { std::vector<uint8_t> out(cap); size_t n = cap; if (fn(size, data, &n, out.data()) == 1) { out.resize(n); return out; } }
  throw Error("brob box: brotli stream invalid or too large");
}

// A frame that is shown as it is: full canvas, replaces what was there, and the first frame the reference would receive as a full image.
static bool FrameIsPlain(const FrameHeader& fh, const ImageMetadata& m) {
  const bool shown = (fh.frame_type == kFrameRegular || fh.frame_type == kFrameSkipProgressive) && (fh.is_last || fh.duration > 0);
  const bool full = !fh.have_crop || (fh.x0 <= 0 && fh.y0 <= 0 && int64_t(fh.x0) + fh.width >= int64_t(m.xsize) && int64_t(fh.y0) + fh.height >= int64_t(m.ysize));
  return shown && full && fh.blending.mode == 0;
}

// ---------------------------------------------------------------- pass 1: info + metadata
struct Headers { ContainerInfo ci; ImageMetadata meta; size_t frame_pos = 0; /* byte offset of the first frame in the codestream */ };

static int KnownProfileOf(const ColorEncoding& c) {   // N/Decoder/JxlDecoder.cpp:36-108
  if (c.want_icc || c.have_gamma) return -1;
  if (c.color_space == kCsRGB && c.white_point == kWpD65) {
    if (c.tf == kTfLinear) { if (c.primaries == kPrSRGB) return 1; if (c.primaries == kPr2100) return 6; }
    else if (c.tf == kTfSRGB) { if (c.primaries == kPrSRGB) return 0; if (c.primaries == kPrP3) return 4; }
    else if (c.tf == kTf709) { if (c.primaries == kPrSRGB) return 5; }
    else if (c.primaries == kPr2100) { if (c.tf == kTfPQ) return 7; }
  } else if (c.color_space == kCsGray && c.white_point == kWpD65) { if (c.tf == kTfLinear) return 2; if (c.tf == kTfSRGB) return 3; }
  return -1;
}
// Output encoding of the samples (Appendix C-1): original enum encoding when expressible without a CMS, else sRGB.
static ColorEncoding OutputEncoding(const ImageMetadata& m) {
  ColorEncoding t; if (!m.xyb_encoded) return m.ce;
  bool ok = !m.ce.want_icc && (m.ce.have_gamma || m.ce.tf != kTfUnknown) && m.ce.color_space != kCsXYB && m.ce.color_space != kCsUnknown;
  if (ok) return m.ce; t.color_space = m.ce.color_space == kCsGray ? kCsGray : kCsRGB; t.intent = 0; return t;
}

static void ParseHeadersInto(const uint8_t* data, size_t size, Headers* h, ParsedInfo* info) {
  int sig = SignatureCheck(data, size); if (sig == 0) throw StatusError(DecoderStatus_InvalidFileSignature);
  h->ci = ParseContainer(data, size); info->is_container = h->ci.is_container; const ByteSpan& cs = h->ci.codestream;
  JXLG_CHECK(cs.size() >= 2 && cs[0] == 0xFF && cs[1] == 0x0A, "codestream signature");
  BitReader br(cs.data() + 2, cs.size() - 2); h->meta = ReadImageHeaders(br); const ImageMetadata& m = h->meta; h->frame_pos = 2 + br.pos / 8;
  // BASIC_INFO decisions, N/Decoder/JxlDecoder.cpp:461-561
  if (m.xsize > 0x7fffffffu || m.ysize > 0x7fffffffu) throw StatusError(DecoderStatus_ImageDimensionExceedsInt32);
  int alpha = m.alpha_index(); uint32_t alpha_bits = alpha >= 0 ? m.ec[alpha].bd.bits : 0; info->has_alpha = alpha_bits != 0; int black = -1; bool first_alpha = false;
  for (size_t i = 0; i < m.ec.size(); i++) {
    if (m.ec[i].type == kEcBlack) { if (black < 0) black = int(i); else throw StatusError(DecoderStatus_UnsupportedChannelFormat); }
    else if (m.ec[i].type == kEcAlpha) { if (info->has_alpha && !first_alpha) first_alpha = true; else throw StatusError(DecoderStatus_UnsupportedChannelFormat); }
  }
  int cc = m.num_color_channels(); info->num_channels = cc + (info->has_alpha ? 1 : 0); info->format = cc == 1 ? 0 : (black >= 0 ? 2 : 1); info->sample_type = 0; info->width = m.xsize; info->height = m.ysize;
  if (m.bd.exp_bits > 0) {
    JXLG_CHECK(info->format != 2, "Floating point CMYK images are not supported.");
    if (m.bd.bits <= 16) info->sample_type = 2; else if (m.bd.bits <= 32) info->sample_type = 3; else throw Error("Unsupported floating point bit depth: " + std::to_string(m.bd.bits) + ".");
  } else if (m.bd.bits > 8) {
    if (m.bd.bits <= 16) { JXLG_CHECK(info->format != 2, "CMYK64 images are not supported."); info->sample_type = 1; }
    else throw Error("Unsupported integer bit depth: " + std::to_string(m.bd.bits) + ".");
  }
  if (m.orientation >= 5) std::swap(info->width, info->height);
  // COLOR_ENCODING, :562-686 — the profile reported is the one describing the delivered samples
  ColorEncoding out_ce = OutputEncoding(m); info->known_profile = KnownProfileOf(out_ce); if (m.ce.want_icc && !m.xyb_encoded) info->icc = m.icc;
  // encodings libjxl can express but the 8 known enums cannot (custom primaries / white point, pure gamma, DCI): synthesised ICC (SURVEY §8f-2)
  if (info->known_profile < 0 && info->icc.empty() && !out_ce.want_icc) info->icc = SynthesizeIcc(out_ce);
  // BOX events, :687-784: first Exif box only, every xml box, brob decompressed; container files only
  for (const Box& b : h->ci.boxes) {
    const uint8_t* p = b.data; size_t n = b.size; char type[5]; memcpy(type, b.type, 5); std::vector<uint8_t> tmp;
    if (!strcmp(type, "brob") && n >= 4) { memcpy(type, p, 4); type[4] = 0; if (!strcmp(type, "Exif") || !strcmp(type, "xml ")) { tmp = BrotliDecompress(p + 4, n - 4); p = tmp.data(); n = tmp.size(); } }
    if (!strcmp(type, "Exif")) { if (!info->has_exif) { info->has_exif = true; info->exif.assign(p, p + n); } } else if (!strcmp(type, "xml ")) info->xmp.emplace_back(p, p + n);
  }
}

ParsedInfo ParseInfo(const uint8_t* data, size_t size) { Headers h; ParsedInfo info; ParseHeadersInto(data, size, &h, &info); return info; }

// ---------------------------------------------------------------- blob builder
struct Blob {
  std::vector<uint8_t> b; bool uses_lz77 = false;   // some code of this frame is LZ77-enabled: the kernels need their windows
  uint32_t Add(const void* p, size_t n, size_t align = 16) { if (b.empty()) b.resize(16, 0);   /* offset 0 means "no table" to the kernels */ size_t o = (b.size() + align - 1) / align * align; b.resize(o + n); if (n) memcpy(&b[o], p, n); JXLG_CHECK(b.size() < (size_t(1) << 31), "table blob too large"); return uint32_t(o); }
  DCode AddCode(const Code& c) {
    DCode d; memset(&d, 0, sizeof(d)); d.num_ctx = uint32_t(c.ctx_map.size()); d.num_clusters = uint32_t(c.cfg.size()); d.log_alpha = uint32_t(c.log_alpha); d.use_prefix = c.use_prefix;
    d.ctx_map_off = Add(c.ctx_map.data(), c.ctx_map.size()); std::vector<DHybrid> cfg(c.cfg.size()); for (size_t i = 0; i < cfg.size(); i++) cfg[i] = DHybrid{uint8_t(c.cfg[i].split_exp), uint8_t(c.cfg[i].msb), uint8_t(c.cfg[i].lsb), 0};
    d.cfg_off = Add(cfg.data(), cfg.size() * sizeof(DHybrid));
    std::vector<uint32_t> info(c.cfg.size());
    for (size_t k = 0; k < c.cfg.size(); k++) { uint32_t cs = 0xffff;
      if (!c.use_prefix) { for (size_t sy = 0; sy < c.ans[k].freq.size(); sy++) if (c.ans[k].freq[sy] == kAnsTab) cs = uint32_t(sy); } else if (c.prefix[k].max_len == 0) cs = uint32_t(c.prefix[k].single);
      info[k] = c.cfg[k].split_exp | (c.cfg[k].msb << 8) | (c.cfg[k].lsb << 12) | (cs << 16); }
    d.info_off = Add(info.data(), info.size() * 4);
    if (c.lz77) { d.lz77 = 1; d.lz_min_symbol = c.lz_min_symbol; d.lz_min_length = c.lz_min_length; d.lz_len_info = c.lz_len_cfg.split_exp | (c.lz_len_cfg.msb << 8) | (c.lz_len_cfg.lsb << 12);
      d.lz_dist_cluster = c.ctx_map.back(); uses_lz77 = true; }
    if (!c.use_prefix) {
      size_t ts = size_t(1) << c.log_alpha; std::vector<DAlias> al(c.ans.size() * ts);
      for (size_t k = 0; k < c.ans.size(); k++) { const AnsTable& t = c.ans[k]; for (size_t i = 0; i < ts; i++) al[k * ts + i] = PackAlias(t.cutoff[i], t.right[i], t.off1[i], t.freq[i], t.freq[t.right[i]]); }
      d.alias_off = Add(al.data(), al.size() * 8);
    } else {
      std::vector<uint32_t> desc(2 * c.prefix.size());
      for (size_t k = 0; k < c.prefix.size(); k++) { const PrefixTable& t = c.prefix[k]; std::vector<uint32_t> lut(size_t(1) << t.max_len);
        if (t.max_len == 0) lut[0] = uint32_t(t.single) << 4; else for (size_t i = 0; i < lut.size(); i++) lut[i] = (uint32_t(t.lut_sym[i]) << 4) | t.lut_len[i];
        desc[2 * k] = Add(lut.data(), lut.size() * 4); desc[2 * k + 1] = uint32_t(t.max_len); }
      d.prefix_off = Add(desc.data(), desc.size() * 4);
    }
    return d;
  }
};

static const std::vector<float>& DefaultDequant(int t) { static std::vector<float> tab[kNumQuantTables]; static std::once_flag once; std::call_once(once, []() { for (int i = 0; i < kNumQuantTables; i++) tab[i] = ComputeDequantTable(i, LibraryEncoding(i)); }); return tab[t]; }
static const std::vector<uint32_t>& NaturalOrderCached(int o) { static std::vector<uint32_t> tab[kNumOrders]; static std::once_flag once; std::call_once(once, []() { for (int i = 0; i < kNumOrders; i++) { int s = kOrderStrategy[i]; tab[i] = NaturalOrder(std::min(kCoveredX[s], kCoveredY[s]), std::max(kCoveredX[s], kCoveredY[s])); } }); return tab[o]; }

static QuantEncoding ReadQuantEncodingHost(BitReader& br, int t) {
  auto read_params = [&](DctParams& p) { p.num_bands = int(br.ReadBits(4)) + 1; for (int c = 0; c < 3; c++) { for (int i = 0; i < p.num_bands; i++) p.bands[c][i] = br.F16(); JXLG_CHECK(p.bands[c][0] >= 1e-8f, "distance band"); p.bands[c][0] *= 64.0f; } };
  QuantEncoding e; e.mode = int(br.ReadBits(3)); bool small = kTableRows[t] == 1 && kTableCols[t] == 1;
  switch (e.mode) {
    case kQModeLibrary: return LibraryEncoding(t);
    case kQModeId: JXLG_CHECK(small, "quant mode/table mismatch"); for (int c = 0; c < 3; c++) for (int i = 0; i < 3; i++) e.idw[c][i] = br.F16() * 64.0f; break;
    case kQModeDCT2: JXLG_CHECK(small, "quant mode/table mismatch"); for (int c = 0; c < 3; c++) for (int i = 0; i < 6; i++) e.dct2w[c][i] = br.F16() * 64.0f; break;
    case kQModeDCT4: JXLG_CHECK(small, "quant mode/table mismatch"); for (int c = 0; c < 3; c++) for (int i = 0; i < 2; i++) e.dct4mul[c][i] = br.F16(); read_params(e.dct4); break;
    case kQModeDCT4x8: JXLG_CHECK(small, "quant mode/table mismatch"); for (int c = 0; c < 3; c++) e.dct4x8mul[c] = br.F16(); read_params(e.dct4x8); break;
    case kQModeDCT: read_params(e.dct); break;
    default: throw Error("AFV / RAW quant table encodings are not supported");
  }
  return e;
}

LayeredStill::LayeredStill() : Error("layered (multi-frame) files are decoded by LoadImage / JxlB200LoadImageBgra only, not by the batch and band calls") {}

// ---------------------------------------------------------------- the job
class DecodeJob {
 public:
  Headers hd; ParsedInfo info; FrameHeader fh; Toc toc; DFrame h; Blob blob; bool bgra = false, device_output = false, layer = false; DLocalTree global_local = DLocalTree(); std::vector<DModOp> ops_host; bool mod_has_lf_level = false; uint64_t mod_total_ints = 0;   /* int32 samples of all Modular planes: coded channels + the outputs of palette expansions */
  Buf d_frame, d_blob, d_comp, d_lfq, d_lf, d_lf_tmp, d_acs, d_qf, d_sharp, d_lfidx, d_ytox, d_ytob, d_hfmeta, d_coeffs, d_xyb, d_xyb_tmp, d_sigma, d_mod, d_wp, d_out, d_err, h_out, h_err, h_comp, h_blob, h_misc, d_gother, d_nz, d_acend, d_lz, d_gpal, d_layer_out, h_layer_out;   /* *_layer_out: the finished canvas of a layered file (owned by the job of the frame that is shown) */
  std::function<void()> ac_budget; int ac_lanes = 1; bool phased = false; size_t coeffs_bytes = 0, xyb_row_shift = 0;
  bool defer_entropy = false, lf_pending = false, ac_pending = false;   // bundle mode: the LF / AC entropy launch is left to DecodeBundleLaunch*
  cudaStream_t stream = nullptr; cudaEvent_t ev[8] = {nullptr}; bool timed = false; size_t out_bytes = 0; size_t comp_size = 0; const uint8_t* frame_ptr = nullptr; size_t frame_off = 0;
  bool has_tree = false; Tree tree; Code tree_code; uint64_t global_data_bitpos = 0; bool global_has_data = false;
  std::vector<Code> ac_codes; uint32_t hf_blob_mark = 0; uint32_t frame_uploads = 0; uint8_t* ext_out_device = nullptr; uint8_t* ext_out_pinned = nullptr;
  ~DecodeJob() { for (auto& e : ev) if (e) cudaEventDestroy(e); }

  void Setup(const DecodeRequest& req);
  void RunLf(const DecodeRequest& req); void RunAc(); void RunRender();
  void ReservePools(size_t count) { Buf* all[] = {&d_frame, &d_blob, &d_comp, &d_lfq, &d_lf, &d_lf_tmp, &d_acs, &d_qf, &d_sharp, &d_lfidx, &d_ytox, &d_ytob, &d_hfmeta, &d_coeffs, &d_xyb, &d_xyb_tmp, &d_sigma, &d_mod, &d_wp, &d_out, &d_err, &h_out, &h_err, &h_comp, &h_blob, &h_misc, &d_gother, &d_nz, &d_acend};
    // several buffers of a job share a size class (the small ones all round to 4 KiB): reserve count x multiplicity per class
    std::map<std::pair<Pool*, size_t>, size_t> mult;
    for (Buf* b : all) if (b->p && b->pool) mult[std::make_pair(b->pool, Pool::Round(b->n))]++;
    for (auto& kv : mult) kv.first.first->Reserve(kv.first.second, (count + 1) * kv.second); }
  void Run(const DecodeRequest& req) { RunLf(req); RunAc(); RunRender(); }
  void ParseLfGlobal(BitReader& br); uint32_t AddTree(const Tree& t, uint32_t* uses_wp); DLocalTree ParseLocalTree(BitReader& br, size_t pixels);
  void ParseHfGlobal(BitReader& br);
  void AllocateAndUpload(const DecodeRequest& req);
  void UploadFrame();
};

// An MA tree as the kernels walk it (flat int4 nodes in the blob); *uses_wp: some node needs the weighted predictor's state.
uint32_t DecodeJob::AddTree(const Tree& t, uint32_t* uses_wp) {
  std::vector<DTreeNode> nodes(t.size());
  for (size_t i = 0; i < t.size(); i++) { const TreeNode& n = t[i];
    if (n.property >= 0) { nodes[i] = make_int4(n.property, n.splitval, n.lchild, n.rchild); if (n.property == 15) *uses_wp = 1;
      JXLG_CHECK(n.property < 16 + 4 * 4, "MA-tree properties of more than four previous channels are not supported by the GPU decoder"); }
    else { nodes[i] = make_int4(-1, (n.leaf_id << 4) | n.predictor, n.offset, int(n.multiplier)); if (n.predictor == 6) *uses_wp = 1; } }
  return blob.Add(nodes.data(), nodes.size() * sizeof(DTreeNode));
}
// A sub-bitstream with its own MA tree (use_global_tree = 0): tree and code follow its header; parsed here, tables into the blob.
DLocalTree DecodeJob::ParseLocalTree(BitReader& br, size_t pixels) {
  DLocalTree lt; memset(&lt, 0, sizeof(lt));
  Tree t = DecodeTree(br, std::max<size_t>(std::min<size_t>(size_t(1) << 22, 1024 + pixels), 1 << 10)); Code code = DecodeCode(br, NumLeaves(t)); JXLG_CHECK(!br.overrun, "local MA tree truncated");
  uint32_t wp = 0; lt.tree_off = AddTree(t, &wp); lt.tree_size = uint32_t(t.size()); lt.uses_wp = wp; lt.code = blob.AddCode(code); lt.present = 1; if (wp) h.uses_wp = 1;   // the weighted-predictor kernels for the whole frame
  return lt;
}

// The global Modular image: its channels as coded (the forward side of every transform its header lists, SURVEY.md A.7; libjxl's MetaApply)
// and the inverse transforms as device ops.
struct ModPlan {
  std::vector<DModChannel> coded, out;   // the channels as coded / the image's own channels after the inverse transforms, each with its plane
  std::vector<DModOp> ops;               // the inverse transforms in the order the kernels run them: last transform first
  size_t global_channels = 0;            // coded channels [0, global_channels) are held by the global section
  bool has_lf_level = false;             // some later channel is coded in the LF-group sections
  uint64_t total_ints = 0;               // int32 samples of all planes: coded channels + the outputs of the ops
};
// The walk keeps channel identities (indices into `geo`), not positions. An RCT works in place on three of them; a palette consumes
// begin..end and creates an index and a palette channel; a squeeze step creates an average and a residual channel for each channel it
// consumes. Every op outputs the channels its transform consumed, so each channel is either coded or made by exactly one op.
static ModPlan PlanModularImage(const ImageMetadata& m, const FrameHeader& fh, const GroupHeader& gh) {
  std::vector<DModChannel> geo;   // every channel the forward transforms pass through; the image's own channels first
  if (fh.encoding == 1) { JXLG_CHECK(!m.xyb_encoded, "XYB-encoded Modular frames are not supported"); int nc = m.ce.color_space == kCsGray ? 1 : 3; for (int c = 0; c < nc; c++) geo.push_back(DModChannel{fh.xsize, fh.ysize, 0, 0, 0}); }
  for (size_t i = 0; i < m.ec.size(); i++) { JXLG_CHECK(fh.ec_upsampling[i] == 1, "upsampling is not supported"); uint32_t s = m.ec[i].dim_shift; geo.push_back(DModChannel{DivCeil(fh.xsize, 1u << s), DivCeil(fh.ysize, 1u << s), s, s, 0}); }
  JXLG_CHECK(geo.size() <= 8, "too many Modular channels"); const size_t num_image_channels = geo.size();
  std::vector<uint32_t> ch(num_image_channels); for (size_t i = 0; i < ch.size(); i++) ch[i] = uint32_t(i);   // the channel list
  auto add = [&](DModChannel c) { geo.push_back(c); return uint32_t(geo.size() - 1); };
  ModPlan plan; std::vector<DModOp>& ops = plan.ops;
  // an op goes in front of the ops of earlier transforms; `at` keeps the channels of one squeeze step in order
  auto new_op = [&](uint32_t kind, size_t at) -> DModOp& { JXLG_CHECK(ops.size() < 1024, "too many Modular transform steps"); DModOp& o = *ops.insert(ops.begin() + at, DModOp()); o.kind = kind; return o; };
  int nb_meta = 0;
  for (const Transform& t : gh.transforms) {
    if (t.id == 0) {
      JXLG_CHECK(t.begin_c + 3 <= ch.size(), "RCT channel range"); const DModChannel a = geo[ch[t.begin_c]];
      for (int k = 1; k < 3; k++) JXLG_CHECK(geo[ch[t.begin_c + k]].w == a.w && geo[ch[t.begin_c + k]].h == a.h, "RCT channel sizes");
      DModOp& op = new_op(0, 0); op.rct_type = t.rct_type; op.w = a.w; op.h = a.h; for (int k = 0; k < 3; k++) op.p[k] = ch[t.begin_c + k];
      continue;
    }
    if (t.id == 1) {
      const uint32_t end_c = t.begin_c + t.num_c - 1; JXLG_CHECK(t.num_c >= 1 && t.num_c <= 4 && end_c < ch.size(), "palette channel range"); const DModChannel first = geo[ch[t.begin_c]];
      for (uint32_t c = t.begin_c + 1; c <= end_c; c++) { const DModChannel& o = geo[ch[c]]; JXLG_CHECK(o.w == first.w && o.h == first.h && o.hshift == first.hshift && o.vshift == first.vshift, "palette channel sizes"); }
      if (int(t.begin_c) < nb_meta) { JXLG_CHECK(int(end_c) < nb_meta, "palette across the meta-channel boundary"); nb_meta += 2 - int(t.num_c); } else nb_meta += 1;
      JXLG_CHECK(t.nb_deltas == 0 || t.predictor != 6, "delta palettes with the weighted predictor are not supported");
      DModOp& op = new_op(1, 0); op.num_c = t.num_c; op.pal_w = t.nb_colors + t.nb_deltas; op.nb_deltas = t.nb_deltas; op.predictor = t.predictor; op.w = first.w; op.h = first.h;
      for (uint32_t k = 0; k < t.num_c; k++) op.out[k] = ch[t.begin_c + k];
      op.p[0] = add(first); op.p[1] = add(DModChannel{op.pal_w, t.num_c, 0, 0, 0});   // the palette itself: one row per colour channel, always coded in the global section
      ch.erase(ch.begin() + t.begin_c + 1, ch.begin() + end_c + 1); ch[t.begin_c] = uint32_t(op.p[0]); ch.insert(ch.begin(), uint32_t(op.p[1]));
      continue;
    }
    // Squeeze: every step halves its channels (average, shift + 1) and appends / inserts the residual channels
    std::vector<SqueezeParams> steps = t.squeezes;
    if (steps.empty()) {   // default parameters (libjxl's DefaultSqueezeParameters): chroma first when the first two channels match, then alternate until <= 8 x 8
      const int nb = int(ch.size()) - nb_meta; JXLG_CHECK(nb > 0, "squeeze without channels"); uint32_t w = geo[ch[nb_meta]].w, hh = geo[ch[nb_meta]].h;
      if (nb > 2 && geo[ch[nb_meta + 1]].w == w && geo[ch[nb_meta + 1]].h == hh) { SqueezeParams p; p.horizontal = true; p.in_place = false; p.begin_c = uint32_t(nb_meta + 1); p.num_c = 2; steps.push_back(p); p.horizontal = false; steps.push_back(p); }
      SqueezeParams p; p.begin_c = uint32_t(nb_meta); p.num_c = uint32_t(nb); p.in_place = true;
      if (!(w > hh)) { if (hh > 8) { p.horizontal = false; steps.push_back(p); hh = (hh + 1) / 2; } }
      while (w > 8 || hh > 8) { if (w > 8) { p.horizontal = true; steps.push_back(p); w = (w + 1) / 2; } if (hh > 8) { p.horizontal = false; steps.push_back(p); hh = (hh + 1) / 2; } }
    }
    for (const SqueezeParams& sq : steps) {
      const uint32_t end_c = sq.begin_c + sq.num_c - 1; JXLG_CHECK(sq.num_c >= 1 && end_c < ch.size(), "squeeze channel range"); JXLG_CHECK(int(sq.begin_c) >= nb_meta, "squeeze of meta channels is not supported");
      const size_t offset = sq.in_place ? size_t(end_c) + 1 : ch.size();
      for (uint32_t c = sq.begin_c; c <= end_c; c++) {
        const DModChannel in = geo[ch[c]]; DModChannel a = in, r;
        if (sq.horizontal) { a.w = (in.w + 1) / 2; a.hshift++; r = DModChannel{in.w - a.w, a.h, a.hshift, a.vshift, 0}; }
        else { a.h = (in.h + 1) / 2; a.vshift++; r = DModChannel{a.w, in.h - a.h, a.hshift, a.vshift, 0}; }
        JXLG_CHECK(a.hshift < 30 && a.vshift < 30, "squeeze depth");
        DModOp& op = new_op(2, c - sq.begin_c); op.rct_type = sq.horizontal ? 1 : 0; op.w = a.w; op.h = a.h; op.num_c = r.w; op.pal_w = r.h; op.out[0] = ch[c];
        op.p[0] = ch[c] = add(a); op.p[1] = add(r); ch.insert(ch.begin() + offset + (c - sq.begin_c), uint32_t(op.p[1]));
      }
    }
  }
  JXLG_CHECK(ch.size() <= 255, "too many Modular channels");
  // planes: the coded channels in coded order, then the outputs of the ops in the order they run; p[] and out[] turn from channels into planes
  uint64_t off = 0; for (uint32_t id : ch) { DModChannel& c = geo[id]; c.plane_off = off; off += uint64_t(c.w) * c.h; plan.coded.push_back(c); }
  for (DModOp& op : ops) {
    const uint32_t nout = op.kind == 0 ? 0 : op.kind == 1 ? op.num_c : 1;
    for (uint32_t k = 0; k < nout; k++) { DModChannel& c = geo[op.out[k]]; c.plane_off = off; off += uint64_t(c.w) * c.h; op.out[k] = c.plane_off; }
    for (int k = 0; k < (op.kind == 0 ? 3 : 2); k++) op.p[k] = geo[op.p[k]].plane_off;
  }
  plan.out.assign(geo.begin(), geo.begin() + num_image_channels); plan.total_ints = off;
  // which channels the global section holds: meta channels always, then every channel up to the first one larger than a group
  const std::vector<DModChannel>& cc = plan.coded; size_t c = 0; for (; c < cc.size(); c++) if (int(c) >= nb_meta && (cc[c].w > fh.group_dim || cc[c].h > fh.group_dim)) break;
  plan.global_channels = c;
  for (size_t i = c; i < cc.size(); i++) if (std::min(cc[i].hshift, cc[i].vshift) >= 3 && cc[i].w && cc[i].h) plan.has_lf_level = true;   // coded in the LF-group sections
  return plan;
}

void DecodeJob::ParseLfGlobal(BitReader& br) {
  const ImageMetadata& m = hd.meta;
  JXLG_CHECK(!(fh.flags & (kFlagPatches | kFlagSplines | kFlagNoise)), "patches/splines/noise are not supported");
  float lf_dequant[3] = {1.0f / 4096, 1.0f / 512, 1.0f / 256}; uint32_t global_scale = 1, quant_lf = 16; BlockCtxMap bctx; uint32_t color_factor = 84; float base_x = 0.f, base_b = 1.f; int32_t xlf = 0, blf = 0;
  // LfChannelDequantization is read for every frame encoding: Modular frames carry the bundle too (unused there)
  if (!br.Bool()) for (int c = 0; c < 3; c++) { lf_dequant[c] = br.F16() * (1.0f / 128.0f); JXLG_CHECK(lf_dequant[c] >= 1e-8f, "lf dequant"); }
  if (fh.encoding == 0) {
    JXLG_CHECK(!(fh.flags & kFlagUseLfFrame), "LF frames are not supported");
    global_scale = br.U32(BitsOffset(11, 1), BitsOffset(11, 2049), BitsOffset(12, 4097), BitsOffset(16, 8193)); quant_lf = br.U32(Val(16), BitsOffset(5, 1), BitsOffset(8, 1), BitsOffset(16, 1));
    if (!br.Bool()) {
      bctx.num_lf_ctxs = 1; for (int j = 0; j < 3; j++) { uint32_t n = br.ReadBits(4); bctx.lf_thr[j].resize(n); for (auto& t : bctx.lf_thr[j]) t = UnpackSigned(br.U32(Bits(4), BitsOffset(8, 16), BitsOffset(16, 272), BitsOffset(32, 65808))); bctx.num_lf_ctxs *= n + 1; }
      uint32_t nq = br.ReadBits(4); bctx.qf_thr.resize(nq); for (auto& t : bctx.qf_thr) t = br.U32(Bits(2), BitsOffset(3, 4), BitsOffset(5, 12), BitsOffset(8, 44)) + 1;
      JXLG_CHECK(bctx.num_lf_ctxs * (nq + 1) <= 64, "block context map too large"); size_t ncl = 0; bctx.map = DecodeContextMap(br, size_t(3) * kNumOrders * bctx.num_lf_ctxs * (nq + 1), &ncl); JXLG_CHECK(ncl <= 16, "too many block contexts"); bctx.num_ctxs = uint32_t(ncl);
    }
    if (!br.Bool()) { color_factor = br.U32(Val(84), Val(256), BitsOffset(8, 2), BitsOffset(16, 258)); base_x = br.F16(); base_b = br.F16(); xlf = int32_t(br.ReadBits(8)) - 128; blf = int32_t(br.ReadBits(8)) - 128; }
    float inv_gs = 65536.0f / float(global_scale), lfinv = inv_gs / float(quant_lf);
    for (int c = 0; c < 3; c++) h.lf_fac[c] = lf_dequant[c] * lfinv;
    h.inv_color_factor = 1.0f / float(color_factor); h.base_x = base_x; h.base_b = base_b; h.cfl_x_lf = base_x + float(xlf) / float(color_factor); h.cfl_b_lf = base_b + float(blf) / float(color_factor);
    h.inv_gs = inv_gs; h.quant_scale = float(global_scale) / 65536.0f; h.xm = std::pow(0.8f, float(fh.x_qm_scale) - 2.0f); h.bm = std::pow(0.8f, float(fh.b_qm_scale) - 2.0f);
    for (int i = 0; i < 4; i++) h.quant_bias[i] = m.opsin.quant_bias[i];
    h.nb_block_ctx = bctx.num_ctxs; h.num_lf_ctxs = bctx.num_lf_ctxs; h.n_qf_thr = uint32_t(bctx.qf_thr.size()); for (size_t i = 0; i < bctx.qf_thr.size(); i++) h.qf_thr[i] = bctx.qf_thr[i];
    for (int j = 0; j < 3; j++) { h.n_lf_thr[j] = uint32_t(bctx.lf_thr[j].size()); for (size_t i = 0; i < bctx.lf_thr[j].size(); i++) h.lf_thr[j][i] = bctx.lf_thr[j][i]; }
    h.bctx_map_off = blob.Add(bctx.map.data(), bctx.map.size());
  }
  has_tree = br.Bool();
  if (has_tree) {
    size_t nch = (fh.encoding == 1 ? 3 : 0) + m.ec.size(); size_t limit = std::min<size_t>(size_t(1) << 22, 1024 + size_t(fh.xsize) * fh.ysize * std::max<size_t>(nch, 1) / 16); limit = std::max<size_t>(limit, 1 << 16);
    tree = DecodeTree(br, limit); tree_code = DecodeCode(br, NumLeaves(tree));
    uint32_t uses_wp = 0; h.tree_off = AddTree(tree, &uses_wp); h.tree_size = uint32_t(tree.size()); h.uses_wp = uses_wp; h.mod_code = blob.AddCode(tree_code);
  }
  h.has_tree = has_tree;
  h.mod_bitdepth = m.bd.bits; { uint32_t mb = m.bd.bits; for (const auto& e : m.ec) mb = std::max(mb, e.bd.bits); h.mod_wide = (mb > 20 || !m.modular_16bit) ? 1 : 0; }
  // global Modular image: colour channels (Modular frames) + extra channels
  GroupHeader gheader; ModPlan plan;
  if (fh.encoding == 1 || !m.ec.empty()) { gheader = ReadGroupHeader(br); plan = PlanModularImage(m, fh, gheader); }
  const std::vector<DModChannel>& ch = plan.coded; const size_t nglobal = plan.global_channels;
  h.num_mod_channels = uint32_t(ch.size()); h.first_group_channel = uint32_t(nglobal); mod_has_lf_level = plan.has_lf_level; mod_total_ints = plan.total_ints; global_has_data = false;
  h.mod_ch_off = 0; if (ch.size() <= 8) { for (size_t i = 0; i < ch.size(); i++) h.mod_ch[i] = ch[i]; } else h.mod_ch_off = blob.Add(ch.data(), ch.size() * sizeof(DModChannel));
  for (size_t i = 0; i < plan.out.size(); i++) h.out_ch[i] = plan.out[i];
  if (!ch.empty()) {
    size_t nonempty = 0; for (size_t i = 0; i < nglobal; i++) if (ch[i].w && ch[i].h) nonempty++;
    if (nonempty) {
      global_has_data = true;
      if (!gheader.use_global_tree) { size_t px = 0; for (size_t i = 0; i < nglobal; i++) px += size_t(ch[i].w) * ch[i].h; global_local = ParseLocalTree(br, px); }   // data starts where this parse stops
      else JXLG_CHECK(has_tree, "the global Modular stream uses the global MA tree, but the frame has none");
    }
    const WPHeader& gw = gheader.wp; h.global_wp.p1 = gw.p1; h.global_wp.p2 = gw.p2; h.global_wp.p3a = gw.p3a; h.global_wp.p3b = gw.p3b; h.global_wp.p3c = gw.p3c; h.global_wp.p3d = gw.p3d; h.global_wp.p3e = gw.p3e;
    for (int i = 0; i < 4; i++) h.global_wp.w[i] = gw.w[i];
  }
  ops_host = plan.ops; h.num_ops = uint32_t(ops_host.size()); h.ops_off = 0;
  if (ops_host.size() <= 4) { for (size_t i = 0; i < ops_host.size(); i++) h.ops[i] = ops_host[i]; } else h.ops_off = blob.Add(ops_host.data(), ops_host.size() * sizeof(DModOp));
}

void DecodeJob::ParseHfGlobal(BitReader& br) {
  bool all_default = br.Bool();
  const StaticBlob& sb = DeviceStaticBlob(); h.static_blob = sb.dev;
  for (int t = 0; t < kNumQuantTables; t++) { if (all_default) h.dq_off[t] = sb.dq_off[t]; else { std::vector<float> d = ComputeDequantTable(t, ReadQuantEncodingHost(br, t)); h.dq_off[t] = blob.Add(d.data(), d.size() * 4); } }
  h.num_hf_presets = 1 + br.ReadBits(CeilLog2(fh.num_groups));
  ac_codes.resize(fh.passes.num_passes);
  for (uint32_t p = 0; p < fh.passes.num_passes; p++) {
    uint32_t used = br.U32(Val(0x5F), Val(0x13), Val(0), Bits(13)); for (int i = 0; i < kNumOrders * 3; i++) h.order_off[p][i] = sb.nat_off[i / 3];
    if (used) { Code c = DecodeCode(br, 8); SymbolReader r(&c, &br);
      for (int o = 0; o < kNumOrders; o++) if (used >> o & 1) for (int chn = 0; chn < 3; chn++) { const auto& nat = NaturalOrderCached(o); size_t size = nat.size(); std::vector<uint32_t> perm = ReadPermutation(r, size / 64, size), out(size);
        for (size_t k = 0; k < size; k++) out[k] = nat[perm[k]]; h.order_off[p][o * 3 + chn] = blob.Add(out.data(), out.size() * 4); }
      JXLG_CHECK(r.CheckFinal(), "coefficient order ANS final state"); }
    ac_codes[p] = DecodeCode(br, size_t(495) * h.num_hf_presets * h.nb_block_ctx); h.ac_code[p] = blob.AddCode(ac_codes[p]);
  }
}

void DecodeJob::Setup(const DecodeRequest& req) {
  const ImageMetadata& m = hd.meta; const ByteSpan& cs = hd.ci.codestream; size_t pos = req.layer ? req.layer_pos : hd.frame_pos; layer = req.layer;
  if (m.have_preview && !req.layer) { ImageMetadata pm = m; pm.xsize = m.preview_x; pm.ysize = m.preview_y; BitReader br(cs.data() + pos, cs.size() - pos); FrameHeader pf = ReadFrameHeader(br, pm); Toc t = ReadToc(br, pf); pos += br.pos / 8 + t.total; JXLG_CHECK(pos <= cs.size(), "preview frame truncated"); }
  BitReader br(cs.data() + pos, cs.size() - pos); fh = ReadFrameHeader(br, m);
  JXLG_CHECK(fh.frame_type != kFrameLF, "LF frames are not supported");
  JXLG_CHECK(fh.upsampling == 1, "upsampling is not supported"); JXLG_CHECK(!fh.do_ycbcr, "YCbCr (JPEG-recompressed) frames are not supported");
  if (!req.layer) {   // the plain single-frame file; layered files go through DecodeOnGpu's compositing loop, which sets req.layer for every frame
    const bool full = !fh.have_crop || (fh.x0 == 0 && fh.y0 == 0 && fh.width == m.xsize && fh.height == m.ysize);
    if (!FrameIsPlain(fh, m) || !full) throw LayeredStill();
  }
  JXLG_CHECK(fh.passes.num_passes <= uint32_t(kMaxPasses), "too many passes");
  JXLG_CHECK(fh.encoding != 0 || m.xyb_encoded, "VarDCT frames that are not XYB-encoded are not supported");
  toc = ReadToc(br, fh); frame_off = pos + br.pos / 8; JXLG_CHECK(frame_off + toc.total <= cs.size(), "JxlDecoderProcessInput needs more input, but it already received the entire image.");
  info.frame_name = fh.name; info.bpp = double(cs.size()) * 8.0 / (double(m.xsize) * m.ysize);
  memset(&h, 0, sizeof(h)); bgra = req.bgra; device_output = req.device_output;
  ac_lanes = 1; while (ac_lanes * 2 <= req.ac_lanes && ac_lanes < 32) ac_lanes *= 2;
  h.xsize = fh.xsize; h.ysize = fh.ysize; h.xb = fh.xblocks; h.yb = fh.yblocks; h.xpad = h.xb * 8; h.ypad = h.yb * 8; h.xt = (h.xb + 7) / 8; h.yt = (h.yb + 7) / 8; h.xgroups = fh.xgroups; h.ygroups = fh.ygroups; h.num_groups = fh.num_groups;
  h.xlfgroups = fh.xlfgroups; h.ylfgroups = fh.ylfgroups; h.num_lf_groups = fh.num_lf_groups; h.group_dim = fh.group_dim; h.num_passes = fh.passes.num_passes; h.encoding = fh.encoding; h.flags = uint32_t(fh.flags);
  info.group_dim = h.group_dim; info.num_group_rows = h.ygroups;
  if (req.band_begin || req.band_end) {
    JXLG_CHECK(req.band_begin < req.band_end && req.band_end <= h.ygroups, "band decode: group-row range out of bounds"); JXLG_CHECK(m.orientation == 1, "band decode needs identity orientation");
    h.band_on = 1; h.out_g0 = req.band_begin; h.out_g1 = req.band_end; h.comp_g0 = req.band_begin ? req.band_begin - 1 : 0; h.comp_g1 = std::min(h.ygroups, req.band_end + 1);
    h.out_y0 = h.out_g0 * h.group_dim; h.out_y1 = std::min(h.ysize, h.out_g1 * h.group_dim);
  }
  for (uint32_t p = 0; p < h.num_passes; p++) { h.pass_shift[p] = p + 1 < h.num_passes ? fh.passes.shift[p] : 0;
    int min_shift = 3, max_shift = 2; for (uint32_t i = 0;; i++) { for (uint32_t j = 0; j < fh.passes.num_ds; j++) if (i == fh.passes.last_pass[j]) min_shift = FloorLog2(fh.passes.downsample[j]); if (i + 1 == h.num_passes) min_shift = 0; if (i == p) break; max_shift = min_shift - 1; }
    h.pass_min_shift[p] = min_shift; h.pass_max_shift[p] = max_shift; }
  const LoopFilter& l = fh.lf; h.lpf.gab = l.gab; h.lpf.epf_iters = l.epf_iters; memcpy(h.lpf.gab_w, l.gab_w, sizeof(l.gab_w)); memcpy(h.lpf.epf_sharp_lut, l.epf_sharp_lut, sizeof(l.epf_sharp_lut)); memcpy(h.lpf.epf_channel_scale, l.epf_channel_scale, sizeof(l.epf_channel_scale));
  h.lpf.epf_quant_mul = l.epf_quant_mul; h.lpf.pass0_sigma_scale = l.epf_pass0_sigma_scale; h.lpf.pass2_sigma_scale = l.epf_pass2_sigma_scale; h.lpf.border_sad_mul = l.epf_border_sad_mul; h.lpf.sigma_for_modular = l.epf_sigma_for_modular;
  if (fh.encoding == 1) JXLG_CHECK(!l.gab && !l.epf_iters, "restoration filters on Modular frames are not supported by the GPU decoder yet");
  // colour
  DColor& c = h.color; memcpy(c.opsin_inv, m.opsin.inv, sizeof(c.opsin_inv)); for (int i = 0; i < 3; i++) { c.opsin_bias[i] = m.opsin.bias[i]; c.opsin_bias_cbrt[i] = std::cbrt(m.opsin.bias[i]); }
  c.itscale = 255.0f / m.tm.intensity_target; c.intensity_target = m.tm.intensity_target; c.xyb_encoded = m.xyb_encoded; c.num_color = m.ce.color_space == kCsGray && !m.xyb_encoded ? 1 : 3; if (fh.encoding == 1) c.num_color = m.ce.color_space == kCsGray ? 1 : 3;
  ColorEncoding oe = OutputEncoding(m); c.tf = oe.have_gamma ? 0 : oe.tf; c.gamma = oe.have_gamma ? float(oe.gamma) * 1e-7f : 1.0f;
  { // linear sRGB -> target primaries
    for (int i = 0; i < 9; i++) c.to_target[i] = (i % 4 == 0) ? 1.f : 0.f;
    if (!(oe.primaries == kPrSRGB && oe.white_point == kWpD65) && oe.color_space == kCsRGB) {
      auto prim = [](const ColorEncoding& ce, double p[3][2], double w[2]) {
        switch (ce.white_point) { case kWpD65: w[0] = 0.3127; w[1] = 0.3290; break; case kWpE: w[0] = w[1] = 1.0 / 3; break; case kWpDCI: w[0] = 0.314; w[1] = 0.351; break; default: w[0] = ce.white_xy[0] * 1e-6; w[1] = ce.white_xy[1] * 1e-6; }
        static const double srgb[3][2] = {{0.639998686, 0.330010138}, {0.300003784, 0.600003357}, {0.150002046, 0.059997204}}, bt2100[3][2] = {{0.708, 0.292}, {0.170, 0.797}, {0.131, 0.046}}, p3[3][2] = {{0.680, 0.320}, {0.265, 0.690}, {0.150, 0.060}};
        const double (*src)[2] = ce.primaries == kPr2100 ? bt2100 : ce.primaries == kPrP3 ? p3 : srgb; for (int i = 0; i < 3; i++) for (int k = 0; k < 2; k++) p[i][k] = ce.primaries == kPrCustom ? ce.prim_xy[i][k] * 1e-6 : src[i][k]; };
      auto inv3 = [](const double mm[9], double o[9]) { double det = mm[0] * (mm[4] * mm[8] - mm[5] * mm[7]) - mm[1] * (mm[3] * mm[8] - mm[5] * mm[6]) + mm[2] * (mm[3] * mm[7] - mm[4] * mm[6]); JXLG_CHECK(std::fabs(det) > 1e-12, "singular colour matrix"); double id = 1 / det;
        o[0] = (mm[4] * mm[8] - mm[5] * mm[7]) * id; o[1] = (mm[2] * mm[7] - mm[1] * mm[8]) * id; o[2] = (mm[1] * mm[5] - mm[2] * mm[4]) * id; o[3] = (mm[5] * mm[6] - mm[3] * mm[8]) * id; o[4] = (mm[0] * mm[8] - mm[2] * mm[6]) * id; o[5] = (mm[2] * mm[3] - mm[0] * mm[5]) * id;
        o[6] = (mm[3] * mm[7] - mm[4] * mm[6]) * id; o[7] = (mm[1] * mm[6] - mm[0] * mm[7]) * id; o[8] = (mm[0] * mm[4] - mm[1] * mm[3]) * id; };
      auto rgb2xyz = [&](const double p[3][2], const double w[2], double mm[9]) { double P[9]; for (int i = 0; i < 3; i++) { P[i] = p[i][0] / p[i][1]; P[3 + i] = 1.0; P[6 + i] = (1 - p[i][0] - p[i][1]) / p[i][1]; } double W[3] = {w[0] / w[1], 1.0, (1 - w[0] - w[1]) / w[1]}, Pi[9]; inv3(P, Pi);
        double S[3]; for (int i = 0; i < 3; i++) S[i] = Pi[3 * i] * W[0] + Pi[3 * i + 1] * W[1] + Pi[3 * i + 2] * W[2]; for (int r = 0; r < 3; r++) for (int cc = 0; cc < 3; cc++) mm[3 * r + cc] = P[3 * r + cc] * S[cc]; };
      ColorEncoding s; double ps[3][2], ws[2], pt[3][2], wt[2], A[9], B[9], Bi[9]; prim(s, ps, ws); prim(oe, pt, wt); rgb2xyz(ps, ws, A); rgb2xyz(pt, wt, B); inv3(B, Bi);
      for (int r = 0; r < 3; r++) for (int cc = 0; cc < 3; cc++) { double v = 0; for (int k = 0; k < 3; k++) v += Bi[3 * r + k] * A[3 * k + cc]; c.to_target[3 * r + cc] = float(v); }
    }
  }
  for (int r = 0; r < 3; r++) for (int cc = 0; cc < 3; cc++) { double v = 0; for (int k = 0; k < 3; k++) v += double(c.to_target[3 * r + k]) * double(c.opsin_inv[3 * k + cc]); c.mix_to_target[3 * r + cc] = float(v * double(c.itscale)); }
  // output description
  DOutput& o = h.out; o.sample_type = uint32_t(info.sample_type); o.num_channels = uint32_t(info.num_channels); o.color_channels = uint32_t(m.num_color_channels()); o.orientation = m.orientation; o.bgra = bgra ? 1 : 0;
  o.out_w = m.orientation >= 5 ? fh.ysize : fh.xsize; o.out_h = m.orientation >= 5 ? fh.xsize : fh.ysize; o.bits = m.bd.bits; o.exp_bits = m.bd.exp_bits;
  size_t ec_base = fh.encoding == 1 ? (m.ce.color_space == kCsGray ? 1 : 3) : 0; int alpha = info.has_alpha ? m.alpha_index() : -1, black = m.black_index();
  o.alpha_plane = alpha >= 0 ? int32_t(ec_base + alpha) : -1; o.black_plane = info.format == 2 ? int32_t(ec_base + black) : -1; o.premultiplied = alpha >= 0 && m.ec[alpha].alpha_associated;
  if (alpha >= 0) { o.alpha_bits = m.ec[alpha].bd.bits; o.alpha_exp_bits = m.ec[alpha].bd.exp_bits; } if (black >= 0) o.black_bits = m.ec[black].bd.bits;
  if (bgra) JXLG_CHECK(info.format != 2, "BGRA surface output is not defined for CMYK images");
  if (layer) {   // float samples of the frame itself; orientation, unpremultiply and the sample type are applied to the finished canvas
    JXLG_CHECK(info.format != 2, "multi-frame CMYK images are not supported");
    o.sample_type = 3; o.orientation = 1; o.premultiplied = 0; o.bgra = 0; bgra = false; device_output = true; o.out_w = fh.xsize; o.out_h = fh.ysize;
  }
  if (fh.encoding == 0) for (size_t i = 0; i < m.ec.size(); i++) JXLG_CHECK(m.ec[i].dim_shift < 3, "extra channels with dim_shift >= 3 (Modular LF-group data inside VarDCT frames) are not supported by the GPU decoder yet");
}

void DecodeJob::UploadFrame() { if (!h_misc.p) h_misc.Alloc(2 * sizeof(DFrame) + 64, true); DFrame* slot = h_misc.as<DFrame>() + (frame_uploads++ & 1); *slot = h; CUDA_OK(cudaMemcpyAsync(d_frame.p, slot, sizeof(DFrame), cudaMemcpyHostToDevice, stream)); }

void DecodeJob::AllocateAndUpload(const DecodeRequest& req) {
  const ByteSpan& cs = hd.ci.codestream; comp_size = cs.size();
  // Band decode (one rank's share of a huge frame): the big per-pixel buffers — coefficients, XYB planes, non-zero counts — are allocated
  // for the band's group rows only (comp_g0 .. comp_g1: the band plus one halo row each side), not for the frame. The kernels keep
  // addressing by absolute group / pixel row, so the descriptor carries bases shifted back by the band's first group / row.
  const size_t band_g0 = h.band_on ? size_t(h.comp_g0) * h.xgroups : 0, band_groups = h.band_on ? size_t(h.comp_g1 - h.comp_g0) * h.xgroups : h.num_groups;
  const size_t band_y0 = h.band_on ? size_t(h.comp_g0) * h.group_dim : 0;
  if (h.band_on && h.encoding == 0) h.ypad = uint32_t(std::min<size_t>(h.ypad, size_t(h.comp_g1) * h.group_dim) - band_y0);   // rows per plane = plane stride of the kernels
  size_t cells = size_t(h.xb) * h.yb, px = size_t(h.xpad) * h.ypad, tiles = size_t(h.xt) * h.yt; bool vardct = h.encoding == 0;
  d_frame.Alloc(sizeof(DFrame)); d_err.Alloc(64); h_err.Alloc(64, true); d_gother.Alloc(size_t(h.num_groups) * 4);
  d_comp.Alloc(comp_size + 64);
  if (vardct) {
    d_lfq.Alloc(cells * 3 * 4); d_lf.Alloc(cells * 3 * 4); d_lf_tmp.Alloc(cells * 3 * 4); d_acs.Alloc(cells); d_qf.Alloc(cells); d_sharp.Alloc(cells); d_lfidx.Alloc(cells); d_ytox.Alloc(tiles); d_ytob.Alloc(tiles);
    d_nz.Alloc(band_groups * 3072); d_acend.Alloc(size_t(h.num_groups) * h.num_passes * 8);
    d_hfmeta.Alloc((size_t(h.num_lf_groups) * kHfMetaScratchInts + h.num_lf_groups) * 4); d_coeffs.Alloc(band_groups * 3 * 65536 * 2); coeffs_bytes = band_groups * 3 * 65536 * 2; d_xyb.Alloc(px * 3 * 4);
    d_sigma.Alloc(cells * 4); if (!phased) d_xyb_tmp.Alloc(px * 3 * 4);   // phased (batch) jobs allocate xyb_tmp in RunRender, and only when the frame needs it
  }
  uint64_t mod_ints = mod_total_ints; if (mod_ints) d_mod.Alloc(mod_ints * 4);
  if (h.uses_wp) d_wp.Alloc((size_t(h.num_lf_groups) + h.num_groups + 1) * 5 * 2 * (kMaxWpWidth + 2) * 4); else d_wp.Alloc(16);
  const DOutput& o = h.out; size_t bps = o.sample_type == 0 ? 1 : o.sample_type == 3 ? 4 : 2; size_t chans = bgra ? 4 : (o.num_channels + (o.black_plane >= 0 ? 1 : 0)); if (bgra) bps = 1;
  out_bytes = size_t(o.out_w) * (h.band_on ? h.out_y1 - h.out_y0 : o.out_h) * chans * bps;
  if (req.out_device || req.out_pinned) JXLG_CHECK(req.out_capacity >= out_bytes, "output buffer too small");
  if (!req.out_device) d_out.Alloc(out_bytes); if (!device_output && !req.out_pinned) h_out.Alloc(out_bytes, true);
  ext_out_device = req.out_device; ext_out_pinned = req.out_pinned;
  h.comp = d_comp.as<uint8_t>(); h.lfq = d_lfq.as<int32_t>(); h.lf = d_lf.as<float>(); h.lf_tmp = d_lf_tmp.as<float>(); h.acs = d_acs.as<uint8_t>(); h.hf_mul_m1 = d_qf.as<uint8_t>(); h.sharp = d_sharp.as<uint8_t>(); h.lf_idx = d_lfidx.as<uint8_t>();
  h.ytox = d_ytox.as<int8_t>(); h.ytob = d_ytob.as<int8_t>(); h.hfmeta_scratch = d_hfmeta.as<int32_t>(); h.coeffs = d_coeffs.as<int16_t>() - band_g0 * 3 * 65536; h.xyb = d_xyb.as<float>() - band_y0 * h.xpad; h.xyb_tmp = d_xyb_tmp.p ? d_xyb_tmp.as<float>() - band_y0 * h.xpad : nullptr; xyb_row_shift = band_y0 * h.xpad; h.inv_sigma = d_sigma.as<float>();
  h.mod_planes = d_mod.as<int32_t>(); h.wp_scratch = d_wp.as<int32_t>(); h.out_px = req.out_device ? req.out_device : d_out.as<uint8_t>(); h.err = d_err.as<uint32_t>(); h.end_bitpos = reinterpret_cast<uint64_t*>(d_err.as<uint8_t>() + 16); h.tables = DeviceTables();
  bool smooth = vardct && !(h.flags & kFlagSkipAdaptiveLfSmoothing) && h.xb > 2 && h.yb > 2; h.lf_src = smooth ? h.lf_tmp : h.lf;
  memset(h_err.p, 0, 64); h.host_flags = h_err.as<uint32_t>() + 12; h.group_other = d_gother.as<uint32_t>(); h.nz_scratch = d_nz.as<uint8_t>() - band_g0 * 3072; h.ac_endpos = d_acend.as<uint64_t>();
  h.group_pal = nullptr;   // palette channels of palettes listed in group sections' own headers (16 KB per group)
  if (h.num_mod_channels > h.first_group_channel) { d_gpal.Alloc(size_t(h.num_groups) * kGroupPalInts * 4); h.group_pal = d_gpal.as<int32_t>(); }
  h.lz_window = nullptr;
  if (blob.uses_lz77) { d_lz.Alloc((size_t(std::max(h.num_lf_groups, h.num_groups)) + 1) * (size_t(1) << 20) * 4); h.lz_window = d_lz.as<uint32_t>(); }
  CUDA_OK(cudaMemsetAsync(d_err.p, 0, 64, stream)); CUDA_OK(cudaMemsetAsync(d_gother.p, 0, size_t(h.num_groups) * 4, stream));
  if (req.device_input && hd.ci.contiguous_offset != size_t(-1)) CUDA_OK(cudaMemcpyAsync(d_comp.p, req.device_input + hd.ci.contiguous_offset, comp_size, cudaMemcpyDeviceToDevice, stream));
  else { h_comp.Alloc(comp_size, true); memcpy(h_comp.p, cs.data(), comp_size); CUDA_OK(cudaMemcpyAsync(d_comp.p, h_comp.p, comp_size, cudaMemcpyHostToDevice, stream)); }   // pinned staging: a pageable source would serialise the stream
  CUDA_OK(cudaMemsetAsync(d_comp.as<uint8_t>() + comp_size, 0, 64, stream));
}

static const char* DevErrorText(uint32_t e) {
  switch (e) { case kErrOverrun: return "section truncated (read past its end)"; case kErrAnsFinal: return "ANS final state mismatch"; case kErrBadStrategy: return "invalid or unsupported (AFV) AC strategy"; case kErrBlockBounds: return "AC strategy block out of bounds";
    case kErrTooManyNz: return "too many non-zero coefficients"; case kErrNzMismatch: return "non-zero count mismatch"; case kErrUnsupportedStream: return "unsupported Modular stream geometry"; case kErrCoefRange: return "coefficient exceeds 16 bits";
    case kErrHfMeta: return "HF metadata inconsistent"; case kErrLocalTree: return "local MA trees are not supported by the GPU decoder yet"; case kErrGroupTransform: return "per-group Modular transforms are not supported by the GPU decoder yet";
    case kErrHybrid: return "hybrid integer too large"; case kErrPrefix: return "invalid prefix code"; case kErrCflRange: return "CfL factor out of range"; case kErrSharpness: return "EPF sharpness out of range"; case kErrPreset: return "invalid HF preset"; case kErrRefProps: return "unsupported MA-tree property";
    case kErrPaletteDelta: return "delta-palette entries (negative palette indices) are not supported";
    default: return "device decode error"; }
}

// Phase 1: host parse of the global sections, uploads, the global Modular stream and the LF-group entropy kernel.
void DecodeJob::RunLf(const DecodeRequest& req) {
  const ByteSpan& cs = hd.ci.codestream; const bool vardct = h.encoding == 0; const size_t nsec = toc.size.size(); const bool single = nsec == 1;
  const size_t nlog = size_t(h.num_passes) * h.num_groups + h.num_lf_groups + 2;
  // host parse: LfGlobal (+ HfGlobal when it has its own section)
  BitReader lfg(cs.data() + frame_off + toc.offset[0], toc.size[0]); ParseLfGlobal(lfg); JXLG_CHECK(!lfg.overrun, "LfGlobal truncated");
  uint64_t base_bits = uint64_t(frame_off) * 8; uint64_t after_lfglobal = (uint64_t(frame_off) + toc.offset[0]) * 8 + lfg.pos;
  if (!single && vardct) { BitReader hb(cs.data() + frame_off + toc.offset[1 + h.num_lf_groups], toc.size[1 + h.num_lf_groups]); ParseHfGlobal(hb); JXLG_CHECK(!hb.overrun, "HfGlobal truncated"); }
  {  // shared-memory budgets for the staged tables (host knows the exact sizes)
    auto code_bytes = [](const DCode& c) { return ((c.num_clusters * 4 + 15) & ~15u) + ((c.num_ctx + 15) & ~15u) + (c.use_prefix ? 0u : (((c.num_clusters << c.log_alpha) * 8 + 15) & ~15u)); };
    uint32_t modb = has_tree ? code_bytes(h.mod_code) + ((h.tree_size * 16 + 15) & ~15u) : 0;
    { static std::atomic<uint32_t> lf_cursor{0}, ac_cursor{0};   // concurrent images start their few long-running CTAs on different SMs
      h.lf_cta_offset = lf_cursor.fetch_add(h.num_lf_groups) % 148u; h.ac_cta_offset = vardct ? ac_cursor.fetch_add(uint32_t(AcCtas(h, ac_lanes))) % 148u : 0; }
    // + the transposed alias table of the speculative LF loop (32 slots x 8 bytes per alias entry), when it stays small
    { const uint32_t spec = has_tree && !h.mod_code.use_prefix ? (256u << h.mod_code.log_alpha) : 0u; const uint32_t copies = h.num_mod_channels > h.first_group_channel ? 4u : 1u;   // k_mod_group: one table per warp, 4 warps per CTA
      h.lf_smem = std::min<uint32_t>(modb + 64 + (spec * copies <= 64 * 1024 ? spec * copies + 64 : (spec <= 64 * 1024 ? spec + 16 : 0)), 96 * 1024); } ac_budget = [this, code_bytes]() { uint32_t acb = 0; bool prefix = false; for (uint32_t p = 0; p < h.num_passes; p++) { acb = std::max(acb, code_bytes(h.ac_code[p])); prefix |= h.ac_code[p].use_prefix != 0; }
      for (uint32_t p = 0; p < h.num_passes; p++) prefix |= h.ac_code[p].lz77 != 0;   // LZ77 streams take the generic reader too
      h.ac_smem = acb + 64; h.ac_fast = (!prefix && h.ac_smem <= 96 * 1024) ? 1 : 0; if (!h.ac_fast) h.ac_smem = 0; };
    if (vardct && !single) ac_budget();
  }
  // ---- sub-bitstreams with their own MA tree. Group sections of Modular frames start with their Modular header, so the host can parse the tree and
  // the code that follow it (VarDCT frames keep their group-local Modular data behind the AC coefficients, where only the device knows the position).
  h.local_off = 0;
  { std::vector<DLocalTree> lts(size_t(h.num_groups) + 1 + h.num_lf_groups); memset(lts.data(), 0, lts.size() * sizeof(DLocalTree)); bool any = false;   // [group g | global | LF group g]
    if (global_local.present) { lts[h.num_groups] = global_local; lts[h.num_groups].data_bitpos = after_lfglobal; any = true; }
    auto section_tree = [&](size_t t, size_t slot, size_t pixels) {   // TOC section t, entry lts[slot], at most `pixels` samples
      if (toc.size[t] == 0) return;
      BitReader gb(cs.data() + frame_off + toc.offset[t], toc.size[t]); const GroupHeader gh = ReadGroupHeader(gb);
      bool only_rct = true; for (const Transform& tr : gh.transforms) only_rct = only_rct && tr.id == 0;
      if (gb.overrun || gh.use_global_tree || !only_rct) return;   // (palette / squeeze inside a section: the kernel reports them)
      lts[slot] = ParseLocalTree(gb, pixels); lts[slot].data_bitpos = base_bits + uint64_t(toc.offset[t]) * 8 + gb.pos; any = true;
    };
    const size_t dim = size_t(h.group_dim);
    if (fh.encoding == 1 && !single && h.num_passes == 1 && h.num_mod_channels > h.first_group_channel)
      for (uint32_t g = 0; g < h.num_groups; g++) section_tree(size_t(2) + h.num_lf_groups + g, g, dim * dim * (h.num_mod_channels - h.first_group_channel));
    if (fh.encoding == 1 && !single && mod_has_lf_level)   // LF-group sections of Modular frames (channels of shift >= 3) start with their Modular header too
      for (uint32_t g = 0; g < h.num_lf_groups; g++) section_tree(size_t(1) + g, size_t(h.num_groups) + 1 + g, dim * dim * h.num_mod_channels);
    if (any) h.local_off = blob.Add(lts.data(), lts.size() * sizeof(DLocalTree)); }
  std::vector<uint64_t> sec(2 * nlog + 2, 0);
  for (size_t i = 0; i < nlog; i++) { size_t t = single ? 0 : i; sec[i] = base_bits + uint64_t(toc.offset[t]) * 8; sec[nlog + i] = base_bits + uint64_t(toc.offset[t] + toc.size[t]) * 8; }
  h.sec_off = blob.Add(sec.data(), sec.size() * 8);
  AllocateAndUpload(req);
  auto upload_blob = [&]() { blob.b.resize((blob.b.size() + 31) / 16 * 16, 0); if (d_blob.n < blob.b.size() + 16) d_blob.Alloc(std::max<size_t>(blob.b.size() * 2, 1 << 16)); h.blob = d_blob.as<uint8_t>(); h_blob.Alloc(blob.b.size(), true); memcpy(h_blob.p, blob.b.data(), blob.b.size()); CUDA_OK(cudaMemcpyAsync(d_blob.p, h_blob.p, blob.b.size(), cudaMemcpyHostToDevice, stream)); UploadFrame(); };
  upload_blob();
  const DFrame* d = d_frame.as<DFrame>();
  if (timed) cudaEventRecord(ev[0], stream);
  // global Modular stream
  if (global_has_data) LaunchModularGlobal(d, h, after_lfglobal, h.first_group_channel, stream);
  else if (single) { uint64_t* slot = reinterpret_cast<uint64_t*>(h_misc.as<uint8_t>() + 2 * sizeof(DFrame)); slot[0] = after_lfglobal; CUDA_OK(cudaMemcpyAsync(h.end_bitpos, slot, 8, cudaMemcpyHostToDevice, stream)); }
  if (!vardct && !single && mod_has_lf_level) LaunchModLfGroups(h, stream);   // Modular frames: channels of shift >= 3 live in the LF-group sections
  if (vardct) { if (defer_entropy && !single) lf_pending = true; else LaunchLfGroups(d, h, stream); }
  else if (single) { /* Modular frame, single section: LF group and HfGlobal parts are empty; groups continue where the global stream ended */ CUDA_OK(cudaMemcpyAsync(h.end_bitpos + 2, h.end_bitpos, 8, cudaMemcpyDeviceToDevice, stream)); }
  if (single && vardct) {   // HfGlobal follows the LF group in the same bit stream: need its end position on the host
    uint64_t pos[3] = {0, 0, 0}; CUDA_OK(cudaMemcpyAsync(h_err.p, d_err.p, 64, cudaMemcpyDeviceToHost, stream)); CUDA_OK(cudaStreamSynchronize(stream));
    uint32_t e = *h_err.as<uint32_t>(); JXLG_CHECK(e == 0, DevErrorText(e)); memcpy(pos, h_err.as<uint8_t>() + 16, 24);
    size_t byte = size_t(pos[1] / 8); JXLG_CHECK(byte <= cs.size(), "LF group ran past the end of the file");
    BitReader hb(cs.data(), cs.size()); hb.pos = size_t(pos[1]); ParseHfGlobal(hb); JXLG_CHECK(!hb.overrun, "HfGlobal truncated"); uint64_t after = hb.pos; ac_budget();
    upload_blob(); { uint64_t* slot = reinterpret_cast<uint64_t*>(h_misc.as<uint8_t>() + 2 * sizeof(DFrame)) + 1; slot[0] = after; CUDA_OK(cudaMemcpyAsync(h.end_bitpos + 2, slot, 8, cudaMemcpyHostToDevice, stream)); }
  }
}

// Phase 2: LF dequantisation (+ adaptive smoothing) and the AC / group-Modular entropy kernels.
void DecodeJob::RunAc() {
  const bool vardct = h.encoding == 0; const DFrame* d = d_frame.as<DFrame>();
  if (timed) cudaEventRecord(ev[1], stream);
  if (vardct) LaunchLfDequant(d, h, h.lf_src == h.lf_tmp, stream);
  if (vardct) CUDA_OK(cudaMemsetAsync(d_coeffs.p, 0, coeffs_bytes, stream));
  if (defer_entropy && vardct && h.num_passes == 1 && h.ac_fast && !(h.num_mod_channels > h.first_group_channel)) ac_pending = true;
  else for (uint32_t p = 0; p < h.num_passes; p++) LaunchAcGroups(d, h, int(p), ac_lanes, stream);
  if (timed) cudaEventRecord(ev[2], stream);
}

// Phase 3: dequant + IDCT, restoration filters, colour transform, pack, and the copy back to the host.
void DecodeJob::RunRender() {
  const bool vardct = h.encoding == 0; const DFrame* d = d_frame.as<DFrame>();
  if (vardct && !d_xyb_tmp.p) {   // phased job: the LF phase has drained, its flag word is already in host memory
    const bool big_blocks = h_err.as<volatile uint32_t>()[12] != 0;   // written by k_lf_group straight into this page-locked word
    if (big_blocks) { d_xyb_tmp.Alloc(size_t(h.xpad) * h.ypad * 3 * 4); h.xyb_tmp = d_xyb_tmp.as<float>() - xyb_row_shift; UploadFrame(); }
  }
  if (vardct) LaunchReconstruct(d, h, stream);
  if (timed) cudaEventRecord(ev[3], stream);
  if (h.num_ops) LaunchInverseRct(d, h, ops_host.data(), stream);
  const bool fused = vardct && LaunchFusedRender(d, h, stream);   // gaborish + EPF + colour + pack in one kernel
  if (timed) cudaEventRecord(ev[4], stream);
  if (!fused) LaunchOutput(d, h, stream);
  if (timed) cudaEventRecord(ev[5], stream);
  if (!device_output) CUDA_OK(cudaMemcpyAsync(ext_out_pinned ? ext_out_pinned : h_out.as<uint8_t>(), h.out_px, out_bytes, cudaMemcpyDeviceToHost, stream));
  CUDA_OK(cudaMemcpyAsync(h_err.p, d_err.p, 64, cudaMemcpyDeviceToHost, stream));
  if (timed) cudaEventRecord(ev[6], stream);
}

// Position of the first frame after an optional preview frame, and whether that frame is a plain single-frame image.
static bool FirstFrameIsPlain(const Headers& hd, size_t* first_pos) {
  const ImageMetadata& m = hd.meta; const ByteSpan& cs = hd.ci.codestream; size_t pos = hd.frame_pos;
  if (m.have_preview) { ImageMetadata pm = m; pm.xsize = m.preview_x; pm.ysize = m.preview_y; BitReader br(cs.data() + pos, cs.size() - pos); FrameHeader pf = ReadFrameHeader(br, pm); Toc t = ReadToc(br, pf); pos += br.pos / 8 + t.total; JXLG_CHECK(pos <= cs.size(), "preview frame truncated"); }
  *first_pos = pos; BitReader br(cs.data() + pos, cs.size() - pos); FrameHeader fh = ReadFrameHeader(br, m);
  const bool exact = !fh.have_crop || (fh.x0 == 0 && fh.y0 == 0 && fh.width == m.xsize && fh.height == m.ysize);
  return FrameIsPlain(fh, m) && exact;
}

// The start of every decode: a job on `stream` (stage events when `timed`) with the headers parsed and the frame set up. With `layered_pos`,
// a file whose first frame is not plain is left for compositing: the job holds only its headers, and *layered_pos receives that frame's position.
static std::shared_ptr<DecodeJob> StartJob(const DecodeRequest& req, cudaStream_t stream, bool timed, size_t* layered_pos = nullptr) {
  std::shared_ptr<DecodeJob> job = std::make_shared<DecodeJob>(); job->stream = stream;
  if (timed) { job->timed = true; for (int i = 0; i < 7; i++) cudaEventCreate(&job->ev[i]); }   // stage timing only: ev calls are not checked
  ParseHeadersInto(req.data, req.size, &job->hd, &job->info);
  if (layered_pos && !FirstFrameIsPlain(job->hd, layered_pos)) return job;
  if (layered_pos) *layered_pos = 0;
  job->Setup(req);
  return job;
}

std::shared_ptr<DecodeJob> DecodeEnqueue(const DecodeRequest& req, cudaStream_t stream, bool lf_phase_only, bool defer_entropy) {
  if (!req.data) throw StatusError(DecoderStatus_NullParameter);
  std::string why; JXLG_CHECK(CudaAvailable(&why), why);
  std::shared_ptr<DecodeJob> job = StartJob(req, stream, false);
  job->phased = lf_phase_only; job->defer_entropy = defer_entropy && lf_phase_only;
  if (lf_phase_only) job->RunLf(req); else job->Run(req);
  return job;
}

// Phased enqueue (batches): phase 1 = DecodeEnqueue(..., lf_phase_only), then DecodeEnqueuePhase(job, 2) and (job, 3), each once
// the stream has drained, so that a queued dependent kernel never blocks a hardware queue shared with other streams.
void DecodeEnqueuePhase(const std::shared_ptr<DecodeJob>& job, int phase) {
  try { if (phase == 2) job->RunAc(); else job->RunRender(); }
  catch (...) { cudaStreamSynchronize(job->stream); throw; }   // the caller drops the failed job: its buffers may go back to the pools only once its work has drained
}
// Bundle mode: the jobs share one stream and were enqueued with defer_entropy; their pending LF (phase 1) or AC (phase 2) entropy kernels
// go out as multi-image launches of up to kMaxBundle frames each.
void DecodeBundleLaunch(const std::vector<std::shared_ptr<DecodeJob>>& jobs, int phase) {
  for (int kind = 0; kind < 2; kind++) {   // LF: narrow / wide Modular kernels; AC: one kind
    DFrameSet set; set.n = 0; cudaStream_t st = nullptr; int lanes = 1;
    auto flush = [&]() { if (!set.n) return; if (phase == 1) LaunchLfGroupsMulti(set, kind == 0, st); else LaunchAcGroupsMulti(set, lanes, st); set.n = 0; };
    for (const auto& j : jobs) {
      if (!j) continue;
      if (phase == 1) { if (!j->lf_pending || LfNarrow(j->h) != (kind == 0)) continue; }
      else { if (kind == 1 || !j->ac_pending) continue; if (set.n && j->ac_lanes != lanes) flush(); lanes = j->ac_lanes; }
      if (set.n == 0) { set.first[0] = 0; set.cta_offset = phase == 1 ? j->h.lf_cta_offset : j->h.ac_cta_offset; st = j->stream; }
      set.f[set.n] = j->h; set.first[set.n + 1] = set.first[set.n] + (phase == 1 ? j->h.num_lf_groups : uint32_t(AcCtas(j->h, j->ac_lanes))); set.n++;
      if (phase == 1) j->lf_pending = false; else j->ac_pending = false;
      if (set.n == uint32_t(kMaxBundle)) flush();
    }
    flush();
  }
}
// Band layout of the first frame (host-only parse): group size in pixels and the number of group rows a caller can shard over.
ParsedInfo DecodeBandLayout(const uint8_t* data, size_t size) { DecodeRequest req; req.data = data; req.size = size; return StartJob(req, nullptr, false)->info; }
// Host-only: byte sizes of the first frame's TOC entries (sections in logical order). Instrumentation for the load-balance analysis of the AC kernel.
SectionSizes DecodeSectionSizes(const uint8_t* data, size_t size) {
  DecodeRequest req; req.data = data; req.size = size; std::shared_ptr<DecodeJob> job = StartJob(req, nullptr, false);
  SectionSizes r; r.sizes.assign(job->toc.size.begin(), job->toc.size.end()); r.num_lf_groups = job->fh.num_lf_groups; r.num_groups = job->fh.num_groups; return r;
}
void DecodeReservePools(const std::shared_ptr<DecodeJob>& job, size_t count) { if (job) job->ReservePools(count); }

DecodeResult DecodeFinish(const std::shared_ptr<DecodeJob>& job) {
  cudaError_t e = cudaStreamSynchronize(job->stream);
  if (e != cudaSuccess) throw Error(std::string("CUDA: ") + cudaGetErrorString(e));
  uint32_t de = *job->h_err.as<uint32_t>();
  JXLG_CHECK(de == 0, DevErrorText(de));
  DecodeResult r;
  r.info = job->info; r.pixels = job->device_output ? job->h.out_px : (job->ext_out_pinned ? job->ext_out_pinned : job->h_out.as<uint8_t>()); r.pixel_bytes = job->out_bytes; r.out_width = job->h.out.out_w; r.out_height = job->h.band_on ? job->h.out_y1 - job->h.out_y0 : job->h.out.out_h; r.job = job;
  if (job->timed) { auto ms = [&](int a, int b) { float t = 0; cudaEventElapsedTime(&t, job->ev[a], job->ev[b]); return t; };
    r.times.lf = ms(0, 1); r.times.ac = ms(1, 2); r.times.recon = ms(2, 3); r.times.filters = ms(3, 4); r.times.output = ms(4, 5); r.times.d2h = ms(5, 6); r.times.total = ms(0, 6); }
  return r;
}

// Layered stills (N/Decoder/JxlDecoder.cpp:252-400: the reference takes the first full image of a coalescing decoder). Every frame up to the
// first one that is shown is decoded by the ordinary pipeline into float samples and blended onto a canvas-sized float image that starts as a
// copy of the frame's source slot (dev/composite_kernels.cu); frames that may be referenced leave their result in a slot. The canvas that is
// shown becomes the output: unpremultiply, sample type, orientation. Reference-only frames saved before the colour transform can only feed
// patches (rejected) and are skipped.
// `head` holds the file's headers.
static DecodeResult DecodeLayered(const DecodeRequest& req, const DecodeJob& head, size_t pos, cudaStream_t st) {
  struct SlotBuf { Buf buf; bool valid = false; }; SlotBuf slots[4]; ParsedInfo info = head.info;
  const ImageMetadata& m = head.hd.meta; const ByteSpan& cs = head.hd.ci.codestream;
  for (int guard = 0; guard < 4096; guard++) {
    JXLG_CHECK(pos < cs.size(), "JxlDecoderProcessInput needs more input, but it already received the entire image.");
    BitReader br(cs.data() + pos, cs.size() - pos); const FrameHeader fh = ReadFrameHeader(br, m); const Toc toc = ReadToc(br, fh); const size_t next = pos + br.pos / 8 + toc.total;
    JXLG_CHECK(next <= cs.size(), "JxlDecoderProcessInput needs more input, but it already received the entire image.");
    JXLG_CHECK(fh.frame_type != kFrameLF, "LF frames are not supported");
    const bool ref_only = fh.frame_type == kFrameReferenceOnly;
    if (ref_only && fh.save_before_ct) { pos = next; continue; }
    const bool shown = !ref_only && (fh.is_last || fh.duration > 0);
    const int alpha = info.has_alpha ? m.alpha_index() : -1; const BlendingInfo cb = fh.blending, ab = alpha >= 0 ? fh.ec_blending[alpha] : BlendingInfo();
    JXLG_CHECK(!(cb.mode == 2 || cb.mode == 3) || (alpha >= 0 && int(cb.alpha_channel) == alpha), "blending needs the image's alpha channel");
    JXLG_CHECK(alpha < 0 || ref_only || ab.source == cb.source, "colour and alpha blended from different reference slots are not supported");
    DecodeRequest r = req; r.layer = true; r.layer_pos = pos; r.device_output = true; r.out_device = nullptr; r.out_pinned = nullptr; r.bgra = false; r.band_begin = r.band_end = 0; r.device_input = nullptr;
    std::shared_ptr<DecodeJob> job = StartJob(r, st, false); job->Run(r); const DecodeResult fr = DecodeFinish(job);
    const int W = int(m.xsize), H = int(m.ysize), C = info.num_channels, cc = int(m.num_color_channels()); const size_t canvas_bytes = size_t(W) * H * C * sizeof(float);
    Buf canvas; canvas.Alloc(canvas_bytes);
    if (!ref_only && slots[cb.source].valid) CUDA_OK(cudaMemcpyAsync(canvas.p, slots[cb.source].buf.p, canvas_bytes, cudaMemcpyDeviceToDevice, st)); else CUDA_OK(cudaMemsetAsync(canvas.p, 0, canvas_bytes, st));
    const bool premul = alpha >= 0 && m.ec[alpha].alpha_associated;
    LaunchBlendLayer(canvas.as<float>(), reinterpret_cast<const float*>(fr.pixels), W, H, int(fh.xsize), int(fh.ysize), ref_only ? 0 : fh.x0, ref_only ? 0 : fh.y0, C, cc,
                     ref_only ? 0u : cb.mode, ref_only ? 0u : ab.mode, cb.clamp, ab.clamp, premul, st);
    if (shown) {
      const uint32_t ori = m.orientation; const size_t bps = req.bgra ? 1 : (info.sample_type == 0 ? 1 : info.sample_type == 3 ? 4 : 2); const size_t chans = req.bgra ? 4 : size_t(C);
      const size_t out_bytes = size_t(W) * H * bps * chans;
      if (req.out_device || req.out_pinned) JXLG_CHECK(req.out_capacity >= out_bytes, "output buffer too small");
      uint8_t* d_final = req.out_device; if (!d_final) { job->d_layer_out.Alloc(out_bytes); d_final = job->d_layer_out.as<uint8_t>(); }
      LaunchFinalizeCanvas(canvas.as<float>(), d_final, W, H, C, cc, premul, uint32_t(info.sample_type), ori, req.bgra, st);
      uint8_t* host = nullptr;
      if (!req.device_output) { host = req.out_pinned; if (!host) { job->h_layer_out.Alloc(out_bytes, true); host = job->h_layer_out.as<uint8_t>(); } CUDA_OK(cudaMemcpyAsync(host, d_final, out_bytes, cudaMemcpyDeviceToHost, st)); }
      CUDA_OK(cudaStreamSynchronize(st));
      DecodeResult res; info.frame_name = fh.name; res.info = info; res.pixels = req.device_output ? d_final : host; res.pixel_bytes = out_bytes;
      res.out_width = ori >= 5 ? uint32_t(H) : uint32_t(W); res.out_height = ori >= 5 ? uint32_t(W) : uint32_t(H); res.job = job; return res;
    }
    CUDA_OK(cudaStreamSynchronize(st));   // the frame's buffers go back to the pools with the job
    const bool can_ref = ref_only || (!fh.is_last && (fh.duration == 0 || fh.save_as_reference != 0));
    if (can_ref) { SlotBuf& s = slots[fh.save_as_reference]; s.buf.Free(); s.buf.Swap(canvas); s.valid = true; }
    pos = next;
  }
  throw Error("too many frames before the first one that is shown");
}

DecodeResult DecodeOnGpu(const DecodeRequest& req) {
  if (!req.data) throw StatusError(DecoderStatus_NullParameter);
  if (SignatureCheck(req.data, req.size) == 0) throw StatusError(DecoderStatus_InvalidFileSignature);
  std::string why; JXLG_CHECK(CudaAvailable(&why), why);
  cudaStream_t st = nullptr; JXLG_CHECK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) == cudaSuccess, "cudaStreamCreate failed");
  struct Stream { cudaStream_t s; ~Stream() { cudaStreamDestroy(s); } } stream{st};   // outlives the job below, and with it the job's pending work
  std::shared_ptr<DecodeJob> job;
  try {
    size_t layered_pos = 0;
    job = StartJob(req, st, true, req.band_begin || req.band_end ? nullptr : &layered_pos);
    if (layered_pos) return DecodeLayered(req, *job, layered_pos, st);
    job->Run(req); return DecodeFinish(job);
  } catch (...) { cudaStreamSynchronize(st); throw; }   // the job gives its buffers back only after its work has drained
}

bool DecodeDebugPlanes(const std::shared_ptr<DecodeJob>& job, int which, std::vector<float>* out, int* xpad, int* ypad) {
  if (!job || job->h.encoding != 0) return false; size_t px = size_t(job->h.xpad) * job->h.ypad; *xpad = int(job->h.xpad); *ypad = int(job->h.ypad);
  const float* src = nullptr; size_t n = px * 3;
  if (which == 0) src = job->h.xyb; else if (which == 3) { src = job->h.lf_src; n = size_t(job->h.xb) * job->h.yb * 3; } else return false;
  out->resize(n); return cudaMemcpy(out->data(), src, n * 4, cudaMemcpyDeviceToHost) == cudaSuccess;
}
bool DecodeDebugCoeffs(const std::shared_ptr<DecodeJob>& job, std::vector<int16_t>* out) {
  if (!job || job->h.encoding != 0) return false; size_t n = size_t(job->h.num_groups) * 3 * 65536; out->resize(n); return cudaMemcpy(out->data(), job->h.coeffs, n * 2, cudaMemcpyDeviceToHost) == cudaSuccess;
}

}  // namespace jxlgpu
