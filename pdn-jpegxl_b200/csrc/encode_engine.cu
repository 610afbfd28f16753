// pdn-jpegxl_b200 engine — encode orchestration behind SaveImage / JxlB200EncodeToMemory.
// Restates what EncoderWriteImage configures and drives through libjxl
// (N/Encoder/JxlEncoder.cpp:147-392): pixel-format decision from a full scan (:33-77, gray only
// without ICC :67), 8-bit samples, XYB VarDCT for lossy / Modular with the original profile
// for lossless (:214,325), container always with uncompressed Exif / xml boxes (:201,284-310).
// The codec arithmetic runs in dev/encode_kernels.cu; the host writes headers, builds the
// entropy codes from device histograms and assembles the sections. No CPU encode path exists.
#include "engine.h"
#include "dev/enc_frame.cuh"
#include "dev/kernels.h"
#include "host/headers.h"
#include "host/modular_host.h"
#include "host/vardct_tables.h"
#include "host/icc.h"
#include <map>
#include <mutex>
#include <cmath>

namespace jxlgpu {

#define CUDA_OK(expr) do { cudaError_t e_ = (expr); if (e_ != cudaSuccess) throw Error(std::string("CUDA: ") + cudaGetErrorString(e_) + " at " #expr); } while (0)

namespace {

// Device buffers come from the engine's caching pool (cudaMalloc / cudaFree cost more than most encoder kernels; cudaFree also synchronises).
// A buffer goes back to the pool only after the work that uses it has been synchronised (the sessions sync their stream before they let go).
struct Buf { void* p = nullptr; size_t n = 0; void* pool = nullptr; void Alloc(size_t b) { Free(); n = b ? b : 1; p = DeviceGet(n, &pool); } void Free() { if (p) DevicePut(p, n, pool); p = nullptr; } ~Buf() { Free(); }
  Buf() {} Buf(const Buf&) = delete; Buf& operator=(const Buf&) = delete; template <class T> T* as() const { return static_cast<T*>(p); } };

// ---- fixed MA trees (same shape the decoder kernels walk; BFS layout as DecodeTree allocates it)
struct TreeBuilder {
  struct Tmp { int prop; int32_t split; int l, r; int pred; }; std::vector<Tmp> n;
  int Leaf(int pred) { n.push_back({-1, 0, -1, -1, pred}); return int(n.size()) - 1; }
  int Split(int prop, int32_t val, int gt, int le) { n.push_back({prop, val, gt, le, 0}); return int(n.size()) - 1; }
  int Range(int prop, const std::vector<int32_t>& thr, int lo, int hi, int pred) { if (lo >= hi) return Leaf(pred); int mid = (lo + hi) / 2; int gt = Range(prop, thr, mid + 1, hi, pred); int le = Range(prop, thr, lo, mid, pred); return Split(prop, thr[mid], gt, le); }
  int ResidualCtx(int pred) { static const std::vector<int32_t> thr = {-64, -24, -8, -3, -1, 0, 2, 7, 23, 63}; return Range(8, thr, 0, int(thr.size()), pred); }
  int Channels(int nch, int first, int pred) { if (nch == 1) return ResidualCtx(pred); int mid = first + nch / 2 - 1; int gt = Channels(nch - nch / 2, mid + 1, pred); int le = Channels(nch / 2, first, pred); return Split(0, mid, gt, le); }
  Tree Flatten(int root) {
    Tree tree; std::vector<int> queue{root}; size_t head = 0; int leaf = 0;
    while (head < queue.size()) { const Tmp t = n[queue[head++]]; TreeNode o;
      if (t.prop < 0) { o.property = -1; o.predictor = t.pred; o.leaf_id = leaf++; } else { o.property = t.prop; o.splitval = t.split; o.lchild = int(queue.size()); o.rchild = int(queue.size()) + 1; queue.push_back(t.l); queue.push_back(t.r); }
      tree.push_back(o); }
    return tree;
  }
};
Tree MakeVarDctTree(uint32_t nlf, int num_ec, bool varying_hf_mul, bool varying_cfl) {
  // Zero predictor: constant maps decode as zero-entropy rows. Maps that vary (effort >= 5) are predicted from the left neighbour.
  TreeBuilder b; int sharp = b.Leaf(0), hfmul = b.Leaf(varying_hf_mul ? 1 : 0), strat = b.Leaf(0), cflc = b.Leaf(varying_cfl ? 1 : 0);
  int blockinfo = b.Split(2, 0, hfmul, strat); int hfmeta = b.Split(0, 1, b.Split(0, 2, sharp, blockinfo), cflc);
  int groups = num_ec > 0 ? b.Channels(num_ec, 0, 5) : b.Leaf(5); int upper = b.Split(1, int32_t(3 * nlf + 17), groups, hfmeta);
  int lfc = b.Channels(3, 0, 5); int global = b.Leaf(5); int lower = b.Split(1, 0, lfc, global);
  return b.Flatten(b.Split(1, int32_t(2 * nlf), upper, lower));
}
Tree MakeLosslessTree(int nch) { TreeBuilder b; return b.Flatten(b.Channels(nch, 0, 5)); }
// leaf reached for the given properties (only the properties the fixed trees test: 0 channel, 1 stream, 2 y, 8 previous residual)
const TreeNode& LeafFor(const Tree& t, int chan, int stream, int y, int prop8) {
  int i = 0; while (t[i].property >= 0) { int p = t[i].property; int v = p == 0 ? chan : p == 1 ? stream : p == 2 ? y : prop8; i = v > t[i].splitval ? t[i].lchild : t[i].rchild; } return t[i];
}
const int32_t kProp8Rep[11] = {-100, -40, -10, -5, -2, 0, 1, 5, 10, 40, 100};   // one representative per bucket of ResidualCtx

// tiny host-side Modular tokeniser for the HF-metadata image (a few thousand samples): predictors W (1) and gradient (5)
void TokenizeSmallChannel(const std::vector<int32_t>& px, int w, int h, int chan, int stream, const Tree& tree, std::vector<Token>* out) {
  for (int y = 0; y < h; y++) { int32_t prev_grad = 0; for (int x = 0; x < w; x++) {
    auto at = [&](int yy, int xx) { return px[size_t(yy) * w + xx]; };
    int32_t W = x ? at(y, x - 1) : (y ? at(y - 1, x) : 0), N = y ? at(y - 1, x) : W, NW = (x && y) ? at(y - 1, x - 1) : W;
    const TreeNode& leaf = LeafFor(tree, chan, stream, y, W - prev_grad);
    int32_t pred = leaf.predictor == 0 ? 0 : leaf.predictor == 1 ? W : std::max(std::min(W, N), std::min(std::max(W, N), W + N - NW)); JXLG_CHECK(leaf.predictor == 0 || leaf.predictor == 1 || leaf.predictor == 5, "fixed tree predictor");
    out->push_back({uint32_t(leaf.leaf_id), PackSigned(at(y, x) - pred)}); prev_grad = W + N - NW; } }
}

void QuantizerFromDistance(float d, uint32_t* global_scale, uint32_t* quant_lf, float* q_ac) {
  d = std::max(d, 0.01f); float qac = 0.79f / d; float eff = 0.3f * std::pow(d / 0.3f, 0.83f); eff = std::min(d, std::max(0.5f * d, eff)); float qdc = std::min(50.0f, 1.0959f / eff);
  float scale = 65536.0f * qac / 5.0f; scale = std::min(32768.0f, std::max(1.0f, scale)); int gs = int(scale); int sdc = int(qdc * 4096.0f * 1.6f); if (gs > sdc) gs = std::max(1, sdc);
  *global_scale = uint32_t(gs); float v = qdc * (65536.0f / float(gs)) + 0.5f; *quant_lf = uint32_t(std::max(1.0f, std::min(65536.0f, v))); *q_ac = qac;
}

// appends `nbits` bits of a byte buffer to a bit writer at any alignment
void AppendBits(BitWriter& bw, const uint8_t* p, uint64_t nbits) {
  uint64_t full = nbits / 8; size_t i = 0;
  if ((bw.pos & 7) == 0 && full) {   // byte-aligned destination (an AC stream opens its section): one memcpy
    const size_t byte = bw.pos >> 3, need = byte + full + 16; if (bw.buf.size() < need) bw.buf.resize(need * 2, 0);
    memcpy(&bw.buf[byte], p, full); bw.pos += full * 8; i = full;
  }
  for (; i + 7 <= full; i += 7) { uint64_t v = 0; memcpy(&v, p + i, 7); bw.Write(56, v); } for (; i < full; i++) bw.Write(8, p[i]);
  int rem = int(nbits & 7); if (rem) bw.Write(rem, p[full] & ((1u << rem) - 1));
}

struct DeviceEncCode { Buf ctx_map, freq, start, rev, desc; };
void UploadEncCode(const EncCode& c, DeviceEncCode* d, cudaStream_t st) {
  size_t ncl = c.cfg.size(); std::vector<uint16_t> freq(ncl * kEncAlphabet, 0), start(ncl * kEncAlphabet, 0), rev(c.use_prefix ? 8 : ncl * 4096, 0);
  if (c.use_prefix) {   // prefix codes (efforts 1-2): `freq` carries the code lengths, `start` the bit-reversed code words (k_enc_prefix)
    for (size_t k = 0; k < ncl; k++) { const PrefixTable& p = c.prefix[k]; JXLG_CHECK(p.len.size() <= kEncAlphabet, "encoder alphabet"); for (size_t s = 0; s < p.len.size(); s++) { freq[k * kEncAlphabet + s] = p.max_len ? p.len[s] : 0; start[k * kEncAlphabet + s] = p.max_len ? p.enc_code[s] : 0; } }
  } else
  for (size_t k = 0; k < ncl; k++) { JXLG_CHECK((size_t(1) << c.log_alpha) <= kEncAlphabet, "encoder alphabet"); for (size_t s = 0; s < (size_t(1) << c.log_alpha); s++) { freq[k * kEncAlphabet + s] = c.ans[k].freq[s]; start[k * kEncAlphabet + s] = uint16_t(c.sym_start[k][s]); } memcpy(&rev[k * 4096], c.rev[k].data(), 4096 * 2); }
  d->ctx_map.Alloc(c.ctx_map.size()); d->freq.Alloc(freq.size() * 2); d->start.Alloc(start.size() * 2); d->rev.Alloc(rev.size() * 2); d->desc.Alloc(sizeof(DEncCode));
  CUDA_OK(cudaMemcpyAsync(d->ctx_map.p, c.ctx_map.data(), c.ctx_map.size(), cudaMemcpyHostToDevice, st)); CUDA_OK(cudaMemcpyAsync(d->freq.p, freq.data(), freq.size() * 2, cudaMemcpyHostToDevice, st));
  CUDA_OK(cudaMemcpyAsync(d->start.p, start.data(), start.size() * 2, cudaMemcpyHostToDevice, st)); CUDA_OK(cudaMemcpyAsync(d->rev.p, rev.data(), rev.size() * 2, cudaMemcpyHostToDevice, st));
  DEncCode h{d->ctx_map.as<uint8_t>(), d->freq.as<uint16_t>(), d->start.as<uint16_t>(), d->rev.as<uint16_t>()}; CUDA_OK(cudaMemcpyAsync(d->desc.p, &h, sizeof(h), cudaMemcpyHostToDevice, st)); CUDA_OK(cudaStreamSynchronize(st));
}

std::vector<std::vector<uint64_t>> HistFromDevice(const uint32_t* d_hist, size_t num_ctx, cudaStream_t st) {
  std::vector<uint32_t> raw(num_ctx * kEncAlphabet); CUDA_OK(cudaMemcpyAsync(raw.data(), d_hist, raw.size() * 4, cudaMemcpyDeviceToHost, st)); CUDA_OK(cudaStreamSynchronize(st));
  std::vector<std::vector<uint64_t>> h(num_ctx); for (size_t c = 0; c < num_ctx; c++) { size_t last = 0; bool any = false; for (size_t s = 0; s < kEncAlphabet; s++) if (raw[c * kEncAlphabet + s]) { last = s; any = true; } if (any) { h[c].resize(last + 1); for (size_t s = 0; s <= last; s++) h[c][s] = raw[c * kEncAlphabet + s]; } }
  return h;
}
void AddTokensToHist(const std::vector<Token>& toks, const HybridCfg& cfg, std::vector<std::vector<uint64_t>>* h) { for (const Token& t : toks) { uint32_t tok, nb, bits; HybridEncode(cfg, t.value, &tok, &nb, &bits); auto& hh = (*h)[t.ctx]; if (hh.size() <= tok) hh.resize(tok + 1, 0); hh[tok]++; } }

const DTables* EncDeviceTables() {
  static std::mutex mu; static std::map<int, DTables*> per_dev; std::lock_guard<std::mutex> lk(mu); int dev = 0; CUDA_OK(cudaGetDevice(&dev)); auto it = per_dev.find(dev); if (it != per_dev.end()) return it->second;
  std::unique_ptr<DTables> h(new DTables); FillDeviceTables(h.get()); DTables* d = nullptr; CUDA_OK(cudaMalloc(&d, sizeof(DTables))); CUDA_OK(cudaMemcpy(d, h.get(), sizeof(DTables), cudaMemcpyHostToDevice));
  float lut[256]; for (int i = 0; i < 256; i++) { float v = float(i) * (1.0f / 255.0f); lut[i] = v <= 0.04045f ? v / 12.92f : std::pow((v + 0.055f) / 1.055f, 2.4f); } UploadSrgbLut(lut); per_dev[dev] = d; return d;
}

}  // namespace


// ================================================================================================================================
// The encoder as three steps over a BAND of the frame, so that one frame can be encoded by several GPUs (BASELINE config 5, SURVEY §8e
// "Encode sharding"; N/Encoder/JxlEncoder.cpp:128,367 is where the reference hands the whole frame to libjxl):
//   Begin     upload the band's rows, scan them (isGray / hasTransparency, N/Encoder/JxlEncoder.cpp:33-77)         -> band flags
//   Tokenize  (frame flags = OR over bands)  pixels -> XYB -> DCT -> quantise -> tokens -> histograms              -> band histograms
//   Finish    (frame histograms = sum over bands)  entropy codes -> ANS streams -> this band's sections
// and AssembleFile, which writes headers, LfGlobal, HfGlobal and the TOC around the sections of all bands. A band is a whole number of
// LF-group rows (2048 pixel rows): LF groups, AC groups and Modular groups are then independent of the other bands, and the only things
// the bands share are the two small reductions above (4 bytes and the histograms). SaveImage is the same code with a single band, so a
// frame encoded in bands is bit-identical to the same frame encoded at once.
// ================================================================================================================================
namespace {

const size_t kNumAcCtx = size_t(495) * 15;

// Everything that depends on the frame only (size, options, pixel format), never on pixels.
struct EncPlan {
  bool lossless = false, is_gray = false, has_alpha = false; int ncolor = 3, num_ec = 0, nplanes = 0;
  ImageMetadata m; FrameHeader fh;
  Tree tree; std::vector<Token> tree_tokens; EncCode tree_code; size_t nleaves = 0; std::vector<uint16_t> leaf_lut;
  EncOptions mopt, aopt; uint32_t global_scale = 1, quant_lf = 16; float q_ac = 1;
  bool groups_have_modular = false, global_has_modular = false, single = false, aq = false, cfl = false; GroupHeader plain, gheader;
  size_t HistWords() const { return (nleaves + (lossless ? 0 : kNumAcCtx)) * kEncAlphabet; }
};

EncPlan MakePlan(uint32_t xs, uint32_t ys, uint32_t flags, const EncodeRequest& req) {
  EncPlan p; p.lossless = req.lossless;
  p.is_gray = !(flags & 1) && req.icc_size == 0; p.has_alpha = (flags & 2) != 0;
  ImageMetadata& m = p.m; m.xsize = xs; m.ysize = ys; m.xyb_encoded = !p.lossless; m.ce.intent = 0;   // sRGB, perceptual intent (N/Encoder/JxlEncoder.cpp:269-282)
  if (p.is_gray) m.ce.color_space = kCsGray;
  if (req.icc_size) { m.ce.want_icc = true; m.icc.assign(req.icc, req.icc + req.icc_size); }        // N/Encoder/JxlEncoder.cpp:258-262
  if (p.has_alpha) { ExtraChannelInfo a; a.type = kEcAlpha; m.ec.push_back(a); }
  p.num_ec = p.has_alpha ? 1 : 0; p.ncolor = p.is_gray ? 1 : 3; p.nplanes = p.lossless ? p.ncolor + p.num_ec : p.num_ec;
  FrameHeader& fh = p.fh; fh.encoding = p.lossless ? 1 : 0; fh.ec_upsampling.assign(p.num_ec, 1); fh.ec_blending.assign(p.num_ec, BlendingInfo());
  if (p.lossless) { fh.group_size_shift = 1; fh.lf.gab = false; fh.lf.epf_iters = 0; }
  else {
    const bool hi = req.effort >= 5; int epf = 0;
    if (hi) { const float thr[3] = {0.7f, 1.5f, 4.0f}; for (float t : thr) if (req.distance >= t) epf++; }
    fh.lf.gab = hi; fh.lf.epf_iters = uint32_t(epf);
  }
  DeriveFrameDims(fh, m);
  const uint32_t nlf = fh.num_lf_groups;
  p.single = NumTocEntries(fh) == 1;
  // effort >= 5: adaptive quantisation and chroma from luma (block-local decisions made on the device; what libjxl's higher efforts add first)
  p.aq = p.cfl = !p.lossless && req.effort >= 5;
  p.tree = p.lossless ? MakeLosslessTree(p.ncolor + p.num_ec) : MakeVarDctTree(nlf, p.num_ec, p.aq, p.cfl); TokenizeTree(p.tree, &p.tree_tokens);
  EncOptions topt; topt.cfg = HybridCfg{4, 1, 0}; p.mopt.cfg = HybridCfg{4, 1, 0}; p.mopt.max_clusters = 48; p.aopt.cfg = HybridCfg{4, 2, 0}; p.aopt.max_clusters = 64;
  if (req.effort <= 2) { p.mopt.use_prefix = true; p.aopt.use_prefix = true; }   // the fastest efforts write prefix codes: no serial state chain in the stream writer
  p.tree_code = BuildCode({&p.tree_tokens}, 6, topt); p.nleaves = NumLeaves(p.tree);
  // leaf LUT for the device tokeniser: kind 0 = LF coefficient streams, 1 = pass-group streams, 2 = global stream
  p.leaf_lut.assign(3 * 8 * 11, 0);
  for (int kind = 0; kind < 3; kind++) for (int c = 0; c < 8; c++) for (int b = 0; b < 11; b++) {
    const int stream = kind == 0 ? 1 : kind == 1 ? int(1 + 3 * nlf + 17) : 0;
    p.leaf_lut[(kind * 8 + c) * 11 + b] = uint16_t(LeafFor(p.tree, c, stream, 1, kProp8Rep[b]).leaf_id);
  }
  if (!p.lossless) QuantizerFromDistance(req.distance, &p.global_scale, &p.quant_lf, &p.q_ac);
  const uint32_t gd = fh.group_dim;
  p.groups_have_modular = p.nplanes > 0 && (xs > gd || ys > gd); p.global_has_modular = p.nplanes > 0 && !p.groups_have_modular;
  p.plain.use_global_tree = true; p.gheader = p.plain;
  if (p.lossless && p.ncolor == 3) { Transform t; t.id = 0; t.begin_c = 0; t.rct_type = 6; p.gheader.transforms.push_back(t); }
  return p;
}

std::vector<std::vector<uint64_t>> TrimmedHist(const uint64_t* flat, size_t num_ctx) {
  std::vector<std::vector<uint64_t>> h(num_ctx);
  for (size_t c = 0; c < num_ctx; c++) {
    const uint64_t* row = flat + c * kEncAlphabet; size_t last = 0; bool any = false;
    for (size_t s = 0; s < kEncAlphabet; s++) if (row[s]) { last = s; any = true; }
    if (any) h[c].assign(row, row + last + 1);
  }
  return h;
}

}  // namespace

// kind: 0 global Modular stream, 1 LF group, 2 pass group. The payload is either owned (`bytes`) or a view into a band's serialised blob.
struct BandSection { uint32_t kind = 0, index = 0; uint64_t bits = 0; std::vector<uint8_t> bytes; const uint8_t* view = nullptr; size_t view_n = 0;
  const uint8_t* data() const { return view ? view : bytes.data(); } size_t size() const { return view ? view_n : bytes.size(); } };

class BandEncoder {
 public:
  explicit BandEncoder(const EncodeRequest& r) : req(r) {}
  ~BandEncoder() { if (st) { cudaStreamSynchronize(st); cudaStreamDestroy(st); } }
  uint32_t Begin();                                         // -> flags of this band (bit 0: a non-gray pixel, bit 1: a non-opaque pixel)
  std::vector<uint64_t> Tokenize(uint32_t frame_flags);     // -> this band's histograms, [context][kEncAlphabet] (Modular contexts, then AC contexts)
  std::vector<BandSection> Finish(const std::vector<uint64_t>& frame_hist);
  int64_t DebugStage(int32_t which, void* out, int64_t capacity, int64_t* dims4);   // JxlB200BandEncoderDebugStage
  const EncPlan& Plan() const { return plan; }
  float device_ms = 0;

 private:
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

uint32_t BandEncoder::Begin() {
  std::string why; JXLG_CHECK(CudaAvailable(&why), why);
  JXLG_CHECK(req.width > 0 && req.height > 0 && req.stride >= req.width * 4, "invalid bitmap");
  frame_h = req.frame_height ? req.frame_height : req.height;
  if (req.frame_height) {   // band of a larger frame
    JXLG_CHECK(req.band_y0 % 2048 == 0 && uint64_t(req.band_y0) + req.height <= frame_h, "band: the first row must be a multiple of 2048 (one LF-group row) inside the frame");
    JXLG_CHECK(req.band_y0 + req.height == frame_h || req.height % 2048 == 0, "band: the row count must be a multiple of 2048 unless the band ends the frame");
    JXLG_CHECK(req.halo_top == std::min<uint32_t>(8, req.band_y0) && req.halo_bottom == std::min<uint32_t>(8, frame_h - (req.band_y0 + req.height)), "band: 8 halo rows are needed on every side that has a neighbour");
  } else JXLG_CHECK(req.band_y0 == 0 && req.halo_top == 0 && req.halo_bottom == 0, "band fields without a frame height");
  CUDA_OK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
  Timer t(st, &device_ms);
  const size_t rows = size_t(req.halo_top) + req.height + req.halo_bottom, in_bytes = size_t(req.stride) * rows;
  const uint8_t* base = req.bgra;
  if (!req.device_input) { d_in.Alloc(in_bytes); CUDA_OK(cudaMemcpyAsync(d_in.p, req.bgra, in_bytes, cudaMemcpyHostToDevice, st)); base = d_in.as<uint8_t>(); }
  d_bgra = base + size_t(req.halo_top) * req.stride;
  d_flags.Alloc(16); CUDA_OK(cudaMemsetAsync(d_flags.p, 0, 16, st)); EncLaunchScan(d_bgra, req.width, req.height, req.stride, d_flags.as<uint32_t>(), st);
  uint32_t flags = 0; CUDA_OK(cudaMemcpyAsync(&flags, d_flags.p, 4, cudaMemcpyDeviceToHost, st)); CUDA_OK(cudaStreamSynchronize(st));
  return flags;
}

std::vector<uint64_t> BandEncoder::Tokenize(uint32_t frame_flags) {
  Timer t(st, &device_ms); stages_valid = false;
  const uint32_t xs = req.width, ys = req.height;
  plan = MakePlan(xs, frame_h, frame_flags, req);
  const bool lossless = plan.lossless; const int nplanes = plan.nplanes;
  // lossy with an ICC source profile: libjxl gets the source -> XYB mapping from a CMS, the engine reads a matrix/TRC profile directly
  IccMatrixTrc src_profile; bool has_src_profile = false;
  if (req.icc_size && !lossless) { std::string why; JXLG_CHECK(ParseMatrixTrcIcc(req.icc, req.icc_size, &src_profile, &why), why + " — lossy encoding of this profile needs a CMS, which the engine does not have"); has_src_profile = true; }
  // the band as an image of its own: same width, same options, its own block / group / LF-group grid
  { ImageMetadata mb = plan.m; mb.ysize = ys; fb = plan.fh; DeriveFrameDims(fb, mb); }
  const uint32_t nlf = fb.num_lf_groups, ng = fb.num_groups, gd = fb.group_dim;
  lf_group0 = (req.band_y0 / 2048) * plan.fh.xlfgroups; group0 = (req.band_y0 / gd) * plan.fh.xgroups;
  JXLG_CHECK(fb.xlfgroups == plan.fh.xlfgroups && fb.xgroups == plan.fh.xgroups, "band layout");
  // ---- device frame
  memset(&e, 0, sizeof(e)); e.xsize = xs; e.ysize = ys; e.stride = req.stride; e.xb = fb.xblocks; e.yb = fb.yblocks; e.xpad = e.xb * 8; e.ypad = e.yb * 8;
  e.xgroups = fb.xgroups; e.ygroups = fb.ygroups; e.num_groups = ng; e.gray = plan.is_gray; e.alpha = plan.has_alpha;
  const bool gab = !lossless && plan.fh.lf.gab;
  e.ext_top = gab ? req.halo_top : 0; e.ext_rows = e.ext_top + e.ypad + ((gab && req.halo_bottom) ? 8 : 0);
  e.src_row_min = -int32_t(req.halo_top); e.src_row_max = int32_t(ys) - 1 + int32_t(req.halo_bottom);
  if (has_src_profile) {
    d_srclut.Alloc(sizeof(src_profile.lut)); CUDA_OK(cudaMemcpyAsync(d_srclut.p, src_profile.lut, sizeof(src_profile.lut), cudaMemcpyHostToDevice, st));
    e.src_lut = d_srclut.as<float>(); e.has_src_profile = 1; for (int i = 0; i < 9; i++) e.src_matrix[i] = float(src_profile.to_linear_srgb[i]);
  }
  e.tables = EncDeviceTables();
  const size_t npx = size_t(xs) * ys, epx = size_t(e.xpad) * e.ext_rows, cells = size_t(e.xb) * e.yb;
  e.alpha_plane = lossless ? uint32_t(plan.ncolor) : 0;
  d_e.Alloc(sizeof(DEncFrame)); if (nplanes) d_planes.Alloc(npx * nplanes * 4); e.planes = d_planes.as<int32_t>();
  d_lut.Alloc(plan.leaf_lut.size() * 2); CUDA_OK(cudaMemcpyAsync(d_lut.p, plan.leaf_lut.data(), plan.leaf_lut.size() * 2, cudaMemcpyHostToDevice, st));
  // ---- Modular streams: LF coefficients per LF group (VarDCT), then alpha / lossless colour per group (or one global stream for a one-group frame)
  uint64_t token_cursor = 0; byte_cursor = 0; max_mod_tokens = 0; mod_streams.clear(); m_streams.clear();
  auto add_mod_stream = [&](uint32_t x0, uint32_t y0, uint32_t w, uint32_t h, uint32_t kind, uint32_t nch) {
    DEncModStream s{x0, y0, w, h, kind, 0, token_cursor}; mod_streams.push_back(s);
    const uint32_t cnt = w * h * nch; DEncStream es{token_cursor, byte_cursor, cnt, 0}; m_streams.push_back(es);
    token_cursor += cnt; byte_cursor += (size_t(cnt) * 6 + 16 + 15) / 16 * 16; max_mod_tokens = std::max(max_mod_tokens, cnt);
  };
  first_lf_stream = 0;
  if (!lossless) for (uint32_t g = 0; g < nlf; g++) { const uint32_t gx = g % fb.xlfgroups, gy = g / fb.xlfgroups; add_mod_stream(gx * 256, gy * 256, std::min<uint32_t>(256, e.xb - gx * 256), std::min<uint32_t>(256, e.yb - gy * 256), 0, 3); }
  first_group_stream = uint32_t(mod_streams.size());
  if (plan.groups_have_modular) for (uint32_t g = 0; g < ng; g++) { const uint32_t gx = g % fb.xgroups, gy = g / fb.xgroups; add_mod_stream(gx * gd, gy * gd, std::min(gd, xs - gx * gd), std::min(gd, ys - gy * gd), 1, uint32_t(nplanes)); }
  else if (plan.global_has_modular) add_mod_stream(0, 0, xs, ys, 2, uint32_t(nplanes));
  const uint64_t ac_token_off = token_cursor; if (!lossless) token_cursor += uint64_t(ng) * kMaxAcTokensPerGroup; e.ac_token_off = ac_token_off;
  d_tokens.Alloc(std::max<uint64_t>(token_cursor, 1) * 8); e.tokens = d_tokens.as<uint2>();
  if (!lossless) {
    const float inv_gs = 65536.0f / float(plan.global_scale); OpsinInverse op;
    e.hf_mul = uint32_t(std::max(1, std::min(255, int(std::lrintf(plan.q_ac * 65536.0f / float(plan.global_scale)))))); e.inv_gs = inv_gs;
    e.xm = std::pow(0.8f, float(plan.fh.x_qm_scale) - 2.0f); e.bm = std::pow(0.8f, float(plan.fh.b_qm_scale) - 2.0f); e.kx = 0.f; e.kb = 1.f;
    const float lfd[3] = {1.0f / 4096, 1.0f / 512, 1.0f / 256}; for (int c = 0; c < 3; c++) e.lf_fac[c] = lfd[c] * inv_gs / float(plan.quant_lf);
    e.cfl_x_lf = 0.f; e.cfl_b_lf = 1.f; for (int i = 0; i < 4; i++) e.quant_bias[i] = op.quant_bias[i];
    d_xyb.Alloc(epx * 12); d_lf.Alloc(cells * 12); d_lfq.Alloc(cells * 12); d_coeffs.Alloc(size_t(ng) * 3 * 65536 * 2); d_nz.Alloc(cells * 3); d_account.Alloc(size_t(ng) * 4);
    std::vector<float> dq = ComputeDequantTable(0, LibraryEncoding(0)); d_dq.Alloc(dq.size() * 4); CUDA_OK(cudaMemcpyAsync(d_dq.p, dq.data(), dq.size() * 4, cudaMemcpyHostToDevice, st));
    std::vector<uint32_t> nat = NaturalOrder(1, 1); std::vector<uint16_t> o16(nat.begin(), nat.end()); d_order.Alloc(128); CUDA_OK(cudaMemcpyAsync(d_order.p, o16.data(), 128, cudaMemcpyHostToDevice, st));
    e.xyb = d_xyb.as<float>(); e.lf = d_lf.as<float>(); e.lfq = d_lfq.as<int32_t>(); e.coeffs = d_coeffs.as<int16_t>(); e.nz = d_nz.as<uint8_t>();
    e.dequant8 = d_dq.as<float>(); e.order8 = d_order.as<uint16_t>(); e.ac_token_count = d_account.as<uint32_t>();
    CUDA_OK(cudaMemsetAsync(d_coeffs.p, 0, d_coeffs.n, st));
    e.xt = (e.xb + 7) / 8; e.yt = (e.yb + 7) / 8;
    if (plan.aq || plan.cfl) {
      d_hfm.Alloc(cells); d_ytox.Alloc(size_t(e.xt) * e.yt); d_ytob.Alloc(size_t(e.xt) * e.yt); d_stats.Alloc(cells * 16);
      e.hf_mul_map = d_hfm.as<uint8_t>(); e.ytox_map = d_ytox.as<int8_t>(); e.ytob_map = d_ytob.as<int8_t>(); e.block_stats = d_stats.as<float>();
      e.aq_on = plan.aq; e.cfl_on = plan.cfl; e.aq_ref = 0.05f;
    }
  }
  d_bytes.Alloc(std::max<uint64_t>(byte_cursor + (lossless ? 0 : uint64_t(ng) * (size_t(kMaxAcTokensPerGroup) * 6 + 16)), 16)); d_bits.Alloc((mod_streams.size() + ng + 1) * 8);
  e.stream_bytes = d_bytes.as<uint8_t>(); e.stream_bits = d_bits.as<uint64_t>();
  CUDA_OK(cudaMemcpyAsync(d_e.p, &e, sizeof(e), cudaMemcpyHostToDevice, st)); const DEncFrame* de = d_e.as<DEncFrame>();
  // ---- pixels -> planes / XYB -> DCT + quant
  if (lossless) EncLaunchToPlanes(de, e, d_bgra, st);
  else {
    EncLaunchToXyb(de, e, d_bgra, st);
    if (gab) {   // approximate inverse gaborish: two Van Cittert iterations against the decoder's own kernel. Mirrored edges at the borders of the extended plane:
                 // the padded frame's own borders where the band touches them, halo rows (discarded afterwards) where a neighbouring band lies
      d_tmp1.Alloc(epx * 12); d_tmp2.Alloc(epx * 12); d_gabframe.Alloc(sizeof(DFrame));
      DFrame gf; memset(&gf, 0, sizeof(gf)); gf.xsize = e.xpad; gf.ysize = e.ext_rows; gf.xpad = e.xpad; gf.ypad = e.ext_rows; gf.lpf.gab = 1; memcpy(gf.lpf.gab_w, plan.fh.lf.gab_w, sizeof(gf.lpf.gab_w));
      CUDA_OK(cudaMemcpyAsync(d_gabframe.p, &gf, sizeof(gf), cudaMemcpyHostToDevice, st)); CUDA_OK(cudaMemcpyAsync(d_tmp1.p, d_xyb.p, epx * 12, cudaMemcpyDeviceToDevice, st));
      for (int it = 0; it < 2; it++) { LaunchGaborishPlanes(d_gabframe.as<DFrame>(), gf, e.xyb, d_tmp2.as<float>(), st); EncLaunchSharpen(e.xyb, d_tmp1.as<float>(), d_tmp2.as<float>(), epx * 3, st); }
    }
    if (e.hf_mul_map) EncLaunchBlockParams(de, e, st);
    EncLaunchDct8(de, e, st); EncLaunchAcTokens(de, e, st);
  }
  // ---- Modular tokens on the device
  d_modstreams.Alloc(std::max<size_t>(mod_streams.size(), 1) * sizeof(DEncModStream));
  if (!mod_streams.empty()) CUDA_OK(cudaMemcpyAsync(d_modstreams.p, mod_streams.data(), mod_streams.size() * sizeof(DEncModStream), cudaMemcpyHostToDevice, st));
  if (!lossless && nlf) { uint32_t mx = 0; for (uint32_t g = 0; g < nlf; g++) mx = std::max(mx, m_streams[first_lf_stream + g].count);
    EncLaunchModTokens(de, d_modstreams.as<DEncModStream>() + first_lf_stream, nlf, mx, e.lfq, e.xb, e.yb, 3, d_lut.as<uint16_t>(), st); }
  if (mod_streams.size() > first_group_stream) { const uint32_t n = uint32_t(mod_streams.size()) - first_group_stream; uint32_t mx = 0; for (uint32_t i = 0; i < n; i++) mx = std::max(mx, m_streams[first_group_stream + i].count);
    EncLaunchModTokens(de, d_modstreams.as<DEncModStream>() + first_group_stream, n, mx, e.planes, xs, ys, uint32_t(nplanes), d_lut.as<uint16_t>(), st); }
  // ---- AC stream descriptors need the per-group token counts
  a_streams.clear(); ac_counts.assign(ng, 0);
  if (!lossless) { CUDA_OK(cudaMemcpyAsync(ac_counts.data(), d_account.p, size_t(ng) * 4, cudaMemcpyDeviceToHost, st)); CUDA_OK(cudaStreamSynchronize(st));
    for (uint32_t g = 0; g < ng; g++) { DEncStream s{ac_token_off + uint64_t(g) * kMaxAcTokensPerGroup, byte_cursor, ac_counts[g], 0}; a_streams.push_back(s); byte_cursor += (size_t(ac_counts[g]) * 6 + 16 + 15) / 16 * 16; } }
  std::vector<DEncStream> all = m_streams; all.insert(all.end(), a_streams.begin(), a_streams.end());
  d_streams.Alloc(std::max<size_t>(all.size(), 1) * sizeof(DEncStream)); if (!all.empty()) CUDA_OK(cudaMemcpyAsync(d_streams.p, all.data(), all.size() * sizeof(DEncStream), cudaMemcpyHostToDevice, st));
  const DEncStream* d_m = d_streams.as<DEncStream>(); const DEncStream* d_a = d_m + m_streams.size();
  // ---- histograms
  const size_t nleaves = plan.nleaves;
  d_hist_m.Alloc(nleaves * kEncAlphabet * 4); CUDA_OK(cudaMemsetAsync(d_hist_m.p, 0, d_hist_m.n, st)); EncLaunchHistogram(e.tokens, d_m, uint32_t(m_streams.size()), max_mod_tokens, d_hist_m.as<uint32_t>(), st);
  uint32_t max_ac = 0; for (uint32_t c : ac_counts) max_ac = std::max(max_ac, c);
  if (!lossless) { d_hist_a.Alloc(kNumAcCtx * kEncAlphabet * 4); CUDA_OK(cudaMemsetAsync(d_hist_a.p, 0, d_hist_a.n, st)); EncLaunchHistogram(e.tokens, d_a, ng, max_ac, d_hist_a.as<uint32_t>(), st); }
  std::vector<uint64_t> hist(plan.HistWords(), 0);
  { std::vector<uint32_t> raw(nleaves * kEncAlphabet); CUDA_OK(cudaMemcpyAsync(raw.data(), d_hist_m.p, raw.size() * 4, cudaMemcpyDeviceToHost, st)); CUDA_OK(cudaStreamSynchronize(st)); for (size_t i = 0; i < raw.size(); i++) hist[i] = raw[i]; }
  if (!lossless) { std::vector<uint32_t> raw(kNumAcCtx * kEncAlphabet); CUDA_OK(cudaMemcpyAsync(raw.data(), d_hist_a.p, raw.size() * 4, cudaMemcpyDeviceToHost, st)); CUDA_OK(cudaStreamSynchronize(st)); uint64_t* dst = hist.data() + nleaves * kEncAlphabet; for (size_t i = 0; i < raw.size(); i++) dst[i] = raw[i]; }
  // HF metadata is tokenised on the host: every block DCT8, constant EPF sharpness; the quantiser multipliers and chroma-from-luma factors are
  // constants below effort 5 and device-computed maps from effort 5 on (one byte per block / per tile to download)
  std::vector<uint8_t> h_hfm; std::vector<int8_t> h_ytox, h_ytob;
  if (e.hf_mul_map) { h_hfm.resize(cells); h_ytox.resize(size_t(e.xt) * e.yt); h_ytob.resize(h_ytox.size());
    CUDA_OK(cudaMemcpyAsync(h_hfm.data(), d_hfm.p, h_hfm.size(), cudaMemcpyDeviceToHost, st)); CUDA_OK(cudaMemcpyAsync(h_ytox.data(), d_ytox.p, h_ytox.size(), cudaMemcpyDeviceToHost, st));
    CUDA_OK(cudaMemcpyAsync(h_ytob.data(), d_ytob.p, h_ytob.size(), cudaMemcpyDeviceToHost, st)); CUDA_OK(cudaStreamSynchronize(st)); }
  hfmeta_tokens.assign(nlf, {}); hfmeta_nb.assign(nlf, 0);
  if (!lossless) for (uint32_t g = 0; g < nlf; g++) {
    const uint32_t gx = g % fb.xlfgroups, gy = g / fb.xlfgroups; const int w = int(std::min<uint32_t>(256, e.xb - gx * 256)), h = int(std::min<uint32_t>(256, e.yb - gy * 256)), tw = (w + 7) / 8, th = (h + 7) / 8, nb = w * h; hfmeta_nb[g] = uint32_t(nb);
    const int sid = int(1 + 2 * plan.fh.num_lf_groups + lf_group0 + g);
    std::vector<int32_t> cflx(size_t(tw) * th, 0), cflb(size_t(tw) * th, 0), info(size_t(nb) * 2, 0), sharp(size_t(w) * h, plan.fh.lf.epf_iters ? 4 : 0); for (int i = 0; i < nb; i++) info[nb + i] = int32_t(e.hf_mul) - 1;
    if (!h_hfm.empty()) {   // maps decided on the device: per-block multiplier, per-tile chroma-from-luma factors
      for (int y = 0; y < h; y++) for (int x = 0; x < w; x++) info[size_t(nb) + size_t(y) * w + x] = int32_t(h_hfm[size_t(gy * 256 + y) * e.xb + gx * 256 + x]) - 1;
      for (int y = 0; y < th; y++) for (int x = 0; x < tw; x++) { const size_t t = size_t(gy * 32 + y) * e.xt + gx * 32 + x; cflx[size_t(y) * tw + x] = h_ytox[t]; cflb[size_t(y) * tw + x] = h_ytob[t]; }
    }
    TokenizeSmallChannel(cflx, tw, th, 0, sid, plan.tree, &hfmeta_tokens[g]); TokenizeSmallChannel(cflb, tw, th, 1, sid, plan.tree, &hfmeta_tokens[g]);
    TokenizeSmallChannel(info, nb, 2, 2, sid, plan.tree, &hfmeta_tokens[g]); TokenizeSmallChannel(sharp, w, h, 3, sid, plan.tree, &hfmeta_tokens[g]);
    for (const Token& t : hfmeta_tokens[g]) { uint32_t tok, nbits, bits; HybridEncode(plan.mopt.cfg, t.value, &tok, &nbits, &bits); JXLG_CHECK(tok < kEncAlphabet, "HF metadata token"); hist[size_t(t.ctx) * kEncAlphabet + tok]++; }
  }
  stages_valid = true;
  return hist;
}

// Copies one device buffer of the session to `out` (see JxlB200BandEncoderDebugStage for the layouts). dims4 receives the shape even when
// `out` is too small, so that a caller can size its buffer with a first call.
int64_t BandEncoder::DebugStage(int32_t which, void* out, int64_t capacity, int64_t* dims4) {
  JXLG_CHECK(stages_valid, "stage dumps exist only between Tokenize and Finish");
  JXLG_CHECK(which >= 0 && which <= 9, "unknown stage");
  JXLG_CHECK(which == 9 || !plan.lossless, "a lossless session has no VarDCT stages");
  JXLG_CHECK(!(which >= 2 && which <= 4) || e.hf_mul_map, "block statistics and the HF maps exist from effort 5 on");
  const size_t cells = size_t(e.xb) * e.yb, epx = size_t(e.xpad) * e.ext_rows, tiles = size_t(e.xt) * e.yt;
  struct Piece { const void* p; size_t n; }; std::vector<Piece> pieces; int64_t d[4] = {0, 0, 0, 0};
  std::vector<uint32_t> counts;   // stage 9: token count of every stream, written ahead of the tokens
  switch (which) {
    case 0: pieces.push_back({plan.fh.lf.gab ? d_tmp1.p : d_xyb.p, epx * 12}); d[0] = 3; d[1] = e.ext_rows; d[2] = e.xpad; break;
    case 1: pieces.push_back({d_xyb.p, epx * 12}); d[0] = 3; d[1] = e.ext_rows; d[2] = e.xpad; break;
    case 2: pieces.push_back({d_stats.p, cells * 16}); d[0] = e.yb; d[1] = e.xb; d[2] = 4; break;
    case 3: pieces.push_back({d_hfm.p, cells}); d[0] = e.yb; d[1] = e.xb; break;
    case 4: pieces.push_back({d_ytox.p, tiles}); pieces.push_back({d_ytob.p, tiles}); d[0] = 2; d[1] = e.yt; d[2] = e.xt; break;
    case 5: pieces.push_back({d_lf.p, cells * 12}); d[0] = 3; d[1] = e.yb; d[2] = e.xb; break;
    case 6: pieces.push_back({d_lfq.p, cells * 12}); d[0] = 3; d[1] = e.yb; d[2] = e.xb; break;
    case 7: pieces.push_back({d_coeffs.p, size_t(e.num_groups) * 3 * 65536 * 2}); d[0] = e.num_groups; d[1] = 3; d[2] = 1024; d[3] = 64; break;
    case 8: pieces.push_back({d_nz.p, cells * 3}); d[0] = 3; d[1] = e.yb; d[2] = e.xb; break;
    default: {
      uint64_t total = 0;
      for (const std::vector<DEncStream>* v : {&m_streams, &a_streams}) for (const DEncStream& s : *v) {
        counts.push_back(s.count); total += s.count; if (s.count) pieces.push_back({d_tokens.as<uint2>() + s.token_off, size_t(s.count) * 8}); }
      d[0] = int64_t(counts.size()); d[1] = int64_t(total); d[2] = int64_t(m_streams.size());
    }
  }
  if (dims4) memcpy(dims4, d, sizeof(d));
  size_t bytes = counts.size() * 4; for (const Piece& p : pieces) bytes += p.n;
  JXLG_CHECK(out && int64_t(bytes) <= capacity, "stage buffer too small: " + std::to_string(bytes) + " bytes needed");
  uint8_t* o = static_cast<uint8_t*>(out); if (!counts.empty()) { memcpy(o, counts.data(), counts.size() * 4); o += counts.size() * 4; }
  for (const Piece& p : pieces) { CUDA_OK(cudaMemcpyAsync(o, p.p, p.n, cudaMemcpyDeviceToHost, st)); o += p.n; }
  CUDA_OK(cudaStreamSynchronize(st));
  return int64_t(bytes);
}

namespace {
struct FrameCodes { EncCode mcode, acode; };
FrameCodes CodesFromHist(const EncPlan& plan, const std::vector<uint64_t>& hist) {
  JXLG_CHECK(hist.size() == plan.HistWords(), "histogram size");
  FrameCodes c; c.mcode = BuildCodeFromHist(TrimmedHist(hist.data(), plan.nleaves), plan.nleaves, plan.mopt);
  if (!plan.lossless) c.acode = BuildCodeFromHist(TrimmedHist(hist.data() + plan.nleaves * kEncAlphabet, kNumAcCtx), kNumAcCtx, plan.aopt);
  return c;
}
}  // namespace

std::vector<BandSection> BandEncoder::Finish(const std::vector<uint64_t>& frame_hist) {
  const bool lossless = plan.lossless; const uint32_t nlf = fb.num_lf_groups, ng = fb.num_groups;
  stages_valid = false;
  FrameCodes codes = CodesFromHist(plan, frame_hist);
  std::vector<uint64_t> bits_m(m_streams.size(), 0), bits_a(ng, 0), dense_off; std::vector<uint8_t> bytes;
  {
    Timer t(st, &device_ms);
    DeviceEncCode dm, da; UploadEncCode(codes.mcode, &dm, st); if (!lossless) UploadEncCode(codes.acode, &da, st);
    const DEncFrame* de = d_e.as<DEncFrame>(); const DEncStream* d_m = d_streams.as<DEncStream>(); const DEncStream* d_a = d_m + m_streams.size();
    // the Modular streams (few and long: an LF group is one serial stream of 196 608 tokens) and the AC streams (many) are independent: two CUDA streams
    cudaStream_t st2 = nullptr; cudaEvent_t ready = nullptr, done2 = nullptr; CUDA_OK(cudaStreamCreateWithFlags(&st2, cudaStreamNonBlocking)); cudaEventCreateWithFlags(&ready, cudaEventDisableTiming); cudaEventCreateWithFlags(&done2, cudaEventDisableTiming);
    cudaEventRecord(ready, st); cudaStreamWaitEvent(st2, ready, 0);
    const uint32_t nm = uint32_t(m_streams.size());
    if (codes.mcode.use_prefix) EncLaunchPrefix(de, d_m, nm, dm.desc.as<DEncCode>(), 0, st); else EncLaunchAns(de, d_m, nm, dm.desc.as<DEncCode>(), 0, st);
    if (!lossless) { if (codes.acode.use_prefix) EncLaunchPrefix(de, d_a, ng, da.desc.as<DEncCode>(), nm, st2); else EncLaunchAns(de, d_a, ng, da.desc.as<DEncCode>(), nm, st2); }
    cudaEventRecord(done2, st2); cudaStreamWaitEvent(st, done2, 0);
    if (nm) CUDA_OK(cudaMemcpyAsync(bits_m.data(), e.stream_bits, size_t(nm) * 8, cudaMemcpyDeviceToHost, st));
    if (!lossless) CUDA_OK(cudaMemcpyAsync(bits_a.data(), e.stream_bits + nm, size_t(ng) * 8, cudaMemcpyDeviceToHost, st));
    CUDA_OK(cudaStreamSynchronize(st)); cudaStreamDestroy(st2); cudaEventDestroy(ready); cudaEventDestroy(done2);
    // dense copy of what was written: stream k (Modular streams first, then AC) lands at dense_off[k] of `bytes`
    const size_t ns = size_t(nm) + (lossless ? 0 : ng); dense_off.assign(ns + 1, 0);
    for (size_t k = 0; k < ns; k++) { const uint64_t b = k < nm ? bits_m[k] : bits_a[k - nm]; dense_off[k + 1] = dense_off[k] + ((b + 7) / 8 + 15) / 16 * 16; }
    bytes.assign(dense_off[ns], 0);
    if (dense_off[ns]) {
      Buf d_off, d_dense; d_off.Alloc(ns * 8); d_dense.Alloc(dense_off[ns]);
      CUDA_OK(cudaMemcpyAsync(d_off.p, dense_off.data(), ns * 8, cudaMemcpyHostToDevice, st));
      EncLaunchCompact(e.stream_bytes, d_m, uint32_t(ns), e.stream_bits, d_off.as<uint64_t>(), d_dense.as<uint8_t>(), st);
      CUDA_OK(cudaMemcpyAsync(bytes.data(), d_dense.p, dense_off[ns], cudaMemcpyDeviceToHost, st)); CUDA_OK(cudaStreamSynchronize(st));
    }
  }
  std::vector<BandSection> out;
  auto emit = [&](uint32_t kind, uint32_t index, BitWriter& bw) { BandSection s; s.kind = kind; s.index = index; s.bits = bw.pos; s.bytes = bw.Finish(); out.push_back(std::move(s)); };
  if (plan.global_has_modular) { BitWriter bw; const DEncStream& s = m_streams[first_group_stream]; (void)s; AppendBits(bw, &bytes[dense_off[first_group_stream]], bits_m[first_group_stream]); emit(0, 0, bw); }
  if (!lossless) for (uint32_t g = 0; g < nlf; g++) {
    BitWriter bw; bw.Write(2, 0); WriteGroupHeader(bw, plan.plain); AppendBits(bw, &bytes[dense_off[first_lf_stream + g]], bits_m[first_lf_stream + g]);
    const uint32_t gx = g % fb.xlfgroups, gy = g / fb.xlfgroups; const uint64_t wh = uint64_t(std::min<uint32_t>(256, e.xb - gx * 256)) * std::min<uint32_t>(256, e.yb - gy * 256);
    bw.Write(CeilLog2(wh), hfmeta_nb[g] - 1); WriteGroupHeader(bw, plan.plain); WriteTokens(bw, codes.mcode, hfmeta_tokens[g]);
    emit(1, lf_group0 + g, bw);
  }
  for (uint32_t g = 0; g < ng; g++) {
    BitWriter bw;
    if (!lossless) AppendBits(bw, &bytes[dense_off[m_streams.size() + g]], bits_a[g]);
    if (plan.groups_have_modular) { WriteGroupHeader(bw, plan.plain); AppendBits(bw, &bytes[dense_off[first_group_stream + g]], bits_m[first_group_stream + g]); }
    emit(2, group0 + g, bw);
  }
  return out;
}

// Writes the file around the sections of all bands: headers, TOC, LfGlobal (quantiser, MA tree, Modular code), HfGlobal (AC code).
std::vector<uint8_t> AssembleFile(const EncPlan& plan, const std::vector<uint64_t>& frame_hist, const std::vector<const BandSection*>& sections, const EncodeRequest& meta) {
  const FrameHeader& fh = plan.fh; const uint32_t nlf = fh.num_lf_groups, ng = fh.num_groups; const size_t nsec = NumTocEntries(fh); const bool single = plan.single, lossless = plan.lossless;
  FrameCodes codes = CodesFromHist(plan, frame_hist);
  std::vector<const BandSection*> lf_sec(nlf, nullptr), grp_sec(ng, nullptr); const BandSection* global_sec = nullptr;
  for (const BandSection* s : sections) {
    if (s->kind == 0) { JXLG_CHECK(!global_sec, "two global Modular streams"); global_sec = s; }
    else if (s->kind == 1) { JXLG_CHECK(s->index < nlf && !lf_sec[s->index], "LF-group section index"); lf_sec[s->index] = s; }
    else { JXLG_CHECK(s->kind == 2 && s->index < ng && !grp_sec[s->index], "group section index"); grp_sec[s->index] = s; }
  }
  if (!lossless) for (uint32_t g = 0; g < nlf; g++) JXLG_CHECK(lf_sec[g], "a band is missing: LF group without a section");
  for (uint32_t g = 0; g < ng; g++) JXLG_CHECK(grp_sec[g], "a band is missing: group without a section");
  JXLG_CHECK(!plan.global_has_modular || global_sec, "global Modular stream missing");
  if (!single) {
    // Every section of a multi-section frame is byte-aligned and arrives padded: LfGlobal and HfGlobal are written here, the TOC follows from the
    // sizes, and the bands' sections are copied ONCE, straight into the file (a 1 GP frame is 119 MB of sections: every extra pass over them counts).
    BitWriter lfg; lfg.Bool(true);
    if (!lossless) { lfg.U32(BitsOffset(11, 1), BitsOffset(11, 2049), BitsOffset(12, 4097), BitsOffset(16, 8193), plan.global_scale); lfg.U32(Val(16), BitsOffset(5, 1), BitsOffset(8, 1), BitsOffset(16, 1), plan.quant_lf); lfg.Bool(true); lfg.Bool(true); }
    lfg.Bool(true); WriteCode(lfg, plan.tree_code); WriteTokens(lfg, plan.tree_code, plan.tree_tokens); WriteCode(lfg, codes.mcode);
    if (plan.nplanes > 0) WriteGroupHeader(lfg, plan.gheader);
    BitWriter hfg; if (!lossless) { hfg.Bool(true); hfg.Write(CeilLog2(ng), 0); hfg.U32(Val(0x5F), Val(0x13), Val(0), Bits(13), 0); WriteCode(hfg, codes.acode); }
    const std::vector<uint8_t> lfg_bytes = lfg.Finish(), hfg_bytes = hfg.Finish();
    std::vector<size_t> sizes(nsec, 0); sizes[0] = lfg_bytes.size(); sizes[1 + nlf] = hfg_bytes.size();
    for (uint32_t g = 0; g < nlf; g++) sizes[1 + g] = lf_sec[g] ? lf_sec[g]->size() : 0;
    for (uint32_t g = 0; g < ng; g++) sizes[2 + nlf + g] = grp_sec[g]->size();
    BitWriter cs; cs.Write(16, 0x0AFF); WriteImageHeaders(cs, plan.m); WriteFrameHeader(cs, fh, plan.m); WriteToc(cs, sizes); const std::vector<uint8_t> head = cs.Finish();
    uint64_t payload = head.size(); for (size_t v : sizes) payload += v;
    std::vector<uint8_t> file = ContainerPrologue();
    if (meta.exif_size) AppendBox(file, "Exif", meta.exif, meta.exif_size); if (meta.xmp_size) AppendBox(file, "xml ", meta.xmp, meta.xmp_size);
    file.reserve(file.size() + 16 + payload);
    {   // the jxlc box header (extended size past 4 GB), then the payload piece by piece
      uint64_t total = payload + 8; if (total > 0xffffffffull) { total += 8; uint8_t hh[16] = {0, 0, 0, 1, 'j', 'x', 'l', 'c'}; for (int i = 0; i < 8; i++) hh[8 + i] = uint8_t(total >> (56 - 8 * i)); file.insert(file.end(), hh, hh + 16); }
      else { uint8_t hh[8] = {uint8_t(total >> 24), uint8_t(total >> 16), uint8_t(total >> 8), uint8_t(total), 'j', 'x', 'l', 'c'}; file.insert(file.end(), hh, hh + 8); } }
    file.insert(file.end(), head.begin(), head.end()); file.insert(file.end(), lfg_bytes.begin(), lfg_bytes.end());
    for (uint32_t g = 0; g < nlf; g++) if (lf_sec[g]) file.insert(file.end(), lf_sec[g]->data(), lf_sec[g]->data() + lf_sec[g]->size());
    file.insert(file.end(), hfg_bytes.begin(), hfg_bytes.end());
    for (uint32_t g = 0; g < ng; g++) file.insert(file.end(), grp_sec[g]->data(), grp_sec[g]->data() + grp_sec[g]->size());
    return file;
  }
  std::vector<BitWriter> secw(single ? 1 : nsec); auto W = [&](size_t i) -> BitWriter& { return single ? secw[0] : secw[i]; };
  auto append = [&](BitWriter& bw, const BandSection* s) { if (s) AppendBits(bw, s->data(), s->bits); };
  { BitWriter& bw = W(0);
    bw.Bool(true);   // LfChannelDequantization all_default: present for Modular frames too
    if (!lossless) { bw.U32(BitsOffset(11, 1), BitsOffset(11, 2049), BitsOffset(12, 4097), BitsOffset(16, 8193), plan.global_scale); bw.U32(Val(16), BitsOffset(5, 1), BitsOffset(8, 1), BitsOffset(16, 1), plan.quant_lf); bw.Bool(true); bw.Bool(true); }
    bw.Bool(true); WriteCode(bw, plan.tree_code); WriteTokens(bw, plan.tree_code, plan.tree_tokens); WriteCode(bw, codes.mcode);
    if (plan.nplanes > 0) { WriteGroupHeader(bw, plan.gheader); if (plan.global_has_modular) append(bw, global_sec); } }
  for (uint32_t g = 0; g < nlf; g++) { if (lossless) continue; append(W(1 + g), lf_sec[g]); }
  { BitWriter& bw = W(1 + nlf); if (!lossless) { bw.Bool(true); bw.Write(CeilLog2(ng), 0); bw.U32(Val(0x5F), Val(0x13), Val(0), Bits(13), 0); WriteCode(bw, codes.acode); } }
  for (uint32_t g = 0; g < ng; g++) append(W(2 + nlf + g), grp_sec[g]);
  BitWriter cs; cs.Write(16, 0x0AFF); WriteImageHeaders(cs, plan.m); WriteFrameHeader(cs, fh, plan.m);
  std::vector<std::vector<uint8_t>> secs; std::vector<size_t> sizes; for (auto& w : secw) secs.push_back(w.Finish()); for (auto& s : secs) sizes.push_back(s.size());
  WriteToc(cs, sizes); std::vector<uint8_t> code = cs.Finish(); for (auto& s : secs) code.insert(code.end(), s.begin(), s.end());
  // container always (JxlEncoderUseBoxes, N/Encoder/JxlEncoder.cpp:201); Exif / xml boxes uncompressed, blobs passed through (:284-310)
  std::vector<uint8_t> file = ContainerPrologue();
  if (meta.exif_size) AppendBox(file, "Exif", meta.exif, meta.exif_size); if (meta.xmp_size) AppendBox(file, "xml ", meta.xmp, meta.xmp_size);
  AppendBox(file, "jxlc", code.data(), code.size());
  return file;
}

EncodeResult EncodeOnGpu(const EncodeRequest& req) {
  EncodeResult res;
  if (!req.bgra) { res.status = EncStatus::NullParameter; return res; }
  try {
    std::string why; if (!CudaAvailable(&why)) { res.status = EncStatus::EncodeError; res.message = why; return res; }
    BandEncoder enc(req);
    const uint32_t flags = enc.Begin();
    const std::vector<uint64_t> hist = enc.Tokenize(flags);
    const std::vector<BandSection> secs = enc.Finish(hist);
    std::vector<const BandSection*> ptrs; for (const BandSection& s : secs) ptrs.push_back(&s);
    res.file = AssembleFile(enc.Plan(), hist, ptrs, req);
    res.pixel_format = enc.Plan().is_gray ? (enc.Plan().has_alpha ? 1 : 0) : (enc.Plan().has_alpha ? 3 : 2); res.times.total = enc.device_ms;
  } catch (const std::bad_alloc&) { res.status = EncStatus::OutOfMemory; }
  catch (const std::exception& ex) { res.status = EncStatus::EncodeError; res.message = ex.what(); }
  return res;
}

// ---- band sessions behind the C ABI (JxlB200BandEncoder*)
struct BandSession { std::unique_ptr<BandEncoder> enc; std::vector<uint8_t> icc, exif, xmp; EncodeRequest req; };

static std::vector<uint8_t> SerializeSections(const std::vector<BandSection>& secs) {
  std::vector<uint8_t> out; auto put = [&](const void* p, size_t n) { const uint8_t* b = static_cast<const uint8_t*>(p); out.insert(out.end(), b, b + n); };
  const uint32_t magic = 0x4253584a, count = uint32_t(secs.size()); put(&magic, 4); put(&count, 4);
  for (const BandSection& s : secs) { put(&s.kind, 4); put(&s.index, 4); put(&s.bits, 8); const uint64_t nb = s.bytes.size(); put(&nb, 8); put(s.bytes.data(), s.bytes.size()); }
  return out;
}
static std::vector<BandSection> ParseSections(const uint8_t* p, size_t n) {
  std::vector<BandSection> out; size_t pos = 0; auto get = [&](void* d, size_t k) { JXLG_CHECK(k <= n - pos, "band sections truncated"); memcpy(d, p + pos, k); pos += k; };
  uint32_t magic = 0, count = 0; get(&magic, 4); get(&count, 4); JXLG_CHECK(magic == 0x4253584a, "band sections: bad magic");
  for (uint32_t i = 0; i < count; i++) { BandSection s; uint64_t nb = 0; get(&s.kind, 4); get(&s.index, 4); get(&s.bits, 8); get(&nb, 8); JXLG_CHECK(nb <= n - pos && s.bits <= nb * 8, "band sections truncated"); s.view = p + pos; s.view_n = size_t(nb); pos += nb; out.push_back(std::move(s)); }   // a view: the blob outlives the assembly
  return out;
}

BandSession* BandEncoderCreate(const EncodeRequest& r, uint32_t* flags, EncStatus* status, std::string* message) {
  std::unique_ptr<BandSession> s(new BandSession); s->req = r;
  try {
    if (r.icc_size) { s->icc.assign(r.icc, r.icc + r.icc_size); s->req.icc = s->icc.data(); }   // the session outlives the call: keep copies of the metadata
    s->req.exif = nullptr; s->req.exif_size = 0; s->req.xmp = nullptr; s->req.xmp_size = 0;
    s->enc.reset(new BandEncoder(s->req)); *flags = s->enc->Begin(); *status = EncStatus::Ok; return s.release();
  } catch (const std::bad_alloc&) { *status = EncStatus::OutOfMemory; } catch (const std::exception& ex) { *status = EncStatus::EncodeError; *message = ex.what(); }
  return nullptr;
}
EncStatus BandEncoderTokenize(BandSession* s, uint32_t frame_flags, std::vector<uint64_t>* hist, std::string* message) {
  try { *hist = s->enc->Tokenize(frame_flags); return EncStatus::Ok; } catch (const std::bad_alloc&) { return EncStatus::OutOfMemory; } catch (const std::exception& ex) { *message = ex.what(); return EncStatus::EncodeError; }
}
EncStatus BandEncoderFinish(BandSession* s, const uint64_t* hist, size_t words, std::vector<uint8_t>* sections, float* device_ms, std::string* message) {
  try { std::vector<uint64_t> h(hist, hist + words); *sections = SerializeSections(s->enc->Finish(h)); if (device_ms) *device_ms = s->enc->device_ms; return EncStatus::Ok; }
  catch (const std::bad_alloc&) { return EncStatus::OutOfMemory; } catch (const std::exception& ex) { *message = ex.what(); return EncStatus::EncodeError; }
}
void BandEncoderDestroy(BandSession* s) { delete s; }
int64_t BandEncoderDebugStage(BandSession* s, int32_t which, void* out, int64_t capacity, int64_t* dims4, std::string* message) {
  try { return s->enc->DebugStage(which, out, capacity, dims4); } catch (const std::exception& ex) { *message = ex.what(); return 0; }
}
EncStatus AssembleBands(const EncodeRequest& frame, uint32_t frame_flags, const uint64_t* hist, size_t words, const uint8_t* const* blobs, const size_t* sizes, size_t count, std::vector<uint8_t>* file, std::string* message) {
  try {
    EncPlan plan = MakePlan(frame.width, frame.height, frame_flags, frame); std::vector<uint64_t> h(hist, hist + words);
    std::vector<std::vector<BandSection>> all; for (size_t i = 0; i < count; i++) all.push_back(ParseSections(blobs[i], sizes[i]));
    std::vector<const BandSection*> ptrs; for (auto& v : all) for (auto& s : v) ptrs.push_back(&s);
    *file = AssembleFile(plan, h, ptrs, frame); return EncStatus::Ok;
  } catch (const std::bad_alloc&) { return EncStatus::OutOfMemory; } catch (const std::exception& ex) { *message = ex.what(); return EncStatus::EncodeError; }
}

}  // namespace jxlgpu
