// ORACLE — test infrastructure only (see jxlo_bits.h header). PARITY UNPINNED.
// C API over the oracle for ctypes (tests/, __graft_entry__.smoke(), bench.py cpu_baseline).
#include "jxlo_encoder.h"
#include "jxlo_icc.h"
#include <dlfcn.h>

namespace jxlo {
std::vector<uint8_t> BrotliDecompress(const uint8_t* data, size_t size) {
  typedef int (*Fn)(size_t, const uint8_t*, size_t*, uint8_t*);
  static Fn fn = []() -> Fn { void* h = dlopen("libbrotlidec.so.1", RTLD_NOW); return h ? reinterpret_cast<Fn>(dlsym(h, "BrotliDecoderDecompress")) : nullptr; }();
  JXLO_CHECK(fn != nullptr, "brob box: libbrotlidec.so.1 not available");
  for (size_t cap = std::max<size_t>(size * 8, 1 << 16); cap <= (size_t(1) << 31); cap *= 4) {
    std::vector<uint8_t> out(cap); size_t n = cap; if (fn(size, data, &n, out.data()) == 1) { out.resize(n); return out; }
  }
  throw Error("brob box: brotli stream invalid or too large");
}
}  // namespace jxlo

using namespace jxlo;

extern "C" {

struct jxlo_encode_params {
  float distance; int32_t effort; int32_t lossless; int32_t gab; int32_t epf; int32_t varblocks; int32_t cfl; int32_t adaptive_quant; int32_t force_strategy;
  int32_t use_prefix; int32_t container; int32_t modular_group_shift; int32_t orientation; int32_t skip_lf_smoothing; int32_t threads;
  int32_t bits; int32_t exp_bits; int32_t color_space; int32_t white_point; int32_t primaries; int32_t tf; int32_t intent; float intensity_target; int32_t premultiplied; int32_t black_channel; int32_t num_passes; int32_t pass_shift; float varblock_scale; int32_t varblock_pattern;
  int32_t canvas_w, canvas_h, crop_x0, crop_y0, blend_mode, alpha_blend_mode, blend_source, blend_clamp, is_last, save_as_reference, frame_only;
};

static thread_local std::vector<uint8_t> g_next_icc;
static void SetErr(char* err, size_t n, const char* msg) { if (err && n) { strncpy(err, msg, n - 1); err[n - 1] = 0; } }

void jxlo_default_params(jxlo_encode_params* p) {
  EncodeParams d; memset(p, 0, sizeof(*p)); p->distance = d.distance; p->effort = d.effort; p->gab = -1; p->epf = -1; p->varblocks = -1; p->cfl = -1; p->adaptive_quant = -1; p->force_strategy = -1;
  p->container = 1; p->modular_group_shift = 1; p->orientation = 1; p->threads = 1; p->bits = 8; p->color_space = 0; p->white_point = 1; p->primaries = 1; p->tf = 13; p->intent = 1; p->intensity_target = 255.f; p->num_passes = 1; p->pass_shift = 1; p->varblock_scale = 1.0f; p->is_last = 1;
}

// pixels: interleaved u8 (is_float=0) or f32 (is_float=1) with num_color + alpha (+black before alpha) channels
int jxlo_encode(const void* pixels, int is_float, uint32_t width, uint32_t height, int num_color, int has_alpha, const jxlo_encode_params* cp,
                const uint8_t* exif, size_t exif_size, const uint8_t* xmp, size_t xmp_size, uint8_t** out, size_t* out_size, char* err, size_t errlen) {
  try {
    EncodeParams p; p.distance = cp->distance; p.effort = cp->effort; p.lossless = cp->lossless != 0; p.gab = cp->gab; p.epf = cp->epf; p.varblocks = cp->varblocks; p.cfl = cp->cfl; p.adaptive_quant = cp->adaptive_quant;
    p.force_strategy = cp->force_strategy; p.use_prefix = cp->use_prefix != 0; p.container = cp->container != 0; p.modular_group_shift = cp->modular_group_shift; p.orientation = uint32_t(cp->orientation); p.skip_lf_smoothing = cp->skip_lf_smoothing != 0;
    p.threads = cp->threads; p.bd.bits = uint32_t(cp->bits); p.bd.exp_bits = uint32_t(cp->exp_bits); p.bd.float_sample = cp->exp_bits > 0; p.ce.color_space = uint32_t(cp->color_space); p.ce.white_point = uint32_t(cp->white_point);
    p.ce.primaries = uint32_t(cp->primaries); p.ce.tf = uint32_t(cp->tf); p.ce.intent = uint32_t(cp->intent); p.intensity_target = cp->intensity_target; p.premultiplied = cp->premultiplied != 0; p.black_channel = cp->black_channel != 0; p.num_passes = cp->num_passes; p.pass_shift = cp->pass_shift; p.varblock_scale = cp->varblock_scale; p.varblock_pattern = cp->varblock_pattern;
    p.canvas_w = uint32_t(cp->canvas_w); p.canvas_h = uint32_t(cp->canvas_h); p.crop_x0 = cp->crop_x0; p.crop_y0 = cp->crop_y0; p.blend_mode = uint32_t(cp->blend_mode); p.alpha_blend_mode = uint32_t(cp->alpha_blend_mode);
    p.blend_source = uint32_t(cp->blend_source); p.blend_clamp = cp->blend_clamp != 0; p.is_last = cp->is_last != 0; p.save_as_reference = uint32_t(cp->save_as_reference); p.frame_only = cp->frame_only != 0;
    EncodeInput in; in.width = width; in.height = height; in.num_color = num_color; in.has_alpha = has_alpha != 0; if (is_float) in.f32 = static_cast<const float*>(pixels); else in.u8 = static_cast<const uint8_t*>(pixels);
    in.exif = exif; in.exif_size = exif_size; in.xmp = xmp; in.xmp_size = xmp_size;
    std::vector<uint8_t> icc; icc.swap(g_next_icc); in.icc = icc.data(); in.icc_size = icc.size();
    std::vector<uint8_t> v = EncodeImage(in, p); *out = static_cast<uint8_t*>(malloc(v.size() ? v.size() : 1)); memcpy(*out, v.data(), v.size()); *out_size = v.size(); return 0;
  } catch (const std::exception& e) { SetErr(err, errlen, e.what()); return 1; }
}
void jxlo_free(void* p) { free(p); }
void jxlo_last_encode_strategy_cells(int64_t* out27) { memcpy(out27, LastEncodeStrategyCells(), 27 * sizeof(int64_t)); }
// ICC profile attached to the NEXT jxlo_encode call of this thread (keeps jxlo_encode's signature stable); cleared by that call.
void jxlo_set_next_icc(const uint8_t* icc, size_t n) { g_next_icc.assign(icc, icc + n); }
// ICC stream codec alone (bit stream as it sits in the codestream after ImageMetadata)
int jxlo_icc_stream_write(const uint8_t* icc, size_t n, uint8_t** out, size_t* out_size, char* err, size_t errlen) {
  try { BitWriter bw; WriteIccStream(bw, std::vector<uint8_t>(icc, icc + n)); std::vector<uint8_t> b = bw.Finish(); *out = static_cast<uint8_t*>(malloc(b.size() ? b.size() : 1)); memcpy(*out, b.data(), b.size()); *out_size = b.size(); return 0; }
  catch (const std::exception& e) { SetErr(err, errlen, e.what()); return 1; }
}
int jxlo_icc_stream_read(const uint8_t* data, size_t n, uint8_t** out, size_t* out_size, char* err, size_t errlen) {
  try { BitReader br(data, n); std::vector<uint8_t> v = ReadIccStream(br); JXLO_CHECK(!br.overrun, "ICC stream truncated"); *out = static_cast<uint8_t*>(malloc(v.size() ? v.size() : 1)); memcpy(*out, v.data(), v.size()); *out_size = v.size(); return 0; }
  catch (const std::exception& e) { SetErr(err, errlen, e.what()); return 1; }
}
// Replays a hand-written predicted-ICC byte string (commands + data) through the predictor only: lets the tests exercise every command.
int jxlo_icc_unpredict(const uint8_t* enc, size_t n, uint8_t** out, size_t* out_size, char* err, size_t errlen) {
  try { std::vector<uint8_t> v = UnpredictIcc(std::vector<uint8_t>(enc, enc + n)); *out = static_cast<uint8_t*>(malloc(v.size() ? v.size() : 1)); memcpy(*out, v.data(), v.size()); *out_size = v.size(); return 0; }
  catch (const std::exception& e) { SetErr(err, errlen, e.what()); return 1; }
}

struct jxlo_image { DecodedImage img; };

int jxlo_decode(const uint8_t* data, size_t size, int threads, int keep_stages, jxlo_image** out, char* err, size_t errlen) {
  try { DecodeOptions o; o.threads = threads; o.keep_stages = keep_stages != 0; jxlo_image* r = new jxlo_image; r->img = DecodeImage(data, size, o); *out = r; return 0; }
  catch (const std::exception& e) { SetErr(err, errlen, e.what()); return 1; }
}
void jxlo_image_free(jxlo_image* i) { delete i; }
// info: width,height,format,sample_type,has_alpha,num_channels,xpad,ypad,known_profile,orientation,is_container,has_exif,num_xmp,bits,exp_bits,xyb
void jxlo_image_info(const jxlo_image* i, int32_t* info) {
  const DecodedImage& d = i->img; info[0] = int32_t(d.width); info[1] = int32_t(d.height); info[2] = d.format; info[3] = d.sample_type; info[4] = d.has_alpha; info[5] = d.num_channels; info[6] = d.xpad; info[7] = d.ypad;
  info[8] = KnownProfileOf(d.meta.ce); info[9] = int32_t(d.meta.orientation); info[10] = d.is_container; info[11] = d.has_exif; info[12] = int32_t(d.xmp.size()); info[13] = int32_t(d.meta.bd.bits); info[14] = int32_t(d.meta.bd.exp_bits); info[15] = d.meta.xyb_encoded;
}
const uint8_t* jxlo_image_pixels(const jxlo_image* i, size_t* n) { *n = i->img.pixels.size(); return i->img.pixels.data(); }
const char* jxlo_image_name(const jxlo_image* i, size_t* n) { *n = i->img.frame_name.size(); return i->img.frame_name.data(); }
const uint8_t* jxlo_image_icc(const jxlo_image* i, size_t* n) { *n = i->img.meta.icc.size(); return i->img.meta.icc.data(); }
const uint8_t* jxlo_image_exif(const jxlo_image* i, size_t* n) { *n = i->img.exif.size(); return i->img.exif.data(); }
const uint8_t* jxlo_image_xmp(const jxlo_image* i, int k, size_t* n) { *n = i->img.xmp[k].size(); return i->img.xmp[k].data(); }
// which: 0 idct, 1 gab, 2 epf (3 planes xpad*ypad floats), 3 lf (3 planes xb*yb); returns element count
size_t jxlo_image_stage_f32(const jxlo_image* i, int which, const float** p) { const std::vector<float>& v = which == 0 ? i->img.stage_idct : which == 1 ? i->img.stage_gab : which == 2 ? i->img.stage_epf : i->img.stage_lf; *p = v.data(); return v.size(); }
// which: 0 quantised LF (3 planes xb*yb, channel order X, Y, B), 1 hf_mul (xb*yb), 2 ytox, 3 ytob (xt*yt), 4 quantiser {global_scale, quant_lf,
// x_qm_scale, b_qm_scale}; returns element count
size_t jxlo_image_stage_i32(const jxlo_image* i, int which, const int32_t** p) {
  const DecodedImage& d = i->img; const std::vector<int32_t>& v = which == 0 ? d.stage_lfq : which == 1 ? d.stage_hf_mul : which == 2 ? d.stage_ytox : which == 3 ? d.stage_ytob : d.stage_quant;
  *p = v.data(); return v.size();
}
size_t jxlo_image_stage_coeffs(const jxlo_image* i, const int32_t** p) { *p = i->img.stage_coeffs.data(); return i->img.stage_coeffs.size(); }

int jxlo_signature_check(const uint8_t* d, size_t n) { return SignatureCheck(d, n); }

// ---- stage-level entry points for kernel parity tests
void jxlo_transform_to_pixels(int strategy, const float* coef, float* px, size_t stride) { TransformToPixels(strategy, coef, px, stride); }
void jxlo_transform_from_pixels(int strategy, const float* px, size_t stride, float* coef) { TransformFromPixels(strategy, px, stride, coef); }
void jxlo_llf_from_dc(int strategy, const float* dc, size_t dc_stride, float* block) { LowestFrequenciesFromDC(strategy, dc, dc_stride, block); }
size_t jxlo_dequant_table(int table, float* out) { std::vector<float> t = ComputeDequantTable(table, LibraryEncoding(table)); if (out) memcpy(out, t.data(), t.size() * sizeof(float)); return t.size(); }
size_t jxlo_natural_order(int order_id, uint32_t* out) { int s = kOrderStrategy[order_id]; std::vector<uint32_t> o = NaturalOrder(std::min(kCoveredX[s], kCoveredY[s]), std::max(kCoveredX[s], kCoveredY[s])); if (out) memcpy(out, o.data(), o.size() * 4); return o.size(); }
void jxlo_xyb_to_srgb8(const float* x, const float* y, const float* b, size_t n, uint8_t* rgb) {
  OpsinInverse o; ColorEncoding ce; for (size_t i = 0; i < n; i++) { float lin[3]; XybToLinear(x[i], y[i], b[i], o, 1.0f, lin); for (int c = 0; c < 3; c++) StoreSample(rgb + 3 * i + c, kU8, TfFromLinear(lin[c], ce, 255.f)); }
}
void jxlo_srgb8_to_xyb(const uint8_t* rgb, size_t n, float* x, float* y, float* b) {
  for (size_t i = 0; i < n; i++) { float lin[3], o[3]; for (int c = 0; c < 3; c++) lin[c] = SrgbToLinear(rgb[3 * i + c] * (1.0f / 255.0f)); LinearToXyb(lin, o); x[i] = o[0]; y[i] = o[1]; b[i] = o[2]; }
}

}  // extern "C"
