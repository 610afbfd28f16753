// ORACLE — test infrastructure only (see jxlo_bits.h header). PARITY UNPINNED.
// Whole-file decode: the oracle's restatement of DecoderReadImage's observable behaviour
// (N/Decoder/JxlDecoder.cpp:796-852) — signature gate, format decisions (:461-561),
// metadata boxes (:687-784), first frame only (:398-400), output buffer layout (:289-323) —
// on top of the codestream restatement in jxlo_decoder.h / jxlo_render.h.
#pragma once
#include "jxlo_render.h"

namespace jxlo {

inline void SetupFrameArrays(FrameState& fs) {
  const FrameHeader& fh = fs.fh; fs.xb = int(fh.xblocks); fs.yb = int(fh.yblocks); fs.xpad = fs.xb * 8; fs.ypad = fs.yb * 8; fs.xt = (fs.xb + 7) / 8; fs.yt = (fs.yb + 7) / 8;
  if (fh.encoding == 0) {
    size_t n = size_t(fs.xb) * fs.yb; for (int c = 0; c < 3; c++) { fs.lfq[c].assign(n, 0); fs.lf[c] = Plane(fs.xb, fs.yb); fs.xyb[c] = Plane(fs.xpad, fs.ypad); }
    fs.strategy.assign(n, 255); fs.is_first.assign(n, 0); fs.hf_mul.assign(n, 1); fs.sharp.assign(n, 0); fs.lf_idx.assign(n, 0); fs.ytox.assign(size_t(fs.xt) * fs.yt, 0); fs.ytob.assign(size_t(fs.xt) * fs.yt, 0);
  }
}

// Decodes one frame whose header starts at br (byte aligned). Leaves reconstructed XYB (VarDCT) in fs.xyb
// and the global modular image (colour for Modular frames, extra channels always) in fs.gimg.
inline void DecodeFrame(FrameState& fs, const uint8_t* data, size_t size, size_t* pos_bytes, const DecodeOptions& opt, DecodedImage* dbg) {
  BitReader br(data + *pos_bytes, size - *pos_bytes);
  fs.fh = ReadFrameHeader(br, fs.meta); const FrameHeader& fh = fs.fh;
  JXLO_CHECK(fh.upsampling == 1, "upsampling is not supported"); JXLO_CHECK(!fh.do_ycbcr, "YCbCr (JPEG-recompressed) frames are not supported");
  fs.toc = ReadToc(br, fh); size_t hdr_bytes = br.pos / 8; fs.frame_data = data + *pos_bytes + hdr_bytes; fs.frame_size = size - *pos_bytes - hdr_bytes;
  JXLO_CHECK(fs.toc.total <= fs.frame_size, "frame data truncated");
  SetupFrameArrays(fs);
  size_t nlf = fh.num_lf_groups, ng = fh.num_groups, np = fh.passes.num_passes; bool single = fs.toc.size.size() == 1;
  SectionReaders sr(&fs);
  { BitReader b = sr.Get(0); DecodeLfGlobal(fs, b); sr.Done(b); }
  auto lf_job = [&](size_t g) { BitReader b = sr.Get(1 + g); DecodeLfGroup(fs, b, uint32_t(g)); sr.Done(b); };
  if (single) lf_job(0); else ParallelFor(nlf, opt.threads, lf_job);
  if (fh.encoding == 0) { for (size_t i = 0; i < fs.strategy.size(); i++) JXLO_CHECK(fs.strategy[i] != 255, "HF metadata does not cover every block"); }
  { BitReader b = sr.Get(1 + nlf); if (fh.encoding == 0) DecodeHfGlobal(fs, b); sr.Done(b); }
  if (fh.encoding == 0 && !(fh.flags & kFlagSkipAdaptiveLfSmoothing)) AdaptiveLfSmoothing(fs);
  if (dbg && opt.keep_stages && fh.encoding == 0) { dbg->stage_lf.clear(); for (int c = 0; c < 3; c++) dbg->stage_lf.insert(dbg->stage_lf.end(), fs.lf[c].d.begin(), fs.lf[c].d.end()); dbg->stage_coeffs.assign(size_t(3) * fs.xpad * fs.ypad, 0);
    dbg->stage_lfq.clear(); for (int c = 0; c < 3; c++) dbg->stage_lfq.insert(dbg->stage_lfq.end(), fs.lfq[c].begin(), fs.lfq[c].end());
    dbg->stage_hf_mul = fs.hf_mul; dbg->stage_ytox.assign(fs.ytox.begin(), fs.ytox.end()); dbg->stage_ytob.assign(fs.ytob.begin(), fs.ytob.end());
    dbg->stage_quant = {int32_t(fs.q.global_scale), int32_t(fs.q.quant_lf), int32_t(fh.x_qm_scale), int32_t(fh.b_qm_scale)}; }
  auto group_job = [&](size_t g) {
    std::vector<int32_t> coeffs[3]; std::vector<uint16_t> nz[3];
    if (fh.encoding == 0) for (auto& c : coeffs) c.assign(256 * 256, 0);
    int gx = int(g % fh.xgroups), gy = int(g / fh.xgroups);
    for (size_t p = 0; p < np; p++) {
      BitReader b = sr.Get(2 + nlf + p * ng + g);
      if (fh.encoding == 0) DecodeAcGroup(fs, b, uint32_t(p), uint32_t(g), coeffs, nz);
      int min_shift = 3, max_shift = 2;   // Passes::GetDownsamplingBracket (A.7 channel distribution)
      for (size_t i = 0;; i++) {
        for (uint32_t j = 0; j < fh.passes.num_ds; j++) if (i == fh.passes.last_pass[j]) min_shift = FloorLog2(fh.passes.downsample[j]);
        if (i + 1 == np) min_shift = 0;
        if (i == p) break;
        max_shift = min_shift - 1;
      }
      DecodeModularGroup(fs, b, gx * int(fh.group_dim), gy * int(fh.group_dim), int(fh.group_dim), int(fh.group_dim), min_shift, max_shift, StreamIdModularGroup(fh, uint32_t(p), uint32_t(g)));
      sr.Done(b);
    }
    if (fh.encoding == 0) {
      ReconstructGroup(fs, uint32_t(g), coeffs);
      if (dbg && opt.keep_stages) { int w = std::min(32, fs.xb - gx * 32), h = std::min(32, fs.yb - gy * 32);
        for (int c = 0; c < 3; c++) for (int by = 0; by < h; by++) for (int bx = 0; bx < w; bx++) for (int k = 0; k < 64; k++)
          dbg->stage_coeffs[size_t(c) * fs.xpad * fs.ypad + (size_t(gy * 32 + by) * fs.xb + gx * 32 + bx) * 64 + k] = coeffs[c][(size_t(by) * 32 + bx) * 64 + k]; }
    }
  };
  if (single) group_job(0); else ParallelFor(ng, opt.threads, group_job);
  *pos_bytes += hdr_bytes + fs.toc.total;
  if (!fs.gimg.ch.empty()) UndoTransforms(fs.gimg, fs.gheader);
}

inline void SkipFrame(const ImageMetadata& meta_in, const uint8_t* data, size_t size, size_t* pos_bytes, bool preview) {
  ImageMetadata m = meta_in; if (preview) { m.xsize = m.preview_x; m.ysize = m.preview_y; }
  BitReader br(data + *pos_bytes, size - *pos_bytes); FrameHeader fh = ReadFrameHeader(br, m); Toc t = ReadToc(br, fh); *pos_bytes += br.pos / 8 + t.total; JXLO_CHECK(*pos_bytes <= size, "frame truncated");
}

struct ImageInfo { int format = 1; int sample_type = kU8; bool has_alpha = false; int num_channels = 3; int status = 0; std::string error; };
enum { kStOk = 0, kStDimExceeds = 6, kStUnsupportedChannel = 7, kStDecodeError = 10 };

// Restates the BASIC_INFO branch of ReadImageInfoAndMetadata (N/Decoder/JxlDecoder.cpp:461-561).
inline ImageInfo DecideFormat(const ImageMetadata& m) {
  ImageInfo r; int alpha = m.alpha_index(); uint32_t alpha_bits = alpha >= 0 ? m.ec[alpha].bd.bits : 0; r.has_alpha = alpha_bits != 0;
  if (m.xsize > 0x7fffffffu || m.ysize > 0x7fffffffu) { r.status = kStDimExceeds; return r; }
  int black = -1; bool first_alpha = false, ok = true;
  for (size_t i = 0; i < m.ec.size() && ok; i++) {
    if (m.ec[i].type == kEcBlack) { if (black < 0) black = int(i); else ok = false; }
    else if (m.ec[i].type == kEcAlpha) { if (r.has_alpha && !first_alpha) first_alpha = true; else ok = false; }
  }
  int cc = m.num_color_channels();
  if (!ok) { r.status = kStUnsupportedChannel; return r; }
  r.num_channels = cc + (r.has_alpha ? 1 : 0); r.format = cc == 1 ? 0 : (black >= 0 ? 2 : 1);
  if (m.bd.exp_bits > 0) {
    if (r.format == 2) { r.status = kStDecodeError; r.error = "Floating point CMYK images are not supported."; return r; }
    if (m.bd.bits <= 16) r.sample_type = kF16; else if (m.bd.bits <= 32) r.sample_type = kF32; else { r.status = kStDecodeError; r.error = "Unsupported floating point bit depth: " + std::to_string(m.bd.bits) + "."; return r; }
  } else if (m.bd.bits > 8) {
    if (m.bd.bits <= 16) { if (r.format == 2) { r.status = kStDecodeError; r.error = "CMYK64 images are not supported."; return r; } r.sample_type = kU16; }
    else { r.status = kStDecodeError; r.error = "Unsupported integer bit depth: " + std::to_string(m.bd.bits) + "."; return r; }
  }
  return r;
}

// KnownColorProfile mapping (N/Decoder/JxlDecoder.cpp:36-108); -1 = not one of the eight enums.
inline int KnownProfileOf(const ColorEncoding& c) {
  if (c.want_icc || c.have_gamma) return -1;
  if (c.color_space == kCsRGB && c.white_point == kWpD65) {
    if (c.tf == kTfLinear) { if (c.primaries == kPrSRGB) return 1; if (c.primaries == kPr2100) return 6; }
    else if (c.tf == kTfSRGB) { if (c.primaries == kPrSRGB) return 0; if (c.primaries == kPrP3) return 4; }
    else if (c.tf == kTf709) { if (c.primaries == kPrSRGB) return 5; }
    else if (c.primaries == kPr2100) { if (c.tf == kTfPQ) return 7; }
  } else if (c.color_space == kCsGray && c.white_point == kWpD65) { if (c.tf == kTfLinear) return 2; if (c.tf == kTfSRGB) return 3; }
  return -1;
}

inline void ApplyOrientation(std::vector<uint8_t>& px, uint32_t* w, uint32_t* h, size_t bpp, uint32_t orientation) {
  if (orientation <= 1) return; uint32_t W = *w, H = *h; bool swap = orientation >= 5; uint32_t ow = swap ? H : W, oh = swap ? W : H; std::vector<uint8_t> out(px.size());
  for (uint32_t y = 0; y < oh; y++) for (uint32_t x = 0; x < ow; x++) {
    uint32_t sx, sy;
    switch (orientation) { case 2: sx = W - 1 - x; sy = y; break; case 3: sx = W - 1 - x; sy = H - 1 - y; break; case 4: sx = x; sy = H - 1 - y; break;
      case 5: sx = y; sy = x; break; case 6: sx = y; sy = H - 1 - x; break; case 7: sx = W - 1 - y; sy = H - 1 - x; break; default: sx = W - 1 - y; sy = x; break; }
    memcpy(&out[(size_t(y) * ow + x) * bpp], &px[(size_t(sy) * W + sx) * bpp], bpp);
  }
  px.swap(out); *w = ow; *h = oh;
}

std::vector<uint8_t> BrotliDecompress(const uint8_t* data, size_t size);   // jxlo_capi.cc (dlopen of the system libbrotlidec)

// Blends one pixel of a new frame (fg) onto the canvas (bg), both R, G, B, alpha in the output encoding; bg receives the result.
// Modes (frame header BlendingInfo): 0 replace, 1 add, 2 blend (alpha compositing, "over"), 3 alpha-weighted add, 4 multiply. The colour
// channels follow `cmode`, the alpha channel itself `amode`. [M]: restated from memory of libjxl's PerformBlending; unpinned.
inline void BlendPixel(uint32_t cmode, uint32_t amode, bool cclamp, bool aclamp, bool premultiplied, bool has_alpha, const float* fg, float* bg) {
  const float ba = bg[3]; float fa = fg[3];
  auto clamp01 = [](float v) { return std::min(1.f, std::max(0.f, v)); };
  // alpha channel
  float out_a = ba;
  if (has_alpha) {
    const float fac = aclamp ? clamp01(fa) : fa;
    switch (amode) { case 0: out_a = fa; break; case 1: out_a = ba + fa; break; case 2: out_a = 1.f - (1.f - fac) * (1.f - ba); break; case 3: out_a = ba; break; default: out_a = ba * fac; break; }
  }
  // colour channels
  const float fac = cclamp ? clamp01(fa) : fa;
  for (int c = 0; c < 3; c++) {
    const float f = fg[c], b = bg[c]; float o;
    switch (cmode) {
      case 0: o = f; break;
      case 1: o = b + f; break;
      case 2:
        if (premultiplied) o = f + b * (1.f - fac);
        else { const float na = 1.f - (1.f - fac) * (1.f - ba); const float rna = na > 0.f ? 1.f / na : 0.f; o = (f * fac + b * ba * (1.f - fac)) * rna; }
        break;
      case 3: o = b + f * fac; break;
      default: o = b * (cclamp ? clamp01(f) : f); break;
    }
    bg[c] = o;
  }
  bg[3] = has_alpha ? out_a : 1.f;
}

inline DecodedImage DecodeImage(const uint8_t* data, size_t size, const DecodeOptions& opt) {
  DecodedImage out; ContainerInfo ci = ParseContainer(data, size); out.is_container = ci.is_container;
  const std::vector<uint8_t>& cs = ci.codestream; JXLO_CHECK(cs.size() >= 2 && cs[0] == 0xFF && cs[1] == 0x0A, "codestream signature");
  BitReader hb(cs.data() + 2, cs.size() - 2); FrameState fs; fs.meta = ReadImageHeaders(hb); out.meta = fs.meta; const ImageMetadata& m = fs.meta;
  // metadata boxes (first Exif only, every xml box; brob decompressed) — N/Decoder/JxlDecoder.cpp:687-784
  for (const Box& b : ci.boxes) {
    const uint8_t* p = b.data; size_t n = b.size; char type[5]; memcpy(type, b.type, 5); std::vector<uint8_t> tmp;
    if (!strcmp(type, "brob") && n >= 4) { memcpy(type, p, 4); type[4] = 0; if (!strcmp(type, "Exif") || !strcmp(type, "xml ")) { tmp = BrotliDecompress(p + 4, n - 4); p = tmp.data(); n = tmp.size(); } }
    if (!strcmp(type, "Exif")) { if (!out.has_exif) { out.has_exif = true; out.exif.assign(p, p + n); } } else if (!strcmp(type, "xml ")) out.xmp.emplace_back(p, p + n);
  }
  ImageInfo info = DecideFormat(m); JXLO_CHECK(info.status == kStOk, info.error.empty() ? "unsupported channel format" : info.error);
  out.format = info.format; out.sample_type = info.sample_type; out.has_alpha = info.has_alpha; out.num_channels = info.num_channels;
  size_t pos = 2 + hb.pos / 8;
  if (m.have_preview) SkipFrame(m, cs.data(), cs.size(), &pos, true);
  const int alpha = info.has_alpha ? m.alpha_index() : -1, black = m.black_index(); const bool premul = alpha >= 0 && m.ec[alpha].alpha_associated;
  const int C = info.num_channels, cc = m.num_color_channels(); const size_t bps = BytesPerSample(info.sample_type); size_t bpp = bps * C;
  // output colour transform (Appendix C-1: default output encoding of a freshly reset decoder)
  bool to_target = m.xyb_encoded && !m.ce.want_icc; ColorEncoding target = to_target ? m.ce : ColorEncoding(); if (m.xyb_encoded && m.ce.want_icc && m.ce.color_space == kCsGray) target.color_space = kCsGray;
  if (to_target && !target.have_gamma && target.tf == kTfUnknown) { target = ColorEncoding(); target.color_space = m.ce.color_space; }
  float mat[9]; LinearSrgbToTarget(target, mat); const float itscale = 255.0f / m.tm.intensity_target;

  // One decoded frame as float samples in the output encoding: [ys][xs][4] = R, G, B (gray replicated), alpha (1 when the image has none);
  // black: the K channel as 8-bit samples (CMYK, single-frame files only).
  struct FrameSamples { int xs = 0, ys = 0; std::vector<float> px; std::vector<uint8_t> black; };
  auto render_frame = [&](FrameSamples* fsm) {
    const FrameHeader& fh = fs.fh; const int xs = int(fh.xsize), ys = int(fh.ysize); const LoopFilter& lf = fh.lf;
    Plane col[3]; int ncol = 3;
    if (fh.encoding == 0) { for (int c = 0; c < 3; c++) col[c] = std::move(fs.xyb[c]); }
    else {
      JXLO_CHECK(!m.xyb_encoded, "XYB-encoded Modular frames are not supported");
      ncol = (m.ce.color_space == kCsGray) ? 1 : 3;
      for (int c = 0; c < ncol; c++) { const Channel& ch = fs.gimg.ch[c]; JXLO_CHECK(ch.w == xs && ch.h == ys, "modular colour channel size"); col[c] = Plane(xs, ys); for (size_t i = 0; i < ch.d.size(); i++) col[c].d[i] = IntToFloatSample(ch.d[i], m.bd); }
    }
    bool filters = (fh.encoding == 0) || (ncol == 3 && (lf.gab || lf.epf_iters));
    if (opt.keep_stages && fh.encoding == 0) { out.xpad = fs.xpad; out.ypad = fs.ypad; for (int c = 0; c < 3; c++) out.stage_idct.insert(out.stage_idct.end(), col[c].d.begin(), col[c].d.end()); }
    if (filters) {
      JXLO_CHECK(ncol == 3, "restoration filters on a single-channel frame are not supported");
      if (lf.gab) Gaborish(col, xs, ys, lf, opt.threads);
      if (opt.keep_stages && fh.encoding == 0) for (int c = 0; c < 3; c++) out.stage_gab.insert(out.stage_gab.end(), col[c].d.begin(), col[c].d.end());
      if (lf.epf_iters) { if (fh.encoding == 1) { fs.xb = (xs + 7) / 8; fs.yb = (ys + 7) / 8; } std::vector<float> is = ComputeInvSigma(fs);
        if (lf.epf_iters == 3) EpfPass(col, xs, ys, fs.xb, is, lf, 0, opt.threads); EpfPass(col, xs, ys, fs.xb, is, lf, 1, opt.threads); if (lf.epf_iters >= 2) EpfPass(col, xs, ys, fs.xb, is, lf, 2, opt.threads); }
      if (opt.keep_stages && fh.encoding == 0) for (int c = 0; c < 3; c++) out.stage_epf.insert(out.stage_epf.end(), col[c].d.begin(), col[c].d.end());
    }
    const size_t ec_base = fh.encoding == 1 ? size_t(ncol) : 0;
    auto ec_sample = [&](int ec, int x, int y) -> float { const Channel& ch = fs.gimg.ch[ec_base + ec]; int s = int(m.ec[ec].dim_shift); return IntToFloatSample(ch.row(std::min(y >> s, ch.h - 1))[std::min(x >> s, ch.w - 1)], m.ec[ec].bd); };
    fsm->xs = xs; fsm->ys = ys; fsm->px.assign(size_t(xs) * ys * 4, 0.f); if (info.format == 2) fsm->black.assign(size_t(xs) * ys, 0);
    ParallelFor(size_t(ys), opt.threads, [&](size_t yy) {
      const int y = int(yy); float* dst = fsm->px.data() + size_t(y) * xs * 4;
      for (int x = 0; x < xs; x++, dst += 4) {
        if (m.xyb_encoded) {
          float lin[3]; XybToLinear(col[0].row(y)[x], col[1].row(y)[x], col[2].row(y)[x], m.opsin, itscale, lin);
          for (int c = 0; c < 3; c++) dst[c] = TfFromLinear(mat[3 * c] * lin[0] + mat[3 * c + 1] * lin[1] + mat[3 * c + 2] * lin[2], target, m.tm.intensity_target);
        } else for (int c = 0; c < 3; c++) dst[c] = col[std::min(c, ncol - 1)].row(y)[x];
        dst[3] = alpha >= 0 ? ec_sample(alpha, x, y) : 1.0f;
        if (info.format == 2) StoreSample(&fsm->black[size_t(y) * xs + x], kU8, ec_sample(black, x, y));
      }
    });
  };
  // Float samples -> what setLayerData receives: unpremultiply (JxlDecoderSetUnpremultiplyAlpha, N/Decoder/JxlDecoder.cpp:233), sample
  // type, CMYK merge (:159-215), orientation.
  auto finalize = [&](const FrameSamples& f) {
    const int xs = f.xs, ys = f.ys; out.width = uint32_t(xs); out.height = uint32_t(ys); out.pixels.assign(size_t(xs) * ys * bpp, 0);
    ParallelFor(size_t(ys), opt.threads, [&](size_t yy) {
      const int y = int(yy); uint8_t* dst = out.pixels.data() + size_t(y) * xs * bpp; const float* src = f.px.data() + size_t(y) * xs * 4;
      for (int x = 0; x < xs; x++, src += 4, dst += bpp) {
        float rgb[3] = {src[0], src[1], src[2]}; const float a = src[3];
        if (premul) { float mul = 1.0f / std::max(1.0f / float(1u << 26), a); for (float& v : rgb) v *= mul; }
        for (int c = 0; c < cc; c++) StoreSample(dst + bps * c, info.sample_type, rgb[c]);
        if (alpha >= 0) StoreSample(dst + bps * cc, info.sample_type, a);
      }
    });
    if (info.format == 2) {   // SetCmykImageDataUInt8, N/Decoder/JxlDecoder.cpp:159-215
      int tc = 4 + (info.has_alpha ? 1 : 0); std::vector<uint8_t> merged(size_t(xs) * ys * tc);
      for (size_t i = 0; i < size_t(xs) * ys; i++) { const uint8_t* sp = &out.pixels[i * C]; uint8_t* d = &merged[i * tc]; d[0] = uint8_t(0xff - sp[0]); d[1] = uint8_t(0xff - sp[1]); d[2] = uint8_t(0xff - sp[2]); d[3] = uint8_t(0xff - f.black[i]); if (info.has_alpha) d[4] = sp[3]; }
      out.pixels.swap(merged); bpp = size_t(tc);
    }
    if (m.orientation > 1) ApplyOrientation(out.pixels, &out.width, &out.height, bpp, m.orientation);
  };

  // ---- frames. The reference takes the first JXL_DEC_FULL_IMAGE of a coalescing decoder (N/Decoder/JxlDecoder.cpp:252-400): zero-duration
  // frames are layers that are blended onto the canvas / a reference slot until the first frame that is shown (is_last, or a duration > 0).
  struct Slot { bool valid = false; std::vector<float> px; };   // canvas-sized [H][W][4]
  Slot slots[4]; const int W = int(m.xsize), H = int(m.ysize); bool first = true;
  for (;;) {
    BitReader peek(cs.data() + pos, cs.size() - pos); FrameHeader ph = ReadFrameHeader(peek, m);
    JXLO_CHECK(ph.frame_type != kFrameLF, "LF frames are not supported");
    JXLO_CHECK(!(ph.flags & (kFlagPatches | kFlagSplines | kFlagNoise)), "patches/splines/noise are not supported");
    if (ph.frame_type == kFrameReferenceOnly && ph.save_before_ct) { SkipFrame(m, cs.data(), cs.size(), &pos, false); continue; }   // only patches could use it
    const bool shown = ph.frame_type != kFrameReferenceOnly && (ph.is_last || ph.duration > 0);
    const bool full = !ph.have_crop || (ph.x0 == 0 && ph.y0 == 0 && ph.width == m.xsize && ph.height == m.ysize);
    DecodeFrame(fs, cs.data(), cs.size(), &pos, opt, &out); const FrameHeader& fh = fs.fh; FrameSamples frame; render_frame(&frame);
    if (first && shown && full && fh.blending.mode == 0) { out.frame_name = fh.name; finalize(frame); return out; }   // the plain single-frame file
    first = false;
    JXLO_CHECK(info.format != 2, "multi-frame CMYK images are not supported");
    // blend onto the source slot
    const BlendingInfo& cb = fh.blending; const BlendingInfo ab = alpha >= 0 ? fh.ec_blending[alpha] : BlendingInfo();
    JXLO_CHECK(!(cb.mode == 2 || cb.mode == 3) || (alpha >= 0 && int(cb.alpha_channel) == alpha), "blending needs the image's alpha channel");
    const bool is_ref_only = fh.frame_type == kFrameReferenceOnly;
    std::vector<float> canvas;
    if (is_ref_only) { canvas.assign(size_t(W) * H * 4, 0.f); }
    else { const Slot& src = slots[cb.source]; if (src.valid) canvas = src.px; else canvas.assign(size_t(W) * H * 4, 0.f); }
    if (alpha >= 0 && !is_ref_only && ab.source != cb.source) { const Slot& as = slots[ab.source]; for (size_t i = 0; i < size_t(W) * H; i++) canvas[i * 4 + 3] = as.valid ? as.px[i * 4 + 3] : 0.f; }
    const int x0 = is_ref_only ? 0 : fh.x0, y0 = is_ref_only ? 0 : fh.y0;
    for (int y = 0; y < frame.ys; y++) { const int cy = y + y0; if (cy < 0 || cy >= H) continue;
      for (int x = 0; x < frame.xs; x++) { const int cx = x + x0; if (cx < 0 || cx >= W) continue;
        const float* fg = &frame.px[(size_t(y) * frame.xs + x) * 4]; float* bg = &canvas[(size_t(cy) * W + cx) * 4];
        BlendPixel(is_ref_only ? 0 : cb.mode, is_ref_only ? 0 : ab.mode, cb.clamp, ab.clamp, premul, alpha >= 0, fg, bg); } }
    const bool can_ref = is_ref_only || (!fh.is_last && (fh.duration == 0 || fh.save_as_reference != 0));
    if (shown) { out.frame_name = fh.name; FrameSamples whole; whole.xs = W; whole.ys = H; whole.px.swap(canvas); finalize(whole); return out; }
    if (can_ref) { slots[fh.save_as_reference].valid = true; slots[fh.save_as_reference].px.swap(canvas); }
  }
}

}  // namespace jxlo
