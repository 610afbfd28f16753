// ORACLE — test infrastructure only (see jxlo_bits.h header). PARITY UNPINNED.
// Reconstruction after entropy decode: HF dequant + chroma-from-luma + LLF-from-LF + inverse
// transforms (A.8 "Dequant", A.9), adaptive LF smoothing (A.8 [M]), gaborish + EPF (A.10 [M]),
// XYB -> linear -> transfer function -> sample type (A.10), and the reference's own output
// decisions: channel count / sample type (N/Decoder/JxlDecoder.cpp:494-556), straight alpha
// (:233), CMYK merge and inversion (:159-215).
#pragma once
#include "jxlo_decoder.h"

namespace jxlo {

inline float AdjustQuantBias(int32_t q, float bias1, float bias3) { if (q == 0) return 0.f; if (q == 1) return bias1; if (q == -1) return -bias1; return float(q) - bias3 / float(q); }

// Dequantises and inverse-transforms every varblock of group g into fs.xyb.
inline void ReconstructGroup(FrameState& fs, uint32_t g, const std::vector<int32_t>* coeffs) {
  const FrameHeader& fh = fs.fh; int gx = int(g % fh.xgroups), gy = int(g / fh.xgroups), cx0 = gx * 32, cy0 = gy * 32;
  int w = std::min(32, fs.xb - cx0), h = std::min(32, fs.yb - cy0);
  float inv_gs = fs.q.InvGlobalScale(); float xm = std::pow(0.8f, float(fh.x_qm_scale) - 2.0f), bm = std::pow(0.8f, float(fh.b_qm_scale) - 2.0f);
  const float* qb = fs.meta.opsin.quant_bias; std::vector<float> blk[3], px;
  for (int by = 0; by < h; by++) for (int bx = 0; bx < w; bx++) {
    size_t o = size_t(cy0 + by) * fs.xb + cx0 + bx; if (!fs.is_first[o]) continue;
    int s = fs.strategy[o], bw = kCoveredX[s], bh = kCoveredY[s]; size_t size = size_t(bw) * bh * 64; int t = kQuantTableOf[s];
    const float* dq = fs.dequant[t].data(); float scale = inv_gs / float(fs.hf_mul[o]);
    size_t tile = size_t((cy0 + by) / 8) * fs.xt + (cx0 + bx) / 8; float kx = fs.cfl.YtoX(fs.ytox[tile]), kb = fs.cfl.YtoB(fs.ytob[tile]);
    for (int c = 0; c < 3; c++) blk[c].assign(size, 0.f);
    for (uint32_t p = 0; p < size; p++) {
      size_t a = CoefAddr(by, bx, bw, p);
      float y = AdjustQuantBias(coeffs[1][a], qb[1], qb[3]) * dq[size + p] * scale;
      float x = AdjustQuantBias(coeffs[0][a], qb[0], qb[3]) * dq[p] * (scale * xm) + kx * y;
      float b = AdjustQuantBias(coeffs[2][a], qb[2], qb[3]) * dq[2 * size + p] * (scale * bm) + kb * y;
      blk[0][p] = x; blk[1][p] = y; blk[2][p] = b;
    }
    for (int c = 0; c < 3; c++) {
      LowestFrequenciesFromDC(s, fs.lf[c].row(cy0 + by) + cx0 + bx, size_t(fs.xb), blk[c].data());
      TransformToPixels(s, blk[c].data(), fs.xyb[c].row((cy0 + by) * 8) + (cx0 + bx) * 8, size_t(fs.xpad));
    }
  }
}

// A.8 adaptive LF smoothing (skipped when flag 128 is set or the LF image is smaller than 3x3)
inline void AdaptiveLfSmoothing(FrameState& fs) {
  int w = fs.xb, h = fs.yb; if (w <= 2 || h <= 2) return;
  const float kW1 = 0.20345139757231578f, kW2 = 0.0334829185968739f, kW0 = 1.0f - 4.0f * (kW1 + kW2);
  float inv = fs.q.InvGlobalScale() / float(fs.q.quant_lf); float fac[3]; for (int c = 0; c < 3; c++) fac[c] = fs.lf_dequant[c] * inv;
  Plane out[3]; for (int c = 0; c < 3; c++) out[c] = fs.lf[c];
  for (int y = 1; y + 1 < h; y++) for (int x = 1; x + 1 < w; x++) {
    float sm[3], gap = 0.5f;
    for (int c = 0; c < 3; c++) { const float* t = fs.lf[c].row(y - 1); const float* m = fs.lf[c].row(y); const float* b = fs.lf[c].row(y + 1);
      float corner = t[x - 1] + t[x + 1] + b[x - 1] + b[x + 1], edge = t[x] + m[x - 1] + m[x + 1] + b[x]; sm[c] = m[x] * kW0 + edge * kW1 + corner * kW2;
      gap = std::max(gap, std::fabs((m[x] - sm[c]) / fac[c])); }
    float factor = std::max(0.f, 3.0f - 4.0f * gap);
    for (int c = 0; c < 3; c++) { float mc = fs.lf[c].row(y)[x]; out[c].row(y)[x] = (sm[c] - mc) * factor + mc; }
  }
  for (int c = 0; c < 3; c++) fs.lf[c] = out[c];
}

inline int Mirror(int x, int n) { while (x < 0 || x >= n) { if (x < 0) x = -x - 1; else x = 2 * n - 1 - x; } return x; }

// planes have stride p.w >= xs; only [0,xs) x [0,ys) is meaningful and filtered.
inline void Gaborish(Plane* xyb, int xs, int ys, const LoopFilter& lf, int threads = 1) {
  for (int c = 0; c < 3; c++) {
    float w1 = lf.gab_w[2 * c], w2 = lf.gab_w[2 * c + 1]; float mul = 1.0f / (1.0f + 4.0f * (w1 + w2)); float wc = mul, we = w1 * mul, wd = w2 * mul;
    Plane out = xyb[c];
    ParallelFor(size_t(ys), threads, [&](size_t yy) { int y = int(yy); const float* t = xyb[c].row(Mirror(y - 1, ys)); const float* m = xyb[c].row(y); const float* b = xyb[c].row(Mirror(y + 1, ys)); float* o = out.row(y);
      for (int x = 0; x < xs; x++) { int xl = Mirror(x - 1, xs), xr = Mirror(x + 1, xs); o[x] = m[x] * wc + (t[x] + b[x] + m[xl] + m[xr]) * we + (t[xl] + t[xr] + b[xl] + b[xr]) * wd; } });
    xyb[c] = std::move(out);
  }
}

static const float kInvSigmaNum = -1.1715728752538099024f;
static const float kMinSigma = -3.90524291751269967465540850526868f;

// inv_sigma per 8x8 cell (A.10 EPF [M]); Modular frames use a constant.
inline std::vector<float> ComputeInvSigma(const FrameState& fs) {
  const LoopFilter& lf = fs.fh.lf; std::vector<float> is(size_t(fs.xb) * fs.yb);
  if (fs.fh.encoding == 1) { std::fill(is.begin(), is.end(), kInvSigmaNum / lf.epf_sigma_for_modular); return is; }
  float quant_scale = float(fs.q.global_scale) / 65536.0f;
  for (size_t i = 0; i < is.size(); i++) {
    float sigma_quant = lf.epf_quant_mul / (quant_scale * float(fs.hf_mul[i]) * kInvSigmaNum);
    float sigma = sigma_quant * lf.epf_sharp_lut[fs.sharp[i]]; sigma = std::min(-1e-4f, sigma); is[i] = 1.0f / sigma;
  }
  return is;
}

// One EPF pass. pass: 0 (12 neighbours, plus-SAD), 1 (4 neighbours, plus-SAD), 2 (4 neighbours, 1-px SAD).
inline void EpfPass(Plane* xyb, int xs, int ys, int xb, const std::vector<float>& inv_sigma, const LoopFilter& lf, int pass, int threads = 1) {
  static const int n12[12][2] = {{-2, 0}, {-1, -1}, {-1, 0}, {-1, 1}, {0, -2}, {0, -1}, {0, 1}, {0, 2}, {1, -1}, {1, 0}, {1, 1}, {2, 0}};   // {dy,dx}
  static const int n4[4][2] = {{-1, 0}, {0, -1}, {0, 1}, {1, 0}};
  static const int plus[5][2] = {{0, 0}, {-1, 0}, {1, 0}, {0, -1}, {0, 1}};
  float sigma_scale = pass == 0 ? lf.epf_pass0_sigma_scale : pass == 2 ? lf.epf_pass2_sigma_scale : 1.0f; float sm = sigma_scale * 1.65f, bsm = sm * lf.epf_border_sad_mul;
  const int (*nb)[2] = pass == 0 ? n12 : n4; int nn = pass == 0 ? 12 : 4;
  Plane out[3] = {xyb[0], xyb[1], xyb[2]};
  ParallelFor(size_t(ys), threads, [&](size_t yy) { const int y = int(yy); for (int x = 0; x < xs; x++) {
    float is = inv_sigma[size_t(y / 8) * xb + x / 8]; if (is < kMinSigma) continue;
    bool border = (y % 8 == 0 || y % 8 == 7 || x % 8 == 0 || x % 8 == 7); float inv = is * (border ? bsm : sm);
    float wsum = 1.0f, acc[3]; for (int c = 0; c < 3; c++) acc[c] = xyb[c].row(y)[x];
    for (int i = 0; i < nn; i++) {
      float sad = 0;
      for (int c = 0; c < 3; c++) { float s = 0;
        if (pass == 2) s = std::fabs(xyb[c].row(Mirror(y + nb[i][0], ys))[Mirror(x + nb[i][1], xs)] - xyb[c].row(y)[x]);
        else for (int k = 0; k < 5; k++) { int yy = y + plus[k][0], xx = x + plus[k][1]; s += std::fabs(xyb[c].row(Mirror(yy + nb[i][0], ys))[Mirror(xx + nb[i][1], xs)] - xyb[c].row(Mirror(yy, ys))[Mirror(xx, xs)]); }
        sad += s * lf.epf_channel_scale[c]; }
      float wgt = std::max(0.f, 1.0f + sad * inv); wsum += wgt;
      for (int c = 0; c < 3; c++) acc[c] += wgt * xyb[c].row(Mirror(y + nb[i][0], ys))[Mirror(x + nb[i][1], xs)];
    }
    float iw = 1.0f / wsum; for (int c = 0; c < 3; c++) out[c].row(y)[x] = acc[c] * iw;
  } });
  for (int c = 0; c < 3; c++) xyb[c] = std::move(out[c]);
}

// ------------------------------------------------------------------ colour
inline void XybToLinear(float X, float Y, float B, const OpsinInverse& o, float itscale, float* rgb) {
  float g[3] = {Y + X, Y - X, B}, m[3];
  for (int c = 0; c < 3; c++) { float cb = std::cbrt(o.bias[c]); float v = g[c] - cb; m[c] = v * v * v + o.bias[c]; }
  for (int c = 0; c < 3; c++) rgb[c] = (o.inv[3 * c] * m[0] + o.inv[3 * c + 1] * m[1] + o.inv[3 * c + 2] * m[2]) * itscale;
}
inline float TfFromLinear(float v, const ColorEncoding& ce, float intensity_target) {
  float a = std::fabs(v), r;
  if (ce.have_gamma) r = std::pow(a, float(ce.gamma) * 1e-7f);
  else switch (ce.tf) {
    case kTfLinear: r = a; break;
    case kTfSRGB: r = a <= 0.0031308f ? 12.92f * a : 1.055f * std::pow(a, 1.0f / 2.4f) - 0.055f; break;
    case kTf709: r = a < 0.018f ? 4.5f * a : 1.099f * std::pow(a, 0.45f) - 0.099f; break;
    case kTfPQ: { const double m1 = 2610.0 / 16384, m2 = 2523.0 / 4096 * 128, c1 = 3424.0 / 4096, c2 = 2413.0 / 4096 * 32, c3 = 2392.0 / 4096 * 32;
      double yv = std::min(1.0, double(a) * intensity_target / 10000.0); double p = std::pow(yv, m1); r = float(std::pow((c1 + c2 * p) / (1 + c3 * p), m2)); break; }
    case kTfDCI: r = std::pow(a, 1.0f / 2.6f); break;
    // ARIB STD-B67 OETF on the nominal range [0, 1] (12 E = the 0..12 scene range); an HLG-tagged file comes back in its own encoding, so no
    // OOTF is involved (display light is only derived when the output encoding differs from the file's, which the reference never asks for)
    case kTfHLG: { const double ha = 0.17883277, hb = 0.28466892, hc = 0.55991073; r = a <= 1.0f / 12 ? float(std::sqrt(3.0 * a)) : float(ha * std::log(12.0 * a - hb) + hc); break; }
    default: throw Error("unsupported transfer function for output");
  }
  return v < 0 ? -r : r;
}
inline void PrimariesXY(const ColorEncoding& ce, double p[3][2], double w[2]) {
  switch (ce.white_point) { case kWpD65: w[0] = 0.3127; w[1] = 0.3290; break; case kWpE: w[0] = w[1] = 1.0 / 3; break; case kWpDCI: w[0] = 0.314; w[1] = 0.351; break; default: w[0] = ce.white_xy[0] * 1e-6; w[1] = ce.white_xy[1] * 1e-6; }
  static const double srgb[3][2] = {{0.639998686, 0.330010138}, {0.300003784, 0.600003357}, {0.150002046, 0.059997204}}, bt2100[3][2] = {{0.708, 0.292}, {0.170, 0.797}, {0.131, 0.046}}, p3[3][2] = {{0.680, 0.320}, {0.265, 0.690}, {0.150, 0.060}};
  const double (*src)[2] = ce.primaries == kPr2100 ? bt2100 : ce.primaries == kPrP3 ? p3 : srgb;
  for (int i = 0; i < 3; i++) for (int k = 0; k < 2; k++) p[i][k] = ce.primaries == kPrCustom ? ce.prim_xy[i][k] * 1e-6 : src[i][k];
}
inline void Inv3x3(const double m[9], double o[9]) {
  double det = m[0] * (m[4] * m[8] - m[5] * m[7]) - m[1] * (m[3] * m[8] - m[5] * m[6]) + m[2] * (m[3] * m[7] - m[4] * m[6]); JXLO_CHECK(std::fabs(det) > 1e-12, "singular colour matrix"); double id = 1 / det;
  o[0] = (m[4] * m[8] - m[5] * m[7]) * id; o[1] = (m[2] * m[7] - m[1] * m[8]) * id; o[2] = (m[1] * m[5] - m[2] * m[4]) * id;
  o[3] = (m[5] * m[6] - m[3] * m[8]) * id; o[4] = (m[0] * m[8] - m[2] * m[6]) * id; o[5] = (m[2] * m[3] - m[0] * m[5]) * id;
  o[6] = (m[3] * m[7] - m[4] * m[6]) * id; o[7] = (m[1] * m[6] - m[0] * m[7]) * id; o[8] = (m[0] * m[4] - m[1] * m[3]) * id;
}
inline void RgbToXyzMatrix(const double p[3][2], const double w[2], double m[9]) {
  double P[9]; for (int i = 0; i < 3; i++) { P[i] = p[i][0] / p[i][1]; P[3 + i] = 1.0; P[6 + i] = (1 - p[i][0] - p[i][1]) / p[i][1]; }
  double W[3] = {w[0] / w[1], 1.0, (1 - w[0] - w[1]) / w[1]}, Pi[9]; Inv3x3(P, Pi); double S[3]; for (int i = 0; i < 3; i++) S[i] = Pi[3 * i] * W[0] + Pi[3 * i + 1] * W[1] + Pi[3 * i + 2] * W[2];
  for (int r = 0; r < 3; r++) for (int c = 0; c < 3; c++) m[3 * r + c] = P[3 * r + c] * S[c];
}
// 3x3 taking linear sRGB (D65) to the linear RGB of `ce` (identity for sRGB primaries + D65)
inline void LinearSrgbToTarget(const ColorEncoding& ce, float out[9]) {
  if (ce.primaries == kPrSRGB && ce.white_point == kWpD65) { for (int i = 0; i < 9; i++) out[i] = (i % 4 == 0) ? 1.f : 0.f; return; }
  ColorEncoding s; double ps[3][2], ws[2], pt[3][2], wt[2], A[9], B[9], Bi[9]; PrimariesXY(s, ps, ws); PrimariesXY(ce, pt, wt); RgbToXyzMatrix(ps, ws, A); RgbToXyzMatrix(pt, wt, B); Inv3x3(B, Bi);
  for (int r = 0; r < 3; r++) for (int c = 0; c < 3; c++) { double v = 0; for (int k = 0; k < 3; k++) v += Bi[3 * r + k] * A[3 * k + c]; out[3 * r + c] = float(v); }
}

inline uint16_t F32ToF16(float f) { return BitWriter::FloatToHalf(f); }
inline float F16ToF32(uint16_t b) { uint32_t sign = b >> 15, e = (b >> 10) & 31, m = b & 1023; float v; if (e == 0) v = std::ldexp(float(m), -24); else if (e == 31) v = m ? NAN : INFINITY; else v = std::ldexp(float(m | 1024), int(e) - 25); return sign ? -v : v; }

// Interprets a Modular integer sample as a float sample of the stream's bit depth (A.7 "To samples").
inline float IntToFloatSample(int32_t v, const BitDepth& bd) {
  if (!bd.float_sample) return float(double(v) / double((uint64_t(1) << bd.bits) - 1));
  if (bd.bits == 32 && bd.exp_bits == 8) { float f; memcpy(&f, &v, 4); return f; }
  int mant_bits = int(bd.bits) - int(bd.exp_bits) - 1; uint32_t u = uint32_t(v); bool sign = (u >> (bd.bits - 1)) & 1; u &= (1u << (bd.bits - 1)) - 1;
  if (u == 0) return sign ? -0.f : 0.f;
  int exp = int(u >> mant_bits); uint32_t mant = u & ((1u << mant_bits) - 1); int bias = (1 << (bd.exp_bits - 1)) - 1; double r;
  if (exp == 0) r = std::ldexp(double(mant), 1 - bias - mant_bits); else r = std::ldexp(double(mant | (1u << mant_bits)), exp - bias - mant_bits);
  return float(sign ? -r : r);
}

enum SampleType { kU8 = 0, kU16 = 1, kF16 = 2, kF32 = 3 };
struct DecodedImage {
  uint32_t width = 0, height = 0; int format = 1; /* DecoderImageFormat: 0 gray 1 rgb 2 cmyk */ int sample_type = kU8; bool has_alpha = false; int num_channels = 3;
  std::vector<uint8_t> pixels;        // what setLayerData receives (after the CMYK merge when format == 2)
  ImageMetadata meta; std::string frame_name; bool is_container = false; std::vector<uint8_t> exif; std::vector<std::vector<uint8_t>> xmp; bool has_exif = false;
  // stage dumps (keep_stages)
  int xpad = 0, ypad = 0; std::vector<float> stage_idct, stage_gab, stage_epf, stage_lf; std::vector<int32_t> stage_coeffs;
  // the HF metadata and LF integers the file carries: quantised LF [3 (X, Y, B)][yb][xb], hf_mul [yb][xb], ytox / ytob [yt][xt], and the
  // quantiser {global_scale, quant_lf, x_qm_scale, b_qm_scale}
  std::vector<int32_t> stage_lfq, stage_hf_mul, stage_ytox, stage_ytob, stage_quant;
};

inline size_t BytesPerSample(int t) { return t == kU8 ? 1 : t == kF32 ? 4 : 2; }

inline void StoreSample(uint8_t* dst, int type, float v) {
  switch (type) {
    case kU8: { float c = std::min(1.f, std::max(0.f, v)) * 255.0f; *dst = uint8_t(std::lrintf(c)); break; }
    case kU16: { float c = std::min(1.f, std::max(0.f, v)) * 65535.0f; uint16_t u = uint16_t(std::lrintf(c)); memcpy(dst, &u, 2); break; }
    case kF16: { uint16_t h = F32ToF16(v); memcpy(dst, &h, 2); break; }
    default: memcpy(dst, &v, 4);
  }
}

}  // namespace jxlo
