// pdn-jpegxl_b200 engine — encode kernels (sm_100a) behind SaveImage, low-effort pipeline:
//   k_enc_scan        BGRA scan: isGray / hasTransparency            (N/Encoder/JxlEncoder.cpp:33-77), 4 B/px read
//   k_enc_to_xyb      BGRA -> linear -> XYB planes (+ alpha plane)    (BgraTo* of N/Encoder/PixelFormatConversion.cpp:16-121 fused in), 4 + 12 B/px
//   k_enc_to_planes   BGRA -> integer planes + YCgCo RCT (lossless)
//   k_enc_sharpen     Van Cittert step of the inverse gaborish
//   k_enc_dct8        forward DCT8 + quantise + LF extraction          (SURVEY.md A.9/A.11), 12 + 6 B/px
//   k_enc_lf_quant    LF quantisation with chroma-from-luma
//   k_enc_mod_tokens  Modular tokenisation (gradient predictor, fixed MA tree), one thread per sample
//   k_enc_ac_tokens   AC tokenisation with the A.8 context model, one thread per 256x256 group
//   k_enc_histogram   token histograms; k_enc_ans: ANS stream writer, one thread per section stream
// Replaces the libjxl work behind JxlEncoderAddImageFrame / JxlEncoderFlushInput (N/Encoder/JxlEncoder.cpp:128,367).
#include "enc_frame.cuh"
#include "kernels.h"

namespace jxlgpu {

__device__ __constant__ float kSrgbLut[256];
void UploadSrgbLut(const float* lut) { CUDA_OK(cudaMemcpyToSymbol(kSrgbLut, lut, 256 * sizeof(float))); }

__global__ void k_enc_scan(const uint8_t* __restrict__ bgra, uint32_t w, uint32_t h, uint32_t stride, uint32_t* flags) {
  uint32_t x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y; uint32_t f = 0;
  if (x < w && y < h) { uchar4 p = *reinterpret_cast<const uchar4*>(bgra + size_t(y) * stride + size_t(x) * 4); if (!(p.z == p.y && p.y == p.x)) f |= 1; if (p.w < 255) f |= 2; }
  f = __reduce_or_sync(0xffffffffu, f); if ((threadIdx.x & 31) == 0 && f) atomicOr(flags, f);
}

__global__ void k_enc_to_xyb(const DEncFrame* ep, const uint8_t* __restrict__ bgra) {
  // yy counts rows of the extended plane (halo rows first); `bgra` points at the first row of the band itself, halo rows lie before it
  const DEncFrame& e = *ep; int xx = blockIdx.x * blockDim.x + threadIdx.x, ye = blockIdx.y * blockDim.y + threadIdx.y; if (xx >= int(e.xpad) || ye >= int(e.ext_rows)) return;
  const int yy = ye - int(e.ext_top);
  int x = min(xx, int(e.xsize) - 1), y = max(e.src_row_min, min(yy, e.src_row_max)); uchar4 p = *reinterpret_cast<const uchar4*>(bgra + ptrdiff_t(y) * ptrdiff_t(e.stride) + size_t(x) * 4);
  float r, g, b;
  if (e.has_src_profile) {   // matrix/TRC ICC source: tone curves from the profile, then its colorants -> linear sRGB (what libjxl's CMS step does)
    const float lr = e.src_lut[p.z], lg = e.src_lut[256 + p.y], lb = e.src_lut[512 + p.x]; const float* m = e.src_matrix;
    r = m[0] * lr + m[1] * lg + m[2] * lb; g = m[3] * lr + m[4] * lg + m[5] * lb; b = m[6] * lr + m[7] * lg + m[8] * lb;
  } else { r = kSrgbLut[e.gray ? p.x : p.z]; g = kSrgbLut[e.gray ? p.x : p.y]; b = kSrgbLut[p.x]; }   // gray takes the B channel (N/Encoder/PixelFormatConversion.cpp:34)
  const float bias = 0.0037930732552754493f, cb = cbrtf(bias);
  float m0 = 0.30f * r + 0.622f * g + 0.078f * b + bias, m1 = 0.23f * r + 0.692f * g + 0.078f * b + bias, m2 = 0.24342268924547819f * r + 0.20476744424496821f * g + 0.55180986650955360f * b + bias;
  float g0 = cbrtf(fmaxf(m0, 0.f)) - cb, g1 = cbrtf(fmaxf(m1, 0.f)) - cb, g2 = cbrtf(fmaxf(m2, 0.f)) - cb;
  size_t plane = size_t(e.xpad) * e.ext_rows, at = size_t(ye) * e.xpad + xx; e.xyb[at] = 0.5f * (g0 - g1); e.xyb[plane + at] = 0.5f * (g0 + g1); e.xyb[2 * plane + at] = g2;
  if (e.alpha && xx < int(e.xsize) && yy >= 0 && yy < int(e.ysize)) e.planes[size_t(e.alpha_plane) * e.xsize * e.ysize + size_t(yy) * e.xsize + xx] = p.w;
}

__global__ void k_enc_to_planes(const DEncFrame* ep, const uint8_t* __restrict__ bgra) {
  const DEncFrame& e = *ep; int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y; if (x >= int(e.xsize) || y >= int(e.ysize)) return;
  uchar4 p = *reinterpret_cast<const uchar4*>(bgra + size_t(y) * e.stride + size_t(x) * 4); size_t n = size_t(e.xsize) * e.ysize, at = size_t(y) * e.xsize + x;
  if (e.gray) e.planes[at] = p.x;
  else { int32_t R = p.z, G = p.y, B = p.x; int32_t Co = R - B; int32_t t = B + (Co >> 1); int32_t Cg = G - t; int32_t Y = t + (Cg >> 1); e.planes[at] = Y; e.planes[n + at] = Co; e.planes[2 * n + at] = Cg; }
  if (e.alpha) e.planes[size_t(e.alpha_plane) * n + at] = p.w;
}

__global__ void k_enc_sharpen(float* __restrict__ cur, const float* __restrict__ orig, const float* __restrict__ blur, size_t n) {
  size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; if (i < n) cur[i] += orig[i] - blur[i];
}

// Forward DCT8 of one block in the storage layout of square blocks (S[hf * 8 + vf]); S[0] is the LF sample.
__device__ __forceinline__ void ForwardDct8(const float* px, size_t stride, const float* cos8, float* S) {
  float t[64];
  for (int y = 0; y < 8; y++) { float v[8]; for (int x = 0; x < 8; x++) v[x] = px[size_t(y) * stride + x]; for (int k = 0; k < 8; k++) { float a = 0; for (int x = 0; x < 8; x++) a += v[x] * cos8[k * 8 + x]; t[y * 8 + k] = a * 0.125f; } }
  for (int hf = 0; hf < 8; hf++) for (int vf = 0; vf < 8; vf++) { float a = 0; for (int y = 0; y < 8; y++) a += t[y * 8 + hf] * cos8[vf * 8 + y]; S[hf * 8 + vf] = a * 0.125f; }
}

// Effort >= 5, step 1: per-block statistics of the unquantised coefficients — activity (sum of |AC| of Y) and the three sums of the
// least-squares chroma-from-luma fit over the AC coefficients. One thread per block; block_stats[cell] = {activity, sum X*Y, sum B*Y, sum Y*Y}.
__global__ void __launch_bounds__(64) k_enc_block_stats(const DEncFrame* ep) {
  const DEncFrame& e = *ep; const int cell = blockIdx.x * blockDim.x + threadIdx.x; if (cell >= int(e.xb * e.yb)) return;
  const int cy = cell / int(e.xb), cx = cell % int(e.xb); const float* cos8 = e.tables->cosines + CosOff(3); const size_t plane = size_t(e.xpad) * e.ext_rows;
  const float* base = e.xyb + (size_t(e.ext_top) + size_t(cy) * 8) * e.xpad + size_t(cx) * 8; float Y[64], C[64];
  ForwardDct8(base + plane, e.xpad, cos8, Y);
  float act = 0, syy = 0; for (int k = 1; k < 64; k++) { act += fabsf(Y[k]); syy += Y[k] * Y[k]; }
  ForwardDct8(base, e.xpad, cos8, C); float sxy = 0; for (int k = 1; k < 64; k++) sxy += C[k] * Y[k];
  ForwardDct8(base + 2 * plane, e.xpad, cos8, C); float sby = 0; for (int k = 1; k < 64; k++) sby += C[k] * Y[k];
  reinterpret_cast<float4*>(e.block_stats)[cell] = make_float4(act, sxy, sby, syy);
}
// Step 2: one warp per 64x64 tile (8 x 8 blocks, two per lane, summed in a fixed order: the result does not depend on scheduling).
//   chroma from luma: ytox = round(84 * sum(XY) / sum(YY)), ytob = round(84 * (sum(BY) / sum(YY) - 1))   (kx = ytox / 84, kb = 1 + ytob / 84)
//   adaptive quantisation: the block's multiplier is the frame's base multiplier times (aq_ref / activity)^0.2, limited to [0.75, 1.35] and
//   snapped to five levels (the map costs < 0.02 bpp): finer steps where the block is smooth, coarser where texture masks the error.
//   aq_ref is a constant of the encoder, not a statistic of the frame, so bands of a sharded encode need no exchange for it.
__global__ void __launch_bounds__(128) k_enc_tile_params(const DEncFrame* ep) {
  const DEncFrame& e = *ep; const int lane = threadIdx.x & 31; const uint32_t tile = blockIdx.x * 4 + (threadIdx.x >> 5); if (tile >= e.xt * e.yt) return;
  const uint32_t ty = tile / e.xt, tx = tile % e.xt; float sxy = 0, sby = 0, syy = 0;
  for (int k = 0; k < 2; k++) {
    const uint32_t by = ty * 8 + uint32_t(lane >> 3) + 4u * k, bx = tx * 8 + uint32_t(lane & 7);
    if (by < e.yb && bx < e.xb) {
      const size_t cell = size_t(by) * e.xb + bx; const float4 st = reinterpret_cast<const float4*>(e.block_stats)[cell]; sxy += st.y; sby += st.z; syy += st.w;
      if (e.aq_on) {
        const float mulq = fminf(1.35f, fmaxf(0.75f, __powf(e.aq_ref / (st.x + 1e-4f), 0.2f)));
        const float level = mulq < 0.81f ? 0.75f : mulq < 0.93f ? 0.87f : mulq < 1.08f ? 1.0f : mulq < 1.25f ? 1.16f : 1.35f;
        e.hf_mul_map[cell] = uint8_t(max(1, min(255, __float2int_rn(float(e.hf_mul) * level))));
      } else e.hf_mul_map[cell] = uint8_t(e.hf_mul);
    }
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) { sxy += __shfl_xor_sync(0xffffffffu, sxy, d); sby += __shfl_xor_sync(0xffffffffu, sby, d); syy += __shfl_xor_sync(0xffffffffu, syy, d); }
  if (lane == 0) {
    int fx = 0, fb = 0; if (e.cfl_on && syy > 1e-12f) { fx = __float2int_rn(84.0f * (sxy / syy)); fb = __float2int_rn(84.0f * (sby / syy - 1.0f)); }
    e.ytox_map[tile] = int8_t(max(-128, min(127, fx))); e.ytob_map[tile] = int8_t(max(-128, min(127, fb)));
  }
}

// One thread per 8x8 block; channels in order Y, X, B because X/B quantise against the dequantised Y (A.8 chroma from luma).
__global__ void __launch_bounds__(64) k_enc_dct8(const DEncFrame* ep) {
  const DEncFrame& e = *ep; int cell = blockIdx.x * blockDim.x + threadIdx.x; if (cell >= int(e.xb * e.yb)) return;
  int cy = cell / int(e.xb), cx = cell % int(e.xb); int g = (cy >> 5) * int(e.xgroups) + (cx >> 5); int by = cy & 31, bx = cx & 31;
  const float* cos8 = e.tables->cosines + CosOff(3); const float* dq = e.dequant8; size_t plane = size_t(e.xpad) * e.ext_rows, lfplane = size_t(e.xb) * e.yb;
  const uint32_t hfm = e.hf_mul_map ? e.hf_mul_map[cell] : e.hf_mul; float kx = e.kx, kb = e.kb;
  if (e.ytox_map) { const size_t tile = size_t(cy >> 3) * e.xt + (cx >> 3); kx = float(e.ytox_map[tile]) * (1.0f / 84.0f); kb = 1.0f + float(e.ytob_map[tile]) * (1.0f / 84.0f); }
  float scale = e.inv_gs / float(hfm); float ydq[64]; uint32_t nzc[3];
#pragma unroll 1
  for (int ci = 0; ci < 3; ci++) {
    const int c = ci == 0 ? 1 : ci == 1 ? 0 : 2; const float* px = e.xyb + c * plane + (size_t(e.ext_top) + size_t(cy) * 8) * e.xpad + size_t(cx) * 8; float S[64];
    ForwardDct8(px, e.xpad, cos8, S);
    e.lf[c * lfplane + cell] = S[0];
    int16_t* out = e.coeffs + (size_t(g) * 3 + c) * 65536 + (size_t(by) * 32 + bx) * 64; uint32_t nz = 0;
    const float mulc = c == 1 ? scale : c == 0 ? scale * e.xm : scale * e.bm, kc = c == 0 ? kx : kb;
    for (int p = 0; p < 64; p++) {
      int q = 0;
      if (p) { float step = dq[c * 64 + p] * mulc; float v = S[p]; if (c != 1) v -= kc * ydq[p]; float qf = v / step; if (fabsf(qf) >= 0.56f) q = __float2int_rn(qf); q = max(-32768, min(32767, q));
        if (c == 1) { float a = q == 0 ? 0.f : q == 1 ? e.quant_bias[1] : q == -1 ? -e.quant_bias[1] : float(q) - e.quant_bias[3] / float(q); ydq[p] = a * step; } nz += q != 0; }
      out[p] = int16_t(q);
    }
    nzc[c] = nz;
  }
  e.nz[cell] = uint8_t(nzc[0]); e.nz[lfplane + cell] = uint8_t(nzc[1]); e.nz[2 * lfplane + cell] = uint8_t(nzc[2]);
}

__global__ void k_enc_lf_quant(const DEncFrame* ep) {
  const DEncFrame& e = *ep; size_t n = size_t(e.xb) * e.yb, i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; if (i >= n) return;
  float fy = e.lf_fac[1]; int32_t qy = __float2int_rn(e.lf[n + i] / fy); float ydq = float(qy) * fy;
  int32_t qx = __float2int_rn((e.lf[i] - e.cfl_x_lf * ydq) / e.lf_fac[0]), qb = __float2int_rn((e.lf[2 * n + i] - e.cfl_b_lf * ydq) / e.lf_fac[2]);
  e.lfq[i] = qy; e.lfq[n + i] = qx; e.lfq[2 * n + i] = qb;   // stream channel order Y, X, B
}

__device__ __forceinline__ uint32_t PackSignedDev(int32_t v) { return (uint32_t(v) << 1) ^ uint32_t(v >> 31); }
// token word: ctx[0,16) | symbol[16,24) | nbits[24,30); second word: extra bits
__device__ __forceinline__ void MakeToken(uint32_t ctx, uint32_t value, uint32_t split_exp, uint32_t msb, uint2* out) {
  uint32_t split = 1u << split_exp, tok, nb = 0, bits = 0;
  if (value < split) tok = value; else { uint32_t n = 31 - __clz(value), m = value - (1u << n); tok = split + ((n - split_exp) << msb) + (m >> (n - msb)); nb = n - msb; bits = m & ((1u << nb) - 1); }
  *out = make_uint2(ctx | (tok << 16) | (nb << 24), bits);
}

// Modular tokenisation: stream s covers rect (x0,y0,w,h) of `nch` planes of size (pw x ph); tokens in channel-major raster order.
__global__ void k_enc_mod_tokens(const DEncFrame* ep, const DEncModStream* streams, const int32_t* __restrict__ planes, uint32_t pw, uint32_t ph, uint32_t nch, const uint16_t* __restrict__ leaf_lut /*[kind][8 ch][11]*/) {
  const DEncFrame& e = *ep; const DEncModStream s = streams[blockIdx.y]; uint32_t per = s.w * s.h, total = per * nch, i = blockIdx.x * blockDim.x + threadIdx.x; if (i >= total) return;
  uint32_t c = i / per, r = i % per; int y = int(r / s.w), x = int(r % s.w); const int32_t* p = planes + size_t(c) * pw * ph + size_t(s.y0) * pw + s.x0; const int W = int(pw);
  auto at = [&](int yy, int xx) -> int32_t { return p[size_t(yy) * W + xx]; };
  int32_t Wv = x ? at(y, x - 1) : (y ? at(y - 1, x) : 0), N = y ? at(y - 1, x) : Wv, NW = (x && y) ? at(y - 1, x - 1) : Wv;
  int32_t lo = min(Wv, N), hi = max(Wv, N), pred = max(lo, min(hi, Wv + N - NW));
  int32_t prev_grad = 0; if (x) { int xp = x - 1; int32_t Wp = xp ? at(y, xp - 1) : (y ? at(y - 1, xp) : 0), Np = y ? at(y - 1, xp) : Wp, NWp = (xp && y) ? at(y - 1, xp - 1) : Wp; prev_grad = Wp + Np - NWp; }
  int32_t prop8 = Wv - prev_grad; const int32_t thr[10] = {-64, -24, -8, -3, -1, 0, 2, 7, 23, 63}; int bucket = 0; for (int k = 0; k < 10; k++) bucket += prop8 > thr[k];
  uint32_t ctx = leaf_lut[(s.kind * 8 + c) * 11 + bucket];
  MakeToken(ctx, PackSignedDev(at(y, x) - pred), 4, 1, e.tokens + s.token_off + i);
}

__device__ __constant__ uint8_t kFreqCtxE[64] = {0, 0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 15, 16, 16, 17, 17, 18, 18, 19, 19, 20, 20, 21, 21, 22, 22,
  23, 23, 23, 23, 24, 24, 24, 24, 25, 25, 25, 25, 26, 26, 26, 26, 27, 27, 27, 27, 28, 28, 28, 28, 29, 29, 29, 29, 30, 30, 30, 30};
__device__ __constant__ uint8_t kNumNzCtxE[64] = {0, 0, 31, 62, 62, 93, 93, 93, 93, 123, 123, 123, 123, 152, 152, 152, 152, 152, 152, 152, 152, 180, 180, 180, 180, 180, 180, 180, 180, 180, 180, 180, 180,
  206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206};

// AC tokenisation for DCT8-only frames (default block-context map: 15 contexts, order id 0). One CTA per 256x256 group, one thread per
// 8x8 block: a block's token count is known from its coefficients alone (1 + the scan position of the last non-zero coefficient, per
// channel), so a CTA-wide exclusive scan in raster order gives every block its place in the group's token stream and all blocks are
// written at once. (r01: one THREAD per group walked its 1024 blocks serially.)
__global__ void __launch_bounds__(1024) k_enc_ac_tokens(const DEncFrame* ep) {
  const DEncFrame& e = *ep; const int g = blockIdx.x;
  const int gx = g % int(e.xgroups), gy = g / int(e.xgroups), cx0 = gx * 32, cy0 = gy * 32, w = min(32, int(e.xb) - cx0), h = min(32, int(e.yb) - cy0); const size_t lfplane = size_t(e.xb) * e.yb;
  const int tid = threadIdx.x, by = tid >> 5, bx = tid & 31, lane = tid & 31, warp = tid >> 5; const bool active = by < h && bx < w;
  const uint32_t nbctx = 15; const uint8_t bctx_of[3] = {7, 0, 7};   // default map, order 0: Y->0, X->7, B->7 (A.8)
  const uint16_t* order = e.order8; const size_t cell = size_t(cy0 + by) * e.xb + cx0 + bx;
  __shared__ uint32_t warp_total[32];
  // ---- count: per channel, the scan position of the last non-zero coefficient (0: the block has none)
  uint32_t last[3] = {0, 0, 0}, cnt = 0;
  if (active) {
#pragma unroll 1
    for (int c = 0; c < 3; c++) {
      if (e.nz[c * lfplane + cell]) { const int16_t* co = e.coeffs + (size_t(g) * 3 + c) * 65536 + (size_t(by) * 32 + bx) * 64; int k = 63; while (k > 0 && co[order[k]] == 0) k--; last[c] = uint32_t(k); }
      cnt += 1 + last[c];
    }
  }
  // ---- exclusive scan over the CTA in raster order
  uint32_t incl = cnt;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) { const uint32_t v = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl += v; }
  if (lane == 31) warp_total[warp] = incl;
  __syncthreads();
  if (warp == 0) { uint32_t v = warp_total[lane], iv = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const uint32_t u = __shfl_up_sync(0xffffffffu, iv, d); if (lane >= d) iv += u; }
    warp_total[lane] = iv - v; if (lane == 31) e.ac_token_count[g] = iv; }
  __syncthreads();
  if (!active) return;
  uint2* out = e.tokens + e.ac_token_off + size_t(g) * kMaxAcTokensPerGroup + warp_total[warp] + (incl - cnt);
  // ---- emit: channels in the order Y, X, B
#pragma unroll 1
  for (int ci = 0; ci < 3; ci++) {
    const int c = ci == 0 ? 1 : ci == 1 ? 0 : 2; const uint8_t* nzp = e.nz + c * lfplane; uint32_t nz = nzp[cell];
    uint32_t pred; if (bx == 0) pred = by == 0 ? 32 : nzp[cell - e.xb]; else if (by == 0) pred = nzp[cell - 1]; else pred = (uint32_t(nzp[cell - e.xb]) + nzp[cell - 1] + 1) >> 1;
    const uint32_t nzb = pred < 8 ? pred : (pred >= 64 ? 36 : 4 + pred / 2), bc = bctx_of[c];
    MakeToken(nzb * nbctx + bc, nz, 4, 2, out++);
    const int16_t* co = e.coeffs + (size_t(g) * 3 + c) * 65536 + (size_t(by) * 32 + bx) * 64; const uint32_t histo = nbctx * 37 + 458 * bc; uint32_t prev = nz > 4 ? 0 : 1;
    for (uint32_t k = 1; k <= last[c]; k++) { const int32_t v = co[order[k]]; const uint32_t zctx = (uint32_t(kNumNzCtxE[nz]) + kFreqCtxE[k]) * 2 + prev; MakeToken(histo + zctx, PackSignedDev(v), 4, 2, out++); prev = v != 0; nz -= prev; }
  }
}

// Token histograms. Neighbouring tokens of a stream mostly share their (context, symbol) pair (runs of zeros in one context), so a warp first
// groups its lanes by key and one lane per group adds the group's size: same-address atomics, which serialise in L2, drop several-fold.
__global__ void k_enc_histogram(const uint2* __restrict__ tokens, const DEncStream* streams, uint32_t* hist) {
  const DEncStream s = streams[blockIdx.y]; const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; const bool valid = i < s.count;
  const uint32_t t = valid ? tokens[s.token_off + i].x : 0xffffffffu; const uint32_t key = valid ? (t & 0x00ffffffu) : 0xffffffffu;   // ctx[0,16) | symbol[16,24)
  const uint32_t peers = __match_any_sync(0xffffffffu, key); const int leader = __ffs(peers) - 1;
  if (valid && int(threadIdx.x & 31) == leader) atomicAdd(hist + size_t(key & 0xffff) * kEncAlphabet + (key >> 16), uint32_t(__popc(peers)));
}

// ANS writer (A.6 "ANS symbol read" mirrored), one WARP per section stream. The state chain is serial (token i needs the state after token
// i + 1), but everything around it is not:
//   reverse pass: the lanes load 32 tokens at once and look up cluster, frequency, reciprocal and reverse-table base for them; then the warp
//                 steps through the 32 tokens with the state held redundantly in every lane (shuffles hand out token k's operands), so a step
//                 is a reciprocal multiply + one dependent table load, not five dependent global loads;
//   forward pass: lengths (16 flush bits + extra bits) are prefix-summed across the warp, every lane ORs its bits into a shared-memory
//                 window, whole words go to HBM with coalesced stores.
// (r01: one THREAD per stream: 32 lanes of a warp walked 32 different streams with scattered loads, 70 ms per launch at 12 MP.)
__global__ void __launch_bounds__(128) k_enc_ans(const DEncFrame* ep, const DEncStream* streams, uint32_t nstreams, const DEncCode* code, uint32_t bits_off) {
  const DEncFrame& e = *ep; const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5; const uint32_t si = blockIdx.x * 4 + warp;
  __shared__ uint32_t window[4][56];
  if (si >= nstreams) return;   // whole warps leave; only __syncwarp below
  const DEncStream s = streams[si]; uint2* tk = e.tokens + s.token_off; const uint32_t count = s.count; uint32_t state = 0x130000u;
  const uint8_t* ctx_map = code->ctx_map; const uint16_t* freq = code->freq; const uint16_t* start = code->start; const uint16_t* rev = code->rev;
  // One step of the chain for token k of the chunk: the operands come from lane k, the state is uniform across the warp. Both candidates of
  // the quotient (with and without the 16-bit flush) are started before the flush decision is known.
  auto step = [&](int k, uint32_t f, uint32_t m, uint32_t rb, uint32_t& myflush) {
    const uint32_t fk = __shfl_sync(0xffffffffu, f, k), mk = __shfl_sync(0xffffffffu, m, k), rk = __shfl_sync(0xffffffffu, rb, k);
    const bool fl = (state >> 20) >= fk; const uint32_t flush = fl ? (0x10000u | (state & 0xffff)) : 0u, x = fl ? (state >> 16) : state;
    uint32_t q = __umulhi(x, mk), r = x - q * fk; if (r >= fk) { q++; r -= fk; } if (r >= fk) { q++; r -= fk; }
    state = (q << 12) + rev[rk + r];
    if (lane == k) myflush = flush;
  };
  for (int64_t base = count ? int64_t((count - 1) & ~31u) : -1; base >= 0; base -= 32) {
    const uint32_t i = uint32_t(base) + lane; const bool valid = i < count; uint32_t t = 0, f = 1, rb = 0;
    if (valid) { t = tk[i].x; const uint32_t cl = ctx_map[t & 0xffff], sym = (t >> 16) & 0xff; f = freq[cl * kEncAlphabet + sym]; rb = cl * 4096 + start[cl * kEncAlphabet + sym]; }
    const uint32_t m = 0xffffffffu / max(f, 1u);   // floor((2^32 - 1) / f): umulhi(state, m) is state / f or up to 2 less
    uint32_t myflush = 0; const int kmax = int(min(uint32_t(31), count - 1 - uint32_t(base)));
    if (kmax == 31) {   // full chunk: straight-line code, so the shuffles of later tokens issue while a table load is in flight
#pragma unroll
      for (int k = 31; k >= 0; k--) step(k, f, m, rb, myflush);
    } else for (int k = kmax; k >= 0; k--) step(k, f, m, rb, myflush);
    if (valid) tk[i].x = (t & 0x3f000000u) | myflush;   // keep nbits, replace ctx / symbol by the flush word
  }
  __syncwarp();
  // ---- forward: the final state first (32 bits), then per token [16 flush bits][extra bits]
  uint32_t* out = reinterpret_cast<uint32_t*>(e.stream_bytes + s.byte_off); uint32_t* win = window[warp];
  if (lane == 0) out[0] = state;
  uint64_t pos = 32; uint32_t carry = 0;   // bits written so far; the partial last word
  for (uint32_t base = 0; base < count; base += 32) {
    const uint32_t i = base + lane; uint32_t len = 0; uint64_t val = 0;
    if (i < count) { const uint2 t = tk[i]; const uint32_t nb = (t.x >> 24) & 0x3f; if (t.x & 0x10000u) { val = (t.x & 0xffff) | (uint64_t(t.y) << 16); len = 16 + nb; } else { val = t.y; len = nb; } }
    uint32_t incl = len;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const uint32_t v = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl += v; }
    const uint32_t total = __shfl_sync(0xffffffffu, incl, 31), lead = uint32_t(pos & 31), at = lead + incl - len;
    win[lane] = lane == 0 ? carry : 0; if (lane < 24) win[32 + lane] = 0;
    __syncwarp();
    if (len) { const uint32_t wd = at >> 5, sh = at & 31; const uint64_t lo = val << sh; atomicOr(&win[wd], uint32_t(lo)); const uint32_t mid = uint32_t(lo >> 32); if (mid) atomicOr(&win[wd + 1], mid);
      if (sh + len > 64) atomicOr(&win[wd + 2], uint32_t(val >> (64 - sh))); }
    __syncwarp();
    const uint32_t filled = lead + total, nfull = filled >> 5; uint32_t* dst = out + (pos >> 5);
    for (uint32_t j = lane; j < nfull; j += 32) dst[j] = win[j];
    carry = win[nfull]; pos += total;
    __syncwarp();
  }
  if (lane == 0) { if (pos & 31) out[pos >> 5] = carry; e.stream_bits[bits_off + si] = pos; }
}

// Prefix-code writer (efforts 1-2: what libjxl's fastest efforts use too). A prefix code has no state chain, so a stream is one warp-parallel pass:
// every lane looks up its token's code (length in `freq`, bit-reversed code word in `start` of the cluster's row), the lengths (code + extra bits)
// are prefix-summed and the bits packed through the same shared-memory window as the ANS writer's forward pass. The four LF-group streams that
// bound an ANS encode (589 824 tokens each, ~20 ms serial) take well under a millisecond this way.
__global__ void __launch_bounds__(128) k_enc_prefix(const DEncFrame* ep, const DEncStream* streams, uint32_t nstreams, const DEncCode* code, uint32_t bits_off) {
  const DEncFrame& e = *ep; const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5; const uint32_t si = blockIdx.x * 4 + warp;
  __shared__ uint32_t window[4][56];
  if (si >= nstreams) return;
  const DEncStream s = streams[si]; const uint2* tk = e.tokens + s.token_off; const uint32_t count = s.count;
  const uint8_t* ctx_map = code->ctx_map; const uint16_t* plen = code->freq; const uint16_t* pcode = code->start;
  uint32_t* out = reinterpret_cast<uint32_t*>(e.stream_bytes + s.byte_off); uint32_t* win = window[warp];
  uint64_t pos = 0; uint32_t carry = 0;
  for (uint32_t base = 0; base < count; base += 32) {
    const uint32_t i = base + lane; uint32_t len = 0; uint64_t val = 0;
    if (i < count) { const uint2 t = tk[i]; const uint32_t cl = ctx_map[t.x & 0xffff], sym = (t.x >> 16) & 0xff, nb = (t.x >> 24) & 0x3f, cl_len = plen[cl * kEncAlphabet + sym];
      val = uint64_t(pcode[cl * kEncAlphabet + sym]) | (uint64_t(t.y) << cl_len); len = cl_len + nb; }
    uint32_t incl = len;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const uint32_t v = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl += v; }
    const uint32_t total = __shfl_sync(0xffffffffu, incl, 31), lead = uint32_t(pos & 31), at = lead + incl - len;
    win[lane] = lane == 0 ? carry : 0; if (lane < 24) win[32 + lane] = 0;
    __syncwarp();
    if (len) { const uint32_t wd = at >> 5, sh = at & 31; const uint64_t lo = val << sh; atomicOr(&win[wd], uint32_t(lo)); const uint32_t mid = uint32_t(lo >> 32); if (mid) atomicOr(&win[wd + 1], mid);
      if (sh + len > 64) atomicOr(&win[wd + 2], uint32_t(val >> (64 - sh))); }
    __syncwarp();
    const uint32_t filled = lead + total, nfull = filled >> 5; uint32_t* dst = out + (pos >> 5);
    for (uint32_t j = lane; j < nfull; j += 32) dst[j] = win[j];
    carry = win[nfull]; pos += total;
    __syncwarp();
  }
  if (lane == 0) { if (pos & 31) out[pos >> 5] = carry; e.stream_bits[bits_off + si] = pos; }
}

// The ANS writer leaves every stream at the start of a slot sized for its worst case (6 bytes per token); the host wants the bytes that
// were actually written. One CTA per stream copies ceil(bits / 8) bytes, 16 at a time, to its place in a dense buffer (offsets are
// multiples of 16), so that the device-to-host copy carries the compressed size, not the worst case (r02: 1.6 GB -> 60 MB per 537 MP band).
__global__ void __launch_bounds__(256) k_enc_compact(const uint8_t* __restrict__ src, const DEncStream* streams, const uint64_t* __restrict__ bits, const uint64_t* __restrict__ dst_off, uint8_t* __restrict__ dst) {
  const uint32_t si = blockIdx.x; const uint64_t nvec = ((bits[si] + 7) / 8 + 15) / 16;
  const uint4* s = reinterpret_cast<const uint4*>(src + streams[si].byte_off); uint4* d = reinterpret_cast<uint4*>(dst + dst_off[si]);
  for (uint64_t i = threadIdx.x; i < nvec; i += 256) d[i] = s[i];
}
void EncLaunchCompact(const uint8_t* src, const DEncStream* streams, uint32_t nstreams, const uint64_t* bits, const uint64_t* dst_off, uint8_t* dst, cudaStream_t st) {
  if (!nstreams) return; Launch<k_enc_compact>(nstreams, 256, 0, st, src, streams, bits, dst_off, dst);
}
void EncLaunchScan(const uint8_t* bgra, uint32_t w, uint32_t h, uint32_t stride, uint32_t* flags, cudaStream_t st) { dim3 grid((w + 255) / 256, h); Launch<k_enc_scan>(grid, 256, 0, st, bgra, w, h, stride, flags); }
void EncLaunchToXyb(const DEncFrame* d, const DEncFrame& h, const uint8_t* bgra, cudaStream_t st) { dim3 blk(32, 8), grid((h.xpad + 31) / 32, (h.ext_rows + 7) / 8); Launch<k_enc_to_xyb>(grid, blk, 0, st, d, bgra); }
void EncLaunchToPlanes(const DEncFrame* d, const DEncFrame& h, const uint8_t* bgra, cudaStream_t st) { dim3 blk(32, 8), grid((h.xsize + 31) / 32, (h.ysize + 7) / 8); Launch<k_enc_to_planes>(grid, blk, 0, st, d, bgra); }
void EncLaunchSharpen(float* cur, const float* orig, const float* blur, size_t n, cudaStream_t st) { Launch<k_enc_sharpen>(unsigned((n + 255) / 256), 256, 0, st, cur, orig, blur, n); }
void EncLaunchBlockParams(const DEncFrame* d, const DEncFrame& h, cudaStream_t st) {
  const uint32_t cells = h.xb * h.yb, tiles = h.xt * h.yt; Launch<k_enc_block_stats>((cells + 63) / 64, 64, 0, st, d); Launch<k_enc_tile_params>((tiles + 3) / 4, 128, 0, st, d);
}
void EncLaunchDct8(const DEncFrame* d, const DEncFrame& h, cudaStream_t st) { uint32_t cells = h.xb * h.yb; Launch<k_enc_dct8>((cells + 63) / 64, 64, 0, st, d); Launch<k_enc_lf_quant>((cells + 255) / 256, 256, 0, st, d); }
void EncLaunchModTokens(const DEncFrame* d, const DEncModStream* streams, uint32_t nstreams, uint32_t max_tokens, const int32_t* planes, uint32_t pw, uint32_t ph, uint32_t nch, const uint16_t* leaf_lut, cudaStream_t st) {
  if (!nstreams || !max_tokens) return; dim3 grid((max_tokens + 255) / 256, nstreams); Launch<k_enc_mod_tokens>(grid, 256, 0, st, d, streams, planes, pw, ph, nch, leaf_lut);
}
void EncLaunchAcTokens(const DEncFrame* d, const DEncFrame& h, cudaStream_t st) { if (!h.num_groups) return; Launch<k_enc_ac_tokens>(h.num_groups, 1024, 0, st, d); }
void EncLaunchHistogram(const uint2* tokens, const DEncStream* streams, uint32_t nstreams, uint32_t max_count, uint32_t* hist, cudaStream_t st) {
  if (!nstreams || !max_count) return; dim3 grid((max_count + 255) / 256, nstreams); Launch<k_enc_histogram>(grid, 256, 0, st, tokens, streams, hist);
}
void EncLaunchPrefix(const DEncFrame* d, const DEncStream* streams, uint32_t nstreams, const DEncCode* code, uint32_t bits_off, cudaStream_t st) { if (!nstreams) return; Launch<k_enc_prefix>((nstreams + 3) / 4, 128, 0, st, d, streams, nstreams, code, bits_off); }
void EncLaunchAns(const DEncFrame* d, const DEncStream* streams, uint32_t nstreams, const DEncCode* code, uint32_t bits_off, cudaStream_t st) { if (!nstreams) return; Launch<k_enc_ans>((nstreams + 3) / 4, 128, 0, st, d, streams, nstreams, code, bits_off); }

}  // namespace jxlgpu
