// pdn-jpegxl_b200 engine — reconstruction kernels (sm_100a), all HBM-bound fp32 stages:
//   k_reconstruct : HF dequant + chroma-from-luma + LLF-from-LF + inverse transform for every varblock of a
//                   256x256 group (SURVEY.md A.8 "Dequant", A.9). int16 coefficients in, fp32 XYB planes out:
//                   6 B + 12 B = 18 algorithmic bytes per pixel.
//   k_inv_sigma : the EPF's 1/sigma per 8x8 block. k_gaborish : one gaborish pass over whole planes (the encoder's inverse gaborish).
//   k_render_wide_tma, k_render : restoration filters (A.10) + colour + pack fused, one tile and its halo at a time in shared memory.
//   k_output / k_output_int : XYB -> linear -> transfer function -> sample type, interleave, optional
//                   fused BGRA32 surface pack (15-16 B/px for 8-bit RGB/BGRA), bit-exact integer path for lossless.
// Replaces libjxl's dequant / IDCT / render-pipeline stages reached from N/Decoder/JxlDecoder.cpp:252 and the
// managed repack loops I/DecoderLayerData.cs:667-992 + S/JpegXLLoad.cs:219-249 (bgra mode).
#include "frame.cuh"
#include "kernels.h"
#include "enc_frame.cuh"
#include "idct_tables.inc"
#include <cuda_fp16.h>
#include <cuda.h>
#include <cmath>
#include <stdexcept>

namespace jxlgpu {

void FillDeviceTables(DTables* t) {
  for (int l = 0; l <= 8; l++) { int n = 1 << l; float* c = t->cosines + CosOff(l);
    for (int k = 0; k < n; k++) for (int i = 0; i < n; i++) c[size_t(k) * n + i] = float((k == 0 ? 1.0 : std::sqrt(2.0)) * std::cos((2 * i + 1) * k * M_PI / (2.0 * n))); }
  for (int l = 0; l < 6; l++) { int n = 1 << l; for (int u = 0; u < 32; u++) { double p = 1; if (u < n) for (int k = 0; k < 3; k++) p *= std::cos(u * M_PI * double(1 << k) / (16.0 * n)); t->resample[l][u] = float(1.0 / p); } }
}

__device__ __forceinline__ float AdjustQuantBiasDev(int q, float b1, float b3) { if (q == 0) return 0.f; if (q == 1) return b1; if (q == -1) return -b1; return float(q) - b3 / float(q); }
__device__ __forceinline__ int Log2Dev(int n) { return 31 - __clz(n); }

// 8x8 special transforms (A.9 [L]); coef/px in registers or shared memory, stride in floats
__device__ void SpecialTransform8x8(int s, const float* coef, float* px, size_t stride, const float* cos4, const float* cos8) {
  if (s == 2) {   // DCT2X2: three Hadamard levels
    float b[64], t[64]; for (int i = 0; i < 64; i++) b[i] = coef[i];
    for (int S = 2; S <= 8; S *= 2) { int n = S / 2;
      for (int y = 0; y < n; y++) for (int x = 0; x < n; x++) { float c00 = b[y * 8 + x], c01 = b[y * 8 + n + x], c10 = b[(y + n) * 8 + x], c11 = b[(y + n) * 8 + n + x];
        t[y * 2 * 8 + x * 2] = c00 + c01 + c10 + c11; t[y * 2 * 8 + x * 2 + 1] = c00 + c01 - c10 - c11; t[(y * 2 + 1) * 8 + x * 2] = c00 - c01 + c10 - c11; t[(y * 2 + 1) * 8 + x * 2 + 1] = c00 - c01 - c10 + c11; }
      for (int y = 0; y < S; y++) for (int x = 0; x < S; x++) b[y * 8 + x] = t[y * 8 + x]; }
    for (int y = 0; y < 8; y++) for (int x = 0; x < 8; x++) px[y * stride + x] = b[y * 8 + x];
    return;
  }
  if (s == 3 || s == 1) {
    float a = coef[0], b = coef[1], c = coef[8], d = coef[9]; float dcs[4] = {a + b + c + d, a + b - c - d, a - b + c - d, a - b - c + d};
    for (int y = 0; y < 2; y++) for (int x = 0; x < 2; x++) {
      if (s == 3) {   // DCT4X4: storage blk[hf][vf]
        float blk[16]; blk[0] = dcs[y * 2 + x]; for (int iy = 0; iy < 4; iy++) for (int ix = 0; ix < 4; ix++) if (ix || iy) blk[iy * 4 + ix] = coef[(y + iy * 2) * 8 + x + ix * 2];
        float tmp[16];
        for (int hf = 0; hf < 4; hf++) for (int py = 0; py < 4; py++) { float sacc = 0; for (int vf = 0; vf < 4; vf++) sacc += blk[hf * 4 + vf] * cos4[vf * 4 + py]; tmp[hf * 4 + py] = sacc; }
        for (int py = 0; py < 4; py++) for (int pxx = 0; pxx < 4; pxx++) { float sacc = 0; for (int hf = 0; hf < 4; hf++) sacc += tmp[hf * 4 + py] * cos4[hf * 4 + pxx]; px[(y * 4 + py) * stride + x * 4 + pxx] = sacc; }
      } else {        // IDENTITY
        float block_dc = dcs[y * 2 + x], rs = 0; for (int iy = 0; iy < 4; iy++) for (int ix = 0; ix < 4; ix++) if (ix || iy) rs += coef[(y + iy * 2) * 8 + x + ix * 2];
        float center = block_dc - rs * (1.0f / 16); px[(4 * y + 1) * stride + 4 * x + 1] = center;
        for (int iy = 0; iy < 4; iy++) for (int ix = 0; ix < 4; ix++) { if (ix == 1 && iy == 1) continue; px[(y * 4 + iy) * stride + x * 4 + ix] = coef[(y + iy * 2) * 8 + x + ix * 2] + center; }
        px[y * 4 * stride + x * 4] = coef[(y + 2) * 8 + x + 2] + center;
      }
    }
    return;
  }
  // DCT4X8 (s==12): two 4-row x 8-col halves stacked vertically, storage blk[vf(4)][hf(8)];
  // DCT8X4 (s==13): two 8-row x 4-col halves side by side, storage blk[hf(4)][vf(8)]
  float dcs[2] = {coef[0] + coef[8], coef[0] - coef[8]};
  for (int k = 0; k < 2; k++) {
    float blk[32]; blk[0] = dcs[k]; for (int iy = 0; iy < 4; iy++) for (int ix = 0; ix < 8; ix++) if (ix || iy) blk[iy * 8 + ix] = coef[(k + iy * 2) * 8 + ix];
    float tmp[32];   // tmp[r][j]: r = short-axis frequency (4), j = long-axis position (8)
    for (int r = 0; r < 4; r++) for (int j = 0; j < 8; j++) { float sacc = 0; for (int c = 0; c < 8; c++) sacc += blk[r * 8 + c] * cos8[c * 8 + j]; tmp[r * 8 + j] = sacc; }
    for (int i = 0; i < 4; i++) for (int j = 0; j < 8; j++) { float sacc = 0; for (int r = 0; r < 4; r++) sacc += tmp[r * 8 + j] * cos4[r * 4 + i];
      if (s == 12) px[(k * 4 + i) * stride + j] = sacc; else px[j * stride + k * 4 + i] = sacc; }
  }
}

// LLF corner from the LF samples of the block (A.9 "LLF from DC"). lanes cooperate; writes into storage-layout S.
__device__ void LlfFromLf(const DFrame& f, int c, int cy, int cx, const float* lfp, int lf_stride, float* S, int SW, int lane, int nlanes) {
  const DTables& t = *f.tables; const int ly = Log2Dev(cy), lx = Log2Dev(cx); const float* cv = t.cosines + CosOff(ly); const float* ch = t.cosines + CosOff(lx);
  for (int idx = lane; idx < cy * cx; idx += nlanes) { int v = idx / cx, hfr = idx % cx; float acc = 0;
    for (int y = 0; y < cy; y++) { float rowacc = 0; for (int x = 0; x < cx; x++) rowacc += lfp[y * lf_stride + x] * ch[hfr * cx + x]; acc += rowacc * cv[v * cy + y]; }
    float val = acc / float(cy * cx) * t.resample[ly][v] * t.resample[lx][hfr];
    if (cy < cx) S[v * SW + hfr] = val; else S[hfr * SW + v] = val; }
  (void)c;
}

// ------------------------------------------------------------------ DCT8 fast path
// c[k*8+i] = ck * cos((2i+1) k pi / 16), c0 = 1, ck = sqrt(2) (A.9 scaling: inverse is the plain DCT-III sum)
__device__ constexpr float kCos8[64] = {1.000000000e+00f, 1.000000000e+00f, 1.000000000e+00f, 1.000000000e+00f, 1.000000000e+00f, 1.000000000e+00f, 1.000000000e+00f, 1.000000000e+00f, 1.387039845e+00f, 1.175875602e+00f, 7.856949584e-01f, 2.758993793e-01f, -2.758993793e-01f, -7.856949584e-01f, -1.175875602e+00f, -1.387039845e+00f, 1.306562965e+00f, 5.411961001e-01f, -5.411961001e-01f, -1.306562965e+00f, -1.306562965e+00f, -5.411961001e-01f, 5.411961001e-01f, 1.306562965e+00f, 1.175875602e+00f, -2.758993793e-01f, -1.387039845e+00f, -7.856949584e-01f, 7.856949584e-01f, 1.387039845e+00f, 2.758993793e-01f, -1.175875602e+00f, 1.000000000e+00f, -1.000000000e+00f, -1.000000000e+00f, 1.000000000e+00f, 1.000000000e+00f, -1.000000000e+00f, -1.000000000e+00f, 1.000000000e+00f, 7.856949584e-01f, -1.387039845e+00f, 2.758993793e-01f, 1.175875602e+00f, -1.175875602e+00f, -2.758993793e-01f, 1.387039845e+00f, -7.856949584e-01f, 5.411961001e-01f, -1.306562965e+00f, 1.306562965e+00f, -5.411961001e-01f, -5.411961001e-01f, 1.306562965e+00f, -1.306562965e+00f, 5.411961001e-01f, 2.758993793e-01f, -7.856949584e-01f, 1.175875602e+00f, -1.387039845e+00f, 1.387039845e+00f, -1.175875602e+00f, 7.856949584e-01f, -2.758993793e-01f};

// 8-point inverse DCT in the codestream's scaling (y[n] = X0 + sqrt2 * sum_k X[k] cos((2n+1) k pi / 16)) as an even/odd split:
// 34 flops instead of the 64 of the matrix form (kCos8 rows 1,3,5,7 are +-{k1,k3,k5,k7}, rows 2,6 are +-{1.3066, 0.5412}, row 4 is +-1).
__device__ __forceinline__ void Idct8(const float X[8], float y[8]) {
  const float k1 = 1.387039845e+00f, k3 = 1.175875602e+00f, k5 = 7.856949584e-01f, k7 = 2.758993793e-01f, r2 = 1.306562965e+00f, r6 = 5.411961001e-01f;
  const float a0 = X[0] + X[4], a1 = X[0] - X[4];
  const float b0 = fmaf(r2, X[2], r6 * X[6]), b1 = fmaf(r6, X[2], -r2 * X[6]);
  const float e0 = a0 + b0, e3 = a0 - b0, e1 = a1 + b1, e2 = a1 - b1;
  const float o0 = fmaf(k1, X[1], fmaf(k3, X[3], fmaf(k5, X[5], k7 * X[7])));
  const float o1 = fmaf(k3, X[1], fmaf(-k7, X[3], fmaf(-k1, X[5], -k5 * X[7])));
  const float o2 = fmaf(k5, X[1], fmaf(-k1, X[3], fmaf(k7, X[5], k3 * X[7])));
  const float o3 = fmaf(k7, X[1], fmaf(-k5, X[3], fmaf(k3, X[5], -k1 * X[7])));
  y[0] = e0 + o0; y[7] = e0 - o0; y[1] = e1 + o1; y[6] = e1 - o1; y[2] = e2 + o2; y[5] = e2 - o2; y[3] = e3 + o3; y[4] = e3 - o3;
}

// N-point inverse DCT (N = 8, 16, 32) on register arrays by the even/odd recursion: the even-indexed coefficients are an N/2-point
// IDCT, the odd ones an (N/2)x(N/2) product with compile-time constants (FFMA immediates after unrolling): 114 flops for N = 16 and
// 402 for N = 32 instead of N^2, and no cosine-table loads.
template <int N> struct IdctN;
template <> struct IdctN<8> { static __device__ __forceinline__ void Run(const float* X, float* y) { Idct8(X, y); } };
template <> struct IdctN<16> { static __device__ __forceinline__ void Run(const float* X, float* y) {
  float e[8], ye[8];
#pragma unroll
  for (int i = 0; i < 8; i++) e[i] = X[2 * i];
  Idct8(e, ye);
#pragma unroll
  for (int n = 0; n < 8; n++) { float o = 0.f;
#pragma unroll
    for (int i = 0; i < 8; i++) o = fmaf(kOdd16[i][n], X[2 * i + 1], o);
    y[n] = ye[n] + o; y[15 - n] = ye[n] - o; } } };
template <> struct IdctN<32> { static __device__ __forceinline__ void Run(const float* X, float* y) {
  float e[16], ye[16];
#pragma unroll
  for (int i = 0; i < 16; i++) e[i] = X[2 * i];
  IdctN<16>::Run(e, ye);
#pragma unroll
  for (int n = 0; n < 16; n++) { float o = 0.f;
#pragma unroll
    for (int i = 0; i < 16; i++) o = fmaf(kOdd32[i][n], X[2 * i + 1], o);
    y[n] = ye[n] + o; y[31 - n] = ye[n] - o; } } };

// Both passes of a separable SW x SH inverse transform for one warp. S holds the dequantised block in storage layout (SH rows of SW
// coefficients, row stride STR = SW + 4 floats so that LDS.128 by 8 consecutive rows is conflict-free), T is scratch of the same shape.
// Pass 1: lane r transforms storage row r (SW-point IDCT in registers). Pass 2: lane j transforms column j (SH-point) and writes
// pixels: a contiguous run of SH floats per lane when the block is at least as tall as wide, one coalesced row per step otherwise.
template <int SW, int SH>
__device__ __forceinline__ void InverseSeparable(const float* S, float* T, float* out, size_t xpad, bool tall, int lane) {
  constexpr int STR = SW + 4;
  if (lane < SH) {
    float X[SW], y[SW];
#pragma unroll
    for (int k = 0; k < SW; k += 4) { const float4 v = *reinterpret_cast<const float4*>(S + lane * STR + k); X[k] = v.x; X[k + 1] = v.y; X[k + 2] = v.z; X[k + 3] = v.w; }
    IdctN<SW>::Run(X, y);
#pragma unroll
    for (int k = 0; k < SW; k += 4) *reinterpret_cast<float4*>(T + lane * STR + k) = make_float4(y[k], y[k + 1], y[k + 2], y[k + 3]);
  }
  __syncwarp();
  if (lane < SW) {
    float X[SH], y[SH];
#pragma unroll
    for (int r = 0; r < SH; r++) X[r] = T[r * STR + lane];
    IdctN<SH>::Run(X, y);
    if (tall) {   // long axis vertical: lane = pixel row, y[] runs along x
#pragma unroll
      for (int i = 0; i < SH; i += 4) *reinterpret_cast<float4*>(out + size_t(lane) * xpad + i) = make_float4(y[i], y[i + 1], y[i + 2], y[i + 3]);
    } else {      // long axis horizontal: lane = pixel column, y[] runs along y
#pragma unroll
      for (int i = 0; i < SH; i++) out[size_t(i) * xpad + lane] = y[i];
    }
  }
  __syncwarp();
}

// Dequant + chroma-from-luma + LLF + 8x8 IDCT for every DCT8 varblock. A work item is one row of 32 cells of a 256x256 group; a CTA of
// 8 warps walks items with a grid stride (persistent: the grid is a multiple of the SM count).
//   phase A  thread (cell, storage row r): one 16-byte load per channel (8 int16 coefficients; a cell's 3 x 128 bytes are contiguous, a
//            warp reads 16 cells x 2 rows = full 32-byte sectors), dequantise + CfL in registers, 8-point IDCT along the row, two
//            STS.128 into a [cell][68] transposition buffer. Warps own a row PAIR, so the high-frequency pairs, which are all zero in
//            most cells, skip the arithmetic warp-uniformly.
//   phase B  thread (channel, half of the pixel rows, cell): eight LDS.128 (four pixel rows of the column-transformed block), four
//            8-point IDCTs, and per pixel row two float4 stores: a warp writes 32 cells x 32 bytes = 1 KB contiguous per pixel row.
// The buffer is double-buffered, so an item costs one __syncthreads. Everything the next item reads from global memory is requested
// before the current one is transformed. 6 B/px read (int16 coefficients) + 12 B/px written (fp32 XYB) = 18 algorithmic bytes per pixel.
static const int kD8Stride = 68;   // floats per cell in the transposition buffer: 64 + 4, so 8 consecutive cells hit 8 different 16-byte bank groups
__global__ void __launch_bounds__(256, 3) k_reconstruct_dct8(const __grid_constant__ DFrame f, const int num_items) {
  extern __shared__ __align__(16) float s_t_raw[];   // [2 buffers][3 channels][32 cells * kD8Stride] (dynamic: 51 KB)
  float (*s_t)[3][32 * kD8Stride] = reinterpret_cast<float (*)[3][32 * kD8Stride]>(s_t_raw);
  __shared__ __align__(16) float s_dq[192];
  __shared__ uint8_t s_valid[2][32];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int bxA = (warp >> 2) * 16 + (lane & 15), rA = (warp & 3) * 2 + (lane >> 4);   // phase A role
  const int cB = warp % 3, yhalf = warp / 3;                                            // phase B role (warps 0..5), cell = lane
  if (tid < 192) s_dq[tid] = reinterpret_cast<const float*>(BlobAt(f, f.dq_off[0]))[tid];
  __syncthreads();
  const size_t plane = size_t(f.xpad) * f.ypad, lfplane = size_t(f.xb) * f.yb;
  struct Pre { int4 raw[3]; float lf[3]; int acs, hf, tx, tb; };
  auto geometry = [&](int item, int& cx0, int& cy0, int& by, int& w) -> bool {
    const int g = item >> 5; by = item & 31; const int gx = g % int(f.xgroups), gy = g / int(f.xgroups); cx0 = gx * 32; cy0 = gy * 32;
    w = min(32, int(f.xb) - cx0); return by < min(32, int(f.yb) - cy0) && GroupInBand(f, g);
  };
  auto fetch = [&](int item, Pre& p) {
    p.raw[0] = p.raw[1] = p.raw[2] = make_int4(0, 0, 0, 0); p.lf[0] = p.lf[1] = p.lf[2] = 0.f; p.acs = 0; p.hf = 0; p.tx = 0; p.tb = 0;
    int cx0, cy0, by, w; if (item >= num_items || !geometry(item, cx0, cy0, by, w) || bxA >= w) return;
    const size_t o = size_t(cy0 + by) * f.xb + cx0 + bxA, tile = size_t((cy0 + by) >> 3) * f.xt + ((cx0 + bxA) >> 3);
    const int16_t* cp = f.coeffs + size_t(item >> 5) * 3 * 65536 + (by * 32 + bxA) * 64 + rA * 8;
    p.raw[0] = __ldcs(reinterpret_cast<const int4*>(cp)); p.raw[1] = __ldcs(reinterpret_cast<const int4*>(cp + 65536)); p.raw[2] = __ldcs(reinterpret_cast<const int4*>(cp + 2 * 65536));
    p.acs = f.acs[o]; p.hf = f.hf_mul_m1[o]; p.tx = f.ytox[tile]; p.tb = f.ytob[tile];
    if (rA == 0) { p.lf[0] = f.lf_src[o]; p.lf[1] = f.lf_src[lfplane + o]; p.lf[2] = f.lf_src[2 * lfplane + o]; }
  };
  Pre cur; fetch(blockIdx.x, cur);
  int buf = 0;
#pragma unroll 1
  for (int item = blockIdx.x; item < num_items; item += gridDim.x, buf ^= 1) {
    Pre nxt; fetch(item + int(gridDim.x), nxt);
    int cx0, cy0, by, w; const bool row_ok = geometry(item, cx0, cy0, by, w);
    if (!row_ok) { cur = nxt; continue; }   // uniform over the CTA
    // ---- phase A
    const bool valid = bxA < w && cur.acs == 0x80;   // strategy 0 (DCT8), first (only) cell
    if (rA == 0) s_valid[buf][bxA] = valid ? 1 : 0;
    const bool any = valid && (((cur.raw[0].x | cur.raw[0].y | cur.raw[0].z | cur.raw[0].w | cur.raw[1].x | cur.raw[1].y | cur.raw[1].z | cur.raw[1].w | cur.raw[2].x | cur.raw[2].y | cur.raw[2].z | cur.raw[2].w) != 0) || rA == 0);
    const bool warp_any = __any_sync(0xffffffffu, any);   // voted by every lane, before the lanes of other strategies drop out
    if (valid) {
      const float scale = f.inv_gs / float(cur.hf + 1), kx = f.base_x + float(cur.tx) * f.inv_color_factor, kb = f.base_b + float(cur.tb) * f.inv_color_factor;
      float* dst = &s_t[buf][0][bxA * kD8Stride + rA * 8];
      if (!warp_any) {   // the whole row pair of these 16 cells is zero: the row transform of zeros is zeros
        const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int c = 0; c < 3; c++) { *reinterpret_cast<float4*>(dst + c * 32 * kD8Stride) = z; *reinterpret_cast<float4*>(dst + c * 32 * kD8Stride + 4) = z; }
      } else {
        float y8[8];
#pragma unroll
        for (int ci = 0; ci < 3; ci++) {
          const int c = ci == 0 ? 1 : ci == 1 ? 0 : 2; float v[8], t[8];
          const int4 raw = cur.raw[c];
          const int q[8] = {int(short(raw.x & 0xffff)), raw.x >> 16, int(short(raw.y & 0xffff)), raw.y >> 16, int(short(raw.z & 0xffff)), raw.z >> 16, int(short(raw.w & 0xffff)), raw.w >> 16};
          const float mulc = c == 1 ? scale : c == 0 ? scale * f.xm : scale * f.bm, kc = c == 0 ? kx : kb, b1 = f.quant_bias[c], b3 = f.quant_bias[3];
          const float4 d0 = *reinterpret_cast<const float4*>(&s_dq[c * 64 + rA * 8]), d1 = *reinterpret_cast<const float4*>(&s_dq[c * 64 + rA * 8 + 4]);
          const float dq[8] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w};
#pragma unroll
          for (int j = 0; j < 8; j++) {
            const float qf = float(q[j]);   // quantisation-bias adjustment: 0 -> 0, +-1 -> +-b1, else q - b3 / q
            const float adj = fabsf(qf) >= 1.5f ? qf - __fdividef(b3, qf) : qf * b1;
            float a = adj * dq[j] * mulc; if (c == 1) y8[j] = a; else a = fmaf(kc, y8[j], a); v[j] = a;
          }
          if (rA == 0) v[0] = cur.lf[c];   // LLF of an 8x8 block is the LF sample itself
          Idct8(v, t);
          *reinterpret_cast<float4*>(dst + c * 32 * kD8Stride) = make_float4(t[0], t[1], t[2], t[3]);
          *reinterpret_cast<float4*>(dst + c * 32 * kD8Stride + 4) = make_float4(t[4], t[5], t[6], t[7]);
        }
      }
    }
    __syncthreads();
    // ---- phase B
    if (warp < 6 && lane < w && s_valid[buf][lane]) {
      const float* src = &s_t[buf][cB][lane * kD8Stride + yhalf * 4];
      float4 in[8];
#pragma unroll
      for (int hf = 0; hf < 8; hf++) in[hf] = *reinterpret_cast<const float4*>(src + hf * 8);
      float* out = f.xyb + cB * plane + (size_t(cy0 + by) * 8 + yhalf * 4) * f.xpad + size_t(cx0 + lane) * 8;
#pragma unroll
      for (int yy = 0; yy < 4; yy++) {
        float X[8], px[8];
#pragma unroll
        for (int hf = 0; hf < 8; hf++) X[hf] = yy == 0 ? in[hf].x : yy == 1 ? in[hf].y : yy == 2 ? in[hf].z : in[hf].w;
        Idct8(X, px);
        __stcs(reinterpret_cast<float4*>(out + size_t(yy) * f.xpad), make_float4(px[0], px[1], px[2], px[3]));
        __stcs(reinterpret_cast<float4*>(out + size_t(yy) * f.xpad + 4), make_float4(px[4], px[5], px[6], px[7]));
      }
    }
    cur = nxt;
  }
}

static const int kReconWarps = 8;
// Two instantiations, launched one after the other: kSide = 16 takes the varblocks whose longer side is at most 16 px (DCT16x16, 16x8, 8x16 and
// the 8x8 special transforms: up to 85 registers, 3.8 KB of shared memory per warp, 3 CTAs per SM), kSide = 32 the 32-px ones and the >= 64-px pass
// (128 registers for the 32-point IDCT, 2 CTAs per SM). One kernel for both ran everything at the occupancy of the widest transform.
template <int kSide>
__global__ void __launch_bounds__(kReconWarps * 32, kSide == 16 ? 3 : 2) k_reconstruct(const DFrame* fp) {
  const DFrame& f = *fp; const int g = blockIdx.x >> 2, quarter = blockIdx.x & 3, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;   // four CTAs share a group's small varblocks
  if (!GroupInBand(f, g) || f.group_other[g] == 0) return;   // every varblock of this group is a DCT8: k_reconstruct_dct8 did all the work
  const int gx = g % int(f.xgroups), gy = g / int(f.xgroups), cx0 = gx * 32, cy0 = gy * 32, w = min(32, int(f.xb) - cx0), h = min(32, int(f.yb) - cy0);
  constexpr int kBuf = kSide * (kSide + 4);   // floats per buffer: kSide rows of kSide + 4
  extern __shared__ __align__(16) float smem[]; float* Sy = smem + warp * 3 * kBuf; float* Sc = Sy + kBuf; float* T = Sc + kBuf;   // per warp: Sy, Sc, T
  const int16_t* coef = f.coeffs + size_t(g) * 3 * 65536; const size_t plane = size_t(f.xpad) * f.ypad, lfplane = size_t(f.xb) * f.yb; const DTables& tb = *f.tables;
  // ---- small varblocks (both sides <= 32 px): one warp per block. Separable DCTs of 8/16/32 points run as register-resident straight-line
  // code (InverseSeparable); the 8x8 special transforms (IDENTITY, DCT2X2, DCT4X4, DCT4X8, DCT8X4) are rare and stay with lane 0.
  // A warp owns one row of 32 cells: the lanes read the row's strategy bytes with one coalesced load and vote which cells start a small
  // non-DCT8 varblock (a serial scan would pay one dependent global load per cell), then the warp works through the set bits.
  const int by = quarter * kReconWarps + warp;
  uint32_t my_a = 0;
  if (by < h && lane < w) my_a = f.acs[size_t(cy0 + by) * f.xb + cx0 + lane];
  { const int ms = min(int(my_a & 31), 26); const uint32_t lx = CoveredXLog2Dev(ms), ly = CoveredYLog2Dev(ms); const bool wide32 = lx == 2 || ly == 2;
    const bool cand = (my_a & 0x80) && ms != 0 && lx <= 2 && ly <= 2 && wide32 == (kSide == 32); if (!cand) my_a = 0; }
  uint32_t todo = __ballot_sync(0xffffffffu, my_a != 0);
  while (todo) {
    const int bx = __ffs(int(todo)) - 1; todo &= todo - 1;
    const uint32_t a = __shfl_sync(0xffffffffu, my_a, bx);
    const size_t o = size_t(cy0 + by) * f.xb + cx0 + bx;
    const int s = min(int(a & 31), 26), bw = 1 << CoveredXLog2Dev(s), bh = 1 << CoveredYLog2Dev(s);
    const int size = bw * bh * 64, H = bh * 8, W = bw * 8, SW = max(H, W), SH = min(H, W), STR = (s >= 4 && s <= 11) ? SW + 4 : SW; const float* dq = reinterpret_cast<const float*>(BlobAt(f, f.dq_off[QuantTableOf(s)]));
    const float scale = f.inv_gs / float(int(f.hf_mul_m1[o]) + 1); const size_t tile = size_t((cy0 + by) / 8) * f.xt + (cx0 + bx) / 8;
    const float kx = f.base_x + float(f.ytox[tile]) * f.inv_color_factor, kb = f.base_b + float(f.ytob[tile]) * f.inv_color_factor;
    const bool plain = s >= 4 && s <= 11; const int lsw = Log2Dev(SW);
    for (int c3 = 0; c3 < 3; c3++) {
      const int c = c3 == 0 ? 1 : c3 == 1 ? 0 : 2; float* S = c == 1 ? Sy : Sc;
      const float mulc = c == 1 ? scale : c == 0 ? scale * f.xm : scale * f.bm, kc = c == 0 ? kx : kb, b1 = f.quant_bias[c], b3 = f.quant_bias[3];
      if (plain) {   // 8 coefficients per lane and step: one 16-byte coefficient load, two 16-byte table loads, two STS.128
        for (int p8 = lane * 8; p8 < size; p8 += 256) {
          const int j = p8 >> 6, sp = (p8 >> lsw) * STR + (p8 & (SW - 1));
          const int4 raw = *reinterpret_cast<const int4*>(coef + c * 65536 + ((by + j / bw) * 32 + bx + j % bw) * 64 + (p8 & 63));
          const float4 d0 = *reinterpret_cast<const float4*>(dq + c * size + p8), d1 = *reinterpret_cast<const float4*>(dq + c * size + p8 + 4);
          const int q[8] = {int(short(raw.x & 0xffff)), raw.x >> 16, int(short(raw.y & 0xffff)), raw.y >> 16, int(short(raw.z & 0xffff)), raw.z >> 16, int(short(raw.w & 0xffff)), raw.w >> 16};
          const float dd[8] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w}; float v[8];
#pragma unroll
          for (int k = 0; k < 8; k++) { const float qf = float(q[k]); const float adj = fabsf(qf) >= 1.5f ? qf - __fdividef(b3, qf) : qf * b1; v[k] = adj * dd[k] * mulc; }
          if (c != 1) { const float4 y0 = *reinterpret_cast<const float4*>(Sy + sp), y1 = *reinterpret_cast<const float4*>(Sy + sp + 4);
            v[0] = fmaf(kc, y0.x, v[0]); v[1] = fmaf(kc, y0.y, v[1]); v[2] = fmaf(kc, y0.z, v[2]); v[3] = fmaf(kc, y0.w, v[3]); v[4] = fmaf(kc, y1.x, v[4]); v[5] = fmaf(kc, y1.y, v[5]); v[6] = fmaf(kc, y1.z, v[6]); v[7] = fmaf(kc, y1.w, v[7]); }
          *reinterpret_cast<float4*>(S + sp) = make_float4(v[0], v[1], v[2], v[3]); *reinterpret_cast<float4*>(S + sp + 4) = make_float4(v[4], v[5], v[6], v[7]);
        }
      } else for (int p = lane; p < size; p += 32) { const int sp = (p >> lsw) * STR + (p & (SW - 1)); int q = coef[c * 65536 + CoefAddr(by, bx, bw, uint32_t(p))];
        float v = AdjustQuantBiasDev(q, b1, b3) * dq[c * size + p] * mulc; if (c != 1) v += kc * Sy[sp]; S[sp] = v; }
      __syncwarp();
      LlfFromLf(f, c, bh, bw, f.lf_src + c * lfplane + o, int(f.xb), S, STR, lane, 32);
      __syncwarp();
      float* out = f.xyb + c * plane + size_t(cy0 + by) * 8 * f.xpad + size_t(cx0 + bx) * 8;
      if (plain) {
        const bool tall = H >= W;
        if (kSide == 16) { if (SH == 16) InverseSeparable<16, 16>(S, T, out, f.xpad, tall, lane); else InverseSeparable<16, 8>(S, T, out, f.xpad, tall, lane); }
        else if (SH == 32) InverseSeparable<32, 32>(S, T, out, f.xpad, tall, lane);
        else if (SH == 8) InverseSeparable<32, 8>(S, T, out, f.xpad, tall, lane);
        else InverseSeparable<32, 16>(S, T, out, f.xpad, tall, lane);
      } else if (s >= 14 && s <= 17) { if (lane == 0) SetError(f.err, kErrBadStrategy); }
      else if (lane == 0) SpecialTransform8x8(s, S, out, f.xpad, tb.cosines + CosOff(2), tb.cosines + CosOff(3));   // 8x8 block, unpadded rows (STR = 8)
      __syncwarp();
    }
  }
  if (kSide != 32 || quarter != 0 || (f.group_other[g] >> 16) == 0) return;   // high half of group_other: number of varblocks with a side of 64 px or more (uniform over the CTA, so no barrier is skipped by part of it)
  __syncthreads();
  // ---- large varblocks (a side >= 64 px): the whole CTA per block, staged through the XYB planes themselves (first of the group's four CTAs)
  const int NT = kReconWarps * 32;
  for (int cell = 0; cell < 1024; cell++) {
    const int by = cell >> 5, bx = cell & 31; if (by >= h || bx >= w) continue;
    const size_t o = size_t(cy0 + by) * f.xb + cx0 + bx; const uint8_t a = f.acs[o]; if (!(a & 0x80)) continue;
    const int s = min(int(a & 31), 26), bw = 1 << CoveredXLog2Dev(s), bh = 1 << CoveredYLog2Dev(s); if (bw <= 4 && bh <= 4) continue;
    const int size = bw * bh * 64, H = bh * 8, W = bw * 8, SW = max(H, W), SH = min(H, W); const float* dq = reinterpret_cast<const float*>(BlobAt(f, f.dq_off[QuantTableOf(s)]));
    const float scale = f.inv_gs / float(int(f.hf_mul_m1[o]) + 1); const size_t tile = size_t((cy0 + by) / 8) * f.xt + (cx0 + bx) / 8;
    const float kx = f.base_x + float(f.ytox[tile]) * f.inv_color_factor, kb = f.base_b + float(f.ytob[tile]) * f.inv_color_factor;
    const size_t base = size_t(cy0 + by) * 8 * f.xpad + size_t(cx0 + bx) * 8;
    // stage 0: dequantised coefficients, storage position p kept at linear index p of the block's pixel rect (in xyb_tmp)
    for (int p = tid; p < size; p += NT) { uint32_t ad = CoefAddr(by, bx, bw, uint32_t(p)); size_t dst = base + size_t(p / W) * f.xpad + p % W;
      float y = AdjustQuantBiasDev(coef[65536 + ad], f.quant_bias[1], f.quant_bias[3]) * dq[size + p] * scale;
      float x = AdjustQuantBiasDev(coef[ad], f.quant_bias[0], f.quant_bias[3]) * dq[p] * (scale * f.xm) + kx * y;
      float b = AdjustQuantBiasDev(coef[2 * 65536 + ad], f.quant_bias[2], f.quant_bias[3]) * dq[2 * size + p] * (scale * f.bm) + kb * y;
      f.xyb_tmp[dst] = x; f.xyb_tmp[plane + dst] = y; f.xyb_tmp[2 * plane + dst] = b; }
    __syncthreads();
    {  // LLF corner
      const int ly = Log2Dev(bh), lx = Log2Dev(bw); const float* cv = tb.cosines + CosOff(ly); const float* ch = tb.cosines + CosOff(lx);
      for (int idx = tid; idx < 3 * bh * bw; idx += NT) { int c = idx / (bh * bw), r = idx % (bh * bw), v = r / bw, hfr = r % bw; const float* lfp = f.lf_src + c * lfplane + o; float acc = 0;
        for (int y = 0; y < bh; y++) { float ra = 0; for (int x = 0; x < bw; x++) ra += lfp[size_t(y) * f.xb + x] * ch[hfr * bw + x]; acc += ra * cv[v * bh + y]; }
        float val = acc / float(bh * bw) * tb.resample[ly][v] * tb.resample[lx][hfr]; int p = bh < bw ? v * SW + hfr : hfr * SW + v;
        f.xyb_tmp[c * plane + base + size_t(p / W) * f.xpad + p % W] = val; }
    }
    __syncthreads();
    const float* cl = tb.cosines + CosOff(Log2Dev(SW)); const float* cs = tb.cosines + CosOff(Log2Dev(SH));
    for (int c = 0; c < 3; c++) {   // pass A: along the long axis, xyb_tmp -> xyb (linear index = r*SW + j)
      for (int idx = tid; idx < size; idx += NT) { int r = idx / SW, j = idx % SW; float acc = 0;
        for (int k = 0; k < SW; k++) { int p = r * SW + k; acc += f.xyb_tmp[c * plane + base + size_t(p / W) * f.xpad + p % W] * cl[k * SW + j]; }
        f.xyb[c * plane + base + size_t(idx / W) * f.xpad + idx % W] = acc; }
    }
    __syncthreads();
    for (int c = 0; c < 3; c++) {   // pass B: along the short axis, xyb -> xyb_tmp at final pixel positions
      for (int idx = tid; idx < size; idx += NT) { int i = idx / SW, j = idx % SW; float acc = 0;
        for (int r = 0; r < SH; r++) { int p = r * SW + j; acc += f.xyb[c * plane + base + size_t(p / W) * f.xpad + p % W] * cs[r * SH + i]; }
        int py = H >= W ? j : i, pxx = H >= W ? i : j; f.xyb_tmp[c * plane + base + size_t(py) * f.xpad + pxx] = acc; }
    }
    __syncthreads();
    for (int c = 0; c < 3; c++) for (int idx = tid; idx < size; idx += NT) { size_t ad = c * plane + base + size_t(idx / W) * f.xpad + idx % W; f.xyb[ad] = f.xyb_tmp[ad]; }
    __syncthreads();
  }
}

// ------------------------------------------------------------------ restoration filters
__device__ __forceinline__ int MirrorDev(int x, int n) { while (x < 0 || x >= n) { if (x < 0) x = -x - 1; else x = 2 * n - 1 - x; } return x; }

__global__ void k_inv_sigma(const DFrame* fp) {
  const DFrame& f = *fp; size_t n = size_t(f.xb) * f.yb; size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; if (i >= n) return;
  const float kInvSigmaNum = -1.1715728752538099024f;
  if (f.encoding == 1) { f.inv_sigma[i] = kInvSigmaNum / f.lpf.sigma_for_modular; return; }
  float sigma_quant = f.lpf.epf_quant_mul / (f.quant_scale * float(int(f.hf_mul_m1[i]) + 1) * kInvSigmaNum);
  float sigma = fminf(-1e-4f, sigma_quant * f.lpf.epf_sharp_lut[f.sharp[i]]); f.inv_sigma[i] = 1.0f / sigma;
}

__global__ void k_gaborish(const DFrame* fp, const float* __restrict__ src, float* __restrict__ dst) {
  const DFrame& f = *fp; const int xs = int(f.xsize), ys = int(f.ysize); const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y; if (x >= xs || y >= ys) return;
  const size_t plane = size_t(f.xpad) * f.ypad; const int yu = MirrorDev(y - 1, ys), yd = MirrorDev(y + 1, ys), xl = MirrorDev(x - 1, xs), xr = MirrorDev(x + 1, xs);
#pragma unroll
  for (int c = 0; c < 3; c++) { const float* p = src + c * plane; const float* t = p + size_t(yu) * f.xpad; const float* m = p + size_t(y) * f.xpad; const float* b = p + size_t(yd) * f.xpad;
    float w1 = f.lpf.gab_w[2 * c], w2 = f.lpf.gab_w[2 * c + 1]; float mul = 1.0f / (1.0f + 4.0f * (w1 + w2));
    dst[c * plane + size_t(y) * f.xpad + x] = m[x] * mul + (t[x] + b[x] + m[xl] + m[xr]) * (w1 * mul) + (t[xl] + t[xr] + b[xl] + b[xr]) * (w2 * mul); }
}

// ------------------------------------------------------------------ inverse RCT on the global Modular image
__global__ void k_inverse_rct(const DFrame* fp, uint32_t op_index) {
  const DFrame& f = *fp; const DModOp& op = ModOp(f, op_index); const uint32_t type = op.rct_type; const size_t n = size_t(op.w) * op.h; size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; if (i >= n) return;
  int32_t* p0 = f.mod_planes + op.p[0]; int32_t* p1 = f.mod_planes + op.p[1]; int32_t* p2 = f.mod_planes + op.p[2];
  uint32_t perm = type / 7, k = type % 7; int32_t A = p0[i], B = p1[i], C = p2[i], o[3];
  if (k == 6) { int32_t t = A - (C >> 1); int32_t G = C + t; int32_t Bl = t - (B >> 1); int32_t R = Bl + B; o[0] = R; o[1] = G; o[2] = Bl; }
  else { int32_t D = A, E = B, F = C; if (k & 1) F += A; if ((k >> 1) == 1) E += A; if ((k >> 1) == 2) E += (A + F) >> 1; o[0] = D; o[1] = E; o[2] = F; }
  int32_t r[3]; r[perm % 3] = o[0]; r[(perm + 1 + perm / 3) % 3] = o[1]; r[(perm + 2 - perm / 3) % 3] = o[2];
  p0[i] = r[0]; p1[i] = r[1]; p2[i] = r[2];
}

// ------------------------------------------------------------------ inverse Palette on the global Modular image (SURVEY.md A.7 "Palette")
// Index -> colour: explicit entries [0, pal_w), then the implicit 4x4x4 cube (64 entries, offset by 2^(bitdepth-3)) and the implicit 5x5x5
// cube. Negative indices address the 72-entry delta palette, whose table is not available offline: they raise kErrPaletteDelta.
__device__ __forceinline__ int32_t PaletteValue(const int32_t* pal_row, int index, int c, int pal_w, int bitdepth, uint32_t* err) {
  bool bad = false; const int32_t v = PaletteLookup(pal_row, index, c, pal_w, bitdepth, &bad); if (bad) SetError(err, kErrPaletteDelta); return v;
}
// Pure gather: one thread per sample and output channel (blockIdx.y). Used when the palette has no delta entries.
__global__ void k_inverse_palette(const DFrame* fp, uint32_t op_index) {
  const DFrame& f = *fp; const DModOp& op = ModOp(f, op_index); const size_t n = size_t(op.w) * op.h; const size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; if (i >= n) return;
  const int c = blockIdx.y; const int32_t* idx = f.mod_planes + op.p[0]; const int32_t* pal = f.mod_planes + op.p[1] + size_t(c) * op.pal_w;
  f.mod_planes[op.out[c] + i] = PaletteValue(pal, idx[i], c, int(op.pal_w), int(f.mod_bitdepth), f.err);
}
// Palettes with delta entries (index < nb_deltas: the entry is ADDED to a prediction from the already reconstructed neighbours of the same
// output channel): serial in raster order, one thread per output channel. A rare path (lossy-palette files); correctness only.
__global__ void k_inverse_palette_delta(const DFrame* fp, uint32_t op_index) {
  const DFrame& f = *fp; const DModOp& op = ModOp(f, op_index); const int c = blockIdx.x; if (threadIdx.x) return;
  const int32_t* idx = f.mod_planes + op.p[0]; const int32_t* pal = f.mod_planes + op.p[1] + size_t(c) * op.pal_w; int32_t* out = f.mod_planes + op.out[c]; const int w = int(op.w), h = int(op.h);
  for (int y = 0; y < h; y++) for (int x = 0; x < w; x++) {
    const int index = idx[size_t(y) * w + x]; int32_t v = PaletteValue(pal, index, c, int(op.pal_w), int(f.mod_bitdepth), f.err);
    if (index >= 0 && index < int(op.nb_deltas)) {
      const int32_t* p = out + size_t(y) * w + x;
      const long long W = x ? p[-1] : (y ? p[-w] : 0), N = y ? p[-w] : W, NW = (x && y) ? p[-w - 1] : W, NE = (y && x + 1 < w) ? p[-w + 1] : N, NN = y > 1 ? p[-2 * w] : N, WW = x > 1 ? p[-2] : W, NEE = (y && x + 2 < w) ? p[-w + 2] : NE;
      v = int32_t(v + ModMath<long long>::Prediction(int(op.predictor), N, W, NW, NE, NN, WW, NEE, 0));
    }
    out[size_t(y) * w + x] = v;
  }
}

// ------------------------------------------------------------------ output
// a^e for a >= 0 through the SFU (lg2 + ex2): relative error of a few 1e-7 here (|e * log2 a| < 16), far inside the 1-LSB / 1e-4 bounds
// of the output formats; libm powf costs ~70 instructions per call and was 29 % of the fused kernel's issue slots (profiles/).
__device__ __forceinline__ float PowSfu(float a, float e) {   // lg2(0) = -inf -> ex2(-inf) = +0: no branch needed for a == 0 (e > 0)
  float l, r; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l) : "f"(a)); asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(l * e)); return r; }
__device__ __forceinline__ float TfFromLinearDev(float v, uint32_t tf, float gamma, float intensity_target) {
  float a = fabsf(v), r;
  switch (tf) {
    case 0: r = PowSfu(a, gamma); break;
    case 8: r = a; break;
    case 13: r = a <= 0.0031308f ? 12.92f * a : 1.055f * PowSfu(a, 1.0f / 2.4f) - 0.055f; break;
    case 1: r = a < 0.018f ? 4.5f * a : 1.099f * PowSfu(a, 0.45f) - 0.099f; break;
    // PQ in double: the outer exponent (78.84) multiplies every fp32 rounding of the ratio by ~80, which alone is 1e-5..1e-4 relative on the code value
    case 16: { const double m1 = 2610.0 / 16384, m2 = 2523.0 / 4096 * 128, c1 = 3424.0 / 4096, c2 = 2413.0 / 4096 * 32, c3 = 2392.0 / 4096 * 32;
      const double yv = fmin(1.0, double(a) * double(intensity_target) / 10000.0); const double p = pow(yv, m1); r = float(pow((c1 + c2 * p) / (1.0 + c3 * p), m2)); break; }
    case 17: r = PowSfu(a, 1.0f / 2.6f); break;
    case 18: r = a <= 1.0f / 12 ? sqrtf(3.0f * a) : 0.17883277f * logf(12.0f * a - 0.28466892f) + 0.55991073f; break;   // HLG OETF (ARIB STD-B67), no OOTF: the file's own encoding
    default: r = a; break;
  }
  return v < 0 ? -r : r;
}
__device__ __forceinline__ float IntToFloatSampleDev(int32_t v, uint32_t bits, uint32_t exp_bits) {
  if (exp_bits == 0) return float(double(v) / double((1ull << bits) - 1));
  if (bits == 32 && exp_bits == 8) return __int_as_float(v);
  int mant_bits = int(bits) - int(exp_bits) - 1; uint32_t u = uint32_t(v); bool sign = (u >> (bits - 1)) & 1; u &= (1u << (bits - 1)) - 1; if (u == 0) return sign ? -0.f : 0.f;
  int e = int(u >> mant_bits); uint32_t mant = u & ((1u << mant_bits) - 1); int bias = (1 << (exp_bits - 1)) - 1; double r;
  if (e == 0) r = ldexp(double(mant), 1 - bias - mant_bits); else r = ldexp(double(mant | (1u << mant_bits)), e - bias - mant_bits);
  return float(sign ? -r : r);
}
__device__ __forceinline__ void StoreSampleDev(uint8_t* dst, uint32_t type, float v) {
  switch (type) {
    case 0: *dst = uint8_t(__float2int_rn(fminf(1.f, fmaxf(0.f, v)) * 255.0f)); break;
    case 1: *reinterpret_cast<uint16_t*>(dst) = uint16_t(__float2int_rn(fminf(1.f, fmaxf(0.f, v)) * 65535.0f)); break;
    case 2: *reinterpret_cast<__half*>(dst) = __float2half_rn(v); break;
    default: *reinterpret_cast<float*>(dst) = v; break;
  }
}
// (x,y) in decoded frame coordinates -> element index in the oriented output image
__device__ __forceinline__ size_t OrientedIndex(const DFrame& f, int x, int y) {
  const int W = int(f.xsize), H = int(f.ysize); int ox, oy;
  switch (f.out.orientation) { case 2: ox = W - 1 - x; oy = y; break; case 3: ox = W - 1 - x; oy = H - 1 - y; break; case 4: ox = x; oy = H - 1 - y; break;
    case 5: ox = y; oy = x; break; case 6: ox = H - 1 - y; oy = x; break; case 7: ox = H - 1 - y; oy = W - 1 - x; break; case 8: ox = y; oy = W - 1 - x; break; default: ox = x; oy = y; }
  return size_t(oy - int(f.out_y0)) * f.out.out_w + ox;   // out_y0: first output row of a band decode (0 otherwise; bands need orientation 1)
}

// Colour + sample conversion + store of one pixel. For VarDCT frames (X,Y,B) are the filtered XYB samples.
// XYB -> target-encoded RGB of one VarDCT sample (shared by every output path, so they agree bit for bit)
__device__ __forceinline__ void XybToRgbDev(const DFrame& f, float X, float Y, float B, float rgb[3]) {
    float gm[3] = {Y + X, Y - X, B}, mix[3];
#pragma unroll
    for (int c = 0; c < 3; c++) { float v = gm[c] - f.color.opsin_bias_cbrt[c]; mix[c] = v * v * v + f.color.opsin_bias[c]; }
    float lin[6];   // lin[3..5]: linear light in the target primaries (opsin inverse, intensity scale and primaries change are one matrix)
#pragma unroll
    for (int c = 0; c < 3; c++) lin[c + 3] = fmaf(f.color.mix_to_target[3 * c], mix[0], fmaf(f.color.mix_to_target[3 * c + 1], mix[1], f.color.mix_to_target[3 * c + 2] * mix[2]));
    if (f.color.tf == 13) {   // sRGB curve, the common case: branch-free per channel
#pragma unroll
      for (int c = 0; c < 3; c++) { const float v = lin[c + 3], a = fabsf(v), r = a <= 0.0031308f ? 12.92f * a : 1.055f * PowSfu(a, 1.0f / 2.4f) - 0.055f; rgb[c] = v < 0 ? -r : r; }
    } else {
#pragma unroll
      for (int c = 0; c < 3; c++) rgb[c] = TfFromLinearDev(lin[c + 3], f.color.tf, f.color.gamma, f.color.intensity_target);
    }
}
__device__ __forceinline__ void OutputPixel(const DFrame& f, int x, int y, float X, float Y, float B) {
  const DOutput& o = f.out; float rgb[3];
  if (f.encoding == 0) XybToRgbDev(f, X, Y, B, rgb);
  else {
    const uint32_t nc = f.color.num_color;
    for (uint32_t c = 0; c < 3; c++) { const DModChannel& ch = f.out_ch[c < nc ? c : nc - 1]; rgb[c] = IntToFloatSampleDev(f.mod_planes[ch.plane_off + size_t(y) * ch.w + x], o.bits, o.exp_bits); }
  }
  float a = 1.0f;
  if (o.alpha_plane >= 0) { const DModChannel& ch = f.out_ch[o.alpha_plane]; int sx = min(x >> ch.hshift, int(ch.w) - 1), sy = min(y >> ch.vshift, int(ch.h) - 1); a = IntToFloatSampleDev(f.mod_planes[ch.plane_off + size_t(sy) * ch.w + sx], o.alpha_bits, o.alpha_exp_bits); }
  if (o.premultiplied) { float mul = 1.0f / fmaxf(1.0f / 67108864.0f, a); rgb[0] *= mul; rgb[1] *= mul; rgb[2] *= mul; }
  const size_t oi = OrientedIndex(f, x, y);
  if (o.bgra) {   // BGRA32 surface: B,G,R from the 8-bit conversion, A = alpha plane mapped to 8 bits (I/TransparencyMapping.cs:19-32) or 255
    uint8_t r8 = uint8_t(__float2int_rn(fminf(1.f, fmaxf(0.f, rgb[0])) * 255.0f)), g8 = uint8_t(__float2int_rn(fminf(1.f, fmaxf(0.f, rgb[1])) * 255.0f)), b8 = uint8_t(__float2int_rn(fminf(1.f, fmaxf(0.f, rgb[2])) * 255.0f));
    if (o.color_channels == 1) { g8 = r8; b8 = r8; }
    uint8_t a8 = 255; if (o.alpha_plane >= 0) a8 = uint8_t(__float2int_rn(fminf(1.f, fmaxf(0.f, a)) * 255.0f));
    reinterpret_cast<uint32_t*>(f.out_px)[oi] = uint32_t(b8) | (uint32_t(g8) << 8) | (uint32_t(r8) << 16) | (uint32_t(a8) << 24); return;
  }
  const uint32_t bps = o.sample_type == 0 ? 1 : o.sample_type == 3 ? 4 : 2; uint8_t* dst = f.out_px + oi * size_t(bps) * (o.num_channels + (o.black_plane >= 0 ? 1 : 0));
  if (o.black_plane >= 0) {   // CMYK merge, N/Decoder/JxlDecoder.cpp:159-215 (u8 only): 255 - C,M,Y,K then optional A
    const DModChannel& ch = f.out_ch[o.black_plane]; float k = IntToFloatSampleDev(f.mod_planes[ch.plane_off + size_t(min(y >> ch.vshift, int(ch.h) - 1)) * ch.w + min(x >> ch.hshift, int(ch.w) - 1)], o.black_bits, 0);
    uint8_t t[4]; for (int c = 0; c < 3; c++) StoreSampleDev(&t[c], 0, rgb[c]); StoreSampleDev(&t[3], 0, k);
    for (int c = 0; c < 4; c++) dst[c] = uint8_t(0xff - t[c]); if (o.alpha_plane >= 0) StoreSampleDev(dst + 4, 0, a); return;
  }
  for (uint32_t c = 0; c < o.color_channels; c++) StoreSampleDev(dst + bps * c, o.sample_type, rgb[c]);
  if (o.alpha_plane >= 0) StoreSampleDev(dst + bps * o.color_channels, o.sample_type, a);
}

__global__ void k_output(const __grid_constant__ DFrame f, const float* __restrict__ xyb) {
  const int xs = int(f.xsize), ys = int(f.ysize); const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y; if (x >= xs || y >= ys) return;
  if (f.band_on && (y < int(f.out_y0) || y >= int(f.out_y1))) return;
  float X = 0.f, Y = 0.f, B = 0.f;
  if (f.encoding == 0) { const size_t plane = size_t(f.xpad) * f.ypad, at = size_t(y) * f.xpad + x; X = xyb[at]; Y = xyb[plane + at]; B = xyb[2 * plane + at]; }
  OutputPixel(f, x, y, X, Y, B);
}

// Fused restoration + colour kernel: one 32x32 output tile per CTA. The tile plus its halo (1 for gaborish, 3/2/1 for EPF
// pass 0/1/2) is loaded once into shared memory with mirrored image borders (the filters are mirror-equivariant, so filtering
// the mirrored halo reproduces the mirrored filtered image), the passes ping-pong between two shared buffers, and the last
// buffer goes straight through the colour transform to the output image: 12 B/px read + 3-4 B/px written instead of
// 24 B/px per pass. SURVEY.md A.10; replaces libjxl's render pipeline stages reached from N/Decoder/JxlDecoder.cpp:252.
// FAST: plain RGB8 output (3 colour channels, no alpha / CMYK / BGRA, identity orientation, rows 4-byte aligned): the tile's bytes are
// packed in shared memory and leave as 32-bit words, 96 contiguous bytes per row, instead of three byte stores per pixel.
template <int GAB, int EPF, bool FAST>
__global__ void __launch_bounds__(256) k_render(const __grid_constant__ DFrame f) {
  constexpr int R0 = EPF == 3 ? 3 : 0, R1 = EPF >= 1 ? 2 : 0, R2 = EPF >= 2 ? 1 : 0, H = GAB + R0 + R1 + R2, D = 32 + 2 * H, N = D * D;
  if (f.band_on && (blockIdx.y * 32 + 32 <= f.out_y0 || blockIdx.y * 32 >= f.out_y1)) return;   // band decode: tiles outside the band
  extern __shared__ float rs[]; float* A = rs; float* Bf = rs + 3 * N; float* Mh = rs + 6 * N; float* Mv = rs + 7 * N; float* s_is = rs + (EPF ? 8 : 6) * N;   // s_is: 8x8 blocks of 1/sigma
  const int xs = int(f.xsize), ys = int(f.ysize), tx0 = blockIdx.x * 32 - H, ty0 = blockIdx.y * 32 - H, tid = threadIdx.x; const size_t plane = size_t(f.xpad) * f.ypad;
  const int bx0 = max(tx0, 0) >> 3, by0 = max(ty0, 0) >> 3;
  if (EPF && tid < 64) { const int by = by0 + (tid >> 3), bx = bx0 + (tid & 7); s_is[tid] = (by < int(f.yb) && bx < int(f.xb)) ? f.inv_sigma[size_t(by) * f.xb + bx] : 0.f; }
  {  // tile + halo: a thread owns one column (mirrored x resolved once) and every (256/D)-th row
    constexpr int S = 256 / D; const int lx = tid % D, gx = MirrorDev(tx0 + lx, xs);
    if (tid < S * D) for (int ly = tid / D; ly < D; ly += S) { const size_t at = size_t(MirrorDev(ty0 + ly, ys)) * f.xpad + gx; const int i = ly * D + lx;
      A[i] = f.xyb[at]; A[N + i] = f.xyb[plane + at]; A[2 * N + i] = f.xyb[2 * plane + at]; }
  }
  __syncthreads();
  int off = 0;   // valid region of the current buffer is [off, D-off)^2
  float* src = A; float* dst = Bf;
  if (GAB) {   // column strips: a thread walks down its column with a rolling 3x3 window per channel (3 shared loads per sample instead of 9)
    off += 1; constexpr int n = D - 2, S = 256 / n, R = (n + S - 1) / S;
    if (tid < n * S) {
      const int x = off + tid % n, y0 = off + (tid / n) * R, y1 = min(y0 + R, off + n);
#pragma unroll
      for (int c = 0; c < 3; c++) {
        const float* s = src + c * N + x; float* d = dst + c * N + x; const float w1 = f.lpf.gab_w[2 * c], w2 = f.lpf.gab_w[2 * c + 1], mul = 1.0f / (1.0f + 4.0f * (w1 + w2)), m1 = w1 * mul, m2 = w2 * mul;
        float a0 = s[(y0 - 1) * D - 1], a1 = s[(y0 - 1) * D], a2 = s[(y0 - 1) * D + 1], b0 = s[y0 * D - 1], b1 = s[y0 * D], b2 = s[y0 * D + 1];
#pragma unroll
        for (int k = 0; k < R; k++) { const int y = y0 + k; if (y >= y1) break; const float c0 = s[(y + 1) * D - 1], c1 = s[(y + 1) * D], c2 = s[(y + 1) * D + 1];
          d[y * D] = b1 * mul + (a1 + c1 + b0 + b2) * m1 + (a0 + a2 + c0 + c2) * m2; a0 = b0; a1 = b1; a2 = b2; b0 = c0; b1 = c1; b2 = c2; }
      }
    }
    __syncthreads(); float* t = src; src = dst; dst = t;
  }
#pragma unroll
  for (int pass = 0; pass < 3; pass++) {
    const int r = pass == 0 ? R0 : pass == 1 ? R1 : R2; if (r == 0) continue;
    off += r; const int n = D - 2 * off;
    const float sigma_scale = pass == 0 ? f.lpf.pass0_sigma_scale : pass == 2 ? f.lpf.pass2_sigma_scale : 1.0f, sm = sigma_scale * 1.65f, smb = sm * f.lpf.border_sad_mul;
    const float cs0 = f.lpf.epf_channel_scale[0], cs1 = f.lpf.epf_channel_scale[1], cs2 = f.lpf.epf_channel_scale[2];
    if (pass == 1) {
      // The 5-tap-cross SAD towards a 4-neighbour is a sum of five adjacent-sample differences, so two maps of channel-weighted
      // |horizontal| and |vertical| differences are built once, and a pixel reads 16 map entries instead of 120 samples.
      { const int lo = off - 2, m = D - 2 * lo - 1;
        for (int i = tid; i < m * m; i += 256) { const int q = (lo + i / m) * D + lo + i % m; const float a0 = src[q], a1 = src[N + q], a2 = src[2 * N + q];
          Mh[q] = fabsf(src[q + 1] - a0) * cs0 + fabsf(src[N + q + 1] - a1) * cs1 + fabsf(src[2 * N + q + 1] - a2) * cs2;
          Mv[q] = fabsf(src[q + D] - a0) * cs0 + fabsf(src[N + q + D] - a1) * cs1 + fabsf(src[2 * N + q + D] - a2) * cs2; } }
      __syncthreads();
      constexpr int n1 = D - 2 * (GAB + R0 + R1), S = 256 / n1, R = (n1 + S - 1) / S;
      if (tid < n * S) {   // column strips with rolling registers: 16 shared loads per pixel
        const int x = off + tid % n, y0 = off + (tid / n) * R, y1 = min(y0 + R, off + n); const int gx = MirrorDev(tx0 + x, xs); const bool xborder = (gx & 7) == 0 || (gx & 7) == 7; const int isx = (gx >> 3) - bx0;
        float h[3][4], v[4][3], pu[3], pl[3], pc[3], pr[3], pd[3];
#pragma unroll
        for (int rr = 0; rr < 3; rr++) for (int j = 0; j < 4; j++) h[rr][j] = Mh[(y0 - 1 + rr) * D + x - 2 + j];
#pragma unroll
        for (int rr = 0; rr < 4; rr++) for (int j = 0; j < 3; j++) v[rr][j] = Mv[(y0 - 2 + rr) * D + x - 1 + j];
#pragma unroll
        for (int c = 0; c < 3; c++) { const float* s = src + c * N + y0 * D + x; pu[c] = s[-D]; pl[c] = s[-1]; pc[c] = s[0]; pr[c] = s[1]; pd[c] = s[D]; }
#pragma unroll
        for (int k = 0; k < R; k++) {
          const int y = y0 + k; if (y >= y1) break;
          const int p = y * D + x, gy = MirrorDev(ty0 + y, ys); const float is = s_is[((gy >> 3) - by0) * 8 + isx];
          if (is < -3.90524291751269967465540850526868f) { dst[p] = pc[0]; dst[N + p] = pc[1]; dst[2 * N + p] = pc[2]; }
          else {
            const bool border = xborder || (gy & 7) == 0 || (gy & 7) == 7; const float inv = is * (border ? smb : sm);
            const float sad_u = v[1][1] + v[0][1] + v[2][1] + v[1][0] + v[1][2];   // neighbour (y-1, x)
            const float sad_l = h[1][1] + h[0][1] + h[2][1] + h[1][0] + h[1][2];   // neighbour (y, x-1)
            const float sad_r = h[1][2] + h[0][2] + h[2][2] + h[1][1] + h[1][3];   // neighbour (y, x+1)
            const float sad_d = v[2][1] + v[1][1] + v[3][1] + v[2][0] + v[2][2];   // neighbour (y+1, x)
            const float wu = fmaxf(0.f, 1.0f + sad_u * inv), wl = fmaxf(0.f, 1.0f + sad_l * inv), wr = fmaxf(0.f, 1.0f + sad_r * inv), wd = fmaxf(0.f, 1.0f + sad_d * inv);
            const float iw = 1.0f / (1.0f + wu + wl + wr + wd);
#pragma unroll
            for (int c = 0; c < 3; c++) dst[c * N + p] = (pc[c] + wu * pu[c] + wl * pl[c] + wr * pr[c] + wd * pd[c]) * iw;
          }
          if (y + 1 < y1) {   // roll the window one row down
#pragma unroll
            for (int j = 0; j < 4; j++) { h[0][j] = h[1][j]; h[1][j] = h[2][j]; h[2][j] = Mh[(y + 2) * D + x - 2 + j]; }
#pragma unroll
            for (int j = 0; j < 3; j++) { v[0][j] = v[1][j]; v[1][j] = v[2][j]; v[2][j] = v[3][j]; v[3][j] = Mv[(y + 2) * D + x - 1 + j]; }
#pragma unroll
            for (int c = 0; c < 3; c++) { const float* s = src + c * N + (y + 1) * D + x; pu[c] = pc[c]; pc[c] = pd[c]; pl[c] = s[-1]; pr[c] = s[1]; pd[c] = s[D]; }
          }
        }
      }
    } else {
      for (int i = tid; i < n * n; i += 256) {
        const int y = off + i / n, x = off + i % n, p = y * D + x; const int gy = MirrorDev(ty0 + y, ys), gx = MirrorDev(tx0 + x, xs);
        const float is = s_is[((gy >> 3) - by0) * 8 + (gx >> 3) - bx0];
        if (is < -3.90524291751269967465540850526868f) { dst[p] = src[p]; dst[N + p] = src[N + p]; dst[2 * N + p] = src[2 * N + p]; continue; }
        const bool border = ((gy & 7) == 0 || (gy & 7) == 7 || (gx & 7) == 0 || (gx & 7) == 7); const float inv = is * (border ? smb : sm);
        float wsum = 1.0f, acc0 = src[p], acc1 = src[N + p], acc2 = src[2 * N + p];
        const int nn = pass == 0 ? 12 : 4;
        const int d12[12] = {-2 * D, -D - 1, -D, -D + 1, -2, -1, 1, 2, D - 1, D, D + 1, 2 * D}; const int d4[4] = {-D, -1, 1, D};
#pragma unroll
        for (int k = 0; k < nn; k++) {
          const int d = pass == 0 ? d12[k] : d4[k]; float sad = 0.f;
#pragma unroll
          for (int c = 0; c < 3; c++) { const float* s = src + c * N + p; float sc;
            if (pass == 2) sc = fabsf(s[d] - s[0]);
            else sc = fabsf(s[d] - s[0]) + fabsf(s[d - D] - s[-D]) + fabsf(s[d + D] - s[D]) + fabsf(s[d - 1] - s[-1]) + fabsf(s[d + 1] - s[1]);
            sad += sc * (c == 0 ? cs0 : c == 1 ? cs1 : cs2); }
          const float wgt = fmaxf(0.f, 1.0f + sad * inv); wsum += wgt; acc0 += wgt * src[p + d]; acc1 += wgt * src[N + p + d]; acc2 += wgt * src[2 * N + p + d];
        }
        const float iw = 1.0f / wsum; dst[p] = acc0 * iw; dst[N + p] = acc1 * iw; dst[2 * N + p] = acc2 * iw;
      }
    }
    __syncthreads(); float* t = src; src = dst; dst = t;
  }
  if (FAST) {
    uint8_t* sb = reinterpret_cast<uint8_t*>(dst);   // the other plane buffer is free after the last pass: 32 rows x 96 bytes
    for (int i = tid; i < 32 * 32; i += 256) { const int ly = i >> 5, lx = i & 31, p = (H + ly) * D + H + lx; float rgb[3]; XybToRgbDev(f, src[p], src[N + p], src[2 * N + p], rgb);
#pragma unroll
      for (int c = 0; c < 3; c++) sb[ly * 96 + lx * 3 + c] = uint8_t(__float2int_rn(fminf(1.f, fmaxf(0.f, rgb[c])) * 255.0f)); }
    __syncthreads();
    const int x0 = blockIdx.x * 32, y0 = blockIdx.y * 32, nbytes = min(32, xs - x0) * 3;
    for (int i = tid; i < 32 * 24; i += 256) { const int ly = i / 24, b0 = (i - ly * 24) * 4, y = y0 + ly; if (y >= ys || b0 >= nbytes) continue;
      if (f.band_on && (y < int(f.out_y0) || y >= int(f.out_y1))) continue;
      uint8_t* row = f.out_px + (size_t(y - int(f.out_y0)) * xs + x0) * 3;
      if (b0 + 4 <= nbytes) *reinterpret_cast<uint32_t*>(row + b0) = *reinterpret_cast<const uint32_t*>(sb + ly * 96 + b0); else for (int b = b0; b < nbytes; b++) row[b] = sb[ly * 96 + b]; }
    return;
  }
  for (int i = tid; i < 32 * 32; i += 256) { const int ly = i >> 5, lx = i & 31, y = blockIdx.y * 32 + ly, x = blockIdx.x * 32 + lx; if (x >= xs || y >= ys) continue;
    if (f.band_on && (y < int(f.out_y0) || y >= int(f.out_y1))) continue;
    const int p = (H + ly) * D + H + lx; OutputPixel(f, x, y, src[p], src[N + p], src[2 * N + p]); }
}

// ------------------------------------------------------------------ fused render, wide-tile version
// gaborish + EPF pass 1 (+ pass 2) + XYB -> RGB8 for the common output (RGB8, identity orientation) with 64x32 output tiles and
// vector shared-memory accesses. Same arithmetic as k_render; what changes is the work per instruction:
//   * 64x32 tiles: halo overhead (70x38)/(64x32) = 1.30 instead of 1.41 for 32x32, and rows of 72 floats so that every row starts
//     16-byte aligned (x = -4 sits in column 0): filters read LDS.128;
//   * gaborish: a thread owns (channel, 4 columns, 9 rows) with a rolling three-row window: 3 shared loads per 4 outputs;
//   * EPF: the 5-tap-cross SADs are sums of channel-weighted |horizontal| / |vertical| difference maps Dh, Dv built once; a thread
//     filters a 4x2 patch and builds the cross sums of its patch from LDS.128 rows, ~6 shared loads per pixel instead of 16;
//   * colour + pack in registers, 12 contiguous bytes per thread and row.
// Buffers: A[3][38][72] (raw XYB; later Dh = A[0], Dv = A[1]), B[3][38][72] (after gaborish). Row r <-> y = ty0 - 3 + r, column c <-> x = tx0 - 4 + c.
static const int kRfS = 72, kRfRows = 38, kRfPlane = kRfS * kRfRows;
static const int kRfBuf = (3 * kRfPlane * 4 + 127) / 128 * 128 / 4;   // floats per three-plane buffer, padded so that every buffer starts 128-byte aligned (TMA destination)
__host__ __device__ __forceinline__ bool WideTileInterior(const DFrame& f, int tx0, int ty0) { return tx0 >= 4 && tx0 + 68 <= int(f.xsize) && ty0 >= 3 && ty0 + 35 <= int(f.ysize); }
// tile + halo -> A with mirrored image borders (the slow path of border tiles; interior tiles arrive by TMA)
__device__ __forceinline__ void WideTileFillMirrored(const DFrame& f, float* A, int tx0, int ty0, int tid) {
  const int xs = int(f.xsize), ys = int(f.ysize); const size_t plane = size_t(f.xpad) * f.ypad;
  for (int i = tid; i < 3 * kRfRows * kRfS; i += 256) { const int c = i / kRfPlane, rem = i - c * kRfPlane, r = rem / kRfS, col = rem - r * kRfS;
    A[i] = f.xyb[c * plane + size_t(MirrorDev(ty0 - 3 + r, ys)) * f.xpad + MirrorDev(tx0 - 4 + col, xs)]; }
}
// Stages 1-3 on a tile whose raw samples sit in A (visible to every thread). Ends with the pixel stores; the caller synchronises before
// A or B are written again.
template <int EPF, bool BGRA>
__device__ __forceinline__ void WideTileStages(const DFrame& f, float* A, float* B, const float* s_is, const int tx0, const int ty0, const int tid) {
  static_assert(EPF == 1, "pass 2 is handled by k_render");
  const int xs = int(f.xsize), ys = int(f.ysize);
  // ---- stage 1: gaborish A -> B on rows 1..36 (y = -2..33); thread = (channel, quad column, 9-row strip)
  if (tid < 216) {
    const int c = tid / 72, rem = tid - c * 72, q = rem % 18, strip = rem / 18, r0 = 1 + strip * 9;
    const float w1 = f.lpf.gab_w[2 * c], w2 = f.lpf.gab_w[2 * c + 1], m0 = 1.0f / (1.0f + 4.0f * (w1 + w2)), m1 = w1 * m0, m2 = w2 * m0;
    const float* src = A + c * kRfPlane + 4 * q; float* dst = B + c * kRfPlane + 4 * q; const int lo = q == 0 ? 0 : -1, hi = q == 17 ? 3 : 4;
    auto load = [&](int r, float4& v, float4& sd) { const float* p = src + r * kRfS; v = *reinterpret_cast<const float4*>(p); const float L = p[lo], R = p[hi];
      sd = make_float4(L + v.y, v.x + v.z, v.y + v.w, v.z + R); };
    float4 c0, s0, c1, s1, c2, s2; load(r0 - 1, c0, s0); load(r0, c1, s1);
#pragma unroll
    for (int k = 0; k < 9; k++) {
      load(r0 + k + 1, c2, s2);
      float4 o;
      o.x = c1.x * m0 + (c0.x + c2.x + s1.x) * m1 + (s0.x + s2.x) * m2; o.y = c1.y * m0 + (c0.y + c2.y + s1.y) * m1 + (s0.y + s2.y) * m2;
      o.z = c1.z * m0 + (c0.z + c2.z + s1.z) * m1 + (s0.z + s2.z) * m2; o.w = c1.w * m0 + (c0.w + c2.w + s1.w) * m1 + (s0.w + s2.w) * m2;
      *reinterpret_cast<float4*>(dst + (r0 + k) * kRfS) = o; c0 = c1; s0 = s1; c1 = c2; s1 = s2;
    }
  }
  __syncthreads();
  // ---- stage 2: difference maps from B: Dh(r, c) = sum_ch scale * |B(r, c+1) - B(r, c)| -> A[0], Dv(r, c) = sum_ch scale * |B(r+1, c) - B(r, c)| -> A[1], rows 1..35
  if (tid < 252) {
    const int q = tid % 18, part = tid / 18, r0 = 1 + (part < 7 ? part * 3 : 21 + (part - 7) * 2), nr = part < 7 ? 3 : 2, hi = q == 17 ? 3 : 4;
    const float cs[3] = {f.lpf.epf_channel_scale[0], f.lpf.epf_channel_scale[1], f.lpf.epf_channel_scale[2]};
    float4 cur[3];
#pragma unroll
    for (int c = 0; c < 3; c++) cur[c] = *reinterpret_cast<const float4*>(B + c * kRfPlane + r0 * kRfS + 4 * q);
    for (int k = 0; k < nr; k++) {
      const int r = r0 + k; float4 dh = make_float4(0.f, 0.f, 0.f, 0.f), dv = dh;
#pragma unroll
      for (int c = 0; c < 3; c++) {
        const float* p = B + c * kRfPlane + r * kRfS + 4 * q; const float R = p[hi]; const float4 nx = *reinterpret_cast<const float4*>(p + kRfS), v = cur[c];
        dh.x = fmaf(fabsf(v.y - v.x), cs[c], dh.x); dh.y = fmaf(fabsf(v.z - v.y), cs[c], dh.y); dh.z = fmaf(fabsf(v.w - v.z), cs[c], dh.z); dh.w = fmaf(fabsf(R - v.w), cs[c], dh.w);
        dv.x = fmaf(fabsf(nx.x - v.x), cs[c], dv.x); dv.y = fmaf(fabsf(nx.y - v.y), cs[c], dv.y); dv.z = fmaf(fabsf(nx.z - v.z), cs[c], dv.z); dv.w = fmaf(fabsf(nx.w - v.w), cs[c], dv.w);
        cur[c] = nx;
      }
      *reinterpret_cast<float4*>(A + r * kRfS + 4 * q) = dh; *reinterpret_cast<float4*>(A + kRfPlane + r * kRfS + 4 * q) = dv;
    }
  }
  __syncthreads();
  // ---- stage 3: EPF pass 1 on a 4x2 patch per thread, then colour + pack
  const int px = tid & 15, py = tid >> 4, col = 4 + 4 * px, r0 = 3 + 2 * py;   // patch: columns col..col+3 (x = 4 px ..), rows r0, r0+1 (y = 2 py, 2 py + 1)
  const float* Dh = A; const float* Dv = A + kRfPlane;
  float outv[3][2][4];
  {
    const float is = s_is[(py >> 2) * 8 + (px >> 1)];
    if (is < -3.90524291751269967465540850526868f) {
#pragma unroll
      for (int c = 0; c < 3; c++)
#pragma unroll
        for (int j = 0; j < 2; j++) { const float4 v = *reinterpret_cast<const float4*>(B + c * kRfPlane + (r0 + j) * kRfS + col); outv[c][j][0] = v.x; outv[c][j][1] = v.y; outv[c][j][2] = v.z; outv[c][j][3] = v.w; }
    } else {
      // cross sums Ch(r, c) = Dh(r-1,c) + Dh(r,c) + Dh(r+1,c) + Dh(r,c-1) + Dh(r,c+1) at columns col-1..col+3, rows r0, r0+1:
      // SAD towards the right neighbour of pixel (r, c) is Ch(r, c), towards the left neighbour Ch(r, c-1)
      float hrow[4][5];   // Dh rows r0-1..r0+2, columns col-1..col+3
#pragma unroll
      for (int k = 0; k < 4; k++) { const float* p = Dh + (r0 - 1 + k) * kRfS + col; const float4 v = *reinterpret_cast<const float4*>(p); hrow[k][0] = p[-1]; hrow[k][1] = v.x; hrow[k][2] = v.y; hrow[k][3] = v.z; hrow[k][4] = v.w; }
      float Ch[2][5];
#pragma unroll
      for (int j = 0; j < 2; j++) {
        const float* p = Dh + (r0 + j) * kRfS + col; const float l2 = p[-2], r4 = p[4];
#pragma unroll
        for (int i = 0; i < 5; i++) { const float left = i == 0 ? l2 : hrow[j + 1][i - 1], right = i == 4 ? r4 : hrow[j + 1][i + 1]; Ch[j][i] = hrow[j][i] + hrow[j + 1][i] + hrow[j + 2][i] + left + right; }
      }
      // Cv(r, c) = Dv(r-1,c) + Dv(r,c) + Dv(r+1,c) + Dv(r,c-1) + Dv(r,c+1) at rows r0-1..r0+1, columns col..col+3:
      // SAD towards the lower neighbour of pixel (r, c) is Cv(r, c), towards the upper neighbour Cv(r-1, c)
      float vrow[5][4];   // Dv rows r0-2..r0+2
#pragma unroll
      for (int k = 0; k < 5; k++) { const float4 v = *reinterpret_cast<const float4*>(Dv + (r0 - 2 + k) * kRfS + col); vrow[k][0] = v.x; vrow[k][1] = v.y; vrow[k][2] = v.z; vrow[k][3] = v.w; }
      float Cv[3][4];
#pragma unroll
      for (int j = 0; j < 3; j++) {
        const float* p = Dv + (r0 - 1 + j) * kRfS + col; const float l1 = p[-1], r4 = p[4];
#pragma unroll
        for (int i = 0; i < 4; i++) { const float left = i == 0 ? l1 : vrow[j + 1][i - 1], right = i == 3 ? r4 : vrow[j + 1][i + 1]; Cv[j][i] = vrow[j][i] + vrow[j + 1][i] + vrow[j + 2][i] + left + right; }
      }
      const float sm = 1.65f, smb = sm * f.lpf.border_sad_mul;   // pass 1 has sigma scale 1
      float wl[2][4], wr[2][4], wu[2][4], wd[2][4], iw[2][4];
#pragma unroll
      for (int j = 0; j < 2; j++)
#pragma unroll
        for (int i = 0; i < 4; i++) {
          const int xm = (4 * px + i) & 7, ym = (2 * py + j) & 7; const bool border = xm == 0 || xm == 7 || ym == 0 || ym == 7; const float inv = is * (border ? smb : sm);
          wr[j][i] = fmaxf(0.f, fmaf(Ch[j][i + 1], inv, 1.0f)); wl[j][i] = fmaxf(0.f, fmaf(Ch[j][i], inv, 1.0f));
          wd[j][i] = fmaxf(0.f, fmaf(Cv[j + 1][i], inv, 1.0f)); wu[j][i] = fmaxf(0.f, fmaf(Cv[j][i], inv, 1.0f));
          iw[j][i] = __fdividef(1.0f, 1.0f + wu[j][i] + wl[j][i] + wr[j][i] + wd[j][i]);   // MUFU.RCP: the sum is in [1, 5]
        }
#pragma unroll
      for (int c = 0; c < 3; c++) {
        float prow[4][6];   // B rows r0-1..r0+2, columns col-1..col+4 (the corner entries of the outer rows are not used)
#pragma unroll
        for (int k = 0; k < 4; k++) { const float* p = B + c * kRfPlane + (r0 - 1 + k) * kRfS + col; const float4 v = *reinterpret_cast<const float4*>(p); prow[k][1] = v.x; prow[k][2] = v.y; prow[k][3] = v.z; prow[k][4] = v.w;
          if (k == 1 || k == 2) { prow[k][0] = p[-1]; prow[k][5] = p[4]; } }
#pragma unroll
        for (int j = 0; j < 2; j++)
#pragma unroll
          for (int i = 0; i < 4; i++)
            outv[c][j][i] = (prow[j + 1][i + 1] + wu[j][i] * prow[j][i + 1] + wl[j][i] * prow[j + 1][i] + wr[j][i] * prow[j + 1][i + 2] + wd[j][i] * prow[j + 2][i + 1]) * iw[j][i];
      }
    }
  }
  // ---- colour + pack: 4 pixels = 12 bytes per row (RGB8) or one 16-byte store (BGRA32 surface, A = 255: S/JpegXLLoad.cs:219-249 with an opaque layer)
#pragma unroll
  for (int j = 0; j < 2; j++) {
    const int y = ty0 + 2 * py + j, x = tx0 + 4 * px; uint32_t b[12];
#pragma unroll
    for (int i = 0; i < 4; i++) { float rgb[3]; XybToRgbDev(f, outv[0][j][i], outv[1][j][i], outv[2][j][i], rgb);
#pragma unroll
      for (int c = 0; c < 3; c++) b[3 * i + c] = uint32_t(__float2int_rn(fminf(1.f, fmaxf(0.f, rgb[c])) * 255.0f)); }
    if (y >= ys || x >= xs) continue;
    if (f.band_on && (y < int(f.out_y0) || y >= int(f.out_y1))) continue;
    if (BGRA) {
      uint32_t* row4 = reinterpret_cast<uint32_t*>(f.out_px) + size_t(y - int(f.out_y0)) * xs + x; uint32_t v[4];
#pragma unroll
      for (int i = 0; i < 4; i++) v[i] = b[3 * i + 2] | (b[3 * i + 1] << 8) | (b[3 * i] << 16) | 0xff000000u;
      if (x + 4 <= xs && (xs & 3) == 0) *reinterpret_cast<uint4*>(row4) = make_uint4(v[0], v[1], v[2], v[3]);
      else {
#pragma unroll
        for (int i = 0; i < 4; i++) if (x + i < xs) row4[i] = v[i];
      }
      continue;
    }
    uint8_t* row = f.out_px + (size_t(y - int(f.out_y0)) * xs + x) * 3;
    if (x + 4 <= xs && (reinterpret_cast<uintptr_t>(row) & 3) == 0) {
      uint32_t* w = reinterpret_cast<uint32_t*>(row);
      w[0] = b[0] | (b[1] << 8) | (b[2] << 16) | (b[3] << 24); w[1] = b[4] | (b[5] << 8) | (b[6] << 16) | (b[7] << 24); w[2] = b[8] | (b[9] << 8) | (b[10] << 16) | (b[11] << 24);
    } else {
#pragma unroll
      for (int i = 0; i < 4; i++) if (x + i < xs) { row[3 * i] = uint8_t(b[3 * i]); row[3 * i + 1] = uint8_t(b[3 * i + 1]); row[3 * i + 2] = uint8_t(b[3 * i + 2]); }
    }
  }
}

// Frame row of the first row the XYB planes hold: a band decode allocates them from its first reconstructed group row (the halo row above
// the band) and addresses them through a base shifted back by that many rows; a whole-frame decode starts at row 0.
__host__ __device__ __forceinline__ int XybFirstRow(const DFrame& f) { return f.band_on ? int(f.comp_g0 * f.group_dim) : 0; }
// Persistent CTAs, two per SM, walk the tiles [t0, t1) with a grid stride (a band decode passes its own tile rows). The raw 72x38x3 box of
// the NEXT tile is fetched by one TMA operation (cp.async.bulk.tensor.3d, completion on an mbarrier) into the second raw buffer while the
// current tile is filtered, so no warp waits on HBM latency inside the stages (profiles/r02_render_tma_ab.md). Border tiles (mirrored
// samples: TMA can only zero-fill) are loaded by the threads. Interior tiles of a band stay inside its allocated rows: the band carries one
// group row of halo on each side, more than the 3 rows above and 35 below that WideTileInterior asks for.
__device__ __forceinline__ uint32_t SmemU32(const void* p) { return uint32_t(__cvta_generic_to_shared(p)); }
template <int EPF, bool BGRA>
__global__ void __launch_bounds__(256, 2) k_render_wide_tma(const __grid_constant__ DFrame f, const __grid_constant__ CUtensorMap tmap, const int ntx, const int t0, const int t1) {
  extern __shared__ __align__(128) float rw[];
  float* B = rw + 2 * kRfBuf;   // raw buffers: rw + b * kRfBuf, b = 0, 1
  __shared__ __align__(8) unsigned long long bar[2]; __shared__ float s_is[32];
  const int tid = threadIdx.x;
  if (tid == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(SmemU32(&bar[0])));
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(SmemU32(&bar[1])));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  auto tile_xy = [&](int t, int& tx0, int& ty0) { tx0 = (t % ntx) * 64; ty0 = (t / ntx) * 32; };
  auto issue = [&](int t, int b) {   // one thread: arm the barrier with the box size and start the bulk copy
    int tx0, ty0; tile_xy(t, tx0, ty0);
    if (tid != 0 || !WideTileInterior(f, tx0, ty0)) return;
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // the buffer was last written through the generic proxy (difference maps)
    const uint32_t bytes = 3u * kRfPlane * 4u, mb = SmemU32(&bar[b]);
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mb), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
                 ::"r"(SmemU32(rw + b * kRfBuf)), "l"(reinterpret_cast<uint64_t>(&tmap)), "r"(mb), "r"(tx0 - 4), "r"(ty0 - 3 - XybFirstRow(f)), "r"(0) : "memory");
  };
  uint32_t phase_bits = 0u;   // bit b: parity of buffer b's barrier
  int t = t0 + int(blockIdx.x); if (t < t1) issue(t, 0);
  for (int b = 0; t < t1; t += int(gridDim.x), b ^= 1) {
    if (t + int(gridDim.x) < t1) issue(t + int(gridDim.x), b ^ 1);
    int tx0, ty0; tile_xy(t, tx0, ty0);
    float* A = rw + b * kRfBuf;
    if (tid < 32) { const int by = (ty0 >> 3) + (tid >> 3), bx = (tx0 >> 3) + (tid & 7); s_is[tid] = (by < int(f.yb) && bx < int(f.xb)) ? f.inv_sigma[size_t(by) * f.xb + bx] : 0.f; }
    if (WideTileInterior(f, tx0, ty0)) {
      const uint32_t mb = SmemU32(&bar[b]), ph = (phase_bits >> b) & 1u; uint32_t ok = 0;
      while (!ok) asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }" : "=r"(ok) : "r"(mb), "r"(ph) : "memory");
      phase_bits ^= 1u << b;
    } else WideTileFillMirrored(f, A, tx0, ty0, tid);
    __syncthreads();
    WideTileStages<EPF, BGRA>(f, A, B, s_is, tx0, ty0, tid);
    __syncthreads();   // every read of A / B is done before the next copy lands in A's partner and before B is rewritten
  }
}

// Lossless 8/16-bit integer fast path: samples pass through untouched (bit-exact by construction).
__global__ void k_output_int(const DFrame* fp) {
  const DFrame& f = *fp; const int xs = int(f.xsize), ys = int(f.ysize); const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y; if (x >= xs || y >= ys) return;
  if (f.band_on && (y < int(f.out_y0) || y >= int(f.out_y1))) return;
  const DOutput& o = f.out; const size_t oi = OrientedIndex(f, x, y); const uint32_t nc = f.color.num_color; int32_t v[4]; uint32_t n = 0;
  for (uint32_t c = 0; c < o.color_channels; c++) { const DModChannel& ch = f.out_ch[c < nc ? c : nc - 1]; v[n++] = f.mod_planes[ch.plane_off + size_t(y) * ch.w + x]; }
  if (o.alpha_plane >= 0) { const DModChannel& ch = f.out_ch[o.alpha_plane]; v[n++] = f.mod_planes[ch.plane_off + size_t(y) * ch.w + x]; }
  const int32_t mx = o.sample_type == 0 ? 255 : 65535;
  if (o.bgra) { uint8_t r8 = uint8_t(min(max(v[0], 0), 255)), g8 = o.color_channels == 1 ? r8 : uint8_t(min(max(v[1], 0), 255)), b8 = o.color_channels == 1 ? r8 : uint8_t(min(max(v[2], 0), 255)); uint8_t a8 = o.alpha_plane >= 0 ? uint8_t(min(max(v[n - 1], 0), 255)) : 255;
    reinterpret_cast<uint32_t*>(f.out_px)[oi] = uint32_t(b8) | (uint32_t(g8) << 8) | (uint32_t(r8) << 16) | (uint32_t(a8) << 24); return; }
  if (o.sample_type == 0) { uint8_t* dst = f.out_px + oi * n; for (uint32_t c = 0; c < n; c++) dst[c] = uint8_t(min(max(v[c], 0), mx)); }
  else { uint16_t* dst = reinterpret_cast<uint16_t*>(f.out_px) + oi * n; for (uint32_t c = 0; c < n; c++) dst[c] = uint16_t(min(max(v[c], 0), mx)); }
}

void LaunchReconstruct(const DFrame* d, const DFrame& h, cudaStream_t st) {
  const size_t smem16 = size_t(kReconWarps) * 3 * 16 * 20 * sizeof(float), smem32 = size_t(kReconWarps) * 3 * 32 * 36 * sizeof(float);
  { const int items = int(h.num_groups) * 32; const int grid = std::min(items, 148 * 3); const size_t d8smem = size_t(2) * 3 * 32 * kD8Stride * sizeof(float);
    Launch<k_reconstruct_dct8>(grid, 256, d8smem, st, h, items); }
  Launch<k_reconstruct<16>>(h.num_groups * 4, kReconWarps * 32, smem16, st, d); Launch<k_reconstruct<32>>(h.num_groups * 4, kReconWarps * 32, smem32, st, d);
}
void LaunchGaborishPlanes(const DFrame* d, const DFrame& h, const float* src, float* dst, cudaStream_t st) { dim3 blk(32, 8), grid((h.xsize + 31) / 32, (h.ysize + 7) / 8); Launch<k_gaborish>(grid, blk, 0, st, d, src, dst); }
// TMA descriptor of the three XYB planes as one rank-3 fp32 tensor {xpad, ypad, 3}, box {72, 38, 3}: one bulk copy fetches a whole
// tile-plus-halo into the dense [plane][row][72] layout the filters read. The tensor starts at the planes' first allocated row (XybFirstRow),
// so a band's map covers exactly its ypad rows. The driver entry point is looked up at run time (no libcuda link).
static bool EncodeXybTensorMap(const DFrame& h, CUtensorMap* out) {
  typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                               CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  static EncodeFn fn = []() -> EncodeFn { void* p = nullptr; cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) { cudaGetLastError(); return nullptr; } return reinterpret_cast<EncodeFn>(p); }();
  if (!fn) return false;
  const cuuint64_t gdim[3] = {h.xpad, h.ypad, 3}, gstride[2] = {cuuint64_t(h.xpad) * 4, cuuint64_t(h.xpad) * h.ypad * 4}; const cuuint32_t box[3] = {kRfS, kRfRows, 3}, es[3] = {1, 1, 1};
  return fn(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, h.xyb + size_t(XybFirstRow(h)) * h.xpad, gdim, gstride, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
// k_render_wide_tma for the RGB8 or opaque BGRA32 output of a frame with gaborish + one EPF iteration
static void LaunchRenderWide(const DFrame& h, bool bgra, cudaStream_t st) {
  const size_t smem = size_t(3) * kRfBuf * sizeof(float);
  const int ntx = int(h.xsize + 63) / 64;
  // tile rows of the output rows: a band's out_y0 is a multiple of the group size, hence of the 32-row tile height
  const int t0 = h.band_on ? int(h.out_y0 / 32) * ntx : 0, t1 = int(((h.band_on ? h.out_y1 : h.ysize) + 31) / 32) * ntx;
  CUtensorMap tmap{};
  // Tile (64, 32) is the first that can be interior: a frame smaller than 132 x 67 has no interior tile, issues no copy and gets the zero map.
  if (WideTileInterior(h, 64, 32) && !EncodeXybTensorMap(h, &tmap)) throw std::runtime_error("cuTensorMapEncodeTiled failed for the render kernel's XYB planes");
  const int grid = std::min(t1 - t0, 148 * 2);
  if (bgra) Launch<k_render_wide_tma<1, true>>(grid, 256, smem, st, h, tmap, ntx, t0, t1); else Launch<k_render_wide_tma<1, false>>(grid, 256, smem, st, h, tmap, ntx, t0, t1);
}
// gaborish + EPF + colour in one pass over the frame (VarDCT frames with at least one restoration filter)
template <int GAB, int EPF> static void LaunchRenderT(const DFrame& h, cudaStream_t st) {
  constexpr int H = GAB + (EPF == 3 ? 3 : 0) + (EPF >= 1 ? 2 : 0) + (EPF >= 2 ? 1 : 0), D = 32 + 2 * H; size_t smem = (size_t(EPF ? 8 : 6) * D * D + 64) * sizeof(float);
  constexpr bool kWide = GAB == 1 && EPF == 1;   // RGB8 output of these filters takes k_render_wide_tma, so k_render<1, 1, true> is never built
  const DOutput& o = h.out;
  const bool rgb8 = !o.bgra && o.sample_type == 0 && o.num_channels == 3 && o.color_channels == 3 && o.alpha_plane < 0 && o.black_plane < 0 && !o.premultiplied && o.orientation == 1;
  dim3 grid((h.xsize + 31) / 32, (h.ysize + 31) / 32);
  if constexpr (kWide) {
    // opaque BGRA32 surface of an 8-bit RGB image (JxlB200LoadImageBgra, BASELINE config 2): the same kernel with a 16-byte store per 4 pixels
    const bool fast_bgra = o.bgra && o.color_channels == 3 && o.alpha_plane < 0 && o.black_plane < 0 && !o.premultiplied && o.orientation == 1 && (reinterpret_cast<uintptr_t>(h.out_px) & 15) == 0;
    if (rgb8 || fast_bgra) LaunchRenderWide(h, fast_bgra, st);   // rows that are not 4-byte aligned fall back to byte stores inside the kernel
    else Launch<k_render<1, 1, false>>(grid, 256, smem, st, h);
  } else {
    const bool fast = rgb8 && (size_t(h.xsize) * 3) % 4 == 0 && (reinterpret_cast<uintptr_t>(h.out_px) & 3) == 0;
    if (fast) Launch<k_render<GAB, EPF, true>>(grid, 256, smem, st, h); else Launch<k_render<GAB, EPF, false>>(grid, 256, smem, st, h);
  }
}
bool LaunchFusedRender(const DFrame* d, const DFrame& h, cudaStream_t st) {
  if (h.encoding != 0 || (!h.lpf.gab && !h.lpf.epf_iters)) return false;
  if (h.lpf.epf_iters) { size_t n = size_t(h.xb) * h.yb; Launch<k_inv_sigma>(unsigned((n + 255) / 256), 256, 0, st, d); }
  const int g = h.lpf.gab ? 1 : 0;
  switch (g * 4 + int(h.lpf.epf_iters)) {
    case 1: LaunchRenderT<0, 1>(h, st); break; case 2: LaunchRenderT<0, 2>(h, st); break; case 3: LaunchRenderT<0, 3>(h, st); break;
    case 4: LaunchRenderT<1, 0>(h, st); break; case 5: LaunchRenderT<1, 1>(h, st); break; case 6: LaunchRenderT<1, 2>(h, st); break; case 7: LaunchRenderT<1, 3>(h, st); break;
    default: return false;
  }
  return true;
}
// ------------------------------------------------------------------ inverse Squeeze on the global Modular image (SURVEY.md A.7 "Squeeze")
// avg, residual -> the two interleaved samples: diff = residual + tendency(previous output, avg, next avg); first = avg + diff / 2 (C division);
// second = first - diff. The tendency term makes sample k depend on sample k - 1 along the squeezed direction: one thread per row (horizontal)
// or per column (vertical, coalesced) walks that direction serially.
__device__ __forceinline__ long long SmoothTendencyDev(long long B, long long a, long long n) {
  long long diff = 0;
  if (B >= a && a >= n) { diff = (4 * B - 3 * n - a + 6) / 12; if (diff - (diff & 1) > 2 * (B - a)) diff = 2 * (B - a) + 1; if (diff + (diff & 1) > 2 * (a - n)) diff = 2 * (a - n); }
  else if (B <= a && a <= n) { diff = (4 * B - 3 * n - a - 6) / 12; if (diff + (diff & 1) < 2 * (B - a)) diff = 2 * (B - a) - 1; if (diff - (diff & 1) < 2 * (a - n)) diff = 2 * (a - n); }
  return diff;
}
__global__ void k_unsqueeze(const DFrame* fp, uint32_t op_index) {
  const DFrame& f = *fp; const DModOp& op = ModOp(f, op_index); const int aw = int(op.w), ah = int(op.h), rw = int(op.num_c), rh = int(op.pal_w);
  const int32_t* avg = f.mod_planes + op.p[0]; const int32_t* res = f.mod_planes + op.p[1]; int32_t* out = f.mod_planes + op.out[0];
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (op.rct_type) {   // horizontal: out is (aw + rw) x ah, thread = row
    if (t >= ah) return; const int ow = aw + rw; const int32_t* pa = avg + size_t(t) * aw; const int32_t* pr = res + size_t(t) * rw; int32_t* po = out + size_t(t) * ow;
    for (int x = 0; x < rw; x++) { const long long a = pa[x], nx = x + 1 < aw ? pa[x + 1] : a, left = x ? po[2 * x - 1] : a; const long long diff = pr[x] + SmoothTendencyDev(left, a, nx); const long long A = a + diff / 2; po[2 * x] = int32_t(A); po[2 * x + 1] = int32_t(A - diff); }
    if (ow & 1) po[ow - 1] = pa[aw - 1];
  } else {             // vertical: out is aw x (ah + rh), thread = column
    if (t >= aw) return; const int oh = ah + rh;
    for (int y = 0; y < rh; y++) { const long long a = avg[size_t(y) * aw + t], nx = y + 1 < ah ? avg[size_t(y + 1) * aw + t] : a, top = y ? out[size_t(2 * y - 1) * aw + t] : a;
      const long long diff = res[size_t(y) * aw + t] + SmoothTendencyDev(top, a, nx); const long long A = a + diff / 2; out[size_t(2 * y) * aw + t] = int32_t(A); out[size_t(2 * y + 1) * aw + t] = int32_t(A - diff); }
    if (oh & 1) out[size_t(oh - 1) * aw + t] = avg[size_t(ah - 1) * aw + t];
  }
}

void LaunchInverseRct(const DFrame* d, const DFrame& h, const DModOp* ops, cudaStream_t st) {   // every inverse transform of the global Modular image, in execution order
  for (uint32_t i = 0; i < h.num_ops; i++) {
    const DModOp& op = ops[i]; const size_t n = size_t(op.w) * op.h;
    if (op.kind == 2) { const unsigned threads = op.rct_type ? op.h : op.w; if (!threads) continue; Launch<k_unsqueeze>((threads + 63) / 64, 64, 0, st, d, i); continue; }
    if (!n) continue;
    if (op.kind == 0) Launch<k_inverse_rct>(unsigned((n + 255) / 256), 256, 0, st, d, i);
    else if (op.nb_deltas == 0) Launch<k_inverse_palette>(dim3(unsigned((n + 255) / 256), op.num_c), 256, 0, st, d, i);
    else Launch<k_inverse_palette_delta>(op.num_c, 32, 0, st, d, i);
  }
}
void LaunchOutput(const DFrame* d, const DFrame& h, cudaStream_t st) {
  dim3 blk(32, 8), grid((h.xsize + 31) / 32, (h.ysize + 7) / 8);
  bool int_path = h.encoding == 1 && !h.color.xyb_encoded && h.out.exp_bits == 0 && h.out.black_plane < 0 && !h.out.premultiplied && (h.out.sample_type == 0 ? h.out.bits == 8 : (h.out.sample_type == 1 && h.out.bits == 16)) &&
                  (h.out.alpha_plane < 0 || (h.out.alpha_bits == h.out.bits && h.out.alpha_exp_bits == 0 && h.out_ch[h.out.alpha_plane].hshift == 0));
  if (int_path) Launch<k_output_int>(grid, blk, 0, st, d); else Launch<k_output>(grid, blk, 0, st, h, h.xyb);
}

}  // namespace jxlgpu
