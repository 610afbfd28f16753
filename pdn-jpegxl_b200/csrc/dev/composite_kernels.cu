// pdn-jpegxl_b200 engine — layers of a multi-frame still blended on the GPU.
//
// The reference takes the first JXL_DEC_FULL_IMAGE of a coalescing libjxl decoder (N/Decoder/JxlDecoder.cpp:252-400): every frame of zero
// duration before the first frame that is shown is a LAYER, blended onto the canvas or onto one of four reference slots with the frame
// header's BlendingInfo (replace / add / blend / alpha-weighted add / multiply), inside its crop rectangle. Each frame is decoded by the
// ordinary pipeline into float samples of the output encoding (interleaved colour [+ alpha], the frame's own size); k_blend_layer folds it
// into a canvas-sized float image that starts as a copy of the source slot; k_finalize_canvas turns the canvas shown into what
// setLayerData receives (unpremultiply: JxlDecoderSetUnpremultiplyAlpha, :233; sample type; orientation).
// Blend arithmetic as in oracle/jxlo_image.h BlendPixel ([M]: restated from memory of libjxl's blending stage, unpinned).
#include <cuda_fp16.h>
#include "kernels.h"

namespace jxlgpu {

__device__ __forceinline__ float Clamp01(float v) { return fminf(1.f, fmaxf(0.f, v)); }

// One thread per pixel of the frame. C = samples per pixel (colour channels + alpha), cc = colour channels (1 or 3).
__global__ void __launch_bounds__(256) k_blend_layer(float* __restrict__ canvas, const float* __restrict__ frame, int W, int H, int fw, int fh, int x0, int y0, int C, int cc,
                                                     uint32_t cmode, uint32_t amode, uint32_t cclamp, uint32_t aclamp, uint32_t premultiplied) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y; if (x >= fw || y >= fh) return;
  const int cx = x + x0, cy = y + y0; if (cx < 0 || cx >= W || cy < 0 || cy >= H) return;
  const float* fg = frame + (size_t(y) * fw + x) * C; float* bg = canvas + (size_t(cy) * W + cx) * C; const bool has_alpha = C > cc;
  const float ba = has_alpha ? bg[cc] : 1.f, fa = has_alpha ? fg[cc] : 1.f;
  if (has_alpha) {
    const float fac = aclamp ? Clamp01(fa) : fa; float oa;
    switch (amode) { case 0: oa = fa; break; case 1: oa = ba + fa; break; case 2: oa = 1.f - (1.f - fac) * (1.f - ba); break; case 3: oa = ba; break; default: oa = ba * fac; break; }
    bg[cc] = oa;
  }
  const float fac = cclamp ? Clamp01(fa) : fa;
  for (int c = 0; c < cc; c++) {
    const float f = fg[c], b = bg[c]; float o;
    switch (cmode) {
      case 0: o = f; break;
      case 1: o = b + f; break;
      case 2:
        if (premultiplied) o = f + b * (1.f - fac);
        else { const float na = 1.f - (1.f - fac) * (1.f - ba); const float rna = na > 0.f ? 1.f / na : 0.f; o = (f * fac + b * ba * (1.f - fac)) * rna; }
        break;
      case 3: o = b + f * fac; break;
      default: o = b * (cclamp ? Clamp01(f) : f); break;
    }
    bg[c] = o;
  }
}

__device__ __forceinline__ void StoreSampleC(uint8_t* dst, uint32_t type, float v) {
  switch (type) {
    case 0: *dst = uint8_t(__float2int_rn(Clamp01(v) * 255.0f)); break;
    case 1: *reinterpret_cast<uint16_t*>(dst) = uint16_t(__float2int_rn(Clamp01(v) * 65535.0f)); break;
    case 2: *reinterpret_cast<__half*>(dst) = __float2half_rn(v); break;
    default: *reinterpret_cast<float*>(dst) = v; break;
  }
}

// One thread per canvas pixel: unpremultiply, convert, store at the oriented position (orientation 1..8 as in the image header).
__global__ void __launch_bounds__(256) k_finalize_canvas(const float* __restrict__ canvas, uint8_t* __restrict__ out, int W, int H, int C, int cc, uint32_t premultiplied, uint32_t sample_type, uint32_t orientation) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y; if (x >= W || y >= H) return;
  const float* src = canvas + (size_t(y) * W + x) * C; float v[4]; for (int c = 0; c < C; c++) v[c] = src[c];
  if (C > cc && premultiplied) { const float mul = 1.0f / fmaxf(1.0f / 67108864.0f, v[cc]); for (int c = 0; c < cc; c++) v[c] *= mul; }
  int ox, oy;
  switch (orientation) { case 2: ox = W - 1 - x; oy = y; break; case 3: ox = W - 1 - x; oy = H - 1 - y; break; case 4: ox = x; oy = H - 1 - y; break;
    case 5: ox = y; oy = x; break; case 6: ox = H - 1 - y; oy = x; break; case 7: ox = H - 1 - y; oy = W - 1 - x; break; case 8: ox = y; oy = W - 1 - x; break; default: ox = x; oy = y; }
  const int out_w = orientation >= 5 ? H : W; const uint32_t bps = sample_type == 0 ? 1 : sample_type == 3 ? 4 : 2;
  uint8_t* dst = out + (size_t(oy) * out_w + ox) * bps * C;
  for (int c = 0; c < C; c++) StoreSampleC(dst + bps * c, sample_type, v[c]);
}

// BGRA32 surface from the canvas (JxlB200LoadImageBgra on a layered file): colour to 8 bits, gray replicated, alpha to 8 bits or 255.
__global__ void __launch_bounds__(256) k_finalize_canvas_bgra(const float* __restrict__ canvas, uint32_t* __restrict__ out, int W, int H, int C, int cc, uint32_t premultiplied, uint32_t orientation) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y; if (x >= W || y >= H) return;
  const float* src = canvas + (size_t(y) * W + x) * C; float v[4]; for (int c = 0; c < C; c++) v[c] = src[c];
  if (C > cc && premultiplied) { const float mul = 1.0f / fmaxf(1.0f / 67108864.0f, v[cc]); for (int c = 0; c < cc; c++) v[c] *= mul; }
  int ox, oy;
  switch (orientation) { case 2: ox = W - 1 - x; oy = y; break; case 3: ox = W - 1 - x; oy = H - 1 - y; break; case 4: ox = x; oy = H - 1 - y; break;
    case 5: ox = y; oy = x; break; case 6: ox = H - 1 - y; oy = x; break; case 7: ox = H - 1 - y; oy = W - 1 - x; break; case 8: ox = y; oy = W - 1 - x; break; default: ox = x; oy = y; }
  const int out_w = orientation >= 5 ? H : W;
  const uint32_t r8 = uint32_t(__float2int_rn(Clamp01(v[0]) * 255.0f)), g8 = cc == 1 ? r8 : uint32_t(__float2int_rn(Clamp01(v[1]) * 255.0f)), b8 = cc == 1 ? r8 : uint32_t(__float2int_rn(Clamp01(v[2]) * 255.0f));
  const uint32_t a8 = C > cc ? uint32_t(__float2int_rn(Clamp01(v[cc]) * 255.0f)) : 255u;
  out[size_t(oy) * out_w + ox] = b8 | (g8 << 8) | (r8 << 16) | (a8 << 24);
}

void LaunchBlendLayer(float* canvas, const float* frame, int W, int H, int fw, int fh, int x0, int y0, int C, int cc, uint32_t cmode, uint32_t amode, bool cclamp, bool aclamp, bool premultiplied, cudaStream_t st) {
  if (fw <= 0 || fh <= 0) return; dim3 grid((fw + 255) / 256, fh);
  Launch<k_blend_layer>(grid, 256, 0, st, canvas, frame, W, H, fw, fh, x0, y0, C, cc, cmode, amode, cclamp, aclamp, premultiplied);
}
void LaunchFinalizeCanvas(const float* canvas, uint8_t* out, int W, int H, int C, int cc, bool premultiplied, uint32_t sample_type, uint32_t orientation, bool bgra, cudaStream_t st) {
  dim3 grid((W + 255) / 256, H);
  if (bgra) Launch<k_finalize_canvas_bgra>(grid, 256, 0, st, canvas, reinterpret_cast<uint32_t*>(out), W, H, C, cc, premultiplied, orientation);
  else Launch<k_finalize_canvas>(grid, 256, 0, st, canvas, out, W, H, C, cc, premultiplied, sample_type, orientation);
}

}  // namespace jxlgpu
