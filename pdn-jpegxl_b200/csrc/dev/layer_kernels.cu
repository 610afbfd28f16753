// pdn-jpegxl_b200 engine — the managed layer repack of the reference as one GPU epilogue.
//
// After LoadImage returns, the reference's managed side splits the interleaved native buffer into the two bitmaps a Paint.NET layer
// is made of (I/DecoderLayerData.cs:127-992, eighteen Set*ImageData variants): a colour bitmap — Rgb24 / Rgb48 / Rgb48Half / Rgb96Float
// with gray replicated into R, G and B (:294-616), Cmyk32 for CMYK (:164-243) — and an Alpha8 transparency bitmap whose samples go
// through TransparencyMapping.ToEightBit (I/TransparencyMapping.cs:18-32: u16 / 257, clamp(half) * 255 and clamp(float) * 255,
// truncated). k_split_layers does that split on the device, straight from the decoder's output buffer, so that only the two final
// bitmaps cross PCIe (JxlB200LoadImageLayers).
#include <cuda_fp16.h>
#include "kernels.h"

namespace jxlgpu {

__device__ __forceinline__ uint8_t AlphaToEightBit(uint8_t v) { return v; }
__device__ __forceinline__ uint8_t AlphaToEightBit(uint16_t v) { return uint8_t(v / 257u); }
__device__ __forceinline__ uint8_t AlphaToEightBit(__half v) {
  // Half.Clamp(value, 0, 1) * 255 is evaluated in half precision (the product is rounded to a half) and then truncated
  const __half c = __hmin(__hmax(v, __float2half(0.0f)), __float2half(1.0f));
  const __half p = __float2half_rn(__half2float(c) * 255.0f);   // one rounding: the exact product fits a float
  const float f = __half2float(p); return (f != f) ? uint8_t(0) : uint8_t(int(f));
}
__device__ __forceinline__ uint8_t AlphaToEightBit(float v) { const float c = fminf(fmaxf(v, 0.0f), 1.0f) * 255.0f; return (c != c) ? uint8_t(0) : uint8_t(int(c)); }

// One thread per pixel. SRC = interleaved channels per pixel in the native buffer, NCOL = colour channels there (1 gray, 3 RGB,
// 4 CMYK), DST = channels of the colour bitmap (3, or 4 for CMYK). Rows are tightly packed on both sides.
template <typename T, int NCOL, int DST, bool ALPHA>
__global__ void __launch_bounds__(256) k_split_layers(const T* __restrict__ src, T* __restrict__ color, uint8_t* __restrict__ alpha, size_t npix) {
  const size_t i = size_t(blockIdx.x) * 256 + threadIdx.x; if (i >= npix) return;
  constexpr int SRC = NCOL + (ALPHA ? 1 : 0);
  T v[SRC];
#pragma unroll
  for (int c = 0; c < SRC; c++) v[c] = src[i * SRC + c];
#pragma unroll
  for (int c = 0; c < DST; c++) color[i * DST + c] = v[NCOL == 1 ? 0 : c];
  if (ALPHA) alpha[i] = AlphaToEightBit(v[NCOL]);
}

template <typename T>
static void SplitT(const void* src, void* color, uint8_t* alpha, size_t npix, int format, bool has_alpha, cudaStream_t st) {
  const unsigned grid = unsigned((npix + 255) / 256); const T* s = static_cast<const T*>(src); T* c = static_cast<T*>(color);
  if (format == 0) { if (has_alpha) Launch<k_split_layers<T, 1, 3, true>>(grid, 256, 0, st, s, c, alpha, npix); else Launch<k_split_layers<T, 1, 3, false>>(grid, 256, 0, st, s, c, alpha, npix); }
  else if (format == 1) { if (has_alpha) Launch<k_split_layers<T, 3, 3, true>>(grid, 256, 0, st, s, c, alpha, npix); else Launch<k_split_layers<T, 3, 3, false>>(grid, 256, 0, st, s, c, alpha, npix); }
  else { if (has_alpha) Launch<k_split_layers<T, 4, 4, true>>(grid, 256, 0, st, s, c, alpha, npix); else Launch<k_split_layers<T, 4, 4, false>>(grid, 256, 0, st, s, c, alpha, npix); }
}

// format: DecoderImageFormat (0 Gray, 1 Rgb, 2 Cmyk); sample_type: 0 u8, 1 u16, 2 f16, 3 f32
void LaunchSplitLayers(const void* src, void* color, uint8_t* alpha, size_t npix, int format, int sample_type, bool has_alpha, cudaStream_t st) {
  if (!npix) return;
  switch (sample_type) {
    case 0: SplitT<uint8_t>(src, color, alpha, npix, format, has_alpha, st); break;
    case 1: SplitT<uint16_t>(src, color, alpha, npix, format, has_alpha, st); break;
    case 2: SplitT<__half>(src, color, alpha, npix, format, has_alpha, st); break;
    default: SplitT<float>(src, color, alpha, npix, format, has_alpha, st); break;
  }
}

}  // namespace jxlgpu
