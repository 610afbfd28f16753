// pdn-jpegxl_b200 engine — host-side bitstream front-end (bit reader/writer and field codes).
// Part of the product: parses what must be parsed serially on the CPU (container, image and
// frame headers, TOC, entropy-code headers, MA tree) and hands flat tables to the sm_100a
// kernels. Replaces the libjxl work reached from N/Decoder/JxlDecoder.cpp:252,454 and
// N/Encoder/JxlEncoder.cpp:128,367 of the reference. Field codes per ISO/IEC 18181-1 as
// digested in SURVEY.md Appendix A (A.2).
#pragma once
#include <cstdint>
#include <cstddef>
#include <cstring>
#include <cmath>
#include <vector>
#include <string>
#include <stdexcept>
#include <algorithm>

namespace jxlgpu {

struct Error : std::runtime_error {
  explicit Error(const std::string& s) : std::runtime_error(s) {}
};
// A failure the C ABI reports with its own status (a DecoderStatus or EncoderStatus) instead of DecodeError / EncodeError.
struct StatusError : Error {
  int32_t status;
  explicit StatusError(int32_t st, const std::string& s = std::string()) : Error(s), status(st) {}
};
#define JXLG_CHECK(c, msg) do { if (!(c)) throw ::jxlgpu::Error(msg); } while (0)

// U32 distribution descriptor: Val(c) | Bits(n) | BitsOffset(n, off)   (SURVEY A.2)
struct Dist { int nbits; uint32_t off; };
inline constexpr Dist Val(uint32_t c) { return Dist{0, c}; }
inline constexpr Dist Bits(int n) { return Dist{n, 0}; }
inline constexpr Dist BitsOffset(int n, uint32_t o) { return Dist{n, o}; }

inline int CeilLog2(uint64_t x) { int r = 0; while ((uint64_t(1) << r) < x) r++; return r; }   // x>=1
inline int FloorLog2(uint64_t x) { int r = 0; while (x >>= 1) r++; return r; }                    // x>=1
inline uint32_t PackSigned(int32_t v) { return (uint32_t(v) << 1) ^ uint32_t(v >> 31); }
inline int32_t UnpackSigned(uint32_t u) { return int32_t(u >> 1) ^ -int32_t(u & 1); }

// LSB-first bit reader over a byte range (SURVEY A.2). Reads past the end return zeros and
// latch `overrun`; callers turn that into the reference's truncated-input DecodeError
// (N/Decoder/JxlDecoder.cpp:402-406).
struct BitReader {
  const uint8_t* d = nullptr; size_t n = 0; size_t pos = 0; bool overrun = false;
  BitReader() {}
  BitReader(const uint8_t* data, size_t size) : d(data), n(size) {}
  inline uint64_t Peek(int nb) {  // nb <= 56
    size_t byte = pos >> 3; int sh = pos & 7; uint64_t v = 0;
    if (byte + 8 <= n) { memcpy(&v, d + byte, 8); }
    else { for (size_t i = 0; i < 8 && byte + i < n; i++) v |= uint64_t(d[byte + i]) << (8 * i); }
    v >>= sh;
    return nb >= 64 ? v : (v & ((uint64_t(1) << nb) - 1));
  }
  inline void Skip(size_t nb) { pos += nb; if (pos > n * 8) overrun = true; }
  inline uint32_t ReadBits(int nb) { if (nb == 0) return 0; uint64_t v = Peek(nb); Skip(nb); return uint32_t(v); }
  inline bool Bool() { return ReadBits(1) != 0; }
  uint32_t U32(Dist d0, Dist d1, Dist d2, Dist d3) {
    Dist ds[4] = {d0, d1, d2, d3}; Dist d_ = ds[ReadBits(2)];
    return ReadBits(d_.nbits) + d_.off;
  }
  uint64_t U64() {
    uint32_t sel = ReadBits(2);
    if (sel == 0) return 0; if (sel == 1) return 1 + ReadBits(4); if (sel == 2) return 17 + ReadBits(8);
    uint64_t v = ReadBits(12); int s = 12;
    while (ReadBits(1)) { if (s == 60) { v |= uint64_t(ReadBits(4)) << 60; break; } v |= uint64_t(ReadBits(8)) << s; s += 8; }
    return v;
  }
  float F16() {
    uint32_t b = ReadBits(16); uint32_t sign = b >> 15, e = (b >> 10) & 31, m = b & 1023;
    JXLG_CHECK(e != 31, "F16 inf/nan");
    float v;
    if (e == 0) v = std::ldexp(float(m), -24); else v = std::ldexp(float(m | 1024), int(e) - 25);
    return sign ? -v : v;
  }
  uint32_t Enum() { uint32_t v = U32(Val(0), Val(1), BitsOffset(4, 2), BitsOffset(6, 18)); JXLG_CHECK(v < 64, "enum"); return v; }
  uint32_t U8() { if (!ReadBits(1)) return 0; int nb = ReadBits(3); return (1u << nb) + ReadBits(nb); }
  void ZeroPadToByte() { int r = (8 - (pos & 7)) & 7; uint32_t v = ReadBits(r); JXLG_CHECK(v == 0, "non-zero padding"); }
  void Extensions() {
    uint64_t ext = U64(); if (!ext) return; uint64_t total = 0;
    for (int i = 0; i < 64; i++) if (ext >> i & 1) total += U64();
    Skip(total);
  }
};

struct BitWriter {
  std::vector<uint8_t> buf; size_t pos = 0;  // pos in bits
  void Write(int nb, uint64_t v) {           // nb <= 56
    if (nb == 0) return;
    size_t need = (pos + nb + 7) / 8 + 8; if (buf.size() < need) buf.resize(need * 2, 0);
    size_t byte = pos >> 3; int sh = pos & 7; uint64_t cur; memcpy(&cur, &buf[byte], 8);
    cur |= (v & ((nb >= 64) ? ~uint64_t(0) : ((uint64_t(1) << nb) - 1))) << sh; memcpy(&buf[byte], &cur, 8);
    if (sh + nb > 64) buf[byte + 8] |= uint8_t(v >> (64 - sh));
    pos += nb;
  }
  void Bool(bool b) { Write(1, b); }
  // Chooses the first distribution that can represent v.
  void U32(Dist d0, Dist d1, Dist d2, Dist d3, uint32_t v) {
    Dist ds[4] = {d0, d1, d2, d3};
    for (int i = 0; i < 4; i++) {
      uint64_t lo = ds[i].off, hi = uint64_t(ds[i].off) + ((uint64_t(1) << ds[i].nbits) - 1);
      if (v >= lo && v <= hi) { Write(2, i); Write(ds[i].nbits, v - ds[i].off); return; }
    }
    throw Error("U32 value not representable");
  }
  void U64(uint64_t v) {
    if (v == 0) { Write(2, 0); return; } if (v <= 16) { Write(2, 1); Write(4, v - 1); return; }
    if (v <= 272) { Write(2, 2); Write(8, v - 17); return; }
    Write(2, 3); Write(12, v & 4095); v >>= 12; int s = 12;
    while (v) { Write(1, 1); if (s == 60) { Write(4, v & 15); return; } Write(8, v & 255); v >>= 8; s += 8; }
    Write(1, 0);
  }
  static uint16_t FloatToHalf(float f) {   // exact only for representable values; RNE otherwise
    uint32_t x; memcpy(&x, &f, 4); uint32_t sign = (x >> 16) & 0x8000; int e = int((x >> 23) & 255) - 127 + 15; uint32_t m = x & 0x7fffff;
    if (e <= 0) { if (e < -10) return sign; m |= 0x800000; int sh = 14 - e; uint32_t r = m >> sh; uint32_t rem = m & ((1u << sh) - 1), half = 1u << (sh - 1);
      if (rem > half || (rem == half && (r & 1))) r++; return sign | r; }
    if (e >= 31) return sign | 0x7bff;
    uint32_t r = (uint32_t(e) << 10) | (m >> 13); uint32_t rem = m & 0x1fff; if (rem > 0x1000 || (rem == 0x1000 && (r & 1))) r++;
    return sign | r;
  }
  void F16(float f) { Write(16, FloatToHalf(f)); }
  void Enum(uint32_t v) { U32(Val(0), Val(1), BitsOffset(4, 2), BitsOffset(6, 18), v); }
  void U8(uint32_t v) { if (v == 0) { Write(1, 0); return; } Write(1, 1); int nb = FloorLog2(v); Write(3, nb); Write(nb, v - (1u << nb)); }
  void ZeroPadToByte() { pos = (pos + 7) & ~size_t(7); }
  void AppendBytes(const uint8_t* p, size_t n) { ZeroPadToByte(); for (size_t i = 0; i < n; i++) Write(8, p[i]); }
  std::vector<uint8_t> Finish() { ZeroPadToByte(); std::vector<uint8_t> out(buf.begin(), buf.begin() + std::min(buf.size(), pos / 8)); out.resize(pos / 8, 0); return out; }
};

}  // namespace jxlgpu
