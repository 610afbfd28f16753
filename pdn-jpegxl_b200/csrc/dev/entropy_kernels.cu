// pdn-jpegxl_b200 engine — entropy-decoding kernels (sm_100a).
//   k_lf_group : one CTA per LF group (2048x2048 px): LF coefficients (Modular, 3 channels at 1/8 res),
//                HF metadata (CfL maps, block strategies + hf multipliers, EPF sharpness), varblock placement.
//   k_ac_vardct: AC coefficients of the 256x256 groups of one pass: ANS/prefix decode with the context model of
//                SURVEY.md A.8 "PassGroup AC decode"; one lane per section, 1..32 sections per warp.
//   k_mod_group: the groups' Modular channels (alpha / lossless colour).
// A section is a serial bit stream (per-symbol adaptive contexts), so one thread is productive per CTA; the
// other lanes zero-fill, stage tables and post-process. Throughput comes from the number of sections in
// flight (192 AC groups for 12 MP, x batch). Replaces libjxl's DecodeGroup / ModularFrameDecoder work reached
// from N/Decoder/JxlDecoder.cpp:252.
#include "frame.cuh"
#include "kernels.h"
#include <cstdlib>
#include <algorithm>

namespace jxlgpu {

__device__ __constant__ uint8_t kFreqCtx[64] = {0, 0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 15, 16, 16, 17, 17, 18, 18, 19, 19, 20, 20, 21, 21, 22, 22,
  23, 23, 23, 23, 24, 24, 24, 24, 25, 25, 25, 25, 26, 26, 26, 26, 27, 27, 27, 27, 28, 28, 28, 28, 29, 29, 29, 29, 30, 30, 30, 30};
__device__ __constant__ uint8_t kNumNzCtx[64] = {0, 0, 31, 62, 62, 93, 93, 93, 93, 123, 123, 123, 123, 152, 152, 152, 152, 152, 152, 152, 152, 180, 180, 180, 180, 180, 180, 180, 180, 180, 180, 180, 180,
  206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206};

// Parses a Modular GroupHeader (A.7 "Sub-bitstream header"). Streams that need host-side parsing
// (local MA trees, per-group transforms) are reported as unsupported instead of being mis-decoded.
__device__ __forceinline__ const DLocalTree* LocalTreeOf(const DFrame& f, uint32_t index) { return f.local_off ? reinterpret_cast<const DLocalTree*>(f.blob + f.local_off) + index : nullptr; }
// Switches the decoder to a stream's own MA tree and code (tables in global memory: the speculative shared-memory loop does not apply)
__device__ void BindLocalTree(ModDecoder& md, const DFrame& f, const DLocalTree& lt) {
  md.tree = reinterpret_cast<const DTreeNode*>(f.blob + lt.tree_off); md.cv.Bind(f.blob, lt.code); md.uses_wp = lt.uses_wp != 0; md.rd.br.Init(f.comp, lt.data_bitpos);
}
__device__ bool ReadGroupHeaderDev(ModDecoder& md, const DFrame& f, const DLocalTree* lt = nullptr, bool rct_allowed = false) {
  BitRd& br = md.rd.br;
  bool use_global = br.Read(1);
  if (!br.Read(1)) { md.wp.p1 = br.Read(5); md.wp.p2 = br.Read(5); md.wp.p3a = br.Read(5); md.wp.p3b = br.Read(5); md.wp.p3c = br.Read(5); md.wp.p3d = br.Read(5); md.wp.p3e = br.Read(5); for (int i = 0; i < 4; i++) md.wp.w[i] = br.Read(4); }
  else { md.wp.p1 = 16; md.wp.p2 = 10; md.wp.p3a = 7; md.wp.p3b = 7; md.wp.p3c = 7; md.wp.p3d = 0; md.wp.p3e = 0; md.wp.w[0] = 13; md.wp.w[1] = 12; md.wp.w[2] = 12; md.wp.w[3] = 12; }
  uint32_t nt = br.ReadU32(0, 0, 0, 1, 4, 2, 8, 18);
  GroupTransforms* gt = md.gt; if (gt) gt->n = 0;
  if (nt != 0 && (!rct_allowed || !gt || nt > uint32_t(GroupTransforms::kMax))) { md.rd.err = kErrGroupTransform; return false; }
  for (uint32_t i = 0; i < nt; i++) {
    const uint32_t id = br.Read(2); if (id > 1) { md.rd.err = kErrGroupTransform; return false; }   // squeeze inside a group section
    const uint32_t begin_c = br.ReadU32(3, 0, 6, 8, 10, 72, 13, 1096); uint32_t a, b = 0;
    if (id == 0) { a = br.ReadU32(0, 6, 2, 0, 4, 2, 6, 10); if (a >= 42) { md.rd.err = kErrGroupTransform; return false; } }
    else {
      a = br.ReadU32(0, 1, 0, 3, 0, 4, 13, 1); b = br.ReadU32(8, 0, 10, 256, 12, 1280, 16, 5376); const uint32_t nb_deltas = br.ReadU32(0, 0, 8, 1, 10, 257, 16, 1281); br.Read(4);   // predictor: only used by delta entries
      if (nb_deltas != 0 || a > 4) { md.rd.err = kErrGroupTransform; return false; }
    }
    gt->kind[gt->n] = id; gt->begin[gt->n] = begin_c; gt->a[gt->n] = a; gt->b[gt->n] = b; gt->n++;
  }
  if (!use_global) {   // the tree and the code follow in the stream: the host has parsed them (Modular frames) or the stream is not supported
    if (!lt || !lt->present) { md.rd.err = kErrLocalTree; return false; }
    BindLocalTree(md, f, *lt); return true;
  }
  if (!f.has_tree) { md.rd.err = kErrLocalTree; return false; }
  return true;
}

__device__ void BindModDecoder(ModDecoder& md, const DFrame& f, ChanLut* lut) {
  md.cv.Bind(f.blob, f.mod_code); md.tree = reinterpret_cast<const DTreeNode*>(f.blob + f.tree_off); md.uses_wp = f.uses_wp != 0; md.wide = f.mod_wide != 0; md.rd.err = 0; md.lut = lut;
}
// Stages the Modular code tables and the MA tree into shared memory (all threads of the CTA call this, then sync).
__device__ void StageModDecoder(ModDecoder& md, const DFrame& f, uint8_t* dsm, uint32_t cap, uint32_t& used, int tid, int nt) {
  if (!f.has_tree) return;
  md.cv.Stage(dsm, cap, used, tid, nt); md.tree = static_cast<const DTreeNode*>(StageBytes(dsm, cap, used, md.tree, f.tree_size * 16, tid, nt));
}

template <bool kNarrow>
__device__ __forceinline__ void LfGroupBody(const DFrame& f, const int g) {
  const int lane = threadIdx.x;
  if (f.band_on) {   // band decode: only the LF groups that cover the block rows of the band (+1 row each side for smoothing / LLF context)
    const int r0 = (g / int(f.xlfgroups)) * 256, r1 = r0 + 256, need0 = int(f.comp_g0 * (f.group_dim >> 3)) - 1, need1 = int(f.comp_g1 * (f.group_dim >> 3)) + 1;
    if (r1 <= need0 || r0 >= need1) return;
  }
  const int gx = g % int(f.xlfgroups), gy = g / int(f.xlfgroups), cx0 = gx * 256, cy0 = gy * 256;
  const int w = min(256, int(f.xb) - cx0), h = min(256, int(f.yb) - cy0), tw = (w + 7) / 8, th = (h + 7) / 8;
  int32_t* scratch = f.hfmeta_scratch + size_t(g) * kHfMetaScratchInts;
  int32_t* s_cflx = scratch; int32_t* s_cflb = scratch + 1024; int32_t* s_info = scratch + 2048; int32_t* s_sharp = scratch + 2048 + 2 * 65536;
  __shared__ uint32_t sh_nb, sh_ok, sh_hdr_ok; __shared__ ChanLut sh_lut; __shared__ LeanSpecPrep sh_prep; extern __shared__ __align__(16) uint8_t dsm[];
  uint32_t used = 0;
  ModDecoder md; BindModDecoder(md, f, &sh_lut); StageModDecoder(md, f, dsm, f.lf_smem, used, lane, 32);
  // LF coefficients and HF metadata are small integers whatever the bit depth of the image (|LF| < 2^24 even at the finest quantiser): 32-bit
  // arithmetic is exact for them, so a float32 / 32-bit image does not push its LF groups onto the 64-bit path (r02: 100 ms -> 29 ms at 8K float32)
  md.wide = false;
  __syncthreads();
  // room left in the dynamic shared memory for the transposed alias table of the speculative loop (DecodeRowsLeanSpec)
  const uint32_t spec_off = (used + 15u) & ~15u, spec_bytes = f.lf_smem > spec_off ? f.lf_smem - spec_off : 0u;
  const uint64_t* sec = SecBitPos(f); const uint32_t nsec = f.num_passes * f.num_groups + f.num_lf_groups + 2; const bool single = (f.num_groups == 1 && f.num_passes == 1);
  const uint64_t end = single ? sec[nsec] : sec[nsec + 1 + g];
  int32_t* wp = f.wp_scratch + size_t(g) * WPScratchInts(kMaxWpWidth);
  const size_t plane = size_t(f.xb) * f.yb; const int lf_sid = 1 + g;
  // ---- part A (lane 0): section start, LF-coefficient sub-bitstream header
  if (lane == 0) {
    sh_ok = 0; sh_nb = 0;
    const uint64_t start = single ? f.end_bitpos[0] : sec[1 + g];
    md.rd.br.Init(f.comp, start); if (f.lz_window) md.rd.win = f.lz_window + size_t(g) * kLzWindow; md.dist_mult = uint32_t(w);
    uint32_t extra_prec = md.rd.br.Read(2);
    f.hfmeta_scratch[size_t(f.num_lf_groups) * kHfMetaScratchInts + g] = int32_t(extra_prec);
    const bool ok = ReadGroupHeaderDev(md, f);
    if (ok) md.rd.Init(md.cv);
    sh_hdr_ok = ok ? 1 : 0;
  }
  __syncwarp();
  // ---- part B (whole warp): the three LF-coefficient channels; stream channel order is Y, X, B (A.8 LfGroup)
  if (sh_hdr_ok) {
    for (int c = 0; c < 3; c++) {
      const int dstc = c == 0 ? 1 : c == 1 ? 0 : 2; int32_t* dst = f.lfq + dstc * plane + size_t(cy0) * f.xb + cx0;
      if (lane == 0) { if (c == 0) md.ResetChannels(); md.NoteChannel(dst, f.xb, w, h, 3, 3); sh_prep.ok = 0; if (!(kNarrow && md.PrepareLeanSpec(c, lf_sid, sh_prep, spec_bytes))) md.DecodeChannel<kNarrow>(c, lf_sid, dst, f.xb, w, h, wp); }
      __syncwarp();
      if (sh_prep.ok) {   // uniform: written by lane 0 before the barrier
        DecodeRowsLeanSpec(sh_prep, reinterpret_cast<const uint8_t*>(md.cv.alias), md.cv.log_alpha, reinterpret_cast<uint2*>(dsm + spec_off), dst, f.xb, w, h, lane);
        if (lane == 0) md.FinishLeanSpec(sh_prep);
      }
      __syncwarp();
    }
  }
  // ---- part C (lane 0): HF metadata
  if (lane == 0) {
    bool ok = sh_hdr_ok != 0;
    if (ok && !md.rd.FinalOk(md.cv)) md.rd.err = md.rd.err ? md.rd.err : kErrAnsFinal;
    // (Modular LF-group channels — extra channels with dim_shift >= 3 — are rejected on the host.)
    if (ok && !md.rd.err) {
      uint32_t nb = md.rd.br.Read(CeilLog2Dev(uint32_t(w * h))) + 1; sh_nb = nb;
      ok = ReadGroupHeaderDev(md, f);
      if (ok) {
        md.rd.Init(md.cv); const int sid = 1 + 2 * int(f.num_lf_groups) + g; md.dist_mult = uint32_t(max(max(tw, w), int(min(nb, 65536u))));
        md.ResetChannels();
        md.NoteChannel(s_cflx, tw, tw, th, 3, 3); md.DecodeChannel<kNarrow>(0, sid, s_cflx, tw, tw, th, wp); md.NoteChannel(s_cflb, tw, tw, th, 3, 3); md.DecodeChannel<kNarrow>(1, sid, s_cflb, tw, tw, th, wp);
        if (nb <= 65536u) { md.NoteChannel(s_info, nb, int(nb), 2, 0, 0); md.DecodeChannel<kNarrow>(2, sid, s_info, nb, int(nb), 2, wp); md.NoteChannel(s_sharp, w, w, h, 0, 0); md.DecodeChannel<kNarrow>(3, sid, s_sharp, w, w, h, wp); } else md.rd.err = kErrHfMeta;
        if (!md.rd.FinalOk(md.cv)) md.rd.err = md.rd.err ? md.rd.err : kErrAnsFinal;
      }
    }
    uint64_t pos = md.rd.br.BitPos(); if (pos > end) md.rd.err = md.rd.err ? md.rd.err : kErrOverrun;
    if (single) f.end_bitpos[1] = pos;
    SetError(f.err, md.rd.err); sh_ok = (ok && !md.rd.err) ? 1 : 0;
  }
  __syncwarp();
  if (!sh_ok) return;
  // ---- parallel post-processing: CfL maps, sharpness, clear block map
  uint32_t bad = 0;
  for (int i = lane; i < tw * th; i += 32) { int y = i / tw, x = i % tw; int32_t a = s_cflx[i], b = s_cflb[i]; if (a < -128 || a > 127 || b < -128 || b > 127) bad = kErrCflRange;
    size_t o = size_t(cy0 / 8 + y) * f.xt + cx0 / 8 + x; f.ytox[o] = int8_t(a); f.ytob[o] = int8_t(b); }
  for (int i = lane; i < w * h; i += 32) { int y = i / w, x = i % w; int32_t v = s_sharp[i]; if (v < 0 || v > 7) bad = kErrSharpness; size_t o = size_t(cy0 + y) * f.xb + cx0 + x; f.sharp[o] = uint8_t(v); f.acs[o] = 0xFF; }
  if (bad) SetError(f.err, bad);
  __syncwarp();
  // ---- varblock placement: raster scan, each block at the first uncovered cell (A.8 LfGroup)
  const uint32_t nb = sh_nb; bool all1 = nb == uint32_t(w * h);
  if (all1) for (uint32_t i = lane; i < nb; i += 32) { int32_t s = s_info[i]; if (s < 0 || s >= 27 || (CoveredXLog2Dev(s) | CoveredYLog2Dev(s)) != 0) all1 = false; }
  all1 = __all_sync(0xffffffffu, all1);
  if (all1) {   // common case (only 8x8 strategies): block i sits in cell i, fully parallel
    for (uint32_t i = lane; i < nb; i += 32) { const int yy = cy0 + int(i / w), xx = cx0 + int(i % w); size_t o = size_t(yy) * f.xb + xx; f.acs[o] = uint8_t(s_info[i] | 0x80); f.hf_mul_m1[o] = uint8_t(max(0, min(255, s_info[nb + i])));
      if (s_info[i] != 0) atomicAdd(f.group_other + (yy >> 5) * f.xgroups + (xx >> 5), 1u); }
  } else {
    // Mixed strategies. Pass 1 (lane 0): walk the blocks in order against a coverage bitmap in shared memory (one bit per cell: the next free
    // cell is a find-first-set on a word, not a chain of dependent global loads) and note each block's first cell in the upper bits of its
    // s_info entry. Pass 2 (all lanes): fill the strategy / multiplier maps block by block.
    __shared__ uint32_t cov[256][8];
    for (int idx = lane; idx < 256 * 8; idx += 32) { const int row = idx >> 3, k = idx & 7, lo = k * 32;
      cov[row][k] = row >= h ? 0xffffffffu : (w >= lo + 32 ? 0u : (w <= lo ? 0xffffffffu : (0xffffffffu << (w - lo)))); }   // cells outside the group count as covered
    __syncwarp();
    if (lane == 0) {
      uint32_t e = 0; int y = 0, x = 0;
      for (uint32_t num = 0; num < nb && !e; num++) {
        for (;;) {   // first uncovered cell at or after (y, x)
          if (y >= h) { e = kErrHfMeta; break; }
          const uint32_t free_bits = ~(cov[y][x >> 5] | ((1u << (x & 31)) - 1u));
          if (free_bits) { x = (x & ~31) + __ffs(int(free_bits)) - 1; break; }
          x = (x & ~31) + 32; if (x >= w) { x = 0; y++; }
        }
        if (e) break;
        const int32_t s = s_info[num]; if (s < 0 || s >= 27) { e = kErrBadStrategy; break; }
        const int bw = 1 << CoveredXLog2Dev(s), bh = 1 << CoveredYLog2Dev(s);
        if (x + bw > w || y + bh > h || (x & 31) + bw > 32 || (y & 31) + bh > 32) { e = kErrBlockBounds; break; }
        const uint32_t m = (bw == 32 ? 0xffffffffu : ((1u << bw) - 1u)) << (x & 31);
        for (int iy = 0; iy < bh; iy++) { if (cov[y + iy][x >> 5] & m) e = kErrBlockBounds; cov[y + iy][x >> 5] |= m; }
        s_info[num] = s | (x << 8) | (y << 16);
        if (bw > 4 || bh > 4) { atomicOr(f.err + 12, 1u); *reinterpret_cast<volatile uint32_t*>(f.host_flags) = 1u; }   // host_flags: page-locked host word, read by the host once this kernel has drained: a transform of 64 px or more needs the second plane set (xyb_tmp)
        x += bw; if (x >= w) { x = 0; y++; }
      }
      SetError(f.err, e);
    }
    __syncwarp();
    uint32_t bad_cov = 0;   // every cell must be covered once the blocks are placed
    for (int idx = lane; idx < h * 8; idx += 32) if (cov[idx >> 3][idx & 7] != 0xffffffffu) bad_cov = kErrHfMeta;
    if (bad_cov) SetError(f.err, bad_cov);
    for (uint32_t i = lane; i < nb; i += 32) {
      const int32_t info = s_info[i]; const int s = info & 0xff, x = (info >> 8) & 0xff, y = (info >> 16) & 0xff; if (s >= 27) continue;
      const int bw = 1 << CoveredXLog2Dev(s), bh = 1 << CoveredYLog2Dev(s); if (x + bw > w || y + bh > h) continue;   // (pass 1 stopped on an error: entries beyond it are unplaced)
      const uint8_t qf = uint8_t(max(0, min(255, s_info[nb + i]))); const size_t o = size_t(cy0 + y) * f.xb + cx0 + x;
      for (int iy = 0; iy < bh; iy++) for (int ix = 0; ix < bw; ix++) { const size_t p = o + size_t(iy) * f.xb + ix; f.acs[p] = uint8_t(s); f.hf_mul_m1[p] = qf; }
      f.acs[o] = uint8_t(s | 0x80);
      if (s != 0) atomicAdd(f.group_other + ((cy0 + y) >> 5) * f.xgroups + ((cx0 + x) >> 5), 1u + ((bw > 4 || bh > 4) ? 0x10000u : 0u));   // low half: non-DCT8 varblocks, high half: those of 64 px and more
    }
  }
}

// The first-wave CTA->SM mapping is deterministic, so concurrent images would stack their few LF CTAs on the same SMs:
// each launch prepends `lf_cta_offset` empty CTAs to land on different SMs.
// Register budget: one warp per CTA, at least 12 CTAs per SM (a 256-image batch of 12 MP files keeps about 7 LF CTAs on each SM), which
// allows up to 168 registers. Left to ptxas's default target, the narrow variants get 96 and spill around the decode calls.
constexpr int kLfMinCtasPerSm = 12;
template <bool kNarrow>
__global__ void __launch_bounds__(32, kLfMinCtasPerSm) k_lf_group(const __grid_constant__ DFrame f) {
  if (blockIdx.x < f.lf_cta_offset) return;
  LfGroupBody<kNarrow>(f, int(blockIdx.x - f.lf_cta_offset));
}
// Several images per launch (DFrameSet): the image is found from the CTA index.
template <bool kNarrow>
__global__ void __launch_bounds__(32, kLfMinCtasPerSm) k_lf_group_multi(const __grid_constant__ DFrameSet s) {
  if (blockIdx.x < s.cta_offset) return;
  const uint32_t cta = blockIdx.x - s.cta_offset; uint32_t img = 0; while (img + 1 < s.n && cta >= s.first[img + 1]) img++;
  LfGroupBody<kNarrow>(s.f[img], int(cta - s.first[img]));
}

// LF dequantisation + chroma-from-luma + block-context LF index (A.8 "Dequant", BlockCtxMap)
__global__ void k_lf_dequant(const DFrame* fp) {
  const DFrame& f = *fp; size_t plane = size_t(f.xb) * f.yb; size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; if (i >= plane) return;
  int y = int(i / f.xb), x = int(i % f.xb); int g = (y / 256) * int(f.xlfgroups) + x / 256;
  float mul = 1.0f / float(1u << uint32_t(f.hfmeta_scratch[size_t(f.num_lf_groups) * kHfMetaScratchInts + g]));
  int32_t qx = f.lfq[i], qy = f.lfq[plane + i], qb = f.lfq[2 * plane + i];
  float Y = float(qy) * (f.lf_fac[1] * mul); f.lf[plane + i] = Y; f.lf[i] = float(qx) * (f.lf_fac[0] * mul) + f.cfl_x_lf * Y; f.lf[2 * plane + i] = float(qb) * (f.lf_fac[2] * mul) + f.cfl_b_lf * Y;
  uint32_t bx = 0, by = 0, bb = 0;
  for (uint32_t t = 0; t < f.n_lf_thr[0]; t++) bx += qx > f.lf_thr[0][t]; for (uint32_t t = 0; t < f.n_lf_thr[1]; t++) by += qy > f.lf_thr[1][t]; for (uint32_t t = 0; t < f.n_lf_thr[2]; t++) bb += qb > f.lf_thr[2][t];
  f.lf_idx[i] = uint8_t((bx * (f.n_lf_thr[2] + 1) + bb) * (f.n_lf_thr[1] + 1) + by);
}

// Adaptive LF smoothing (A.8): lf -> lf_tmp, 3 channels; borders copied.
__global__ void k_lf_smooth(const DFrame* fp) {
  const DFrame& f = *fp; const int w = int(f.xb), h = int(f.yb); size_t plane = size_t(w) * h; size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; if (i >= plane) return;
  int y = int(i / w), x = int(i % w);
  if (x == 0 || y == 0 || x == w - 1 || y == h - 1) { for (int c = 0; c < 3; c++) f.lf_tmp[c * plane + i] = f.lf[c * plane + i]; return; }
  const float kW1 = 0.20345139757231578f, kW2 = 0.0334829185968739f, kW0 = 1.0f - 4.0f * (kW1 + kW2);
  float sm[3], mc[3], gap = 0.5f;
  for (int c = 0; c < 3; c++) { const float* p = f.lf + c * plane + i; float corner = p[-w - 1] + p[-w + 1] + p[w - 1] + p[w + 1], edge = p[-w] + p[-1] + p[1] + p[w]; mc[c] = p[0]; sm[c] = mc[c] * kW0 + edge * kW1 + corner * kW2;
    gap = fmaxf(gap, fabsf((mc[c] - sm[c]) / f.lf_fac[c])); }
  float factor = fmaxf(0.f, 3.0f - 4.0f * gap);
  for (int c = 0; c < 3; c++) f.lf_tmp[c * plane + i] = (sm[c] - mc[c]) * factor + mc[c];
}

// Decodes the group-local Modular channels (extra channels of VarDCT frames, everything of Modular frames). Warp-collective: lane 0 owns the
// bit stream and parses; channels that qualify run through the speculative loop with every lane (DecodeRowsLeanSpec), the others on lane 0.
// `prep` / `flag` are this warp's shared-memory words, `T` its room for the transposed alias table (spec_bytes bytes, may be 0).
// A section covers the square (x0, y0, dim) of the frame and holds the channels whose shift min(hshift, vshift) lies in [min_shift, max_shift]:
// pass groups take the bracket of their pass (0..2 for a single pass), LF groups everything from 3 up (channels squeezed or subsampled 8x or more).
template <bool kNarrow>
__device__ void DecodeModularGroupDev(ModDecoder& md, const DFrame& f, int g, int x0, int y0, int gd, int min_shift, int max_shift, int sid, const DLocalTree* lt, int32_t* wp, int lane,
                                      LeanSpecPrep& prep, volatile uint32_t* flag, uint2* T, uint32_t spec_bytes) {
  auto region = [&](uint32_t c, int& rx0, int& ry0, int& rw, int& rh) -> bool {
    const DModChannel& ch = ModCh(f, c); const int shift = int(min(ch.hshift, ch.vshift)); if (shift > max_shift || shift < min_shift) return false;
    rx0 = x0 >> ch.hshift; ry0 = y0 >> ch.vshift; if (rx0 >= int(ch.w) || ry0 >= int(ch.h)) return false;
    rw = min(gd >> ch.hshift, int(ch.w) - rx0); rh = min(gd >> ch.vshift, int(ch.h) - ry0); return rw > 0 && rh > 0;
  };
  // the section's channel list: rectangles of the frame's channels (every lane derives the same list from the frame descriptor)
  struct Loc { int32_t* p; int stride, w, h, hs, vs; };
  static const int kMaxLoc = 44; Loc loc[kMaxLoc]; int nloc = 0; uint32_t dm = 0;   // a squeezed image has a few dozen residual channels per section
  bool too_many = false;
  for (uint32_t c = f.first_group_channel; c < f.num_mod_channels; c++) {
    int rx0, ry0, rw, rh; if (!region(c, rx0, ry0, rw, rh)) continue;
    if (nloc >= kMaxLoc - 4) { too_many = true; break; }   // more channels in one section than the list holds: refused, never truncated
    const DModChannel& ch = ModCh(f, c); loc[nloc++] = Loc{f.mod_planes + ch.plane_off + size_t(ry0) * ch.w + rx0, int(ch.w), rw, rh, int(ch.hshift), int(ch.vshift)}; dm = max(dm, uint32_t(rw));
  }
  if (too_many) { if (lane == 0) md.rd.err = kErrUnsupportedStream; return; }
  if (nloc == 0) return;
  GroupTransforms gts; md.gt = &gts;
  if (lane == 0) { const bool ok = ReadGroupHeaderDev(md, f, lt, true); *flag = ok ? 1u : 0u; }
  md.gt = nullptr;
  __syncwarp();
  if (!*flag) return;
  // the transforms of this section's own header, for every lane (lane 0 parsed them)
  const int gt_n = int(__shfl_sync(0xffffffffu, gts.n, 0)); uint32_t gt_kind[GroupTransforms::kMax], gt_begin[GroupTransforms::kMax], gt_a[GroupTransforms::kMax], gt_b[GroupTransforms::kMax];
#pragma unroll
  for (int i = 0; i < GroupTransforms::kMax; i++) { gt_kind[i] = __shfl_sync(0xffffffffu, gts.kind[i], 0); gt_begin[i] = __shfl_sync(0xffffffffu, gts.begin[i], 0); gt_a[i] = __shfl_sync(0xffffffffu, gts.a[i], 0); gt_b[i] = __shfl_sync(0xffffffffu, gts.b[i], 0); }
  // ---- the channel list as coded: a palette replaces its channels by one index channel and puts the palette itself in front (meta channel)
  Loc saved[GroupTransforms::kMax][3]; int nb_meta = 0; uint32_t pal_used = 0; bool bad = false;
  for (int t = 0; t < gt_n && !bad; t++) {
    if (gt_kind[t] != 1) continue;
    const int b0 = int(gt_begin[t]), nc = int(gt_a[t]), ncol = int(gt_b[t]);
    if (b0 < nb_meta || b0 + nc > nloc || nloc + 1 > kMaxLoc || pal_used + uint32_t(ncol * nc) > kGroupPalInts || !f.group_pal) { bad = true; break; }
    for (int j = 1; j < nc; j++) { bad = bad || loc[b0 + j].w != loc[b0].w || loc[b0 + j].h != loc[b0].h; saved[t][j - 1] = loc[b0 + j]; }
    for (int j = b0 + nc; j < nloc; j++) loc[j - (nc - 1)] = loc[j];
    nloc -= nc - 1;
    for (int j = nloc; j > 0; j--) loc[j] = loc[j - 1];
    loc[0] = Loc{f.group_pal + size_t(g) * kGroupPalInts + pal_used, ncol, ncol, nc, -1, -1}; nloc++; nb_meta++; pal_used += uint32_t(ncol * nc); dm = max(dm, uint32_t(ncol));
  }
  if (bad) { if (lane == 0) md.rd.err = kErrGroupTransform; return; }
  if (lane == 0) { md.rd.Init(md.cv); md.dist_mult = dm; }
  for (int k = 0; k < nloc; k++) {
    const Loc& L = loc[k];
    if (lane == 0) { if (k == 0) md.ResetChannels(); md.NoteChannel(L.p, size_t(L.stride), L.w, L.h, L.hs, L.vs); prep.ok = 0; if (!(kNarrow && md.PrepareLeanSpec(k, sid, prep, spec_bytes))) md.DecodeChannel<kNarrow>(k, sid, L.p, size_t(L.stride), L.w, L.h, wp); }
    __syncwarp();
    if (prep.ok) { DecodeRowsLeanSpec(prep, reinterpret_cast<const uint8_t*>(md.cv.alias), md.cv.log_alpha, T, L.p, size_t(L.stride), L.w, L.h, lane); if (lane == 0) md.FinishLeanSpec(prep); }
    __syncwarp();
  }
  if (lane == 0 && !md.rd.FinalOk(md.cv)) md.rd.err = md.rd.err ? md.rd.err : kErrAnsFinal;
  // ---- undo the section's own transforms on its rectangles, last listed first
  __syncwarp();
  for (int t = gt_n - 1; t >= 0; t--) {
    const int b0 = int(gt_begin[t]);
    if (gt_kind[t] == 0) {
      if (b0 < nb_meta || b0 + 3 > nloc || loc[b0 + 1].w != loc[b0].w || loc[b0 + 2].w != loc[b0].w || loc[b0 + 1].h != loc[b0].h || loc[b0 + 2].h != loc[b0].h) { if (lane == 0) md.rd.err = md.rd.err ? md.rd.err : kErrGroupTransform; break; }
      const uint32_t perm = gt_a[t] / 7, kind = gt_a[t] % 7; const int rw0 = loc[b0].w, rh0 = loc[b0].h;
      for (int i = lane; i < rw0 * rh0; i += 32) {
        const int y = i / rw0, x = i - y * rw0; int32_t* q0 = loc[b0].p + size_t(y) * loc[b0].stride + x; int32_t* q1 = loc[b0 + 1].p + size_t(y) * loc[b0 + 1].stride + x; int32_t* q2 = loc[b0 + 2].p + size_t(y) * loc[b0 + 2].stride + x;
        const int32_t A = *q0, B = *q1, C = *q2; int32_t o[3];
        if (kind == 6) { const int32_t tt = A - (C >> 1), G = C + tt, Bl = tt - (B >> 1), R = Bl + B; o[0] = R; o[1] = G; o[2] = Bl; }
        else { int32_t D = A, E = B, F = C; if (kind & 1) F += A; if ((kind >> 1) == 1) E += A; if ((kind >> 1) == 2) E += (A + F) >> 1; o[0] = D; o[1] = E; o[2] = F; }
        int32_t r[3]; r[perm % 3] = o[0]; r[(perm + 1 + perm / 3) % 3] = o[1]; r[(perm + 2 - perm / 3) % 3] = o[2];
        *q0 = r[0]; *q1 = r[1]; *q2 = r[2];
      }
    } else {   // palette: loc[0] is the palette, loc[b0 + 1] the index channel; colour 0 overwrites the index plane, the others go back to their own planes
      const Loc pal = loc[0], idx = loc[b0 + 1]; const int nc = int(gt_a[t]); bool neg = false;
      for (int i = lane; i < idx.w * idx.h; i += 32) {
        const int y = i / idx.w, x = i - y * idx.w; const int index = idx.p[size_t(y) * idx.stride + x];
        for (int c = nc - 1; c >= 0; c--) { const int32_t v = PaletteLookup(pal.p + size_t(c) * pal.stride, index, c, pal.w, int(f.mod_bitdepth), &neg); const Loc& o = c == 0 ? idx : saved[t][c - 1]; o.p[size_t(y) * o.stride + x] = v; }
      }
      if (__any_sync(0xffffffffu, neg) && lane == 0) md.rd.err = md.rd.err ? md.rd.err : kErrPaletteDelta;   // only lane 0's error word is reported
      for (int j = 0; j + 1 < nloc; j++) loc[j] = loc[j + 1];   // drop the palette: the index channel is now at b0
      nloc--; nb_meta--;
      for (int j = nloc - 1; j > b0; j--) loc[j + nc - 1] = loc[j];
      for (int j = 1; j < nc; j++) loc[b0 + j] = saved[t][j - 1];
      nloc += nc - 1;
    }
    __syncwarp();
  }
}

// AC coefficients of 256x256 groups (A.8 "PassGroup AC decode"), SIMT over independent sections.
// Every section is a serial, adaptive-context bit stream, so one LANE walks one section; `lanes` (1..32) sections share a
// warp. The walk is a flat one-symbol-per-iteration state machine (block/channel set-up and coefficient placement are the
// divergent arms, the ANS step is the convergent one), so lanes at different blocks still share the instruction stream.
// lanes = 1 gives the lowest single-image latency (192 warps for 12 MP); batches raise it so that the number of resident
// sections is not capped by the register file (a lone lane still holds a full warp's registers).
// kSmem: ANS code with every table staged in shared memory (the host checks sizes before choosing the instantiation).
// Warps per CTA: the code tables are staged once per CTA, and the CTAs resident on an SM are capped by that shared memory (a
// 60 KB table set allows 3). Wide CTAs (12 warps = a whole 12 MP image at 16 sections per warp) share one copy between 12 warps, so
// a batch keeps 24 AC warps resident per SM instead of 12; single-image decodes keep small CTAs that spread over more SMs.
static const int kAcMaxWarps = 12;
static const uint32_t kAcBatchSmem = 0;   // bytes of shared memory a batch-mode AC CTA asks for at least (0: only what its tables need)
static inline int AcWarpsFor(int lanes) { return lanes >= 8 ? kAcMaxWarps : 4; }
template <bool kSmem>
__device__ __forceinline__ void AcVardctBody(const DFrame& f, const int pass, const int lanes, const int cta) {
  extern __shared__ __align__(16) uint8_t dsm[]; __shared__ uint8_t s_freq[64], s_numnz[64];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  CodeView cv; cv.Bind(f.blob, f.ac_code[pass]);
  if (tid < 64) { s_freq[tid] = kFreqCtx[tid]; s_numnz[tid] = kNumNzCtx[tid]; }
  if (kSmem) { uint32_t used = 0; cv.Stage(dsm, f.ac_smem, used, tid, int(blockDim.x)); }
  __syncthreads();
  if (kSmem) cv.AssumeShared();
  const int g = (cta * int(blockDim.x >> 5) + warp) * lanes + lane;
  if (lane >= lanes || g >= int(f.num_groups) || !GroupInBand(f, g)) return;
  const int xb = int(f.xb), cx0 = (g % int(f.xgroups)) * 32, cy0 = (g / int(f.xgroups)) * 32, w = min(32, xb - cx0), h = min(32, int(f.yb) - cy0);
  const uint64_t* sec = SecBitPos(f); const uint32_t nsec = f.num_passes * f.num_groups + f.num_lf_groups + 2; const bool single = (f.num_groups == 1 && f.num_passes == 1);
  const uint32_t sidx = 2 + f.num_lf_groups + uint32_t(pass) * f.num_groups + g;
  const uint64_t start = single ? f.end_bitpos[2] : sec[sidx], end = single ? sec[nsec] : sec[nsec + sidx];
  SymReader rd; rd.br.Init(f.comp, start); rd.err = 0; if (f.lz_window) rd.win = f.lz_window + size_t(g) * kLzWindow;
  uint32_t err = 0, bad_range = 0;
  const uint32_t preset = rd.br.Read(CeilLog2Dev(f.num_hf_presets));
  if (preset >= f.num_hf_presets) { SetError(f.err, kErrPreset); return; }
  rd.Init(cv);
  const uint32_t nbctx = f.nb_block_ctx, ctx_offset = 495 * nbctx * preset, shift = f.pass_shift[pass], n_qf_thr = f.n_qf_thr, num_lf_ctxs = f.num_lf_ctxs;
  const uint8_t* bmap = f.blob + f.bctx_map_off; int16_t* coef = f.coeffs + size_t(g) * 3 * 65536; uint8_t* nzs = f.nz_scratch + size_t(g) * 3072;
  int bx = -1, by = 0, ci = 2, cell = 0, ord = 0, bw = 1, bh = 1, c = 0;
  uint32_t nz_left = 0, covered = 1, log2c = 0, size = 64, lbw = 0, bwm = 0, qf_idx = 0, lfi = 0, bctx = 0;
  uint32_t k = 0, nzctx = 0, histo = 0, prev = 0; const uint32_t* order = nullptr; int16_t* cc = nullptr; uint8_t* nzrow = nzs;
  for (;;) {
    uint32_t ctx; const bool blk = nz_left == 0;
    if (blk) {   // next (varblock, channel): number-of-nonzeros symbol
      if (++ci == 3) {
        ci = 0; bool found = false; uint32_t a = 0; size_t o = 0;
        for (;;) { if (++bx >= w) { bx = 0; if (++by >= h) break; } o = size_t(cy0 + by) * xb + cx0 + bx; a = f.acs[o]; if (a & 0x80) { found = true; break; } }
        if (!found) break;
        const int s = min(int(a & 31), 26); lbw = CoveredXLog2Dev(s); const uint32_t lbh = CoveredYLog2Dev(s); bw = 1 << lbw; bh = 1 << lbh; log2c = lbw + lbh; covered = 1u << log2c; size = covered * 64; ord = int(StrategyOrderDev(s));
        const uint32_t qf = uint32_t(f.hf_mul_m1[o]) + 1; qf_idx = 0; for (uint32_t t = 0; t < n_qf_thr; t++) qf_idx += qf > f.qf_thr[t];
        lfi = f.lf_idx[o]; bwm = uint32_t(bw) - 1; cell = by * 32 + bx;
      }
      c = ci == 0 ? 1 : ci == 1 ? 0 : 2; nzrow = nzs + c * 1024;
      uint32_t pred; if (bx == 0) pred = by == 0 ? 32 : nzrow[cell - 32]; else if (by == 0) pred = nzrow[cell - 1]; else pred = (uint32_t(nzrow[cell - 32]) + nzrow[cell - 1] + 1) >> 1;
      uint32_t idx = c < 2 ? uint32_t(c ^ 1) : 2u; idx = idx * 13 + ord; idx = idx * (n_qf_thr + 1) + qf_idx; idx = idx * num_lf_ctxs + lfi; bctx = bmap[idx];
      uint32_t nzb = pred > 64 ? 64 : pred; nzb = nzb < 8 ? nzb : (nzb >= 64 ? 36 : 4 + nzb / 2);
      ctx = ctx_offset + nzb * nbctx + bctx;
    } else {
      ctx = nzctx + uint32_t(s_freq[k >> log2c]) * 2 + prev;
    }
    const uint32_t u = kSmem ? rd.ReadAns(cv, ctx) : (cv.lz77 ? rd.ReadLz(cv, ctx, 0) : rd.Read(cv, ctx));
    if (blk) {
      if (u + covered > size) { err = kErrTooManyNz; break; }
      const uint32_t v = (u + covered - 1) >> log2c;
      if (covered == 1) nzrow[cell] = uint8_t(v); else for (int iy = 0; iy < bh; iy++) for (int ix = 0; ix < bw; ix++) nzrow[cell + iy * 32 + ix] = uint8_t(v);
      if (u) {
        order = reinterpret_cast<const uint32_t*>(BlobAt(f, f.order_off[pass][ord * 3 + c])); histo = ctx_offset + nbctx * 37 + 458 * bctx; prev = u > size / 16 ? 0 : 1;
        cc = coef + c * 65536 + cell * 64; nzctx = uint32_t(s_numnz[v]) * 2 + histo; k = covered; nz_left = u;
      }
    } else {
      prev = u != 0;
      if (u) {
        int32_t v = int32_t(uint32_t(UnpackSignedDev(u)) << shift); const uint32_t p = order[k], j = p >> 6; const uint32_t addr = (((j >> lbw) << 5) + (j & bwm)) * 64 + (p & 63);
        if (pass) v += cc[addr]; bad_range |= uint32_t(v + 32768) >> 16; cc[addr] = int16_t(v); nz_left--; nzctx = uint32_t(s_numnz[(nz_left + covered - 1) >> log2c]) * 2 + histo;
      }
      k++;
      if (k >= size && nz_left) { err = kErrNzMismatch; break; }
    }
  }
  if (!err && !rd.FinalOk(cv)) err = kErrAnsFinal;
  if (!err && bad_range) err = kErrCoefRange;
  if (!err) err = rd.err;
  const uint64_t pos = rd.br.BitPos(); if (!err && pos > end) err = kErrOverrun;
  f.ac_endpos[size_t(pass) * f.num_groups + g] = pos;
  SetError(f.err, err);
}

template <bool kSmem>
__global__ void __launch_bounds__(32 * kAcMaxWarps, 2) k_ac_vardct(const __grid_constant__ DFrame f, int pass, int lanes) {
  if (blockIdx.x < f.ac_cta_offset) return;   // spreads concurrent images over different SMs (see k_lf_group)
  AcVardctBody<kSmem>(f, pass, lanes, int(blockIdx.x - f.ac_cta_offset));
}
template <bool kSmem>
__global__ void __launch_bounds__(32 * kAcMaxWarps, 2) k_ac_vardct_multi(const __grid_constant__ DFrameSet s, int lanes) {   // pass 0 of single-pass frames
  if (blockIdx.x < s.cta_offset) return;
  const uint32_t cta = blockIdx.x - s.cta_offset; uint32_t img = 0; while (img + 1 < s.n && cta >= s.first[img + 1]) img++;
  AcVardctBody<kSmem>(s.f[img], 0, lanes, int(cta - s.first[img]));
}

// Group-local Modular channels (alpha / extra channels of VarDCT frames, everything of Modular frames): warp w of a CTA owns
// group blockIdx.x*kModGroupsPerCta + w, lane 0 walks the bit stream, and the warps share one staged copy of the tables.
// In VarDCT frames the stream continues where the group's AC coefficients ended (ac_endpos, written by k_ac_vardct).
static const int kModGroupsPerCta = 4;
template <bool kNarrow>
__global__ void __launch_bounds__(32 * kModGroupsPerCta) k_mod_group(const __grid_constant__ DFrame f, int pass) {
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31; const int g = blockIdx.x * kModGroupsPerCta + warp; const bool active = g < int(f.num_groups);
  __shared__ ChanLut sh_lut[kModGroupsPerCta]; __shared__ LeanSpecPrep sh_prep[kModGroupsPerCta]; __shared__ uint32_t sh_flag[kModGroupsPerCta]; extern __shared__ __align__(16) uint8_t dsm[];
  ModDecoder md; BindModDecoder(md, f, &sh_lut[warp]); uint32_t used = 0;
  StageModDecoder(md, f, dsm, f.lf_smem, used, tid, 32 * kModGroupsPerCta);
  __syncthreads();
  if (!active || !GroupInBand(f, g)) return;   // whole warps leave; inside a warp every lane stays (the speculative loop is warp-collective)
  // each warp's share of the dynamic shared memory left after the staged tables: room for its transposed alias table
  const uint32_t spec_off = (used + 15u) & ~15u, spec_all = f.lf_smem > spec_off ? f.lf_smem - spec_off : 0u, spec_bytes = (spec_all / kModGroupsPerCta) & ~15u;
  uint2* T = reinterpret_cast<uint2*>(dsm + spec_off + size_t(warp) * spec_bytes);
  const uint64_t* sec = SecBitPos(f); const uint32_t nsec = f.num_passes * f.num_groups + f.num_lf_groups + 2; const bool single = (f.num_groups == 1 && f.num_passes == 1);
  const uint32_t sidx = 2 + f.num_lf_groups + uint32_t(pass) * f.num_groups + g;
  uint64_t start = single ? f.end_bitpos[2] : sec[sidx], end = single ? sec[nsec] : sec[nsec + sidx];
  if (f.encoding == 0) start = f.ac_endpos[size_t(pass) * f.num_groups + g];
  md.rd.br.Init(f.comp, start); if (f.lz_window) md.rd.win = f.lz_window + size_t(g) * kLzWindow;
  md.rd.err = 0;
  { const int gd = int(f.group_dim), sid = 1 + 3 * int(f.num_lf_groups) + 17 + pass * int(f.num_groups) + g;
    DecodeModularGroupDev<kNarrow>(md, f, g, (g % int(f.xgroups)) * gd, (g / int(f.xgroups)) * gd, gd, f.pass_min_shift[pass], f.pass_max_shift[pass], sid,
                                   f.encoding == 1 && pass == 0 ? LocalTreeOf(f, uint32_t(g)) : nullptr, f.wp_scratch + (size_t(f.num_lf_groups) + g) * WPScratchInts(kMaxWpWidth), lane, sh_prep[warp], &sh_flag[warp], T, spec_bytes); }
  if (lane != 0) return;
  uint32_t err = md.rd.err; uint64_t pos = md.rd.br.BitPos(); if (!err && pos > end) err = kErrOverrun;
  SetError(f.err, err);
}

// Modular frames: the LF-group sections hold the channels of shift >= 3 (squeezed / subsampled 8x or more), one 8x8-group square per section.
template <bool kNarrow>
__global__ void __launch_bounds__(32 * kModGroupsPerCta) k_mod_lf_group(const __grid_constant__ DFrame f) {
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31; const int g = blockIdx.x * kModGroupsPerCta + warp; const bool active = g < int(f.num_lf_groups);
  __shared__ ChanLut sh_lut[kModGroupsPerCta]; __shared__ LeanSpecPrep sh_prep[kModGroupsPerCta]; __shared__ uint32_t sh_flag[kModGroupsPerCta]; extern __shared__ __align__(16) uint8_t dsm[];
  ModDecoder md; BindModDecoder(md, f, &sh_lut[warp]); uint32_t used = 0;
  StageModDecoder(md, f, dsm, f.lf_smem, used, tid, 32 * kModGroupsPerCta);
  __syncthreads();
  if (!active) return;
  const uint32_t spec_off = (used + 15u) & ~15u, spec_all = f.lf_smem > spec_off ? f.lf_smem - spec_off : 0u, spec_bytes = (spec_all / kModGroupsPerCta) & ~15u;
  uint2* T = reinterpret_cast<uint2*>(dsm + spec_off + size_t(warp) * spec_bytes);
  const uint64_t* sec = SecBitPos(f); const uint32_t nsec = f.num_passes * f.num_groups + f.num_lf_groups + 2; const bool single = (f.num_groups == 1 && f.num_passes == 1);
  if (single) return;   // a one-group frame keeps every channel in its global stream
  const uint64_t start = sec[1 + g], end = sec[nsec + 1 + g];
  md.rd.br.Init(f.comp, start); if (f.lz_window) md.rd.win = f.lz_window + size_t(g) * kLzWindow;
  md.rd.err = 0; const int dim = int(f.group_dim) * 8;
  DecodeModularGroupDev<kNarrow>(md, f, g, (g % int(f.xlfgroups)) * dim, (g / int(f.xlfgroups)) * dim, dim, 3, 1000, 1 + int(f.num_lf_groups) + g, LocalTreeOf(f, f.num_groups + 1 + uint32_t(g)),
                                 f.wp_scratch + size_t(g) * WPScratchInts(kMaxWpWidth), lane, sh_prep[warp], &sh_flag[warp], T, spec_bytes);
  if (lane != 0) return;
  uint32_t err = md.rd.err; const uint64_t pos = md.rd.br.BitPos(); if (!err && pos > end) err = kErrOverrun;
  SetError(f.err, err);
}

// Global Modular stream (channels small enough to live in the LfGlobal section), decoded by one thread.
__global__ void k_modular_global(const __grid_constant__ DFrame f, uint64_t start_bitpos, uint32_t num_channels) {
  __shared__ ChanLut sh_lut; extern __shared__ __align__(16) uint8_t dsm[];
  ModDecoder md; BindModDecoder(md, f, &sh_lut); { uint32_t used = 0; StageModDecoder(md, f, dsm, f.lf_smem, used, threadIdx.x, 32); }
  __syncthreads();
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  md.rd.br.Init(f.comp, start_bitpos);
  // header already parsed on the host (it carries the global transforms, the weighted-predictor parameters and, if local, the tree and code); the ANS state word follows
  md.wp = f.global_wp;
  { const DLocalTree* lt = LocalTreeOf(f, f.num_groups); if (lt && lt->present) BindLocalTree(md, f, *lt); }   // data_bitpos == start_bitpos: the host stopped right after the code
  if (f.lz_window) md.rd.win = f.lz_window + size_t(max(f.num_lf_groups, f.num_groups)) * kLzWindow;
  { uint32_t dm = 0; for (uint32_t c = 0; c < num_channels; c++) dm = max(dm, ModCh(f, c).w); md.dist_mult = dm; }
  md.rd.Init(md.cv);
  int32_t* wp = f.wp_scratch + (size_t(f.num_lf_groups) + f.num_groups) * WPScratchInts(kMaxWpWidth);
  md.ResetChannels();
  for (uint32_t c = 0; c < num_channels; c++) { const DModChannel& ch = ModCh(f, c); md.NoteChannel(f.mod_planes + ch.plane_off, ch.w, int(ch.w), int(ch.h), int(ch.hshift), int(ch.vshift)); md.DecodeChannel(int(c), 0, f.mod_planes + ch.plane_off, ch.w, int(ch.w), int(ch.h), wp); }
  if (!md.rd.FinalOk(md.cv)) md.rd.err = md.rd.err ? md.rd.err : kErrAnsFinal;
  f.end_bitpos[0] = md.rd.br.BitPos();
  SetError(f.err, md.rd.err);
}

void LaunchLfGroups(const DFrame* d, const DFrame& h, cudaStream_t st) { if (!h.num_lf_groups) return; const bool narrow = LfNarrow(h);
  if (narrow) Launch<k_lf_group<true>>(h.num_lf_groups + h.lf_cta_offset, 32, h.lf_smem, st, h); else Launch<k_lf_group<false>>(h.num_lf_groups + h.lf_cta_offset, 32, h.lf_smem, st, h); }
// Bundle launches (JxlB200DecodeBatch): the images of `set` share one stream; all must be VarDCT, multi-section, of the same kind
// (narrow Modular path for LF; single pass + shared-memory ANS tables for AC) — the caller checks with BundleCompatible*.
bool LfNarrow(const DFrame& h) { return !h.uses_wp; }   // the image's bit depth (mod_wide) does not matter for LF groups: see LfGroupBody
void LaunchLfGroupsMulti(const DFrameSet& set, bool narrow, cudaStream_t st) {
  uint32_t smem = 0; for (uint32_t i = 0; i < set.n; i++) smem = std::max(smem, set.f[i].lf_smem); const unsigned grid = set.first[set.n] + set.cta_offset;
  if (narrow) Launch<k_lf_group_multi<true>>(grid, 32, smem, st, set); else Launch<k_lf_group_multi<false>>(grid, 32, smem, st, set);
}
void LaunchAcGroupsMulti(const DFrameSet& set, int lanes, cudaStream_t st) {   // every frame: encoding 0, num_passes 1, ac_fast
  uint32_t smem = 0; for (uint32_t i = 0; i < set.n; i++) smem = std::max(smem, set.f[i].ac_smem);
  // Occupancy cap: a padded shared-memory request bounds the AC CTAs resident per SM, which leaves registers and shared memory for the
  // tile kernels (reconstruction, render) of images that are further along (they otherwise queue behind ~70 ms entropy CTAs).
  if (lanes >= 8) smem = std::max(smem, kAcBatchSmem);
  Launch<k_ac_vardct_multi<true>>(set.first[set.n] + set.cta_offset, 32 * AcWarpsFor(lanes), smem, st, set, lanes);
}
void LaunchLfDequant(const DFrame* d, const DFrame& h, bool smooth, cudaStream_t st) {
  size_t plane = size_t(h.xb) * h.yb; unsigned blocks = unsigned((plane + 255) / 256); Launch<k_lf_dequant>(blocks, 256, 0, st, d); if (smooth) Launch<k_lf_smooth>(blocks, 256, 0, st, d);
}
// `lanes`: sections per warp for the AC walk (power of two, 1..32).
int AcCtas(const DFrame& h, int lanes) { const unsigned per_cta = unsigned(AcWarpsFor(lanes) * lanes); return int((h.num_groups + per_cta - 1) / per_cta); }
void LaunchAcGroups(const DFrame* d, const DFrame& h, int pass, int lanes, cudaStream_t st) {
  if (h.encoding == 0) {
    const unsigned nw = unsigned(AcWarpsFor(lanes)), per_cta = nw * unsigned(lanes), ctas = (h.num_groups + per_cta - 1) / per_cta;
    if (h.ac_fast) Launch<k_ac_vardct<true>>(ctas + h.ac_cta_offset, 32 * nw, h.ac_smem, st, h, pass, lanes); else Launch<k_ac_vardct<false>>(ctas + h.ac_cta_offset, 32 * nw, 0, st, h, pass, lanes);
  }
  if (h.num_mod_channels > h.first_group_channel) { const unsigned ctas = (h.num_groups + kModGroupsPerCta - 1) / kModGroupsPerCta;
    if (!h.uses_wp && !h.mod_wide) Launch<k_mod_group<true>>(ctas, 32 * kModGroupsPerCta, h.lf_smem, st, h, pass); else Launch<k_mod_group<false>>(ctas, 32 * kModGroupsPerCta, h.lf_smem, st, h, pass); }
}
void LaunchModLfGroups(const DFrame& h, cudaStream_t st) {
  if (!h.num_lf_groups) return; const unsigned ctas = (h.num_lf_groups + kModGroupsPerCta - 1) / kModGroupsPerCta;
  if (!h.uses_wp && !h.mod_wide) Launch<k_mod_lf_group<true>>(ctas, 32 * kModGroupsPerCta, h.lf_smem, st, h); else Launch<k_mod_lf_group<false>>(ctas, 32 * kModGroupsPerCta, h.lf_smem, st, h);
}
void LaunchModularGlobal(const DFrame* d, const DFrame& h, uint64_t start_bitpos, uint32_t num_channels, cudaStream_t st) { Launch<k_modular_global>(1, 32, h.lf_smem, st, h, start_bitpos, num_channels); }

}  // namespace jxlgpu
