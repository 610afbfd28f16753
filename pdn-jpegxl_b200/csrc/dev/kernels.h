// pdn-jpegxl_b200 engine — host-callable launch wrappers for the sm_100a kernels.
#pragma once
#include "frame.cuh"

namespace jxlgpu {
// decode
void LaunchLfGroups(const DFrame* d, const DFrame& h, cudaStream_t st);
void LaunchLfDequant(const DFrame* d, const DFrame& h, bool smooth, cudaStream_t st);
int AcCtas(const DFrame& h, int lanes);
bool LfNarrow(const DFrame& h);
void LaunchLfGroupsMulti(const DFrameSet& set, bool narrow, cudaStream_t st);
void LaunchAcGroupsMulti(const DFrameSet& set, int lanes, cudaStream_t st);
int LaunchAcGroups(const DFrame* d, const DFrame& h, int pass, int lanes, cudaStream_t st);
void LaunchModLfGroups(const DFrame& h, cudaStream_t st);   // Modular frames: channels of shift >= 3 in the LF-group sections
void LaunchModularGlobal(const DFrame* d, const DFrame& h, uint64_t start_bitpos, uint32_t num_channels, cudaStream_t st);
void LaunchReconstruct(const DFrame* d, const DFrame& h, cudaStream_t st);       // dequant + CfL + LLF + inverse transforms
bool LaunchFusedRender(const DFrame* d, const DFrame& h, cudaStream_t st);       // gaborish + EPF + colour fused (returns false when not applicable)
void LaunchInverseRct(const DFrame* d, const DFrame& h, const DModOp* ops, cudaStream_t st);   // ops: host copy of the op table (h.ops or the blob table)
void LaunchOutput(const DFrame* d, const DFrame& h, cudaStream_t st);            // colour transform + sample conversion + interleave (+BGRA)
void LaunchSplitLayers(const void* src, void* color, uint8_t* alpha, size_t npix, int format, int sample_type, bool has_alpha, cudaStream_t st);   // I/DecoderLayerData.cs repack
// layers of a multi-frame still (dev/composite_kernels.cu): float canvas [H][W][C], frame [fh][fw][C]
void LaunchBlendLayer(float* canvas, const float* frame, int W, int H, int fw, int fh, int x0, int y0, int C, int cc, uint32_t cmode, uint32_t amode, bool cclamp, bool aclamp, bool premultiplied, cudaStream_t st);
void LaunchFinalizeCanvas(const float* canvas, uint8_t* out, int W, int H, int C, int cc, bool premultiplied, uint32_t sample_type, uint32_t orientation, bool bgra, cudaStream_t st);
void FillDeviceTables(DTables* host_tables);
int LaunchCount();                                                                 // kernels launched by this process so far (bench gpu_launches)
void CountLaunch(int n = 1);
}  // namespace jxlgpu
