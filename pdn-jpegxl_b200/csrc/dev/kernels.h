// pdn-jpegxl_b200 engine — host-callable launch wrappers for the sm_100a kernels.
#pragma once
#include "frame.cuh"
#include "../host/bits.h"
#include <atomic>
#include <mutex>

// A runtime call that fails throws Error("CUDA: <the runtime's text> at <the call>").
#define CUDA_OK(expr) do { cudaError_t e_ = (expr); if (e_ != cudaSuccess) throw ::jxlgpu::Error(std::string("CUDA: ") + cudaGetErrorString(e_) + " at " #expr); } while (0)

namespace jxlgpu {
// decode
void LaunchLfGroups(const DFrame* d, const DFrame& h, cudaStream_t st);
void LaunchLfDequant(const DFrame* d, const DFrame& h, bool smooth, cudaStream_t st);
int AcCtas(const DFrame& h, int lanes);
bool LfNarrow(const DFrame& h);
void LaunchLfGroupsMulti(const DFrameSet& set, bool narrow, cudaStream_t st);
void LaunchAcGroupsMulti(const DFrameSet& set, int lanes, cudaStream_t st);
void LaunchAcGroups(const DFrame* d, const DFrame& h, int pass, int lanes, cudaStream_t st);
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

inline std::atomic<int> g_launch_count{0};
inline int LaunchCount() { return g_launch_count.load(); }                      // kernels launched by this process so far (bench gpu_launches)

// Throws for a launch, or the shared-memory opt-in of one, that the runtime refused.
[[noreturn]] inline void ThrowLaunchError(cudaError_t e, const void* kernel) {
  const char* name = nullptr; if (cudaFuncGetName(&name, kernel) != cudaSuccess) name = nullptr;
  throw Error(std::string("CUDA: ") + cudaGetErrorString(e) + " launching " + (name ? name : "a kernel"));
}
// Opts Kernel in to `smem` bytes of dynamic shared memory on the current device: once per (kernel, device), and again only when a launch asks for
// more (the lock is taken only then). Any size is opted in, not only those over 48 KB: the default 48 KB also holds the kernel's static shared memory.
template <auto Kernel> void AllowDynamicSmem(size_t smem) {
  static std::atomic<size_t> allowed[64]; static std::mutex mu;
  int dev = 0; CUDA_OK(cudaGetDevice(&dev)); JXLG_CHECK(dev < 64, "CUDA: device index over 63");
  if (smem <= allowed[dev].load()) return;
  std::lock_guard<std::mutex> lk(mu); if (smem <= allowed[dev].load()) return;
  const cudaError_t e = cudaFuncSetAttribute(reinterpret_cast<const void*>(Kernel), cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
  if (e != cudaSuccess) ThrowLaunchError(e, reinterpret_cast<const void*>(Kernel));
  allowed[dev].store(smem);
}
// Every kernel of the engine is launched here. A launch the runtime refuses (a grid dimension over its limit, too much shared memory) throws
// instead of leaving the output buffers as they were. cudaGetLastError reads the calling thread's state, which Guard (abi.cu) clears around
// every engine call, so a refusal is reported to the call that made it. Counted for LaunchCount.
template <auto Kernel, class... Args> void Launch(dim3 grid, dim3 block, size_t smem, cudaStream_t st, const Args&... args) {
  if (smem) AllowDynamicSmem<Kernel>(smem);
  Kernel<<<grid, block, smem, st>>>(args...);
  if (const cudaError_t e = cudaGetLastError(); e != cudaSuccess) ThrowLaunchError(e, reinterpret_cast<const void*>(Kernel));
  g_launch_count.fetch_add(1);
}
}  // namespace jxlgpu
