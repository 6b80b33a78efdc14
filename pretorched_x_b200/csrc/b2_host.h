// b2_host.h -- host-side helpers shared by the C-ABI translation units (defined in b2_host.cu): error reporting, launch
// accounting and CUtensorMap construction through the driver entry point (no -lcuda link needed).
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>

#include <atomic>

#include "../../include/b2_pretorched.h"

namespace b2 {

int set_error(int code, const char* fmt, ...);
void count_launch(int n = 1);

#define B2_CHECK_ARG(cond, ...)                                   \
  do {                                                            \
    if (!(cond)) return ::b2::set_error(B2_ERR_INVALID, __VA_ARGS__); \
  } while (0)

#define B2_TRY(expr)                              \
  do {                                            \
    const int rc__ = (expr);                      \
    if (rc__ != B2_OK) return rc__;               \
  } while (0)

#define B2_CHECK_CUDA(expr)                                                                         \
  do {                                                                                              \
    cudaError_t e__ = (expr);                                                                       \
    if (e__ != cudaSuccess)                                                                         \
      return ::b2::set_error(B2_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), \
                             __FILE__, __LINE__);                                                   \
  } while (0)

// after a kernel launch: picks up launch-configuration errors without synchronising
#define B2_CHECK_LAUNCH(name)                                                                        \
  do {                                                                                               \
    cudaError_t e__ = cudaGetLastError();                                                            \
    if (e__ != cudaSuccess)                                                                          \
      return ::b2::set_error(B2_ERR_CUDA, "launch of %s failed: %s", name, cudaGetErrorString(e__)); \
    ::b2::count_launch();                                                                            \
  } while (0)

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) is a PER-DEVICE property of a kernel: a single process that drives several
// GPUs (nn.DataParallel -- the reference's only multi-GPU construct -- or model.to('cuda:1')) must opt in on each of them.
// One bit per device ordinal, set after the first successful call on that device.
int current_device();
int sm_count();          // SM count of the current device (cached per ordinal); 148, the B200's, when there is no device
#define B2_OPT_IN_SMEM(kernel, bytes)                                                                          \
  do {                                                                                                         \
    static std::atomic<unsigned long long> done__{0};                                                          \
    const unsigned long long bit__ = 1ull << (::b2::current_device() & 63);                                    \
    if (!(done__.load(std::memory_order_relaxed) & bit__)) {                                                   \
      B2_CHECK_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(bytes)));  \
      done__.fetch_or(bit__, std::memory_order_relaxed);                                                       \
    }                                                                                                          \
  } while (0)

// A CUtensorMap as plain values: what cuTensorMapEncodeTiled takes (strides in bytes, for dims 1 .. rank-1).  The builders
// below check what can be checked on the host (alignment, pitch, box limits) and fill one; encode_tmap makes the map.
struct TmapSpec {
  const void* base;
  CUtensorMapDataType dtype;
  int rank;
  cuuint64_t dims[4];
  cuuint64_t strides[3];
  cuuint32_t box[4];
  cuuint32_t estr[4];
  bool swizzle128;
};
int encode_tmap(CUtensorMap* out, const TmapSpec& spec);

// 2-D fp16 tensor map: `inner` contiguous elements per row, `outer` rows of pitch `pitch_elems`;
// box = [box_inner x box_outer]; swizzle128 selects CU_TENSOR_MAP_SWIZZLE_128B (box_inner must be 64).
// Out-of-bounds elements read as zero and are dropped on store.
int tmap_2d_f16(TmapSpec* out, const void* base, uint64_t inner, uint64_t outer, uint64_t pitch_elems, uint32_t box_inner,
                uint32_t box_outer, bool swizzle128);
int make_tmap_2d_f16(CUtensorMap* out, const void* base, uint64_t inner, uint64_t outer, uint64_t pitch_elems,
                     uint32_t box_inner, uint32_t box_outer, bool swizzle128);

// 4-D fp16 tensor map over an NDHWC activation viewed as (C, W, H, N*T); smem box = (64, box_w, box_h, box_planes) pixels
// taken every stride_hw-th column / row (TMA elementStrides), SWIZZLE_128B.  Negative / out-of-range box coordinates read zeros (halo columns, rows above/below the image).
int tmap_ndhwc_slab(TmapSpec* out, const void* base, uint64_t C, uint64_t W, uint64_t H, uint64_t planes, uint32_t box_w,
                    uint32_t box_h, uint32_t stride_hw, uint32_t box_planes = 1);

int require_sm100();

// Launch with programmatic stream serialization (see pdl_wait() in b2_ptx.cuh).  B2_PDL=0 in the environment turns
// the attribute off (A/B measurements).
bool pdl_enabled();
template <typename... KArgs, typename... Args>
cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = pdl_enabled() ? 1 : 0;
  cfg.attrs = attr; cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}   // B2_OK when the current device is compute capability 10.x

}  // namespace b2
