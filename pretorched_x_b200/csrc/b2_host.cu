// b2_host.cu -- library-wide host helpers declared in b2_host.h: error / launch bookkeeping, device queries, CUtensorMap
// construction and the programmatic-dependent-launch switch.
#include <mutex>
#include <stdlib.h>

#include "b2_host.h"

namespace b2 {

// ------------------------------------------------------------------------------------------
// error + launch bookkeeping
// ------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";
static std::atomic<uint64_t> g_launches{0};

int set_error(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
void count_launch(int n) { g_launches.fetch_add(static_cast<uint64_t>(n), std::memory_order_relaxed); }

int require_sm100() {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return set_error(B2_ERR_CUDA, "no CUDA device: %s", cudaGetErrorString(e));
  int major = 0;
  e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  if (e != cudaSuccess) return set_error(B2_ERR_CUDA, "cudaDeviceGetAttribute: %s", cudaGetErrorString(e));
  if (major != 10)
    return set_error(B2_ERR_UNSUPPORTED, "this library targets sm_100a (B200); device is sm_%d0 and there is no fallback",
                     major);
  return B2_OK;
}

int current_device() {
  int dev = 0;
  cudaGetDevice(&dev);
  return dev;
}

int sm_count() {               // per device ordinal (a process may drive several GPUs)
  static std::atomic<int> cache[64];
  const int dev = current_device() & 63;
  int n = cache[dev].load(std::memory_order_relaxed);
  if (n == 0) {
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cache[dev].store(n, std::memory_order_relaxed);
  }
  return n;
}

bool pdl_enabled() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("B2_PDL"); v = (e && e[0] == '0') ? 0 : 1; }
  return v != 0;
}

// ------------------------------------------------------------------------------------------
// tensor maps
// ------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode_tiled() {
  static PFN_encodeTiled fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_encodeTiled>(p);
  });
  return fn;
}

int tmap_2d_f16(TmapSpec* out, const void* base, uint64_t inner, uint64_t outer, uint64_t pitch_elems, uint32_t box_inner,
                uint32_t box_outer, bool swizzle128) {
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0) return set_error(B2_ERR_INVALID, "tensor base not 16-byte aligned");
  if ((pitch_elems * 2) % 16 != 0) return set_error(B2_ERR_INVALID, "row pitch %llu elements is not a multiple of 8",
                                                    (unsigned long long)pitch_elems);
  *out = TmapSpec{base, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, {inner, outer}, {pitch_elems * 2}, {box_inner, box_outer}, {1, 1},
                  swizzle128};
  return B2_OK;
}

int tmap_ndhwc_slab(TmapSpec* out, const void* base, uint64_t C, uint64_t W, uint64_t H, uint64_t planes, uint32_t box_w,
                    uint32_t box_h, uint32_t stride_hw, uint32_t box_planes) {
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0) return set_error(B2_ERR_INVALID, "tensor base not 16-byte aligned");
  // with element strides the box is given in traversed (full-resolution) elements; smem receives every
  // stride_hw-th pixel / row, i.e. box_w x box_h dense pixels
  *out = TmapSpec{base, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, {C, W, H, planes}, {C * 2, W * C * 2, H * W * C * 2},
                  {64, stride_hw * (box_w - 1) + 1, stride_hw * (box_h - 1) + 1, box_planes}, {1, stride_hw, stride_hw, 1}, true};
  if (out->box[1] > 256 || out->box[2] > 256)
    return set_error(B2_ERR_UNSUPPORTED, "slab box %ux%u exceeds the TMA box limit", out->box[1], out->box[2]);
  return B2_OK;
}

int encode_tmap(CUtensorMap* out, const TmapSpec& s) {
  PFN_encodeTiled enc = get_encode_tiled();
  if (!enc) return set_error(B2_ERR_CUDA, "cuTensorMapEncodeTiled entry point unavailable (no driver?)");
  CUresult r = enc(out, s.dtype, (cuuint32_t)s.rank, const_cast<void*>(s.base), s.dims, s.strides, s.box, s.estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, s.swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return set_error(B2_ERR_CUDA, "cuTensorMapEncodeTiled(%dd) failed (%d) dims=%llux%llu.. box=%ux%u..", s.rank, (int)r,
                     (unsigned long long)s.dims[0], (unsigned long long)s.dims[1], s.box[0], s.box[1]);
  return B2_OK;
}

int make_tmap_2d_f16(CUtensorMap* out, const void* base, uint64_t inner, uint64_t outer, uint64_t pitch_elems,
                     uint32_t box_inner, uint32_t box_outer, bool swizzle128) {
  TmapSpec s;
  const int rc = tmap_2d_f16(&s, base, inner, outer, pitch_elems, box_inner, box_outer, swizzle128);
  return rc != B2_OK ? rc : encode_tmap(out, s);
}

}  // namespace b2

extern "C" {
const char* b2_last_error(void) { return b2::g_err; }
uint64_t b2_launch_count(void) { return b2::g_launches.load(std::memory_order_relaxed); }
}
