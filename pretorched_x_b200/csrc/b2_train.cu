// b2_train.cu -- the kernels of the frozen-BatchNorm block backward (fine-tuning of the residual stages): the implicit
// tcgen05 weight gradient (b2_conv_ndhwc_wgrad), the ReLU mask with its per-channel gradient sum, and the two scatters of
// the strided data gradient.  Like b2_aux.cu, the element-wise kernels move 8 fp16 channels (16 bytes) per access with the
// channel index fastest.
#include "b2_host.h"
#include "b2_ptx.cuh"

#include <cuda_fp16.h>

namespace b2 {

static inline int div_up_t(long long a, long long b) { return (int)((a + b - 1) / b); }

__device__ __forceinline__ void unpack8(const uint4 v, float f[8]) {
  const uint32_t u[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const float2 t = __half22float2(*reinterpret_cast<const __half2*>(&u[e]));
    f[2 * e] = t.x; f[2 * e + 1] = t.y;
  }
}

__device__ __forceinline__ uint4 pack8(const float f[8]) {
  uint32_t o[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    __half2 h = __floats2half2_rn(f[2 * e], f[2 * e + 1]);
    o[e] = *reinterpret_cast<uint32_t*>(&h);
  }
  return make_uint4(o[0], o[1], o[2], o[3]);
}

// ------------------------------------------------------------------------------------------
// ReLU backward + per-channel sums.  Block = C8 lanes x R row groups (R * C8 <= 256); block b owns rows
// [b * rows_per_block, ...) and walks them in a fixed order, the R partial sums meet in shared memory in a fixed order,
// and b2_relu_grad_sum_reduce adds the per-block rows in block order: the sums do not depend on scheduling.
// ------------------------------------------------------------------------------------------
constexpr int kMaskThreads = 256;

__global__ void __launch_bounds__(kMaskThreads)
relu_grad_kernel(const __half* __restrict__ y, int ldy8, const __half* __restrict__ g, int ldg8, __half* __restrict__ gz,
                 int C8, long long M, int rows_per_block, float* __restrict__ partial) {
  __shared__ float red[kMaskThreads][9];
  const int R = kMaskThreads / C8;
  const int lane = threadIdx.x % C8, grp = threadIdx.x / C8;
  float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  const long long r0 = (long long)blockIdx.x * rows_per_block;
  const long long r1 = min(M, r0 + rows_per_block);
  if (grp < R) {
    for (long long r = r0 + grp; r < r1; r += R) {
      float fy[8], fg[8];
      unpack8(__ldg(reinterpret_cast<const uint4*>(y) + r * ldy8 + lane), fy);
      unpack8(__ldg(reinterpret_cast<const uint4*>(g) + r * ldg8 + lane), fg);
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        fg[e] = fy[e] > 0.f ? fg[e] : 0.f;
        acc[e] += fg[e];
      }
      reinterpret_cast<uint4*>(gz)[r * ldy8 + lane] = pack8(fg);
    }
  }
#pragma unroll
  for (int e = 0; e < 8; ++e) red[threadIdx.x][e] = acc[e];
  __syncthreads();
  if (grp == 0) {
    for (int q = 1; q < R; ++q)
#pragma unroll
      for (int e = 0; e < 8; ++e) acc[e] += red[q * C8 + lane][e];
#pragma unroll
    for (int e = 0; e < 8; ++e) partial[(size_t)blockIdx.x * C8 * 8 + lane * 8 + e] = acc[e];
  }
}

__global__ void relu_grad_reduce_kernel(const float* __restrict__ partial, int blocks, int C, float* __restrict__ sum) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  float s = 0.f;
  for (int b = 0; b < blocks; ++b) s += partial[(size_t)b * C + c];
  sum[c] = s;
}

// ------------------------------------------------------------------------------------------
// Strided scatters of the data gradient
// ------------------------------------------------------------------------------------------
// y (input geometry T x H x W, pitch 8*ld8) = g at positions (s*to, s*ho, s*wo), zero elsewhere
__global__ void zero_dilate_kernel(const __half* __restrict__ g, __half* __restrict__ y, int T, int H, int W, int To, int Ho,
                                   int Wo, int ld8, int s, long long total) {
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int c8 = (int)(i % ld8);
  long long q = i / ld8;
  const int w = (int)(q % W); q /= W;
  const int h = (int)(q % H); q /= H;
  const int t = (int)(q % T);
  const long long n = q / T;
  uint4 v = make_uint4(0, 0, 0, 0);
  if (t % s == 0 && h % s == 0 && w % s == 0 && t / s < To && h / s < Ho && w / s < Wo)
    v = __ldg(reinterpret_cast<const uint4*>(g) + (((n * To + t / s) * Ho + h / s) * (long long)Wo + w / s) * ld8 + c8);
  reinterpret_cast<uint4*>(y)[i] = v;
}

// y[n, s*to, s*ho, s*wo, c] += g[n, to, ho, wo, c] for c < 8*C8 (each y element is touched by at most one thread)
__global__ void strided_add_kernel(const __half* __restrict__ g, int ldg8, __half* __restrict__ y, int ldy8, int T, int H,
                                   int W, int To, int Ho, int Wo, int C8, int s, long long total) {
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int c8 = (int)(i % C8);
  long long q = i / C8;
  const int wo = (int)(q % Wo); q /= Wo;
  const int ho = (int)(q % Ho); q /= Ho;
  const int to = (int)(q % To);
  const long long n = q / To;
  uint4* dst = reinterpret_cast<uint4*>(y) + (((n * T + (long long)to * s) * H + (long long)ho * s) * W + (long long)wo * s) * ldy8 + c8;
  float a[8], b[8];
  unpack8(*dst, a);
  unpack8(__ldg(reinterpret_cast<const uint4*>(g) + (((n * To + to) * Ho + ho) * (long long)Wo + wo) * ldg8 + c8), b);
#pragma unroll
  for (int e = 0; e < 8; ++e) a[e] += b[e];
  *dst = pack8(a);
}


// ------------------------------------------------------------------------------------------
// Implicit-GEMM weight gradient on tcgen05: dW[k][tap][c] = sum_p g[p][k] * x[p*s + tap - pad][c].
// A CTA owns one output tile (128 filters k x 128 channels c of one tap) and one split range of position rectangles.
// A rectangle is 8 x 8 output positions (h, w) of one (n, t) plane: the TMA box of g at those positions and the box of
// x at the shifted (and, with elementStrides, strided) positions hold the same 64 positions in the same row order, each
// as [64 positions][64 channels] with 128-byte swizzle -- MN-major for both operands (instruction-descriptor bits 15
// and 16), 64 positions deep.  Out-of-range h / w read zeros from TMA; a tap whose input frame t lies outside the clip
// contributes nothing and is skipped.  No transposed or im2col copy exists in HBM.  Split ranges write fp32 partials
// that b2_wgrad_reduce sums in split order, so results do not depend on scheduling.
// ------------------------------------------------------------------------------------------
constexpr int kWgStages = 4;
constexpr int kWgStageBytes = 4 * 8192;            // A: 2 x [64 pos][64 k], B: 2 x [64 pos][64 c]
constexpr int kWgThreads = 192;                    // warps 0-3 epilogue, 4 TMA, 5 MMA + TMEM
constexpr int kWgSmem = kWgStages * kWgStageBytes + 1024;

__host__ __device__ inline void wgrad_split_range(long long rects, int S, int s, long long* r0, long long* r1) {
  *r0 = rects * s / S;
  *r1 = rects * (s + 1) / S;
}

struct WgradParams {
  float* out;                 // [S][K][taps][C] fp32 (S == 1: the result)
  int K, C, taps, kt, kh, kw, st, pt, ph, pw;
  int T, To, Ho, Wo, mt, nt, S;
  int rw, rh;                 // rectangles per row / column of a plane
  long long rects;            // N * To * rh * rw
};

__global__ void __launch_bounds__(kWgThreads, 1)
wgrad_kernel(const __grid_constant__ CUtensorMap tmG, const __grid_constant__ CUtensorMap tmX, const WgradParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_align<1024>(smem_raw);
  __shared__ __align__(8) uint64_t full_bar[kWgStages], empty_bar[kWgStages], acc_bar;
  __shared__ uint32_t tmem_slot;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  int tile = blockIdx.x;
  const int ct = tile % p.nt; tile /= p.nt;
  const int tap = tile % p.taps;
  const int mtile = tile / p.taps;
  const int dw = tap % p.kw, dh = (tap / p.kw) % p.kh, dt = tap / (p.kw * p.kh);
  long long r0, r1;
  wgrad_split_range(p.rects, p.S, blockIdx.y, &r0, &r1);

  if (tid == 0) {
    for (int s = 0; s < kWgStages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    mbar_init(&acc_bar, 1);
    fence_mbar_init();
    tma_prefetch_desc(&tmG); tma_prefetch_desc(&tmX);
  }
  if (warp == 5) { tmem_alloc(&tmem_slot, 128); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_slot;

  // rectangle r -> (plane of g, first output row / column, input frame); the same decode in both producer and issuer
  auto decode = [&](long long r, int* gplane, int* xplane, int* ho0, int* wo0) -> bool {
    const int cw = (int)(r % p.rw); r /= p.rw;
    const int chh = (int)(r % p.rh); r /= p.rh;
    const int to = (int)(r % p.To);
    const int n = (int)(r / p.To);
    const int ti = to * p.st - p.pt + dt;
    *gplane = n * p.To + to; *xplane = n * p.T + ti; *ho0 = chh * 8; *wo0 = cw * 8;
    return ti >= 0 && ti < p.T;
  };

  if (warp == 4) {
    int it = 0;
    for (long long r = r0; r < r1; ++r) {
      int gp, xp, ho0, wo0;
      if (!decode(r, &gp, &xp, &ho0, &wo0)) continue;
      const int s = it % kWgStages;
      mbar_wait(&empty_bar[s], ((it / kWgStages) & 1) ^ 1);
      if (elect_one()) {
        uint8_t* dst = smem + s * kWgStageBytes;
        mbar_expect_tx(&full_bar[s], kWgStageBytes);
        const int hi = ho0 * p.st - p.ph + dh, wi = wo0 * p.st - p.pw + dw;
        tma_load_4d(dst, &tmG, &full_bar[s], mtile * 128, wo0, ho0, gp);
        tma_load_4d(dst + 8192, &tmG, &full_bar[s], mtile * 128 + 64, wo0, ho0, gp);
        tma_load_4d(dst + 16384, &tmX, &full_bar[s], ct * 128, wi, hi, xp);
        tma_load_4d(dst + 24576, &tmX, &full_bar[s], ct * 128 + 64, wi, hi, xp);
      }
      __syncwarp();
      ++it;
    }
  } else if (warp == 5) {
    // both operands MN-major, 128B swizzle: LBO = 8192 B between the two 64-wide k / c blocks, +2048 B per 16 positions
    constexpr uint32_t idesc = make_idesc_f16(128, 128, 0) | (1u << 15) | (1u << 16);
    const uint32_t ring = smem_u32(smem);
    int it = 0;
    for (long long r = r0; r < r1; ++r) {
      int gp, xp, ho0, wo0;
      if (!decode(r, &gp, &xp, &ho0, &wo0)) continue;
      const int s = it % kWgStages;
      mbar_wait(&full_bar[s], (it / kWgStages) & 1);
      tc_fence_after();
      const uint32_t base = ring + s * kWgStageBytes;
      const uint32_t a_lo = ((base & 0x3FFFFu) >> 4) | ((8192u >> 4) << 16);
      const uint32_t b_lo = (((base + 16384) & 0x3FFFFu) >> 4) | ((8192u >> 4) << 16);
      if (elect_one()) {
#pragma unroll
        for (int kk = 0; kk < 4; ++kk)
          umma_f16(tmem, desc_from(kSw128DescHi, a_lo + kk * 128), desc_from(kSw128DescHi, b_lo + kk * 128), idesc,
                   (it != 0 || kk != 0) ? 1u : 0u);
        umma_commit(&empty_bar[s]);
      }
      __syncwarp();
      ++it;
    }
    if (elect_one()) {
      if (it > 0) umma_commit(&acc_bar);
      else mbar_arrive(&acc_bar);          // nothing accumulated: the epilogue writes zeros
    }
    __syncwarp();
  } else {
    // epilogue: warp w holds filters mtile*128 + 32w + lane; 128 channels in four 32-column loads
    mbar_wait(&acc_bar, 0);
    tc_fence_after();
    bool any = false;
    for (long long r = r0; r < r1 && !any; ++r) { int a, b, c, d; any = decode(r, &a, &b, &c, &d); }
    const int k = mtile * 128 + warp * 32 + lane;
    float* row = p.out + (((size_t)blockIdx.y * p.K + k) * p.taps + tap) * p.C;
#pragma unroll 1
    for (int j = 0; j < 4; ++j) {
      uint32_t v[32];
      if (any) {
        tmem_ld32(tmem + ((uint32_t)(warp * 32) << 16) + j * 32, v);
        tmem_ld_wait();
      } else {
#pragma unroll
        for (int e = 0; e < 32; ++e) v[e] = 0u;
      }
      const int c0 = ct * 128 + j * 32;
      if (k < p.K && c0 < p.C) {
#pragma unroll
        for (int e = 0; e < 32; e += 4)
          *reinterpret_cast<float4*>(row + c0 + e) = make_float4(__uint_as_float(v[e]), __uint_as_float(v[e + 1]),
                                                                 __uint_as_float(v[e + 2]), __uint_as_float(v[e + 3]));
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 5) tmem_dealloc(tmem, 128);
}

// out[i] = sum_s part[s * n + i], splits in order
__global__ void wgrad_reduce_kernel(const float* __restrict__ part, int S, long long n, float* __restrict__ out) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= n) return;
  float acc = 0.f;
  for (int s = 0; s < S; ++s) acc += part[s * n + i];
  out[i] = acc;
}

struct WgradPlan {
  WgradParams p;
  dim3 grid;
  int block, smem;
  int ldg, ldx, N, H, W;
};

static int odim_t(int in, int k, int s, int pad) { return (in + 2 * pad - k) / s + 1; }

// Tile and split choice; calls no CUDA API except sm_count().  Output tiles alone fill the SMs for wide 3x3x3 layers;
// elsewhere (1x1x1 layers: 4 x 16 tiles for C2048 -> 512) the positions are split so that about two CTAs run per SM,
// keeping at least 4 rectangles per split.
static int plan_wgrad(const b2_wgrad_args* a, WgradPlan* pl) {
  B2_CHECK_ARG(a && a->x && a->g && a->dw, "null tensor pointer");
  B2_CHECK_ARG(a->N > 0 && a->T > 0 && a->H > 0 && a->W > 0 && a->K > 0 && a->C > 0, "non-positive dimension");
  B2_CHECK_ARG(a->C % 64 == 0 && a->ldx % 8 == 0 && a->ldx >= a->C && a->ldg % 8 == 0 && a->ldg >= a->K,
               "wgrad needs C a multiple of 64 and pitches that are multiples of 8 covering C / K");
  B2_CHECK_ARG(a->sh == a->sw && a->st > 0 && a->sh > 0, "wgrad needs equal H / W strides");
  B2_CHECK_ARG(a->kt > 0 && a->kh > 0 && a->kw > 0 && a->pt >= 0 && a->ph >= 0 && a->pw >= 0, "bad filter geometry");
  WgradParams& p = pl->p;
  p.out = a->dw; p.K = a->K; p.C = a->C;
  p.kt = a->kt; p.kh = a->kh; p.kw = a->kw; p.taps = a->kt * a->kh * a->kw;
  p.st = a->st; p.pt = a->pt; p.ph = a->ph; p.pw = a->pw;
  p.T = a->T;
  p.To = odim_t(a->T, a->kt, a->st, a->pt); p.Ho = odim_t(a->H, a->kh, a->sh, a->ph); p.Wo = odim_t(a->W, a->kw, a->sw, a->pw);
  B2_CHECK_ARG(p.To > 0 && p.Ho > 0 && p.Wo > 0, "empty output");
  p.mt = (a->K + 127) / 128; p.nt = (a->C + 127) / 128;
  p.rw = (p.Wo + 7) / 8; p.rh = (p.Ho + 7) / 8;
  p.rects = (long long)a->N * p.To * p.rh * p.rw;
  const long long tiles = (long long)p.mt * p.taps * p.nt;
  B2_CHECK_ARG(tiles < (1ll << 31), "too many output tiles");
  long long S = (2ll * sm_count() + tiles - 1) / tiles;
  S = S < p.rects / 4 ? S : p.rects / 4;
  S = S < 1 ? 1 : (S > 65535 ? 65535 : S);
  p.S = (int)S;
  pl->grid = dim3((unsigned)tiles, (unsigned)S, 1);
  pl->block = kWgThreads;
  pl->smem = kWgSmem;
  pl->ldg = a->ldg; pl->ldx = a->ldx; pl->N = a->N; pl->H = a->H; pl->W = a->W;
  return B2_OK;
}

}  // namespace b2

using namespace b2;

extern "C" {

int b2_relu_grad_sum_partials(long long M, int ld) {
  return div_up_t(M, ld >= 512 ? 256 : 512);
}

int b2_relu_grad_sum(const void* y, int ldy, const void* g, int ldg, void* gz, long long M, float* partial, float* sum,
                     void* stream) {
  B2_CHECK_ARG(y && g && gz && partial && sum && M > 0, "bad argument");
  B2_CHECK_ARG(ldy % 8 == 0 && ldg % 8 == 0 && ldg >= ldy && ldy <= 8 * kMaskThreads,
               "pitches must be multiples of 8 with ldg >= ldy and ldy <= %d", 8 * kMaskThreads);
  const int C8 = ldy / 8;
  const int blocks = b2_relu_grad_sum_partials(M, ldy);
  const int rows = (int)((M + blocks - 1) / blocks);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  relu_grad_kernel<<<blocks, kMaskThreads, 0, st>>>((const __half*)y, C8, (const __half*)g, ldg / 8, (__half*)gz, C8, M, rows,
                                                    partial);
  B2_CHECK_LAUNCH("relu_grad");
  relu_grad_reduce_kernel<<<div_up_t(ldy, 128), 128, 0, st>>>(partial, blocks, ldy, sum);
  B2_CHECK_LAUNCH("relu_grad_reduce");
  return B2_OK;
}

int b2_zero_dilate_scatter(const void* g, void* y, int N, int T, int H, int W, int ld, int stride, void* stream) {
  B2_CHECK_ARG(g && y && N > 0 && T > 0 && H > 0 && W > 0 && stride > 0 && ld % 8 == 0, "bad argument");
  const int To = (T - 1) / stride + 1, Ho = (H - 1) / stride + 1, Wo = (W - 1) / stride + 1;
  const long long total = (long long)N * T * H * W * (ld / 8);
  zero_dilate_kernel<<<div_up_t(total, 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      (const __half*)g, (__half*)y, T, H, W, To, Ho, Wo, ld / 8, stride, total);
  B2_CHECK_LAUNCH("zero_dilate_scatter");
  return B2_OK;
}

int b2_strided_scatter_add(const void* g, int ldg, void* y, int ldy, int N, int T, int H, int W, int C, int stride, void* stream) {
  B2_CHECK_ARG(g && y && N > 0 && T > 0 && H > 0 && W > 0 && stride > 0, "bad argument");
  B2_CHECK_ARG(C % 8 == 0 && ldg % 8 == 0 && ldy % 8 == 0 && C <= ldg && C <= ldy, "channel count / pitches must be multiples of 8");
  const int To = (T - 1) / stride + 1, Ho = (H - 1) / stride + 1, Wo = (W - 1) / stride + 1;
  const long long total = (long long)N * To * Ho * Wo * (C / 8);
  strided_add_kernel<<<div_up_t(total, 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      (const __half*)g, ldg / 8, (__half*)y, ldy / 8, T, H, W, To, Ho, Wo, C / 8, stride, total);
  B2_CHECK_LAUNCH("strided_scatter_add");
  return B2_OK;
}

size_t b2_wgrad_workspace_floats(const b2_wgrad_args* a) {
  WgradPlan pl;
  if (plan_wgrad(a, &pl) != B2_OK || pl.p.S == 1) return 0;
  return (size_t)pl.p.S * a->K * pl.p.taps * a->C;
}

int b2_conv_ndhwc_wgrad(const b2_wgrad_args* a, void* stream) {
  WgradPlan pl;
  B2_TRY(plan_wgrad(a, &pl));
  B2_TRY(require_sm100());
  const long long n = (long long)a->K * pl.p.taps * a->C;
  if (pl.p.S > 1) {
    B2_CHECK_ARG(a->work != nullptr, "split weight gradient needs b2_wgrad_workspace_floats() floats of workspace");
    pl.p.out = a->work;
  }
  CUtensorMap tmG, tmX;
  TmapSpec sg, sx;
  B2_TRY(tmap_ndhwc_slab(&sg, a->g, (uint64_t)a->ldg, (uint64_t)pl.p.Wo, (uint64_t)pl.p.Ho, (uint64_t)a->N * pl.p.To, 8, 8, 1));
  B2_TRY(tmap_ndhwc_slab(&sx, a->x, (uint64_t)a->ldx, (uint64_t)a->W, (uint64_t)a->H, (uint64_t)a->N * a->T, 8, 8, a->sh));
  B2_TRY(encode_tmap(&tmG, sg));
  B2_TRY(encode_tmap(&tmX, sx));
  B2_OPT_IN_SMEM(wgrad_kernel, kWgSmem);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  wgrad_kernel<<<pl.grid, pl.block, pl.smem, st>>>(tmG, tmX, pl.p);
  B2_CHECK_LAUNCH("conv_ndhwc_wgrad");
  if (pl.p.S > 1) {
    wgrad_reduce_kernel<<<div_up_t(n, 256), 256, 0, st>>>(a->work, pl.p.S, n, a->dw);
    B2_CHECK_LAUNCH("wgrad_reduce");
  }
  return B2_OK;
}

/* Host-only view of plan_wgrad: grid_x, grid_y, block, smem, m tiles, n tiles, taps, rectangles (low 31 bits), splits,
 * rectangles per row, rectangles per column. */
int b2_debug_wgrad_plan(const b2_wgrad_args* a, int* out, int n) {
  WgradPlan pl;
  B2_TRY(plan_wgrad(a, &pl));
  const int v[11] = {(int)pl.grid.x, (int)pl.grid.y, pl.block, pl.smem, pl.p.mt, pl.p.nt, pl.p.taps, (int)pl.p.rects, pl.p.S,
                     pl.p.rw, pl.p.rh};
  for (int i = 0; i < n && i < 11; ++i) out[i] = v[i];
  return B2_OK;
}

/* The rectangle range [r0, r1) split `s` of that plan reduces over (the same function the kernel calls). */
int b2_debug_wgrad_split(const b2_wgrad_args* a, int s, long long* r0r1) {
  WgradPlan pl;
  B2_TRY(plan_wgrad(a, &pl));
  B2_CHECK_ARG(s >= 0 && s < pl.p.S, "split %d outside [0, %d)", s, pl.p.S);
  wgrad_split_range(pl.p.rects, pl.p.S, s, &r0r1[0], &r0r1[1]);
  return B2_OK;
}

}  // extern "C"
