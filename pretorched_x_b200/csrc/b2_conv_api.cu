// b2_conv_api.cu -- C-ABI entry points for the tcgen05 convolution and dense GEMM kernels.  A host-only planner decides which
// kernel runs a call and with what tiling (plan_conv / plan_gemm: a ConvPlan, no CUDA call but sm_count()); launch_plan runs it.
#include <stdlib.h>
#include <string.h>

#include "b2_host.h"
#include "b2_igemm.cuh"
#include "b2_densem.cuh"
#include "b2_pgemm.cuh"
#include "b2_slabconv.cuh"
#include "b2_slabts.cuh"
#include "b2_tstack.cuh"
#include "b2_stemconv.cuh"

namespace b2 {

// ------------------------------------------------------------------------------------------
// kernel-selection knobs (debug / tuning): read from the environment once, changed by the b2_debug_set_* entry points
// ------------------------------------------------------------------------------------------
struct Tuning {
  int conv_algo = 0;       // 0 auto, 1 gather kernel for every convolution the stem / dense-M kernels do not take (A/B comparisons)
  int gemm_algo = 0;       // 0 auto (persistent kernel where it applies), 1 force the per-tile kernel
  int tstack = -1;         // temporal stack kernel: -1 rule, 0 never (B2_TSTACK=0), 1 whenever the shape is eligible
  bool slabts = true;      // temporal-group slab kernel (B2_SLABTS=0 disables)
  int slab_mt = 0;         // M tiles per slab work item: 0 cost model, > 0 forced (B2_SLAB_MT)
  bool slab_mp = true;     // multi-plane slab work items (B2_SLAB_MP=0 disables)
  int slab_wide = -1;      // 256-column N tiles for channel counts that are multiples of 256: -1 rule, 0 never, 1 always
  int densem_maxm = -1;    // dense-M kernel: -1 rule, 0 never, > 0 replaces both M thresholds (B2_DENSEM_MAXM)
  int densem_s = 0;        // > 0 caps the dense-M cluster size (B2_DENSEM_S)
  bool stem_pair = true;   // pair-of-planes items of the stem kernel (B2_STEM_PAIR=0 disables)
};

static bool env_off(const char* name) { const char* e = getenv(name); return e && e[0] == '0'; }
static int env_int(const char* name, int absent) { const char* e = getenv(name); return e ? atoi(e) : absent; }
static Tuning& tuning() {
  static Tuning t{0, 0, env_off("B2_TSTACK") ? 0 : -1, !env_off("B2_SLABTS"), env_int("B2_SLAB_MT", 0) > 0 ? env_int("B2_SLAB_MT", 0) : 0,
                  !env_off("B2_SLAB_MP"), -1, env_int("B2_DENSEM_MAXM", -1) >= 0 ? env_int("B2_DENSEM_MAXM", -1) : -1,
                  env_int("B2_DENSEM_S", 0), !env_off("B2_STEM_PAIR")};
  return t;
}

// ------------------------------------------------------------------------------------------
// the plan: one launch of one kernel instance, as plain values
// ------------------------------------------------------------------------------------------
enum ConvKernel {          // one value per launched template instance; _lib.CONV_KERNELS names them in this order
  KERN_NONE = 0, KERN_TSTACK, KERN_SLABTS, KERN_SLAB64, KERN_SLAB128, KERN_SLABN, KERN_STEM64, KERN_STEM128, KERN_DENSEM,
  KERN_PGEMM64, KERN_PGEMM64_GAN, KERN_PGEMM128, KERN_PGEMM128_GAN, KERN_IGEMM64, KERN_IGEMM128
};
static const char* const kKernelName[] = {"none", "tstack_kernel", "slabts_kernel", "slabconv_kernel", "slabconv_kernel",
                                          "slabconv_kernel", "stemconv_kernel", "stemconv_kernel", "densem_kernel", "pgemm_kernel",
                                          "pgemm_kernel", "pgemm_kernel", "pgemm_kernel", "igemm_kernel", "igemm_kernel"};

static const int kNumTmaps[] = {0, 2, 2, 2, 2, 2, 1, 1, 2, 7, 7, 7, 7, 4, 4};
constexpr int kMaxTmaps = 7;
struct ConvPlan {
  int kernel;                       // ConvKernel
  dim3 grid, block;
  int smem;                         // dynamic shared memory bytes
  int cluster;                      // CTAs per thread-block cluster along z (dense-M split-K); 1: plain launch
  TmapSpec tm[kMaxTmaps];           // the kernel's tensor maps, in argument order (kNumTmaps[kernel] of them)
  signed char tm_copy[kMaxTmaps];   // >= 0: the same map as tm[tm_copy[i]] (an operand the kernel does not read)
  union {
    SlabParams slab;                // slab kernels and the temporal-group slab kernel
    TstackParams tstack;
    StemParams stem;
    DensemParams densem;
    IgemmParams igemm;
    PgemmParams pgemm;
  } p;
};

static int set_launch(ConvPlan* pl, int kernel, dim3 grid, int block, int smem, int cluster = 1) {
  pl->kernel = kernel; pl->grid = grid; pl->block = dim3(block); pl->smem = smem; pl->cluster = cluster;
  return B2_OK;
}
static dim3 persistent_grid(long long work) { return dim3((unsigned)(work < sm_count() ? work : sm_count())); }   // min(work, SMs)

// ------------------------------------------------------------------------------------------
// slab convolution (stride 1 / 2, "same" padding): geometry and tiling
// ------------------------------------------------------------------------------------------
static int slab_naff(int ldy) { return (ldy + 31) / 32 * 32 + 256; }   // chunk reads may run past ldy inside the last N tile
static long long slab_smem(long long slab_bytes, int w_stage, int ldy) {
  return kSlabSStages * slab_bytes + kSlabWStages * w_stage + 256 + 2 * slab_naff(ldy) * 4 + 1024;
}

static int slab_rows(int MT, int PW, int reach, int P) {
  int R = 0;
  for (int q0 = 0; q0 < P; q0 += MT * 128) {
    int lo = q0 - reach;
    lo = (lo >= 0) ? lo / PW : -((-lo + PW - 1) / PW);
    const int hi = (q0 + MT * 128 - 1 + reach) / PW;
    R = (hi - lo + 1) > R ? (hi - lo + 1) : R;
  }
  return R;
}

// Fills the geometry part of SlabParams (sub-image / tap tables).  Returns false when the convolution is not of a
// shape the slab kernel handles.
static bool slab_geometry(const b2_conv_args* a, SlabParams* p, int wc_hint) {
  if (a->mode != B2_CONV_AUTO || a->out_f32) return false;
  if ((a->kt & 1) == 0 || (a->kh & 1) == 0 || (a->kw & 1) == 0) return false;
  if (a->pt != (a->kt - 1) / 2 || a->ph != (a->kh - 1) / 2 || a->pw != (a->kw - 1) / 2) return false;
  if (a->sh != a->sw || (a->sh != 1 && a->sh != 2) || (a->st != 1 && a->st != 2)) return false;
  if (a->kh * a->kw > kSlabMaxTaps) return false;
  const int ss = a->sh;
  if (a->kt * a->kh * a->kw == 1) return false;   // 1x1x1: persistent GEMM (stride 1) / gather kernel (strided): no tap reuse to exploit
  memset(p, 0, sizeof(*p));
  p->T = a->T; p->C = a->C;
  p->To = (a->T + 2 * a->pt - a->kt) / a->st + 1;
  p->Ho = (a->H + 2 * a->ph - a->kh) / ss + 1;
  p->Wo = (a->W + 2 * a->pw - a->kw) / ss + 1;
  p->kt = a->kt; p->khw = a->kh * a->kw; p->st = a->st; p->ss = ss; p->pt = a->pt;
  p->cchunks = (a->C + 63) / 64;
  // tap (dh, dw) reads input (ss*ho + dh - ph, ss*wo + dw - pw) = phase (rh, rw), sub-image pixel (ho + oi, wo + oj)
  int oi[8], rh[8], oj[8], rw[8];
  int min_oj = 0, max_oj = 0;
  for (int d = 0; d < a->kh; ++d) { int v = d - a->ph; rh[d] = ((v % ss) + ss) % ss; oi[d] = (v - rh[d]) / ss; }
  for (int d = 0; d < a->kw; ++d) {
    int v = d - a->pw; rw[d] = ((v % ss) + ss) % ss; oj[d] = (v - rw[d]) / ss;
    if (oj[d] < min_oj) min_oj = oj[d];
    if (oj[d] > max_oj) max_oj = oj[d];
  }
  p->halo_l = -min_oj;
  // W chunking: rows longer than a TMA box (256 pixels incl. halo) are cut into chunks of WC output columns.  For the
  // temporal remap (kw = 1, "rows" are H*W positions of one frame) a short chunk keeps MT+kt-1 frames in one slab.
  p->WC = p->Wo; p->wchunks = 1;
  const int wc_box = (ss == 1 ? 256 : 128) - p->halo_l - max_oj;                            // TMA box <= 256 traversed pixels
  const int wc_max = (wc_hint > 0 && wc_hint < wc_box) ? wc_hint : wc_box;
  if (p->Wo > wc_max) {
    int best = 0;
    for (int c = wc_max; c >= (wc_max * 3) / 4; --c) if (p->Wo % c == 0) { best = c; break; }   // prefer an exact divisor
    p->WC = best ? best : wc_max;
    p->wchunks = (p->Wo + p->WC - 1) / p->WC;
  }
  p->PW = p->WC + p->halo_l + max_oj;
  p->P = p->Ho * p->PW;
  p->n_sub = 0;
  p->reach = 0;
  for (int ph_ = 0; ph_ < ss; ++ph_)
    for (int pw_ = 0; pw_ < ss; ++pw_) {
      int n = 0;
      const int sidx = p->n_sub;
      for (int dh = 0; dh < a->kh; ++dh)
        for (int dw = 0; dw < a->kw; ++dw)
          if (rh[dh] == ph_ && rw[dw] == pw_) {
            const int off = oi[dh] * p->PW + oj[dw];
            p->sub_off[sidx][n] = (short)off;
            p->sub_tap[sidx][n] = (unsigned char)(dh * a->kw + dw);
            if (off > p->reach) p->reach = off;
            if (-off > p->reach) p->reach = -off;
            ++n;
          }
      if (n == 0) continue;
      p->sub_ntaps[sidx] = n;
      p->sub_h0[sidx] = ph_;                               // + ss * r_lo at run time
      p->sub_w0[sidx] = pw_ - ss * p->halo_l;              // slab column 0 = sub-image column -halo_l
      ++p->n_sub;
    }
  if (a->upsample) {
    // 3x3 conv of the nearest-2x upsampled image: output (2h + py, 2w + px) reads low-res rows {h - 1, h} (py = 0) or
    // {h, h + 1} (py = 1), same for columns; the folded 2x2 filters of phase ph are weight taps ph*4 .. ph*4 + 3
    const int s_h0 = p->sub_h0[0], s_w0 = p->sub_w0[0];
    for (int ph = 0; ph < 4; ++ph) {
      const int py = ph >> 1, px = ph & 1;
      for (int ai = 0; ai < 2; ++ai)
        for (int bi = 0; bi < 2; ++bi) {
          const int ro = ai - 1 + py, co = bi - 1 + px;
          p->sub_off[ph][ai * 2 + bi] = (short)(ro * p->PW + co);
          p->sub_tap[ph][ai * 2 + bi] = (unsigned char)(ph * 4 + ai * 2 + bi);
        }
      p->sub_ntaps[ph] = 4; p->sub_h0[ph] = s_h0; p->sub_w0[ph] = s_w0;
    }
    p->khw = 16; p->up = 1; p->n_sub = 1;
  }
  return p->n_sub > 0 && p->PW <= 256;
}

// Fills the run-time part of SlabParams that the slab and temporal-group kernels share; the caller sets the N tile, the
// accumulator sets, the N tiles and the work items.
static void slab_fill(const b2_conv_args* a, SlabParams& p, int MT, int R) {
  p.R = R;
  p.planes_total = a->N * p.To;
  p.plane_stride = R * p.PW * 128;
  p.slab_bytes = ((R * p.PW * 128 * (p.mp > 1 ? p.mp : 1)) + 1023) / 1024 * 1024;
  p.MT = MT;
  p.Ncols = a->K;
  p.scale = a->scale; p.shift = a->shift;
  p.residual = reinterpret_cast<const __half*>(a->residual);
  p.ldr = a->ldr;
  p.y = reinterpret_cast<__half*>(a->y);
  p.ldy = a->ldy;
  p.relu = a->relu;
  p.aff_ld = a->aff_ld;
  p.naff = slab_naff(a->ldy);
  p.tiles_q = p.mp > 1 ? 1 : (p.P + MT * 128 - 1) / (MT * 128);
  p.fd_tiles_q = make_fastdiv(p.tiles_q); p.fd_wchunks = make_fastdiv(p.wchunks); p.fd_PW = make_fastdiv(p.PW);
}

struct SlabTiles {
  int bn;          // N tile
  bool flex;       // runtime-N instance (slabconv_kernel<0>)
  int mt, R;       // M tiles per work item and slab rows; mt == 0: no configuration fits in shared memory
  double cost;     // modelled cycles
};

// Picks the N tile (fixed 64 / 128 or runtime), the M tiles per work item and the slab rows for a geometry.
static SlabTiles slab_pick_tiles(const b2_conv_args* a, SlabParams& p, bool wide) {
  const Tuning& t = tuning();
  int BN = (a->ldy <= 64) ? 64 : 128;
  const int planes = a->N * p.To;
  int ntn = (a->ldy + BN - 1) / BN;
  // Channel counts that tile badly by 128 (144, 288, 576 ... of R(2+1)D) take the runtime-N instance: the fewest
  // tiles of <= 256 columns, each a multiple of 16 wide.
  bool flex = false;
  if (a->ldy > 128) {
    const int tn = (a->ldy + 255) / 256;
    const int bn = (((a->ldy + tn - 1) / tn) + 15) / 16 * 16;
    if ((long long)bn * tn * 21 <= (long long)ntn * 128 * 20 || ((wide || t.slab_wide == 1) && a->ldy % 256 == 0)) {
      flex = true; BN = bn; ntn = tn;
      p.bn = bn; p.wbytes = (bn * 128 + 1023) / 1024 * 1024; p.accs = (bn + 31) / 32 * 32;
    }
  } else if (a->ldy <= 16) {
    // a handful of output channels (the generator's RGB head): the narrowest MMA (N = 16) instead of a 64-wide tile
    // that is 95% padding -- the A operand still streams through shared memory once per tap, so this saves a third
    flex = true; BN = 16; ntn = 1;
    p.bn = 16; p.wbytes = 2048; p.accs = 32;
  }
  const int acc_stride = flex ? p.accs : BN;
  const int w_stage = flex ? p.wbytes : BN * 128;
  // Pick the M tiles per work item from a cycle model of one SM's share: rounds of items x the slower of the MMA
  // stream and the slab/weight loads, plus the epilogue when a single accumulator set leaves it exposed.  (Constants
  // from ncu: a 128xNx16 MMA retires in ~40 + N/2 cycles, TMA delivers ~48 B/cycle/SM out of L2.)
  int best_mt = 0, best_R = 0;
  double best_cost = 0.0;
  const int force_mt = t.slab_mt;
  int ksteps = 0;
  for (int cc = 0; cc < p.cchunks; ++cc) { const int k = (a->C - cc * 64 + 15) / 16; ksteps += k > 4 ? 4 : k; }
  int taps_hw = 0;
  for (int sidx = 0; sidx < p.n_sub; ++sidx) taps_hw += p.sub_ntaps[sidx];
  // planes of at most one M tile whose temporal taps do not differ from plane to plane: the MT accumulators of an item are MT
  // consecutive PLANES (SlabParams::mp), see b2_slabconv.cuh
  const bool mp_ok = t.slab_mp && p.P <= 128 && (a->kt == 1 || a->T == 1) && p.ss == 1 && !p.up && p.wchunks == 1 && planes > 1 &&
                     !a->aff_ld;      // (a per-sample affine is read once per item: its tiles must belong to one image)
  p.mp = 0;
  for (int MT = 512 / acc_stride > 4 ? 4 : 512 / acc_stride; MT >= 1; --MT) {
    if (force_mt > 0 && MT != force_mt && MT != 1) continue;
    // (multi-plane: rows one plane's positions and taps can touch -- slab_rows assumes a full 128-position tile)
    const int R = mp_ok ? (p.P - 1 + p.reach) / p.PW + (p.reach + p.PW - 1) / p.PW + 1 : slab_rows(MT, p.PW, p.reach, p.P);
    if (p.ss * (R - 1) + 1 > 256) continue;
    const long long slab_b = ((long long)R * p.PW * 128 * (mp_ok ? MT : 1) + 1023) / 1024 * 1024;
    if (slab_smem(slab_b, w_stage, a->ldy) > 227 * 1024) continue;
    const long long tq = mp_ok ? 1 : (p.P + MT * 128 - 1) / (MT * 128);
    const long long items = (long long)ntn * tq * (mp_ok ? (planes + MT - 1) / MT : planes) * p.wchunks * (p.up ? 4 : 1);
    const double rounds = (double)((items + sm_count() - 1) / sm_count());
    const double tiles_per_item = mp_ok ? (double)MT : (double)((p.P + 127) / 128) / (double)tq;   // average (the last item of a plane is short)
    // (A per-weight-tile issue floor of ~650 cycles was tried here after profiles/ncu_r02 showed the issuing warp, not the tensor
    // pipe, pacing one-tile items with a narrow N; it moved the (1,3,3) C64->144 layer from MT = 1 with two accumulator sets to MT = 2
    // with one, which measured 59 us instead of 44 us -- losing the epilogue overlap costs more than the amortised issue work gains.)
    const double mma = tiles_per_item * p.kt * taps_hw * ksteps * (40.0 + 0.5 * BN);
    // small planes: every SM streams the whole filter per item at the same time, and what bounds that is the aggregate L2 -> SM rate
    // (~7 TB/s = 26 B/cycle/SM: 192 items x 884 KB in 25 us on the 7x7 C256->576 layer), not one SM's TMA rate
    const double bpc = mp_ok ? 26.0 : 48.0;
    const double load = (double)p.kt * p.n_sub * p.cchunks * slab_b / bpc + (double)p.kt * taps_hw * p.cchunks * w_stage / bpc;
    const double epi = (MT * acc_stride <= 256) ? 0.0 : tiles_per_item * ((BN + 31) / 32) * 250.0;
    const double cost = rounds * ((mma > load ? mma : load) + epi + 1500.0);
    if (best_mt == 0 || cost < best_cost || (force_mt > 0 && MT == force_mt)) { best_mt = MT; best_R = R; best_cost = cost; }
    if (force_mt > 0 && MT == force_mt) break;
  }
  if (mp_ok && best_mt >= 2 && best_mt < 4 && force_mt <= 0 && 4 * acc_stride <= 512) {
    // measured (profiles/slab_mp_sweep_r02.txt): four planes per item beat two by ~10% as long as a full wave of items remains
    const int R4 = (p.P - 1 + p.reach) / p.PW + (p.reach + p.PW - 1) / p.PW + 1;
    const long long slab4 = ((long long)R4 * p.PW * 128 * 4 + 1023) / 1024 * 1024;
    const long long items4 = (long long)ntn * ((planes + 3) / 4);
    if (slab_smem(slab4, w_stage, a->ldy) <= 227 * 1024 && items4 >= sm_count()) { best_mt = 4; best_R = R4; }
  }
  p.mp = (mp_ok && best_mt > 1) ? best_mt : 0;
  return SlabTiles{BN, flex, best_mt, best_R, best_cost};
}

// The slab kernel.  Declines (B2_OK, no kernel) shapes it does not take.
static int plan_slab(const b2_conv_args* a_in, ConvPlan* pl) {
  b2_conv_args remap;
  const b2_conv_args* a = a_in;
  int wc_hint = 0;
  if (a_in->kt > 1 && a_in->kh == 1 && a_in->kw == 1 && a_in->st == 1 && a_in->sh == 1 && a_in->sw == 1 && a_in->ph == 0 &&
      a_in->pw == 0) {
    // (kt,1,1) over [N][T][H][W] == (1,kt,1) over N images of T rows x (H*W) columns
    remap = *a_in;
    remap.T = 1; remap.H = a_in->T; remap.W = a_in->H * a_in->W;
    remap.kt = 1; remap.kh = a_in->kt; remap.kw = 1;
    remap.pt = 0; remap.ph = a_in->pt; remap.pw = 0;
    a = &remap;
    wc_hint = 64;
  }
  // W chunking candidates: the default (whole rows, or <= 256-pixel chunks) and narrower chunks.  Narrow chunks make the
  // slab of a work item shorter, which (a) lets 256-pixel rows fit the two slab stages at all and (b) admits more M tiles
  // per item for wide images -- with few-tap 2-D filters the per-item costs (decode, epilogue set-up, slab latency) are
  // what the cycle model trades against the extra halo columns.  The cheapest modelled configuration wins.
  const int wc_try[3] = {wc_hint, 128, 64};
  SlabParams& p = pl->p.slab;
  SlabTiles best = {};
  for (int attempt = 0; attempt < 3; ++attempt) {
    if (attempt > 0 && (wc_hint > 0 || wc_try[attempt] >= a->W)) continue;
    SlabParams q;
    if (!slab_geometry(a, &q, wc_try[attempt])) { if (attempt == 0) return B2_OK; else continue; }
    if (attempt > 0 && q.wchunks == 1) continue;              // same geometry as the default
    SlabTiles c = slab_pick_tiles(a, q, false);
    if (tuning().slab_wide < 0 && a->ldy % 256 == 0 && !c.flex) {
      // 256-column N tiles (one A read per 256 output channels instead of per 128): measured with tools/conv_sweep.py
      // (profiles/slab_wide_sweep_r02.txt) they win by 5-35% wherever at least 64 work items of at least two M tiles remain, and lose
      // when halving the number of N tiles leaves SMs idle (M = 6272: 33 -> 41 us) or an item is a single tile (7x7 planes: 23 -> 29 us)
      SlabParams qw = q;
      const SlabTiles w = slab_pick_tiles(a, qw, true);
      if (w.mt != 0 && w.flex) {
        const long long tq = (qw.P + w.mt * 128 - 1) / (w.mt * 128);
        const long long items_w = (long long)((a->ldy + w.bn - 1) / w.bn) * tq * a->N * qw.To * qw.wchunks * (qw.up ? 4 : 1);
        const double tiles_per_item = (double)((qw.P + 127) / 128) / (double)tq;
        if (items_w >= 64 && tiles_per_item >= 2.0) { q = qw; c = w; c.cost = w.cost * 0.8; }
      }
    }
    if (c.mt == 0) continue;
    if (best.mt == 0 || c.cost < best.cost) { p = q; best = c; }
  }
  if (best.mt == 0) return B2_OK;
  if (!best.flex) { p.bn = best.bn; p.wbytes = best.bn * 128; p.accs = best.bn; }
  slab_fill(a, p, best.mt, best.R);
  p.nacc = (best.mt * p.accs <= 256) ? 2 : 1;
  p.tiles_n = (a->ldy + p.bn - 1) / p.bn;
  const long long plane_items = p.mp > 1 ? ((long long)a->N * p.To + p.mp - 1) / p.mp : (long long)a->N * p.To;
  const long long items = (long long)p.tiles_n * p.tiles_q * p.wchunks * plane_items * (p.up ? 4 : 1);
  if (items >= (1ll << 31)) return set_error(B2_ERR_INVALID, "slab problem too large");
  p.items_total = (int)items;
  p.fd_tiles_n = make_fastdiv(p.tiles_n); p.fd_To = make_fastdiv(p.To);
  if (a->aff_ld && ((a->aff_ld & 3) || (reinterpret_cast<uintptr_t>(a->scale) & 15) || (reinterpret_cast<uintptr_t>(a->shift) & 15)))
    return set_error(B2_ERR_INVALID, "per-sample scale/shift must be 16-byte aligned with a pitch that is a multiple of 4 floats");
  const int taps = p.up ? 16 : a->kt * a->kh * a->kw;
  B2_TRY(tmap_ndhwc_slab(&pl->tm[0], a->x, (uint64_t)a->C, (uint64_t)a->W, (uint64_t)a->H, (uint64_t)a->N * a->T, (uint32_t)p.PW,
                         (uint32_t)p.R, (uint32_t)p.ss, (uint32_t)(p.mp > 1 ? p.mp : 1)));
  B2_TRY(tmap_2d_f16(&pl->tm[1], a->w, (uint64_t)taps * a->C, (uint64_t)a->K, (uint64_t)taps * a->C, 64, p.bn, true));
  return set_launch(pl, best.flex ? KERN_SLABN : best.bn == 64 ? KERN_SLAB64 : KERN_SLAB128, persistent_grid(p.items_total), kSlabThreads,
                    (int)slab_smem(p.slab_bytes, p.wbytes, a->ldy));
}

// ------------------------------------------------------------------------------------------
// temporal-group slab kernel (b2_slabts.cuh): 3 x kh x kw stride-1 "same" convolutions with <= 64 output channels
// ------------------------------------------------------------------------------------------
static int plan_slabts(const b2_conv_args* a, ConvPlan* pl) {
  if (!tuning().slabts) return B2_OK;
  if (a->kt != 3 || a->st != 1 || a->pt != 1 || a->sh != 1 || a->sw != 1 || a->ldy > 64 || a->T < 3) return B2_OK;
  // Measured (CUDA-graph replays, profiles/README_r02.md): 180 vs 186 us on the 3x3x3 C64->64 layer of resnet3d50 -- the operand
  // traffic it saves in shared memory comes back as 2.5x more weight bytes per output tile from L2 (one 24 KB stack per tap and input
  // frame, two M tiles per item) -- and it LOSES where the single accumulator set exposes a residual read (243 vs 190 us) or the
  // in-plane filter is 1x1 (the (3,1,1) convolutions of R(2+1)D: 64 vs 31 us against the frames-as-rows remap).  So: true 3-D
  // filters without a residual only.
  if (a->kh * a->kw < 9 || a->residual) return B2_OK;
  SlabParams& p = pl->p.slab;
  if (!slab_geometry(a, &p, 0) || p.n_sub != 1) return B2_OK;
  int MT = p.P > 128 ? 2 : 1, R = 0;
  long long smem = 0;
  for (; MT >= 1; --MT) {
    R = slab_rows(MT, p.PW, p.reach, p.P);
    smem = slab_smem(((long long)R * p.PW * 128 + 1023) / 1024 * 1024, kTsWBytes, a->ldy);
    if (R <= 256 && smem <= 227 * 1024) break;
  }
  if (MT < 1) return B2_OK;
  slab_fill(a, p, MT, R);
  p.nacc = 1; p.bn = kTsBN; p.wbytes = kTsWBytes; p.accs = kTsBN;
  p.tiles_n = 1;
  const int groups = (p.To + kTsGroup - 1) / kTsGroup;
  const long long items = (long long)p.tiles_q * p.wchunks * a->N * groups;
  if (items >= (1ll << 31)) return B2_OK;
  p.items_total = (int)items;
  p.fd_tiles_n = make_fastdiv(1); p.fd_To = make_fastdiv(groups);
  const int taps = a->kt * a->kh * a->kw;
  B2_TRY(tmap_ndhwc_slab(&pl->tm[0], a->x, (uint64_t)a->C, (uint64_t)a->W, (uint64_t)a->H, (uint64_t)a->N * a->T, (uint32_t)p.PW,
                         (uint32_t)R, 1u));
  B2_TRY(tmap_2d_f16(&pl->tm[1], a->w, (uint64_t)taps * a->C, (uint64_t)a->K, (uint64_t)taps * a->C, 64, kTsBN, true));
  return set_launch(pl, KERN_SLABTS, persistent_grid(p.items_total), kSlabThreads, (int)smem);
}

// ------------------------------------------------------------------------------------------
// temporal stack kernel (b2_tstack.cuh): (kt,1,1) stride-1 "same" convolutions with <= 64 output channels, resident filter
// ------------------------------------------------------------------------------------------
static int plan_tstack(const b2_conv_args* a, ConvPlan* pl) {
  const int mode = tuning().tstack;
  if (mode == 0) return B2_OK;
  if (a->kh != 1 || a->kw != 1 || a->kt < 3 || !(a->kt & 1) || a->st != 1 || a->sh != 1 || a->sw != 1 || a->pt != a->kt / 2 || a->ph != 0 ||
      a->pw != 0 || a->ldy > 64 || a->T < 2)
    return B2_OK;
  const int cchunks = (a->C + 63) / 64;
  const long long wbytes = (long long)cchunks * a->kt * kTkWBlock;
  if (wbytes > 144 * 1024) return B2_OK;                     // the filter must stay resident next to the A ring
  const long long HW = (long long)a->H * a->W;
  if (HW >= (1ll << 24)) return B2_OK;
  TstackParams& p = pl->p.tstack;
  p = TstackParams{};
  p.T = a->T; p.HW = (int)HW; p.C = a->C;
  p.kt = a->kt; p.pt = a->pt;
  p.cchunks = cchunks;
  p.groups = (a->T + kTkG - 1) / kTkG;
  p.tiles_q = (int)((HW + 127) / 128);
  const long long items = (long long)a->N * p.groups * p.tiles_q;
  if (items >= (1ll << 31)) return B2_OK;
  // Below one work item per SM the frames-as-rows form of the slab kernel (more, smaller items) keeps more SMs busy
  // (2 clips of the (3,1,1) C144 layer, 56 items: 9.6 vs 11.0 us, profiles/tstack_sweep_r02.txt).
  if (mode < 0 && items < sm_count()) return B2_OK;
  p.items_total = (int)items;
  p.Ncols = a->K; p.ldy = a->ldy; p.ldr = a->ldr; p.relu = a->relu;
  p.scale = a->scale; p.shift = a->shift;
  p.residual = reinterpret_cast<const __half*>(a->residual);
  p.y = reinterpret_cast<__half*>(a->y);
  p.fd_tiles_q = make_fastdiv(p.tiles_q); p.fd_groups = make_fastdiv(p.groups);
  B2_TRY(tmap_ndhwc_slab(&pl->tm[0], a->x, (uint64_t)a->C, (uint64_t)HW, 1, (uint64_t)a->N * a->T, 128u, 1u, 1u));
  B2_TRY(tmap_2d_f16(&pl->tm[1], a->w, (uint64_t)a->kt * a->C, (uint64_t)a->K, (uint64_t)a->kt * a->C, 64, 64, true));
  return set_launch(pl, KERN_TSTACK, persistent_grid(p.items_total), kTkThreads, (int)(1024 + kTkStages * kTkABytes + wbytes + 128 + 512 + 64));
}

// ------------------------------------------------------------------------------------------
// stem convolution (Toeplitz-descriptor kernel)
// ------------------------------------------------------------------------------------------
static int plan_stem(const b2_conv_args* a, int BN, ConvPlan* pl) {
  StemParams& p = pl->p.stem;
  memset(&p, 0, sizeof(p));
  p.T = a->T; p.H = a->H; p.W = a->W;
  p.To = (a->T + 2 * a->pt - a->kt) / a->st + 1;
  p.Ho = (a->H + 2 * a->ph - a->kh) / 2 + 1;
  p.Wo = (a->W + 6 - 7) / 2 + 1;
  p.kt = a->kt; p.kh = a->kh; p.pt = a->pt; p.ph = a->ph;
  p.G = 256 / BN;
  p.rows = 2 * (p.G - 1) + a->kh;
  if (p.rows > kStemMaxRows) return set_error(B2_ERR_UNSUPPORTED, "stem kernel height %d too large", a->kh);
  for (int i = 0; i < p.rows; ++i) {
    int g_lo = i - (a->kh - 1);
    g_lo = g_lo > 0 ? (g_lo + 1) / 2 : 0;
    int g_hi = i / 2;
    if (g_hi > p.G - 1) g_hi = p.G - 1;
    p.row_glo[i] = (signed char)g_lo;
    p.row_ghi[i] = (signed char)g_hi;
    p.row_slot[i] = (signed char)(g_lo <= g_hi ? stem_slot(i - 2 * g_lo, a->kh) : 0);
  }
  p.w_bytes = a->kh * BN * 64;
  p.stage_bytes = ((p.rows * kStemPitch + p.w_bytes) + 127) / 128 * 128;
  const int tail_bytes = 128 + 2048 + 1024 + 256;     // barriers, scale / shift, W-pool exchange slots
  p.nstages = (227 * 1024 - tail_bytes) / p.stage_bytes;
  if (p.nstages > kStemMaxStages) p.nstages = kStemMaxStages;
  if (p.nstages < 1) return set_error(B2_ERR_UNSUPPORTED, "stem slab does not fit in shared memory (kh=%d)", a->kh);
  p.Ncols = a->K;
  p.ntiles_n = (a->ldy + BN - 1) / BN;
  if (p.ntiles_n * BN > 256) return set_error(B2_ERR_UNSUPPORTED, "stem convolution supports at most 256 output channels");
  p.tiles_w = (p.Wo + kStemTileW - 1) / kStemTileW;
  p.tiles_h = (p.Ho + p.G - 1) / p.G;
  p.planes_total = a->N * p.To;
  p.pair = (tuning().stem_pair && a->kt == 1 && a->pt == 0 && p.Wo <= 60 && !a->pool_w && a->W <= 120) ? 1 : 0;
  const long long plane_items = p.pair ? (p.planes_total + 1) / 2 : p.planes_total;
  const long long items = (long long)p.tiles_w * p.tiles_h * p.ntiles_n * plane_items;
  if (items >= (1ll << 31)) return set_error(B2_ERR_INVALID, "stem problem too large");
  p.items_total = (int)items;
  p.wimg = reinterpret_cast<const __half*>(a->w);
  p.scale = a->scale; p.shift = a->shift;
  p.y = reinterpret_cast<__half*>(a->y);
  p.ldy = a->ldy;
  p.relu = a->relu;
  p.pool_w = a->pool_w; p.Wp = (p.Wo - 1) / 2 + 1;
  if (a->pool_w && (!a->relu || p.tiles_w != 1))
    return set_error(B2_ERR_UNSUPPORTED, "fused W pooling needs ReLU and an output row of at most %d columns (got %d)", kStemTileW, p.Wo);
  // input viewed as 8-byte pixels (W, H, N*T); box (256, rows, 1); no swizzle -> dense 2 KB rows in smem
  TmapSpec& tm = pl->tm[0];
  tm = TmapSpec{a->x, CU_TENSOR_MAP_DATA_TYPE_UINT64, 3, {(cuuint64_t)a->W, (cuuint64_t)a->H, (cuuint64_t)a->N * a->T},
                {(cuuint64_t)a->W * 8, (cuuint64_t)a->H * a->W * 8}, {(cuuint32_t)kStemRowPx, (cuuint32_t)p.rows, 1}, {1, 1, 1}, false};
  if (p.pair) {      // (W, plane, H): box (128 pixels, 2 planes, rows) -> smem [row][plane][1024 B]
    tm.dims[1] = (cuuint64_t)a->N * a->T; tm.dims[2] = (cuuint64_t)a->H;
    tm.strides[0] = (cuuint64_t)a->H * a->W * 8; tm.strides[1] = (cuuint64_t)a->W * 8;
    tm.box[0] = 128; tm.box[1] = 2; tm.box[2] = (cuuint32_t)p.rows;
  }
  return set_launch(pl, BN == 64 ? KERN_STEM64 : KERN_STEM128, persistent_grid(p.items_total), kStemThreads, p.nstages * p.stage_bytes + tail_bytes);
}

// ------------------------------------------------------------------------------------------
// GEMM-shaped launches shared by convolutions and the GEMM entry points
// ------------------------------------------------------------------------------------------
struct IgemmLaunch {
  IgemmParams p;
  // optional second operand pair (persistent GEMM only): D += A2[M][k2] . B2[N][k2]^T
  const void* a2 = nullptr; int lda2 = 0; const void* w2 = nullptr; int ldb2 = 0; int k2 = 0;
  const void* a_mat;      // AMODE_TMA: A as [M][lda]
  int lda;
  int a_cols;             // logical K extent of A (columns readable)
  const void* w;          // B as [Ncols][ldb]
  int ldb;
  int b_cols;             // logical K extent of B
};

// Which layers take the dense-M kernel (measured with tools/conv_sweep.py as CUDA-graph replays, profiles/smallm_sweep_r02.txt):
// it beats the slab kernel only where a plane fills a small part of a 128-row tile AND the K loop is long enough to split --
// stride-1 multi-tap convolutions with M <= 1024 output positions (4x4 planes: 12% tile fill), strided multi-tap convolutions
// (whose slab form needs four phase sub-images per tap) with M <= 8192.  1x1x1 convolutions stay on the persistent GEMM.
// Only plain per-column affines without the generator's extras qualify; the callers test that.
static bool densem_wanted(long long M, int taps, bool strided) {
  const Tuning& t = tuning();
  if (t.gemm_algo != 0) return false;
  if (t.densem_maxm >= 0) return t.densem_maxm > 0 && M <= t.densem_maxm;
  if (taps <= 1) return false;
  return strided ? M <= 8192 : M <= 1024;
}

// N tile (multiple of 32, <= 256, least padding then widest) and cluster size S (bn / S a multiple of 32, >= 2 K blocks per CTA):
// the smallest S that gives every SM a work unit, else the largest admissible one.
static bool densem_split_ok(int bn, int S, int nkb) {      // bn / S a multiple of 32 and every CTA of the cluster gets >= 1 K block
  if (S < 1 || bn % (32 * S) != 0 || S > nkb) return false;
  const int per = (nkb + S - 1) / S;
  return (S - 1) * per < nkb;
}
static int plan_densem(const IgemmLaunch& L, ConvPlan* pl) {
  const IgemmParams& p = L.p;
  const int width = (p.epi == EPI_DIRECT_F32) ? p.Ncols : p.ldy;
  int bn = 256, best_waste = 1 << 30;
  for (int c = 256; c >= 64; c -= 32) {
    const int waste = (width + c - 1) / c * c - width;
    if (waste < best_waste) { best_waste = waste; bn = c; }
  }
  if (width <= 32) bn = 32;
  const int tiles = ((p.M_total + 127) / 128) * ((width + bn - 1) / bn);
  const int force_s = tuning().densem_s;
  int S = 1;
  for (int cand = 1; cand <= 8; ++cand) {
    if (!densem_split_ok(bn, cand, p.nkb) || (cand > 1 && p.nkb / cand < 2)) continue;
    if (force_s > 0) { if (cand <= force_s) S = cand; continue; }
    S = cand;
    if (tiles * cand >= 64) break;                  // measured: beyond ~half the SMs the cluster / DSMEM cost outgrows the gain
  }
  DensemParams& dp = pl->p.densem;
  memset(&dp, 0, sizeof(dp));
  dp.g = p;
  dp.bn = bn; dp.bbytes = bn * 128; dp.stage_bytes = kBM * kBK * 2 + dp.bbytes;
  dp.tmem_cols = bn <= 32 ? 32 : bn <= 64 ? 64 : bn <= 128 ? 128 : 256;
  dp.ksplit = S;
  dp.kb_per = (p.nkb + S - 1) / S;
  dp.nstages = (227 * 1024 - 256 - 1024) / dp.stage_bytes;
  if (dp.nstages > kDmMaxStages) dp.nstages = kDmMaxStages;
  B2_TRY(tmap_2d_f16(&pl->tm[1], L.w, (uint64_t)L.b_cols, (uint64_t)p.Ncols, (uint64_t)L.ldb, kBK, (uint32_t)bn, true));
  if (p.amode == AMODE_TMA) B2_TRY(tmap_2d_f16(&pl->tm[0], L.a_mat, (uint64_t)L.a_cols, (uint64_t)p.M_total, (uint64_t)L.lda, kBK, kBM, true));
  else pl->tm_copy[0] = 1;
  return set_launch(pl, KERN_DENSEM, dim3((width + bn - 1) / bn, (p.M_total + kBM - 1) / kBM, S), kDmThreads,
                    dp.nstages * dp.stage_bytes + 256 + 1024, S);
}

static int plan_pgemm(const IgemmLaunch& L, int BN, bool gan, ConvPlan* pl) {
  const IgemmParams& ip = L.p;
  B2_TRY(tmap_2d_f16(&pl->tm[0], L.a_mat, (uint64_t)L.a_cols, (uint64_t)ip.M_total, (uint64_t)L.lda, 64, 128, true));
  B2_TRY(tmap_2d_f16(&pl->tm[1], L.w, (uint64_t)L.b_cols, (uint64_t)ip.Ncols, (uint64_t)L.ldb, 64, BN, true));
  B2_TRY(tmap_2d_f16(&pl->tm[4], ip.y, (uint64_t)ip.ldy, (uint64_t)ip.M_total, (uint64_t)ip.ldy, 64, 128, true));
  const int up_W = ip.up_W > 0 ? ip.up_W : 2;
  const int res_rows = up_W >= 128 ? 64 : 32;
  if (ip.residual && ip.res_up) {
    // low-res skip tensor: a tile's 128 output rows read res_rows consecutive rows of it (see PgemmParams::res_up)
    if (!(up_W % 128 == 0 || (up_W <= 64 && 64 % up_W == 0)))
      return set_error(B2_ERR_UNSUPPORTED, "residual_up needs an output width that is a multiple of 128 or divides 64 (got %d)", up_W);
    B2_TRY(tmap_2d_f16(&pl->tm[5], ip.residual, (uint64_t)ip.ldr, (uint64_t)ip.M_total / 4, (uint64_t)ip.ldr, 64, res_rows, true));
  } else if (ip.residual) {
    B2_TRY(tmap_2d_f16(&pl->tm[5], ip.residual, (uint64_t)ip.ldr, (uint64_t)ip.M_total, (uint64_t)ip.ldr, 64, 128, true));
  } else {
    pl->tm_copy[5] = 4;
  }
  if (ip.y2) B2_TRY(tmap_2d_f16(&pl->tm[6], ip.y2, (uint64_t)ip.ldy, (uint64_t)ip.M_total, (uint64_t)ip.ldy, 64, 128, true));
  else pl->tm_copy[6] = 4;
  if (L.k2 > 0) {
    B2_TRY(tmap_2d_f16(&pl->tm[2], L.a2, (uint64_t)L.k2, (uint64_t)ip.M_total, (uint64_t)L.lda2, 64, 128, true));
    B2_TRY(tmap_2d_f16(&pl->tm[3], L.w2, (uint64_t)L.k2, (uint64_t)ip.Ncols, (uint64_t)L.ldb2, 64, BN, true));
  } else {
    pl->tm_copy[2] = 0; pl->tm_copy[3] = 1;
  }
  PgemmParams& p = pl->p.pgemm;
  p = PgemmParams{};
  p.M = ip.M_total; p.Ncols = ip.Ncols; p.ldy = ip.ldy; p.nkb = ip.nkb;
  p.nkb2 = (L.k2 + 63) / 64;
  p.tiles_n = (ip.ldy + BN - 1) / BN;
  p.tiles_total = p.tiles_n * ((ip.M_total + 127) / 128);
  p.scale = ip.scale; p.shift = ip.shift;
  p.has_residual = ip.residual != nullptr;
  p.relu = ip.relu;
  p.aff_ld = ip.aff_ld; p.aff_rows = ip.aff_rows;
  p.res_up = ip.res_up ? ip.residual : nullptr;
  p.res_ld = ip.ldr; p.Wh = up_W; p.Hh = ip.up_H > 0 ? ip.up_H : 2; p.res_rows = res_rows;
  p.fd_Wh = make_fastdiv(p.Wh); p.fd_Hh = make_fastdiv(p.Hh);
  p.res_pre = ip.res_pre;
  p.in_scale = gan ? ip.in_scale : nullptr; p.in_shift = ip.in_shift; p.in_ld = ip.in_ld; p.in_rows = ip.in_rows > 0 ? ip.in_rows : 128;
  p.dual = ip.y2 != nullptr; p.scale2 = ip.scale2; p.shift2 = ip.shift2; p.aff2_ld = ip.aff2_ld; p.aff2_rows = ip.aff2_rows > 0 ? ip.aff2_rows : 128;
  const int kernel = BN == 64 ? (gan ? KERN_PGEMM64_GAN : KERN_PGEMM64) : (gan ? KERN_PGEMM128_GAN : KERN_PGEMM128);
  return set_launch(pl, kernel, persistent_grid(p.tiles_total), gan ? kPgThreadsGan : kPgThreads,
                    BN == 64 ? PgemmSmem<64>::kTotal : PgemmSmem<128>::kTotal);
}

static int plan_igemm(const IgemmLaunch& L, ConvPlan* pl) {
  const IgemmParams& p = L.p;
  // 64-wide tiles for narrow outputs, 128 otherwise
  const int BN = ((p.epi == EPI_TMA_F16) ? p.ldy : p.Ncols) <= 64 ? 64 : 128;
  B2_TRY(tmap_2d_f16(&pl->tm[1], L.w, (uint64_t)L.b_cols, (uint64_t)p.Ncols, (uint64_t)L.ldb, kBK, BN, true));
  if (p.amode == AMODE_TMA) B2_TRY(tmap_2d_f16(&pl->tm[0], L.a_mat, (uint64_t)L.a_cols, (uint64_t)p.M_total, (uint64_t)L.lda, kBK, kBM, true));
  else pl->tm_copy[0] = 1;
  if (p.epi == EPI_TMA_F16) {
    B2_TRY(tmap_2d_f16(&pl->tm[2], p.y, (uint64_t)p.ldy, (uint64_t)p.M_total, (uint64_t)p.ldy, 64, kBM, true));
    if (p.residual) B2_TRY(tmap_2d_f16(&pl->tm[3], p.residual, (uint64_t)p.ldr, (uint64_t)p.M_total, (uint64_t)p.ldr, 64, kBM, true));
    else pl->tm_copy[3] = 2;
  } else {
    pl->tm_copy[2] = 1; pl->tm_copy[3] = 1;
  }
  pl->p.igemm = p;
  return set_launch(pl, BN == 64 ? KERN_IGEMM64 : KERN_IGEMM128,
                    dim3((p.epi == EPI_TMA_F16 ? (p.ldy + BN - 1) / BN : (p.Ncols + BN - 1) / BN), (p.M_total + kBM - 1) / kBM, 1),
                    kThreads, BN == 64 ? IgemmSmem<64>::kTotalBytes : IgemmSmem<128>::kTotalBytes);
}

// dense_m: the caller found the launch plain and small enough for the dense-M kernel
static int plan_gemm_shaped(const IgemmLaunch& L, bool dense_m, ConvPlan* pl) {
  const IgemmParams& p = L.p;
  if (dense_m) return plan_densem(L, pl);
  if (tuning().gemm_algo == 0 && p.amode == AMODE_TMA && p.epi == EPI_TMA_F16 && !p.per_row) {
    // the generator's extras need the GAN instance; a second output needs the 64-wide one (it has a second staging tile)
    const bool gan = p.y2 || p.res_up || p.res_pre || p.in_scale;
    return plan_pgemm(L, (p.y2 || p.ldy <= 64) ? 64 : 128, gan, pl);
  }
  if (p.aff_ld)
    return set_error(B2_ERR_UNSUPPORTED, "per-sample affine is implemented by the slab convolution and the persistent GEMM only");
  if (p.res_up || p.res_pre || p.y2 || p.in_scale)
    return set_error(B2_ERR_UNSUPPORTED, "upsampled / pre-scale residuals, second outputs and input affines are implemented by the persistent GEMM (1x1 convolutions, fp16) only");
  return plan_igemm(L, pl);
}

// ------------------------------------------------------------------------------------------
// the planners of the entry points, and the launcher
// ------------------------------------------------------------------------------------------
static int conv_out_dim(int in, int k, int s, int p) { return (in + 2 * p - k) / s + 1; }

// Order: dense-M pre-check -> temporal stack -> temporal-group slab -> slab -> stem / 1x1x1 / gather GEMM.
static int plan_conv(const b2_conv_args* a, ConvPlan* pl) {
  pl->kernel = KERN_NONE;
  memset(pl->tm_copy, -1, sizeof(pl->tm_copy));
  const Tuning& t = tuning();
  const int To = conv_out_dim(a->T, a->kt, a->st, a->pt), Ho = conv_out_dim(a->H, a->kh, a->sh, a->ph),
            Wo = conv_out_dim(a->W, a->kw, a->sw, a->pw);
  const int taps = a->kt * a->kh * a->kw;
  const bool extras = a->aff_ld || a->y2 || a->residual_up || a->residual_pre || a->in_scale;
  // a plain convolution: what the temporal stack / temporal-group kernels (and the dense-M kernel, fp32 output aside) implement
  const bool plain = a->mode == B2_CONV_AUTO && !a->out_f32 && !a->upsample && !extras;
  const bool dense_m = a->mode == B2_CONV_AUTO && !a->upsample && !extras &&
                       densem_wanted((long long)a->N * To * Ho * Wo, taps, a->st > 1 || a->sh > 1 || a->sw > 1);
  int rc;
  if (!dense_m && t.conv_algo == 0) {
    if (plain && ((rc = plan_tstack(a, pl)) != B2_OK || pl->kernel != KERN_NONE)) return rc;
    if (plain && ((rc = plan_slabts(a, pl)) != B2_OK || pl->kernel != KERN_NONE)) return rc;
    if ((rc = plan_slab(a, pl)) != B2_OK || pl->kernel != KERN_NONE) return rc;
  }
  if (a->upsample) return set_error(B2_ERR_UNSUPPORTED, "fused upsampling needs the slab kernel, which does not take this shape");

  IgemmLaunch L;
  memset(&L, 0, sizeof(L));
  IgemmParams& p = L.p;
  p.x = reinterpret_cast<const __half*>(a->x);
  p.N = a->N; p.T = a->T; p.H = a->H; p.W = a->W; p.C = a->C;
  p.To = To; p.Ho = Ho; p.Wo = Wo;
  p.kt = a->kt; p.kh = a->kh; p.kw = a->kw;
  p.st = a->st; p.sh = a->sh; p.sw = a->sw;
  p.pt = a->pt; p.ph = a->ph; p.pw = a->pw;
  const long long M = (long long)a->N * p.To * p.Ho * p.Wo;
  B2_CHECK_ARG(M < (1ll << 31), "output too large");
  p.M_total = (int)M;
  p.Ncols = a->K;
  p.scale = a->scale; p.shift = a->shift;
  p.residual = reinterpret_cast<const __half*>(a->residual);
  p.ldr = a->ldr;
  p.y = a->y; p.ldy = a->ldy;
  p.relu = a->relu; p.per_row = 0; p.accumulate = a->accumulate;
  p.epi = a->out_f32 ? EPI_DIRECT_F32 : EPI_TMA_F16;
  p.aff_ld = a->aff_ld;
  p.res_up = a->residual_up; p.res_pre = a->residual_pre; p.up_H = p.Ho; p.up_W = p.Wo;
  p.y2 = a->y2; p.scale2 = a->scale2; p.shift2 = a->shift2; p.aff2_ld = a->aff2_ld; p.aff2_rows = p.To * p.Ho * p.Wo;
  if (a->y2) {
    B2_CHECK_ARG(a->scale2 && a->shift2 && a->aff2_ld >= a->K && !a->out_f32 && taps == 1,
                 "second output needs scale2 / shift2 (fp32 [N][aff2_ld >= K]) and a 1x1 convolution with fp16 output");
    if (p.aff2_rows % 128 != 0)
      return set_error(B2_ERR_UNSUPPORTED, "second output with a per-sample affine needs To*Ho*Wo %% 128 == 0 (got %d)", p.aff2_rows);
  }
  if (a->in_scale) {
    B2_CHECK_ARG(a->in_shift && a->in_aff_ld >= a->C && (a->in_aff_ld & 3) == 0 && !a->out_f32 && taps == 1 && a->st == 1 &&
                     a->sh == 1 && a->sw == 1 && (reinterpret_cast<uintptr_t>(a->in_scale) & 15) == 0 &&
                     (reinterpret_cast<uintptr_t>(a->in_shift) & 15) == 0,
                 "input affine needs in_shift, a 16-byte aligned fp32 [N][in_aff_ld >= C] pair (pitch %% 4 == 0) and a 1x1 stride-1 convolution with fp16 output");
    if ((p.To * p.Ho * p.Wo) % 128 != 0 || a->C % 64 != 0)
      return set_error(B2_ERR_UNSUPPORTED, "input affine needs To*Ho*Wo %% 128 == 0 and a channel pitch that is a multiple of 64 (got %d, %d)",
                       p.To * p.Ho * p.Wo, a->C);
    p.in_scale = a->in_scale; p.in_shift = a->in_shift; p.in_ld = a->in_aff_ld; p.in_rows = p.To * p.Ho * p.Wo;
  }
  p.aff_rows = p.To * p.Ho * p.Wo;
  if (a->aff_ld && p.aff_rows % 128 != 0)
    return set_error(B2_ERR_UNSUPPORTED, "per-sample affine on a 1x1x1 convolution needs To*Ho*Wo %% 128 == 0 (got %d)", p.aff_rows);
  L.w = a->w;

  if (a->mode == B2_CONV_STEM7) {
    B2_CHECK_ARG(!a->out_f32 && a->residual == nullptr, "stem convolution has no residual / fp32 output");
    B2_CHECK_ARG(a->st == 1 && a->sh == 2, "stem convolution needs strides (1, 2, 2)");
    return plan_stem(a, a->K <= 64 ? 64 : 128, pl);
  } else if (taps == 1 && a->st == 1 && a->sh == 1 && a->sw == 1 && a->pt == 0 && a->ph == 0 && a->pw == 0) {
    // 1x1x1 stride-1: A is literally the [M][C] activation matrix -> TMA on both operands
    p.amode = AMODE_TMA;
    p.nkb = (a->C + kBK - 1) / kBK;
    L.a_mat = a->x; L.lda = a->C; L.a_cols = a->C;
    L.ldb = a->C; L.b_cols = a->C;
  } else {
    p.amode = AMODE_GATHER;
    p.cchunks = (a->C + kBK - 1) / kBK;
    p.nkb = taps * p.cchunks;
    L.ldb = taps * a->C;
    L.b_cols = L.ldb;
    // When C % 64 != 0 the last K block of a tap also covers the first columns of the next tap's
    // weights; the activation side zero-fills channels >= C, so those products vanish.
  }
  return plan_gemm_shaped(L, dense_m, pl);
}

static int plan_gemm(const b2_gemm_args* g, const void* a2, int lda2, const void* b2, int ldb2, int k2, ConvPlan* pl) {
  pl->kernel = KERN_NONE;
  memset(pl->tm_copy, -1, sizeof(pl->tm_copy));
  IgemmLaunch L;
  memset(&L, 0, sizeof(L));
  IgemmParams& p = L.p;
  p.amode = AMODE_TMA;
  p.M_total = g->M;
  p.Ncols = g->N;
  p.nkb = (g->Kd + kBK - 1) / kBK;
  p.scale = g->scale; p.shift = g->shift;
  p.residual = reinterpret_cast<const __half*>(g->residual);
  p.ldr = g->ldr;
  p.y = g->d; p.ldy = g->ldd;
  p.relu = g->relu; p.per_row = g->per_row; p.accumulate = g->accumulate;
  p.epi = g->out_f32 ? EPI_DIRECT_F32 : EPI_TMA_F16;
  B2_CHECK_ARG(g->aff_ld >= 0 && (g->aff_ld == 0 || (g->aff_ld >= g->N && g->aff_rows > 0 && g->aff_rows % 128 == 0 &&
                                                     !g->out_f32 && !g->per_row)),
               "bad per-sample affine (pitch %d, rows per sample %d)", g->aff_ld, g->aff_rows);
  p.aff_ld = g->aff_ld; p.aff_rows = g->aff_rows;
  if (g->d2) {
    B2_CHECK_ARG(g->scale2 && g->shift2 && g->aff2_ld >= g->N && g->aff2_rows > 0 && g->aff2_rows % 128 == 0 && !g->out_f32 && !g->per_row,
                 "second output needs scale2 / shift2 (fp32 [M / aff2_rows][aff2_ld >= N], aff2_rows %% 128 == 0) and fp16 output");
    p.y2 = g->d2; p.scale2 = g->scale2; p.shift2 = g->shift2; p.aff2_ld = g->aff2_ld; p.aff2_rows = g->aff2_rows;
  }
  p.x = reinterpret_cast<const __half*>(g->a);
  L.a_mat = g->a; L.lda = g->lda; L.a_cols = g->Kd;
  L.w = g->b; L.ldb = g->ldb; L.b_cols = g->Kd;
  L.a2 = a2; L.lda2 = lda2; L.w2 = b2; L.ldb2 = ldb2; L.k2 = k2;
  if (k2 > 0 && tuning().gemm_algo != 0) return set_error(B2_ERR_UNSUPPORTED, "two-operand GEMM needs the persistent kernel");
  const bool dense_m = k2 == 0 && !g->aff_ld && !g->d2 && (g->out_f32 || !g->per_row) && densem_wanted(g->M, 1, false);
  return plan_gemm_shaped(L, dense_m, pl);
}

static int launch_plan(const ConvPlan& pl, cudaStream_t stream) {
  CUtensorMap tm[kMaxTmaps];
  for (int i = 0; i < kNumTmaps[pl.kernel]; ++i)
    if (pl.tm_copy[i] < 0) B2_TRY(encode_tmap(&tm[i], pl.tm[i]));
  for (int i = 0; i < kNumTmaps[pl.kernel]; ++i)
    if (pl.tm_copy[i] >= 0) tm[i] = tm[pl.tm_copy[i]];
  const dim3 g = pl.grid, b = pl.block;
  const size_t smem = (size_t)pl.smem;
  cudaError_t e = cudaSuccess;
  // shared memory opt-in (once per kernel and device), then the launch with programmatic stream serialization
#define B2_RUN(kernel, optin, ...) B2_OPT_IN_SMEM(kernel, optin); e = launch_pdl(kernel, g, b, smem, stream, __VA_ARGS__); break
  switch (pl.kernel) {
    case KERN_TSTACK: B2_RUN(tstack_kernel, 227 * 1024, tm[0], tm[1], pl.p.tstack);
    case KERN_SLABTS: B2_RUN(slabts_kernel, 227 * 1024, tm[0], tm[1], pl.p.slab);
    case KERN_SLAB64: B2_RUN(slabconv_kernel<64>, 227 * 1024, tm[0], tm[1], pl.p.slab);
    case KERN_SLAB128: B2_RUN(slabconv_kernel<128>, 227 * 1024, tm[0], tm[1], pl.p.slab);
    case KERN_SLABN: B2_RUN(slabconv_kernel<0>, 227 * 1024, tm[0], tm[1], pl.p.slab);
    case KERN_STEM64: B2_RUN(stemconv_kernel<64>, 227 * 1024, tm[0], pl.p.stem);
    case KERN_STEM128: B2_RUN(stemconv_kernel<128>, 227 * 1024, tm[0], pl.p.stem);
    case KERN_PGEMM64: B2_RUN((pgemm_kernel<64, 0>), PgemmSmem<64>::kTotal, tm[0], tm[1], tm[2], tm[3], tm[4], tm[5], tm[6], pl.p.pgemm);
    case KERN_PGEMM64_GAN: B2_RUN((pgemm_kernel<64, 1>), PgemmSmem<64>::kTotal, tm[0], tm[1], tm[2], tm[3], tm[4], tm[5], tm[6], pl.p.pgemm);
    case KERN_PGEMM128: B2_RUN((pgemm_kernel<128, 0>), PgemmSmem<128>::kTotal, tm[0], tm[1], tm[2], tm[3], tm[4], tm[5], tm[6], pl.p.pgemm);
    case KERN_PGEMM128_GAN: B2_RUN((pgemm_kernel<128, 1>), PgemmSmem<128>::kTotal, tm[0], tm[1], tm[2], tm[3], tm[4], tm[5], tm[6], pl.p.pgemm);
    case KERN_IGEMM64: B2_RUN(igemm_kernel<64>, IgemmSmem<64>::kTotalBytes, tm[0], tm[1], tm[2], tm[3], pl.p.igemm);
    case KERN_IGEMM128: B2_RUN(igemm_kernel<128>, IgemmSmem<128>::kTotalBytes, tm[0], tm[1], tm[2], tm[3], pl.p.igemm);
    case KERN_DENSEM: {     // split-K over a thread-block cluster along z
      B2_OPT_IN_SMEM(densem_kernel, 227 * 1024);
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = g; cfg.blockDim = b; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
      cudaLaunchAttribute attr[2];
      attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
      attr[0].val.programmaticStreamSerializationAllowed = pdl_enabled() ? 1 : 0;
      attr[1].id = cudaLaunchAttributeClusterDimension;
      attr[1].val.clusterDim.x = 1; attr[1].val.clusterDim.y = 1; attr[1].val.clusterDim.z = pl.cluster;
      cfg.attrs = attr; cfg.numAttrs = 2;
      e = cudaLaunchKernelEx(&cfg, densem_kernel, tm[0], tm[1], pl.p.densem);
      break;
    }
    default: return set_error(B2_ERR_INVALID, "no kernel planned");
  }
#undef B2_RUN
  if (e != cudaSuccess) return set_error(B2_ERR_CUDA, "launch of %s failed: %s", kKernelName[pl.kernel], cudaGetErrorString(e));
  B2_CHECK_LAUNCH(kKernelName[pl.kernel]);
  return B2_OK;
}

// Host-only view of a plan for the b2_debug_*_plan entry points; fields the kernel does not have stay 0:
// {kernel, grid x, y, z, block, smem, cluster, bn, MT, R, PW, WC, wchunks, items, flex, remap, groups, tiles, cchunks, wbytes, S}
constexpr int kPlanFields = 21;
static int plan_view(const ConvPlan& pl, int kt_in, int* out, int n) {
  int v[kPlanFields] = {pl.kernel, (int)pl.grid.x, (int)pl.grid.y, (int)pl.grid.z, (int)pl.block.x, pl.smem, pl.cluster};
  if (pl.kernel >= KERN_SLABTS && pl.kernel <= KERN_SLABN) {
    const SlabParams& s = pl.p.slab;
    const int slab[] = {s.bn, s.MT, s.R, s.PW, s.WC, s.wchunks, s.items_total, pl.kernel == KERN_SLABN, s.kt != kt_in};
    memcpy(v + 7, slab, sizeof(slab));
    v[18] = s.cchunks;
  } else if (pl.kernel == KERN_TSTACK) {
    const TstackParams& s = pl.p.tstack;
    v[13] = s.items_total; v[16] = s.groups; v[17] = s.tiles_q; v[18] = s.cchunks; v[19] = s.cchunks * s.kt * kTkWBlock;
  } else if (pl.kernel == KERN_DENSEM) {
    v[7] = pl.p.densem.bn; v[20] = pl.p.densem.ksplit;
  }
  for (int i = 0; i < n; ++i) out[i] = i < kPlanFields ? v[i] : 0;
  return B2_OK;
}

static int g_last_conv_kernel = KERN_NONE;   // kernel of the last b2_conv_ndhwc_fprop launch (tests pin the dispatch)

}  // namespace b2

using namespace b2;

static int validate_conv(const b2_conv_args* a) {
  B2_CHECK_ARG(a != nullptr, "null args");
  B2_CHECK_ARG(a->x && a->w && a->scale && a->shift && a->y, "null tensor pointer");
  B2_CHECK_ARG(a->N > 0 && a->T > 0 && a->H > 0 && a->W > 0 && a->C > 0 && a->K > 0, "non-positive dimension");
  B2_CHECK_ARG(a->kt > 0 && a->kh > 0 && a->kw > 0 && a->st > 0 && a->sh > 0 && a->sw > 0, "bad kernel/stride");
  B2_CHECK_ARG(a->pt >= 0 && a->ph >= 0 && a->pw >= 0, "negative padding");
  B2_CHECK_ARG(a->ldy >= a->K, "ldy < K");
  B2_CHECK_ARG(a->residual == nullptr || a->ldr >= a->K, "ldr < K");
  B2_CHECK_ARG(conv_out_dim(a->T, a->kt, a->st, a->pt) > 0 && conv_out_dim(a->H, a->kh, a->sh, a->ph) > 0 &&
                   conv_out_dim(a->W, a->kw, a->sw, a->pw) > 0,
               "empty output");
  B2_CHECK_ARG(!a->pool_w || a->mode == B2_CONV_STEM7, "pool_w is implemented by the stem convolution only");
  if (a->mode == B2_CONV_STEM7) {
    B2_CHECK_ARG(a->C == 4, "STEM7 needs NDHWC4 input (C == 4), got %d", a->C);
    B2_CHECK_ARG(a->kw == 7 && a->sw == 2 && a->pw == 3, "STEM7 needs kw=7, sw=2, pw=3");
    B2_CHECK_ARG(a->W % 2 == 0, "STEM7 needs an even input width, got %d", a->W);
  } else {
    B2_CHECK_ARG(a->mode == B2_CONV_AUTO, "unknown conv mode %d", a->mode);
    B2_CHECK_ARG(a->C % 8 == 0, "channel pitch %d is not a multiple of 8", a->C);
  }
  if (a->residual_up || a->residual_pre) {
    B2_CHECK_ARG(a->residual != nullptr && a->kt * a->kh * a->kw == 1 && a->st == 1 && a->sh == 1 && a->sw == 1 && a->T == 1 &&
                     !a->out_f32 && a->mode == B2_CONV_AUTO,
                 "residual_up / residual_pre need a residual and a 1x1 stride-1 2-D convolution with fp16 output");
    B2_CHECK_ARG(!a->residual_up || (a->H % 2 == 0 && a->W % 2 == 0), "residual_up needs even output height and width");
  }
  if (a->upsample)
    B2_CHECK_ARG(a->upsample == 1 && a->mode == B2_CONV_AUTO && !a->out_f32 && a->kt == 1 && a->kh == 3 && a->kw == 3 && a->st == 1 &&
                     a->sh == 1 && a->sw == 1 && a->pt == 0 && a->ph == 1 && a->pw == 1,
                 "fused upsampling is implemented for 1x3x3 stride-1 'same' convolutions with fp16 output only");
  B2_CHECK_ARG(a->aff_ld >= 0 && (a->aff_ld == 0 || (a->aff_ld >= a->K && !a->out_f32 && a->mode == B2_CONV_AUTO)),
               "bad per-sample affine pitch %d", a->aff_ld);
  if (!a->out_f32) {
    B2_CHECK_ARG(a->ldy % 8 == 0, "ldy %d is not a multiple of 8", a->ldy);
    B2_CHECK_ARG(a->residual == nullptr || a->ldr % 8 == 0, "ldr %d is not a multiple of 8", a->ldr);
    B2_CHECK_ARG(!a->accumulate, "accumulate requires out_f32");
  }
  return B2_OK;
}

static int validate_gemm(const b2_gemm_args* g, bool pair, const void* a2, int lda2, const void* b2, int ldb2, int k2) {
  if (pair) {        // b2_gemm2_f16
    B2_CHECK_ARG(g != nullptr && a2 && b2 && k2 > 0, "null / empty second operand pair");
    B2_CHECK_ARG(lda2 % 8 == 0 && ldb2 % 8 == 0 && lda2 >= k2 && ldb2 >= k2, "bad second operand pitch");
    B2_CHECK_ARG(!g->out_f32 && !g->per_row, "the fused two-operand GEMM produces fp16 output with per-column affine");
  }
  B2_CHECK_ARG(g != nullptr, "null args");
  B2_CHECK_ARG(g->a && g->b && g->scale && g->shift && g->d, "null tensor pointer");
  B2_CHECK_ARG(g->M > 0 && g->N > 0 && g->Kd > 0, "non-positive dimension");
  B2_CHECK_ARG(g->lda % 8 == 0 && g->ldb % 8 == 0 && g->lda >= g->Kd && g->ldb >= g->Kd, "bad operand pitch");
  B2_CHECK_ARG(g->ldd >= g->N, "ldd < N");
  if (!g->out_f32) {
    B2_CHECK_ARG(g->ldd % 8 == 0, "ldd not a multiple of 8");
    B2_CHECK_ARG(!g->accumulate, "accumulate requires out_f32");
    B2_CHECK_ARG(g->residual == nullptr || (g->ldr % 8 == 0 && g->ldr >= g->N), "bad residual pitch");
  }
  return B2_OK;
}

static int run_gemm(bool pair, const b2_gemm_args* g, const void* a2, int lda2, const void* b2, int ldb2, int k2, void* stream) {
  ConvPlan pl;
  B2_TRY(validate_gemm(g, pair, a2, lda2, b2, ldb2, k2));
  B2_TRY(require_sm100());
  B2_TRY(plan_gemm(g, a2, lda2, b2, ldb2, k2, &pl));
  return launch_plan(pl, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" {

int b2_version(void) { return 103; }   // 103: split-K / fused (2+1)D / pooled-stem entry points (round 2); 102: generator fields

int b2_conv_ndhwc_fprop(const b2_conv_args* a, void* stream) {
  ConvPlan pl;
  g_last_conv_kernel = KERN_NONE;
  B2_TRY(validate_conv(a));
  B2_TRY(require_sm100());
  B2_TRY(plan_conv(a, &pl));
  B2_TRY(launch_plan(pl, reinterpret_cast<cudaStream_t>(stream)));
  g_last_conv_kernel = pl.kernel;
  return B2_OK;
}

int b2_gemm_f16(const b2_gemm_args* g, void* stream) { return run_gemm(false, g, nullptr, 0, nullptr, 0, 0, stream); }

int b2_gemm2_f16(const b2_gemm_args* g, const void* a2, int lda2, const void* b2, int ldb2, int k2, void* stream) {
  return run_gemm(true, g, a2, lda2, b2, ldb2, k2, stream);
}

/* Debug entry points (not in the public header).  The *_plan probes validate and plan a call exactly as the entry point would,
   without a launch or a device: out[0 .. n) = the plan_view fields (kernel id as in enum ConvKernel, grid, block, dynamic shared
   memory, cluster size, then the kernel's tiling).  Without a device sm_count() is 148, the B200's, so these are B200 plans. */
int b2_debug_conv_plan(const b2_conv_args* a, int* out, int n) {
  ConvPlan pl;
  B2_TRY(validate_conv(a));
  B2_TRY(plan_conv(a, &pl));
  return plan_view(pl, a->kt, out, n);
}
/* k2 > 0: the two-operand GEMM of b2_gemm2_f16, with the second pair at the first pair's addresses and pitch round_up(k2, 8) */
int b2_debug_gemm_plan(const b2_gemm_args* g, int k2, int* out, int n) {
  ConvPlan pl;
  const int ld2 = (k2 + 7) / 8 * 8;
  const void* a2 = k2 > 0 && g ? g->a : nullptr;
  const void* b2 = k2 > 0 && g ? g->b : nullptr;
  B2_TRY(validate_gemm(g, k2 > 0, a2, ld2, b2, ld2, k2));
  B2_TRY(plan_gemm(g, a2, ld2, b2, ld2, k2, &pl));
  return plan_view(pl, 1, out, n);
}
int b2_debug_last_conv_kernel(void) { return g_last_conv_kernel; }
int b2_debug_last_conv_path(void) { return g_last_conv_kernel == KERN_TSTACK; }   /* 1: the temporal stack kernel took it */
/* 0 = auto, 1 = no slab / temporal-group / temporal stack kernels */
int b2_debug_set_conv_algo(int algo) {
  if (algo != 0 && algo != 1) return set_error(B2_ERR_INVALID, "conv algo %d: 0 (auto) or 1 (gather)", algo);
  tuning().conv_algo = algo;
  return B2_OK;
}
int b2_debug_set_gemm_algo(int algo) { tuning().gemm_algo = algo; return B2_OK; }
int b2_debug_set_slab_wide(int on) { tuning().slab_wide = on; return B2_OK; }   /* -1 rule, 0 never, 1 always */
int b2_debug_set_tstack(int mode) { tuning().tstack = mode < -1 ? -1 : (mode > 1 ? 1 : mode); return B2_OK; }   /* -1 rule, 0 never, 1 whenever eligible */
int b2_debug_set_slab_mt(int mt) { tuning().slab_mt = mt < 0 ? 0 : mt; return B2_OK; }
/* small-M path: layers with M <= maxm take the dense-M kernel (0 = never, < 0 = the rule); force_s > 0 caps the cluster size */
int b2_debug_set_densem(int maxm, int force_s) { tuning().densem_maxm = maxm < 0 ? -1 : maxm; tuning().densem_s = force_s; return B2_OK; }

}  // extern "C"
