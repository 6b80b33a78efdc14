/* b2_pretorched.h -- C ABI of the B200-native forward engine for pretorched-x's video-ConvNet hot path.
 *
 * The reference (alexandonian/pretorched-x @ 36a5754) has no FFI layer of its own: every FLOP of
 * its hot path is a torch.nn call inside a Python `forward` body.  Each entry point below therefore
 * cites the reference *operator call site(s)* it replaces (file:line under /root/reference).  The
 * Python host side (pretorched_x_b200/) binds these with ctypes; INTEGRATION.md shows the stub a
 * reference maintainer would add.
 *
 * Conventions
 *   - All data pointers are DEVICE pointers owned by the caller.  The library never allocates, frees
 *     or retains them; work is enqueued on `stream` (a cudaStream_t passed as void*) and the call
 *     returns immediately.  Safe under CUDA-graph capture (no syncs, no allocations).
 *   - Activations are fp16 NDHWC ("channels last"), i.e. a dense matrix [N*T*H*W][ld] with channel
 *     pitch `ld` (elements) a multiple of 8.  Channels in [C, ld) must be zero.
 *   - Returns 0 on success, a negative B2_ERR_* code otherwise; b2_last_error() returns a
 *     thread-local message.  No C++ exception crosses the ABI.
 *   - There is NO CPU fallback: on a machine without an sm_100 GPU every compute call fails with
 *     B2_ERR_CUDA / B2_ERR_UNSUPPORTED.
 */
#ifndef B2_PRETORCHED_H_
#define B2_PRETORCHED_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2_OK 0
#define B2_ERR_INVALID (-1)     /* bad argument (shape, alignment, null pointer) */
#define B2_ERR_CUDA (-2)        /* a CUDA runtime / driver call failed */
#define B2_ERR_UNSUPPORTED (-3) /* valid request the engine does not implement */

#define B2_CONV_AUTO 0  /* generic implicit GEMM: x has channel pitch C (multiple of 8)            */
#define B2_CONV_STEM7 1 /* kw == 7, strides (1,2,2), pw == 3, Cin <= 4 stored as NDHWC4 (stem convs)  */

int b2_version(void);
const char* b2_last_error(void);
/* number of kernels this library has launched from the calling process so far (bench bookkeeping) */
uint64_t b2_launch_count(void);

/* ---------------------------------------------------------------------------------------------
 * Convolution as implicit GEMM on tcgen05 tensor cores, with the eval-mode BatchNorm affine
 * (scale/shift), the residual add and the ReLU fused into the epilogue:
 *     y[m, k] = act( scale[k] * sum_{tap,c} x[m @ tap, c] * w[k, tap, c] + shift[k] + residual[m, k] )
 * Replaces nn.Conv3d -> nn.BatchNorm3d -> (+=residual) -> nn.ReLU chains at
 *   resnet3D.py:91-106 (BasicBlock.forward), resnet3D.py:125-143 (Bottleneck.forward),
 *   resnet3D.py:176-185 (type-B shortcut), r2plus1d.py:85-88 (SpatioTemporalConv.forward),
 *   nonlocalnet.py:143-166 (theta/phi/g/W 1x1x1 convs), torchvision_models.py:448-452 (stem).
 * ------------------------------------------------------------------------------------------- */
typedef struct b2_conv_args {
  const void* x;        /* fp16 [N,T,H,W,C]; C is the channel pitch                               */
  const void* w;        /* fp16 packed [K][taps][C] (b2_pack_conv_weight), taps = kt*kh*kw        */
  const float* scale;   /* fp32 [K]                                                                */
  const float* shift;   /* fp32 [K]                                                                */
  const void* residual; /* nullable; fp16 [M][ldr], M = N*To*Ho*Wo                                 */
  void* y;              /* fp16 [M][ldy]  (fp32 when out_f32)                                      */
  int32_t N, T, H, W, C;
  int32_t K;            /* logical output channels; columns [K, ldy) of y are written as zero      */
  int32_t ldy, ldr;
  int32_t kt, kh, kw;
  int32_t st, sh, sw;
  int32_t pt, ph, pw;
  int32_t relu;
  int32_t out_f32;      /* y is fp32 (direct-store epilogue)                                       */
  int32_t accumulate;   /* out_f32 only: y += result                                               */
  int32_t mode;         /* B2_CONV_AUTO | B2_CONV_STEM7                                            */
  int32_t aff_ld;       /* 0: scale/shift are [K].  > 0: per-SAMPLE affine, scale/shift are fp32 [N][aff_ld], 16-byte aligned,
                           aff_ld % 4 == 0
                           (class-conditional BatchNorm of the layer that FOLLOWS this convolution, BigGAN GBlock);
                           multi-tap "same" convolutions and 1x1x1 convolutions with To*Ho*Wo % 128 == 0 only      */
  int32_t upsample;     /* 1: y = conv3x3(nearest_upsample_2x(x)) without materialising the upsampled image (GBlock conv2):
                           x is the LOW-resolution input [N,1,H,W,C], y has (2H) x (2W) pixels per image, and w is the
                           phase-folded filter bank [K][16][C] written by b2_pack_upconv3x3_weight.  kt=1, kh=kw=3,
                           strides 1, padding (0,1,1) only                                                        */
  int32_t residual_up;  /* 1: `residual` is the LOW-resolution tensor [N][H/2][W/2][ldr] of the skip path and is nearest-2x
                           upsampled on the fly (GBlock: h + upsample(x[:, :out]); the channel drop is the pitch ldr).
                           1x1 stride-1 2-D convolutions only                                                     */
  int32_t residual_pre; /* 1: y = act(scale * (acc + residual) + shift) -- the residual joins BEFORE the affine (BatchNorm of
                           the block output folded into its closing convolution).  1x1 convolutions only           */
  void* y2;             /* nullable second output, fp16 [M][ldy]: y2 = relu(y * scale2[n] + shift2[n]) with y the fp32 value of
                           the first output -- the class-conditional BatchNorm + ReLU that OPENS the next GBlock, produced
                           while the tile is still on chip.  1x1 stride-1 convolutions with To*Ho*Wo % 128 == 0 only */
  const float* scale2;  /* fp32 [N][aff2_ld] */
  const float* shift2;
  int32_t aff2_ld;
  int32_t pool_w;       /* B2_CONV_STEM7 only, needs relu: the MaxPool (k = 3, stride 2, padding 1 ALONG W) that follows the stem
                           (resnet3D.py:156, torchvision_models.py:452) is applied in the epilogue.  y then has
                           Wp = (Wo - 1) / 2 + 1 columns per output row ([N*To*Ho*Wp][ldy]); the H / T directions of the pool
                           are a second b2_maxpool3d_ndhwc call with kernel (kt, kh, 1) -- max-pooling is separable -- over a
                           tensor half the size.  Output rows of at most 120 columns                                   */
  const float* in_scale; /* nullable.  Per-SAMPLE affine + ReLU applied to the INPUT of a 1x1 stride-1 convolution on its way to the
                            tensor core: the convolution sees relu(x * in_scale[n][c] + in_shift[n][c]) -- the class-conditional
                            BatchNorm + ReLU that opens a GBlock, without a stand-alone pass over x (x itself stays untouched in
                            memory: the block's skip path reads it raw).  fp32 [N][in_aff_ld], 16-byte aligned, in_aff_ld % 4 == 0,
                            To*Ho*Wo % 128 == 0                                                                           */
  const float* in_shift;
  int32_t in_aff_ld;
} b2_conv_args;

int b2_conv_ndhwc_fprop(const b2_conv_args* a, void* stream);
/* Same contract on plain CUDA cores (one thread per output element, fp32 accumulate).  A debugging
 * cross-check for the tensor-core path; never used by the model forward. */
int b2_conv_ndhwc_fprop_simt(const b2_conv_args* a, void* stream);

/* fp32 [K][Cin][kt][kh][kw] (nn.Conv3d.weight layout, resnet3D.py:60,115-119) -> fp16 packed
 * [K][taps][C] with zero padding of channels [Cin, C).  mode B2_CONV_STEM7: a pre-laid-out shared-memory image
 * [ntile][kt][kh taps, even dh descending then odd dh descending][BN x 32] (see csrc/b2_stemconv.cuh). */
size_t b2_pack_conv_weight_elems(int K, int Cin, int kt, int kh, int kw, int C, int mode);
int b2_pack_conv_weight(const float* w_oidhw, void* w_packed, int K, int Cin, int kt, int kh, int kw, int C,
                        int mode, void* stream);

/* fp32 [K][Cin][3][3] (nn.Conv2d.weight) -> fp16 [K][16][C]: the four 2x2 filters that a 3x3 convolution of a nearest-2x
 * upsampled image collapses to, one per output phase ph = 2*py + px, tap index ph*4 + 2*a + b.  Output pixel (2h+py, 2w+px)
 * reads low-res rows h-1+py+a, columns w-1+px+b (a, b in {0,1}); the folded weight is the sum of the 3x3 taps that land on
 * that low-res pixel (rows: py=0 -> {0},{1,2}; py=1 -> {0,1},{2}).  2.25x fewer MACs, input read at 1/4 of the size. */
int b2_pack_upconv3x3_weight(const float* w_oihw, void* w_packed, int K, int Cin, int C, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Dense layer / 1x1x1 convolution as a plain GEMM:  D[M][N] = act(scale * (A[M][Kd] . B[N][Kd]^T) + shift
 * + residual).  scale/shift index the N dimension, or the M dimension when per_row != 0 (swap-AB use:
 * D^T = B . A^T with the affine following the rows).  Replaces nn.Linear at
 * resnet3D.py:162 / torchvision_models.py:460-464 (head), trn.py:39-49 (Relation MLP).
 * ------------------------------------------------------------------------------------------- */
typedef struct b2_gemm_args {
  const void* a; /* fp16 [M][lda] */
  const void* b; /* fp16 [N][ldb] */
  const float* scale;
  const float* shift;
  const void* residual; /* nullable fp16 [M][ldr] */
  void* d;              /* fp16 [M][ldd] or fp32 when out_f32 */
  int32_t M, N, Kd;
  int32_t lda, ldb, ldd, ldr;
  int32_t per_row;
  int32_t relu;
  int32_t out_f32;
  int32_t accumulate;
  int32_t aff_ld;   /* 0: scale/shift are [N] (or [M] when per_row).  > 0: per-sample affine, fp32 [M / aff_rows][aff_ld]:
                       row m uses scale[(m / aff_rows) * aff_ld + n]; fp16 output only, aff_rows % 128 == 0 */
  int32_t aff_rows;
  void* d2;             /* nullable second output fp16 [M][ldd]: d2 = relu(d * scale2[m / aff2_rows] + shift2[...]) (see y2 above) */
  const float* scale2;
  const float* shift2;
  int32_t aff2_ld, aff2_rows;
} b2_gemm_args;
int b2_gemm_f16(const b2_gemm_args* a, void* stream);
/* D = act(scale * (A.B^T + A2.B2^T) + shift + residual): both products accumulate in the same TMEM tile.  Used to
 * fuse the type-B shortcut projection (resnet3D.py:176-185) into the block-closing 1x1x1 convolution
 * (resnet3D.py:136-143) with the two BatchNorm scales folded into B and B2: the shortcut never touches HBM.
 * fp16 output, per-column affine only. */
int b2_gemm2_f16(const b2_gemm_args* a, const void* a2, int lda2, const void* b2, int ldb2, int k2, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Non-local block core (nonlocalnet.py:143-211):
 *     mode 0:  O[b] = softmax_rows(Q[b] . K[b]^T) . V[b]   (`_embedded_gaussian` :143-166, `_gaussian` :168-190;
 *                                                          unscaled logits, softmax over keys)
 *     mode 1:  O[b] = (Q[b] . K[b]^T / Nk) . V[b]          (`_dot_product` :192-211)
 *     mode 2:  O[b] = (relu(Q[b] . K[b]^T) / Nk) . V[b]    (`_concatenation` :213-243: concat_project's 1x1 conv over
 *                                                          [theta_i ; phi_j] is a_i + b_j, which the caller encodes as the
 *                                                          rank-2 product Q_i = [a_i, 1, 0..], K_j = [1, b_j, 0..])
 * Q: fp16 [B*Nq][ldq] (d columns used); K, V: fp16 [B*Nk][ld] (d resp. dv columns; Nk < Nq when phi and g were
 * max-pooled, `sub_sample=True` :126-131); O: fp16 [B*Nq][ldo].  One fused kernel, the Nq x Nk matrix is never
 * materialised.
 * ------------------------------------------------------------------------------------------- */
int b2_nonlocal_attention(const void* q, int ldq, const void* k, int ldk, const void* v, int ldv, void* o,
                          int ldo, int B, int Nq, int Nk, int d, int dv, int mode, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Pooling / layout / elementwise helpers (all HBM-bound, 128-bit accesses)
 * ------------------------------------------------------------------------------------------- */
/* nn.MaxPool3d (resnet3D.py:156): padding taps are skipped (== -inf padding). */
int b2_maxpool3d_ndhwc(const void* x, void* y, int N, int T, int H, int W, int C, int kt, int kh, int kw,
                       int st, int sh, int sw, int pt, int ph, int pw, void* stream);
/* nn.AdaptiveAvgPool3d(1) (resnet3D.py:161): x fp16 [N][S][C] -> y fp16 [N][C], fp32 accumulation. */
int b2_avgpool_global_ndhwc(const void* x, void* y, int N, int S, int C, void* stream);
/* fp32 NCDHW (the reference's input layout) -> fp16 NDHWC with channel pitch Cp (zero padded). */
int b2_ncdhw_f32_to_ndhwc_f16(const float* x, void* y, int N, int C, int T, int H, int W, int Cp, void* stream);
/* Same for callers that already hold fp16 clips (halves the host->device traffic of the input). */
int b2_ncdhw_f16_to_ndhwc_f16(const void* x, void* y, int N, int C, int T, int H, int W, int Cp, void* stream);
/* fp16 NDHWC (pitch Cp) -> fp32 NCDHW, for `features()` callers that want the reference layout. */
int b2_ndhwc_f16_to_ncdhw_f32(const void* x, float* y, int N, int C, int T, int H, int W, int Cp, void* stream);
/* y[r][c] = (relu ? max(x,0) : x) as fp16, rows x cols with pitches ldx / ldy; columns [cols, ldy) zeroed.
 * Used for the leading nn.ReLU of the TRN relation MLP (trn.py:40-41). */
int b2_cast_f32_to_f16(const float* x, int ldx, void* y, int ldy, int rows, int cols, int relu, void* stream);
/* Parameter-free type-A shortcut (resnet3D.py:65-74, nonlocalnet.py:322-332): spatial/temporal
 * subsampling by `stride` and zero-padding of channels [C, Cout). */
int b2_shortcut_a_ndhwc(const void* x, void* y, int N, int T, int H, int W, int C, int stride, int Cout,
                        void* stream);
/* y[r] = [a[r][0:Ca] | b[r][0:Cb] | 0]: torch.cat(dim=1) of two channels-last activations (SlowFast lateral
 * connections, slowfast.py:143-150, and its two-pathway head, slowfast.py:392).  Ca, Cb multiples of 8. */
int b2_concat_channels(const void* a, int lda, int Ca, const void* b, int ldb, int Cb, void* y, int ldy, long long rows,
                       void* stream);
/* y[n][j*F + f] = x[n][idx[j]][f]: frame-tuple gather of MultiScaleRelation (trn.py:108), fp16. */
int b2_gather_frames(const void* x, void* y, const int32_t* idx_dev, int N, int T, int F, int n_idx,
                     void* stream);
/* All tuples of one scale at once: y[n * n_tuples + t][j*F + f] = x[n][idx[t][j]][f], idx_dev int32 [n_tuples][n_idx] on the
 * device (one table for the whole forward, filled by a single host->device copy: trn.py:100-110 without a copy per tuple). */
int b2_gather_frame_tuples(const void* x, void* y, const int32_t* idx_dev, int N, int T, int F, int n_idx, int n_tuples,
                           void* stream);

/* ---------------------------------------------------------------------------------------------
 * Image preprocessing on the device -- TransformImage (pretorched/transforms/utils.py:34-81; used by
 * examples/imagenet_logits.py:38-43): transforms.Resize (Pillow 8-bit BILINEAR: horizontal pass then vertical pass,
 * 22-bit fixed-point coefficients, each pass rounds to uint8) -> Center/RandomCrop -> flips -> ToTensor -> ToSpaceBGR ->
 * ToRange255 -> Normalize, bit-exact with the Pillow + torchvision pipeline the reference composes.
 *   img       uint8 [H][W][3] RGB on the device
 *   hbounds/hk  int32 [Wr][2] (first source column, count) and [Wr][hksize] coefficients of the horizontal pass (null when Wr == W)
 *   vbounds/vk  the same for the vertical pass to Hr rows (null when Hr == H);  tmp: uint8 [H][Wr][3] scratch (horizontal result)
 *   top/left/crop_h/crop_w  crop window inside the resized [Hr][Wr] image
 *   flags     bit 0 horizontal flip, bit 1 vertical flip, bit 2 BGR, bit 3 range 255
 *   mean/stdv HOST pointers to 3 floats each
 *   out_f32   nullable fp32 [3][crop_h][crop_w] (what the reference returns); out_h4: nullable fp16 [crop_h*crop_w][4]
 *             (NDHWC4: the stem convolution's input layout, channel 3 zero)
 * ------------------------------------------------------------------------------------------- */
/* Decoded video frames, uint8 [N*T*H*W][3] (channels last, RGB) -> the stem's fp16 NDHWC4 input with ToTensor (/255), ToSpaceBGR,
 * ToRange255 and Normalize applied per pixel (the per-frame tail of TransformImage, transforms/utils.py:72-75, for clips that are
 * already at network resolution): a clip crosses PCIe as 3 bytes per pixel instead of 12.  flags: bit 2 BGR, bit 3 range 255;
 * mean / stdv: HOST pointers to 3 floats. */
int b2_u8_frames_to_ndhwc4_f16(const uint8_t* frames, void* y, long long pixels, int flags, const float* mean, const float* stdv,
                               void* stream);
int b2_transform_image_u8(const uint8_t* img, int H, int W, const int32_t* hbounds, const int32_t* hk, int hksize, int Wr,
                          const int32_t* vbounds, const int32_t* vk, int vksize, int Hr, uint8_t* tmp, int top, int left,
                          int crop_h, int crop_w, int flags, const float* mean, const float* stdv, float* out_f32,
                          void* out_h4, void* stream);

/* ---------------------------------------------------------------------------------------------
 * BigGAN-deep generator helpers (BASELINE.json configs[4]).  The architecture is NOT in the reference tree
 * (SURVEY.md section 8a row a14): these replace the F.batch_norm * (1 + gain(y)) + bias(y) -> ReLU ->
 * F.interpolate(scale_factor=2) chain of the published GBlock, its embedding lookup + torch.cat, and the final
 * torch.tanh; see oracle/biggan.py for the restatement they are checked against.
 * ------------------------------------------------------------------------------------------- */
/* v[b] = [ (embedded ? embedded[b] : table[labels[b]]) (ds) | z[b] (dz) | 0 ], D = round_up(ds + dz, 8) entries.
 * split == 0: y[b] = fp16(v), pitch ldy >= D.  split != 0: y[b] = [ hi | lo | hi ] (hi = fp16(v), lo = fp16(v - hi)),
 * pitch ldy >= 3 * D -- the A operand of an fp16 GEMM against [ W_hi | W_hi | W_lo ] that reproduces v . W to ~fp32
 * accuracy.  z, table, embedded fp32; labels int64 (clamped to [0, n_classes)). */
int b2_embed_concat(const float* z, const long long* labels, const float* table, const float* embedded, void* y, int B,
                    int dz, int ds, int n_classes, int ldy, int split, void* stream);
/* y[n, up*h+i, up*w+j, c] = act(x[n,h,w,c] * scale[n*lda + c] + shift[n*lda + c]) for c < C, i,j < up (up = 1 or 2,
 * nearest-neighbour upsampling); channels [C, ldy) written as zero.  scale/shift fp32 [N][lda] (lda = 0: one row shared
 * by all samples, i.e. a plain BatchNorm), or both NULL for a pure copy / channel slice / upsample. */
int b2_ccbn_act_ndhwc(const void* x, int ldx, void* y, int ldy, const float* scale, const float* shift, int lda, int N,
                      int H, int W, int C, int up, int relu, void* stream);
/* RGB head of the generator (3x3 convolution to K <= 4 channels, + bias, tanh, NCHW write) split in two: a 1x1 GEMM
 * (b2_gemm_f16) writes partial[q][(dh*3+dw)*4 + k] = sum_c x[q][c] * w[k][c][dh][dw] for every pixel q (36 columns, pitch
 * ldp >= 36), and this call gathers y[n][k][h][w] = tanh(bias[k] + sum_taps partial[(n,h+dh-1,w+dw-1)][tap*4 + k]) with
 * zero padding.  One pass of the tensor core over x instead of nine shifted passes that use 3 of 16 MMA columns. */
int b2_rgb_head_gather_tanh(const void* partial, int ldp, const float* bias, void* y, int N, int H, int W, int K, int out_f32,
                            void* stream);
/* y[n][c][s] = tanh(x[n*S + s][c]): fp16 channels-last (pitch ldx) -> NCHW planes, fp32 (out_f32) or fp16. */
int b2_tanh_nhwc_to_nchw(const void* x, int ldx, void* y, int N, int C, long long S, int out_f32, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Backward of the residual blocks with frozen BatchNorm statistics (fine-tuning of the last stages, b2_train.cu).
 * ------------------------------------------------------------------------------------------- */
/* gz[r][c] = (y[r][c] > 0) ? g[r][c] : 0 over M rows of pitch ldy (g: pitch ldg >= ldy), fp16; sum[c] = sum_r gz[r][c] in
 * fp32 for c < ldy.  partial: fp32 scratch of b2_relu_grad_sum_partials(M, ldy) * ldy floats.  The sums are reduced in a
 * fixed order (per-block partials, then the blocks in order): two calls give bit-identical results.  ldy <= 2048. */
int b2_relu_grad_sum_partials(long long M, int ld);
int b2_relu_grad_sum(const void* y, int ldy, const void* g, int ldg, void* gz, long long M, float* partial, float* sum,
                     void* stream);
/* y [N][T][H][W][ld] = g at the positions (s*to, s*ho, s*wo) and zero elsewhere; g has the stride-s output geometry
 * (floor((T - 1) / s) + 1, ...) and pitch ld.  The data gradient of a stride-s, k = 2p + 1 convolution is the stride-1
 * convolution of y with the flipped, transposed filter. */
int b2_zero_dilate_scatter(const void* g, void* y, int N, int T, int H, int W, int ld, int stride, void* stream);
/* y[n, s*to, s*ho, s*wo, c] += g[n, to, ho, wo, c] for c < C (fp32 add, fp16 store): the data gradient of a stride-s
 * subsampling (the type-A shortcut, the strided 1x1x1 projection).  y: [N][T][H][W] pitch ldy; g: the subsampled
 * geometry, pitch ldg. */
int b2_strided_scatter_add(const void* g, int ldg, void* y, int ldy, int N, int T, int H, int W, int C, int stride, void* stream);
/* Weight gradient of a convolution as an implicit GEMM on tcgen05, read straight from the two activation matrices:
 *     dw[k][tap][c] = sum over output positions p of g[p][k] * x[p * stride + tap - pad][c]   (fp32, [K][taps][C])
 * x: fp16 NDHWC [N][T][H][W], pitch ldx; g: fp16 rows of the output geometry, pitch ldg; C a multiple of 64; sh == sw.
 * When the plan splits the positions, `work` must hold b2_wgrad_workspace_floats() floats; the splits are summed in a
 * fixed order, so two calls give bit-identical results. */
typedef struct b2_wgrad_args {
  const void* x;
  const void* g;
  float* dw;
  float* work;
  int32_t N, T, H, W, ldx, C, ldg, K;
  int32_t kt, kh, kw, st, sh, sw, pt, ph, pw;
} b2_wgrad_args;
size_t b2_wgrad_workspace_floats(const b2_wgrad_args* a);
int b2_conv_ndhwc_wgrad(const b2_wgrad_args* a, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B2_PRETORCHED_H_ */
