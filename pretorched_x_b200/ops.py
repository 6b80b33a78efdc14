"""Host-side operator layer: torch tensors in, C-ABI calls out.

Activations travel between kernels as :class:`Act` -- an fp16 NDHWC matrix ``[N*T*H*W, ld]`` plus its
logical dims -- so that every convolution is an (implicit) GEMM over dense rows and every epilogue
writes full 128-byte lines.  The functions here mirror, one for one, the torch.nn calls on the
reference's hot path (file:line given per function); the arithmetic happens in
``csrc/*.cu`` behind ``include/b2_pretorched.h``.  There is no CPU implementation.
"""
import ctypes
import functools

import torch

from . import _lib
from ._lib import ConvArgs, GemmArgs, B2_CONV_AUTO, B2_CONV_STEM7


def _round_up(v, m):
    return (v + m - 1) // m * m


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def _first_cuda_device(args, kwargs):
    for v in list(args) + list(kwargs.values()):
        t = getattr(v, "data", None) if isinstance(v, Act) else v
        if isinstance(t, torch.Tensor) and t.is_cuda:
            return t.device
    return None


def _on_device(fn):
    """Run an operator with the device of its first CUDA tensor current (like torch's own device guard): the kernels launch on
    ``torch.cuda.current_stream()`` of the CURRENT device, so a model moved to ``cuda:1`` in a process whose current device is 0
    (``model.to('cuda:1')``, ``nn.DataParallel`` replicas call this from their own threads) must switch for the launch."""
    @functools.wraps(fn)
    def guarded(*args, **kwargs):
        dev = _first_cuda_device(args, kwargs)
        if dev is None or dev.index == torch.cuda.current_device():
            return fn(*args, **kwargs)
        with torch.cuda.device(dev):
            return fn(*args, **kwargs)
    return guarded


def _require_cuda(t, what):
    if not t.is_cuda:
        raise RuntimeError("%s must live on a CUDA (sm_100a) device: this engine has no CPU path" % what)


# ---------------------------------------------------------------------------------------------
# optional per-launch profiling (bench.py / tools): CUDA events on the launching stream + algorithmic work
# ---------------------------------------------------------------------------------------------
_PROFILE = None


class profile:
    """``with ops.profile() as prof: model(x)`` -> prof.rows = [dict(kind, desc, ms, flops, bytes)] per launch."""

    def __enter__(self):
        global _PROFILE
        self.records = []
        _PROFILE = self.records
        return self

    def __exit__(self, *exc):
        global _PROFILE
        _PROFILE = None
        torch.cuda.synchronize()
        self.rows = [dict(kind=k, desc=d, ms=e0.elapsed_time(e1), flops=f, bytes=b) for (k, d, e0, e1, f, b) in self.records]
        return False


class _timed:
    def __init__(self, kind, desc, flops, nbytes):
        self.meta = (kind, desc, flops, nbytes)

    def __enter__(self):
        if _PROFILE is not None:
            self.e0 = torch.cuda.Event(enable_timing=True)
            self.e1 = torch.cuda.Event(enable_timing=True)
            self.e0.record()
        return self

    def __exit__(self, *exc):
        if _PROFILE is not None:
            self.e1.record()
            k, d, f, b = self.meta
            _PROFILE.append((k, d, self.e0, self.e1, f, b))
        return False


class Act:
    """fp16 channels-last activation: ``data`` is ``[N*T*H*W, ld]`` with channels ``[C, ld)`` zero."""
    __slots__ = ("data", "N", "T", "H", "W", "C")

    def __init__(self, data, N, T, H, W, C):
        self.data, self.N, self.T, self.H, self.W, self.C = data, N, T, H, W, C

    @property
    def ld(self):
        return self.data.shape[1]

    @property
    def M(self):
        return self.data.shape[0]

    @property
    def positions(self):
        return self.T * self.H * self.W

    def __repr__(self):
        return "Act(N=%d,T=%d,H=%d,W=%d,C=%d,ld=%d)" % (self.N, self.T, self.H, self.W, self.C, self.ld)


# ---------------------------------------------------------------------------------------------
# layout
# ---------------------------------------------------------------------------------------------
@_on_device
def from_ncdhw(x, pitch=None):
    """fp32 NCDHW (or NCHW) tensor -> Act.  ``pitch`` = channel pitch (4 for stem inputs)."""
    _require_cuda(x, "input")
    if x.dim() == 4:
        x = x.unsqueeze(2)
    if x.dim() != 5:
        raise ValueError("expected a [N,C,T,H,W] or [N,C,H,W] tensor, got %s" % (tuple(x.shape),))
    half_in = x.dtype == torch.float16
    x = x.contiguous() if half_in else x.contiguous().float()
    N, C, T, H, W = x.shape
    if pitch is None:
        pitch = 4 if C <= 4 else _round_up(C, 8)
    y = torch.empty((N * T * H * W, pitch), dtype=torch.float16, device=x.device)
    lib = _lib.load()
    fn = lib.b2_ncdhw_f16_to_ndhwc_f16 if half_in else lib.b2_ncdhw_f32_to_ndhwc_f16
    with _timed("layout", "ncdhw_%s->ndhwc_f16 C%d px=%d" % ("f16" if half_in else "f32", C, N * T * H * W), 0.0,
                N * T * H * W * (x.element_size() * C + 2.0 * pitch)):
        _lib.check(fn(_ptr(x), _ptr(y), N, C, T, H, W, pitch, _stream()), "b2_ncdhw_to_ndhwc_f16")
    return Act(y, N, T, H, W, C)


@_on_device
def to_ncdhw(a):
    """Act -> fp32 NCDHW tensor (the layout/dtype the reference's ``features`` returns)."""
    y = torch.empty((a.N, a.C, a.T, a.H, a.W), dtype=torch.float32, device=a.data.device)
    lib = _lib.load()
    _lib.check(lib.b2_ndhwc_f16_to_ncdhw_f32(_ptr(a.data), _ptr(y), a.N, a.C, a.T, a.H, a.W, a.ld, _stream()),
               "b2_ndhwc_f16_to_ncdhw_f32")
    return y


# ---------------------------------------------------------------------------------------------
# packed convolution parameters
# ---------------------------------------------------------------------------------------------
class PackedConv:
    """fp16 filter in the engine's [K][taps][C] layout + the folded per-channel affine.

    ``scale``/``shift`` fold the conv bias and the eval-mode BatchNorm that follows the convolution in
    the reference (y = (conv + bias - mean) / sqrt(var + eps) * gamma + beta).
    """
    __slots__ = ("w", "scale", "shift", "K", "Cin", "C", "k", "s", "p", "mode", "up")

    @_on_device
    def __init__(self, weight, bias=None, bn=None, stride=(1, 1, 1), padding=(0, 0, 0), in_pitch=None, stem=False,
                 upsample=False):
        _require_cuda(weight, "conv weight")
        if weight.dim() == 4:       # Conv2d weight -> T = 1
            weight = weight.unsqueeze(2)
        K, Cin, kt, kh, kw = weight.shape
        self.K, self.Cin = K, Cin
        self.k = (kt, kh, kw)
        self.s = tuple(int(v) for v in stride)
        self.p = tuple(int(v) for v in padding)
        self.mode = B2_CONV_STEM7 if stem else B2_CONV_AUTO
        self.C = 4 if stem else (in_pitch if in_pitch is not None else _round_up(Cin, 8))
        self.up = bool(upsample)
        lib = _lib.load()
        w32 = weight.detach().contiguous().float()
        if self.up:
            # conv3x3(nearest_upsample_2x(x)) as four phase-specific 2x2 filters over the low-res image (GBlock conv2)
            if (kt, kh, kw) != (1, 3, 3) or self.s != (1, 1, 1) or self.p != (0, 1, 1) or stem:
                raise ValueError("fused upsampling needs a 3x3 stride-1 'same' convolution")
            self.w = torch.empty(K * 16 * self.C, dtype=torch.float16, device=weight.device)
            _lib.check(lib.b2_pack_upconv3x3_weight(_ptr(w32), _ptr(self.w), K, Cin, self.C, _stream()), "b2_pack_upconv3x3_weight")
        else:
            n = lib.b2_pack_conv_weight_elems(K, Cin, kt, kh, kw, self.C, self.mode)
            self.w = torch.empty(n, dtype=torch.float16, device=weight.device)
            _lib.check(lib.b2_pack_conv_weight(_ptr(w32), _ptr(self.w), K, Cin, kt, kh, kw, self.C, self.mode, _stream()),
                       "b2_pack_conv_weight")
        self.scale, self.shift = fold_affine(K, bias, bn, weight.device)


def dense_from_grouped(weight, groups):
    """Grouped-convolution filter [K][C/groups][...] -> the block-diagonal dense filter [K][C][...] (zeros off the diagonal).
    Output channel k belongs to group k // (K / groups) and reads input channels [g * C/groups, (g + 1) * C/groups)
    (nn.Conv3d semantics, resnext3D.py:86-93).  Groups of the ResNeXt-3D nets are 4..32 channels wide -- far below an MMA
    tile -- so the tensor-core path runs the dense filter; the product with the zero blocks is exact."""
    K, cg = weight.shape[0], weight.shape[1]
    if groups == 1:
        return weight
    if K % groups:
        raise ValueError("output channels %d not divisible by groups %d" % (K, groups))
    dense = weight.new_zeros((K, cg * groups) + tuple(weight.shape[2:]))
    kg = K // groups
    for g in range(groups):
        dense[g * kg:(g + 1) * kg, g * cg:(g + 1) * cg] = weight[g * kg:(g + 1) * kg]
    return dense


def fold_affine(K, bias, bn, device):
    """Per-output-channel (scale, shift) in fp32 for conv(+bias) followed by eval-mode BatchNorm."""
    if bn is not None:
        if bn.training:
            raise RuntimeError("the forward engine is inference-only: call model.eval() (BatchNorm uses running stats)")
        g = bn.weight.detach().double() if bn.weight is not None else torch.ones(K, dtype=torch.float64, device=device)
        b = bn.bias.detach().double() if bn.bias is not None else torch.zeros(K, dtype=torch.float64, device=device)
        inv = torch.rsqrt(bn.running_var.detach().double() + bn.eps)
        scale = g * inv
        shift = b - bn.running_mean.detach().double() * scale
        if bias is not None:
            shift = shift + bias.detach().double() * scale
    else:
        scale = torch.ones(K, dtype=torch.float64, device=device)
        shift = bias.detach().double() if bias is not None else torch.zeros(K, dtype=torch.float64, device=device)
    return scale.float().contiguous(), shift.float().contiguous()


def _out_dim(i, k, s, p):
    return (i + 2 * p - k) // s + 1


# ---------------------------------------------------------------------------------------------
# convolution / dense
# ---------------------------------------------------------------------------------------------
def _out_rows(out, M, ld):
    """Validate a caller-provided output row range (``out=``): fp16 [M][ld], dense rows, 16-byte aligned."""
    if (out.dtype != torch.float16 or out.dim() != 2 or tuple(out.shape) != (M, ld) or out.stride(1) != 1 or out.stride(0) != ld
            or out.data_ptr() % 16):
        raise ValueError("out= must be a dense fp16 [%d][%d] row range, got %s %s strides %s" % (M, ld, out.dtype, tuple(out.shape),
                                                                                                  tuple(out.stride())))
    return out


@_on_device
def conv(a, pc, residual=None, relu=False, simt=False, sample_affine=None, residual_up=False, residual_pre=False,
         next_affine=None, pool_w=False, in_affine=None, out=None):
    """nn.Conv3d -> BatchNorm3d -> (+residual) -> ReLU in one kernel
    (resnet3D.py:91-106, 125-143, 176-185; r2plus1d.py:85-88; torchvision_models.py:449-451).

    ``sample_affine=(scale, shift)``: fp32 ``[N][pitch]`` views -- a per-SAMPLE epilogue affine instead of the packed
    per-channel one (class-conditional BatchNorm of the layer that follows the convolution, BigGAN GBlock).
    ``residual_up``: ``residual`` is the skip tensor at HALF the output resolution, nearest-2x upsampled on the fly (its
    first K channels are used: the GBlock's channel drop); ``residual_pre``: the residual joins before the affine,
    y = act(scale * (conv + residual) + shift).  ``next_affine=(scale2, shift2)`` (fp32 [N][pitch] views): also return
    relu(y * scale2[n] + shift2[n]) -- the ccbn + ReLU that opens the next GBlock -- as a second Act, written by the same
    kernel.  All three: 1x1 convolutions only.  ``out``: preallocated fp16 [M][round_up(K, 8)] rows to write instead of a
    fresh tensor (a row range of a larger batch buffer: the depth-first trunk schedule)."""
    if a.ld != pc.C:
        raise ValueError("activation pitch %d != packed filter pitch %d" % (a.ld, pc.C))
    kt, kh, kw = pc.k
    To, Ho, Wo = (_out_dim(a.T, kt, pc.s[0], pc.p[0]), _out_dim(a.H, kh, pc.s[1], pc.p[1]),
                  _out_dim(a.W, kw, pc.s[2], pc.p[2]))
    if pc.up:                         # the kernel reads the low-res image and writes the 2x upsampled convolution
        Ho, Wo = 2 * Ho, 2 * Wo
    Wconv = Wo
    if pool_w:                        # stem only: MaxPool (k 3, stride 2, pad 1) along W applied in the epilogue (b2_conv_args.pool_w)
        if simt or not relu or pc.mode != B2_CONV_STEM7:
            raise ValueError("pool_w needs the stem convolution kernel with ReLU")
        Wo = (Wo - 1) // 2 + 1
    M = a.N * To * Ho * Wo
    ldy = _round_up(pc.K, 8)
    y = _out_rows(out, M, ldy) if out is not None else torch.empty((M, ldy), dtype=torch.float16, device=a.data.device)
    args = ConvArgs()
    args.x, args.w, args.scale, args.shift = _ptr(a.data), _ptr(pc.w), _ptr(pc.scale), _ptr(pc.shift)
    args.residual = _ptr(residual.data if residual is not None else None)
    args.y = _ptr(y)
    args.N, args.T, args.H, args.W, args.C = a.N, a.T, a.H, a.W, a.ld
    args.K, args.ldy = pc.K, ldy
    args.ldr = residual.ld if residual is not None else 0
    if residual is not None and residual.M * (4 if residual_up else 1) != M:
        raise ValueError("residual rows %d do not match output rows %d" % (residual.M, M))
    if (residual_up or residual_pre) and (residual is None or simt):
        raise ValueError("residual_up / residual_pre need a residual and the tensor-core path")
    args.residual_up, args.residual_pre = int(residual_up), int(residual_pre)
    y2 = None
    if next_affine is not None:
        sc2, sh2 = next_affine
        if simt or sc2.shape != sh2.shape or sc2.shape[0] != a.N or sc2.stride(0) != sh2.stride(0) or sc2.shape[1] < pc.K:
            raise ValueError("next_affine must be two fp32 [N][>=K] views with the same pitch")
        y2 = torch.empty_like(y)
        args.y2, args.scale2, args.shift2, args.aff2_ld = _ptr(y2), _ptr(sc2), _ptr(sh2), sc2.stride(0)
    args.kt, args.kh, args.kw = kt, kh, kw
    args.st, args.sh, args.sw = pc.s
    args.pt, args.ph, args.pw = pc.p
    args.relu, args.out_f32, args.accumulate, args.mode = int(relu), 0, 0, pc.mode
    args.upsample = int(pc.up)
    args.pool_w = int(pool_w)
    if in_affine is not None:         # relu(x * scale[n] + shift[n]) on the A operand of a 1x1 convolution (GBlock bn1 + ReLU)
        isc, ish = in_affine
        if simt or isc.shape != ish.shape or isc.shape[0] != a.N or isc.stride(0) != ish.stride(0) or isc.shape[1] < a.C:
            raise ValueError("input affine must be two fp32 [N][>=C] views with the same pitch")
        args.in_scale, args.in_shift, args.in_aff_ld = _ptr(isc), _ptr(ish), isc.stride(0)
    if pc.up and simt:
        raise ValueError("the CUDA-core cross-check has no fused upsampling")
    if sample_affine is not None:
        sc, sh = sample_affine
        if simt or sc.shape != sh.shape or sc.shape[0] != a.N or sc.stride(0) != sh.stride(0) or sc.shape[1] < pc.K:
            raise ValueError("per-sample affine must be two fp32 [N][>=K] views with the same pitch")
        args.scale, args.shift, args.aff_ld = _ptr(sc), _ptr(sh), sc.stride(0)
    lib = _lib.load()
    fn = lib.b2_conv_ndhwc_fprop_simt if simt else lib.b2_conv_ndhwc_fprop
    taps = kt * kh * kw
    flops = 2.0 * (a.N * To * Ho * Wconv) * pc.K * pc.Cin * taps        # algorithmic (padding taps included)
    res_rows = 0 if residual is None else (M // 4 if residual_up else M)
    nbytes = 2.0 * (a.M * a.C + M * pc.K * (2 if y2 is not None else 1) + res_rows * pc.K + pc.K * pc.Cin * taps)
    desc = "conv %dx%dx%d s%s C%d->%d M=%d%s%s%s%s" % (kt, kh, kw, "".join(map(str, pc.s)), pc.Cin, pc.K, a.N * To * Ho * Wconv,
                                                      " up2" if pc.up else "", " +next" if y2 is not None else "", " +poolW" if pool_w else "",
                                                      " bn1(A)" if in_affine is not None else "")
    with _timed("conv", desc, flops, nbytes):
        _lib.check(fn(ctypes.byref(args), _stream()), "b2_conv_ndhwc_fprop")
    out = Act(y, a.N, To, Ho, Wo, pc.K)
    return (out, Act(y2, a.N, To, Ho, Wo, pc.K)) if y2 is not None else out


@_on_device
def gemm(a2d, b2d, scale, shift, M, N, Kd, residual=None, relu=False, per_row=False, out=None, out_f32=False,
         accumulate=False, second=None, aff_rows=0, next_affine=None):
    """D[M][N] = act(scale * A[M][Kd] . B[N][Kd]^T + shift + residual) on tcgen05 (b2_gemm_f16).
    ``second=(A2, B2, K2)`` adds A2[M][K2] . B2[N][K2]^T into the same accumulator (b2_gemm2_f16)."""
    dev = a2d.device
    if out is None:
        ldd = N if out_f32 else _round_up(N, 8)
        out = torch.empty((M, ldd), dtype=torch.float32 if out_f32 else torch.float16, device=dev)
    g = GemmArgs()
    g.a, g.b, g.scale, g.shift = _ptr(a2d), _ptr(b2d), _ptr(scale), _ptr(shift)
    g.residual = _ptr(residual)
    g.d = _ptr(out)
    g.M, g.N, g.Kd = M, N, Kd
    g.lda, g.ldb, g.ldd = a2d.stride(0), b2d.stride(0), out.stride(0)
    g.ldr = residual.stride(0) if residual is not None else 0
    g.per_row, g.relu, g.out_f32, g.accumulate = int(per_row), int(relu), int(out_f32), int(accumulate)
    if aff_rows:                      # per-sample affine: scale/shift are fp32 [M / aff_rows][pitch] views
        g.aff_ld, g.aff_rows = scale.stride(0), int(aff_rows)
    if next_affine is not None:       # (scale2, shift2, rows per sample): second output relu(D * scale2 + shift2), returned too
        sc2, sh2, rows2 = next_affine
        out2 = torch.empty_like(out)
        g.d2, g.scale2, g.shift2, g.aff2_ld, g.aff2_rows = _ptr(out2), _ptr(sc2), _ptr(sh2), sc2.stride(0), int(rows2)
        with _timed("gemm", "gemm M=%d N=%d K=%d +next" % (M, N, Kd), 2.0 * M * N * Kd,
                    2.0 * (M * Kd + N * Kd) + 2.0 * out.element_size() * M * N + (2.0 * M * N if residual is not None else 0.0)):
            _lib.check(_lib.load().b2_gemm_f16(ctypes.byref(g), _stream()), "b2_gemm_f16")
        return out, out2
    if second is not None:
        a2, b2, k2 = second
        with _timed("gemm", "gemm2 M=%d N=%d K=%d+%d" % (M, N, Kd, k2), 2.0 * M * N * (Kd + k2),
                    2.0 * (M * (Kd + k2) + N * (Kd + k2)) + out.element_size() * M * N):
            _lib.check(_lib.load().b2_gemm2_f16(ctypes.byref(g), _ptr(a2), a2.stride(0), _ptr(b2), b2.stride(0), k2,
                                               _stream()), "b2_gemm2_f16")
        return out
    with _timed("gemm", "gemm M=%d N=%d K=%d" % (M, N, Kd), 2.0 * M * N * Kd,
                2.0 * (M * Kd + N * Kd) + out.element_size() * M * N):
        _lib.check(_lib.load().b2_gemm_f16(ctypes.byref(g), _stream()), "b2_gemm_f16")
    return out


class PackedLinear:
    """nn.Linear weights as an fp16 [out][in_pitch] matrix + fp32 bias (resnet3D.py:162, trn.py:42-44)."""
    __slots__ = ("w", "scale", "shift", "out_features", "in_features", "in_pitch")

    def __init__(self, weight, bias=None):
        _require_cuda(weight, "linear weight")
        out_f, in_f = weight.shape
        self.out_features, self.in_features = out_f, in_f
        self.in_pitch = _round_up(in_f, 8)
        w = torch.zeros((out_f, self.in_pitch), dtype=torch.float16, device=weight.device)
        w[:, :in_f] = weight.detach().to(torch.float16)
        self.w = w
        self.scale, self.shift = fold_affine(out_f, bias, None, weight.device)


def linear(x2d, pl, relu=False, out_f32=False, out=None, accumulate=False):
    """x2d: fp16 [M][in_pitch]  ->  [M][out] (fp16, or fp32 when out_f32)."""
    if x2d.shape[1] < pl.in_features:
        raise ValueError("input has %d features, layer needs %d" % (x2d.shape[1], pl.in_features))
    return gemm(x2d, pl.w, pl.scale, pl.shift, x2d.shape[0], pl.out_features, pl.in_features, relu=relu,
                out_f32=out_f32, out=out, accumulate=accumulate)


# ---------------------------------------------------------------------------------------------
# pooling / shortcuts / casts
# ---------------------------------------------------------------------------------------------
@_on_device
def maxpool3d(a, kernel, stride, padding, out=None):
    """nn.MaxPool3d (resnet3D.py:156; executed at torchvision_models.py:452).  ``out``: see ``conv``."""
    kt, kh, kw = kernel
    st, sh, sw = stride
    pt, ph, pw = padding
    To, Ho, Wo = _out_dim(a.T, kt, st, pt), _out_dim(a.H, kh, sh, ph), _out_dim(a.W, kw, sw, pw)
    My = a.N * To * Ho * Wo
    y = _out_rows(out, My, a.ld) if out is not None else torch.empty((My, a.ld), dtype=torch.float16, device=a.data.device)
    with _timed("maxpool", "maxpool C%d M=%d->%d" % (a.C, a.M, y.shape[0]), 0.0, 2.0 * a.C * (a.M + y.shape[0])):
        _lib.check(_lib.load().b2_maxpool3d_ndhwc(_ptr(a.data), _ptr(y), a.N, a.T, a.H, a.W, a.ld, kt, kh, kw, st, sh, sw,
                                                 pt, ph, pw, _stream()), "b2_maxpool3d_ndhwc")
    return Act(y, a.N, To, Ho, Wo, a.C)


@_on_device
def avgpool_global(a):
    """nn.AdaptiveAvgPool3d(1) + view(B, -1) (torchvision_models.py:460-463): -> fp16 [N][ld]."""
    y = torch.empty((a.N, a.ld), dtype=torch.float16, device=a.data.device)
    with _timed("avgpool", "avgpool C%d M=%d" % (a.C, a.M), 0.0, 2.0 * a.C * (a.M + a.N)):
        _lib.check(_lib.load().b2_avgpool_global_ndhwc(_ptr(a.data), _ptr(y), a.N, a.positions, a.ld, _stream()),
                   "b2_avgpool_global_ndhwc")
    return y


@_on_device
def shortcut_a(a, stride, out_channels):
    """Type-A shortcut: F.avg_pool3d(k=1, stride) + zero channel padding (resnet3D.py:65-74)."""
    To, Ho, Wo = (a.T - 1) // stride + 1, (a.H - 1) // stride + 1, (a.W - 1) // stride + 1
    ldo = _round_up(out_channels, 8)
    y = torch.empty((a.N * To * Ho * Wo, ldo), dtype=torch.float16, device=a.data.device)
    _lib.check(_lib.load().b2_shortcut_a_ndhwc(_ptr(a.data), _ptr(y), a.N, a.T, a.H, a.W, a.ld, stride, ldo, _stream()),
               "b2_shortcut_a_ndhwc")
    return Act(y, a.N, To, Ho, Wo, out_channels)


@_on_device
def concat_rows(a2d, Ca, b2d, Cb):
    """fp16 [rows][>=Ca] ++ [rows][>=Cb] -> [rows][round_up(Ca+Cb, 8)] (torch.cat(dim=1), slowfast.py:143-150, 392)."""
    rows = a2d.shape[0]
    if Ca % 8 or Cb % 8:
        raise ValueError("channel concatenation needs channel counts that are multiples of 8 (got %d, %d)" % (Ca, Cb))
    y = torch.empty((rows, _round_up(Ca + Cb, 8)), dtype=torch.float16, device=a2d.device)
    with _timed("concat", "concat C%d+%d rows=%d" % (Ca, Cb, rows), 0.0, 4.0 * rows * (Ca + Cb)):
        _lib.check(_lib.load().b2_concat_channels(_ptr(a2d), a2d.stride(0), Ca, _ptr(b2d), b2d.stride(0), Cb, _ptr(y),
                                                 y.stride(0), rows, _stream()), "b2_concat_channels")
    return y


def concat_channels(a, b):
    """Act ++ Act along channels (same N, T, H, W)."""
    if (a.N, a.T, a.H, a.W) != (b.N, b.T, b.H, b.W):
        raise ValueError("cannot concatenate %r and %r" % (a, b))
    return Act(concat_rows(a.data, a.C, b.data, b.C), a.N, a.T, a.H, a.W, a.C + b.C)


@_on_device
def cast_rows(x2d, relu=False):
    """fp32 [rows][cols] -> fp16 [rows][round_up(cols, 8)], optional ReLU (trn.py:40-41)."""
    _require_cuda(x2d, "input")
    x2d = x2d.contiguous().float()
    rows, cols = x2d.shape
    y = torch.empty((rows, _round_up(cols, 8)), dtype=torch.float16, device=x2d.device)
    _lib.check(_lib.load().b2_cast_f32_to_f16(_ptr(x2d), x2d.stride(0), _ptr(y), y.stride(0), rows, cols, int(relu),
                                             _stream()), "b2_cast_f32_to_f16")
    return y


@_on_device
def gather_frames(x3d, idx_dev):
    """x3d fp16 [N][T][F], idx int32[n] on device -> [N][n*F] (trn.py:108)."""
    N, T, F = x3d.shape
    n = idx_dev.numel()
    y = torch.empty((N, n * F), dtype=torch.float16, device=x3d.device)
    _lib.check(_lib.load().b2_gather_frames(_ptr(x3d), _ptr(y), _ptr(idx_dev), N, T, F, n, _stream()), "b2_gather_frames")
    return y


@_on_device
def gather_frame_tuples(x3d, idx_dev, n_tuples, n_idx):
    """x3d fp16 [N][T][F], idx int32 [n_tuples][n_idx] on device -> [N * n_tuples][n_idx * F], tuple index fastest
    (trn.py:100-110: every sampled tuple of one scale in one launch)."""
    N, T, F = x3d.shape
    y = torch.empty((N * n_tuples, n_idx * F), dtype=torch.float16, device=x3d.device)
    _lib.check(_lib.load().b2_gather_frame_tuples(_ptr(x3d), _ptr(y), _ptr(idx_dev), N, T, F, n_idx, n_tuples, _stream()),
               "b2_gather_frame_tuples")
    return y


# ---------------------------------------------------------------------------------------------
# non-local attention
# ---------------------------------------------------------------------------------------------
@_on_device
def attention(q2d, k2d, v2d, d, dv, B, Nq, Nk, dot_product=False, mode=None):
    """softmax(Q K^T) V (mode 0), (Q K^T / Nk) V (mode 1, ``dot_product``) or (relu(Q K^T) / Nk) V (mode 2, the
    concatenation mode's rank-2 encoding) -- nonlocalnet.py:143-243.

    q2d: fp16 [B*Nq][>= d]; k2d: fp16 [B*Nk][>= d]; v2d: fp16 [B*Nk][>= dv] (row views of projection outputs, 16-byte
    aligned).  Returns fp16 [B*Nq][dv]."""
    if mode is None:
        mode = 1 if dot_product else 0
    o = torch.empty((B * Nq, _round_up(dv, 8)), dtype=torch.float16, device=q2d.device)
    with _timed("attention", "attention B=%d Nq=%d Nk=%d d=%d dv=%d" % (B, Nq, Nk, d, dv), 2.0 * B * Nq * Nk * (d + dv),
                2.0 * B * (Nq * (d + dv) + Nk * (d + dv))):
        _lib.check(_lib.load().b2_nonlocal_attention(_ptr(q2d), q2d.stride(0), _ptr(k2d), k2d.stride(0), _ptr(v2d),
                                                    v2d.stride(0), _ptr(o), o.stride(0), B, Nq, Nk, d, dv,
                                                    int(mode), _stream()), "b2_nonlocal_attention")
    return o


def nonlocal_attention(qkv, d, dv, B, Npos):
    """Embedded-gaussian core on one fused projection: qkv fp16 [B*Npos][>= 2d + dv] = theta | phi | g."""
    return attention(qkv, qkv[:, d:], qkv[:, 2 * d:], d, dv, B, Npos, Npos)


# ---------------------------------------------------------------------------------------------
# BigGAN-deep generator helpers (architecture absent from the reference tree; see models/biggan_deep.py)
# ---------------------------------------------------------------------------------------------
@_on_device
def embed_concat(z, labels, table, split=False):
    """The conditioning vector every ccbn of the generator consumes, v = [table[labels] | z | 0] (D = round_up(ds+dz, 8)):
    fp16 [B][D], or with ``split`` fp16 [B][3D] = [hi | lo | hi] (v = hi + lo to ~2^-22) for the high-accuracy GEMM against
    [W_hi | W_hi | W_lo].  ``labels`` int64 [B] class indices, or an fp32 [B][shared_dim] tensor that is already embedded."""
    _require_cuda(z, "z")
    z = z.contiguous().float()
    B, dz = z.shape
    ds = table.shape[1]
    D = _round_up(dz + ds, 8)
    ldy = 3 * D if split else D
    y = torch.empty((B, ldy), dtype=torch.float16, device=z.device)
    if labels.dtype in (torch.int64, torch.int32, torch.int16, torch.uint8) and labels.dim() == 1:
        lab, emb = labels.to(torch.int64).contiguous(), None
    else:
        lab, emb = None, labels.contiguous().float()
        if emb.shape != (B, ds):
            raise ValueError("embedded class vectors must be [B, %d], got %s" % (ds, tuple(emb.shape)))
    _lib.check(_lib.load().b2_embed_concat(_ptr(z), _ptr(lab), _ptr(table), _ptr(emb), _ptr(y), B, dz, ds, table.shape[0],
                                          ldy, int(split), _stream()), "b2_embed_concat")
    return y


@_on_device
def ccbn_act(a, scale=None, shift=None, channels=None, up=1, relu=True):
    """act(x * scale[n] + shift[n]) with optional nearest 2x upsampling: the ccbn -> ReLU (-> F.interpolate) chain of a
    GBlock in one HBM pass.  ``scale``/``shift``: fp32 [N][pitch] views (per sample), [1][pitch] (shared), or None
    (pure copy: channel slice x[:, :channels] and/or upsampling of the skip path)."""
    C = a.C if channels is None else channels
    ldy = _round_up(C, 8)
    y = torch.empty((a.N * a.T * a.H * up * a.W * up, ldy), dtype=torch.float16, device=a.data.device)
    if a.T != 1:
        raise ValueError("ccbn_act works on images (T == 1)")
    lda = 0
    if scale is not None:
        lda = scale.stride(0) if scale.shape[0] > 1 else 0
        if scale.shape[0] not in (1, a.N) or scale.shape[1] < C or shift.shape != scale.shape or (
                scale.shape[0] > 1 and shift.stride(0) != lda):
            raise ValueError("ccbn affine must be fp32 [N or 1][>=C] views with one pitch")
    with _timed("ccbn", "ccbn_act C%d px=%d up%d" % (C, a.M, up), 0.0, 2.0 * C * a.M * (1 + up * up)):
        _lib.check(_lib.load().b2_ccbn_act_ndhwc(_ptr(a.data), a.ld, _ptr(y), ldy, _ptr(scale), _ptr(shift), lda, a.N, a.H,
                                                a.W, C, up, int(relu), _stream()), "b2_ccbn_act_ndhwc")
    return Act(y, a.N, 1, a.H * up, a.W * up, C)


def _out_images(out, shape, dtype):
    if tuple(out.shape) != tuple(shape) or out.dtype != dtype or not out.is_contiguous():
        raise ValueError("out= must be a contiguous %s %s tensor, got %s %s" % (dtype, tuple(shape), out.dtype, tuple(out.shape)))
    return out


@_on_device
def tanh_to_nchw(a, out_dtype=torch.float32, out=None):
    """torch.tanh + channels-last -> NCHW: the generator's image write (fp32 like the public model, or fp16).  ``out``: a
    preallocated image range to write (a batch slice of a larger NCHW tensor)."""
    if out_dtype not in (torch.float32, torch.float16):
        raise ValueError("images are written as fp32 or fp16")
    shape = (a.N, a.C, a.H, a.W)
    y = _out_images(out, shape, out_dtype) if out is not None else torch.empty(shape, dtype=out_dtype, device=a.data.device)
    S = a.T * a.H * a.W
    with _timed("tanh", "tanh->nchw C%d px=%d" % (a.C, a.M), 0.0, a.M * (2.0 * a.ld + y.element_size() * a.C)):
        _lib.check(_lib.load().b2_tanh_nhwc_to_nchw(_ptr(a.data), a.ld, _ptr(y), a.N, a.C, S, int(out_dtype == torch.float32),
                                                   _stream()), "b2_tanh_nhwc_to_nchw")
    return y


@_on_device
def rgb_head(partial, bias, N, H, W, K=3, out_dtype=torch.float32, out=None):
    """Second half of the split RGB head: gather the per-tap partial products of the 1x1 GEMM (fp16 [N*H*W][>=36], column
    tap*4 + k), add the bias, tanh, write NCHW images (see b2_rgb_head_gather_tanh).  ``out``: see ``tanh_to_nchw``."""
    if out_dtype not in (torch.float32, torch.float16):
        raise ValueError("images are written as fp32 or fp16")
    y = _out_images(out, (N, K, H, W), out_dtype) if out is not None else torch.empty((N, K, H, W), dtype=out_dtype, device=partial.device)
    M = N * H * W
    with _timed("tanh", "rgb gather+tanh px=%d" % M, 0.0, M * (2.0 * 36 + y.element_size() * K)):
        _lib.check(_lib.load().b2_rgb_head_gather_tanh(_ptr(partial), partial.stride(0), _ptr(bias), _ptr(y), N, H, W, K,
                                                      int(out_dtype == torch.float32), _stream()), "b2_rgb_head_gather_tanh")
    return y


# ---------------------------------------------------------------------------------------------
# backward of the residual blocks (frozen BatchNorm statistics): see engine.py, "fine-tuning"
# ---------------------------------------------------------------------------------------------
@_on_device
def relu_grad_sum(y2d, g2d):
    """ReLU backward: ``(gz, s)`` with gz = g * [y > 0] (fp16, y's shape) and s[c] = sum over rows of gz[:, c] (fp32 [ld]),
    reduced in a fixed order.  y2d: fp16 [M][ld] (a ReLU output), g2d: fp16 [M][>= ld]."""
    M, ld = y2d.shape
    if g2d.shape[0] != M or g2d.shape[1] < ld or g2d.stride(1) != 1 or y2d.stride(0) != ld:
        raise ValueError("gradient %s does not match activation %s" % (tuple(g2d.shape), tuple(y2d.shape)))
    lib = _lib.load()
    gz = torch.empty_like(y2d)
    partial = torch.empty((lib.b2_relu_grad_sum_partials(M, ld), ld), dtype=torch.float32, device=y2d.device)
    s = torch.empty(ld, dtype=torch.float32, device=y2d.device)
    with _timed("bwd_eltwise", "relu_grad_sum C%d M=%d" % (ld, M), 0.0, 6.0 * M * ld):
        _lib.check(lib.b2_relu_grad_sum(_ptr(y2d), ld, _ptr(g2d), g2d.stride(0), _ptr(gz), M, _ptr(partial), _ptr(s), _stream()),
                   "b2_relu_grad_sum")
    return gz, s


def wgrad_args(x, g, K, kernel, stride, padding, dw=None, work=None):
    """WgradArgs for the weight gradient of a convolution with input Act ``x`` and output gradient Act ``g`` (K filters)."""
    from ._lib import WgradArgs
    a = WgradArgs()
    a.x, a.g, a.dw, a.work = _ptr(x.data), _ptr(g.data), _ptr(dw), _ptr(work)
    a.N, a.T, a.H, a.W, a.ldx, a.C = x.N, x.T, x.H, x.W, x.ld, _round_up(x.C, 8)
    a.ldg, a.K = g.ld, K
    (a.kt, a.kh, a.kw), (a.st, a.sh, a.sw), (a.pt, a.ph, a.pw) = kernel, stride, padding
    return a


@_on_device
def conv_wgrad(x, g, K, kernel, stride, padding):
    """Weight gradient sum_p g[p][k] x[p*stride + tap - pad][c] on tcgen05 (b2_conv_ndhwc_wgrad): fp32 [K][taps][C]."""
    taps = kernel[0] * kernel[1] * kernel[2]
    C = _round_up(x.C, 8)
    dw = torch.empty((K, taps, C), dtype=torch.float32, device=x.data.device)
    lib = _lib.load()
    args = wgrad_args(x, g, K, kernel, stride, padding, dw)
    n = lib.b2_wgrad_workspace_floats(ctypes.byref(args))
    work = torch.empty(n, dtype=torch.float32, device=x.data.device) if n else None
    args.work = _ptr(work)
    P = g.N * g.T * g.H * g.W
    with _timed("wgrad", "wgrad %dx%dx%d C%d->%d P=%d" % (kernel + (C, K, P)), 2.0 * P * K * C * taps,
                2.0 * (x.M * x.ld * taps + g.M * g.ld) + 4.0 * dw.numel() * (1 + 2 * (n > 0))):
        _lib.check(lib.b2_conv_ndhwc_wgrad(ctypes.byref(args), _stream()), "b2_conv_ndhwc_wgrad")
    return dw


@_on_device
def zero_dilate(g, T, H, W, stride):
    """Act g of a stride-``stride`` output -> Act of the input geometry (T, H, W) holding g at the strided positions, 0 elsewhere."""
    y = torch.empty((g.N * T * H * W, g.ld), dtype=torch.float16, device=g.data.device)
    with _timed("bwd_eltwise", "zero_dilate C%d M=%d" % (g.C, y.shape[0]), 0.0, 2.0 * (g.M + y.shape[0]) * g.ld):
        _lib.check(_lib.load().b2_zero_dilate_scatter(_ptr(g.data), _ptr(y), g.N, T, H, W, g.ld, stride, _stream()),
                   "b2_zero_dilate_scatter")
    return Act(y, g.N, T, H, W, g.C)


@_on_device
def strided_scatter_add_(y, g2d, C, stride):
    """In place: y[n, s*t, s*h, s*w, :C] += g2d[(n, t, h, w), :C] (the data gradient of a stride-s subsampling)."""
    if g2d.shape[0] != y.N * ((y.T - 1) // stride + 1) * ((y.H - 1) // stride + 1) * ((y.W - 1) // stride + 1):
        raise ValueError("subsampled gradient rows %d do not match %r at stride %d" % (g2d.shape[0], y, stride))
    with _timed("bwd_eltwise", "strided_scatter_add C%d M=%d" % (C, g2d.shape[0]), 0.0, 6.0 * g2d.shape[0] * C):
        _lib.check(_lib.load().b2_strided_scatter_add(_ptr(g2d), g2d.stride(0), _ptr(y.data), y.ld, y.N, y.T, y.H, y.W, C, stride,
                                                     _stream()), "b2_strided_scatter_add")
    return y
