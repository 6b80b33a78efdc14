"""Forward engine: walks a (reference-layout) module tree and replaces the bodies of its hot blocks by
fused sm_100a kernels.

The nn.Modules in ``models/`` are *parameter containers* that keep the reference's ``state_dict``
layout; nothing in them computes.  This file holds the block bodies:

* ``conv_bn_act``        Conv3d/Conv2d/SpatioTemporalConv + BatchNorm (+residual) (+ReLU) -> one or two
                         implicit-GEMM launches                      (resnet3D.py:91-106, 125-143)
* ``run_basic/run_bottleneck``  residual blocks incl. type-A/B shortcuts (resnet3D.py:65-74, 176-185)
* ``run_nonlocal``       fused theta|phi|g projection, fused attention, W+BN+residual (nonlocalnet.py:143-166)
* ``run_stem`` / ``run_head``   stem conv+BN+ReLU+maxpool, global average + last_linear
                         (torchvision_models.py:448-464)

Packed fp16 filters and folded BN affines are cached on the owning module.  The cache key is
``(data_ptr, _version, shape)`` of every source tensor, so ``load_state_dict`` and in-place edits of the
parameter itself (``p.copy_()``, ``p.mul_()`` under ``no_grad``) rebuild the packed copy.  Edits made through
``p.data`` (the reference's own init style, ``m.weight.data.fill_``) bump a *different* version counter and are
NOT seen: ``model.invalidate()`` / ``engine.invalidate(model)`` drops every packed copy, and it runs by itself on
``train()`` / ``eval()`` and on ``.to()`` / ``.half()`` / ``.cuda()`` (``_apply``).

Every block body is entered through a ``torch.autograd.Function`` (``functions.py``, SURVEY.md section 8b-ii): the
Function's ``forward`` is the ctypes call sequence, its outputs are marked non-differentiable (frozen-backbone
semantics: the engine has no backward for the convolutional trunk), and the dense heads (``last_linear``, the TRN
relation MLPs) have a real backward on the same tcgen05 GEMM so that a head can be trained on engine features.
"""
import os

import torch
import torch.nn as nn

from . import ops
from . import functions as Fn
from .ops import Act


# ---------------------------------------------------------------------------------------------
# packed-parameter cache
# ---------------------------------------------------------------------------------------------
def _sig(*tensors):
    return tuple((t.data_ptr(), t._version, tuple(t.shape)) if t is not None else None for t in tensors)


def _bn_tensors(bn):
    if bn is None:
        return ()
    return (bn.weight, bn.bias, bn.running_mean, bn.running_var)


def _cached(owner, slot, sig, build):
    cache = owner.__dict__.setdefault("_b2_cache", {})
    hit = cache.get(slot)
    if hit is not None and hit[0] == sig:
        return hit[1]
    val = build()
    cache[slot] = (sig, val)
    return val


def invalidate(root):
    """Drop every packed filter / folded affine cached under ``root`` (call after editing parameters through ``.data``)."""
    for m in root.modules():
        m.__dict__.pop("_b2_cache", None)
        m.__dict__.pop("_b2_pack", None)
    return root


class CacheOwner:
    """Mixin for engine-backed nn.Modules: packed copies are dropped whenever the module is moved, cast or switched
    between train / eval, and on request (``invalidate()``)."""

    def invalidate(self):
        return invalidate(self)

    def train(self, mode=True):
        invalidate(self)
        return super().train(mode)

    def _apply(self, fn, *args, **kwargs):
        invalidate(self)
        return super()._apply(fn, *args, **kwargs)


def _triple(v):
    if isinstance(v, (tuple, list)):
        v = tuple(int(i) for i in v)
        return (1,) + v if len(v) == 2 else v
    return (int(v),) * 3


def _conv_geometry(conv):
    if isinstance(conv, nn.Conv2d):
        s, p = conv.stride, conv.padding
        return (1, int(s[0]), int(s[1])), (0, int(p[0]), int(p[1]))
    return _triple(conv.stride), _triple(conv.padding)


def packed_conv(conv, bn, in_pitch, stem=False, stride=None):
    """PackedConv for a plain nn.Conv3d / nn.Conv2d followed (optionally) by BatchNorm ``bn``."""
    if any(d != 1 for d in conv.dilation):
        raise NotImplementedError("dilated convolutions are outside the engine's scope")
    if conv.groups != 1 and stem:
        raise NotImplementedError("grouped stem convolutions are outside the engine's scope")
    sig = _sig(conv.weight, conv.bias, *_bn_tensors(bn)) + (in_pitch, stem, id(bn), stride)
    cstride, padding = _conv_geometry(conv)
    if stride is None:
        stride = cstride
    # grouped convolution (ResNeXt-3D, resnext3D.py:86-93): packed as the block-diagonal dense filter, see ops.dense_from_grouped
    return _cached(conv, "pc", sig,
                   lambda: ops.PackedConv(ops.dense_from_grouped(conv.weight.detach(), conv.groups), conv.bias, bn, stride, padding,
                                          in_pitch=in_pitch, stem=stem))


def _is_stem_shape(conv):
    w = conv.weight
    kw = w.shape[-1]
    stride, padding = _conv_geometry(conv)
    return w.shape[1] <= 4 and kw == 7 and stride[2] == 2 and padding[2] == 3


def _st_conv_body(conv, bn, a, residual, relu, simt, out=None):
    """(2+1)D factorised conv (r2plus1d.py:85-88): spatial conv + its own BN + ReLU, then the temporal conv whose
    epilogue carries the *outer* BN / residual / ReLU."""
    mid = conv_bn_act(conv.spatial_conv, conv.bn, a, relu=True, simt=simt)
    return conv_bn_act(conv.temporal_conv, bn, mid, residual=residual, relu=relu, simt=simt, out=out)


def conv_bn_act(conv, bn, a, residual=None, relu=False, simt=False, pool_w=False, out=None):
    """Run ``conv`` (Conv3d / Conv2d / SpatioTemporalConv-like) -> ``bn`` -> (+residual) -> (ReLU).  ``pool_w``: stem only, see
    ``_stem_body``.  ``out``: preallocated output rows (``ops.conv``)."""
    if hasattr(conv, "spatial_conv") and hasattr(conv, "temporal_conv"):
        return Fn.SpatioTemporalConvFunction.run(conv, a, bn, residual, relu, simt, out)
    stem = a.ld == 4
    if stem and not _is_stem_shape(conv):
        raise NotImplementedError("NDHWC4 inputs are only supported by 7-wide stride-2 stem convolutions")
    if a.W % 2 != 0 and stem:
        raise ValueError("stem convolution needs an even input width (got %d)" % a.W)
    stride, padding = _conv_geometry(conv)
    if (not simt and tuple(conv.weight.shape[2:]) in ((1, 1, 1), (1, 1)) and padding == (0, 0, 0)
            and stride[0] == stride[1] == stride[2] and stride[0] > 1 and a.T > 1):
        # strided 1x1x1 projection (type-B shortcut, resnet3D.py:176-185): the strided pixel subset is gathered
        # once (1/s^3 of the input) and the projection becomes a plain HBM-bound GEMM on the persistent kernel
        sub = ops.shortcut_a(a, stride[0], a.C)
        pc = packed_conv(conv, bn, sub.ld, stride=(1, 1, 1))
        return ops.conv(sub, pc, residual=residual, relu=relu, out=out)
    pc = packed_conv(conv, bn, a.ld, stem=stem)
    return ops.conv(a, pc, residual=residual, relu=relu, simt=simt, pool_w=pool_w, out=out)


# ---------------------------------------------------------------------------------------------
# residual blocks
# ---------------------------------------------------------------------------------------------
def _shortcut(block, a, simt):
    ds = block.downsample
    if ds is None:
        return a
    if isinstance(ds, nn.Sequential):          # type B: 1x1x1 conv (stride s) + BN
        return conv_bn_act(ds[0], ds[1], a, relu=False, simt=simt)
    if hasattr(ds, "planes") and hasattr(ds, "stride"):   # type A (ShortcutA)
        return ops.shortcut_a(a, ds.stride, ds.planes)
    raise NotImplementedError("unsupported downsample %r" % (ds,))


def run_basic(block, a, simt=False, out=None):
    """conv-BN-ReLU-conv-BN-(+shortcut)-ReLU (resnet3D.py:91-106)."""
    return Fn.BasicBlockFunction.run(block, a, simt, out)


def _basic_body(block, a, simt=False, out=None):
    res = _shortcut(block, a, simt)
    h = conv_bn_act(block.conv1, block.bn1, a, relu=True, simt=simt)
    return conv_bn_act(block.conv2, block.bn2, h, residual=res, relu=True, simt=simt, out=out)


def _plain_1x1(conv):
    return (isinstance(conv, (nn.Conv3d, nn.Conv2d)) and all(k == 1 for k in conv.weight.shape[2:]) and conv.groups == 1
            and all(p == 0 for p in _conv_geometry(conv)[1]))


def _fused_close_with_projection(block, a, h, out=None):
    """conv3 + bn3 + (downsample conv + bn)(x) + ReLU as ONE two-operand GEMM (resnet3D.py:136-143 with the type-B
    shortcut of resnet3D.py:176-185): both BatchNorm scales are folded into the fp16 weight matrices, both products
    accumulate in the same TMEM tile, and the projected shortcut never goes through HBM."""
    ds_conv, ds_bn = block.downsample[0], block.downsample[1]
    stride = _conv_geometry(ds_conv)[0]
    xs = a if stride == (1, 1, 1) else ops.shortcut_a(a, stride[0], a.C)
    if xs.M != h.M:
        raise RuntimeError("shortcut / main path shape mismatch")
    dev = a.data.device

    def build():
        s3, b3 = ops.fold_affine(block.conv3.weight.shape[0], block.conv3.bias, block.bn3, dev)
        sd, bd = ops.fold_affine(ds_conv.weight.shape[0], ds_conv.bias, ds_bn, dev)
        K = block.conv3.weight.shape[0]
        w3 = torch.zeros((K, h.ld), dtype=torch.float16, device=dev)
        w3[:, :h.C] = (_conv1x1_matrix(block.conv3).float() * s3[:, None]).to(torch.float16)
        wd = torch.zeros((K, xs.ld), dtype=torch.float16, device=dev)
        wd[:, :xs.C] = (_conv1x1_matrix(ds_conv).float() * sd[:, None]).to(torch.float16)
        return w3, wd, torch.ones(K, dtype=torch.float32, device=dev), (b3 + bd).contiguous()

    sig = _sig(block.conv3.weight, block.conv3.bias, *_bn_tensors(block.bn3), ds_conv.weight, ds_conv.bias,
               *_bn_tensors(ds_bn)) + (h.ld, xs.ld)
    w3, wd, ones, shift = _cached(block, "close2", sig, build)
    K = w3.shape[0]
    if out is not None:
        ops._out_rows(out, h.M, ops._round_up(K, 8))
    y = ops.gemm(h.data, w3, ones, shift, h.M, K, h.ld, relu=True, second=(xs.data, wd, xs.ld), out=out)
    return Act(y, h.N, h.T, h.H, h.W, K)


def run_bottleneck(block, a, simt=False, out=None):
    """1x1x1-BN-ReLU, 3x3x3(stride)-BN-ReLU, 1x1x1-BN-(+shortcut)-ReLU (resnet3D.py:125-143)."""
    return Fn.BottleneckFunction.run(block, a, simt, out)


def _fusable_close(block, a, simt):
    ds = block.downsample
    return (not simt and isinstance(ds, nn.Sequential) and len(ds) == 2 and _plain_1x1(ds[0]) and _plain_1x1(block.conv3)
            and not ds[1].training and len(set(_conv_geometry(ds[0])[0])) == 1 and (a.T > 1 or _conv_geometry(ds[0])[0][0] == 1)
            and isinstance(ds[0], nn.Conv3d))


def _bottleneck_body(block, a, simt=False, out=None):
    if _fusable_close(block, a, simt):
        h = conv_bn_act(block.conv1, block.bn1, a, relu=True)
        h = conv_bn_act(block.conv2, block.bn2, h, relu=True)
        return _fused_close_with_projection(block, a, h, out)
    res = _shortcut(block, a, simt)
    h = conv_bn_act(block.conv1, block.bn1, a, relu=True, simt=simt)
    h = conv_bn_act(block.conv2, block.bn2, h, relu=True, simt=simt)
    return conv_bn_act(block.conv3, block.bn3, h, residual=res, relu=True, simt=simt, out=out)


def _bn_relu(bn, a):
    """Stand-alone eval-mode BatchNorm + ReLU over an activation (the pre-activation that opens a pre-act block): one
    element-wise HBM pass with the folded per-channel affine."""
    dev = a.data.device
    sc, sh = _cached(bn, "aff1", _sig(*_bn_tensors(bn)) + (a.ld,),
                     lambda: tuple(t.reshape(1, -1).contiguous() for t in ops.fold_affine(bn.num_features, None, bn, dev)))
    flat = ops.ccbn_act(Act(a.data, a.N, 1, a.T * a.H, a.W, a.C), sc, sh, relu=True)
    return Act(flat.data, a.N, a.T, a.H, a.W, a.C)


def _preact_body(block, a, simt=False, out=None):
    """PreActivationBasicBlock / PreActivationBottleneck (pre_act_resnet3D.py:41-57, 76-96):
    out = conv1(relu(bn1(x))); out = conv2(relu(bn2(out))); [out = conv3(relu(bn3(out)))]; out += shortcut(x); no ReLU.
    bn_{k+1} + ReLU run in conv_k's epilogue; the last convolution's epilogue adds the shortcut of the RAW x."""
    res = _shortcut(block, a, simt)
    h = _bn_relu(block.bn1, a)
    h = conv_bn_act(block.conv1, block.bn2, h, relu=True, simt=simt)
    if hasattr(block, "conv3"):
        h = conv_bn_act(block.conv2, block.bn3, h, relu=True, simt=simt)
        return conv_bn_act(block.conv3, None, h, residual=res, relu=False, simt=simt, out=out)
    return conv_bn_act(block.conv2, None, h, residual=res, relu=False, simt=simt, out=out)


def run_block(block, a, simt=False, out=None):
    """One residual block (+ its non-local block).  ``out``: preallocated rows for the block's result (the last kernel writes there)."""
    nl = getattr(block, "nonlocalblock", None)
    if nl is not None and not getattr(block, "nonlocal_layer", True):
        nl = None
    bout = out if nl is None else None
    if getattr(block, "preactivation", False):
        y = Fn.PreActBlockFunction.run(block, a, simt, bout)
    else:
        y = run_bottleneck(block, a, simt, bout) if hasattr(block, "conv3") else run_basic(block, a, simt, bout)
    if nl is not None:
        y = run_nonlocal(nl, y, simt=simt, out=out)
    return y


# ---------------------------------------------------------------------------------------------
# non-local block (embedded gaussian, no sub-sampling)
# ---------------------------------------------------------------------------------------------
def _conv1x1_matrix(conv):
    return conv.weight.detach().reshape(conv.weight.shape[0], -1)


def _first(m):
    return m[0] if isinstance(m, nn.Sequential) else m


def _pad_cols(x2d, cols):
    """fp16 [rows][ld] -> [rows][cols] with zero columns appended (glue for operands whose K extent must be a multiple of 64)."""
    if x2d.shape[1] == cols:
        return x2d
    y = x2d.new_zeros((x2d.shape[0], cols))
    y[:, :x2d.shape[1]] = x2d
    return y


def run_nonlocal(nl, a, simt=False, out=None):
    return Fn.NonLocalFunction.run(nl, a, simt, out)


def _nonlocal_body(nl, a, simt=False, out=None):
    """z = W(y) + x with y = softmax(theta^T phi) g  (embedded gaussian, nonlocalnet.py:143-166),
    y = softmax(x^T phi(x)) g (gaussian, :168-190), y = (theta^T phi / N) g (dot product, :192-211) or
    y = (relu(w . [theta_i ; phi_j]) / N) g (concatenation, :213-243); phi and g are max-pooled when ``sub_sample``
    (:126-131).

    The attention kernel takes d and dv in multiples of 64: the theta / phi / g projections are packed with zero rows up
    to ``dp = round_up(inter_channels, 64)`` (zero logit contributions, zero output columns -- exact), so any width the
    reference accepts runs (nonlocalresnet3d18/34 put a block on C = 64, d = 32).

    Concatenation mode: ``concat_project`` is a bias-free 1x1 Conv2d over the 2d channels of [theta_i ; phi_j] followed
    by ReLU, i.e. f_ij = relu(a_i + b_j) with a_i = w_theta . theta_i and b_j = w_phi . phi_j.  The N x N x 2d tensor the
    reference materialises is never built: a_i + b_j is the rank-2 product of Q_i = [a_i, 1, 0, ...] and K_j = [1, b_j, 0, ...]
    (64-wide), which goes through the same fused kernel with ReLU in place of the softmax (mode 2)."""
    mode = nl.mode
    if mode not in ("embedded_gaussian", "gaussian", "dot_product", "concatenation"):
        raise NotImplementedError("non-local mode %r is outside the engine's scope" % (mode,))
    d, C = nl.inter_channels, nl.in_channels
    dp = ops._round_up(d, 64)
    dev = a.data.device
    w_conv, w_bn = (nl.W[0], nl.W[1]) if isinstance(nl.W, nn.Sequential) else (nl.W, None)
    g_conv = _first(nl.g)
    concat = mode == "concatenation"
    sub = bool(nl.sub_sample)
    if mode == "gaussian":
        projected = [g_conv]
    elif concat:
        projected = [nl.theta, _first(nl.phi), g_conv]
    else:
        projected = [nl.theta, _first(nl.phi), g_conv]           # column order of the GEMM
    cp_w = nl.concat_project[0].weight if concat else None

    def block(conv):                                             # [dp][ld] fp16 weight rows + fp32 bias of one projection
        w = torch.zeros((dp, a.ld), dtype=torch.float32, device=dev)
        w[:d, :C] = _conv1x1_matrix(conv).float()
        b = torch.zeros(dp, dtype=torch.float32, device=dev)
        if conv.bias is not None:
            b[:d] = conv.bias.detach().float()
        return w, b

    def scalar_block(conv, wvec, slot):
        """64 projection columns [.., wvec . conv(x), ..] with the scalar in column ``slot`` and a constant 1 in the other
        of the first two columns: Q_i = [a_i, 1, 0..] (slot 0) resp. K_j = [1, b_j, 0..] (slot 1)."""
        w = torch.zeros((64, a.ld), dtype=torch.float64, device=dev)
        b = torch.zeros(64, dtype=torch.float64, device=dev)
        w[slot, :C] = wvec.double() @ _conv1x1_matrix(conv).double()
        b[slot] = (wvec.double() @ conv.bias.detach().double()) if conv.bias is not None else 0.0
        b[1 - slot] = 1.0
        return w.float(), b.float()

    def build():
        if concat:
            wv = cp_w.detach().reshape(-1)
            q_w, q_b = scalar_block(nl.theta, wv[:d], 0)
            g_w, g_b = block(g_conv)
            if sub:      # phi must be pooled before w_phi is applied (max is not linear): full-resolution phi | g, then a small GEMM
                p_w, p_b = block(_first(nl.phi))
                ws, bs = [q_w, p_w, g_w], [q_b, p_b, g_b]
                kw = torch.zeros((64, dp), dtype=torch.float16, device=dev)
                kw[1, :d] = wv[d:].to(torch.float16)
                kshift = torch.zeros(64, dtype=torch.float32, device=dev)
                kshift[0] = 1.0
                extra = (kw, torch.ones(64, dtype=torch.float32, device=dev), kshift)
            else:
                k_w, k_b = scalar_block(_first(nl.phi), wv[d:], 1)
                ws, bs, extra = [q_w, k_w, g_w], [q_b, k_b, g_b], None
        else:
            pairs = [block(conv) for conv in projected]
            ws, bs, extra = [w for w, _ in pairs], [b for _, b in pairs], None
        w = torch.cat(ws).to(torch.float16).contiguous()
        b = torch.cat(bs).contiguous()
        wo = torch.zeros((C, dp), dtype=torch.float16, device=dev)
        wo[:, :d] = _conv1x1_matrix(w_conv).to(torch.float16)
        so, bo = ops.fold_affine(C, w_conv.bias, w_bn, dev)
        return w, b, torch.ones(w.shape[0], dtype=torch.float32, device=dev), wo, so, bo, extra

    srcs = [t for conv in projected for t in (conv.weight, conv.bias)]
    sig = _sig(*srcs, w_conv.weight, w_conv.bias, cp_w, *_bn_tensors(w_bn)) + (a.ld, mode, sub)
    wp, bp, ones, wo, so, bo, extra = _cached(nl, "proj", sig, build)

    pool = {3: (2, 2, 2), 2: (1, 2, 2), 1: (1, 1, 2)}[nl.dimension]
    B, Nq = a.N, a.positions
    amode = {"dot_product": 1, "concatenation": 2}.get(mode, 0)
    if mode == "gaussian":
        gv = ops.gemm(a.data, wp, ones, bp, a.M, dp, a.ld)                      # g(x): [M][dp]
        Cq = ops._round_up(C, 64)
        xq = _pad_cols(a.data, Cq)                                               # theta = x itself
        if sub:
            xk = ops.maxpool3d(a, pool, pool, (0, 0, 0))                           # phi = max_pool(x)
            gk = ops.maxpool3d(Act(gv, a.N, a.T, a.H, a.W, dp), pool, pool, (0, 0, 0))
            k2d, v2d, Nk = _pad_cols(xk.data, Cq), gk.data, xk.positions
        else:
            k2d, v2d, Nk = xq, gv, Nq
        y = ops.attention(xq, k2d, v2d, Cq, dp, B, Nq, Nk)
    elif concat and sub:
        q = ops.gemm(a.data, wp[:64], ones[:64], bp[:64], a.M, 64, a.ld)        # [a_i, 1, 0..]
        kv = ops.gemm(a.data, wp[64:], ones[64:], bp[64:], a.M, 2 * dp, a.ld)   # phi | g at full resolution
        kvp = ops.maxpool3d(Act(kv, a.N, a.T, a.H, a.W, 2 * dp), pool, pool, (0, 0, 0))
        kw, kones, kshift = extra
        k = ops.gemm(kvp.data, kw, kones, kshift, kvp.M, 64, dp)                 # [1, w_phi . phi_j, 0..]
        y = ops.attention(q, k, kvp.data[:, dp:], 64, dp, B, Nq, kvp.positions, mode=2)
    elif concat:
        qkv = ops.gemm(a.data, wp, ones, bp, a.M, 128 + dp, a.ld)               # [a_i,1,0..] | [1,b_j,0..] | g
        y = ops.attention(qkv, qkv[:, 64:], qkv[:, 128:], 64, dp, B, Nq, Nq, mode=2)
    elif not sub:
        qkv = ops.gemm(a.data, wp, ones, bp, a.M, 3 * dp, a.ld)                  # [M][3dp]: theta | phi | g
        y = ops.attention(qkv, qkv[:, dp:], qkv[:, 2 * dp:], dp, dp, B, Nq, Nq, mode=amode)
    else:
        q = ops.gemm(a.data, wp[:dp], ones[:dp], bp[:dp], a.M, dp, a.ld)         # theta at full resolution
        kv = ops.gemm(a.data, wp[dp:], ones[dp:], bp[dp:], a.M, 2 * dp, a.ld)    # phi | g ...
        kvp = ops.maxpool3d(Act(kv, a.N, a.T, a.H, a.W, 2 * dp), pool, pool, (0, 0, 0))   # ... max-pooled together
        y = ops.attention(q, kvp.data, kvp.data[:, dp:], dp, dp, B, Nq, kvp.positions, mode=amode)
    # W (1x1 conv with bias) + BN + residual x, no ReLU
    if out is not None:
        ops._out_rows(out, a.M, ops._round_up(C, 8))
    z = ops.gemm(y, wo, so, bo, a.M, C, dp, residual=a.data, out=out)
    return Act(z, a.N, a.T, a.H, a.W, C)


# ---------------------------------------------------------------------------------------------
# stem / trunk / head
# ---------------------------------------------------------------------------------------------
def _pool_args(mp):
    if isinstance(mp, nn.MaxPool2d):
        k, s, p = mp.kernel_size, mp.stride, mp.padding
        two = lambda v: (v, v) if isinstance(v, int) else tuple(v)
        k, s, p = two(k), two(s), two(p)
        return (1, k[0], k[1]), (1, s[0], s[1]), (0, p[0], p[1])
    return _triple(mp.kernel_size), _triple(mp.stride), _triple(mp.padding)


def run_stem(model, x, simt=False, out=None):
    """conv1 -> bn1 -> relu -> maxpool (torchvision_models.py:449-452)."""
    a = x if isinstance(x, Act) else ops.from_ncdhw(x)
    return Fn.StemFunction.run(model, a, simt, out)


def _stem_body(model, a, simt=False, out=None):
    """conv1 -> bn1 -> ReLU -> maxpool.  When the stem runs on the Toeplitz kernel and the pool is the usual 3-wide / stride-2 /
    pad-1 window along W, that direction of the pool is taken in the convolution's epilogue (max-pooling is separable, so this is
    exact): the stem writes half of its output and the remaining (kt, kh, 1) pool reads half as much."""
    k, s, p = _pool_args(model.maxpool)
    conv = model.conv1
    plain = isinstance(conv, (nn.Conv3d, nn.Conv2d))
    if (plain and not simt and a.ld == 4 and _is_stem_shape(conv) and (k[2], s[2], p[2]) == (3, 2, 1)
            and ops._out_dim(a.W, 7, 2, 3) <= 120 and os.environ.get("B2_STEM_POOLW", "1") != "0"):
        a = conv_bn_act(conv, model.bn1, a, relu=True, pool_w=True)
        return ops.maxpool3d(a, (k[0], k[1], 1), (s[0], s[1], 1), (p[0], p[1], 0), out=out)
    a = conv_bn_act(conv, model.bn1, a, relu=True, simt=simt)
    return ops.maxpool3d(a, k, s, p, out=out)


# ---------------------------------------------------------------------------------------------
# trunk schedule: breadth-first (default) or, on request, depth-first in clip chunks
# ---------------------------------------------------------------------------------------------
# Clips are independent in every layer (eval-mode BN, per-clip attention), so the trunk may be walked in any clip order.  The
# breadth-first walk (one launch per layer over the whole batch) is the default.  ``set_dfs("units:clips,...")`` walks consecutive
# segments of trunk units DEPTH-first instead -- a chunk of a few clips goes through stem, pool and a run of residual blocks before
# the next chunk starts, so that a chunk's intermediates are write-then-read inside the 126 MB L2 (the allocator hands the next
# chunk the same addresses) and only a segment's first input and last output cross HBM; the last kernel of a chunk writes straight
# into its row range of the whole-batch tensor (``out=``).  MEASURED on B200 (tools/dfs_sweep.py, profiles/dfs_sweep_r02.txt): it
# never pays.  resnet3d50 at 32 clips of 16x224x224: 3.72 ms breadth-first; stem + layer1 in chunks of 8 / 4 / 2 / 1 clips: 4.07 /
# 4.25 / 4.88 / 6.53 ms; same picture for R(2+1)D-34, the non-local net, resnet18 and the BigGAN generator.  Every extra launch of
# these persistent kernels costs 6-9 us of pipeline fill, drain and tile quantisation, and the layers that look HBM-bound (1x1x1
# convolutions at 0.83 of the copy rate) do not speed up when their operands are L2-resident.  The schedule stays as an opt-in
# (same kernels per output element: results equal the breadth-first walk up to kernel-dispatch boundaries) with the evidence.
_DFS_SPEC = os.environ.get("B2_DFS", "off")


def set_dfs(spec):
    """Trunk schedule: ``"off"`` (breadth-first, the default and the measured optimum) or an explicit
    ``"units:clips,units:clips"`` list -- consecutive segments of trunk units (unit 0 = stem + pool, then the residual blocks in
    order), each walked depth-first in chunks of ``clips``; units not covered run breadth-first."""
    global _DFS_SPEC
    _DFS_SPEC = str(spec)


def _trunk_units(model):
    units = [("stem", model)]
    for name in ("layer1", "layer2", "layer3", "layer4"):
        units += [("block", blk) for blk in getattr(model, name)]
    return units


def dfs_plan(model=None, N=None, geom=None):
    """[(units, clips per chunk)] for ``run_trunk`` (empty = breadth-first)."""
    spec = _DFS_SPEC.strip().lower()
    if spec in ("0", "off", "none", "", "auto"):       # "auto" = the measured rule: never chunk
        return []
    return [tuple(int(v) for v in part.split(":")) for part in spec.split(",")]


def _slice_clips(x, n0, n1):
    if isinstance(x, Act):
        r = x.positions
        return Act(x.data[n0 * r:n1 * r], n1 - n0, x.T, x.H, x.W, x.C)
    return x[n0:n1]


def _run_units(units, a, simt, out=None):
    for j, (kind, m) in enumerate(units):
        o = out if j == len(units) - 1 else None
        a = run_stem(m, a, simt=simt, out=o) if kind == "stem" else run_block(m, a, simt=simt, out=o)
    return a


def _run_segment(units, x, N, clips, simt):
    """Depth-first walk of ``units`` in chunks of ``clips``; the last kernel of each chunk writes straight into its row range of the
    segment's whole-batch output (allocated once the first chunk has shown the output geometry)."""
    buf = None
    for n0 in range(0, N, clips):
        n1 = min(N, n0 + clips)
        o = buf.data[n0 * buf.positions:n1 * buf.positions] if buf is not None else None
        y = _run_units(units, _slice_clips(x, n0, n1), simt, out=o)
        if buf is None:
            buf = Act(torch.empty((N * y.positions, y.ld), dtype=torch.float16, device=y.data.device), N, y.T, y.H, y.W, y.C)
            o = buf.data[:y.M]
        if y.data.data_ptr() != o.data_ptr():      # first chunk, or a unit whose last kernel takes no ``out``
            o.copy_(y.data)
    return buf


def run_trunk(model, x, simt=False, trainable_from=None):
    """The trunk on ``x``.  ``trainable_from`` (1..4): the blocks of ``layer{trainable_from}..layer4`` run breadth-first
    through ``TrainableBlockFunction`` (the depth-first plan only covers the frozen units before them), and the result is a
    ``TrainAct`` that ``run_head`` pools differentiably."""
    units = _trunk_units(model)
    cut = len(units)
    if trainable_from is not None:
        first = getattr(model, "layer%d" % trainable_from)[0]
        cut = next(i for i, (_, m) in enumerate(units) if m is first)
    frozen, trained = units[:cut], units[cut:]
    N = x.N if isinstance(x, Act) else x.shape[0]
    plan = [] if simt else dfs_plan()
    a, ui = x, 0
    for n_units, clips in plan:
        seg = frozen[ui:ui + n_units]
        if not seg:
            break
        ui += len(seg)
        a = _run_segment(seg, a, N, clips, simt) if 0 < clips < N else _run_units(seg, a, simt)
    if ui < len(frozen):
        a = _run_units(frozen[ui:], a, simt)
    if not trained:
        return a
    scale = Fn.GradScale()
    for _, blk in trained:
        a = Fn.TrainableBlockFunction.run(blk, a, scale)
    return TrainAct(a, scale)


def run_head(model, a, head):
    """avgpool -> view(B,-1) -> last_linear (torchvision_models.py:460-464).  Returns fp32 [N][classes]."""
    if isinstance(a, TrainAct):
        # fine-tuned trunk: fp32 pooled features (the same fp16 values as below) through a differentiable pool
        pooled = Fn.PoolFunction.apply(a.data, Fn._geom(a), a.grad_scale)
        return Fn.linear(pooled, head.weight, head.bias) if isinstance(head, nn.Linear) else head(pooled)
    pooled = ops.avgpool_global(a)                     # fp16 [N][ld]
    if isinstance(head, nn.Linear) and torch.is_grad_enabled() and any(p.requires_grad for p in head.parameters()):
        # trainable head on frozen engine features: differentiable GEMM (functions.LinearFunction), same kernel
        return Fn.linear(pooled[:, :head.in_features], head.weight, head.bias)
    if isinstance(head, nn.Linear):
        pl = _cached(head, "pl", _sig(head.weight, head.bias), lambda: ops.PackedLinear(head.weight, head.bias))
        return ops.linear(pooled, pl, out_f32=True)
    # user-swapped head (Identity, Dropout, custom module): hand it the pooled features like the reference does
    return head(pooled[:, :a.C].float())


# ---------------------------------------------------------------------------------------------
# fine-tuning: residual blocks with a backward, BatchNorm statistics frozen
# ---------------------------------------------------------------------------------------------
# Every layer is y = relu(z [+ r]) with z = s * conv(x, W) + shift, s = gamma / sqrt(var + eps), and the running statistics
# fixed.  With gz = g_y * [y > 0] (b2_relu_grad_sum, which also sums gz per channel):
#     dbeta  = sum gz
#     dW     = s * R,                      R[k][c][tap] = sum_p gz[p][k] x[p*stride + tap - pad][c]   (b2_conv_ndhwc_wgrad)
#     dgamma = (sum_{c,tap} W * R - mean * sum gz) / sqrt(var + eps)       (= sum gz * x_hat, without dividing by gamma)
#     g_x    = conv(gz, flip(W * s)^T)                                      (the forward convolution kernels)
# and the residual branch receives gz of the closing layer.  dgamma never divides by gamma, so a zero gamma (a zero-initialised
# last BatchNorm of a block) gives exact gradients, and neither the pre-activation nor the residual has to be saved.
# Gradients travel between blocks as fp16 scaled by one power of two per backward pass (a device scalar, GradScale); only the
# fp32 parameter gradients are unscaled.
class TrainAct(Act):
    """The output Act of a fine-tuned trunk, carrying the GradScale its backward pass shares."""
    __slots__ = ("grad_scale",)

    def __init__(self, a, grad_scale):
        super().__init__(a.data, a.N, a.T, a.H, a.W, a.C)
        self.grad_scale = grad_scale


def trainable_layers(block):
    """[(conv, bn)] of a block in parameter order: conv1/bn1, conv2/bn2[, conv3/bn3][, type-B projection]."""
    pairs = [(block.conv1, block.bn1), (block.conv2, block.bn2)]
    if hasattr(block, "conv3"):
        pairs.append((block.conv3, block.bn3))
    if isinstance(block.downsample, nn.Sequential):
        pairs.append((block.downsample[0], block.downsample[1]))
    return pairs


def train_forward(block, a):
    """The block's forward (the frozen body's kernels and results) and the activations its backward needs."""
    if hasattr(block, "conv3"):
        h1 = conv_bn_act(block.conv1, block.bn1, a, relu=True)
        h2 = conv_bn_act(block.conv2, block.bn2, h1, relu=True)
        if _fusable_close(block, a, False):
            out = _fused_close_with_projection(block, a, h2)
        else:
            out = conv_bn_act(block.conv3, block.bn3, h2, residual=_shortcut(block, a, False), relu=True)
        return out, (h1, h2)
    h1 = conv_bn_act(block.conv1, block.bn1, a, relu=True)
    return conv_bn_act(block.conv2, block.bn2, h1, residual=_shortcut(block, a, False), relu=True), (h1,)


def _dgrad_filter(conv, bn, in_pitch):
    """PackedConv of flip(W * s)^T: the stride-1 convolution of the (dilated) output gradient that gives the input gradient."""
    def build():
        s, _ = ops.fold_affine(conv.weight.shape[0], None, bn, conv.weight.device)
        w = (conv.weight.detach().float() * s[:, None, None, None, None]).transpose(0, 1).flip(2, 3, 4).contiguous()
        return ops.PackedConv(w, None, None, (1, 1, 1), _conv_geometry(conv)[1], in_pitch=in_pitch)
    return _cached(conv, "dgrad", _sig(conv.weight, *_bn_tensors(bn)) + (in_pitch,), build)


def _dgrad(conv, bn, gz, x_geom, residual=None):
    """Input gradient of ``conv`` (x geometry (N, T, H, W, C)) from the masked output gradient ``gz``; ``residual`` (an Act of
    the input geometry) is added in the epilogue."""
    N, T, H, W, _ = x_geom
    stride = _conv_geometry(conv)[0]
    if stride != (1, 1, 1):
        if len(set(stride)) != 1:
            raise NotImplementedError("anisotropic strides have no data gradient here")
        if tuple(conv.weight.shape[2:]) == (1, 1, 1):
            raise ValueError("strided 1x1x1 data gradients go through strided_scatter_add_")
        gz = ops.zero_dilate(gz, T, H, W, stride[0])
    return ops.conv(gz, _dgrad_filter(conv, bn, gz.ld), residual=residual)


def _layer_grads(conv, bn, x, gz, gsum, scale, need_w, need_bn):
    """(dW, dgamma, dbeta) of one conv + frozen BN from its input Act ``x`` and the masked gradient ``gz`` (scaled by ``scale``)."""
    if not (need_w or need_bn):
        return None, None, None
    K, Cin = conv.weight.shape[:2]
    kt, kh, kw = conv.weight.shape[2:]
    stride, padding = _conv_geometry(conv)
    dev = gz.data.device
    R = ops.conv_wgrad(x, gz, K, (kt, kh, kw), stride, padding)
    R = R.view(K, kt, kh, kw, -1)[..., :Cin].permute(0, 4, 1, 2, 3)
    s, _ = ops.fold_affine(K, None, bn, dev)
    inv = torch.rsqrt(bn.running_var.detach().float() + bn.eps)
    dw = (R * (s / scale)[:, None, None, None, None]).contiguous() if need_w else None
    dg = db = None
    if need_bn:
        S = gsum[:K]
        dg = inv * ((conv.weight.detach().float() * R).sum((1, 2, 3, 4)) - bn.running_mean.detach().float() * S) / scale
        db = S / scale
    return dw, dg, db


def train_backward(block, x, acts, out, g, scale, need_x, need_params):
    """Gradients of one block: (g_x Act or None, [dW, dgamma, dbeta per trainable_layers(block)]).  ``x``, ``acts``, ``out``: the
    block's input, hidden activations and output (Acts); ``g``: fp16 gradient of ``out`` scaled by the device scalar ``scale``;
    ``need_params``: one flag per parameter, in the order of the returned list."""
    layers = trainable_layers(block)
    need = [need_params[3 * i:3 * i + 3] for i in range(len(layers))]
    grads = [None] * (3 * len(layers))

    def mask(y, g2d):
        gz, gsum = ops.relu_grad_sum(y.data, g2d)
        return Act(gz, y.N, y.T, y.H, y.W, y.C), gsum

    def record(i, xin, gz, gsum):
        conv, bn = layers[i]
        grads[3 * i:3 * i + 3] = _layer_grads(conv, bn, xin, gz, gsum, scale, need[i][0], need[i][1] or need[i][2])

    gz = mask(out, g)                                      # closing layer; also the residual branch's gradient
    close = gz
    hidden = [x] + list(acts)                              # input of layer i is hidden[i]
    for i in range(len(hidden) - 1, -1, -1):
        record(i, hidden[i], *gz)
        if i == 0:
            break
        conv, bn = layers[i]
        gz = mask(hidden[i], _dgrad(conv, bn, gz[0], _geom_of(hidden[i])).data)
    ds = block.downsample
    sub = None
    if isinstance(ds, nn.Sequential):
        stride = _conv_geometry(ds[0])[0][0]
        record(len(layers) - 1, x, *close)                # the patch gather subsamples x itself
        sub = ops.conv(close[0], _dgrad_filter(ds[0], ds[1], close[0].ld)) if need_x else None
    elif ds is not None:
        stride, sub = ds.stride, close[0] if need_x else None
    else:
        stride, sub = 1, close[0] if need_x else None
    if not need_x:
        return None, grads
    conv1, bn1 = layers[0]
    gx = _dgrad(conv1, bn1, gz[0], _geom_of(x), residual=sub if stride == 1 else None)
    if stride != 1:
        ops.strided_scatter_add_(gx, sub.data, ops._round_up(x.C, 8), stride)
    return gx, grads


def _geom_of(a):
    return (a.N, a.T, a.H, a.W, a.C)
