"""torch.autograd.Function wrappers around the C-ABI call sequences (SURVEY.md section 8b-ii; BASELINE.json north_star:
"exposed to Python through a thin C-ABI/ctypes shim wrapped as torch.autograd.Function").

Two kinds:

* **Frozen block bodies** -- ``StemFunction``, ``BottleneckFunction`` (resnet3D.py:125-143), ``BasicBlockFunction``
  (:91-106), ``SpatioTemporalConvFunction`` (r2plus1d.py:85-88), ``NonLocalFunction`` (nonlocalnet.py:143-243),
  ``GBlockFunction`` (BigGAN-deep GBlock).  ``forward`` is the ctypes launch sequence of ``engine.py`` /
  ``biggan_engine.py`` on fp16 NDHWC matrices; every output is marked non-differentiable, so the modules can sit inside
  an autograd graph as a frozen feature extractor (the way the reference's zoo models are used with a replaced
  ``last_linear``, README.md:520-547).  There is no backward for the convolutional trunk: asking for one raises.
* **Dense heads with a real backward** -- ``LinearFunction`` (``last_linear`` / ``fc``: resnet3D.py:162,
  torchvision_models.py:463-464) and, built from it, the TRN relation MLP (trn.py:39-49).  ``forward`` and both
  gradient products run on the same tcgen05 GEMM (``b2_gemm_f16``: fp16 operands, fp32 accumulation and output), so a
  head can be trained on engine features without leaving the library.
* **Fine-tuned residual blocks** -- ``TrainableBlockFunction`` (resnet3d ``BasicBlock`` / ``Bottleneck`` of the stages
  ``ResNet3D.enable_fine_tuning`` opens, frozen BatchNorm statistics) and ``PoolFunction`` (the global average in front of the
  head) have a backward; their gradients travel in fp16 scaled by one power of two per backward pass (``GradScale``).

Tensors cross a Function boundary as the raw ``[N*T*H*W][ld]`` fp16 matrix of an ``ops.Act`` plus its geometry tuple.
``out`` (optional, last argument of the block bodies): a preallocated ``[rows][ld]`` fp16 row range the body's LAST kernel writes
its result into -- how the depth-first trunk schedule (``engine.run_trunk``) assembles a full-batch tensor chunk by chunk.
"""
import torch

from . import ops
from .ops import Act


def _geom(a):
    return (a.N, a.T, a.H, a.W, a.C)


class _FrozenFunction(torch.autograd.Function):
    """Base: outputs are constants to autograd."""

    @staticmethod
    def backward(ctx, *grads):      # pragma: no cover - unreachable: every output is marked non-differentiable
        raise RuntimeError("pretorched_x_b200 is a forward-pass engine: the convolutional trunk has no backward "
                           "(frozen-backbone semantics); only LinearFunction / the relation MLP are differentiable")

    @classmethod
    def run(cls, module, a, *extra):
        """Act in -> Act out through ``cls.apply``."""
        data, geom = cls.apply(a.data, _geom(a), module, *extra)
        return Act(data, *geom)

    @classmethod
    def _finish(cls, ctx, out):
        ctx.mark_non_differentiable(out.data)
        return out.data, _geom(out)


class StemFunction(_FrozenFunction):
    """conv1 -> bn1 -> relu -> maxpool (torchvision_models.py:449-452).  ``x`` is the NDHWC4 / NDHWC input matrix."""

    @staticmethod
    def forward(ctx, x2d, geom, model, simt=False, out=None):
        from . import engine
        return StemFunction._finish(ctx, engine._stem_body(model, Act(x2d, *geom), simt, out))


class BottleneckFunction(_FrozenFunction):
    @staticmethod
    def forward(ctx, x2d, geom, block, simt=False, out=None):
        from . import engine
        return BottleneckFunction._finish(ctx, engine._bottleneck_body(block, Act(x2d, *geom), simt, out))


class BasicBlockFunction(_FrozenFunction):
    @staticmethod
    def forward(ctx, x2d, geom, block, simt=False, out=None):
        from . import engine
        return BasicBlockFunction._finish(ctx, engine._basic_body(block, Act(x2d, *geom), simt, out))


class PreActBlockFunction(_FrozenFunction):
    """Pre-activation residual blocks (pre_act_resnet3D.py:27-96)."""

    @staticmethod
    def forward(ctx, x2d, geom, block, simt=False, out=None):
        from . import engine
        return PreActBlockFunction._finish(ctx, engine._preact_body(block, Act(x2d, *geom), simt, out))


class SpatioTemporalConvFunction(_FrozenFunction):
    """(1,k,k) conv -> BN -> ReLU -> (k,1,1) conv [-> outer BN -> +residual -> ReLU] (r2plus1d.py:85-88)."""

    @staticmethod
    def forward(ctx, x2d, geom, conv, bn=None, residual=None, relu=False, simt=False, out=None):
        from . import engine
        return SpatioTemporalConvFunction._finish(ctx, engine._st_conv_body(conv, bn, Act(x2d, *geom), residual, relu, simt, out))


class NonLocalFunction(_FrozenFunction):
    @staticmethod
    def forward(ctx, x2d, geom, nl, simt=False, out=None):
        from . import engine
        return NonLocalFunction._finish(ctx, engine._nonlocal_body(nl, Act(x2d, *geom), simt, out))


class GBlockFunction(_FrozenFunction):
    """BigGAN-deep GBlock: ccbn-ReLU-1x1 -> ccbn-ReLU-[up]-3x3 -> ccbn-ReLU-3x3 -> ccbn-ReLU-1x1 (+ skip)."""

    @staticmethod
    def forward(ctx, x2d, geom, blk, aff, pk, kwargs):
        from . import biggan_engine
        out = biggan_engine._gblock_body(blk, Act(x2d, *geom), aff, pk, **kwargs)
        if isinstance(out, tuple):          # (block output, pre-activated input of the next block)
            ctx.mark_non_differentiable(out[0].data, out[1].data)
            return out[0].data, _geom(out[0]), out[1].data, _geom(out[1])
        ctx.mark_non_differentiable(out.data)
        return out.data, _geom(out), None, None


# ---------------------------------------------------------------------------------------------------------------
# dense head with a backward on the same GEMM kernel
# ---------------------------------------------------------------------------------------------------------------
def _f16_padded(t2d):
    """fp32 / fp16 [rows][cols] -> contiguous fp16 [rows][round_up(cols, 8)] with zero padding columns."""
    rows, cols = t2d.shape
    out = torch.zeros((rows, ops._round_up(cols, 8)), dtype=torch.float16, device=t2d.device)
    out[:, :cols] = t2d
    return out


def _unit_affine(n, dev):
    return torch.ones(n, dtype=torch.float32, device=dev), torch.zeros(n, dtype=torch.float32, device=dev)


# One power of two per backward pass, chosen so that the largest gradient entering fp16 lands in [2^7, 2^8): per-element
# gradients of a mean-reduced loss sit near 1e-6 in the last stages, where fp16 has only subnormals left, and the headroom
# below 65504 leaves room for gradients to grow through the trunk.
_GRAD_TARGET = 2.0 ** 8


def pow2_scale(amax):
    """2^floor(log2(target / amax)) as an fp32 device scalar, 1 where amax is 0 or not finite; no host synchronisation."""
    e = torch.floor(torch.log2(_GRAD_TARGET / amax.float())).clamp(-100.0, 100.0)
    return torch.where(torch.isfinite(amax) & (amax > 0), torch.exp2(e), torch.ones_like(e))


class GradScale:
    """The gradient scale one backward pass of a fine-tuned trunk shares: set by ``PoolFunction.backward`` (where the gradient
    enters the trunk) and read by every ``TrainableBlockFunction.backward`` after it."""
    __slots__ = ("value",)

    def __init__(self):
        self.value = None

    def get(self, dev):
        return self.value if self.value is not None else torch.ones((), dtype=torch.float32, device=dev)


class PoolFunction(torch.autograd.Function):
    """Global average pool of a fine-tuned trunk's output -> fp32 [N][C] (exactly the fp16 values the frozen head pools).
    Backward: the scaled fp16 gradient of every position, g / (T*H*W) * scale."""

    @staticmethod
    def forward(ctx, x2d, geom, grad_scale):
        from .ops import avgpool_global
        ctx.geom, ctx.ld, ctx.grad_scale = geom, x2d.shape[1], grad_scale
        return avgpool_global(Act(x2d, *geom))[:, :geom[4]].float()

    @staticmethod
    def backward(ctx, g):
        N, T, H, W, C = ctx.geom
        P = T * H * W
        g = g / P
        s = pow2_scale(g.abs().amax())
        ctx.grad_scale.value = s
        gx = torch.zeros((N, P, ctx.ld), dtype=torch.float16, device=g.device)
        gx[:, :, :C] = (g * s).to(torch.float16)[:, None, :]
        return gx.view(N * P, ctx.ld), None, None


class TrainableBlockFunction(torch.autograd.Function):
    """A resnet3d BasicBlock / Bottleneck with a backward (frozen BatchNorm statistics; engine.train_backward).  The
    parameters of ``engine.trainable_layers(block)`` (conv weight, BN weight, BN bias per layer) are inputs, so autograd
    hands their gradients to them; the gradient of the output travels scaled by ``grad_scale``."""

    @staticmethod
    def forward(ctx, x2d, geom, block, grad_scale, *params):
        from . import engine
        x = Act(x2d, *geom)
        out, acts = engine.train_forward(block, x)
        ctx.block, ctx.grad_scale = block, grad_scale
        ctx.geoms = [geom] + [_geom(h) for h in acts] + [_geom(out)]
        ctx.save_for_backward(x2d, *[h.data for h in acts], out.data)
        return out.data, _geom(out)

    @staticmethod
    def backward(ctx, g, _):
        from . import engine
        saved = ctx.saved_tensors
        acts = [Act(t, *gm) for t, gm in zip(saved, ctx.geoms)]
        gx, grads = engine.train_backward(ctx.block, acts[0], acts[1:-1], acts[-1], g.contiguous(), ctx.grad_scale.get(g.device),
                                          ctx.needs_input_grad[0], ctx.needs_input_grad[4:])
        return (gx.data if gx is not None else None, None, None, None) + tuple(grads)

    @classmethod
    def run(cls, block, a, grad_scale):
        from . import engine
        params = [t for conv, bn in engine.trainable_layers(block) for t in (conv.weight, bn.weight, bn.bias)]
        data, geom = cls.apply(a.data, _geom(a), block, grad_scale, *params)
        return Act(data, *geom)


class LinearFunction(torch.autograd.Function):
    """y = x W^T + b on tcgen05 (fp16 operands, fp32 accumulate / output), with
    dL/dx = g W, dL/dW = g^T x, dL/db = sum_rows g computed by the same kernel (D = A . B^T with K-major operands:
    the gradient products take the transposed fp16 copies as their operands)."""

    @staticmethod
    def forward(ctx, x, weight, bias, relu_input=False):
        if x.dim() != 2:
            raise ValueError("LinearFunction takes a [rows][features] matrix")
        x16 = ops.cast_rows(x, relu=relu_input) if x.dtype != torch.float16 else x
        pl = ops.PackedLinear(weight, bias)
        y = ops.linear(x16, pl, out_f32=True)
        ctx.save_for_backward(x16, weight)
        ctx.has_bias = bias is not None
        ctx.relu_input = relu_input
        ctx.in_features = weight.shape[1]
        return y

    @staticmethod
    def backward(ctx, gy):
        x16, weight = ctx.saved_tensors
        dev = gy.device
        rows, out_f = gy.shape
        in_f = ctx.in_features
        gx = gw = gb = None
        s = pow2_scale(gy.abs().amax())                                  # gy is cast to fp16 scaled, the fp32 products unscaled
        g16 = _f16_padded(gy * s)                                        # [rows][out_p]
        if ctx.needs_input_grad[0]:
            wt = _f16_padded(weight.detach().t())                        # [in][out_p]: B operand, K = out
            one, zero = _unit_affine(in_f, dev)
            gx = ops.gemm(g16, wt, one, zero, rows, in_f, out_f, out_f32=True) / s
            if ctx.relu_input:
                gx = gx * (x16[:, :in_f] > 0)
        if ctx.needs_input_grad[1]:
            gt = _f16_padded((gy * s).t())                               # [out][rows_p]: A operand, K = rows
            xt = _f16_padded(x16[:, :in_f].t())                          # [in][rows_p]
            one, zero = _unit_affine(in_f, dev)
            gw = ops.gemm(gt, xt, one, zero, out_f, in_f, rows, out_f32=True) / s
        if ctx.has_bias and ctx.needs_input_grad[2]:
            gb = gy.sum(0)
        return gx, gw, gb, None


def linear(x, weight, bias=None, relu_input=False):
    return LinearFunction.apply(x, weight, bias, relu_input)
