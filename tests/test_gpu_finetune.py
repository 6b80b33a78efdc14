"""Fine-tuning on the GPU: the backward kernels against torch, one block's gradients and whole-model gradients against CPU
fp32 autograd through oracle.functional (same fp16-rounded inputs and weights), gradient scaling and an SGD step."""
import pytest
import torch
import torch.nn.functional as F

import pretorched_x_b200 as P
from pretorched_x_b200 import engine, functions as Fn, ops
from pretorched_x_b200.models import resnet3d as R
from pretorched_x_b200.models.resnet3d import get_fine_tuning_parameters
from oracle import functional as OF

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
TOL = 1e-2


def _rel(got, want):
    got, want = got.detach().double().cpu(), want.detach().double().cpu()
    return (got - want).abs().max().item() / max(want.abs().max().item(), 1e-30)


def _act(x):
    """fp32 NCDHW (CPU) -> Act on the GPU."""
    return ops.from_ncdhw(x.to(DEV), pitch=ops._round_up(x.shape[1], 8))


def _rows(t):
    """NCDHW -> [N*T*H*W][C] (the Act row order)."""
    return t.permute(0, 2, 3, 4, 1).reshape(-1, t.shape[1])


# ---------------------------------------------------------------------------------------------
# kernels
# ---------------------------------------------------------------------------------------------
def test_relu_grad_sum_matches_torch_and_is_deterministic():
    g0 = torch.Generator().manual_seed(1)
    y = torch.randn(5003, 264, generator=g0).clamp(min=0).half().to(DEV)
    g = torch.randn(5003, 264, generator=g0).half().to(DEV)
    gz, s = ops.relu_grad_sum(y, g)
    want = torch.where(y > 0, g, torch.zeros_like(g))
    assert torch.equal(gz, want)
    assert _rel(s, want.double().sum(0)) < 1e-5
    gz2, s2 = ops.relu_grad_sum(y, g)
    assert torch.equal(s, s2) and torch.equal(gz, gz2)


@pytest.mark.parametrize("N, C, K, T, H, W, k, s", [
    (2, 256, 64, 4, 14, 14, 1, 1),          # 1x1x1 C256 -> 64
    (1, 2048, 512, 2, 7, 7, 1, 1),          # layer4's 1x1x1 C2048 -> 512
    (2, 64, 64, 3, 14, 14, 3, 1),           # 3x3x3, odd T
    (1, 128, 128, 4, 7, 7, 3, 1),
    (1, 512, 512, 2, 7, 7, 3, 1),
    (2, 128, 128, 5, 14, 14, 3, 2),         # 3x3x3 stride 2
    (2, 64, 128, 4, 14, 14, 1, 2),          # strided projection
    (3, 64, 64, 3, 9, 11, 3, 2),            # odd extents, ragged rectangles
])
def test_weight_gradient_matches_conv3d_weight(N, C, K, T, H, W, k, s):
    g0 = torch.Generator().manual_seed(2)
    x = torch.randn(N, C, T, H, W, generator=g0).half().float()
    p = k // 2
    To, Ho, Wo = [(e + 2 * p - k) // s + 1 for e in (T, H, W)]
    gy = torch.randn(N, K, To, Ho, Wo, generator=g0).half().float()
    want = torch.nn.grad.conv3d_weight(x, (K, C, k, k, k), gy, stride=s, padding=p)
    xa = ops.from_ncdhw(x.to(DEV), pitch=C + 8 if C == 64 else C)          # ld > C
    ga = _act(gy)
    outs = [ops.conv_wgrad(xa, ga, K, (k,) * 3, (s,) * 3, (p,) * 3) for _ in range(2)]
    torch.cuda.synchronize()
    assert torch.equal(outs[0], outs[1])
    got = outs[0].view(K, k, k, k, C).permute(0, 4, 1, 2, 3)
    assert _rel(got, want) <= 2e-3


def test_zero_dilate_and_strided_scatter_add():
    g0 = torch.Generator().manual_seed(3)
    g = torch.randn(2, 16, 3, 4, 4, generator=g0).half().float()
    a = _act(g)
    d = ops.zero_dilate(a, 5, 7, 8, 2)
    want = torch.zeros(2, 16, 5, 7, 8)
    want[:, :, ::2, ::2, ::2] = g
    assert torch.equal(ops.to_ncdhw(d).cpu(), want)
    base = torch.randn(2, 16, 5, 7, 8, generator=g0).half().float()
    y = _act(base)
    ops.strided_scatter_add_(y, a.data, 16, 2)
    want = base.clone()
    want[:, :, ::2, ::2, ::2] += g
    assert _rel(ops.to_ncdhw(y).cpu(), want) < 1e-3


# ---------------------------------------------------------------------------------------------
# one block
# ---------------------------------------------------------------------------------------------
# The references are CPU fp32 autograd through oracle.functional's primitives on the same fp16-rounded inputs and weights,
# evaluated at the engine's own forward activations: every ReLU takes its mask from the engine's fp16 output and its value is
# snapped to it (identity gradient through the snap).  Otherwise units within fp16 precision of zero take the other side of a
# ReLU than in the engine's forward, and with the few positions per channel of these shapes one such unit moves a gradient
# entry by a whole term -- a forward difference, not a backward one (the forward is checked against the oracle elsewhere).
def _at(z, y):
    """relu(z) with the mask and the value of the engine's output y (fp32 NCDHW)."""
    r = z * (y > 0)
    return r + (y - r).detach()


def _engine_acts(blk, a):
    """(output Act, [hidden activations..., output] as fp32 NCDHW on the CPU) of one block's trainable forward."""
    with torch.no_grad():
        out, acts = engine.train_forward(blk, a)
    return out, [ops.to_ncdhw(h).cpu() for h in list(acts) + [out]]


def _ref_block(x, sd, p, kind, shortcut, planes, stride, has_ds, acts):
    if kind == "bottleneck":
        h = _at(OF._bn(OF._conv(x, sd, p + '.conv1'), sd, p + '.bn1'), acts[0])
        h = _at(OF._bn(OF._conv(h, sd, p + '.conv2', stride, 1), sd, p + '.bn2'), acts[1])
        out, cout = OF._bn(OF._conv(h, sd, p + '.conv3'), sd, p + '.bn3'), planes * 4
    else:
        h = _at(OF._bn(OF._conv(x, sd, p + '.conv1', stride, 1), sd, p + '.bn1'), acts[0])
        out, cout = OF._bn(OF._conv(h, sd, p + '.conv2', 1, 1), sd, p + '.bn2'), planes
    return _at(out + OF._residual(x, sd, p, 'resnet3d', shortcut, cout, stride, has_ds), acts[-1])


def _block_spec(blk):
    kind = "bottleneck" if hasattr(blk, "conv3") else "basic"
    shortcut = "A" if isinstance(blk.downsample, R.ShortcutA) else "B"
    return kind, shortcut, blk.conv1.out_channels, blk.stride, blk.downsample is not None


def _round_params_(m):
    with torch.no_grad():
        for mod in m.modules():
            if isinstance(mod, torch.nn.Conv3d):
                mod.weight.copy_(mod.weight.half().float())
    return m


def _block(kind, shortcut, stride, cin, planes, zero_gamma=False):
    ds = None
    block = R.Bottleneck if kind == "bottleneck" else R.BasicBlock
    cout = planes * block.expansion
    if stride != 1 or cin != cout:
        ds = R.ShortcutA(cout, stride) if shortcut == "A" else torch.nn.Sequential(
            torch.nn.Conv3d(cin, cout, 1, stride=stride, bias=False), torch.nn.BatchNorm3d(cout))
    torch.manual_seed(4)
    m = block(cin, planes, stride, ds)
    OF.randomize_bn_(m, 5)
    if zero_gamma:
        last = m.bn3 if kind == "bottleneck" else m.bn2
        with torch.no_grad():
            last.weight[0] = 0.0
    return _round_params_(m).eval(), ds is not None


@pytest.mark.parametrize("kind, shortcut, stride, cin, planes, zero_gamma", [
    ("basic", "A", 1, 64, 64, False),
    ("basic", "A", 2, 64, 128, False),
    ("bottleneck", "B", 1, 64, 64, False),
    ("bottleneck", "B", 2, 256, 128, False),
    ("bottleneck", "B", 1, 256, 64, False),          # no shortcut
    ("bottleneck", "B", 1, 256, 64, True),           # one channel with gamma = 0
])
def test_block_gradients_match_cpu_autograd(kind, shortcut, stride, cin, planes, zero_gamma):
    m, has_ds = _block(kind, shortcut, stride, cin, planes, zero_gamma)
    g0 = torch.Generator().manual_seed(6)
    x = torch.randn(2, cin, 4, 10, 10, generator=g0).clamp(min=0).half().float()
    # CPU fp32 reference
    params = dict(m.named_parameters())
    sd = {"b." + k: v.detach().clone().requires_grad_(k in params) for k, v in m.state_dict().items()}
    xr = x.clone().requires_grad_(True)
    md = m.to(DEV)
    a = _act(x)
    _, acts = _engine_acts(md, a)
    ref = _ref_block(xr, sd, "b", kind, shortcut, planes, stride, has_ds, acts)
    G = torch.randn(ref.shape, generator=g0)
    (ref * G).sum().backward()
    # GPU
    a.data.requires_grad_(True)
    out = Fn.TrainableBlockFunction.run(md, a, Fn.GradScale())
    assert _rel(out.data[:, :out.C].float(), _rows(ref.detach())) < TOL
    (out.data[:, :out.C].float() * _rows(G).to(DEV)).sum().backward()
    names = dict(md.named_parameters())
    for k, v in names.items():
        want = sd["b." + k].grad
        assert v.grad is not None, k
        assert _rel(v.grad, want) <= TOL, (k, _rel(v.grad, want))
    assert _rel(a.data.grad[:, :cin], _rows(xr.grad)) <= TOL


# ---------------------------------------------------------------------------------------------
# whole models
# ---------------------------------------------------------------------------------------------
def _model(name):
    torch.manual_seed(7)
    m = getattr(P, name)(num_classes=10, pretrained=None)
    OF.randomize_bn_(m, 8)
    return _round_params_(m).eval()


def _reference_grads(m, md, xd, y, ft):
    """CPU fp32 autograd of layer{ft}..layer4 + head from the engine's own (frozen) input to layer{ft}, at its activations."""
    with torch.no_grad():
        a = engine.run_stem(md, xd)
        for i in range(1, ft):
            for blk in getattr(md, "layer%d" % i):
                a = engine.run_block(blk, a)
        feat = ops.to_ncdhw(a).cpu()
    params = dict(m.named_parameters())
    sd = {k: v.detach().cpu().clone().requires_grad_(k in params) for k, v in m.state_dict().items()}
    for i in range(ft, 5):
        for j, blk in enumerate(getattr(md, "layer%d" % i)):
            a, acts = _engine_acts(blk, a)
            kind, shortcut, planes, stride, has_ds = _block_spec(blk)
            feat = _ref_block(feat, sd, "layer%d.%d" % (i, j), kind, shortcut, planes, stride, has_ds, acts)
    F.cross_entropy(OF.head(feat, sd), y).backward()
    return sd


def _trained(k, ft):
    return any(k.startswith("layer%d." % i) for i in range(ft, 5)) or k.startswith("last_linear")


@pytest.mark.parametrize("name", ["resnet3d18", "resnet3d50"])
@pytest.mark.parametrize("ft", [4, 3])
def test_model_gradients_match_cpu_autograd(name, ft):
    m = _model(name)
    g0 = torch.Generator().manual_seed(9)
    x = torch.randn(2, 3, 8, 64, 64, generator=g0).half().float()
    y = torch.tensor([1, 7])
    md = m.to(DEV).enable_fine_tuning(ft)
    xd = x.to(DEV).requires_grad_(True)
    sd = _reference_grads(m, md, xd, y, ft)
    F.cross_entropy(md(xd), y.to(DEV)).backward()
    grads = {k: v.grad for k, v in md.named_parameters()}
    for k, g in grads.items():
        if _trained(k, ft):
            assert g is not None, k
            assert _rel(g, sd[k].grad) <= TOL, (k, _rel(g, sd[k].grad))
        else:
            assert g is None, k
    assert xd.grad is None
    # the same loss x 1e-6: nothing flushes, gradients scale
    md.zero_grad(set_to_none=True)
    (F.cross_entropy(md(xd), y.to(DEV)) * 1e-6).backward()
    for k, v in md.named_parameters():
        if _trained(k, ft):
            assert _rel(v.grad, grads[k] * 1e-6) <= TOL, k


def test_sgd_step_reaches_next_forward():
    m = _model("resnet3d50").to(DEV).enable_fine_tuning(4)
    g0 = torch.Generator().manual_seed(10)
    x = torch.randn(2, 3, 8, 64, 64, generator=g0).to(DEV)
    before = {k: v.detach().clone() for k, v in m.named_parameters()}
    opt = torch.optim.SGD(get_fine_tuning_parameters(m, 4), lr=1e-3)
    with torch.no_grad():
        old = m(x)
    sd_old = {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}
    F.cross_entropy(m(x), torch.tensor([2, 3], device=DEV)).backward()
    opt.step()
    for k, v in m.named_parameters():
        if _trained(k, 4):
            assert not torch.equal(v.detach(), before[k]), k
        else:
            assert torch.equal(v.detach(), before[k]), k
    with torch.no_grad():
        got = m(x)
        want = OF.forward(x.cpu(), {k: v.cpu() for k, v in m.state_dict().items()}, "resnet3d50")
    assert _rel(got, want) <= 5e-3
    # the trunk alone (the head is not cached) follows the updated layer4 weights: its features match the oracle on the new
    # state dict, and the step moved them by several times that error, so stale packed filters would have been caught
    with torch.no_grad():
        feat = m.features(x).cpu()
    stale = OF.trunk(x.cpu(), sd_old, "resnet3d50")
    fresh = OF.trunk(x.cpu(), {k: v.cpu() for k, v in m.state_dict().items()}, "resnet3d50")
    err = _rel(feat, fresh)
    assert err <= 5e-3 and _rel(fresh, stale) > 4 * err and _rel(feat, stale) > 2 * err
    assert not torch.equal(got, old)
