"""Fine-tuning surface without a GPU: the reference's parameter-group rule, enable_fine_tuning's validation, and the
flip / transpose / dilate algebra the block backward's data gradient rests on."""
import pytest
import torch
import torch.nn.functional as F

import pretorched_x_b200 as P
from pretorched_x_b200.models.resnet3d import get_fine_tuning_parameters


def _reference_rule(model, ft_begin_index, head):
    """resnet3D.py:221-239 restated, with the head under this model's name."""
    names = ['layer%d' % i for i in range(ft_begin_index, 5)] + [head]
    out = []
    for k, v in model.named_parameters():
        out.append((k, v, any(n in k for n in names)))
    return out


@pytest.mark.parametrize("factory", [P.resnet3d18, P.resnet3d50])
@pytest.mark.parametrize("ft", range(0, 6))
def test_get_fine_tuning_parameters_matches_reference_rule(factory, ft):
    m = factory(num_classes=10, pretrained=None)
    before = {k: v.clone() for k, v in m.state_dict().items()}
    groups = get_fine_tuning_parameters(m, ft)
    if ft == 0:
        assert [id(p) for p in groups] == [id(p) for p in m.parameters()]
        return
    want = _reference_rule(m, ft, 'last_linear')
    assert len(groups) == len(want)
    for g, (k, v, trained) in zip(groups, want):
        assert g['params'] is v, k
        assert ('lr' in g) != trained, k
        if not trained:
            assert g['lr'] == 0.0
    assert any('last_linear' in k and t for k, _, t in want)
    assert all(torch.equal(before[k], v) for k, v in m.state_dict().items())
    torch.optim.SGD(groups, lr=0.1)             # the groups are valid optimizer input


def test_get_fine_tuning_parameters_uses_fc_for_fc_heads():
    m = P.r2plus1d18(num_classes=10)
    assert m.head_name == 'fc'
    groups = get_fine_tuning_parameters(m, 4)
    names = [k for k, _ in m.named_parameters()]
    trained = [k for k, g in zip(names, groups) if 'lr' not in g]
    assert 'fc.weight' in trained and 'fc.bias' in trained
    assert all(k.startswith(('layer4', 'fc')) for k in trained)


def test_enable_fine_tuning_validation():
    m = P.resnet3d18(num_classes=10, pretrained=None)
    with pytest.raises(NotImplementedError):
        m.enable_fine_tuning(0)
    with pytest.raises(ValueError):
        m.enable_fine_tuning(6)
    assert m.enable_fine_tuning(3) is m and m._b2_ft_begin == 3
    assert m.enable_fine_tuning(5)._b2_ft_begin is None
    assert m.enable_fine_tuning(None)._b2_ft_begin is None
    P.resnet3d50(num_classes=10, pretrained=None).enable_fine_tuning(1)


@pytest.mark.parametrize("factory, name", [
    (lambda: P.r2plus1d18(num_classes=10), "BasicBlock"),
    (lambda: P.preact_resnet3d18(num_classes=10), "PreActivationBasicBlock"),
    (lambda: P.resnext3d50(num_classes=10), "ResNeXtBottleneck"),
])
def test_enable_fine_tuning_rejects_other_blocks(factory, name):
    m = factory()
    with pytest.raises(NotImplementedError, match=name):
        m.enable_fine_tuning(4)


def _dgrad_by_algebra(g, w, stride, in_shape):
    """The block backward's data gradient in plain torch: dilate g into the input geometry (stride 2), then a stride-1
    'same' convolution with the spatially flipped, channel-transposed filter."""
    pad = w.shape[-1] // 2
    if stride != 1:
        d = g.new_zeros(g.shape[:2] + tuple(in_shape[2:]))
        d[:, :, ::stride, ::stride, ::stride] = g
        g = d
    return F.conv3d(g, w.transpose(0, 1).flip(2, 3, 4), padding=pad)


@pytest.mark.parametrize("k", [1, 3])
@pytest.mark.parametrize("stride", [1, 2])
@pytest.mark.parametrize("extent", [(4, 7, 7), (3, 8, 6), (1, 5, 4)])
def test_dgrad_flip_transpose_dilate_algebra(k, stride, extent):
    torch.manual_seed(0)
    x = torch.randn((2, 5) + extent, dtype=torch.float64)
    w = torch.randn(6, 5, k, k, k, dtype=torch.float64)
    pad = k // 2
    y = F.conv3d(x, w, stride=stride, padding=pad)
    g = torch.randn_like(y)
    if k == 1 and stride != 1:
        # strided 1x1x1: a 1x1x1 product on the subsampled positions, scattered back (strided_scatter_add)
        got = x.new_zeros(x.shape)
        got[:, :, ::stride, ::stride, ::stride] = torch.einsum('nkthw,kc->ncthw', g, w[:, :, 0, 0, 0])
    else:
        got = _dgrad_by_algebra(g, w, stride, x.shape)
    want = F.conv_transpose3d(g, w, stride=stride, padding=pad, output_padding=tuple(
        i - ((o - 1) * stride - 2 * pad + k) for i, o in zip(extent, y.shape[2:])))
    assert got.shape == want.shape
    assert torch.allclose(got, want, atol=1e-10)


def _conv_layers(model):
    """(conv, input T, H, W) of every convolution in layers 1-4 for a 16x112x112 clip."""
    T, H = 8, 28                              # after the stem (stride 1, 2, 2) and the 3x3x3 / 2 pool
    out = []
    for li in range(1, 5):
        for blk in getattr(model, "layer%d" % li):
            s = blk.stride
            convs = [(blk.conv1, (T, H)), (blk.conv2, (T, H) if hasattr(blk, "conv3") else ((T - 1) // s + 1, (H - 1) // s + 1))]
            if hasattr(blk, "conv3"):
                T2, H2 = (T - 1) // s + 1, (H - 1) // s + 1
                convs = [(blk.conv1, (T, H)), (blk.conv2, (T, H)), (blk.conv3, (T2, H2))]
            if isinstance(blk.downsample, torch.nn.Sequential):
                convs.append((blk.downsample[0], (T, H)))
            out += convs
            T, H = (T - 1) // s + 1, (H - 1) // s + 1
    return out


@pytest.mark.parametrize("factory", [P.resnet3d18, P.resnet3d50])
@pytest.mark.parametrize("clips", [1, 2, 32])
def test_wgrad_plan_covers_every_tile_and_partitions_positions(factory, clips):
    from pretorched_x_b200 import _lib
    m = factory(num_classes=10, pretrained=None)
    seen = set()
    for conv, (T, H) in _conv_layers(m):
        K, C, kt, kh, kw = conv.weight.shape
        st, pd = conv.stride[0], conv.padding[0]
        a = _lib.WgradArgs()
        a.x = a.g = a.dw = 16
        a.N, a.T, a.H, a.W, a.ldx, a.C, a.ldg, a.K = clips, T, H, H, C, C, K, K
        a.kt, a.kh, a.kw, a.st, a.sh, a.sw, a.pt, a.ph, a.pw = kt, kh, kw, st, st, st, pd, pd, pd
        key = (K, C, kt, st, T, H)
        if key in seen:
            continue
        seen.add(key)
        plan = _lib.wgrad_plan(a)
        To, Ho = (T + 2 * pd - kt) // st + 1, (H + 2 * pd - kh) // st + 1
        # every (filter tile, tap, channel tile) is one CTA column of the grid, once
        assert plan["mt"] * 128 >= K > (plan["mt"] - 1) * 128 and plan["nt"] * 128 >= C > (plan["nt"] - 1) * 128
        assert plan["taps"] == kt * kh * kw and plan["grid_x"] == plan["mt"] * plan["taps"] * plan["nt"]
        # 8x8 rectangles of output positions, per (n, t) plane
        assert plan["rect_cols"] * 8 >= Ho and plan["rect_rows"] * 8 >= Ho
        assert plan["rects"] == clips * To * plan["rect_cols"] * plan["rect_rows"]
        # the split ranges partition the rectangles
        assert plan["grid_y"] == plan["splits"] == len(plan["ranges"])
        assert plan["ranges"][0][0] == 0 and plan["ranges"][-1][1] == plan["rects"]
        assert all(r1 == r0n for (_, r1), (r0n, _) in zip(plan["ranges"], plan["ranges"][1:]))
        assert all(r1 > r0 for r0, r1 in plan["ranges"])
        # shared memory within the opt-in limit of a B200 block
        assert plan["smem"] + 1024 <= 227 * 1024
