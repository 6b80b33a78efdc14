"""CPU: host-side logic of the drop-in boundary -- factory registry, state_dict layout, reference quirks,
BN folding, sharding arithmetic, and loud failure without a GPU."""
import math

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

import pretorched_x_b200 as P
from pretorched_x_b200 import ops, parallel
from pretorched_x_b200.models import r2plus1d, nonlocalnet
from oracle import functional as OF


def test_factory_registry_matches_reference_names():
    for name in ["resnet18", "resnet3d10", "resnet3d18", "resnet3d34", "resnet3d50", "resnet3d101", "resnet3d152",
                 "resnet3d200", "resneti3d50", "nonlocalresnet3d18", "nonlocalresnet3d34", "nonlocalresnet3d50",
                 "nonlocalresnet3d101"]:
        assert callable(P.__dict__[name]), name
    s = P.pretrained_settings["resnet3d50"]["kinetics-400"]
    assert s["num_classes"] == 400 and s["input_size"] == [3, 224, 224] and s["mean"] == [0.485, 0.456, 0.406]
    assert P.pretrained_settings["resnet3d50"]["moments"]["num_classes"] == 339
    assert "resnet3d50" in P.model_names and "resnet18" in P.model_names


def test_resnet3d50_state_dict_layout():
    m = P.resnet3d50(num_classes=400, pretrained=None)
    sd = m.state_dict()
    assert len(sd) == 320                                   # SURVEY.md 8b
    assert tuple(sd["conv1.weight"].shape) == (64, 3, 7, 7, 7)
    assert tuple(sd["layer2.0.downsample.0.weight"].shape) == (512, 256, 1, 1, 1)
    assert tuple(sd["last_linear.weight"].shape) == (400, 2048) and m.fc is None
    assert not any(k.startswith("fc.") for k in sd)


def test_zoo_checkpoints_with_fc_keys_load():
    m = P.resnet3d10(num_classes=7)
    sd = {k.replace("last_linear.", "fc."): v.clone() for k, v in m.state_dict().items()}
    sd["fc.bias"] += 1.0
    m2 = P.resnet3d10(num_classes=7)
    m2.load_state_dict(sd)
    assert torch.equal(m2.last_linear.bias, sd.get("fc.bias", m2.last_linear.bias))


def test_pretrained_asserts_num_classes_before_download():
    with pytest.raises(AssertionError):
        P.resnet3d50(num_classes=10, pretrained="kinetics-400")


def test_r2plus1d_layout_and_quirks():
    assert r2plus1d.intermediate_channels(3, 64, (7, 7, 7)) == 110       # SURVEY appendix C
    assert r2plus1d.intermediate_channels(64, 64, (3, 3, 3)) == 144
    assert r2plus1d.intermediate_channels(64, 128, (1, 1, 1)) == 42
    P.resnet3d10()                                                       # would break the reference's R2Plus1D
    m = P.r2plus1d34(num_classes=400)
    sd = m.state_dict()
    assert len(sd) == 434
    assert tuple(sd["conv1.spatial_conv.weight"].shape) == (110, 3, 1, 7, 7)
    assert tuple(sd["conv1.temporal_conv.weight"].shape) == (64, 110, 7, 1, 1)
    assert tuple(sd["fc.weight"].shape) == (400, 512) and m.last_linear is m.fc
    m.last_linear = P.Identity()
    assert isinstance(m.fc, P.Identity) and "last_linear" not in dict(m.named_children())


def test_nonlocal_quirks():
    m = P.nonlocalresnet3d50(num_classes=10, pretrained=None)            # num_classes is swallowed upstream
    assert m.last_linear.out_features == 339
    sd = m.state_dict()
    assert not any("downsample" in k for k in sd)                        # type-A shortcuts, no parameters
    nl = [k.split(".nonlocalblock")[0] for k in sd if k.endswith("nonlocalblock.g.weight")]
    assert nl == ["layer2.0", "layer2.2", "layer3.0", "layer3.2", "layer3.4"]
    assert float(m.layer2[0].nonlocalblock.W[1].weight.abs().mean()) == 1.0   # init_weights overrides the zero init
    assert OF.nonlocal_positions([3, 4, 6, 3], [0, 2, 3, 0]) == [[], [0, 2], [0, 2, 4], []]
    cat = nonlocalnet.NonLocalBlock3D(64, mode="concatenation")               # nonlocalnet.py:117-121: 2d -> 1 projection, no bias
    assert tuple(cat.state_dict()["concat_project.0.weight"].shape) == (1, 64, 1, 1) and "concat_project.0.bias" not in cat.state_dict()
    sub = nonlocalnet.NonLocalBlock2D(64, mode="gaussian", sub_sample=True)     # reference layout with sub_sample
    assert set(sub.state_dict()) >= {"g.0.weight", "g.0.bias", "W.0.weight", "W.1.running_mean"}
    assert "theta.weight" not in sub.state_dict()


def test_trn_upstream_defects_are_explicit():
    with pytest.raises(NotImplementedError):
        P.HierarchicalRelation(8, 16, 8, relation_size=4)
    h = P.HierarchicalRelation(8, 16, 8, relation_size=1024)             # what TRN(consensus='HTRN') builds
    assert h.final_relation.bottleneck_dim == 512


def test_fold_affine_equals_eval_batchnorm():
    torch.manual_seed(0)
    bn = nn.BatchNorm3d(12)
    OF.randomize_bn_(bn, 5)
    bn.eval()
    bias = torch.randn(12)
    scale, shift = ops.fold_affine(12, bias, bn, torch.device("cpu"))
    x = torch.randn(2, 12, 3, 4, 5)
    want = bn(x + bias.view(1, -1, 1, 1, 1))
    got = x * scale.view(1, -1, 1, 1, 1) + shift.view(1, -1, 1, 1, 1)
    assert torch.allclose(got, want, atol=1e-5, rtol=1e-5)
    bn.train()
    with pytest.raises(RuntimeError):
        ops.fold_affine(12, None, bn, torch.device("cpu"))


def test_forward_fails_loudly_without_gpu():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    m = P.resnet3d10(num_classes=5).eval()
    with pytest.raises(RuntimeError, match="no CPU path"):
        m(torch.randn(1, 3, 4, 32, 32))
    m.train()
    with pytest.raises(RuntimeError, match="inference-only"):
        m(torch.randn(1, 3, 4, 32, 32))


def test_shard_bounds_cover_batch_exactly():
    for total in (1, 7, 16, 32, 33, 64):
        for world in (1, 2, 4, 8):
            spans = [parallel.shard_bounds(total, world, r) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == total
            assert all(spans[i][1] == spans[i + 1][0] for i in range(world - 1))
            sizes = [b - a for a, b in spans]
            assert max(sizes) - min(sizes) <= 1


def _conv_plan(N, C, T, H, W, K, k, s=(1, 1, 1), pad=None):
    """The plan b2_conv_ndhwc_fprop would launch for a BN + ReLU convolution of these dimensions (host code, no GPU needed)."""
    from pretorched_x_b200 import _lib
    a = _lib.ConvArgs()
    a.x = a.w = a.scale = a.shift = a.y = 1 << 20               # never dereferenced: the probe plans, it does not launch
    a.N, a.T, a.H, a.W, a.C, a.K = N, T, H, W, (C + 7) // 8 * 8, K
    a.ldy = (K + 7) // 8 * 8
    a.kt, a.kh, a.kw = k
    a.st, a.sh, a.sw = s
    a.pt, a.ph, a.pw = pad if pad is not None else (k[0] // 2, k[1] // 2, k[2] // 2)
    return _lib.conv_plan(a)


def test_conv_plan_slab_tiling():
    """The slab kernels' tiling decision (N tile, M tiles per item, slab rows, W chunking) is pure host code behind a debug entry
    point: the shapes of the BASELINE nets must be accepted with a plan that fits TMEM (MT * N <= 512 columns)."""
    plan = _conv_plan
    p = plan(32, 64, 8, 56, 56, 64, (3, 3, 3))                     # resnet3d50 layer1 conv2: the temporal-group slab kernel
    assert p["kernel"] == "slabts" and p["bn"] == 64 and 1 <= p["MT"] <= 4 and p["PW"] == 58 and p["wchunks"] == 1
    p = plan(16, 64, 16, 28, 28, 144, (1, 3, 3))                   # R(2+1)D layer1 spatial: runtime N tile of 144 columns
    assert p["kernel"] == "slab<0>" and p["flex"] and p["bn"] == 144 and p["MT"] * 160 <= 512
    p = plan(2, 144, 16, 28, 28, 64, (3, 1, 1))                    # temporal conv: remapped to frames x positions, 64-wide chunks
    assert p["kernel"] == "slab<64>" and p["remap"] and p["WC"] <= 64 and p["wchunks"] >= 13
    assert plan(16, 144, 16, 28, 28, 64, (3, 1, 1))["kernel"] == "tstack"   # its BASELINE-batch twin: the temporal stack kernel
    p = plan(1, 64, 1, 6, 300, 64, (1, 3, 3))                      # rows longer than a TMA box are cut into W chunks
    assert p["kernel"] == "slab<64>" and p["wchunks"] >= 2 and p["PW"] <= 256
    assert plan(2, 64, 4, 8, 8, 256, (1, 1, 1))["kernel"] == "pgemm<128,0>"   # 1x1x1: persistent GEMM, not the slab kernel


def test_conv_plan_temporal_stack():
    """Which convolutions the temporal stack kernel (b2_tstack.cuh) takes, and with what decomposition: pure host code behind a debug
    entry point.  The 64-wide temporal halves of R(2+1)D-34 at the BASELINE batch are taken with the filter resident; launches with
    less than one work item per SM, wider outputs, strided / spatial filters and filters too big to stay resident are not."""
    from pretorched_x_b200 import _lib
    lib = _lib.load()
    plan = _conv_plan
    lib.b2_debug_set_tstack(-1)
    p = plan(16, 110, 32, 56, 56, 64, (7, 1, 1))                   # R(2+1)D stem, temporal half: 8 groups of 4 frames x 25 tiles x 16 clips
    assert p["kernel"] == "tstack" and (p["items"], p["groups"], p["tiles"], p["cchunks"]) == (3200, 8, 25, 2)
    assert p["wbytes"] == 2 * 7 * 8192 and p["smem"] <= 227 * 1024
    p = plan(16, 144, 16, 28, 28, 64, (3, 1, 1))                   # layer1 temporal halves: 3 channel chunks, 72 KB filter
    assert p["kernel"] == "tstack" and (p["items"], p["groups"], p["tiles"], p["cchunks"], p["wbytes"]) == (448, 4, 7, 3, 73728)
    assert plan(2, 144, 16, 28, 28, 64, (3, 1, 1))["kernel"] == "slab<64>"     # 56 items < one per SM: the slab kernel keeps more SMs busy
    assert plan(16, 288, 8, 14, 14, 128, (3, 1, 1))["kernel"] == "slab<128>"   # 128 output channels: N = 128 MMAs are balanced already
    assert plan(16, 64, 16, 28, 28, 64, (3, 3, 3))["kernel"] == "slabts"       # in-plane taps: slab / slabts
    assert plan(16, 230, 8, 14, 14, 64, (3, 1, 1), s=(2, 1, 1))["kernel"] == "slab<64>"    # temporal stride
    assert plan(16, 64, 16, 28, 28, 64, (3, 1, 1), pad=(0, 0, 0))["kernel"] == "igemm<64>"  # not "same"-padded
    assert plan(64, 1024, 8, 14, 14, 64, (3, 1, 1))["kernel"] == "slab<64>"    # 16 chunks x 3 taps x 8 KB = 384 KB: cannot stay resident
    assert plan(64, 64, 1, 56, 56, 64, (3, 1, 1))["kernel"] == "slab<64>"      # a single frame: only the centre tap ever sees data
    try:
        lib.b2_debug_set_tstack(1)                                 # forced (tests): eligibility without the one-item-per-SM rule
        assert plan(2, 144, 16, 28, 28, 64, (3, 1, 1))["kernel"] == "tstack"
        lib.b2_debug_set_tstack(0)
        assert plan(16, 110, 32, 56, 56, 64, (7, 1, 1))["kernel"] == "slab<64>"
    finally:
        lib.b2_debug_set_tstack(-1)


def test_temporal_stack_slot_algebra():
    """The frame-group / slot / stacked-filter arithmetic of b2_tstack.cuh (tstack_item and the MMA issuer's s_lo, s_hi, r0), transcribed
    and run on scalars for every clip length 2..21 and kt = 3, 5, 7, 9: each output frame must receive exactly the taps of a zero-padded
    temporal convolution, each through the stack block that holds W(dt), every issued MMA must cover a contiguous block range inside
    the stack and at most 4 slots.  (The GPU tests cover a handful of (T, kt); this pins the index algebra for all of them.)"""
    G = 4
    for kt in (3, 5, 7, 9):
        pt = kt // 2
        w = torch.arange(1, kt + 1, dtype=torch.float64) * 0.37 + 1.0          # W(dt), distinct values
        for T in range(2, 22):
            x = torch.arange(1, T + 1, dtype=torch.float64) ** 1.5
            want = torch.nn.functional.conv1d(x.view(1, 1, T), w.view(1, 1, kt), padding=pt).view(T)
            got = torch.zeros(T, dtype=torch.float64)
            groups = (T + G - 1) // G
            for g in range(groups):
                to0 = g * G
                nf = min(G, T - to0)
                fr_lo = max(0, pt - to0)
                fr_hi = min(nf + kt - 2, T - 1 - to0 + pt)
                assert fr_lo <= fr_hi
                for fr in range(fr_lo, fr_hi + 1):
                    f = to0 - pt + fr                                            # absolute input frame (plane_i0 + fr)
                    assert 0 <= f < T
                    s_lo, s_hi = max(0, fr - (kt - 1)), min(nf - 1, fr)
                    nslots = s_hi - s_lo + 1
                    assert 1 <= nslots <= 4                                      # N = 64 * nslots <= 256
                    r0 = kt - 1 - (fr - s_lo)                                    # first block of the stack [W(kt-1); ...; W(0)]
                    assert 0 <= r0 and r0 + nslots - 1 <= kt - 1
                    for j in range(nslots):
                        dt = kt - 1 - (r0 + j)                                   # block r holds W(dt = kt-1-r)
                        got[to0 + s_lo + j] += x[f] * w[dt]
            assert torch.allclose(got, want, rtol=1e-12, atol=1e-9), (kt, T)


def test_library_abi_is_pinned(monkeypatch):
    from pretorched_x_b200 import _lib
    assert _lib.load().b2_version() == _lib.EXPECTED_ABI
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "EXPECTED_ABI", _lib.EXPECTED_ABI + 1)
    with pytest.raises(RuntimeError, match="stale library"):
        _lib.load()
    monkeypatch.undo()
    assert _lib.load().b2_version() == _lib.EXPECTED_ABI


def test_cache_invalidation_hooks():
    """Packed-weight caches are dropped on train()/eval(), _apply and on request (engine.CacheOwner)."""
    m = P.resnet3d10(num_classes=3)
    m.layer1[0].conv1.__dict__["_b2_cache"] = {"pc": ("sig", "packed")}
    m.eval()
    assert "_b2_cache" not in m.layer1[0].conv1.__dict__
    m.layer1[0].conv1.__dict__["_b2_cache"] = {"pc": ("sig", "packed")}
    m.invalidate()
    assert "_b2_cache" not in m.layer1[0].conv1.__dict__
    m.layer1[0].conv1.__dict__["_b2_cache"] = {"pc": ("sig", "packed")}
    m.float()
    assert "_b2_cache" not in m.layer1[0].conv1.__dict__


# ---------------------------------------------------------------------------------------------------------------
# depth-first trunk schedule (engine.run_trunk): plan rule and chunk assembly, on CPU stand-ins for the kernels
# ---------------------------------------------------------------------------------------------------------------
def test_dfs_plan_spec():
    from pretorched_x_b200 import engine
    assert engine.dfs_plan() == []                                   # default: breadth-first (the measured optimum)
    try:
        engine.set_dfs("5:2,4:8")
        assert engine.dfs_plan() == [(5, 2), (4, 8)]
        engine.set_dfs("auto")
        assert engine.dfs_plan() == []
    finally:
        engine.set_dfs("off")


def test_dfs_segments_assemble_the_breadth_first_result(monkeypatch):
    """run_trunk with the kernels replaced by CPU stand-ins: chunked segments (ragged last chunk, units that honour ``out`` and
    units that do not) reproduce the whole-batch walk, and every unit sees only its chunk."""
    from pretorched_x_b200 import engine
    from pretorched_x_b200.ops import Act
    seen = []

    def fake_stem(model, x, simt=False, out=None):
        n = x.shape[0]
        seen.append(("stem", n))
        rows = x.reshape(n, 3, -1).permute(0, 2, 1).reshape(-1, 3)            # [n * px][3]
        y = torch.zeros((rows.shape[0], 8), dtype=torch.float16)
        y[:, :3] = rows.half()
        if out is not None:
            out.copy_(y)
            y = out
        return Act(y, n, 1, x.shape[2], x.shape[3], 3)

    def fake_block(block, a, simt=False, out=None):
        seen.append((block.tag, a.N))
        y = a.data * 2 + block.tag
        y[:, a.C:] = 0
        if out is not None and block.tag % 2 == 0:      # odd blocks ignore ``out``: the scheduler must copy
            out.copy_(y)
            y = out
        return Act(y, a.N, a.T, a.H, a.W, a.C)

    class Blk(nn.Module):
        def __init__(self, tag):
            super().__init__()
            self.tag = tag

    class Net(nn.Module):
        def __init__(self):
            super().__init__()
            self.layer1 = nn.Sequential(Blk(1), Blk(2))
            self.layer2 = nn.Sequential(Blk(3))
            self.layer3 = nn.Sequential(Blk(4), Blk(5))
            self.layer4 = nn.Sequential(Blk(6))

    monkeypatch.setattr(engine, "run_stem", fake_stem)
    monkeypatch.setattr(engine, "run_block", fake_block)
    net = Net()
    x = torch.randn(7, 3, 4, 5)
    try:
        engine.set_dfs("off")
        want = engine.run_trunk(net, x)
        for spec in ("3:2", "1:3,2:2,2:4", "7:3", "2:7", "4:1,3:5"):
            seen.clear()
            engine.set_dfs(spec)
            got = engine.run_trunk(net, x)
            assert (got.N, got.H, got.W, got.C) == (want.N, want.H, want.W, want.C) and torch.equal(got.data, want.data), spec
            first_chunk = int(spec.split(",")[0].split(":")[1])
            assert seen[0] == ("stem", min(first_chunk, 7)), (spec, seen[:3])
            assert len(seen) > 7 or first_chunk >= 7
    finally:
        engine.set_dfs("off")


def test_ops_device_guard_is_transparent_on_cpu_arguments():
    """ops._on_device: operators switch to the device of their first CUDA tensor for the launch (ADVICE r1: `model.to('cuda:1')`);
    with no CUDA tensor in sight the call goes straight through and the no-CPU-path error is what the caller sees."""
    assert ops._first_cuda_device((torch.zeros(2), ops.Act(torch.zeros(4, 8), 1, 1, 2, 2, 3)), {"residual": None}) is None
    assert ops.conv.__name__ == "conv" and "BatchNorm3d" in ops.conv.__doc__
    with pytest.raises(RuntimeError, match="no CPU path"):
        ops.from_ncdhw(torch.zeros(1, 3, 2, 4, 4))
