"""GPU (-m gpu): kernel-level parity of the C-ABI entry points against the CPU oracle (torch fp32 on the same
fp16-rounded operands).  Tolerances are relative to max|reference|: 2e-3 for fp16 outputs (fp32 accumulate,
one fp16 rounding of the result = 2^-11), 1e-4 for fp32 outputs."""
import functools
import json
import os
import zlib

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from oracle import functional as OF

pytestmark = pytest.mark.gpu

TOL_F16 = 2e-3
TOL_F32 = 1e-4


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a B200"
    from pretorched_x_b200 import _lib
    _lib.load()
    return torch.device("cuda:0")


def h(x):
    return x.half().float()


def rel(got, ref):
    return (got.double().cpu() - ref.double()).abs().max().item() / max(ref.abs().max().item(), 1e-12)


def seed_of(name):
    return zlib.crc32(name.encode()) % 100000


@functools.lru_cache(maxsize=None)
def golden_kernels():
    """Case name -> the kernel instance its convolution launched on the B200 that recorded tests/golden/conv_plans.json."""
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "conv_plans.json")) as fh:
        rows = json.load(fh)["rows"]
    return {src.split(":", 1)[1]: r["kernel"] for r in rows for src in r["sources"] if src.startswith(("conv_case:", "tstack_case:"))}


CONV_CASES = [
    # name, N, Cin, T, H, W, K, kernel, stride, padding, residual, relu, bias, bn
    ("1x1x1_tma", 2, 64, 4, 8, 8, 256, (1, 1, 1), (1, 1, 1), (0, 0, 0), True, True, False, True),
    ("1x1x1_reduce", 1, 256, 4, 8, 8, 64, (1, 1, 1), (1, 1, 1), (0, 0, 0), False, True, False, True),
    ("3x3x3_s1", 1, 64, 4, 8, 8, 64, (3, 3, 3), (1, 1, 1), (1, 1, 1), False, True, False, True),
    ("3x3x3_s1_ragged_rows", 1, 64, 3, 7, 5, 64, (3, 3, 3), (1, 1, 1), (1, 1, 1), True, True, False, True),
    ("3x3x3_s2", 1, 128, 4, 8, 8, 128, (3, 3, 3), (2, 2, 2), (1, 1, 1), False, True, False, True),
    ("3x3x3_T1_all_temporal_padding", 2, 128, 1, 7, 7, 128, (3, 3, 3), (1, 1, 1), (1, 1, 1), False, True, False, True),
    ("shortcutB_1x1x1_s2", 1, 256, 4, 8, 8, 512, (1, 1, 1), (2, 2, 2), (0, 0, 0), False, False, False, True),
    ("r2p1d_spatial_144", 1, 64, 4, 8, 8, 144, (1, 3, 3), (1, 1, 1), (0, 1, 1), False, True, False, True),
    ("r2p1d_temporal_from_144", 1, 144, 4, 8, 8, 64, (3, 1, 1), (1, 1, 1), (1, 0, 0), True, True, False, True),
    ("r2p1d_temporal7_from_110", 1, 110, 8, 8, 8, 64, (7, 1, 1), (1, 1, 1), (3, 0, 0), False, False, False, True),
    ("r2p1d_spatial_s2_odd_230", 1, 64, 4, 8, 8, 230, (1, 3, 3), (1, 2, 2), (0, 1, 1), False, True, False, True),
    ("r2p1d_temporal_s2_from_230", 1, 230, 4, 4, 4, 128, (3, 1, 1), (2, 1, 1), (1, 0, 0), False, True, False, True),
    ("nonlocal_theta_bias_no_bn", 1, 128, 2, 4, 4, 64, (1, 1, 1), (1, 1, 1), (0, 0, 0), False, False, True, False),
    ("stem_7x7x7", 1, 3, 4, 32, 32, 64, (7, 7, 7), (1, 2, 2), (3, 3, 3), False, True, False, True),
    ("stem_r2p1d_1x7x7_to_110", 1, 3, 4, 32, 32, 110, (1, 7, 7), (1, 2, 2), (0, 3, 3), False, True, False, True),
    ("single_output_pixel", 1, 64, 1, 1, 1, 64, (3, 3, 3), (1, 1, 1), (1, 1, 1), False, True, False, True),
    # slab kernel: full layer shapes, several planes / tiles / N tiles, strided phases
    ("slab_layer1_56x56", 2, 64, 4, 56, 56, 64, (3, 3, 3), (1, 1, 1), (1, 1, 1), False, True, False, True),
    ("slab_layer2_28x28_res", 2, 128, 3, 28, 28, 128, (3, 3, 3), (1, 1, 1), (1, 1, 1), True, True, False, True),
    ("slab_layer3_14x14", 3, 256, 2, 14, 14, 256, (3, 3, 3), (1, 1, 1), (1, 1, 1), False, True, False, True),
    ("slab_odd_sizes_200ch", 1, 64, 5, 13, 11, 200, (3, 3, 3), (1, 1, 1), (1, 1, 1), False, True, False, True),
    ("slab_s2_56_to_28", 2, 128, 4, 56, 56, 128, (3, 3, 3), (2, 2, 2), (1, 1, 1), False, True, False, True),
    ("slab_s2_odd_input_7x7", 2, 256, 3, 7, 7, 256, (3, 3, 3), (2, 2, 2), (1, 1, 1), False, True, False, True),
    ("slab_2d_3x3_s2_resnet18", 2, 64, 1, 56, 56, 128, (1, 3, 3), (1, 2, 2), (0, 1, 1), False, True, False, True),
    ("slab_temporal7_wide", 1, 110, 8, 56, 56, 64, (7, 1, 1), (1, 1, 1), (3, 0, 0), False, False, False, True),
    # runtime-N slab instance (Cout that tiles badly by 128): several N tiles, residual, strided phases
    ("flexn_144_56x56", 2, 64, 2, 56, 56, 144, (1, 3, 3), (1, 1, 1), (0, 1, 1), False, True, False, True),
    ("flexn_288_28x28_res", 2, 128, 3, 28, 28, 288, (1, 3, 3), (1, 1, 1), (0, 1, 1), True, True, False, True),
    ("flexn_576_14x14_3tiles", 2, 256, 2, 14, 14, 576, (1, 3, 3), (1, 1, 1), (0, 1, 1), False, True, False, True),
    ("flexn_460_s2", 1, 128, 2, 28, 28, 460, (1, 3, 3), (1, 2, 2), (0, 1, 1), False, True, False, True),
    # W chunking: rows longer than one TMA box; temporal filters remapped to (1,kt,1) over frames x positions
    ("wide_row_chunks_3x3", 1, 64, 2, 6, 300, 64, (1, 3, 3), (1, 1, 1), (0, 1, 1), False, True, False, True),
    ("wide_row_chunks_3x3_s2", 1, 64, 1, 9, 301, 128, (1, 3, 3), (1, 2, 2), (0, 1, 1), False, True, False, True),
    ("temporal3_chunked_28x28_res", 2, 288, 6, 28, 28, 128, (3, 1, 1), (1, 1, 1), (1, 0, 0), True, True, False, True),
    ("temporal3_14x14_from_576", 2, 576, 4, 14, 14, 256, (3, 1, 1), (1, 1, 1), (1, 0, 0), False, True, False, True),
    ("temporal5_ragged_positions", 1, 64, 7, 9, 11, 64, (5, 1, 1), (1, 1, 1), (2, 0, 0), False, True, False, True),
    ("projection_1x1x1_s2_subsample", 2, 256, 4, 8, 8, 512, (1, 1, 1), (2, 2, 2), (0, 0, 0), False, False, False, True),
    # stem kernel, pair-of-planes mode (Wo <= 60, kt == 1): odd number of planes (the last pair is half empty), full 112-wide rows
    ("stem_pair_odd_planes_112", 1, 3, 3, 20, 112, 110, (1, 7, 7), (1, 2, 2), (0, 3, 3), False, True, False, True),
    ("stem_pair_2d_7x7_64ch", 3, 3, 1, 48, 96, 64, (1, 7, 7), (1, 2, 2), (0, 3, 3), False, True, False, True),
    # dense-M split-K kernel (cluster / DSMEM reduction): 4x4 planes, long K, ragged M, residual; strided multi-tap convolutions
    ("densem_4x4_1152_split", 5, 512, 2, 4, 4, 1152, (1, 3, 3), (1, 1, 1), (0, 1, 1), False, True, False, True),
    ("densem_temporal_1152_512_res", 5, 1152, 2, 4, 4, 512, (3, 1, 1), (1, 1, 1), (1, 0, 0), True, True, False, True),
    ("densem_3x3x3_s2_odd_200ch", 3, 200, 3, 9, 9, 328, (3, 3, 3), (2, 2, 2), (1, 1, 1), True, True, False, True),
    ("densem_tiny_m_3", 3, 256, 1, 1, 1, 96, (3, 3, 3), (1, 1, 1), (1, 1, 1), False, False, True, False),
    # temporal-group slab kernel (3 x kh x kw, Cout <= 64): frame groups 3 + 2, 3 + 3 + 1, clip boundaries, residual, odd widths, 2 K chunks
    ("slabts_c64_t5_res", 2, 64, 5, 20, 20, 64, (3, 3, 3), (1, 1, 1), (1, 1, 1), True, True, False, True),
    ("slabts_c32_to_48_t7_odd", 1, 32, 7, 13, 19, 48, (3, 3, 3), (1, 1, 1), (1, 1, 1), False, True, False, True),
    ("slabts_c128_to_64_t3", 2, 128, 3, 24, 24, 64, (3, 3, 3), (1, 1, 1), (1, 1, 1), False, False, False, True),
    ("slabts_temporal_3x1x1_to_64", 2, 144, 6, 28, 28, 64, (3, 1, 1), (1, 1, 1), (1, 0, 0), True, True, False, True),
    ("slabts_wide_rows_chunked", 1, 64, 4, 5, 300, 64, (3, 3, 3), (1, 1, 1), (1, 1, 1), False, True, False, True),
    # multi-plane items of the slab kernel (small planes share each weight tile): odd plane counts (partial last group), residual,
    # runtime N tile, T == 1 with a 3-tap temporal filter (only the centre tap is ever valid)
    ("slab_multiplane_7x7_192", 9, 128, 3, 7, 7, 192, (1, 3, 3), (1, 1, 1), (0, 1, 1), True, True, False, True),
    ("slab_multiplane_7x7_T1_3x3x3", 23, 128, 1, 7, 7, 128, (3, 3, 3), (1, 1, 1), (1, 1, 1), False, True, False, True),
    ("slab_multiplane_5x6_c512_256wide", 41, 512, 1, 5, 6, 256, (1, 3, 3), (1, 1, 1), (0, 1, 1), False, True, False, True),
]


@pytest.mark.parametrize("case", CONV_CASES, ids=[c[0] for c in CONV_CASES])
@pytest.mark.parametrize("simt", [False, True], ids=["tcgen05", "simt_crosscheck"])
def test_conv_bn_act_matches_oracle(dev, case, simt):
    check_conv_case(dev, case, simt)


# temporal stack kernel (b2_tstack.cuh: (kt,1,1) filters, Cout <= 64, resident filter, 4 output frames per item, two accumulator
# sets): forced on shapes below its one-item-per-SM rule.  Frame groups 4 + 4, 4 + 1, 4 + 2 + ..., a single group of 2 or 3 frames
# (T < kt: taps that never see a valid frame), clip boundaries between samples, ragged position tiles (HW % 128 != 0, HW < 128),
# residual / no residual / no ReLU / bias without BN, 1 - 3 channel chunks with ragged tails, K < 64 (zero pad columns), kt = 3, 5, 7.
TSTACK_CASES = [
    ("tstack_3_c144_to_64_t8_28x28_res", 2, 144, 8, 28, 28, 64, (3, 1, 1), (1, 1, 1), (1, 0, 0), True, True, False, True),
    ("tstack_3_c144_to_64_t5_res", 3, 144, 5, 14, 14, 64, (3, 1, 1), (1, 1, 1), (1, 0, 0), True, True, False, True),
    ("tstack_7_c110_to_64_t16_56x56", 1, 110, 16, 56, 56, 64, (7, 1, 1), (1, 1, 1), (3, 0, 0), False, False, False, True),
    ("tstack_7_c110_to_64_t6_clips", 3, 110, 6, 20, 20, 64, (7, 1, 1), (1, 1, 1), (3, 0, 0), False, True, False, True),
    ("tstack_7_t3_taps_outside", 2, 64, 3, 24, 24, 64, (7, 1, 1), (1, 1, 1), (3, 0, 0), True, True, False, True),
    ("tstack_5_c64_to_42_t9_ragged", 2, 64, 9, 9, 11, 42, (5, 1, 1), (1, 1, 1), (2, 0, 0), True, False, True, False),
    ("tstack_3_c200_to_48_t2", 5, 200, 2, 12, 12, 48, (3, 1, 1), (1, 1, 1), (1, 0, 0), False, True, False, True),
    ("tstack_3_c24_to_64_t13_tiny_planes", 4, 24, 13, 5, 5, 64, (3, 1, 1), (1, 1, 1), (1, 0, 0), True, True, False, True),
]


@pytest.mark.parametrize("case", TSTACK_CASES, ids=[c[0] for c in TSTACK_CASES])
def test_temporal_stack_kernel_matches_oracle(dev, case):
    from pretorched_x_b200 import _lib
    lib = _lib.load()
    lib.b2_debug_set_tstack(1)
    try:
        check_conv_case(dev, case, False)
        assert lib.b2_debug_last_conv_path() == 1          # the temporal stack kernel, not the slab kernel, produced the result
    finally:
        lib.b2_debug_set_tstack(-1)


def test_temporal_stack_kernel_many_items_per_cta(dev):
    """More work items than SMs x 2 (every CTA walks several items: ring phases, both accumulator sets, re-zeroed accumulators),
    taken by the library's own rule (no forcing) -- the layer1 temporal convolution of R(2+1)D-34 on 6 clips."""
    from pretorched_x_b200 import _lib
    check_conv_case(dev, ("tstack_rule_c144_to_64_t16_28x28_res", 6, 144, 16, 28, 28, 64, (3, 1, 1), (1, 1, 1), (1, 0, 0),
                          True, True, False, True), False)
    assert _lib.load().b2_debug_last_conv_path() == 1


def check_conv_case(dev, case, simt):
    from pretorched_x_b200 import ops, engine
    name, N, Cin, T, H, W, K, k, s, p, res, relu, bias, bn = case
    g = torch.Generator().manual_seed(seed_of(name))
    x = h(torch.randn(N, Cin, T, H, W, generator=g))
    conv = nn.Conv3d(Cin, K, k, stride=s, padding=p, bias=bias)
    with torch.no_grad():
        conv.weight.copy_(h(torch.randn(conv.weight.shape, generator=g) / (Cin * k[0] * k[1] * k[2]) ** 0.5))
        if bias:
            conv.bias.copy_(torch.randn(K, generator=g))
    bnm = OF.randomize_bn_(nn.BatchNorm3d(K), 7).eval() if bn else None
    with torch.no_grad():
        y = conv(x)
        y = bnm(y) if bnm is not None else y
        r = h(torch.randn(y.shape, generator=g)) if res else None
        y = y + r if res else y
        y = F.relu(y) if relu else y
    a = ops.from_ncdhw(x.to(dev))
    ra = ops.from_ncdhw(r.to(dev), pitch=ops._round_up(K, 8)) if res else None
    out = engine.conv_bn_act(conv.to(dev), bnm.to(dev) if bnm is not None else None, a, residual=ra, relu=relu, simt=simt)
    if not simt and name in golden_kernels():              # the case ran on the kernel its name is about
        from pretorched_x_b200 import _lib
        assert _lib.last_conv_kernel() == golden_kernels()[name]
    assert (out.N, out.T, out.H, out.W, out.C) == (y.shape[0], y.shape[2], y.shape[3], y.shape[4], K)
    assert rel(ops.to_ncdhw(out), y) <= TOL_F16
    if out.ld > out.C:                                     # channel padding must stay exactly zero
        assert float(out.data[:, out.C:].abs().max()) == 0.0


GEMM_CASES = [
    ("one_tile", 128, 64, 64, False, False, False, False, False),
    ("bn128", 256, 128, 128, False, True, False, False, False),
    ("ragged_everything", 300, 200, 192, True, True, False, False, False),
    ("deep_k", 1000, 512, 512, True, False, False, False, False),
    ("head_fp32", 64, 400, 2048, False, False, False, True, False),
    ("tiny_m_fp32", 3, 339, 2048, False, False, False, True, False),
    ("swap_ab_per_row", 256, 136, 96, False, False, True, False, False),
    ("fp32_accumulate", 20, 64, 128, False, False, False, True, True),
    ("k_not_multiple_of_64", 130, 72, 200, False, True, False, False, False),
]


@pytest.mark.parametrize("case", GEMM_CASES, ids=[c[0] for c in GEMM_CASES])
def test_gemm_matches_oracle(dev, case):
    from pretorched_x_b200 import ops
    name, M, N, Kd, res, relu, per_row, f32, acc = case
    g = torch.Generator().manual_seed(seed_of(name))
    A, B = h(torch.randn(M, Kd, generator=g)), h(torch.randn(N, Kd, generator=g) / Kd ** 0.5)
    nsc = M if per_row else N
    sc, sh = torch.rand(nsc, generator=g) + 0.5, torch.randn(nsc, generator=g)
    D = A @ B.t()
    D = D * (sc.view(-1, 1) if per_row else sc.view(1, -1)) + (sh.view(-1, 1) if per_row else sh.view(1, -1))
    R = h(torch.randn(M, N, generator=g)) if res else None
    D = D + R if res else D
    D = F.relu(D) if relu else D
    Kp, Np = ops._round_up(Kd, 8), ops._round_up(N, 8)
    Ad = torch.zeros(M, Kp, dtype=torch.float16, device=dev); Ad[:, :Kd] = A.half().to(dev)
    Bd = torch.zeros(N, Kp, dtype=torch.float16, device=dev); Bd[:, :Kd] = B.half().to(dev)
    Rd = None
    if res:
        Rd = torch.zeros(M, Np, dtype=torch.float16, device=dev); Rd[:, :N] = R.half().to(dev)
    out = None
    if acc:
        base = torch.randn(M, N, generator=g)
        out, D = base.clone().to(dev), D + base
    got = ops.gemm(Ad, Bd, sc.to(dev), sh.to(dev), M, N, Kd, residual=Rd, relu=relu, per_row=per_row, out_f32=f32,
                   out=out, accumulate=acc)
    assert rel(got[:, :N].float(), D) <= (TOL_F32 if f32 else TOL_F16)
    if not f32 and Np > N:
        assert float(got[:, N:].abs().max()) == 0.0


ATT_CASES = [("one_block", 1, 128, 64, 64), ("ragged_keys_and_queries", 2, 200, 128, 128), ("odd_positions", 3, 99, 64, 128),
             ("layer2_like", 1, 576, 256, 256), ("layer3_like_dv_split", 2, 72, 512, 512), ("n_lt_64", 1, 16, 64, 64),
             ("three_d_chunks", 2, 300, 192, 64), ("many_blocks_dv128", 2, 1111, 128, 128)]


@pytest.mark.parametrize("case", ATT_CASES, ids=[c[0] for c in ATT_CASES])
def test_nonlocal_attention_matches_oracle(dev, case):
    from pretorched_x_b200 import ops
    name, B, Npos, d, dv = case
    g = torch.Generator().manual_seed(seed_of(name))
    q, k = h(torch.randn(B, Npos, d, generator=g) * 0.3), h(torch.randn(B, Npos, d, generator=g) * 0.3)
    v = h(torch.randn(B, Npos, dv, generator=g))
    ref = torch.softmax(q @ k.transpose(1, 2), dim=-1) @ v            # nonlocalnet.py:156-160, unscaled
    qkv = torch.cat([q, k, v], dim=2).reshape(B * Npos, 2 * d + dv).half().to(dev).contiguous()
    o = ops.nonlocal_attention(qkv, d, dv, B, Npos)
    assert rel(o[:, :dv].float().view(B, Npos, dv), ref) <= 4e-3


@pytest.mark.parametrize("two_pass", [False, True], ids=["single_pass", "two_pass"])
def test_attention_with_growing_logits(dev, two_pass):
    """Keys whose norm grows along the sequence: the running row maximum jumps by far more than 2^8 several times, so
    the single-pass kernel must rescale its TMEM accumulator (lazy rescaling) -- and agree with the exact two-pass one."""
    from pretorched_x_b200 import ops, _lib
    B, Npos, d, dv = 2, 700, 128, 256
    g = torch.Generator().manual_seed(77)
    q = h(torch.randn(B, Npos, d, generator=g))
    k = h(torch.randn(B, Npos, d, generator=g) * torch.linspace(0.05, 2.0, Npos).view(1, Npos, 1))
    v = h(torch.randn(B, Npos, dv, generator=g))
    ref = (torch.softmax((q.double() @ k.double().transpose(1, 2)), dim=-1) @ v.double()).float()
    qkv = torch.cat([q, k, v], dim=2).reshape(B * Npos, 2 * d + dv).half().to(dev).contiguous()
    lib = _lib.load()
    lib.b2_debug_set_attention_algo(1 if two_pass else 0)
    try:
        o = ops.nonlocal_attention(qkv, d, dv, B, Npos)
    finally:
        lib.b2_debug_set_attention_algo(0)
    assert rel(o[:, :dv].float().view(B, Npos, dv), ref) <= 4e-3


def test_two_operand_gemm_matches_oracle(dev):
    """b2_gemm2_f16: D = relu(A.B^T + A2.B2^T + shift) -- the fused conv3 + shortcut-projection GEMM."""
    from pretorched_x_b200 import ops
    g = torch.Generator().manual_seed(11)
    M, N, K1, K2 = 1000, 256, 64, 192
    A1, B1 = h(torch.randn(M, K1, generator=g)), h(torch.randn(N, K1, generator=g) / K1 ** 0.5)
    A2, B2 = h(torch.randn(M, K2, generator=g)), h(torch.randn(N, K2, generator=g) / K2 ** 0.5)
    sh = torch.randn(N, generator=g)
    want = F.relu(A1 @ B1.t() + A2 @ B2.t() + sh)
    got = ops.gemm(A1.half().to(dev), B1.half().to(dev), torch.ones(N, device=dev), sh.to(dev), M, N, K1, relu=True,
                   second=(A2.half().to(dev), B2.half().to(dev), K2))
    assert rel(got.float(), want) <= TOL_F16


def test_bottleneck_with_fused_projection_matches_unfused_blocks(dev):
    """A type-B bottleneck (resnet3D.py:125-143 + 176-185) through the fused two-operand close vs the CPU oracle."""
    from pretorched_x_b200.models import resnet3d
    torch.manual_seed(0)
    ds = nn.Sequential(nn.Conv3d(64, 256, kernel_size=1, stride=2, bias=False), nn.BatchNorm3d(256))
    blk = resnet3d.Bottleneck(64, 64, stride=2, downsample=ds)
    OF.randomize_bn_(blk, 5)
    blk.eval()
    x = OF.seeded_input((2, 64, 4, 16, 16), 6).half().float()
    sd = {"b." + k: v for k, v in blk.state_dict().items()}
    with torch.no_grad():
        want = OF.bottleneck(x, sd, "b", "resnet3d", "B", 64, 2, True)
        got = blk.to(dev)(x.to(dev))
    assert tuple(got.shape) == tuple(want.shape)
    assert rel(got, want) <= 3e-3


def test_fp16_input_is_equivalent_to_fp32_input(dev):
    from pretorched_x_b200 import ops
    x = OF.seeded_input((2, 3, 4, 16, 16), 3)
    a32 = ops.from_ncdhw(x.to(dev))
    a16 = ops.from_ncdhw(x.half().to(dev))
    assert torch.equal(a32.data, a16.data)


def test_attention_rows_are_convex_combinations(dev):
    """Size-independent property: with V == 1 every output must be exactly 1 (softmax rows sum to one)."""
    from pretorched_x_b200 import ops
    B, Npos, d, dv = 2, 1000, 64, 64
    g = torch.Generator().manual_seed(5)
    qkv = (torch.randn(B * Npos, 2 * d + dv, generator=g) * 0.5).half()
    qkv[:, 2 * d:] = 1.0
    o = ops.nonlocal_attention(qkv.to(dev), d, dv, B, Npos)
    assert (o[:, :dv].float() - 1.0).abs().max().item() <= 2e-3


def test_pooling_layout_and_helpers(dev):
    from pretorched_x_b200 import ops
    g = torch.Generator().manual_seed(1)
    x = torch.randn(2, 24, 5, 12, 10, generator=g)
    a = ops.from_ncdhw(x.to(dev))
    assert torch.equal(ops.to_ncdhw(a).cpu(), h(x))
    assert torch.equal(ops.to_ncdhw(ops.maxpool3d(a, (3, 3, 3), (2, 2, 2), (1, 1, 1))).cpu(), F.max_pool3d(h(x), 3, 2, 1))
    assert rel(ops.avgpool_global(a)[:, :24].float(), h(x).mean(dim=(2, 3, 4))) <= 1e-3
    assert torch.equal(ops.to_ncdhw(ops.shortcut_a(a, 2, 40)).cpu(), OF.shortcut_a(h(x), 40, 2))
    x3 = torch.randn(1, 3, 2, 6, 6, generator=g)
    a3 = ops.from_ncdhw(x3.to(dev))
    assert a3.ld == 4 and torch.equal(ops.to_ncdhw(a3).cpu(), h(x3))
    assert float(a3.data[:, 3].abs().max()) == 0.0


def test_conv_linearity_at_full_layer_size(dev):
    """Size-independent property at a BASELINE-sized layer (layer1 conv2 of resnet3d50, 4 clips of 8x56x56):
    with identity BN, no ReLU:  conv(a) + conv(b) == conv(a + b) up to fp16 rounding of the three outputs."""
    from pretorched_x_b200 import ops, engine
    g = torch.Generator().manual_seed(3)
    conv = nn.Conv3d(64, 64, 3, padding=1, bias=False)
    with torch.no_grad():
        conv.weight.copy_(torch.randn(conv.weight.shape, generator=g) / (64 * 27) ** 0.5)
    conv = conv.to(dev)
    xa = torch.randn(4, 64, 8, 56, 56, generator=g).half().float()
    xb = torch.randn(4, 64, 8, 56, 56, generator=g).half().float()
    xs = (xa + xb).half().float()
    ya, yb, ys = (engine.conv_bn_act(conv, None, ops.from_ncdhw(t.to(dev))).data.float() for t in (xa, xb, xs))
    scale = ys.abs().max().item()
    assert (ya + yb - ys).abs().max().item() <= 4e-3 * scale


def test_stem_fused_w_pool_equals_separate_maxpool(dev):
    """b2_conv_args.pool_w: conv 7x7x7 -> BN -> ReLU with the W direction of MaxPool3d(3, 2, 1) in the epilogue, then the (3, 3, 1)
    pass, against (a) the same engine with the stand-alone pool (bit-exact: max-pooling is separable) and (b) the CPU oracle."""
    from pretorched_x_b200 import ops, engine
    g = torch.Generator().manual_seed(11)
    for (N, T, H, W) in ((2, 5, 38, 224), (1, 4, 32, 64), (1, 3, 18, 30)):
        x = h(torch.randn(N, 3, T, H, W, generator=g))
        conv = nn.Conv3d(3, 64, 7, stride=(1, 2, 2), padding=3, bias=False)
        with torch.no_grad():
            conv.weight.copy_(h(torch.randn(conv.weight.shape, generator=g) / 32.0))
        bn = OF.randomize_bn_(nn.BatchNorm3d(64), 7).eval()
        with torch.no_grad():
            want = F.max_pool3d(F.relu(bn(conv(x))), 3, 2, 1)
        a = ops.from_ncdhw(x.to(dev))
        conv, bn = conv.to(dev), bn.to(dev)
        fused = ops.maxpool3d(engine.conv_bn_act(conv, bn, a, relu=True, pool_w=True), (3, 3, 1), (2, 2, 1), (1, 1, 0))
        plain = ops.maxpool3d(engine.conv_bn_act(conv, bn, a, relu=True), (3, 3, 3), (2, 2, 2), (1, 1, 1))
        assert (fused.N, fused.T, fused.H, fused.W) == (plain.N, plain.T, plain.H, plain.W) == (N,) + tuple(want.shape[2:])
        assert torch.equal(fused.data, plain.data)
        assert rel(ops.to_ncdhw(fused), want) <= TOL_F16
