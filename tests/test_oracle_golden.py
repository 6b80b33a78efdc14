"""CPU: pin oracle/functional.py and the package's seeded init against fixtures produced by the unmodified
reference (oracle/make_golden.py).  SURVEY.md section 8c: the reference has no golden vectors of its own."""
import glob
import os

import numpy as np
import pytest
import torch

from oracle import functional as OF
import pretorched_x_b200 as P

GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "*.pt")))
MODEL_FIX = [g for g in GOLDEN if torch.load(g, weights_only=False)["kind"] == "model"]


def build_ours(fx):
    return OF.build_package_model(P, fx)


def test_fixtures_present():
    assert len(MODEL_FIX) >= 5 and len(GOLDEN) >= 8


@pytest.mark.parametrize("path", MODEL_FIX, ids=[os.path.basename(p)[:-3] for p in MODEL_FIX])
def test_seeded_init_matches_reference_digest(path):
    fx = torch.load(path, weights_only=False)
    sd = build_ours(fx).state_dict()
    assert len(sd) == fx["n_state"]
    assert list(sd) == list(fx["weight_digest"])          # same keys, same order as the reference's state_dict
    assert OF.digests_match(OF.state_digest(sd), fx["weight_digest"])


@pytest.mark.parametrize("path", MODEL_FIX, ids=[os.path.basename(p)[:-3] for p in MODEL_FIX])
def test_oracle_reproduces_reference_outputs(path):
    fx = torch.load(path, weights_only=False)
    sd = build_ours(fx).state_dict()
    x = OF.seeded_input(fx["input_shape"], fx["seeds"]["input"])
    stages = {}
    with torch.no_grad():
        out = OF.forward(x, sd, OF.arch_spec(fx["arch"], fx["kwargs"]), stages)
    scale = fx["logits"].abs().max().item()
    assert (out - fx["logits"]).abs().max().item() <= 1e-5 * scale
    for name, ref in fx["stages"].items():
        got = stages[name]
        assert tuple(got.shape) == ref["shape"]
        samp = got.reshape(-1)[::ref["step"]][:ref["sample"].numel()]
        assert (samp - ref["sample"]).abs().max().item() <= 1e-5 * max(ref["absmax"], 1e-6), name


def test_relation_fixtures():
    for name in ("relation_small", "relation_htrn"):
        fx = torch.load(os.path.join(os.path.dirname(__file__), "golden", name + ".pt"), weights_only=False)
        torch.manual_seed(fx["seeds"]["init"])
        ours = P.Relation(fx["T"], fx["F"], fx["out"], bottleneck_dim=fx["bottleneck"])
        assert OF.digests_match(OF.state_digest(ours.state_dict()), fx["weight_digest"])
        x = OF.seeded_input((fx["B"], fx["T"], fx["F"]), fx["seeds"]["input"])
        with torch.no_grad():
            y = OF.relation(x, ours.state_dict(), "", fx["T"], fx["F"])
        assert (y - fx["output"]).abs().max().item() <= 1e-5 * fx["output"].abs().max().item()


def test_multiscale_relation_fixture():
    fx = torch.load(os.path.join(os.path.dirname(__file__), "golden", "msrelation_small.pt"), weights_only=False)
    torch.manual_seed(fx["seeds"]["init"])
    ours = P.MultiScaleRelation(fx["T"], fx["F"], fx["out"], bottleneck_dim=fx["bottleneck"])
    assert OF.digests_match(OF.state_digest(ours.state_dict()), fx["weight_digest"])
    x = OF.seeded_input((fx["B"], fx["T"], fx["F"]), fx["seeds"]["input"])
    np.random.seed(fx["np_seed"])
    with torch.no_grad():
        y = OF.multiscale_relation(x, ours.state_dict(), fx["T"], fx["F"])
    assert (y - fx["output"]).abs().max().item() <= 1e-5 * fx["output"].abs().max().item()
    # the package draws the same tuples from the same NumPy seed as the reference (trn.py:103-106)
    np.random.seed(fx["np_seed"])
    picks = ours.sample_tuples()
    np.random.seed(fx["np_seed"])
    y2 = OF.multiscale_relation(x, ours.state_dict(), fx["T"], fx["F"], tuples=picks)
    assert torch.equal(y, y2)


# the reference's whole state_dict for a few factory calls, as per-tensor hashes (oracle/make_golden.py run_state_cases)
STATE_FIX = torch.load(os.path.join(os.path.dirname(__file__), "golden", "state_hashes.pt"), weights_only=False)["cases"]


def assert_state_matches_reference(case, ours):
    """Every tensor of ``ours`` bit-identical to the reference's, same keys in the same order."""
    got = OF.state_hashes(ours.state_dict())
    assert list(got) == list(case["tensors"]), case["arch"]
    for k, want in case["tensors"].items():
        assert got[k] == want, (case["arch"], k)


def test_state_dict_identical_to_live_reference():
    cases = [c for c in STATE_FIX if not c["arch"].startswith("resnext")]
    assert [c["arch"] for c in cases] == ["r2plus1d18", "resnet3d50", "nonlocalresnet3d50"]
    for c in cases:
        torch.manual_seed(c["seed"])
        arch, kw = c["arch"], c["kwargs"]
        ours = getattr(P, arch)(**kw) if arch.startswith("r2") else getattr(P, arch)(pretrained=None, **kw)
        assert_state_matches_reference(c, ours)


SF_FIX = [g for g in GOLDEN if torch.load(g, weights_only=False)["kind"] == "slowfast"]


def build_slowfast(fx):
    torch.manual_seed(fx["seeds"]["init"])
    m = getattr(P.slowfast, fx["factory"])(mode=fx["mode"], **fx["kwargs"])
    OF.randomize_bn_(m, fx["seeds"]["bn"])
    return m.eval()


@pytest.mark.parametrize("path", SF_FIX, ids=[os.path.basename(p)[:-3] for p in SF_FIX])
def test_slowfast_init_and_oracle_match_reference(path):
    fx = torch.load(path, weights_only=False)
    sd = build_slowfast(fx).state_dict()
    assert list(sd) == list(fx["weight_digest"]) and OF.digests_match(OF.state_digest(sd), fx["weight_digest"])
    x = OF.seeded_input(fx["input_shape"], fx["seeds"]["input"])
    with torch.no_grad():
        y = OF.slowfast_forward(x, sd, fx["layers"], fx["bottleneck"], fx["mode"])
    assert (y - fx["logits"]).abs().max().item() <= 1e-5 * fx["logits"].abs().max().item()


NL_FIX = [g for g in GOLDEN if torch.load(g, weights_only=False)["kind"] == "nlblock"]


def build_nlblock(fx):
    from oracle.make_golden import condition_nlblock_
    from pretorched_x_b200.models import nonlocalnet
    torch.manual_seed(fx["seeds"]["init"])
    cls = getattr(nonlocalnet, "NonLocalBlock%dD" % fx["dimension"])
    blk = cls(fx["channels"], mode=fx["mode"], sub_sample=fx["sub_sample"], bn_layer=fx["bn_layer"])
    return condition_nlblock_(blk, fx["seeds"]["bn"]).eval()


@pytest.mark.parametrize("path", NL_FIX, ids=[os.path.basename(p)[:-3] for p in NL_FIX])
def test_nonlocal_block_modes_init_and_oracle_match_reference(path):
    fx = torch.load(path, weights_only=False)
    blk = build_nlblock(fx)
    assert OF.digests_match(OF.state_digest(blk.state_dict()), fx["weight_digest"])
    x = OF.seeded_input(fx["input_shape"], fx["seeds"]["input"]) * fx["input_scale"]
    with torch.no_grad():
        y = OF.nonlocal_block_nd(x, blk.state_dict(), "", fx["dimension"], fx["mode"], fx["sub_sample"], fx["bn_layer"])
    assert (y - fx["output"]).abs().max().item() <= 1e-5 * fx["output"].abs().max().item()


# ---------------------------------------------------------------------------------------------
# ResNeXt-3D (resnext3D.py; exported by pretorched/__init__.py:66-72)
# ---------------------------------------------------------------------------------------------
RX_FIX = [g for g in GOLDEN if torch.load(g, weights_only=False)["kind"] == "resnext"]


def build_resnext(fx):
    torch.manual_seed(fx["seeds"]["init"])
    m = getattr(P, fx["arch"])(**fx["kwargs"])
    OF.randomize_bn_(m, fx["seeds"]["bn"])
    return m.eval()


@pytest.mark.parametrize("path", RX_FIX, ids=[os.path.basename(p)[:-3] for p in RX_FIX])
def test_resnext3d_init_and_oracle_match_reference(path):
    fx = torch.load(path, weights_only=False)
    sd = build_resnext(fx).state_dict()
    assert len(sd) == fx["n_state"] and list(sd) == list(fx["weight_digest"])
    assert "fc.weight" in sd and "last_linear.weight" not in sd            # no modify_resnets on this family
    assert OF.digests_match(OF.state_digest(sd), fx["weight_digest"])
    x = OF.seeded_input(fx["input_shape"], fx["seeds"]["input"])
    stages = {}
    with torch.no_grad():
        out = OF.forward(x, sd, fx["spec"], stages)
    assert (out - fx["logits"]).abs().max().item() <= 1e-5 * fx["logits"].abs().max().item()
    for name, ref in fx["stages"].items():
        samp = stages[name].reshape(-1)[::ref["step"]][:ref["sample"].numel()]
        assert tuple(stages[name].shape) == ref["shape"]
        assert (samp - ref["sample"]).abs().max().item() <= 1e-5 * max(ref["absmax"], 1e-6), name


def test_resnext_fixtures_present():
    assert len(RX_FIX) >= 2


def test_resnext3d_state_dict_identical_to_live_reference():
    cases = [c for c in STATE_FIX if c["arch"].startswith("resnext")]
    assert [c["arch"] for c in cases] == ["resnext3d50", "resnext3d18", "resnext3d101"]
    for c in cases:
        torch.manual_seed(c["seed"])
        assert_state_matches_reference(c, getattr(P, c["arch"])(**c["kwargs"]))
    assert P.models.resnext3d.pretrained_settings["resnext3d101"]["kinetics-400"]["url"].endswith("resnext3d101_kinetics-8e57b772.pth")
    assert P.models.resnext3d.pretrained_settings["resnext3d50"]["kinetics-400"]["url"] is None


def test_grouped_filter_as_block_diagonal_dense_filter():
    """Host logic behind the engine's grouped convolution: the dense filter built by ops.dense_from_grouped gives exactly the
    grouped convolution (the products with the zero blocks vanish)."""
    import torch.nn.functional as F
    from pretorched_x_b200 import ops
    g = torch.Generator().manual_seed(9)
    for K, C, groups, k in ((64, 64, 32, 3), (24, 12, 4, 3), (16, 16, 1, 1), (128, 128, 32, 3)):
        w = torch.randn(K, C // groups, k, k, k, generator=g)
        x = torch.randn(2, C, 4, 6, 5, generator=g)
        dense = ops.dense_from_grouped(w, groups)
        assert dense.shape == (K, C, k, k, k)
        want = F.conv3d(x, w, None, 1, k // 2, 1, groups)
        got = F.conv3d(x, dense, None, 1, k // 2)
        assert (got - want).abs().max().item() <= 1e-5 * want.abs().max().item()
        assert float((dense != 0).double().mean()) <= 1.0 / groups + 1e-9
    with pytest.raises(ValueError):
        ops.dense_from_grouped(torch.zeros(10, 4, 1, 1, 1), 4)


# ---------------------------------------------------------------------------------------------
# TRN wrapper (trn.py:192-338): fixtures come from the reference with only its backbone factory patched for offline use
# ---------------------------------------------------------------------------------------------
TRN_FIX = [g for g in GOLDEN if torch.load(g, weights_only=False)["kind"] == "trn"]


def build_trn(fx):
    torch.manual_seed(fx["seeds"]["init"])
    m = P.TRN(10, num_segments=fx["segments"], arch=fx["arch"], consensus=fx["consensus"], pretrained=None, **fx["kwargs"])
    OF.randomize_bn_(m, fx["seeds"]["bn"])
    return m.eval()


@pytest.mark.parametrize("path", TRN_FIX, ids=[os.path.basename(p)[:-3] for p in TRN_FIX])
def test_trn_wrapper_init_and_oracle_match_reference(path):
    fx = torch.load(path, weights_only=False)
    sd = build_trn(fx).state_dict()
    assert list(sd) == list(fx["weight_digest"]) and OF.digests_match(OF.state_digest(sd), fx["weight_digest"])
    x = OF.seeded_input(fx["input_shape"], fx["seeds"]["input"])
    if fx["np_seed"] is not None:
        np.random.seed(fx["np_seed"])
    st = {}
    with torch.no_grad():
        y = OF.trn_forward(x, sd, fx["arch"], fx["consensus"], fx["segments"], st)
    assert (st["features"] - fx["features"]).abs().max().item() <= 1e-5 * fx["features"].abs().max().item()
    assert (y - fx["logits"]).abs().max().item() <= 1e-5 * fx["logits"].abs().max().item()
