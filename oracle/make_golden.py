"""Generate tests/golden/*.pt from the UNMODIFIED reference (run in the build container only):

    python -m oracle.make_golden

For every case the script (1) builds the reference model from /root/reference under a fixed seed, (2) gives its
BatchNorms non-trivial statistics (oracle.functional.randomize_bn_), (3) runs the reference's own CPU fp32
forward with per-stage forward hooks -- the pattern of the reference's only value-level check,
pretorched/models/fbresnet/resnet152_load.py:251-270 -- (4) asserts that oracle/functional.py reproduces every
stage bit-for-bit, and (5) stores logits, strided stage samples and a per-tensor weight digest.  The fixtures let
the GPU box (which has no /root/reference) verify that pretorched_x_b200's seeded init equals the reference's
and that its CUDA forward matches the reference's outputs.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import functional as OF            # noqa: E402
from oracle import reference_loader as RL      # noqa: E402

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")
SAMPLE = 4096

# name -> (arch, factory kwargs, input shape)
MODEL_CASES = {
    "resnet3d50_b2_t8_64": ("resnet3d50", dict(num_classes=400), (2, 3, 8, 64, 64)),
    "resnet3d18_b1_t8_64": ("resnet3d18", dict(num_classes=400), (1, 3, 8, 64, 64)),
    "r2plus1d34_b1_t8_64": ("r2plus1d34", dict(num_classes=400), (1, 3, 8, 64, 64)),
    "nonlocalresnet3d50_b1_t16_96": ("nonlocalresnet3d50", dict(), (1, 3, 16, 96, 96)),
    "resnet18_b2_64": ("resnet18", dict(num_classes=1000), (2, 3, 64, 64)),
    "resnet50_b2_64": ("resnet50", dict(num_classes=1000), (2, 3, 64, 64)),       # 2-D bottleneck body: the TRN backbone (trn.py:210)
    # same net with theta/phi rescaled into a trained-like logit regime (oracle.functional.calibrate_nonlocal_)
    "nonlocalresnet3d50_tamed_b1_t16_96": ("nonlocalresnet3d50", dict(), (1, 3, 16, 96, 96)),
    # ---- the BASELINE.json clip sizes themselves (configs[1], [2], [3]): what bench.py times.  Same recipe, the
    #      reference's CPU forward takes seconds per clip; fixtures stay small (strided samples + logits).
    "resnet3d50_b2_t16_224": ("resnet3d50", dict(num_classes=400), (2, 3, 16, 224, 224)),
    "r2plus1d34_b1_t32_112": ("r2plus1d34", dict(num_classes=400), (1, 3, 32, 112, 112)),
    "nonlocalresnet3d50_tamed_b1_t32_224": ("nonlocalresnet3d50", dict(), (1, 3, 32, 224, 224)),
    # pre-activation blocks (pre_act_resnet3D.py:27-96), SURVEY 8f n3
    "preact_resnet3d50_b2_t8_64": ("preact_resnet3d50", dict(num_classes=174), (2, 3, 8, 64, 64)),
    "preact_resnet3d18_b1_t8_64": ("preact_resnet3d18", dict(num_classes=174, shortcut_type='A'), (1, 3, 8, 64, 64)),
}
SEED_INIT, SEED_BN, SEED_INPUT = 0, 1, 2


def sample_of(t):
    flat = t.detach().reshape(-1)
    step = max(1, flat.numel() // SAMPLE)
    return flat[::step][:SAMPLE].clone(), step


def summarize(t):
    s, step = sample_of(t)
    return dict(shape=tuple(t.shape), mean=float(t.double().mean()), std=float(t.double().std()),
                absmax=float(t.abs().max()), sample=s, step=step)


def run_model_case(name, arch, kwargs, shape):
    RL.load()
    if arch.startswith("r2plus1d"):
        RL.load_r2plus1d()
    torch.manual_seed(SEED_INIT)
    ref = RL.build(arch, **kwargs)
    OF.randomize_bn_(ref, SEED_BN)
    ref.eval()
    x = OF.seeded_input(shape, SEED_INPUT)
    nl_factors = OF.calibrate_nonlocal_(ref, x) if "tamed" in name else None

    hooked = {}
    handles = []
    for stage in ("maxpool", "layer1", "layer2", "layer3", "layer4"):
        handles.append(getattr(ref, stage).register_forward_hook(
            lambda m, i, o, stage=stage: hooked.__setitem__(stage, o.detach().clone())))
    with torch.no_grad():
        if arch.startswith("r2plus1d") or arch.startswith("preact_"):
            # R2Plus1D / PreActivationResNet3D inherit ResNet3D.forward, which modify_resnets may have patched at class level to need
            # `last_linear` (SURVEY.md section 0.1).  The unpatched body is conv1..layer4 -> avgpool -> fc:
            feat = ref.layer4(ref.layer3(ref.layer2(ref.layer1(ref.maxpool(ref.relu(ref.bn1(ref.conv1(x))))))))
            logits = ref.fc(ref.avgpool(feat).view(feat.size(0), -1))
        else:
            logits = ref(x)
    for h in handles:
        h.remove()
    hooked["logits"] = logits

    sd = {k: v.detach().clone() for k, v in ref.state_dict().items()}
    stages = {}
    spec = arch
    if kwargs.get("shortcut_type") and OF.ARCHS[arch]["shortcut"] != kwargs["shortcut_type"]:
        spec = dict(OF.ARCHS[arch], shortcut=kwargs["shortcut_type"])
    with torch.no_grad():
        out = OF.forward(x, sd, spec, stages)
    for k, v in hooked.items():
        assert torch.equal(stages[k], v), "oracle restatement differs from the reference at %s/%s" % (name, k)
    assert torch.equal(out, logits)

    fixture = dict(
        kind="model", arch=arch, kwargs=kwargs, input_shape=tuple(shape), nl_factors=nl_factors,
        seeds=dict(init=SEED_INIT, bn=SEED_BN, input=SEED_INPUT),
        logits=logits.clone(), stages={k: summarize(v) for k, v in hooked.items()},
        weight_digest=OF.state_digest(sd), n_state=len(sd),
        torch_version=torch.__version__,
    )
    torch.save(fixture, os.path.join(GOLDEN_DIR, name + ".pt"))
    print("%-32s logits %s absmax %.4f  stages ok: %s" % (name, tuple(logits.shape), logits.abs().max(),
                                                         ",".join(hooked)))


def run_resnext_cases():
    """ResNeXt-3D (resnext3D.py; exported by pretorched/__init__.py:66-72): plain ``**kwargs`` factories and an ``fc`` head, so
    the fixtures get their own kind and their own tests (tests/test_oracle_golden.py, tests/test_gpu_resnext.py)."""
    for name, (arch, kwargs, shape) in {
            "resnext3d50_b1_t8_64": ("resnext3d50", dict(num_classes=400), (1, 3, 8, 64, 64)),
            # (cardinality != 32 is broken upstream: fc is sized cardinality * 32 * expansion, the trunk ends with 2048 channels)
            "resnext3d18_a_b2_t8_64": ("resnext3d18", dict(num_classes=10, shortcut_type='A'), (2, 3, 8, 64, 64)),
    }.items():
        RL.load()
        torch.manual_seed(SEED_INIT)
        ref = RL.build(arch, **kwargs)
        OF.randomize_bn_(ref, SEED_BN)
        ref.eval()
        x = OF.seeded_input(shape, SEED_INPUT)
        hooked, handles = {}, []
        for stage in ("maxpool", "layer1", "layer2", "layer3", "layer4"):
            handles.append(getattr(ref, stage).register_forward_hook(
                lambda m, i, o, stage=stage: hooked.__setitem__(stage, o.detach().clone())))
        with torch.no_grad():
            logits = ref(x)
        for h in handles:
            h.remove()
        hooked["logits"] = logits
        sd = {k: v.detach().clone() for k, v in ref.state_dict().items()}
        spec = dict(OF.ARCHS["resnext3d50"], layers={"resnext3d50": [3, 4, 6, 3], "resnext3d18": [2, 2, 2, 2]}[arch],
                    shortcut=kwargs.get("shortcut_type", "B"), cardinality=kwargs.get("cardinality", 32))
        stages = {}
        with torch.no_grad():
            out = OF.forward(x, sd, spec, stages)
        for k, v in hooked.items():
            assert torch.equal(stages[k], v), "oracle restatement differs from the reference at %s/%s" % (name, k)
        assert torch.equal(out, logits)
        torch.save(dict(kind="resnext", arch=arch, kwargs=kwargs, spec=spec, input_shape=tuple(shape),
                        seeds=dict(init=SEED_INIT, bn=SEED_BN, input=SEED_INPUT), logits=logits.clone(),
                        stages={k: summarize(v) for k, v in hooked.items()}, weight_digest=OF.state_digest(sd), n_state=len(sd),
                        torch_version=torch.__version__), os.path.join(GOLDEN_DIR, name + ".pt"))
        print("%-32s logits %s absmax %.4f  stages ok: %s" % (name, tuple(logits.shape), logits.abs().max(), ",".join(hooked)))


def run_relation_cases():
    trn = RL.load_trn()
    # (a) single Relation, small and at the TRN-wired size (trn.py:230-233: T=8, F=2048, bottleneck 512)
    for name, (T, Fdim, out, bott, B) in {"relation_small": (8, 256, 64, 128, 5),
                                          "relation_htrn": (8, 2048, 1024, 512, 3)}.items():
        torch.manual_seed(SEED_INIT)
        ref = trn.Relation(T, Fdim, out, bottleneck_dim=bott).eval()
        x = OF.seeded_input((B, T, Fdim), SEED_INPUT)
        with torch.no_grad():
            y = ref(x)
            y_or = OF.relation(x, ref.state_dict(), "", T, Fdim)
        assert torch.equal(y, y_or)
        torch.save(dict(kind="relation", T=T, F=Fdim, out=out, bottleneck=bott, B=B,
                        seeds=dict(init=SEED_INIT, input=SEED_INPUT), output=y.clone(),
                        weight_digest=OF.state_digest(ref.state_dict())), os.path.join(GOLDEN_DIR, name + ".pt"))
        print("%-32s out %s" % (name, tuple(y.shape)))
    # (b) MultiScaleRelation; the reference draws frame tuples from NumPy's global RNG on every forward
    T, Fdim, out, bott, B = 8, 256, 64, 128, 4
    torch.manual_seed(SEED_INIT)
    import contextlib, io
    with contextlib.redirect_stdout(io.StringIO()):       # the constructor prints (trn.py:97-98)
        ref = trn.MultiScaleRelation(T, Fdim, out, bottleneck_dim=bott).eval()
    x = OF.seeded_input((B, T, Fdim), SEED_INPUT)
    with torch.no_grad():
        np.random.seed(123)
        y = ref(x)
        np.random.seed(123)
        y_or = OF.multiscale_relation(x, ref.state_dict(), T, Fdim)
    assert torch.equal(y, y_or)
    torch.save(dict(kind="msrelation", T=T, F=Fdim, out=out, bottleneck=bott, B=B, np_seed=123,
                    seeds=dict(init=SEED_INIT, input=SEED_INPUT), output=y.clone(),
                    weight_digest=OF.state_digest(ref.state_dict())), os.path.join(GOLDEN_DIR, "msrelation_small.pt"))
    print("%-32s out %s" % ("msrelation_small", tuple(y.shape)))


TRN_CASES = {
    # name -> (consensus, backbone, segments, batch, frame size, relation kwargs, numpy seed)
    "trn_resnet18_TRN": ("TRN", "resnet18", 8, 2, 64, dict(frame_bottleneck_dim=128, video_feature_dim=64), None),
    "trn_resnet18_HTRN": ("HTRN", "resnet18", 8, 2, 64, dict(), None),
    "trn_resnet18_MSTRN": ("MSTRN", "resnet18", 8, 2, 64, dict(frame_bottleneck_dim=128, video_feature_dim=64), 321),
}


def run_trn_cases():
    """The full TRN wrapper (trn.py:192-338).  Upstream cannot construct it offline (SURVEY.md section 0.8): the backbone
    factory must download a checkpoint to get its preprocessing attributes.  The ONLY patch applied here is to that
    factory: build the same backbone with ``pretrained=None`` and attach the registry's attributes (what
    ``load_pretrained`` does after the download, torchvision_models.py:162-166).  TRN.__init__/features/logits/forward run
    unmodified."""
    import contextlib, io
    trn = RL.load_trn()
    pt = RL.load()
    for name, (consensus, arch, T, B, hw, kw, np_seed) in TRN_CASES.items():
        orig = pt.__dict__[arch]

        def offline(num_classes=1000, pretrained=None, _orig=orig, _arch=arch):
            m = _orig(num_classes=num_classes, pretrained=None)
            for k, v in pt.pretrained_settings[_arch]['imagenet'].items():
                if k in ('input_space', 'input_size', 'input_range', 'mean', 'std'):
                    setattr(m, k, v)
            return m
        pt.__dict__[arch] = offline
        try:
            torch.manual_seed(SEED_INIT)
            with contextlib.redirect_stdout(io.StringIO()):
                ref = trn.TRN(10, num_segments=T, arch=arch, consensus=consensus, pretrained=None, **kw)
        finally:
            pt.__dict__[arch] = orig
        OF.randomize_bn_(ref, SEED_BN)
        ref.eval()
        x = OF.seeded_input((B, T, 3, hw, hw), SEED_INPUT)
        with torch.no_grad():
            if np_seed is not None:
                np.random.seed(np_seed)
            feats = ref.features(x)
            logits = ref.logits(feats)
            sd = {k: v.detach().clone() for k, v in ref.state_dict().items()}
            if np_seed is not None:
                np.random.seed(np_seed)
            st = {}
            out = OF.trn_forward(x, sd, arch, consensus, T, st)
        assert torch.equal(st['features'], feats) and torch.equal(out, logits), "oracle restatement differs from the reference TRN (%s)" % name
        torch.save(dict(kind="trn", consensus=consensus, arch=arch, segments=T, kwargs=kw, input_shape=(B, T, 3, hw, hw), np_seed=np_seed,
                        seeds=dict(init=SEED_INIT, bn=SEED_BN, input=SEED_INPUT), features=feats.clone(), logits=logits.clone(),
                        weight_digest=OF.state_digest(sd), n_state=len(sd)), os.path.join(GOLDEN_DIR, name + ".pt"))
        print("%-32s logits %s absmax %.4f" % (name, tuple(logits.shape), logits.abs().max()))


def run_image_case():
    """BASELINE.json configs[0]: resnet18 on the reference's own test image through the reference's own preprocessing
    (examples/imagenet_logits.py:38-43: LoadImage -> TransformImage(model) -> model; weights random-init, as offline).
    Stores the decoded image (the GPU box has no /root/reference), the preprocessed tensor and the logits."""
    utils = RL.load_transforms()
    pt = RL.load()
    from oracle import image as OI
    torch.manual_seed(SEED_INIT)
    ref = RL.build("resnet18", num_classes=1000)
    OF.randomize_bn_(ref, SEED_BN)
    ref.eval()
    settings = pt.pretrained_settings["resnet18"]["imagenet"]
    img = utils.LoadImage()(os.path.join(RL.REFERENCE_ROOT, "data", "cat.jpg"))
    x = utils.TransformImage(settings)(img)                       # the reference's Compose (transforms/utils.py:53-77)
    u8 = torch.from_numpy(np.array(img, copy=True))
    restated = torch.from_numpy(OI.transform_image(u8.numpy(), settings["input_size"], settings["input_space"],
                                                   settings["input_range"], settings["mean"], settings["std"]))
    assert torch.equal(restated, x), "oracle/image.py differs from the reference's TransformImage"
    hooked, handles = {}, []
    for stage in ("maxpool", "layer1", "layer2", "layer3", "layer4"):
        handles.append(getattr(ref, stage).register_forward_hook(
            lambda m, i, o, stage=stage: hooked.__setitem__(stage, o.detach().clone())))
    with torch.no_grad():
        logits = ref(x.unsqueeze(0))
    for h in handles:
        h.remove()
    sd = {k: v.detach().clone() for k, v in ref.state_dict().items()}
    stages = {}
    with torch.no_grad():
        out = OF.forward(x.unsqueeze(0), sd, "resnet18", stages)
    for k, v in hooked.items():
        assert torch.equal(stages[k], v), k
    assert torch.equal(out, logits)
    hooked["logits"] = logits
    torch.save(dict(kind="image", arch="resnet18", kwargs=dict(num_classes=1000), settings={k: settings[k] for k in
                    ("input_size", "input_space", "input_range", "mean", "std")}, image_u8=u8, input=summarize(x), input_sha=OF.state_digest({"x": x})["x"],
                    seeds=dict(init=SEED_INIT, bn=SEED_BN), logits=logits.clone(),
                    stages={k: summarize(v) for k, v in hooked.items()}, weight_digest=OF.state_digest(sd), n_state=len(sd)),
               os.path.join(GOLDEN_DIR, "resnet18_cat_224.pt"))
    print("%-32s image %s -> %s, logits absmax %.4f" % ("resnet18_cat_224", tuple(u8.shape), tuple(x.shape), logits.abs().max()))


NLBLOCK_CASES = {
    # name -> (dimension, mode, sub_sample, bn_layer, channels, input shape)
    "nlblock3d_gaussian_sub": (3, "gaussian", True, True, 128, (2, 128, 4, 8, 8)),
    "nlblock3d_dot_product": (3, "dot_product", False, True, 128, (2, 128, 2, 7, 7)),
    "nlblock3d_embedded_sub": (3, "embedded_gaussian", True, True, 128, (1, 128, 4, 8, 8)),
    "nlblock2d_embedded": (2, "embedded_gaussian", False, True, 128, (2, 128, 12, 12)),
    "nlblock2d_dot_sub_nobn": (2, "dot_product", True, False, 128, (2, 128, 12, 12)),
    "nlblock1d_gaussian": (1, "gaussian", False, True, 128, (3, 128, 50)),
    # concatenation mode (nonlocalnet.py:213-243), plain and with max-pooled phi / g; and a block whose inter_channels (32)
    # is below the attention kernel's 64-wide granule (the nonlocalresnet3d18/34 placement: C = 64, d = 32)
    "nlblock3d_concat": (3, "concatenation", False, True, 128, (2, 128, 2, 6, 6)),
    "nlblock2d_concat_sub": (2, "concatenation", True, True, 128, (2, 128, 12, 12)),
    "nlblock3d_embedded_c64": (3, "embedded_gaussian", False, True, 64, (2, 64, 2, 8, 8)),
}


def condition_nlblock_(blk, seed):
    """Deterministic, benign parameters for a bare non-local block: BN statistics randomised, projections scaled so
    the logits stay O(1), the zero-initialised output projection (nonlocalnet.py:95-102) replaced by seeded noise."""
    OF.randomize_bn_(blk, seed)
    g = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():
        for name, prm in blk.named_parameters():
            if name.startswith(("theta", "phi")) and name.endswith("weight"):
                prm.mul_(0.3)
            if name in ("W.weight", "W.bias"):
                prm.copy_(torch.randn(prm.shape, generator=g) * 0.05)
    return blk


def run_nlblock_cases(only=None):
    ref_nl = RL.load().models.nonlocalnet
    for name, (dim, mode, sub, bn, C, shape) in NLBLOCK_CASES.items():
        if only is not None and name not in only:
            continue
        cls = getattr(ref_nl, "NonLocalBlock%dD" % dim)
        torch.manual_seed(SEED_INIT)
        ref = condition_nlblock_(cls(C, mode=mode, sub_sample=sub, bn_layer=bn), SEED_BN).eval()
        x = OF.seeded_input(shape, SEED_INPUT) * (0.3 if mode == "gaussian" else 1.0)
        with torch.no_grad():
            y = ref(x)
            y_or = OF.nonlocal_block_nd(x, ref.state_dict(), "", dim, mode, sub, bn)
        assert torch.equal(y, y_or), "oracle restatement differs from the reference for %s" % name
        torch.save(dict(kind="nlblock", dimension=dim, mode=mode, sub_sample=sub, bn_layer=bn, channels=C,
                        input_shape=tuple(shape), input_scale=(0.3 if mode == "gaussian" else 1.0),
                        seeds=dict(init=SEED_INIT, bn=SEED_BN, input=SEED_INPUT), output=y.clone(),
                        weight_digest=OF.state_digest(ref.state_dict())), os.path.join(GOLDEN_DIR, name + ".pt"))
        print("%-32s out %s absmax %.4f" % (name, tuple(y.shape), y.abs().max()))


SLOWFAST_CASES = {
    # name -> (factory, mode, layers, bottleneck, kwargs, input shape)
    "slowfast50_sf_b1_t32_64": ("resnet50", "sf", [3, 4, 6, 3], True, dict(num_classes=12), (1, 3, 32, 64, 64)),
    "slowfast18_sf_b2_t32_64": ("resnet18", "sf", [2, 2, 2, 2], False, dict(num_classes=12), (2, 3, 32, 64, 64)),
    "slowonly50_b1_t32_64": ("resnet50", "s", [3, 4, 6, 3], True, dict(num_classes=12), (1, 3, 32, 64, 64)),
    "fastonly50_b1_t16_64": ("resnet50", "f", [3, 4, 6, 3], True, dict(num_classes=12), (1, 3, 16, 64, 64)),
}


def run_slowfast_cases():
    ref_pkg = RL.load()
    for name, (factory, mode, layers, bott, kwargs, shape) in SLOWFAST_CASES.items():
        torch.manual_seed(SEED_INIT)
        ref = getattr(ref_pkg.slowfast, factory)(mode=mode, **kwargs)
        OF.randomize_bn_(ref, SEED_BN)
        ref.eval()
        x = OF.seeded_input(shape, SEED_INPUT)
        with torch.no_grad():
            y = ref(x)
            sd = {k: v.detach().clone() for k, v in ref.state_dict().items()}
            y_or = OF.slowfast_forward(x, sd, layers, bott, mode)
        assert torch.equal(y, y_or), "oracle restatement differs from the reference for %s" % name
        torch.save(dict(kind="slowfast", factory=factory, mode=mode, layers=layers, bottleneck=bott, kwargs=kwargs,
                        input_shape=tuple(shape), seeds=dict(init=SEED_INIT, bn=SEED_BN, input=SEED_INPUT),
                        logits=y.clone(), weight_digest=OF.state_digest(sd), n_state=len(sd)),
                   os.path.join(GOLDEN_DIR, name + ".pt"))
        print("%-32s logits %s absmax %.4f" % (name, tuple(y.shape), y.abs().max()))


# (arch, factory kwargs, seed): whole-model inits whose every tensor tests/test_oracle_golden.py checks against the reference
STATE_CASES = [
    ("r2plus1d18", dict(num_classes=400), 3), ("resnet3d50", dict(num_classes=400), 3), ("nonlocalresnet3d50", dict(), 3),
    ("resnext3d50", dict(num_classes=400), 5), ("resnext3d18", dict(num_classes=10, shortcut_type="A"), 5), ("resnext3d101", dict(), 5),
]


def run_state_cases():
    """The reference's whole state_dict for each STATE_CASES init, stored as per-tensor hashes (oracle.functional.state_hashes):
    the tensors themselves run to hundreds of MB, the hashes let a test demand bit-identical tensors without them."""
    import warnings
    RL.load()
    RL.load_r2plus1d()
    cases = []
    for arch, kwargs, seed in STATE_CASES:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            torch.manual_seed(seed)
            ref = RL.build(arch, **kwargs)
        cases.append(dict(arch=arch, kwargs=kwargs, seed=seed, tensors=OF.state_hashes(ref.state_dict())))
        print("%-32s %d tensors" % ("state %s" % arch, len(cases[-1]["tensors"])))
    torch.save(dict(kind="state", cases=cases, torch_version=torch.__version__), os.path.join(GOLDEN_DIR, "state_hashes.pt"))


def main(argv=None):
    """``python -m oracle.make_golden`` regenerates everything; ``... name [name ...]`` only the named model / nlblock cases
    or groups (``relations``, ``slowfast``, ``nlblocks``, ``resnext``, ``image``, ``preact``, ``trn``, ``state``)."""
    argv = list(sys.argv[1:] if argv is None else argv)
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    want = (lambda n: True) if not argv else (lambda n: n in argv)
    # R(2+1)D first: see reference_loader.load_r2plus1d
    order = sorted(MODEL_CASES, key=lambda n: 0 if MODEL_CASES[n][0].startswith("r2plus1d") else 1)
    for name in order:
        if want(name):
            run_model_case(name, *MODEL_CASES[name])
    if want("relations"):
        run_relation_cases()
    if want("slowfast"):
        run_slowfast_cases()
    if want("nlblocks") or any(a in NLBLOCK_CASES for a in argv):
        run_nlblock_cases(None if want("nlblocks") else [a for a in argv if a in NLBLOCK_CASES])
    if want("resnext"):
        run_resnext_cases()
    if want("trn"):
        run_trn_cases()
    if want("image"):
        run_image_case()
    if want("state"):
        run_state_cases()


if __name__ == "__main__":
    main()
