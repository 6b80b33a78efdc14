"""Time one fine-tuning step (forward + backward + SGD step) of resnet3d50 with the last stages trainable.

    python tools/finetune_step.py [--batch 32] [--frames 16] [--size 224] [--ft 4 3 2 1] [--steps 10] [--out FILE]

For each ft_begin_index: the median over --steps CUDA-event windows of one whole step, then one profiled step split into the
backward's weight-gradient kernels (b2_conv_ndhwc_wgrad, split reduction included), data-gradient convolutions, head GEMMs
and element-wise passes (ops.profile, its own run), with the weight-gradient rate over the algorithmic FLOPs and the part of
the step no library launch accounts for.  As a reference point the same step in torch's own autograd on the same GPU:
oracle.functional's restatement of the network (frozen BatchNorm, the same semantics) under fp16 autocast, channels-last, cuDNN.
The card's name, power limit and clocks are read in the same run.  Needs a GPU; prints one JSON document.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import pretorched_x_b200 as P                                   # noqa: E402
from pretorched_x_b200 import ops                               # noqa: E402
from pretorched_x_b200.models.resnet3d import get_fine_tuning_parameters   # noqa: E402
from oracle import functional as OF                              # noqa: E402


def _gpu_state():
    q = "name,power.limit,clocks.sm,clocks.max.sm,power.draw,temperature.gpu"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()[0]
        return dict(zip(q.split(","), [v.strip() for v in out.split(",")]))
    except Exception as e:                                      # the measurement stands without it; say so
        return {"error": repr(e)}


def _time(step, steps):
    for _ in range(2):
        step()
    torch.cuda.synchronize()
    ms = []
    for _ in range(steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        step()
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    return statistics.median(ms), ms


def engine_case(x, y, ft, steps):
    torch.manual_seed(0)
    m = P.resnet3d50(num_classes=400, pretrained=None)
    OF.randomize_bn_(m, 1)
    m = m.cuda().eval().enable_fine_tuning(ft)
    opt = torch.optim.SGD(get_fine_tuning_parameters(m, ft), lr=1e-4)

    def step():
        opt.zero_grad(set_to_none=True)
        F.cross_entropy(m(x), y).backward()
        opt.step()

    med, ms = _time(step, steps)
    opt.zero_grad(set_to_none=True)
    with ops.profile() as pf:
        loss = F.cross_entropy(m(x), y)
    with ops.profile() as pb:
        loss.backward()
    split = {}
    for r in pb.rows:
        key = {"wgrad": "wgrad", "conv": "dgrad_conv", "gemm": "head_gemm"}.get(r["kind"], "elementwise")
        d = split.setdefault(key, {"ms": 0.0, "flops": 0.0, "launches": 0})
        d["ms"] += r["ms"]
        d["flops"] += r["flops"]
        d["launches"] += 1
    finite = all(bool(torch.isfinite(p.grad).all()) for p in m.parameters() if p.grad is not None)
    w = split.get("wgrad")
    fwd = sum(r["ms"] for r in pf.rows)
    bwd = sum(d["ms"] for d in split.values())
    # what the library's launches do not cover: torch-side parameter-gradient arithmetic, the SGD step, filter repacking
    # after the step, and host time between launches
    return {"ft_begin_index": ft, "step_ms_median": med, "step_ms": ms,
            "profiled_forward_ms": fwd, "profiled_backward_ms": bwd, "not_in_profile_ms": med - fwd - bwd,
            "backward_split": split, "all_gradients_finite": finite,
            "wgrad_tflops": (w["flops"] / (w["ms"] * 1e-3) / 1e12) if w and w["ms"] > 0 else None}


def torch_case(x, y, ft, steps):
    torch.manual_seed(0)
    m = P.resnet3d50(num_classes=400, pretrained=None)
    OF.randomize_bn_(m, 1)
    sd = {k: v.cuda() for k, v in m.state_dict().items()}
    train = [k for k in sd if any(k.startswith("layer%d." % i) for i in range(ft, 5)) or k.startswith("last_linear")]
    params = []
    for k in train:
        if k.endswith(("weight", "bias")):
            sd[k] = sd[k].clone().requires_grad_(True)
            if sd[k].dim() == 5:
                sd[k] = sd[k].detach().to(memory_format=torch.channels_last_3d).requires_grad_(True)
            params.append(sd[k])
    opt = torch.optim.SGD(params, lr=1e-4)
    xc = x.to(memory_format=torch.channels_last_3d)
    torch.backends.cudnn.benchmark = True

    def step():
        opt.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=torch.float16):
            loss = F.cross_entropy(OF.forward(xc, sd, "resnet3d50"), y)
        loss.backward()
        opt.step()

    med, ms = _time(step, steps)
    return {"ft_begin_index": ft, "step_ms_median": med, "step_ms": ms}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--frames", type=int, default=16)
    ap.add_argument("--size", type=int, default=224)
    ap.add_argument("--ft", type=int, nargs="+", default=[4, 3, 2, 1])
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("finetune_step.py measures on the GPU; no CUDA device here")
    g = torch.Generator().manual_seed(2)
    x = torch.randn(args.batch, 3, args.frames, args.size, args.size, generator=g).cuda()
    y = torch.randint(0, 400, (args.batch,), generator=g).cuda()
    res = {"shape": [args.batch, 3, args.frames, args.size, args.size], "gpu_before": _gpu_state(), "engine": [], "torch": []}
    for ft in args.ft:
        res["engine"].append(engine_case(x, y, ft, args.steps))
        torch.cuda.empty_cache()
        res["torch"].append(torch_case(x, y, ft, args.steps))
        torch.cuda.empty_cache()
    res["gpu_after"] = _gpu_state()
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
