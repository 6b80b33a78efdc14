#!/usr/bin/env python
"""bench.py -- throughput of the forward hot path on B200, one BASELINE.json config per --workload.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

Workloads (BASELINE.json ``configs``):
    resnet3d50  configs[1]  resnet3d50, B=32 clips of 16x224x224 per GPU, weak scaling   (default: the contract's line)
    r2plus1d34  configs[2]  r2plus1d34 (R(2+1)D-34), B=16 clips of 32x112x112 IN TOTAL, strong scaling over 1 -> 8 GPUs
    nonlocal50  configs[3]  nonlocalresnet3d50 (5 non-local blocks), 8 clips of 32x224x224 per GPU (B=64 on 8), weak scaling
    biggan256   configs[4]  BigGAN-deep-256 generator, B=256 z+class -> fp16 images per GPU, weak scaling
    resnet18    configs[0]  resnet18 224x224 images (the reference's CPU-runnable anchor), B=256 per GPU

A step = one forward pass of the hot path over one batch of synthetic input per GPU.  Clips shard with no data-path
collective; one all-gather of the [B, classes] logits per step.  Prints ONE JSON line (rank 0):
  value      CUDA-event time of K CUDA-graph replays, input resident in HBM, max over ranks
  e2e        the same forward through the public API from pinned HOST memory: fp32 NCDHW clips (the reference's input dtype)
             -> H2D -> forward -> D2H logits, every step (copies overlap the previous step's compute); the fp16-host rate beside it
  parity     logits of the timed graph for the first clips of the timed batch against the CPU oracle (asserted before timing)
  roofline   dominant kernel of the step: algorithmic FLOP (or bytes) / its CUDA-event time vs the measured peak
  cpu_baseline  the reference's own CPU forward on the host cores (oracle/_ref = the byte-compiled reference), bounded sample

``--impl reference`` times the reference's CPU fp32 forward itself (rank 0 only) on a bounded sample of the same workload.

``--dump-outputs DIR`` writes, after the timed steps, what the last timed step returned for every GPU workload of the line as
float32 ``DIR/<workload>_logits.npy`` / ``DIR/biggan256_images.npy`` (rank 0; logits gathered over ranks).  An output of more
than DUMP_ELEMS elements is stored as a fixed seeded sample of that many elements (1-D, same positions every run).  Inputs and
weights are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# algorithmic GFLOP per sample: padding taps included, exactly what hooking the reference's modules yields (SURVEY.md section 8a)
WORKLOADS = {
    "resnet3d50": dict(arch="resnet3d50", kwargs=dict(num_classes=400), sample=(3, 16, 224, 224), batch=32, scaling="weak",
                       gflop=79.69, classes=400, unit="clips/s", metric="clips/sec resnet3d50 16x224x224 forward",
                       config="configs[1]", check_clips=2, cpu_sample=2, act_elems=127.9e6),
    "r2plus1d34": dict(arch="r2plus1d34", kwargs=dict(num_classes=400), sample=(3, 32, 112, 112), batch=16, scaling="strong",
                       gflop=51.48, classes=400, unit="clips/s", metric="clips/sec r2plus1d34 32x112x112 forward",
                       config="configs[2]", check_clips=2, cpu_sample=2, act_elems=79.2e6),
    "nonlocal50": dict(arch="nonlocalresnet3d50", kwargs=dict(), sample=(3, 32, 224, 224), batch=8, scaling="weak",
                       gflop=262.22, classes=339, unit="clips/s", metric="clips/sec nonlocalresnet3d50 32x224x224 forward",
                       config="configs[3]", check_clips=1, cpu_sample=1, act_elems=289.3e6,
                       nl_fixture="nonlocalresnet3d50_tamed_b1_t32_224.pt"),
    "resnet18": dict(arch="resnet18", kwargs=dict(num_classes=1000), sample=(3, 224, 224), batch=256, scaling="weak",
                     gflop=3.63, classes=1000, unit="images/s", metric="images/sec resnet18 224x224 forward",
                     config="configs[0]", check_clips=4, cpu_sample=16, act_elems=4.7e6),
    # SURVEY.md 8a rows a10-a12: the TRN wrapper as `trn()` builds it (trn.py:345-355: class defaults => consensus 'HTRN', which
    # degenerates to one 8-frame Relation, SURVEY 0.6) on the 2-D ResNet-50 backbone; 8 frames of 224x224 per clip.
    "trn": dict(arch="trn", builder="trn", kwargs=dict(num_classes=339, num_segments=8, arch="resnet50", pretrained=None),
                sample=(8, 3, 224, 224), batch=32, scaling="weak", gflop=8 * 8.18 + 0.036, classes=339, unit="clips/s",
                metric="clips/sec TRN (resnet50 backbone, 8 segments) forward", config="SURVEY.md 8a rows a10-a12",
                check_clips=1, cpu_sample=2, act_elems=8 * 22.2e6),
}
DEFAULT_WORKLOAD = "resnet3d50"
DUMP_ELEMS = 1 << 22        # 16 MB of float32 per array: the default line's four outputs stay within 64 MB


def dump_array(t):
    """``t`` as a float32 NumPy array; above DUMP_ELEMS elements, a sample of DUMP_ELEMS of them at fixed seeded positions."""
    import torch
    t = t.detach()
    if t.numel() > DUMP_ELEMS:
        idx = torch.randint(0, t.numel(), (DUMP_ELEMS,), generator=torch.Generator().manual_seed(0)).sort().values
        t = t.reshape(-1)[idx.to(t.device)]
    return t.float().cpu().numpy()


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            pk = json.load(fh)
        return dict(hbm_gbs=pk["hbm_gbs"], tflops=pk.get("bf16_tflops_sustained", pk["bf16_tflops"]),
                    tflops_burst=pk["bf16_tflops"], source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, tflops=1400.0, tflops_burst=1590.0, source="fallback (B200_PROFILING.md)")


class ClockSampler(threading.Thread):
    """SM clock, power and throttle reasons sampled DURING the timed region.  NVML (a ~1 ms query, sampled every 5 ms) when the
    bindings are importable -- a 20-step timed region is ~80 ms, which an `nvidia-smi` subprocess (~100 ms per call) samples once
    at best; that subprocess is the fallback."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_evt = index, [], threading.Event()
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and all(v.strip().isdigit() for v in vis.split(",")) else index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _sample_nvml(self):
        n = self.nvml
        sm = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
        try:
            mask = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
        except Exception:
            mask = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
        flag = lambda bit: "Active" if mask & bit else "Not Active"
        return [str(sm), str(self.max_sm), str(n.nvmlDeviceGetPowerUsage(self.handle) / 1e3), flag(n.nvmlClocksThrottleReasonHwSlowdown),
                flag(n.nvmlClocksThrottleReasonHwThermalSlowdown), flag(n.nvmlClocksThrottleReasonSwThermalSlowdown),
                flag(n.nvmlClocksThrottleReasonSwPowerCap)]

    def run(self):
        while not self._stop_evt.is_set():
            try:
                if self.nvml is not None:
                    self.rows.append(self._sample_nvml())
                else:
                    out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                    parts = [p.strip() for p in out.strip().split(",")]
                    if len(parts) >= 7:
                        self.rows.append(parts)
            except Exception:
                pass
            self._stop_evt.wait(0.005 if self.nvml is not None else 0.1)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=10)
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(float(r[0]) for r in self.rows)
        reasons = []
        for i, name in enumerate(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")):
            if any(r[3 + i].lower().startswith("active") for r in self.rows):
                reasons.append(name)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons,
                "samples": len(self.rows), "power_w_max": max(float(r[2]) for r in self.rows),
                "source": "nvml" if self.nvml is not None else "nvidia-smi"}


# ------------------------------------------------------------------------------------------------
# model construction shared by both arms (same seeds => same weights on the reference, the port and the engine)
# ------------------------------------------------------------------------------------------------
def condition_(model, spec):
    """Non-trivial BN statistics; for the non-local net the theta/phi rescale recorded in the committed reference fixture (a
    trained-like logit regime: raw Kaiming-initialised logits reach 1e4..1e8 and make softmax an arg-max, DESIGN.md section 6)."""
    import torch
    from oracle import functional as OF
    OF.randomize_bn_(model, 1)
    if spec.get("nl_fixture"):
        fx = torch.load(os.path.join(ROOT, "tests", "golden", spec["nl_fixture"]), weights_only=False)
        OF.apply_nonlocal_factors_(model, fx["nl_factors"])
    return model


def build_ours(spec):
    import torch
    import pretorched_x_b200 as P
    torch.manual_seed(0)
    arch = spec["arch"]
    if spec.get("builder") == "trn":
        m = P.TRN(**spec["kwargs"])
    else:
        m = getattr(P, arch)(**spec["kwargs"]) if arch.startswith("r2plus1d") else getattr(P, arch)(pretrained=None, **spec["kwargs"])
    return condition_(m, spec).eval()


def oracle_forward(spec, x, sd):
    """The CPU checker's forward for a workload (oracle/functional.py restatements, pinned to reference outputs)."""
    from oracle import functional as OF
    if spec.get("builder") == "trn":
        k = spec["kwargs"]
        return OF.trn_forward(x, sd, k["arch"], "HTRN", k["num_segments"]).reshape(x.shape[0], -1)
    return OF.forward(x, sd, spec["arch"])


# ------------------------------------------------------------------------------------------------
# CPU arm (the reference's own implementation of the path on the host cores)
# ------------------------------------------------------------------------------------------------
def cpu_forward_fn(spec):
    """Returns (callable(x) -> logits, kind).  ``reference``: the unmodified reference modules (source tree in the build
    container, byte-compiled oracle/_ref on the GPU box); ``port``: the oracle restatement, only when neither exists."""
    import torch
    from oracle import functional as OF
    from oracle import reference_loader as RL
    arch = spec["arch"]
    if spec.get("builder") == "trn":
        # upstream's TRN cannot be constructed offline (its backbone factory must download a checkpoint, SURVEY.md 0.8): the CPU
        # leg is the oracle restatement of TRN.forward (pinned by the trn_* fixtures), on the same seeded weights
        sd = build_ours(spec).state_dict()
        return (lambda x: oracle_forward(spec, x, sd)), "port"
    if RL.available():
        RL.load()
        torch.manual_seed(0)
        model = condition_(RL.build(arch, **spec["kwargs"]), spec).eval()
        if arch.startswith("r2plus1d"):
            # R2Plus1D inherits ResNet3D.forward, which a resnet3d* factory call may have patched at class level to need
            # `last_linear` (SURVEY.md section 0.1); its own unpatched body is conv1..layer4 -> avgpool -> fc
            def fwd(x, m=model):
                f = m.layer4(m.layer3(m.layer2(m.layer1(m.maxpool(m.relu(m.bn1(m.conv1(x))))))))
                return m.fc(m.avgpool(f).view(f.size(0), -1))
            return fwd, "reference"
        return (lambda x: model(x)), "reference"
    sd = build_ours(spec).state_dict()
    return (lambda x: OF.forward(x, sd, arch)), "port"


def time_cpu(spec, steps, warmup):
    import torch
    from oracle import functional as OF
    fn, kind = cpu_forward_fn(spec)
    n = spec["cpu_sample"]
    x = OF.seeded_input((n,) + spec["sample"], 2)
    # "all the host threads it can use": torch's default is every core, which oversubscribes badly on large shared hosts --
    # probe a few thread counts with one forward each and keep the fastest
    ncpu = os.cpu_count() or 1
    best = None
    with torch.no_grad():
        fn(x)
        for nt in sorted({ncpu, max(1, ncpu // 2), min(ncpu, 32), min(ncpu, 16)}, reverse=True):
            torch.set_num_threads(nt)
            t0 = time.perf_counter()
            fn(x)
            dt = time.perf_counter() - t0
            if best is None or dt < best[0]:
                best = (dt, nt)
        torch.set_num_threads(best[1])
        for _ in range(warmup):
            fn(x)
        t0 = time.perf_counter()
        for _ in range(steps):
            fn(x)
        dt = time.perf_counter() - t0
    return dict(value=n * steps / dt, unit=spec["unit"], cores=torch.get_num_threads(), kind=kind,
                sample="%d steps x %d samples of %s fp32 on %d host threads (torch %s; %s)" % (
                    steps, n, "x".join(map(str, spec["sample"])), torch.get_num_threads(), torch.__version__,
                    "unmodified reference modules" if kind == "reference" else "oracle restatement"),
                ms_per_step=dt / steps * 1e3)


def run_reference_arm(args, spec, rank):
    if rank != 0:
        return
    steps = max(1, min(args.steps, 6))
    cb = time_cpu(spec, steps, 1)
    print(json.dumps({
        "impl": "reference", "metric": spec["metric"], "value": cb["value"], "unit": spec["unit"], "n_gpus": args.gpus,
        "steps": steps, "warmup": 1, "ms_per_step": cb["ms_per_step"], "higher_is_better": True, "scaling": spec["scaling"],
        "vs_baseline": None, "dtype": "f32", "data": "synthetic (seeded randn input, random-init weights)",
        "config": {"workload": "%s forward, %s (bounded CPU sample: %d per step; BASELINE.json %s)" % (
            spec["arch"], "x".join(map(str, spec["sample"])), spec["cpu_sample"], spec["config"]), "parallelism": "cpu"},
        "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": cb["value"], "unit": spec["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}), flush=True)


# ------------------------------------------------------------------------------------------------
# GPU arm, video / image classifiers
# ------------------------------------------------------------------------------------------------
def run_ours(args, spec, rank, world, local, secondary=False, outputs=None):
    """All GPU work of one classifier workload.  Returns the JSON line (rank 0; None elsewhere) WITHOUT its cpu_baseline: the CPU
    legs run in main() after the process group is gone, so that no rank sits in an NCCL barrier while rank 0 times the host.
    ``secondary``: a compact measurement riding on the default line (no fp16 / uint8 e2e variants, no nested workloads).
    ``outputs``: a dict that receives the logits of the last timed step (``dump_array``) on every rank."""
    import torch
    import torch.distributed as dist
    from pretorched_x_b200 import ops, parallel, _lib, engine
    from pretorched_x_b200.graph import GraphedForward, PipelinedForward
    from oracle import functional as OF           # checker (parity) + cpu_baseline leg only; never on the timed path

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    strong = spec["scaling"] == "strong"
    per_gpu = args.batch if args.batch else spec["batch"]
    if strong:
        total = per_gpu                               # the whole job's batch is fixed; ranks split it
        lo, hi = parallel.shard_bounds(total, world, rank)
        B = hi - lo
        if total % world:
            raise SystemExit("strong scaling of B=%d needs a GPU count that divides it" % total)
    else:
        B, total = per_gpu, per_gpu * world
    model = build_ours(spec).to(dev)
    if world > 1:
        parallel.broadcast_parameters(model)

    g = torch.Generator().manual_seed(1000 + rank)
    host_in = [torch.randn((B,) + spec["sample"], generator=g).pin_memory() for _ in range(2)]   # fp32, as the reference takes
    x_dev = host_in[0].to(dev)
    h2d_bytes = host_in[0].numel() * 4
    d2h_bytes = B * spec["classes"] * 4

    # launches per forward, counted on one eager pass (graph replays re-issue exactly these kernels)
    with torch.no_grad():
        model(x_dev)
        torch.cuda.synchronize()
        c0 = _lib.launch_count()
        model(x_dev)
        torch.cuda.synchronize()
        launches_per_fwd = _lib.launch_count() - c0

    graphed = GraphedForward(model, x_dev, warmup=2)
    # trunk schedule of the timed forward (engine.run_trunk): [(units, clips per chunk)] walked depth-first, the rest breadth-first
    schedule = None
    if hasattr(model, "layer1") and hasattr(model, "conv1"):
        plan = engine.dfs_plan()
        schedule = {"depth_first": [list(p_) for p_ in plan], "units": "0 = stem + pool, then the residual blocks in order",
                    "set_by": "B2_DFS=%s" % os.environ.get("B2_DFS")} if plan else "breadth-first (one launch per layer over the whole batch)"

    # ---- parity of the timed configuration itself (outside the timed region): the graph's logits for the first clips of the
    #      timed batch against the CPU oracle (pinned bit-exact to the reference, tests/test_oracle_golden.py) ----
    parity = None
    if rank == 0 and not args.no_check:
        k = min(spec["check_clips"], B)
        sd = {n_: v.detach().cpu() for n_, v in model.state_dict().items()}
        with torch.no_grad():
            want = oracle_forward(spec, host_in[0][:k], sd)
            got = graphed()[:k].float().cpu().reshape(k, -1)
        scale = want.abs().max().item()
        err = (got.double() - want.double()).abs().max().item() / scale
        agree = bool((got.argmax(1) == want.argmax(1)).all())
        parity = {"clips": k, "max_rel_err": err, "argmax_agree": agree, "tolerance": 5e-3,
                  "checker": "oracle/functional.py on the host (pinned bit-exact to the reference's outputs), same weights, same clips"}
        assert err <= 5e-3 and agree, "timed configuration does not match the CPU oracle: %r" % (parity,)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput ("value") ----
    for _ in range(args.warmup):
        out = graphed()
        if world > 1:
            parallel.gather_logits(out, total)     # also brings the NCCL communicator up outside the timed region
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        out = graphed()
        if world > 1:
            parallel.gather_logits(out, total)
    e1.record()
    barrier()
    clocks = sampler.stop() if sampler else None
    ms = e0.elapsed_time(e1)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    value = total * args.steps / (ms_total / 1e3)
    if outputs is not None:
        outputs[args.workload + "_logits"] = dump_array(parallel.gather_logits(out, total))

    # ---- end to end through the public API (pretorched_x_b200.graph.PipelinedForward): pinned HOST clips -> H2D -> forward ->
    #      D2H logits every step; the copy of batch i+1 overlaps the forward of batch i ----
    del graphed
    torch.cuda.empty_cache()

    def run_e2e(batches, example, fwd=None):
        pipe = PipelinedForward(fwd if fwd is not None else model, example, depth=2)
        for i in range(3):
            pipe.submit(batches[i % 2])
        pipe.drain()
        barrier()
        t0 = time.perf_counter()
        e0.record()
        for i in range(args.steps):
            slot = pipe.submit(batches[i % 2])
            if i >= 1:
                pipe.wait((slot + 1) % 2)             # consume the previous step's logits on the host
        pipe.drain()
        e1.record()
        barrier()
        wall_ms = (time.perf_counter() - t0) * 1e3
        tt = torch.tensor([max(e0.elapsed_time(e1), wall_ms)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        del pipe
        torch.cuda.empty_cache()
        sec = float(tt.item()) / 1e3
        return total * args.steps / sec, sec

    e2e_fp32, sec32 = run_e2e(host_in, x_dev)
    e2e_fp16 = e2e_u8 = None
    if not secondary:
        host_in16 = [h.half().pin_memory() for h in host_in]
        e2e_fp16, _ = run_e2e(host_in16, x_dev.half())
        del host_in16
    # decoded uint8 frames (3 bytes per pixel over PCIe), normalised on the device by ClipToStemInput (video workloads)
    if len(spec["sample"]) == 4 and not secondary and not spec.get("builder"):
        import pretorched_x_b200 as P
        from pretorched_x_b200.transforms import ClipToStemInput
        tf = ClipToStemInput(P.pretrained_settings["resnet3d50"]["kinetics-400"])
        _, T_, H_, W_ = spec["sample"]
        host_u8 = [torch.randint(0, 256, (B, T_, H_, W_, 3), generator=g, dtype=torch.uint8).pin_memory() for _ in range(2)]
        e2e_u8, _ = run_e2e(host_u8, host_u8[0].to(dev), fwd=lambda u8: model(tf(u8)))

    # ---- the other BASELINE.json configs on the same ranks, as compact sub-lines of the default line: BigGAN-deep-256 (the
    #      second half of the metric, configs[4]), R(2+1)D-34 (configs[2], strong scaling) and the non-local net (configs[3]) ----
    others = {}
    if args.workload == DEFAULT_WORKLOAD and not secondary:
        del host_in
        x_keep = x_dev
        todo = ([] if args.no_biggan else ["biggan256"]) + ([] if args.no_others else ["r2plus1d34", "nonlocal50"])
        for name in todo:
            torch.cuda.empty_cache()
            try:
                if name == "biggan256":
                    others[name] = run_biggan(args, rank, world, local, outputs=outputs)
                else:
                    sub = argparse.Namespace(**dict(vars(args), workload=name, batch=0, layers=False))
                    others[name] = run_ours(sub, WORKLOADS[name], rank, world, local, secondary=True, outputs=outputs)
            except Exception as exc:      # the contract's line must survive a failure of a secondary workload
                others[name] = {"error": "%s: %s" % (type(exc).__name__, exc)}
                print("secondary %s measurement failed: %s" % (name, others[name]["error"]), file=sys.stderr)
            torch.cuda.empty_cache()
        x_dev = x_keep
    if rank != 0:
        return None

    # ---- per-launch profile (eager, CUDA events on the launching stream) -> roofline of the dominant kernel ----
    peaks = load_peaks()
    nrep = 2
    with torch.no_grad():
        model(x_dev)
        with ops.profile() as prof:
            for _ in range(nrep):
                model(x_dev)
    rows = prof.rows
    conv_rows = [r for r in rows if r["kind"] in ("conv", "gemm", "attention")]
    conv_ms = sum(r["ms"] for r in conv_rows) / nrep
    conv_flops = sum(r["flops"] for r in conv_rows) / nrep
    all_ms = sum(r["ms"] for r in rows) / nrep
    family_tflops = conv_flops / (conv_ms * 1e-3) / 1e12
    groups = {}
    for r in conv_rows:
        gr = groups.setdefault(r["desc"], dict(ms=0.0, flops=0.0, bytes=0.0, n=0))
        gr["ms"] += r["ms"]; gr["flops"] += r["flops"]; gr["bytes"] += r["bytes"]; gr["n"] += 1
    top_desc, top = max(groups.items(), key=lambda kv: kv[1]["ms"])
    roofline = dominant_roofline(top, peaks)
    whole = spec["gflop"] * 1e9 * value / world / 1e12
    roofline.update({
        "kernel": "%s (%d launch per forward; %s)" % (top_desc, top["n"] // nrep, kernel_of(top_desc)),
        "traffic": None,      # dram bytes need an ncu pass (profiles/ncu_traffic_r02.json); not measurable inside an un-profiled run
        "algorithmic_bytes": top["bytes"] / top["n"], "algorithmic_flop": top["flops"] / top["n"],
        "ms_per_launch": top["ms"] / top["n"], "share_of_step": top["ms"] / nrep / all_ms,
        "family": {"kernels": "all %d tcgen05 conv / GEMM / attention launches of one forward" % (len(conv_rows) // nrep),
                   "achieved": family_tflops, "frac": family_tflops / peaks["tflops"], "share_of_step": conv_ms / all_ms},
        "whole_step_tflops": whole, "whole_step_frac": whole / peaks["tflops"],
        "mixed": mixed_roofline(rows, nrep, peaks, ms_total / args.steps),
    })
    if args.layers:
        print_layers(rows, nrep, all_ms, ms_total / args.steps)

    line = {
        "metric": spec["metric"], "value": value, "unit": spec["unit"], "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": spec["scaling"], "vs_baseline": None,
        "dtype": "f16", "data": "synthetic (seeded randn input, random-init weights, randomised BN statistics)",
        "config": {"workload": "%s forward, %s of %s (BASELINE.json %s)" % (
                       spec["arch"], ("B=%d in total (%d per GPU)" % (total, B)) if strong else ("B=%d per GPU" % B),
                       "x".join(map(str, spec["sample"])), spec["config"]),
                   "global_batch": total, "parallelism": "dp%d" % world,
                   "l2": "input (%.0f MB fp32) and the activations of one step (%.0f MB) exceed the 126 MB L2; no flush needed"
                         % (h2d_bytes / 1e6, spec["act_elems"] * 2 * B / 1e6),
                   "schedule": schedule,
                   "timing": "CUDA events around %d CUDA-graph replays, max over ranks" % args.steps},
        "clocks": clocks,
        "e2e": {"value": e2e_fp32, "unit": spec["unit"], "h2d_bytes_per_step": h2d_bytes * world, "d2h_bytes_per_step": d2h_bytes * world,
                "input": "fp32 NCDHW input in pinned host memory (the reference's dtype and layout); logits read back to pinned host "
                         "memory every step; H2D of step i+1 overlaps the forward of step i",
                "h2d_gbs_per_gpu": h2d_bytes * args.steps / sec32 / 1e9,
                "fp16_input_value": e2e_fp16, "fp16_input_h2d_bytes_per_step": h2d_bytes // 2 * world,
                "uint8_frames_value": e2e_u8, "uint8_frames_h2d_bytes_per_step": (h2d_bytes // 4 * world) if e2e_u8 else None,
                "note": "fp32 clips need %.0f MB per step: at the measured H2D rate the copy alone is %.2f ms per step against %.2f ms of "
                        "compute, so the fp32-host rate is the PCIe line rate; the uint8 / fp16 rows move 1/4 / 1/2 of the bytes"
                        % (h2d_bytes / 1e6, sec32 / args.steps * 1e3, ms_total / args.steps)},
        "gpu_launches": int(launches_per_fwd * args.steps),
        "parity": parity,
        "roofline": roofline,
        "cpu_baseline": None,           # filled in by main() once the process group is gone
    }
    keep = ("metric", "value", "unit", "ms_per_step", "steps", "scaling", "e2e", "gpu_launches", "roofline", "cpu_baseline", "config", "parity")
    for name, sub in others.items():
        if sub is not None:
            line[name] = sub if "error" in sub else {k: sub[k] for k in keep if k in sub}
    return line


def print_layers(rows, nrep, all_ms, step_ms):
    agg = {}
    for r in rows:
        a = agg.setdefault(r["desc"], dict(kind=r["kind"], ms=0.0, flops=0.0, bytes=0.0, n=0))
        a["ms"] += r["ms"] / nrep; a["flops"] += r["flops"] / nrep; a["bytes"] += r["bytes"] / nrep; a["n"] += 1
    peaks = load_peaks()
    print("%-52s %4s %9s %9s %8s %8s %6s" % ("layer", "n", "ms", "TFLOP/s", "GB/s", "%step", "roof"), file=sys.stderr)
    for d, a in sorted(agg.items(), key=lambda kv: -kv[1]["ms"]):
        roof = max(a["flops"] / (peaks["tflops"] * 1e12), a["bytes"] / (peaks["hbm_gbs"] * 1e9)) * 1e3
        print("%-52s %4d %9.3f %9.1f %8.0f %7.1f%% %6.2f" % (d, a["n"] // nrep, a["ms"], a["flops"] / a["ms"] / 1e9 if a["ms"] else 0,
                                                            a["bytes"] / a["ms"] / 1e6 if a["ms"] else 0, 100 * a["ms"] / all_ms,
                                                            roof / a["ms"] if a["ms"] else 0), file=sys.stderr)
    print("eager per-launch total %.3f ms/forward (graph replay: %.3f ms)" % (all_ms, step_ms), file=sys.stderr)


# ------------------------------------------------------------------------------------------------
# BASELINE.json configs[4]: BigGAN-deep-256 generator, images/sec
# ------------------------------------------------------------------------------------------------
BIGGAN_RES, BIGGAN_CH, BIGGAN_CLASSES, BIGGAN_BATCH = 256, 128, 1000, 256
BIGGAN_METRIC = "images/sec BigGAN-deep-256 generator forward"


def biggan_cpu(steps, warmup, sample=4):
    """The CPU restatement (oracle/biggan.py; the reference tree has no GAN code) on the host cores."""
    import torch
    import pretorched_x_b200 as P
    from oracle import biggan as OB
    _, sd, z, labels = OB.build_case(P.biggan_deep, BIGGAN_RES, BIGGAN_CH, BIGGAN_CLASSES, sample, init="ortho")
    ncpu = os.cpu_count() or 1
    best = None
    with torch.no_grad():
        OB.generator_forward(z, labels, sd)
        for nt in sorted({ncpu, max(1, ncpu // 2), min(ncpu, 32), min(ncpu, 16)}, reverse=True):
            torch.set_num_threads(nt)
            t0 = time.perf_counter()
            OB.generator_forward(z, labels, sd)
            dt = time.perf_counter() - t0
            if best is None or dt < best[0]:
                best = (dt, nt)
        torch.set_num_threads(best[1])
        for _ in range(warmup):
            OB.generator_forward(z, labels, sd)
        t0 = time.perf_counter()
        for _ in range(steps):
            OB.generator_forward(z, labels, sd)
        dt = time.perf_counter() - t0
    return dict(value=sample * steps / dt, unit="images/s", cores=torch.get_num_threads(), kind="port",
                sample="%d steps x %d images of BigGAN-deep-256 (ch 128) fp32 on %d host threads, oracle/biggan.py restatement "
                       "(no GAN code in the reference tree; torch %s)" % (steps, sample, torch.get_num_threads(), torch.__version__),
                ms_per_step=dt / steps * 1e3)


def run_biggan_reference_arm(args, rank):
    if rank != 0:
        return
    steps = max(1, min(args.steps, 6))
    cb = biggan_cpu(steps, 1)
    print(json.dumps({
        "impl": "reference", "metric": BIGGAN_METRIC, "value": cb["value"], "unit": "images/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": 1, "ms_per_step": cb["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic (seeded z / classes, random-init weights)",
        "config": {"workload": "BigGAN-deep-256 generator (bounded CPU sample: 4 images per step)", "parallelism": "cpu"},
        "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": cb["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}), flush=True)


def run_biggan(args, rank, world, local, outputs=None):
    import torch
    import torch.distributed as dist
    import pretorched_x_b200 as P
    from pretorched_x_b200 import ops, parallel, _lib, biggan_engine
    from pretorched_x_b200.graph import GraphedForward, PipelinedForward
    from oracle import biggan as OB                 # standing-statistics conditioning, checker, cpu_baseline leg only

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    steps = args.steps
    B = args.batch if args.batch else BIGGAN_BATCH
    # random-init generator with calibrated standing statistics (a tiny CPU pass of the restatement: O(1) activations)
    model, sd_cpu, _, _ = OB.build_case(P.biggan_deep, BIGGAN_RES, BIGGAN_CH, BIGGAN_CLASSES, 4, init="ortho")
    model = model.to(dev)
    if world > 1:
        parallel.broadcast_parameters(model)
    host = []
    for i in range(2):
        z, lab = OB.seeded_inputs(B, BIGGAN_CLASSES, 1000 + 2 * rank + i)
        host.append((z.pin_memory(), lab.pin_memory()))
    z_dev, l_dev = host[0][0].to(dev), host[0][1].to(dev)
    h2d = host[0][0].numel() * 4 + host[0][1].numel() * 8
    d2h = B * 3 * BIGGAN_RES * BIGGAN_RES * 2
    gflop = 2.0 * OB.mac_count(BIGGAN_RES, BIGGAN_CH) / 1e9

    with torch.no_grad():
        model(z_dev, l_dev, out_dtype=torch.float16)
        torch.cuda.synchronize()
        c0 = _lib.launch_count()
        model(z_dev, l_dev, out_dtype=torch.float16)
        torch.cuda.synchronize()
        launches_per_fwd = _lib.launch_count() - c0
    graphed = GraphedForward(model, (z_dev, l_dev), warmup=1, out_dtype=torch.float16)
    gplan = biggan_engine.dfs_plan(model, B, [(i, blk) for i, stage in enumerate(model.blocks) for blk in stage])
    schedule = {"depth_first": [list(p_) for p_ in gplan], "levels": "(first module, end module, images per chunk) by output resolution",
                "set_by": "B2_GAN_DFS=%s" % os.environ.get("B2_GAN_DFS")} if gplan else "whole batch per launch"

    parity = None
    if rank == 0 and not args.no_check:
        # the timed generator's first images against the CPU restatement and its fp16-storage twin (tests/test_gpu_biggan.py's bound)
        k = 2
        with torch.no_grad():
            want = OB.generator_forward(host[0][0][:k], host[0][1][:k], sd_cpu)
            twin = OB.generator_forward(host[0][0][:k], host[0][1][:k], sd_cpu, storage=OB.fp16_storage)
            got = graphed()[:k].float().cpu()
        e_rms = (got - want).pow(2).mean().sqrt().item()
        t_rms = (twin - want).pow(2).mean().sqrt().item()
        parity = {"images": k, "rms_err": e_rms, "fp16_storage_twin_rms_err": t_rms, "bound": "rms <= 1.5 x twin + 5e-4 on (-1, 1) images",
                  "checker": "oracle/biggan.py restatement of the published architecture (parity unpinned: no GAN code in the reference tree)"}
        assert e_rms <= 1.5 * t_rms + 5e-4, "timed generator does not match the CPU restatement: %r" % (parity,)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        graphed()
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        graphed()
    e1.record()
    barrier()
    clocks = sampler.stop() if sampler else None
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    value = B * world * steps / (ms_total / 1e3)
    if outputs is not None:
        outputs["biggan256_images"] = dump_array(graphed.static_out)
    del graphed
    torch.cuda.empty_cache()

    # end to end: pinned host z / class ids -> H2D -> generator -> fp16 images -> D2H into pinned host memory, every step
    pipe = PipelinedForward(model, (z_dev, l_dev), depth=2, out_dtype=torch.float16)
    for i in range(3):
        pipe.submit(host[i % 2])
    pipe.drain()
    barrier()
    t0 = time.perf_counter()
    e0.record()
    for i in range(steps):
        slot = pipe.submit(host[i % 2])
        if i >= 1:
            pipe.wait((slot + 1) % 2)
    pipe.drain()
    e1.record()
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    tt = torch.tensor([max(e0.elapsed_time(e1), wall_ms)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    e2e_value = B * world * steps / (float(tt.item()) / 1e3)
    del pipe
    torch.cuda.empty_cache()
    if rank != 0:
        return None

    peaks = load_peaks()
    with torch.no_grad():
        model(z_dev, l_dev, out_dtype=torch.float16)
        with ops.profile() as prof:
            model(z_dev, l_dev, out_dtype=torch.float16)
    rows = prof.rows
    all_ms = sum(r["ms"] for r in rows)
    agg = {}
    for r in rows:
        a = agg.setdefault(r["desc"], dict(kind=r["kind"], ms=0.0, flops=0.0, bytes=0.0, n=0))
        a["ms"] += r["ms"]; a["flops"] += r["flops"]; a["bytes"] += r["bytes"]; a["n"] += 1
    top_desc, top = max(((d, a) for d, a in agg.items() if a["kind"] in ("conv", "gemm", "attention")), key=lambda kv: kv[1]["ms"])
    hbm_rows = [r for r in rows if r["kind"] in ("ccbn", "tanh", "maxpool")]
    hbm_ms = sum(r["ms"] for r in hbm_rows)
    roofline = dominant_roofline(top, peaks)
    exec_flops = sum(r.get("exec_flops", r["flops"]) for r in rows)
    roofline.update({
        "kernel": "%s (%d launches per forward; %s)" % (top_desc, top["n"], kernel_of(top_desc)),
        "traffic": None, "algorithmic_bytes": top["bytes"] / top["n"], "algorithmic_flop": top["flops"] / top["n"],
        "ms_per_launch": top["ms"] / top["n"], "share_of_step": top["ms"] / all_ms,
        "hbm_passes": {"kernels": "ccbn_act / tanh / maxpool passes (%d launches)" % len(hbm_rows),
                       "achieved_gbs": sum(r["bytes"] for r in hbm_rows) / (hbm_ms * 1e-3) / 1e9 if hbm_ms else None,
                       "peak_gbs": peaks["hbm_gbs"], "share_of_step": hbm_ms / all_ms},
        "whole_step_tflops": gflop * 1e9 * value / world / 1e12,
        "whole_step_frac": gflop * 1e9 * value / world / 1e12 / peaks["tflops"],
        "executed_gflop_per_image": exec_flops / B / 1e9, "algorithmic_gflop_per_image": gflop,
        "mixed": mixed_roofline(rows, 1, peaks, ms_total / steps),
        "mixed_executed": mixed_roofline(rows, 1, peaks, ms_total / steps, key="exec_flops"),
    })
    if args.layers:
        print_layers(rows, 1, all_ms, ms_total / steps)
    line = ({
        "metric": BIGGAN_METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": steps, "warmup": args.warmup,
        "ms_per_step": ms_total / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16",
        "data": "synthetic (seeded z ~ N(0,1), uniform class ids; orthogonal random-init weights, calibrated standing statistics)",
        "config": {"workload": "BigGAN-deep-256 generator (ch 128, 1000 classes, %.1f GFLOP/image), B=%d z+class -> fp16 images per GPU "
                               "(BASELINE.json configs[4]); architecture absent from the reference tree: parity is against "
                               "oracle/biggan.py (unpinned)" % (gflop, B),
                   "global_batch": B * world, "parallelism": "dp%d" % world,
                   "l2": "activations of one step (tens of GB) exceed the 126 MB L2; no flush needed",
                   "schedule": schedule,
                   "timing": "CUDA events around %d CUDA-graph replays, max over ranks" % steps},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": h2d * world, "d2h_bytes_per_step": d2h * world,
                "input": "fp32 z + int64 class ids in pinned host memory; fp16 NCHW images copied back to pinned host memory every step"},
        "gpu_launches": int(launches_per_fwd * steps), "parity": parity, "roofline": roofline, "cpu_baseline": None})
    return line


def mixed_roofline(rows, nrep, peaks, step_ms, key="flops"):
    """Per-launch ("implicit-GEMM") roofline of one step: sum over the profiled launches of max(FLOP / P_tensor, bytes / BW_hbm)
    with each launch's ALGORITHMIC work (SURVEY.md section 8d; ``key='exec_flops'``: the FLOPs the kernel actually executes where
    that is less -- the phase-folded upsampling convolutions) and the measured peaks; ``frac`` = that time / the measured step."""
    p_flops, p_bytes = peaks["tflops"] * 1e12, peaks["hbm_gbs"] * 1e9
    fl = lambda r: r.get(key, r["flops"])
    t = sum(max(fl(r) / p_flops, r["bytes"] / p_bytes) for r in rows) / nrep
    return {"ms_per_step": t * 1e3, "frac": t * 1e3 / step_ms,
            "compute_only_ms": sum(fl(r) for r in rows) / nrep / p_flops * 1e3,
            "memory_only_ms": sum(r["bytes"] for r in rows) / nrep / p_bytes * 1e3,
            "definition": "sum_l max(FLOP_l / %.0f TFLOP/s, bytes_l / %.0f GB/s) over the launches of one step (%s work per "
                          "launch) / measured ms_per_step" % (peaks["tflops"], peaks["hbm_gbs"],
                                                              "executed" if key != "flops" else "algorithmic")}


def dominant_roofline(top, peaks):
    """Roofline entry of a layer group {ms, flops, bytes, n} (algorithmic work, CUDA-event time): the bound is the side of
    the ridge its arithmetic intensity falls on at the measured peaks -- tensor (TFLOP/s) or hbm (GB/s)."""
    seconds = top["ms"] * 1e-3
    intensity = top["flops"] / max(top["bytes"], 1.0)
    ridge = peaks["tflops"] * 1e12 / (peaks["hbm_gbs"] * 1e9)
    if intensity >= ridge:
        achieved = top["flops"] / seconds / 1e12
        return {"bound": "tensor", "achieved": achieved, "peak": peaks["tflops"], "unit": "TFLOP/s", "frac": achieved / peaks["tflops"],
                "peak_source": peaks["source"] + ", sustained bf16/fp16 GEMM", "flop_per_byte": intensity}
    achieved = top["bytes"] / seconds / 1e9
    return {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"],
            "peak_source": peaks["source"] + ", device-to-device copy (read + write bytes)", "flop_per_byte": intensity}


def kernel_of(desc):
    """Kernel that the C ABI dispatches a profiled layer description to (see csrc/b2_conv_api.cu)."""
    if desc.startswith("conv 7x7x7") or desc.startswith("conv 1x7x7"):
        return "stemconv_kernel"
    if desc.startswith("st2p1d"):
        return "st2p1d_kernel (fused (2+1)D pair)"
    if desc.startswith("conv 1x1x1 s111") or desc.startswith("gemm"):
        return "pgemm_kernel"
    if desc.startswith("attention"):
        return "nonlocal_attention_online_kernel"
    return "slabconv_kernel" if desc.startswith("conv") else "?"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=0, help="samples per GPU (weak) / in total (strong); default: the BASELINE config")
    ap.add_argument("--layers", action="store_true", help="print the per-layer table to stderr")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-check", action="store_true", help="skip the in-bench parity check against the CPU oracle")
    ap.add_argument("--no-biggan", action="store_true", help="skip the secondary BigGAN-deep-256 measurement of the default line")
    ap.add_argument("--no-others", action="store_true", help="skip the secondary r2plus1d34 / nonlocal50 measurements of the default line")
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=list(WORKLOADS) + ["biggan256"],
                    help="which BASELINE.json config to time (default resnet3d50 = configs[1], the contract's line)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step of every GPU workload to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    spec = WORKLOADS.get(args.workload)
    if args.impl == "reference":
        if args.workload == "biggan256":
            run_biggan_reference_arm(args, rank)
        else:
            run_reference_arm(args, spec, rank)
        return
    if world > 1:
        # the box exports NCCL_DEBUG=VERSION, which makes NCCL print its version banner on stdout in front of the JSON line
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        from pretorched_x_b200 import parallel
        parallel.init_from_env(backend="nccl")
    outputs = {} if args.dump_outputs else None
    if args.workload == "biggan256":
        line = run_biggan(args, rank, world, local, outputs=outputs)
    else:
        line = run_ours(args, spec, rank, world, local, outputs=outputs)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()          # every rank but 0 is done: nobody spins on a GPU while the host legs run
    if rank != 0 or line is None:
        return
    if outputs is not None:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in outputs.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
    if not args.no_cpu:
        def cpu_of(name, steps):
            cb = biggan_cpu(steps=steps, warmup=1) if name == "biggan256" else time_cpu(WORKLOADS[name], steps=steps, warmup=1)
            return {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
        line["cpu_baseline"] = cpu_of(args.workload, 3)
        for name in ("biggan256", "r2plus1d34", "nonlocal50"):
            if isinstance(line.get(name), dict) and "error" not in line[name]:
                line[name]["cpu_baseline"] = cpu_of(name, 2)
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
