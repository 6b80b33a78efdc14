"""Which kernel each convolution / GEMM call launches, with its grid, block and dynamic shared memory.

    python tools/launch_trace.py OUT.json [--sequence SEQ.json] [--skip-workloads]

Wraps b2_conv_ndhwc_fprop, b2_gemm_f16 and b2_gemm2_f16 on the loaded library and runs, under torch.profiler:
  * every CONV_CASES (tcgen05 leg), TSTACK_CASES (temporal stack kernel forced on) and GEMM_CASES row of
    tests/test_gpu_kernels.py, its rule-driven temporal stack case and its two-operand GEMM case;
  * every line of tools/*_shapes.txt (``N Cin T H W K kt kh kw st sh sw [res]``, "same" padding, BN + ReLU);
  * one eager forward of each bench.py workload at its bench batch (resnet3d50, r2plus1d34, nonlocal50, resnet18, biggan256).
Each call is recorded with its argument struct (pointers reduced to 0 / 1 for null / non-null) and the one kernel launch it
made.  The profiler's shared memory is static plus dynamic bytes; the static part of each kernel comes from the ptxas lines of
pretorched_x_b200/csrc/build.log, and what is stored is the dynamic part.  OUT.json holds one row per distinct (entry point,
argument struct, kernel-selection setting); SEQ.json gets every call in launch order, to compare two builds launch for launch.

Imports go through sys.path, so PYTHONPATH=<other checkout> traces that checkout's library and test cases.
"""
import ctypes
import glob
import json
import os
import re
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# right after the PYTHONPATH entries: a checkout named there takes precedence, and this one over installed packages
sys.path.insert(1 + len([p for p in os.environ.get("PYTHONPATH", "").split(os.pathsep) if p]), ROOT)

import torch  # noqa: E402
import torch.nn as nn  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402

FAMILY = re.compile(r"(tstack|slabts|slabconv|stemconv|densem|pgemm|igemm)_kernel(?:<([^>]*)>|I((?:Li\d+E)+)E)?")
SHORT = {"slabconv": "slab", "stemconv": "stem"}


def kernel_id(name):
    """'void b2::pgemm_kernel<64, 1>(...)' or its mangled form -> 'pgemm<64,1>'; None for kernels of other entry points."""
    m = FAMILY.search(name)
    if not m:
        return None
    fam = SHORT.get(m.group(1), m.group(1))
    targs = re.findall(r"\d+", m.group(2) or m.group(3) or "")
    return fam + ("<%s>" % ",".join(targs) if targs else "")


def static_smem(lib_dir):
    """kernel id -> static shared memory bytes, from the `-Xptxas -v` lines the build logs."""
    out, cur = {}, None
    with open(os.path.join(lib_dir, "build.log")) as fh:
        for line in fh:
            m = re.search(r"Compiling entry function '([^']+)'", line)
            if m:
                cur = kernel_id(m.group(1))
                if cur is not None:
                    out.setdefault(cur, 0)
                continue
            m = re.search(r"(\d+) bytes smem", line)
            if m and cur is not None and line.lstrip().startswith("ptxas info    : Used"):
                out[cur] = int(m.group(1))
    return out


def struct_dict(s):
    return {name: (int(bool(getattr(s, name))) if typ is ctypes.c_void_p else int(getattr(s, name))) for name, typ in s._fields_}


class Recorder:
    def __init__(self, lib):
        self.lib, self.calls, self.source, self.settings, self.active = lib, [], "", {}, False
        conv, gemm, gemm2 = lib.b2_conv_ndhwc_fprop, lib.b2_gemm_f16, lib.b2_gemm2_f16

        def rec(api, args, extra, rc):
            if rc == 0 and self.active:
                self.calls.append(dict(api=api, args=dict(struct_dict(args._obj), **extra), settings=dict(self.settings),
                                       source=self.source))
            return rc

        # ops.py looks the entry points up on the library object per call, so instance attributes take their place
        lib.b2_conv_ndhwc_fprop = lambda a, st: rec("conv", a, {}, conv(a, st))
        lib.b2_gemm_f16 = lambda g, st: rec("gemm", g, {}, gemm(g, st))
        lib.b2_gemm2_f16 = lambda g, a2, lda2, b2, ldb2, k2, st: rec(
            "gemm2", g, dict(a2=int(bool(a2)), lda2=lda2, b2=int(bool(b2)), ldb2=ldb2, k2=k2), gemm2(g, a2, lda2, b2, ldb2, k2, st))

    def run(self, source, fn, settings=None):
        """Runs fn() under the profiler and pairs each successful call it made with its kernel launch."""
        self.source, self.settings = source, settings or {}
        n0 = len(self.calls)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            self.active = True
            try:
                fn()
            finally:
                self.active = False
            torch.cuda.synchronize()
        with tempfile.TemporaryDirectory() as tmp:
            path = os.path.join(tmp, "trace.json")
            prof.export_chrome_trace(path)
            with open(path) as fh:
                events = json.load(fh)["traceEvents"]
        kernels = sorted((e for e in events if e.get("cat") == "kernel" and kernel_id(e["name"])), key=lambda e: e["ts"])
        mine = self.calls[n0:]
        assert len(kernels) == len(mine), "%s: %d convolution / GEMM calls but %d kernel launches" % (source, len(mine), len(kernels))
        for c, k in zip(mine, kernels):
            c["kernel"] = kernel_id(k["name"])
            c["grid"], c["block"], c["smem_total"] = list(k["args"]["grid"]), list(k["args"]["block"]), int(k["args"]["shared memory"])


def test_cases(rec, dev):
    from tests import test_gpu_kernels as tk
    from pretorched_x_b200 import _lib
    lib = _lib.load()
    for case in tk.CONV_CASES:
        rec.run("conv_case:" + case[0], lambda: tk.check_conv_case(dev, case, False))
    lib.b2_debug_set_tstack(1)
    try:
        for case in tk.TSTACK_CASES:
            rec.run("tstack_case:" + case[0], lambda: tk.check_conv_case(dev, case, False), {"tstack": 1})
    finally:
        lib.b2_debug_set_tstack(-1)
    rec.run("tstack_rule_case", lambda: tk.test_temporal_stack_kernel_many_items_per_cta(dev))
    for case in tk.GEMM_CASES:
        rec.run("gemm_case:" + case[0], lambda: tk.test_gemm_matches_oracle(dev, case))
    rec.run("gemm2_case", lambda: tk.test_two_operand_gemm_matches_oracle(dev))


def shape_lines(rec, dev):
    from pretorched_x_b200 import engine, ops
    for path in sorted(glob.glob(os.path.join(ROOT, "tools", "*_shapes.txt"))):
        for i, line in enumerate(open(path)):
            sp = line.split()
            if not sp or line.startswith("#"):
                continue
            N, Cin, T, H, W, K, kt, kh, kw, st, sh, sw = [int(v) for v in sp[:12]]
            torch.manual_seed(0)
            conv = nn.Conv3d(Cin, K, (kt, kh, kw), stride=(st, sh, sw), padding=(kt // 2, kh // 2, kw // 2), bias=False).to(dev)
            bn = nn.BatchNorm3d(K).eval().to(dev)

            def fwd():
                with torch.no_grad():
                    x = ops.from_ncdhw(torch.randn(N, Cin, T, H, W, device=dev))
                    y = engine.conv_bn_act(conv, bn, x, relu=True)
                    if len(sp) > 12:
                        res = ops.Act(torch.zeros_like(y.data), y.N, y.T, y.H, y.W, y.C)
                        engine.conv_bn_act(conv, bn, x, residual=res, relu=True)
            rec.run("shapes:%s:%d" % (os.path.basename(path), i + 1), fwd)


def workloads(rec, dev):
    import bench
    for name in ("resnet3d50", "r2plus1d34", "nonlocal50", "resnet18"):
        spec = bench.WORKLOADS[name]
        m = bench.build_ours(spec).to(dev)
        x = torch.randn((spec["batch"],) + spec["sample"], generator=torch.Generator().manual_seed(1)).to(dev)
        with torch.no_grad():
            m(x)                                      # packs the weights (their own launches) outside the recorded forward
            torch.cuda.synchronize()
            rec.run("workload:" + name, lambda: m(x))
        del m, x
        torch.cuda.empty_cache()
    import pretorched_x_b200 as P
    from oracle import biggan as OB
    model = OB.build_case(P.biggan_deep, bench.BIGGAN_RES, bench.BIGGAN_CH, bench.BIGGAN_CLASSES, 4, init="ortho")[0].to(dev)
    z, lab = OB.seeded_inputs(bench.BIGGAN_BATCH, bench.BIGGAN_CLASSES, 1000)
    z, lab = z.to(dev), lab.to(dev)
    with torch.no_grad():
        model(z, lab, out_dtype=torch.float16)
        torch.cuda.synchronize()
        rec.run("workload:biggan256", lambda: model(z, lab, out_dtype=torch.float16))


def write_json(path, doc):
    """One row per line, so that a changed plan is a one-line diff."""
    with open(path, "w") as fh:
        head = ",\n".join(" %s: %s" % (json.dumps(k), json.dumps(v)) for k, v in doc.items() if k != "rows")
        fh.write("{\n%s,\n \"rows\": [\n  %s\n ]\n}\n" % (head, ",\n  ".join(json.dumps(r, sort_keys=True) for r in doc["rows"])))


def main():
    out_path = sys.argv[1]
    from pretorched_x_b200 import _lib
    lib = _lib.load()
    dev = torch.device("cuda:0")
    rec = Recorder(lib)
    test_cases(rec, dev)
    shape_lines(rec, dev)
    if "--skip-workloads" not in sys.argv:
        workloads(rec, dev)
    static = static_smem(os.path.dirname(_lib.lib_path()))
    rows, seen = [], {}
    for c in rec.calls:
        c["smem"] = c.pop("smem_total") - static[c["kernel"]]
        key = json.dumps([c["api"], c["args"], c["settings"]], sort_keys=True)
        launch = [c["kernel"], c["grid"], c["block"], c["smem"]]
        if key in seen:
            row = rows[seen[key]]
            assert [row["kernel"], row["grid"], row["block"], row["smem"]] == launch, "same arguments, different launch: %s" % key
            row["sources"].append(c["source"])
            continue
        seen[key] = len(rows)
        rows.append(dict(api=c["api"], args=c["args"], settings=c["settings"], sources=[c["source"]], kernel=c["kernel"],
                         grid=c["grid"], block=c["block"], smem=c["smem"]))
    doc = dict(device=torch.cuda.get_device_name(dev), sm_count=torch.cuda.get_device_properties(dev).multi_processor_count,
               rows=rows)
    write_json(out_path, doc)
    if "--sequence" in sys.argv:
        doc["rows"] = [[c["source"], c["kernel"], c["grid"], c["block"], c["smem"]] for c in rec.calls]
        write_json(sys.argv[sys.argv.index("--sequence") + 1], doc)
    print("%d calls, %d distinct rows -> %s" % (len(rec.calls), len(rows), out_path))


if __name__ == "__main__":
    main()
