"""CPU: the host-side planner of the convolution / GEMM entry points against the launches recorded on a B200.

tests/golden/conv_plans.json holds, for every distinct convolution / GEMM call of the kernel tests, the tools/*_shapes.txt layer
lists and one forward of each bench.py workload, the kernel instance, grid, block and dynamic shared memory that call launched
(written by tools/launch_trace.py).  b2_debug_conv_plan / b2_debug_gemm_plan must plan exactly that launch for the same argument
struct, here without a GPU."""
import ctypes
import json
import os

import pytest

from pretorched_x_b200 import _lib

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "conv_plans.json")


def _golden():
    with open(GOLDEN) as fh:
        return json.load(fh)


ROWS = _golden()["rows"]


def _struct(cls, fields):
    """The argument struct of a recorded row: pointers that were non-null become distinct 16-byte aligned stand-ins."""
    s = cls()
    for i, (name, typ) in enumerate(cls._fields_):
        v = fields[name]
        setattr(s, name, ((i + 1) << 20) if (typ is ctypes.c_void_p and v) else (None if typ is ctypes.c_void_p else v))
    return s


def _plan(row):
    a = row["args"]
    if row["api"] == "conv":
        return _lib.conv_plan(_struct(_lib.ConvArgs, a))
    return _lib.gemm_plan(_struct(_lib.GemmArgs, a), a["k2"] if row["api"] == "gemm2" else 0)


@pytest.fixture
def settings():
    """Applies a row's kernel-selection setting for the duration of a test."""
    lib = _lib.load()

    def apply(st):
        lib.b2_debug_set_tstack(st.get("tstack", -1))
    yield apply
    lib.b2_debug_set_tstack(-1)


def test_golden_plans_cover_every_kernel_test_case():
    g = _golden()
    assert g["sm_count"] == 148 and "B200" in g["device"]            # so plans made here, without a device, are B200 plans
    assert {r["api"] for r in ROWS} == {"conv", "gemm", "gemm2"}
    from tests import test_gpu_kernels as tk
    names = {s.split(":", 1)[1] for r in ROWS for s in r["sources"] if s.startswith(("conv_case:", "tstack_case:"))}
    assert {c[0] for c in tk.CONV_CASES + tk.TSTACK_CASES} <= names


@pytest.mark.parametrize("row", ROWS, ids=["%d:%s" % (i, r["sources"][0]) for i, r in enumerate(ROWS)])
def test_plan_matches_recorded_launch(row, settings):
    settings(row["settings"])
    p = _plan(row)
    assert (p["kernel"], [p["grid_x"], p["grid_y"], p["grid_z"]], [p["block"], 1, 1], p["smem"]) == \
        (row["kernel"], row["grid"], row["block"], row["smem"]), row["sources"]


def _conv(N, C, T, H, W, K, k, s=(1, 1, 1)):
    a = _lib.ConvArgs()
    a.x = a.w = a.scale = a.shift = a.y = 1 << 20
    a.N, a.T, a.H, a.W, a.C, a.K, a.ldy = N, T, H, W, C, K, K
    a.kt, a.kh, a.kw = k
    a.st, a.sh, a.sw = s
    a.pt, a.ph, a.pw = k[0] // 2, k[1] // 2, k[2] // 2
    return a


def test_tuning_setters_move_the_decision():
    lib = _lib.load()
    try:
        temporal = _conv(2, 144, 16, 28, 28, 64, (3, 1, 1))          # 56 items: below the temporal stack kernel's rule
        assert _lib.conv_plan(temporal)["kernel"] == "slab<64>"
        lib.b2_debug_set_tstack(1)
        assert _lib.conv_plan(temporal)["kernel"] == "tstack"
        big = _conv(16, 144, 16, 28, 28, 64, (3, 1, 1))
        lib.b2_debug_set_tstack(-1)
        assert _lib.conv_plan(big)["kernel"] == "tstack"
        lib.b2_debug_set_tstack(0)
        assert _lib.conv_plan(big)["kernel"] == "slab<64>"
        lib.b2_debug_set_tstack(-1)

        small_m = _conv(16, 512, 2, 4, 4, 1152, (1, 3, 3))            # M = 512, 9 taps: dense-M split-K
        p = _lib.conv_plan(small_m)
        assert p["kernel"] == "densem" and p["cluster"] == p["S"] > 1 and p["grid_z"] == p["S"]
        lib.b2_debug_set_densem(0, 0)
        assert _lib.conv_plan(small_m)["kernel"] != "densem"
        lib.b2_debug_set_densem(-1, 1)                                 # the rule, cluster size capped at 1
        p = _lib.conv_plan(small_m)
        assert p["kernel"] == "densem" and p["S"] == 1
        lib.b2_debug_set_densem(-1, 0)

        wide = _conv(32, 256, 2, 14, 14, 256, (3, 3, 3))              # ldy % 256 == 0
        lib.b2_debug_set_slab_wide(1)
        p = _lib.conv_plan(wide)
        assert p["kernel"] == "slab<0>" and p["bn"] == 256
        lib.b2_debug_set_slab_wide(0)
        p = _lib.conv_plan(wide)
        assert p["kernel"] == "slab<128>" and p["bn"] == 128
        lib.b2_debug_set_slab_wide(-1)

        lib.b2_debug_set_conv_algo(1)                                  # gather kernel for what the slab family would take
        assert _lib.conv_plan(big)["kernel"] == "igemm<64>"
    finally:
        lib.b2_debug_set_tstack(-1)
        lib.b2_debug_set_densem(-1, 0)
        lib.b2_debug_set_slab_wide(-1)
        lib.b2_debug_set_conv_algo(0)


def test_conv_algo_accepts_only_auto_and_gather():
    lib = _lib.load()
    try:
        assert lib.b2_debug_set_conv_algo(2) == -1                       # B2_ERR_INVALID
        assert lib.b2_debug_set_conv_algo(3) == -1
        assert _lib.conv_plan(_conv(2, 144, 16, 28, 28, 64, (3, 1, 1)))["kernel"] == "slab<64>"   # still auto
    finally:
        lib.b2_debug_set_conv_algo(0)
