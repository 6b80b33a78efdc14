"""ctypes binding of libb2pretorched.so -- the C-ABI boundary declared in include/b2_pretorched.h.

This is the only place Python touches native code.  There is deliberately no fallback: if the shared
library is missing it is built with nvcc (sm_100a); if that is impossible, or a compute entry point
is called without a B200, a RuntimeError carrying b2_last_error() is raised.
"""
import ctypes
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "csrc", "libb2pretorched.so")
_lock = threading.Lock()
_lib = None

B2_OK = 0
# The ABI revision this binding was written against (b2_version() of csrc/b2_conv_api.cu).  The argument structs below
# mirror that revision; a library from another checkout would silently ignore / misread fields, so load() insists on it.
EXPECTED_ABI = 103
B2_CONV_AUTO = 0
B2_CONV_STEM7 = 1

c_void_p = ctypes.c_void_p
c_int = ctypes.c_int
c_i32 = ctypes.c_int32


class ConvArgs(ctypes.Structure):
    """Mirror of `struct b2_conv_args` (include/b2_pretorched.h)."""
    _fields_ = [
        ("x", c_void_p), ("w", c_void_p), ("scale", c_void_p), ("shift", c_void_p),
        ("residual", c_void_p), ("y", c_void_p),
        ("N", c_i32), ("T", c_i32), ("H", c_i32), ("W", c_i32), ("C", c_i32),
        ("K", c_i32), ("ldy", c_i32), ("ldr", c_i32),
        ("kt", c_i32), ("kh", c_i32), ("kw", c_i32),
        ("st", c_i32), ("sh", c_i32), ("sw", c_i32),
        ("pt", c_i32), ("ph", c_i32), ("pw", c_i32),
        ("relu", c_i32), ("out_f32", c_i32), ("accumulate", c_i32), ("mode", c_i32), ("aff_ld", c_i32), ("upsample", c_i32), ("residual_up", c_i32), ("residual_pre", c_i32),
        ("y2", c_void_p), ("scale2", c_void_p), ("shift2", c_void_p), ("aff2_ld", c_i32), ("pool_w", c_i32),
        ("in_scale", c_void_p), ("in_shift", c_void_p), ("in_aff_ld", c_i32),
    ]


class GemmArgs(ctypes.Structure):
    """Mirror of `struct b2_gemm_args`."""
    _fields_ = [
        ("a", c_void_p), ("b", c_void_p), ("scale", c_void_p), ("shift", c_void_p),
        ("residual", c_void_p), ("d", c_void_p),
        ("M", c_i32), ("N", c_i32), ("Kd", c_i32),
        ("lda", c_i32), ("ldb", c_i32), ("ldd", c_i32), ("ldr", c_i32),
        ("per_row", c_i32), ("relu", c_i32), ("out_f32", c_i32), ("accumulate", c_i32),
        ("aff_ld", c_i32), ("aff_rows", c_i32),
        ("d2", c_void_p), ("scale2", c_void_p), ("shift2", c_void_p), ("aff2_ld", c_i32), ("aff2_rows", c_i32),
    ]


class WgradArgs(ctypes.Structure):
    """Mirror of `struct b2_wgrad_args`."""
    _fields_ = [
        ("x", c_void_p), ("g", c_void_p), ("dw", c_void_p), ("work", c_void_p),
        ("N", c_i32), ("T", c_i32), ("H", c_i32), ("W", c_i32), ("ldx", c_i32), ("C", c_i32), ("ldg", c_i32), ("K", c_i32),
        ("kt", c_i32), ("kh", c_i32), ("kw", c_i32), ("st", c_i32), ("sh", c_i32), ("sw", c_i32),
        ("pt", c_i32), ("ph", c_i32), ("pw", c_i32),
    ]


# name -> (restype, argtypes); every symbol include/b2_pretorched.h declares
SYMBOLS = {
    "b2_version": (c_int, []),
    "b2_last_error": (ctypes.c_char_p, []),
    "b2_launch_count": (ctypes.c_uint64, []),
    "b2_conv_ndhwc_fprop": (c_int, [ctypes.POINTER(ConvArgs), c_void_p]),
    "b2_conv_ndhwc_fprop_simt": (c_int, [ctypes.POINTER(ConvArgs), c_void_p]),
    "b2_pack_conv_weight_elems": (ctypes.c_size_t, [c_int] * 7),
    "b2_pack_conv_weight": (c_int, [c_void_p, c_void_p] + [c_int] * 7 + [c_void_p]),
    "b2_pack_upconv3x3_weight": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "b2_gemm_f16": (c_int, [ctypes.POINTER(GemmArgs), c_void_p]),
    "b2_gemm2_f16": (c_int, [ctypes.POINTER(GemmArgs), c_void_p, c_int, c_void_p, c_int, c_int, c_void_p]),
    "b2_nonlocal_attention": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_void_p, c_int,
                                      c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "b2_maxpool3d_ndhwc": (c_int, [c_void_p, c_void_p] + [c_int] * 14 + [c_void_p]),
    "b2_avgpool_global_ndhwc": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "b2_ncdhw_f32_to_ndhwc_f16": (c_int, [c_void_p, c_void_p] + [c_int] * 6 + [c_void_p]),
    "b2_ncdhw_f16_to_ndhwc_f16": (c_int, [c_void_p, c_void_p] + [c_int] * 6 + [c_void_p]),
    "b2_ndhwc_f16_to_ncdhw_f32": (c_int, [c_void_p, c_void_p] + [c_int] * 6 + [c_void_p]),
    "b2_cast_f32_to_f16": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "b2_shortcut_a_ndhwc": (c_int, [c_void_p, c_void_p] + [c_int] * 7 + [c_void_p]),
    "b2_concat_channels": (c_int, [c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_void_p, c_int, ctypes.c_longlong, c_void_p]),
    "b2_gather_frames": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "b2_gather_frame_tuples": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "b2_transform_image_u8": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_int, c_int,
                                      c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "b2_u8_frames_to_ndhwc4_f16": (c_int, [c_void_p, c_void_p, ctypes.c_longlong, c_int, c_void_p, c_void_p, c_void_p]),
    "b2_embed_concat": (c_int, [c_void_p] * 5 + [c_int] * 6 + [c_void_p]),
    "b2_ccbn_act_ndhwc": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p] + [c_int] * 7 + [c_void_p]),
    "b2_rgb_head_gather_tanh": (c_int, [c_void_p, c_int, c_void_p, c_void_p] + [c_int] * 5 + [c_void_p]),
    "b2_tanh_nhwc_to_nchw": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, ctypes.c_longlong, c_int, c_void_p]),
    "b2_relu_grad_sum_partials": (c_int, [ctypes.c_longlong, c_int]),
    "b2_relu_grad_sum": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, ctypes.c_longlong, c_void_p, c_void_p, c_void_p]),
    "b2_zero_dilate_scatter": (c_int, [c_void_p, c_void_p] + [c_int] * 6 + [c_void_p]),
    "b2_wgrad_workspace_floats": (ctypes.c_size_t, [ctypes.POINTER(WgradArgs)]),
    "b2_conv_ndhwc_wgrad": (c_int, [ctypes.POINTER(WgradArgs), c_void_p]),
    "b2_strided_scatter_add": (c_int, [c_void_p, c_int, c_void_p, c_int] + [c_int] * 6 + [c_void_p]),
}


# Kernel ids of the debug plan probes (enum ConvKernel in csrc/b2_conv_api.cu), one per launched template instance
CONV_KERNELS = ("none", "tstack", "slabts", "slab<64>", "slab<128>", "slab<0>", "stem<64>", "stem<128>", "densem",
                "pgemm<64,0>", "pgemm<64,1>", "pgemm<128,0>", "pgemm<128,1>", "igemm<64>", "igemm<128>")
# what b2_debug_conv_plan / b2_debug_gemm_plan write: the launch, then the kernel's tiling (0 where the kernel has no such field)
PLAN_FIELDS = ("kernel", "grid_x", "grid_y", "grid_z", "block", "smem", "cluster", "bn", "MT", "R", "PW", "WC", "wchunks", "items",
               "flex", "remap", "groups", "tiles", "cchunks", "wbytes", "S")


def _plan(name, argtype, args, *extra):
    fn = getattr(load(), name)
    fn.restype = c_int
    fn.argtypes = [ctypes.POINTER(argtype)] + [c_int] * len(extra) + [ctypes.POINTER(c_int), c_int]
    out = (c_int * len(PLAN_FIELDS))()
    check(fn(ctypes.byref(args), *extra, out, len(PLAN_FIELDS)), name)
    plan = dict(zip(PLAN_FIELDS, out))
    plan["kernel"] = CONV_KERNELS[plan["kernel"]]
    return plan


def conv_plan(args):
    """What b2_conv_ndhwc_fprop would launch for ``args`` (a ConvArgs), as a dict of PLAN_FIELDS.  Host code only: without a
    device the library plans for 148 SMs, the B200's count."""
    return _plan("b2_debug_conv_plan", ConvArgs, args)


def gemm_plan(args, k2=0):
    """What b2_gemm_f16 (k2 == 0) or b2_gemm2_f16 (a second operand pair of depth k2) would launch for ``args`` (a GemmArgs)."""
    return _plan("b2_debug_gemm_plan", GemmArgs, args, k2)


WGRAD_PLAN_FIELDS = ("grid_x", "grid_y", "block", "smem", "mt", "nt", "taps", "rects", "splits", "rect_cols", "rect_rows")


def wgrad_plan(args):
    """What b2_conv_ndhwc_wgrad would launch for ``args`` (a WgradArgs), as a dict of WGRAD_PLAN_FIELDS plus ``ranges``, the
    position-rectangle range [r0, r1) of every split.  Host code only (148 SMs without a device)."""
    lib = load()
    fn, rng = lib.b2_debug_wgrad_plan, lib.b2_debug_wgrad_split
    fn.restype, fn.argtypes = c_int, [ctypes.POINTER(WgradArgs), ctypes.POINTER(c_int), c_int]
    rng.restype, rng.argtypes = c_int, [ctypes.POINTER(WgradArgs), c_int, ctypes.POINTER(ctypes.c_longlong)]
    out = (c_int * len(WGRAD_PLAN_FIELDS))()
    check(fn(ctypes.byref(args), out, len(WGRAD_PLAN_FIELDS)), "b2_debug_wgrad_plan")
    plan = dict(zip(WGRAD_PLAN_FIELDS, out))
    ranges = []
    for s in range(plan["splits"]):
        r = (ctypes.c_longlong * 2)()
        check(rng(ctypes.byref(args), s, r), "b2_debug_wgrad_split")
        ranges.append((r[0], r[1]))
    plan["ranges"] = ranges
    return plan


def last_conv_kernel():
    """The kernel the last b2_conv_ndhwc_fprop call launched (a CONV_KERNELS name)."""
    lib = load()
    lib.b2_debug_last_conv_kernel.restype = c_int
    return CONV_KERNELS[lib.b2_debug_last_conv_kernel()]


def lib_path():
    return _LIB_PATH


def load():
    """Return the loaded shared library, building it first if it is not there."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        from .csrc import build as _build
        if _build.sources_present() and _build.have_nvcc():
            _build.build()    # digest check: rebuilds only when a source, header or flag changed since the .so was linked
        elif not os.path.exists(_LIB_PATH):
            raise RuntimeError("libb2pretorched.so is missing and cannot be built here (no nvcc / no sources): the engine has "
                               "no CPU or library fallback")
        lib = ctypes.CDLL(_LIB_PATH)
        lib.b2_version.restype = c_int
        got = lib.b2_version()
        if got != EXPECTED_ABI:
            raise RuntimeError("libb2pretorched.so reports ABI %d, this binding needs %d: stale library from another checkout -- "
                               "run `python -m pretorched_x_b200.csrc.build --force`" % (got, EXPECTED_ABI))
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(lib, name)  # AttributeError if the library does not export the symbol
            fn.restype = res
            fn.argtypes = args
        algo = os.environ.get("B2_CONV_ALGO")          # debug: "gather" disables the slab kernel (A/B timing)
        if algo:
            lib.b2_debug_set_conv_algo.restype = c_int
            lib.b2_debug_set_conv_algo.argtypes = [c_int]
            lib.b2_debug_set_conv_algo(1 if algo == "gather" else 0)
        if os.environ.get("B2_GEMM_ALGO"):             # debug: "tile" disables the persistent GEMM kernel
            lib.b2_debug_set_gemm_algo.restype = c_int
            lib.b2_debug_set_gemm_algo.argtypes = [c_int]
            lib.b2_debug_set_gemm_algo(1 if os.environ["B2_GEMM_ALGO"] == "tile" else 0)
        _lib = lib
    return _lib


def last_error():
    return load().b2_last_error().decode("utf-8", "replace")


def check(rc, what):
    if rc != B2_OK:
        raise RuntimeError("%s failed (code %d): %s" % (what, rc, last_error()))


def launch_count():
    return int(load().b2_launch_count())
