"""CPU: the C-ABI shared library builds for sm_100a, loads, and exports every symbol include/b2_pretorched.h
declares; the ctypes struct mirrors match the C layout.  No compute call is made (no GPU here)."""
import ctypes
import os
import re
import subprocess
import sys

import pytest

from pretorched_x_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "b2_pretorched.h")


def declared_symbols():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(b2_[a-z0-9_]+)\s*\(", src)))


def test_header_declares_expected_surface():
    syms = declared_symbols()
    for must in ("b2_conv_ndhwc_fprop", "b2_gemm_f16", "b2_nonlocal_attention", "b2_maxpool3d_ndhwc",
                 "b2_avgpool_global_ndhwc", "b2_pack_conv_weight", "b2_last_error", "b2_version"):
        assert must in syms


def test_library_exports_every_declared_symbol():
    lib = _lib.load()
    for name in declared_symbols():
        assert hasattr(lib, name), "libb2pretorched.so does not export %s" % name
    assert set(declared_symbols()) == set(_lib.SYMBOLS), "ctypes table and header disagree"
    assert lib.b2_version() == _lib.EXPECTED_ABI == 103


def test_build_digest_covers_every_included_file():
    """The library is rebuilt only when the digest of SOURCES + HEADERS changes: a local header left out of HEADERS would let an
    edited kernel run from a stale library."""
    from pretorched_x_b200.csrc import build
    listed = {os.path.normpath(os.path.join(build.HERE, f)) for f in build.SOURCES + build.HEADERS}
    todo, seen = list(listed), set()
    while todo:
        path = todo.pop()
        if path in seen:
            continue
        seen.add(path)
        for inc in re.findall(r'^\s*#\s*include\s+"([^"]+)"', open(path).read(), flags=re.M):
            todo.append(os.path.normpath(os.path.join(os.path.dirname(path), inc)))
    assert seen <= listed, "included but not in build.HEADERS: %s" % sorted(seen - listed)


def test_ctypes_structs_match_c_layout(tmp_path):
    prog = tmp_path / "layout.c"
    prog.write_text(
        '#include <stdio.h>\n#include <stddef.h>\n#include "b2_pretorched.h"\n'
        'int main(void){printf("%zu %zu %zu %zu %zu %zu\\n", sizeof(b2_conv_args), offsetof(b2_conv_args, N),'
        ' offsetof(b2_conv_args, mode), sizeof(b2_gemm_args), offsetof(b2_gemm_args, M), offsetof(b2_gemm_args, accumulate));'
        'return 0;}\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(prog), "-o", str(exe)])
    vals = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    assert vals == [ctypes.sizeof(_lib.ConvArgs), _lib.ConvArgs.N.offset, _lib.ConvArgs.mode.offset,
                    ctypes.sizeof(_lib.GemmArgs), _lib.GemmArgs.M.offset, _lib.GemmArgs.accumulate.offset]


def test_sass_contains_blackwell_tensor_core_and_tma_instructions():
    cuobjdump = "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    sass = subprocess.run([cuobjdump, "-sass", _lib.lib_path()], capture_output=True, text=True).stdout
    assert "UTCHMMA" in sass      # tcgen05.mma
    assert "LDTM" in sass         # tcgen05.ld
    assert "UTMALDG" in sass      # TMA load
    assert "UTMASTG" in sass      # TMA store
    assert "HMMA." not in sass.replace("UTCHMMA", "")   # no legacy mma.sync path


def test_argument_validation_needs_no_gpu():
    lib = _lib.load()
    args = _lib.ConvArgs()          # all-null
    rc = lib.b2_conv_ndhwc_fprop(ctypes.byref(args), None)
    assert rc == -1 and b"null" in lib.b2_last_error()
