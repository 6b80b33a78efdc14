"""Build libb2pretorched.so (sm_100a only) in-tree with nvcc.

Usage:  python -m pretorched_x_b200.csrc.build [--force] [--verbose]

The shared library is the drop-in boundary (include/b2_pretorched.h); it links only against the
CUDA runtime.  It is git-ignored but travels to the GPU box with the gpurun snapshot.
"""
import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = ["b2_host.cu", "b2_conv_api.cu", "b2_aux.cu", "b2_attention.cu", "b2_gan.cu", "b2_image.cu", "b2_probe.cu", "b2_train.cu"]
HEADERS = ["b2_ptx.cuh", "b2_igemm.cuh", "b2_densem.cuh", "b2_pgemm.cuh", "b2_slabconv.cuh", "b2_slabts.cuh", "b2_tstack.cuh", "b2_stemconv.cuh",
           "b2_host.h", "../../include/b2_pretorched.h"]
LIB = os.path.join(HERE, "libb2pretorched.so")
STAMP = os.path.join(HERE, ".build_stamp")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC",
    "--use_fast_math",
    "-Xptxas", "-v",
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; cannot build the sm_100a extension")


def have_nvcc():
    try:
        _nvcc()
        return True
    except RuntimeError:
        return False


def sources_present():
    return all(os.path.exists(os.path.join(HERE, f)) for f in SOURCES + HEADERS)


def _digest():
    h = hashlib.sha256()
    for f in SOURCES + HEADERS:
        with open(os.path.join(HERE, f), "rb") as fh:
            h.update(fh.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force=False, verbose=False):
    """Compile every CUDA source for sm_100a and link the shared library.  Returns its path."""
    dig = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(STAMP):
        with open(STAMP) as fh:
            if fh.read().strip() == dig:
                return LIB
    nvcc = _nvcc()
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(HERE, src.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + ["-c", os.path.join(HERE, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    log = []
    for src, pr in procs:
        out, _ = pr.communicate()
        log.append("== %s ==\n%s" % (src, out))
        if pr.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s" % (src, out))
    cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart"]
    out = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if out.returncode != 0:
        raise RuntimeError("link failed:\n%s" % out.stdout)
    with open(os.path.join(HERE, "build.log"), "w") as fh:
        fh.write("\n".join(log))
    with open(STAMP, "w") as fh:
        fh.write(dig)
    if verbose:
        print("\n".join(log))
    return LIB


if __name__ == "__main__":
    path = build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(path)
