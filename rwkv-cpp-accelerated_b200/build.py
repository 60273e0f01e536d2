"""In-tree builds (no JIT cache): every artefact lands next to its sources so that it
travels to the GPU box with the repo snapshot.

  librwkv_b200.so        csrc/engine.cu + generate_kernels.cu + kernels.cuh   nvcc, sm_100a only
  tools/genmodel         tools/genmodel.cpp                g++
  bindings/pybind/rwkv*.so   bindings/pybind/c_binding.cpp g++ + pybind11, links librwkv_b200.so
  oracle/librwkv_oracle.so, oracle/_ref/*                  oracle/Makefile (checker only)
"""
import os
import shutil
import subprocess
import sys
import sysconfig

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
LIB = os.path.join(PKG, "librwkv_b200.so")
GENMODEL = os.path.join(PKG, "tools", "genmodel")
ORACLE_DIR = os.path.join(ROOT, "oracle")
ORACLE_LIB = os.path.join(ORACLE_DIR, "librwkv_oracle.so")
REF_HARNESS = os.path.join(ORACLE_DIR, "_ref", "ref_harness")
PYBIND_DIR = os.path.join(PKG, "bindings", "pybind")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC", "-shared", "-cudart", "static",
]


def _newer(target, sources):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources if os.path.exists(s))


def _run(cmd, cwd=None):
    r = subprocess.run(cmd, cwd=cwd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError("build failed: %s\n%s" % (" ".join(cmd), r.stdout))
    return r.stdout


def nvcc():
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found")
    return exe


def build_engine(force=False):
    srcs = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC))]
    srcs.append(os.path.join(ROOT, "include", "rwkv_b200.h"))
    srcs.append(os.path.join(ROOT, "include", "rwkv", "sampler", "typical.h"))
    if force or _newer(LIB, srcs):
        tmp = LIB + ".tmp%d" % os.getpid()  # a snapshot taken during the build never sees a half-written library
        _run([nvcc()] + NVCC_FLAGS + ["-o", tmp, os.path.join(CSRC, "engine.cu"), os.path.join(CSRC, "generate_kernels.cu")])
        os.replace(tmp, LIB)
    return LIB


def build_genmodel(force=False):
    src = os.path.join(PKG, "tools", "genmodel.cpp")
    if force or _newer(GENMODEL, [src, os.path.join(CSRC, "binfmt.h"), os.path.join(CSRC, "q8.h")]):
        _run(["g++", "-O3", "-std=c++17", "-pthread", "-o", GENMODEL, src])
    return GENMODEL


def build_oracle(force=False):
    if force or _newer(ORACLE_LIB, [os.path.join(ORACLE_DIR, "rwkv_oracle.cpp"), os.path.join(CSRC, "binfmt.h")]):
        _run(["make", "-C", ORACLE_DIR, "librwkv_oracle.so"])
    # The reference harness can only be (re)built where /root/reference exists.
    if os.path.exists("/root/reference/include/rwkv/cuda/rwkv.cu"):
        if force or _newer(REF_HARNESS, [os.path.join(ORACLE_DIR, "ref_harness.cpp")]):
            _run(["make", "-C", ORACLE_DIR, "ref"])
        # the reference's own header / example program on top of this engine (make decides what is stale)
        _run(["make", "-C", ORACLE_DIR, "ref-b200"])
    return ORACLE_LIB


def build_pybind(force=False):
    src = os.path.join(PYBIND_DIR, "c_binding.cpp")
    if not os.path.exists(src):
        return None
    suffix = sysconfig.get_config_var("EXT_SUFFIX") or ".so"
    out = os.path.join(PYBIND_DIR, "rwkv" + suffix)
    hdrs = [os.path.join(ROOT, "include", "rwkv", "rwkv", "rwkv.h"),
            os.path.join(ROOT, "include", "rwkv", "tokenizer", "tokenizer.h"),
            os.path.join(ROOT, "include", "rwkv", "sampler", "typical.h")]
    if force or _newer(out, [src, LIB] + hdrs):
        import pybind11
        inc = ["-I" + pybind11.get_include(), "-I" + sysconfig.get_paths()["include"],
               "-I" + os.path.join(ROOT, "include")]
        _run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", src] + inc +
             ["-L" + PKG, "-lrwkv_b200", "-Wl,-rpath," + PKG, "-o", out])
    return out


def build_all(force=False):
    build_engine(force)
    build_genmodel(force)
    build_oracle(force)
    build_pybind(force)


def file_bytes(L, E, V=50277):
    """Size of a reference-format .bin (include/rwkv/rwkv/format.h: file_bytes)."""
    f64 = E + 4 * (L + 1) * E + 5 * L * E + E + 3 * L * E + 2 * L * E + 2 * E + 2 * L * E
    f32 = V * E + V + 2 * E + 6 * L * E + 2 * L * E + (3 * L * E + 2 * L * 4 * E + L * E) + 4 * E + 2 * E
    u8 = 3 * L * E * E + L * E * E + 2 * L * 4 * E * E + L * E * E + V * E
    return 16 + 8 * f64 + 4 * f32 + u8


def genmodel(n_layers, n_embed, seed, path, threads=None):
    """Write a synthetic reference-format model file (see tools/genmodel.cpp). Uses the generator build() made, so
    that bench.py can make its model from a read-only tree; builds it only when it is missing."""
    if not os.path.exists(GENMODEL):
        build_genmodel()
    cmd = [GENMODEL, str(n_layers), str(n_embed), str(seed), path]
    if threads:
        cmd.append(str(threads))
    _run(cmd)
    return path


if __name__ == "__main__":
    build_all(force="--force" in sys.argv)
    print("built:", LIB)
