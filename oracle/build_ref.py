"""TEST INFRASTRUCTURE ONLY -- builds the *unmodified* reference CUDA extensions as an oracle.

Compiles, from the sources where they lie in a checkout of the original project named by the
environment variable TRINERFLET_REFERENCE (never copied into this repo), the reference's own

  * aux_libs/raymarching/src/{raymarching.cu,bindings.cpp}  -> oracle/_ref/_raymarching_ref.so
  * aux_libs/shencoder/src/{shencoder.cu,bindings.cpp}      -> oracle/_ref/_shencoder_ref.so

for sm_100a with the reference's own nvcc flags (aux_libs/raymarching/setup.py:7-10),
except -std=c++17 (torch 2.x headers need it; the reference pins c++14 for torch 2.0).
No fast-math: IEEE division, default FMA contraction -- exactly what the reference ships.

oracle/_ref/ is git-ignored; where the built .so files are present, tests/ use them as the
bit-exact checker for ray marching.  Nothing in the product package imports them.

Usage:  python oracle/build_ref.py [raymarching|shencoder|all]
"""
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))     # (when run as a script)
from oracle import reference_path  # noqa: E402

REF = reference_path("aux_libs")
OUT = os.path.join(HERE, "_ref")

NVCC_FLAGS = [
    "-O3", "-std=c++17",
    "-U__CUDA_NO_HALF_OPERATORS__", "-U__CUDA_NO_HALF_CONVERSIONS__", "-U__CUDA_NO_HALF2_OPERATORS__",
    "-gencode", "arch=compute_100a,code=sm_100a",
]
C_FLAGS = ["-O3", "-std=c++17"]


def build(which):
    from torch.utils.cpp_extension import load
    os.environ.setdefault("TORCH_CUDA_ARCH_LIST", "10.0a")
    os.environ.setdefault("MAX_JOBS", "4")
    name = {"raymarching": "_raymarching_ref", "shencoder": "_shencoder_ref"}[which]
    src = os.path.join(REF, which, "src") if REF else ""
    if not os.path.isdir(src):
        print(f"[build_ref] no sources of the original {which} extension (TRINERFLET_REFERENCE) -- using prebuilt {name}.so if present")
        return
    bdir = os.path.join(OUT, "build_" + which)
    os.makedirs(bdir, exist_ok=True)
    cu = {"raymarching": "raymarching.cu", "shencoder": "shencoder.cu"}[which]
    load(name=name, sources=[os.path.join(src, cu), os.path.join(src, "bindings.cpp")],
         extra_cflags=C_FLAGS, extra_cuda_cflags=NVCC_FLAGS, build_directory=bdir, verbose=True)
    so = os.path.join(bdir, name + ".so")
    dst = os.path.join(OUT, name + ".so")
    if os.path.exists(so):
        import shutil
        shutil.copy2(so, dst)
        print("[build_ref] wrote", dst)


def load_ref(which):
    """Import a prebuilt reference extension (GPU box / tests). Returns module or None."""
    import importlib.util
    import torch  # noqa: F401  (the .so links against libtorch)
    name = {"raymarching": "_raymarching_ref", "shencoder": "_shencoder_ref"}[which]
    path = os.path.join(OUT, name + ".so")
    if not os.path.exists(path):
        return None
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


if __name__ == "__main__":
    arg = sys.argv[1] if len(sys.argv) > 1 else "all"
    for w in (["raymarching", "shencoder"] if arg == "all" else [arg]):
        build(w)
