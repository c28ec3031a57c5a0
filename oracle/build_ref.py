"""TEST INFRASTRUCTURE ONLY.  Recipe for oracle/_ref/: compiles the reference's own CUDA sources, from where they lie under
/root/reference, into shared libraries the golden-fixture generators load on the GPU box.

    python oracle/build_ref.py [--force]

The package build (__graft_entry__.build) does not run this: run it by hand before oracle/gen_golden_prefilter.py, which
loads whatever library oracle/_ref/ holds.

oracle/_ref/libref_cubemap.so = oracle/ref_cubemap_shim.cu (C-ABI launchers, ours)
                                + /root/reference/network/renderutils/c_src/{cubemap.cu (included by the shim), common.cpp}
built with plain nvcc for sm_100a (the reference's own build goes through torch.utils.cpp_extension and its torch binding,
which is not used here).  oracle/_ref/ is git-ignored (no reference code in the history) but travels to the GPU box.
Nothing under tensoflow_b200/ loads these libraries."""
from __future__ import annotations

import shutil
import subprocess
import sys
from pathlib import Path

HERE = Path(__file__).resolve().parent
REF_SRC = Path("/root/reference/network/renderutils/c_src")
OUT = HERE / "_ref"


def build(force: bool = False):
    """Returns the library path, or None when /root/reference is absent (GPU box: the prebuilt file is used)."""
    lib = OUT / "libref_cubemap.so"
    if not REF_SRC.exists():
        return lib if lib.exists() else None
    srcs = [HERE / "ref_cubemap_shim.cu", REF_SRC / "cubemap.cu", REF_SRC / "common.cpp", REF_SRC / "cubemap.h", REF_SRC / "common.h",
            REF_SRC / "tensor.h", REF_SRC / "vec3f.h", REF_SRC / "vec4f.h"]
    if not force and lib.exists() and all(lib.stat().st_mtime >= s.stat().st_mtime for s in srcs):
        return lib
    OUT.mkdir(exist_ok=True)
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-shared", "-Xcompiler", "-fPIC", "-w",
           "-I", str(REF_SRC), "-o", str(lib), str(HERE / "ref_cubemap_shim.cu"), str(REF_SRC / "common.cpp")]
    subprocess.run(cmd, check=True)
    return lib


if __name__ == "__main__":
    print(build(force="--force" in sys.argv))
