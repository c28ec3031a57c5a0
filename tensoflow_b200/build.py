"""Build libtensoflow_b200.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

    python -m tensoflow_b200.build [--force] [--verbose]

The .so is git-ignored but travels to the GPU box with the repo snapshot.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
LIB = PKG / "libtensoflow_b200.so"
STAMP = PKG / ".libtensoflow_b200.stamp"
INCLUDE = PKG.parent / "include"

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden",
    "--expt-relaxed-constexpr",
]


def _nvcc() -> str:
    cand = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(cand):
        raise RuntimeError("nvcc not found: the CUDA library cannot be built")
    return cand


def sources():
    return sorted(CSRC.glob("*.cu"))


def _digest() -> str:
    h = hashlib.sha256()
    for p in sorted(list(CSRC.glob("*.cu")) + list(CSRC.glob("*.cuh")) + list(INCLUDE.glob("*.h"))):
        h.update(p.name.encode())
        h.update(p.read_bytes())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False, experiment: bool = False) -> Path:
    """experiment=True builds libtensoflow_b200_exp.so with -DTF_TC_DEBUG_SWITCHES (phase-timing switches of the stencil
    kernels; results are wrong by construction when a switch is on): only scripts/stencil_phase_probe.py loads it."""
    dig = _digest()
    if experiment:
        return _build_into(PKG / "libtensoflow_b200_exp.so", PKG / "build_exp", [*NVCC_FLAGS, "-DTF_TC_DEBUG_SWITCHES"], verbose)
    if not force and LIB.exists() and STAMP.exists() and STAMP.read_text().strip() == dig:
        return LIB
    _build_into(LIB, PKG / "build", NVCC_FLAGS, verbose)
    STAMP.write_text(dig)
    return LIB


def _build_into(LIB: Path, objdir: Path, NVCC_FLAGS, verbose: bool) -> Path:
    objdir.mkdir(exist_ok=True)
    nvcc = _nvcc()
    procs = []
    objs = []
    for src in sources():
        obj = objdir / (src.stem + ".o")
        objs.append(str(obj))
        cmd = [nvcc, *NVCC_FLAGS, "-I", str(INCLUDE), "-c", str(src), "-o", str(obj)]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write(f"--- {src.name}\n{out}\n")
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    # --no-undefined: a call into another translation unit without a definition fails here rather than when the library loads
    cmd = [nvcc, "-shared", "-Xlinker", "--no-undefined", "-o", str(LIB), *objs, "-lcudart"]
    subprocess.run(cmd, check=True)
    return LIB


PROBE_SRC = PKG.parent / "tests" / "probes" / "tc_probe.cu"
PROBE_BIN = PKG.parent / "tests" / "probes" / "_bin" / "tc_probe"


def build_probes(force: bool = False) -> Path | None:
    """tests/probes/*.cu -> tests/probes/_bin/<name>: standalone probe executables (test infrastructure; nothing of them is
    linked into libtensoflow_b200.so): tc_probe = tcgen05 operand-layout self-test / issue-rate probe, bulk_probe =
    cp.async.bulk ring streaming probe.  Returns the tc_probe path."""
    srcs = sorted(PROBE_SRC.parent.glob("*.cu"))
    if not srcs:
        return None
    h = hashlib.sha256(b"".join(p.read_bytes() for p in srcs) + (CSRC / "tc_common.cuh").read_bytes()).hexdigest()
    stamp = PROBE_BIN.parent / ".stamp"
    bins = [PROBE_BIN.parent / p.stem for p in srcs]
    if not force and all(b.exists() for b in bins) and stamp.exists() and stamp.read_text().strip() == h:
        return PROBE_BIN
    PROBE_BIN.parent.mkdir(parents=True, exist_ok=True)
    for src, out in zip(srcs, bins):
        subprocess.run([_nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-o", str(out),
                        str(src)], check=True)
    stamp.write_text(h)
    return PROBE_BIN


if __name__ == "__main__":
    path = build(force="--force" in sys.argv, verbose="--verbose" in sys.argv, experiment="--experiment" in sys.argv)
    print(path)
    print(build_probes(force="--force" in sys.argv))
