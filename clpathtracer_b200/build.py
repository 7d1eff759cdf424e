"""Build libclpt.so (host C + CUDA for sm_100a) in-tree.

The host side is C11 compiled by gcc with -ffp-contract=off (its fp32 results
are part of the parity contract); the device side is CUDA compiled by nvcc for
sm_100a only.  Everything is linked into ONE shared library,
clpathtracer_b200/libclpt.so, which exports the C ABI declared in include/*.h.
cudart is linked statically; NCCL is resolved at run time (dlopen).
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from pathlib import Path

PKG = Path(__file__).resolve().parent
ROOT = PKG.parent
CSRC = PKG / "csrc"
OBJ = PKG / "_build"
LIB = PKG / "libclpt.so"

HOST_C = ["host/hostlist.c", "host/vecmath.c", "host/kd_build.c", "host/model_io.c", "host/frame_sched.c"]
HOST_CXX = ["cuda/scene_pack.cpp"]
CUDA = ["cuda/render_kernel.cu", "cuda/kd_build_gpu.cu", "cuda/gl_interop.cu", "cuda/clstate.cu",
        "cuda/clhandler.cu"]

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and Path(cand).exists():
            return cand
    raise RuntimeError("nvcc not found: libclpt.so cannot be built (there is no CPU path)")


def _run(cmd: list[str]) -> None:
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
        raise RuntimeError(f"build step failed: {cmd[0]} {cmd[-1]}")


def _stale(out: Path, deps: list[Path]) -> bool:
    if not out.exists():
        return True
    t = out.stat().st_mtime
    return any(d.stat().st_mtime > t for d in deps if d.exists())


def build(force: bool = False, verbose: bool = False, defines: list[str] | None = None,
          tag: str | None = None) -> Path:
    """Build libclpt.so; with `tag`, build an experimental variant libclpt_<tag>.so
    with extra -D defines (selected at run time with $CLPT_LIB)."""
    global OBJ, LIB
    if tag:
        OBJ = PKG / f"_build_{tag}"
        LIB = PKG / f"libclpt_{tag}.so"
    defines = ["-D" + d for d in (defines or [])]
    OBJ.mkdir(exist_ok=True)
    inc = ["-I" + str(ROOT / "include"), "-I" + str(CSRC / "cuda")]
    headers = list((ROOT / "include").glob("*.h")) + list((CSRC / "cuda").glob("*.h")) + \
        list((CSRC / "host").glob("*.h")) + \
        list((CSRC / "cuda").glob("*.cuh")) + [Path(__file__)]
    objs: list[Path] = []
    for rel in HOST_C:
        src, out = CSRC / rel, OBJ / (Path(rel).stem + ".o")
        if force or _stale(out, [src] + headers):
            _run(["gcc", "-std=c11", "-O2", "-fPIC", "-fopenmp", "-ffp-contract=off", "-Wall", "-Wextra",
                  *inc, "-c", str(src), "-o", str(out)])
        objs.append(out)
    for rel in HOST_CXX:
        src, out = CSRC / rel, OBJ / (Path(rel).stem + ".o")
        if force or _stale(out, [src] + headers):
            _run(["g++", "-std=c++17", "-O2", "-fPIC", "-fopenmp", "-ffp-contract=off", "-Wall", *inc,
                  "-c", str(src), "-o", str(out)])
        objs.append(out)
    nvcc = _nvcc()
    for rel in CUDA:
        src, out = CSRC / rel, OBJ / (Path(rel).stem + ".o")
        if force or _stale(out, [src] + headers):
            cmd = [nvcc, *ARCH, "-std=c++17", "-O3", "-lineinfo", "-Xcompiler", "-fPIC", "-Xptxas", "-v",
                   *defines, *inc, "-c", str(src), "-o", str(out)]
            r = subprocess.run(cmd, capture_output=True, text=True)
            if r.returncode != 0:
                sys.stderr.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
                raise RuntimeError(f"nvcc failed on {rel}")
            (OBJ / (Path(rel).stem + ".ptxas.txt")).write_text(r.stderr)
            if verbose:
                sys.stderr.write(r.stderr)
        objs.append(out)
    if force or _stale(LIB, objs):
        _run([nvcc, *ARCH, "-shared", "-o", str(LIB), *[str(o) for o in objs], "-Xcompiler", "-fopenmp",
              "-Xlinker", "-Bsymbolic", "-lgomp", "-ldl", "-lm"])
    return LIB


def build_oracle() -> None:
    """Build the test-only checker (oracle/liboracle.so, and oracle/_ref when the
    reference tree is present).  Building the checker is not using it."""
    _run(["make", "-s", "-C", str(ROOT / "oracle"), "oracle"])
    _run(["make", "-s", "-C", str(ROOT / "oracle"), "ref"])
    # the rigid-instance restatement (oracle/oracle_instances_py.py builds it the same way when missing)
    _run(["gcc", "-std=c11", "-O2", "-fPIC", "-ffp-contract=off", "-fopenmp", "-w", "-shared", "-o",
          str(ROOT / "oracle" / "liboracle_instances.so"), str(ROOT / "oracle" / "oracle_instances.c"), "-lm"])


if __name__ == "__main__":
    if "--tag" in sys.argv:
        t = sys.argv[sys.argv.index("--tag") + 1]
        print(build(force=True, verbose="-v" in sys.argv, defines=[a[2:] for a in sys.argv if a.startswith("-D")], tag=t))
    else:
        print(build(force="--force" in sys.argv, verbose=True))
        build_oracle()
