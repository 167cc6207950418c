"""In-tree build of the native libraries (no cmake, no pip): nvcc for the CUDA C-ABI library and
the generated stage libraries, g++ for the C++ front-end.  Everything lands inside the repo so
that it travels to the GPU box with the snapshot:

  optimal_control_problem_b200/lib/libocp_b200.so        CUDA kernels + C ABI (include/ocp_b200.h)
  optimal_control_problem_b200/lib/libocp_b200_host.so   C++ front-end (reference class surface) + ctypes entry points
  optimal_control_problem_b200/share/code_gen/*.so       nvcc-compiled stage libraries (include/ocp_b200_model.h)

The CPU oracle is built by oracle/build.py (test infrastructure, not part of the package).
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

PKG = Path(__file__).resolve().parent
ROOT = PKG.parent
LIB = PKG / "lib"
OBJ = PKG / "lib" / "obj"
SHARE = PKG / "share"
INCLUDE = ROOT / "include"

NVCC = os.environ.get("OCP_B200_NVCC", "nvcc")
# $CXX in this image points at a wrapper that links libstdc++ statically, which must not be mixed
# with the dynamic libstdc++ of the python process: use the system compiler unless told otherwise
CXX = os.environ.get("OCP_B200_CXX", "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]

HOST_SOURCES = [
    "host/src/casadi_lite.cpp",
    "host/src/OCPConfig.cpp",
    "host/src/OptimalControlProblem.cpp",
    "host/src/OptimalControlProblemSolve.cpp",
    "host/src/AutoDifferentiator.cpp",
    "host/src/SQPOptimizationSolver.cpp",
    "host/src/StageCodegen.cpp",
    "host/src/CasadiCInterop.cpp",
    "host/src/CuCaQP.cpp",
    "host/src/host_capi.cpp",
    "problems/problems.cpp",
]
# the half of the front-end that does not touch the device library (used by the oracle too)
FRONTEND_SOURCES = [
    "host/src/casadi_lite.cpp",
    "host/src/OCPConfig.cpp",
    "host/src/OptimalControlProblem.cpp",
    "problems/problems.cpp",
]
HOST_FLAGS = ["-std=c++17", "-O2", "-fPIC", "-Wall", "-Wno-sign-compare", "-I" + str(PKG / "host"), "-I" + str(PKG),
              "-I" + str(INCLUDE), '-DOCP_B200_INCLUDE_DIR_DEFAULT="' + str(INCLUDE) + '"']


def _run(cmd: list[str]) -> None:
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if res.returncode != 0:
        raise RuntimeError("build command failed:\n  " + " ".join(cmd) + "\n" + res.stdout)


def _stale(target: Path, deps: list[Path]) -> bool:
    if not target.exists():
        return True
    t = target.stat().st_mtime
    return any(d.stat().st_mtime > t for d in deps if d.exists())


def _headers() -> list[Path]:
    return list(PKG.rglob("*.h")) + list(PKG.rglob("*.hpp")) + list(PKG.rglob("*.cuh")) + list(INCLUDE.glob("*.h"))


def compile_objects(sources: list[str], flags: list[str], objdir: Path, tag: str = "") -> list[Path]:
    """g++ -c every source that is newer than its object (or whose headers are)."""
    objdir.mkdir(parents=True, exist_ok=True)
    hdrs = _headers()
    flag_tag = hashlib.sha1((" ".join(flags) + tag).encode()).hexdigest()[:8]
    jobs, objs = [], []
    for src in sources:
        sp = PKG / src
        op = objdir / (sp.stem + "_" + flag_tag + ".o")
        objs.append(op)
        if _stale(op, [sp] + hdrs):
            # the synthetic-input generator must give the same bits in every build (GPU arm, oracle)
            extra = ["-ffp-contract=off"] if sp.name == "problems.cpp" else []
            jobs.append([CXX, *flags, *extra, "-c", str(sp), "-o", str(op)])
    if jobs:
        with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 4)) as ex:
            list(ex.map(_run, jobs))
    return objs


CUDA_SOURCES = ["csrc/ocp_b200.cu", "csrc/direct_smem.cu", "csrc/direct_mixed.cu", "csrc/direct_multi.cu", "csrc/direct_big.cu", "csrc/direct_compact.cu"]
NVCC_FLAGS = [*ARCH, "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC", "-I" + str(INCLUDE), "-I" + str(PKG / "csrc"),
              *os.environ.get("OCP_B200_NVCC_EXTRA", "").split()]


def build_cuda(force: bool = False) -> Path:
    """nvcc -c every CUDA translation unit (in parallel), then link libocp_b200.so."""
    LIB.mkdir(parents=True, exist_ok=True)
    OBJ.mkdir(parents=True, exist_ok=True)
    out = LIB / "libocp_b200.so"
    deps = [*(PKG / "csrc").glob("*.cuh"), *(PKG / "csrc").glob("*.h"), INCLUDE / "ocp_b200.h", INCLUDE / "ocp_b200_model.h"]
    jobs, objs = [], []
    for src in CUDA_SOURCES:
        sp = PKG / src
        op = OBJ / (sp.stem + ".cu.o")
        objs.append(op)
        if force or _stale(op, [sp] + deps):
            jobs.append([NVCC, *NVCC_FLAGS, "-c", str(sp), "-o", str(op)])
    if jobs:
        with ThreadPoolExecutor(max_workers=len(jobs)) as ex:
            list(ex.map(_run, jobs))
    if force or _stale(out, objs):
        _run([NVCC, *ARCH, "-shared", "-o", str(out), *map(str, objs), "-ldl"])
    return out


def build_host(force: bool = False) -> Path:
    out = LIB / "libocp_b200_host.so"
    cuda = build_cuda()
    objs = compile_objects(HOST_SOURCES, HOST_FLAGS, OBJ)
    if force or _stale(out, objs + [cuda]):
        _run([CXX, "-shared", "-o", str(out), *map(str, objs), "-L" + str(LIB), "-locp_b200", "-Wl,-rpath,$ORIGIN",
              "-pthread", "-ldl"])
    return out


def build_all(stage_models: bool = True) -> dict:
    """Builds the two libraries and, unless told otherwise, the stage libraries of the three
    benchmark problems (code generation + nvcc; no GPU needed)."""
    out = {"cuda": build_cuda(), "host": build_host()}
    if stage_models:
        from . import Problem  # noqa: WPS433 (import after the libraries exist)
        libs = []
        for name in ("quadrotor", "cartpole", "centroidal"):
            libs.append(Problem(name).model_library)
        out["stage_libraries"] = libs
    return out


if __name__ == "__main__":
    print(build_all(stage_models="--no-models" not in sys.argv))
