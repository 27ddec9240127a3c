"""In-tree build of the native code.

* ``ops/_srb_cuda.so``  - every sm_100a kernel + the ``torch.ops.srb`` bindings
  (``nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo``; nvcc cross-compiles
  without a GPU).  Kernel ``.cu`` files never include torch headers (seconds each);
  only the three ``*.cpp`` binding files do.
* ``native/_host_runtime.so`` - C++ host runtime (featurise / collate).

Artifacts stay in-tree (git-ignored) so they travel with a repo snapshot to a GPU
box; nothing is written to a JIT cache.  ``python -m spacy_ray_b200.build`` or
``__graft_entry__.build()``.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path
from typing import List

ROOT = Path(__file__).resolve().parent
CSRC = ROOT / "ops" / "csrc"
OUT_CUDA = ROOT / "ops" / "_srb_cuda.so"
OUT_HOST = ROOT / "native" / "_host_runtime.so"
OBJ_DIR = ROOT / "ops" / "_build"

NVCC_ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
CU_FILES = ["elementwise_kernels.cu", "elementwise_fast.cu", "ner_kernels.cu", "tagger_kernels.cu", "parser_kernels.cu", "gemm_tcgen05.cu", "comm_kernels.cu", "textcat_kernels.cu"]
CPP_FILES = ["bindings.cpp", "gemm_binding.cpp", "comm_binding.cpp"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and Path(cand).exists():
            return cand
    raise RuntimeError("nvcc not found")


def _run(cmd: List[str]) -> None:
    proc = subprocess.run(cmd, capture_output=True, text=True)
    if proc.returncode != 0:
        raise RuntimeError(f"build step failed: {' '.join(cmd)}\n{proc.stdout}\n{proc.stderr}")


def _digest(paths: List[Path], extra: str = "") -> str:
    h = hashlib.sha256(extra.encode())
    for p in sorted(paths):
        h.update(p.name.encode())
        h.update(p.read_bytes())
    return h.hexdigest()


def build_host(force: bool = False) -> Path:
    src = ROOT / "native" / "csrc" / "host_runtime.cpp"
    stamp = OUT_HOST.with_suffix(".stamp")
    dig = _digest([src])
    if not force and OUT_HOST.exists() and stamp.exists() and stamp.read_text() == dig:
        return OUT_HOST
    _run(["g++", "-O3", "-std=c++17", "-shared", "-fPIC", "-o", str(OUT_HOST), str(src)])
    stamp.write_text(dig)
    return OUT_HOST


def build_cuda(force: bool = False, verbose: bool = False) -> Path:
    import torch
    from torch.utils.cpp_extension import include_paths

    headers = list(CSRC.glob("*.h")) + list(CSRC.glob("*.cuh"))
    sources = [CSRC / f for f in CU_FILES + CPP_FILES]
    dig = _digest(sources + headers, extra=torch.__version__)
    stamp = OUT_CUDA.with_suffix(".stamp")
    if not force and OUT_CUDA.exists() and stamp.exists() and stamp.read_text() == dig:
        return OUT_CUDA
    OBJ_DIR.mkdir(parents=True, exist_ok=True)
    nvcc = _nvcc()
    cuda_home = Path(nvcc).resolve().parent.parent
    torch_inc = [f"-I{p}" for p in include_paths()]
    abi = f"-D_GLIBCXX_USE_CXX11_ABI={int(torch._C._GLIBCXX_USE_CXX11_ABI)}"
    jobs = []
    objs = []
    for f in CU_FILES:
        obj = OBJ_DIR / (f + ".o")
        objs.append(obj)
        jobs.append([nvcc, *NVCC_ARCH, "-lineinfo", "-O3", "-std=c++17", "--expt-relaxed-constexpr",
                     "-Xcompiler", "-fPIC", "-c", str(CSRC / f), "-o", str(obj)] + (["-Xptxas", "-v"] if verbose else []))
    for f in CPP_FILES:
        obj = OBJ_DIR / (f + ".o")
        objs.append(obj)
        jobs.append(["g++", "-O2", "-std=c++17", "-fPIC", abi, *torch_inc, f"-I{cuda_home / 'include'}",
                     "-DTORCH_EXTENSION_NAME=_srb_cuda", "-c", str(CSRC / f), "-o", str(obj)])
    for old in OBJ_DIR.glob("*.o"):                     # objects of sources that no longer exist
        if old not in objs:
            old.unlink()
    with ThreadPoolExecutor(max_workers=min(8, len(jobs))) as ex:
        list(ex.map(_run, jobs))
    torch_lib = Path(torch.__file__).parent / "lib"
    cudart_dir = Path(torch.__file__).parent.parent / "nvidia" / "cuda_runtime" / "lib"
    link = ["g++", "-shared", "-o", str(OUT_CUDA), *map(str, objs), f"-L{torch_lib}",
            "-lc10", "-ltorch_cpu", "-ltorch", "-lc10_cuda", "-ltorch_cuda"]
    if (cudart_dir / "libcudart.so.12").exists():
        link += [f"-L{cudart_dir}", "-l:libcudart.so.12", f"-Wl,-rpath,{cudart_dir}"]
    else:
        link += [f"-L{cuda_home / 'lib64'}", "-lcudart"]
    link += [f"-Wl,-rpath,{torch_lib}"]
    _run(link)
    stamp.write_text(dig)
    return OUT_CUDA


def build_all(force: bool = False, verbose: bool = False) -> None:
    build_host(force)
    build_cuda(force, verbose)


if __name__ == "__main__":
    build_all(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print("built:", OUT_HOST, OUT_CUDA)
