"""Builds rrnco_b200/librrnco_b200.so (C-ABI, include/rrnco_b200.h) with nvcc for sm_100a, in-tree.

nvcc cross-compiles without a GPU; the .so is git-ignored but travels to the GPU box with the snapshot.
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "librrnco_b200.so")
SOURCES = ["env_kernels.cu", "rollout_kernel.cu", "rollout_kernel_tc.cu", "rollout_lean.cu", "rollout_tiled.cu", "cache_kernel.cu", "ffn_tc_kernel.cu", "step_kernels.cu", "encoder_kernels.cu", "encoder_dur_kernel.cu"]
# development switches (never set for the product build): per-phase cycle stamps, device printf, raw lo split
NVCC_FLAGS = [f"-D{k}" for k in ("RRNCO_PHASE_STAMPS", "RRNCO_DEBUG_PRINT", "RRNCO_SPLIT_LO_RAW", "RRNCO_LEAN_SELECT3") if os.environ.get(k)] + ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xptxas", "-v"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def _digest(paths):
    h = hashlib.sha256()
    for p in sorted(paths):
        with open(p, "rb") as f:
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build_library(force: bool = False, verbose: bool = False) -> str:
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh"))]
    deps.append(os.path.join(os.path.dirname(HERE), "include", "rrnco_b200.h"))
    stamp = os.path.join(HERE, "build", "stamp")
    digest = _digest(deps)
    if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read() == digest:
        return LIB
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    nvcc = _nvcc()

    def compile_one(src):
        obj = os.path.join(HERE, "build", src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        with open(obj + ".ptxas.txt", "w") as f:
            f.write(r.stderr)
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    r = subprocess.run([nvcc, "-shared", "-o", LIB, *objs], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    with open(stamp, "w") as f:
        f.write(digest)
    return LIB


TORCH_LIB = os.path.join(HERE, "librrnco_b200_torch.so")


def build_torch_ops(force: bool = False) -> str:
    """g++ csrc/torch_ops.cpp -> rrnco_b200/librrnco_b200_torch.so: the TORCH_LIBRARY registration of the C-ABI entry points
    (no device code: it links against librrnco_b200.so, which is found next to it through $ORIGIN)."""
    import torch
    from torch.utils import cpp_extension as ce
    build_library()
    src = os.path.join(CSRC, "torch_ops.cpp")
    stamp = os.path.join(HERE, "build", "stamp_torch")
    digest = _digest([src, os.path.join(os.path.dirname(HERE), "include", "rrnco_b200.h")]) + torch.__version__
    if not force and os.path.exists(TORCH_LIB) and os.path.exists(stamp) and open(stamp).read() == digest:
        return TORCH_LIB
    tlib = os.path.join(os.path.dirname(torch.__file__), "lib")
    cuda_home = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    cmd = ["g++", "-O2", "-std=c++17", "-shared", "-fPIC", f"-D_GLIBCXX_USE_CXX11_ABI={int(torch._C._GLIBCXX_USE_CXX11_ABI)}",
           *[f"-I{p}" for p in ce.include_paths()], f"-I{cuda_home}/include", src, "-o", TORCH_LIB,
           f"-L{tlib}", f"-L{HERE}", "-ltorch", "-ltorch_cpu", "-ltorch_cuda", "-lc10", "-lc10_cuda", "-l:librrnco_b200.so",
           f"-L{cuda_home}/lib64", "-lcudart", "-Wl,-rpath,$ORIGIN", f"-Wl,-rpath,{tlib}"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"torch_ops build failed:\n{r.stdout}\n{r.stderr}")
    with open(stamp, "w") as f:
        f.write(digest)
    return TORCH_LIB


TRAIN_LIB = os.path.join(HERE, "librrnco_b200_train.so")
TRAIN_SOURCES = ["ffn_train.cu", "attention_train.cu", "attention_tiled_train.cu", "logits_train.cu", "context_train.cu",
                 "pointer_train.cu", "encoder_train.cu", "encoder_dur_train.cu"]


def build_train_library(force: bool = False) -> str:
    """nvcc csrc_train/*.cu -> rrnco_b200/librrnco_b200_train.so (include/rrnco_b200_train.h): the kernels of the training
    hand-off.  A library of its own: the rollout library's build digest (profiles are stamped with it) covers csrc/ only."""
    tdir = os.path.join(HERE, "csrc_train")
    srcs = [os.path.join(tdir, f) for f in TRAIN_SOURCES if os.path.exists(os.path.join(tdir, f))]
    deps = srcs + [os.path.join(CSRC, f) for f in ("common.cuh", "tc05.cuh", "ffn_pack.cuh")]
    deps += [os.path.join(os.path.dirname(HERE), "include", f) for f in ("rrnco_b200.h", "rrnco_b200_train.h")]
    stamp = os.path.join(HERE, "build", "stamp_train")
    digest = _digest(deps)
    if not force and os.path.exists(TRAIN_LIB) and os.path.exists(stamp) and open(stamp).read() == digest:
        return TRAIN_LIB
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    nvcc = _nvcc()

    def compile_one(src):
        obj = os.path.join(HERE, "build", "train_" + os.path.basename(src).replace(".cu", ".o"))
        r = subprocess.run([nvcc, *NVCC_FLAGS, "-c", src, "-o", obj], capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        with open(obj + ".ptxas.txt", "w") as f:
            f.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=len(srcs)) as ex:
        objs = list(ex.map(compile_one, srcs))
    r = subprocess.run([nvcc, "-shared", "-o", TRAIN_LIB, *objs], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    with open(stamp, "w") as f:
        f.write(digest)
    return TRAIN_LIB


def build_digest() -> str:
    """Digest of the CUDA sources + flags the library on disk was built from (profiles stamp their numbers with it)."""
    stamp = os.path.join(HERE, "build", "stamp")
    return open(stamp).read().strip() if os.path.exists(stamp) else ""


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose=True))
    print(build_torch_ops(force="--force" in sys.argv))
    print(build_train_library(force="--force" in sys.argv))
