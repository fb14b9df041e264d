"""ctypes binding of the rorl_b200 C ABI (include/rorl_b200.h) + the in-tree nvcc build.

The shared library is built IN-TREE (csrc/librorl_b200.so) for sm_100a only, so that it travels to
the GPU box with the repo snapshot.  There is deliberately no CPU implementation behind any of these
entry points: `lib()` raises if the library is missing, and every wrapper raises `RuntimeError` on
a non-zero status (negative = argument error, 1000+ = CUDA launch error).
"""
from __future__ import annotations

import ctypes
import os
import re
import subprocess
from typing import Dict, List, Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
REPO_ROOT = os.path.dirname(_HERE)
HEADER = os.path.join(REPO_ROOT, "include", "rorl_b200.h")
LIB_PATH = os.environ.get("RORL_B200_LIB") or os.path.join(CSRC, "librorl_b200.so")   # override: A/B experiments only
SOURCES = ["scan_real.cu", "scan_complex.cu", "selscan.cu", "conv1d.cu", "addnorm.cu", "losses.cu", "optim.cu",
           "gather.cu", "gru.cu", "lstm.cu", "gemm_bf16.cu", "attn.cu", "reduce.cu", "efc_head.cu", "head.cu",
           "categorical.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xptxas", "-v"]

_lib: Optional[ctypes.CDLL] = None


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def sources() -> List[str]:
    return [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def needs_build() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = sources() + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cuh")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every .cu under csrc/ into csrc/librorl_b200.so (sm_100a; cross-compiles without a GPU)."""
    if not force and not needs_build():
        return LIB_PATH
    objs = []
    procs = []
    os.makedirs(os.path.join(CSRC, "build"), exist_ok=True)
    for src in sources():
        obj = os.path.join(CSRC, "build", os.path.basename(src)[:-3] + ".o")
        objs.append(obj)
        if not force and os.path.exists(obj) and os.path.getmtime(obj) > max(
                os.path.getmtime(src), *[os.path.getmtime(os.path.join(CSRC, f)) for f in os.listdir(CSRC) if f.endswith(".cuh")]):
            continue
        cmd = [_nvcc(), *NVCC_FLAGS, "-I", CSRC, "-I", os.path.join(REPO_ROOT, "include"), "-c", src, "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    log = []
    for src, p in procs:
        out, _ = p.communicate()
        log.append(f"== {os.path.basename(src)}\n{out}")
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{out}")
    link = [_nvcc(), "-shared", "-o", LIB_PATH, *objs, "-gencode", "arch=compute_100a,code=sm_100a"]
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}")
    with open(os.path.join(CSRC, "build", "ptxas.log"), "w") as f:
        f.write("\n".join(log))
    if verbose:
        print("\n".join(log))
    global _lib
    _lib = None
    return LIB_PATH


# ---------------------------------------------------------------------------------------------
# prototypes parsed from the header, so the binding can never drift from include/rorl_b200.h
# ---------------------------------------------------------------------------------------------
_CTYPES = {
    "int": ctypes.c_int, "int64_t": ctypes.c_int64, "int32_t": ctypes.c_int32, "float": ctypes.c_float,
    "double": ctypes.c_double, "cudaStream_t": ctypes.c_void_p, "void": None, "size_t": ctypes.c_size_t,
}


def declared_prototypes() -> Dict[str, tuple]:
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    protos = {}
    for m in re.finditer(r"\b(int|int64_t|void)\s+(rorl_\w+)\s*\(([^)]*)\)\s*;", text):
        ret, name, args = m.group(1), m.group(2), m.group(3).strip()
        argtypes = []
        if args and args != "void":
            for a in args.split(","):
                a = a.strip()
                if "*" in a:
                    argtypes.append(ctypes.c_void_p)
                else:
                    ty = a.replace("const", "").split()[0]
                    argtypes.append(_CTYPES[ty])
        protos[name] = (_CTYPES[ret], argtypes)
    return protos


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"rorl_b200: {LIB_PATH} is missing. Build it with `python -c 'import __graft_entry__ as g; g.build()'`. "
                "There is no CPU fallback for the update hot path.")
        _lib = ctypes.CDLL(LIB_PATH)
        for name, (ret, argtypes) in declared_prototypes().items():
            fn = getattr(_lib, name)
            fn.restype = ret
            fn.argtypes = argtypes
    return _lib


_ERR = {-1: "invalid shape", -2: "misaligned pointer / stride", -3: "null or inconsistent argument",
        -4: "workspace too small"}


def check(status: int, what: str) -> None:
    if status != 0:
        if status >= 1000:
            raise RuntimeError(f"rorl_b200.{what}: CUDA launch error {status - 1000}")
        raise RuntimeError(f"rorl_b200.{what}: {_ERR.get(status, 'error')} (status {status})")


def ptr(t) -> Optional[int]:
    """Device pointer of a torch tensor (None -> NULL). Refuses anything that is not a CUDA fp32/int tensor."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("rorl_b200 kernels take CUDA tensors only; there is no CPU path")
    return t.data_ptr()


def stream() -> int:
    import torch
    return torch.cuda.current_stream().cuda_stream


_launches = 0


def call(name: str, *args) -> None:
    """Invoke an int-returning launcher and raise on failure; counts launches for bench.py."""
    global _launches
    _launches += 1
    check(getattr(lib(), name)(*args), name)


def add_launches(n: int) -> None:
    """Kernel launches replayed from a captured CUDA graph (counted once at capture time, per replay here)."""
    global _launches
    _launches += int(n)


def launch_count() -> int:
    return _launches
