"""Build and load ``libstswin_b200.so`` (the C ABI of include/stswin_b200.h).

The library is compiled in-tree with nvcc for sm_100a (``build()``; called by
``__graft_entry__.build()``) and loaded with ctypes.  There is no fallback: if the
library is missing or a call fails, a Python exception is raised.
"""
from __future__ import annotations

import ctypes
import glob
import os
import shutil
import subprocess
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
# STSWIN_B200_LIB: load another build of the same ABI (A/B timing of a kernel change); never a different implementation
LIB_PATH = os.environ.get("STSWIN_B200_LIB") or os.path.join(_HERE, "libstswin_b200.so")
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "--expt-relaxed-constexpr", "-Xcompiler", "-fPIC", "-shared",
]

_lock = threading.Lock()
_lib = None


class StswinError(RuntimeError):
    """A C-ABI call returned a negative status."""


def _sources():
    return sorted(glob.glob(os.path.join(CSRC, "*.cu")))


def _stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = _sources() + glob.glob(os.path.join(CSRC, "*.h")) + glob.glob(os.path.join(CSRC, "*.cuh"))
    deps.append(os.path.join(os.path.dirname(_HERE), "include", "stswin_b200.h"))
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every CUDA source under csrc/ into one shared library (sm_100a)."""
    if not force and not _stale():
        return LIB_PATH
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise StswinError("nvcc not found: cannot build libstswin_b200.so")
    objs = []
    build_dir = os.path.join(_HERE, "build")
    os.makedirs(build_dir, exist_ok=True)
    procs = []
    for src in _sources():
        obj = os.path.join(build_dir, os.path.basename(src)[:-3] + ".o")
        objs.append(obj)
        cmd = [nvcc] + [f for f in NVCC_FLAGS if f != "-shared"] + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for cmd, p in procs:
        out, _ = p.communicate()
        if verbose and out:
            print(out)
        if p.returncode != 0:
            raise StswinError("nvcc failed: %s\n%s" % (" ".join(cmd), out))
    cmd = [nvcc, "-shared", "-o", LIB_PATH] + objs
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise StswinError("link failed: %s\n%s" % (" ".join(cmd), r.stdout))
    return LIB_PATH


_vp, _i, _i64, _fp = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_void_p

# name -> argtypes; every symbol declared in include/stswin_b200.h must appear here
SIGNATURES = {
    "stswin_abi_version": ([], ctypes.c_int),
    "stswin_last_error": ([], ctypes.c_char_p),
    "stswin_set_device": ([_i], ctypes.c_int),
    "stswin_winattn_lse_elems": ([_i] * 7, ctypes.c_int64),
    "stswin_winattn_fwd": ([_vp, _fp, _vp, _fp] + [_i] * 8 + [ctypes.c_float, _fp, _i, _vp], ctypes.c_int),
    "stswin_winattn_bwd": ([_vp, _fp, _fp, _vp, _vp, _fp, _fp] + [_i] * 8 + [ctypes.c_float, _fp, _i, _vp], ctypes.c_int),
    "stswin_layernorm_fwd": ([_vp, _fp, _fp, _vp, _fp, _fp, _i64, _i, ctypes.c_float, _i, _i, _i, _i, _vp], ctypes.c_int),
    "stswin_layernorm_bwd": ([_vp, _vp, _fp, _fp, _fp, _vp, _vp, _fp, _fp, _fp, _i64, _i, _i, _i, _i, _i, _vp], ctypes.c_int),
    "stswin_transpose": ([_vp, _i, _vp, _i, _i64, _i, _i, _vp], ctypes.c_int),
    "stswin_colsum": ([_vp, _vp, _i64, _i, _vp], ctypes.c_int),
    "stswin_copy_strided": ([_vp, _i64, _vp, _i64, _i64, _i, _vp], ctypes.c_int),
    "stswin_pixloss_labels": ([_vp, _vp] + [_i] * 8 + [_vp] * 7 + [_i64, _vp], ctypes.c_int),
    "stswin_pixloss_prepare": ([_vp, _vp, _vp] + [_i] * 7 + [_vp] * 5 + [_i64, _vp], ctypes.c_int),
    "stswin_pixloss_fwd": ([_vp, _i, _i] + [_vp] * 8 + [_i] * 6 + [_vp] * 8, ctypes.c_int),
    "stswin_pixloss_bwd": ([_vp, _i, _i] + [_vp] * 8 + [_i] * 6 + [_vp] * 4 + [_i] + [_vp] * 2 + [_i, _vp], ctypes.c_int),
    "stswin_ohem_ws_bytes": ([], ctypes.c_int64),
    "stswin_ohem_ce_fwd": ([_vp, _i, _vp, _i, _i, _i64, _i, ctypes.c_float, _i64, _fp, _vp, _fp, _fp, _vp], ctypes.c_int),
    "stswin_ohem_ce_bwd": ([_vp, _i, _vp, _i, _i, _i64, _i, _fp, _fp, _fp, _vp, _vp], ctypes.c_int),
    "stswin_ema_update": ([_vp, _vp, _vp, _vp, _i, ctypes.c_float, ctypes.c_float, _fp, _vp], ctypes.c_int),
    "stswin_lars_sgd_step": ([_vp] * 6 + [_i, _i, _i, ctypes.c_float, _fp] + [ctypes.c_float] * 2 + [_i, ctypes.c_float, _i,
                             ctypes.c_float, ctypes.c_float, _fp, _vp], ctypes.c_int),
    "stswin_adam_step": ([_vp] * 6 + [_i, _i] + [ctypes.c_float] * 6 + [_vp, _vp], ctypes.c_int),
    "stswin_sgd_step": ([_vp] * 6 + [_i, _i, ctypes.c_float, _fp] + [ctypes.c_float] * 2 + [_i, _i] + [ctypes.c_float] * 2
                        + [_vp], ctypes.c_int),
    "stswin_gather_cast": ([_vp, _vp, _vp, _i, _i, _vp], ctypes.c_int),
    "stswin_f32_split": ([_vp, _vp, _i64, _i, _i, _i, _i, _vp], ctypes.c_int),
    "stswin_f32_rowop": ([_vp, _vp, _vp, _vp, _i64, _i, _i, _vp], ctypes.c_int),
    "stswin_f32_colsum": ([_vp, _vp, _i64, _i, _vp], ctypes.c_int),
    "stswin_f32_layernorm_fwd": ([_vp] * 6 + [_i64, _i, ctypes.c_float, _i, _i, _i, _i, _vp], ctypes.c_int),
    "stswin_f32_layernorm_bwd": ([_vp] * 9 + [_i64, _i, _i, _i, _i, _i, _vp], ctypes.c_int),
    "stswin_winattn_f32_fwd": ([_vp] * 4 + [_i] * 8 + [ctypes.c_float, _vp, _i, _vp], ctypes.c_int),
    "stswin_winattn_f32_bwd": ([_vp] * 8 + [_i] * 8 + [ctypes.c_float, _vp, _i, _vp], ctypes.c_int),
    "stswin_gemm_bf16": ([_vp, _i, _i64, _vp, _i, _i64, _vp, _i64, _vp, _vp, _i64, _fp, _fp, _i, _i, _i, _i, _i, _vp], ctypes.c_int),
}


def load():
    """Return the ctypes handle (loading it on first use).  Never builds implicitly on a
    machine without the library unless nvcc is present -- and never falls back."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                build()
            elif _stale() and not os.environ.get("STSWIN_B200_LIB"):
                # sources newer than the library: rebuild when a compiler is here, refuse otherwise -- never run a
                # library that does not match csrc/ silently
                if shutil.which("nvcc") or os.path.exists("/usr/local/cuda/bin/nvcc"):
                    build()
                else:
                    raise StswinError(f"{LIB_PATH} is older than its sources under {CSRC} and nvcc is not available")
            lib = ctypes.CDLL(LIB_PATH, mode=ctypes.RTLD_GLOBAL)
            for name, (argtypes, restype) in SIGNATURES.items():
                fn = getattr(lib, name)
                fn.argtypes = argtypes
                fn.restype = restype
            _lib = lib
    return _lib


def check(status: int, what: str) -> None:
    if status != 0:
        msg = load().stswin_last_error().decode("utf-8", "replace")
        raise StswinError(f"{what} failed with status {status}: {msg}")
