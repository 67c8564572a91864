"""Shared helpers for the test suite (test infrastructure; may import oracle/)."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG_DIR = os.path.join(ROOT, "petit-kernel_b200")
LIB_PATH = os.path.join(PKG_DIR, "petit_kernel", "libpetit_b200.so")
HEADER = os.path.join(ROOT, "include", "causalflow", "petit", "petit.h")
GOLDEN = os.path.join(ROOT, "tests", "golden")
for p in (PKG_DIR, ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)

from oracle import petit_oracle as orc  # noqa: E402


def ensure_built():
    """Build the CUDA library + extension in-tree if they are missing."""
    if not os.path.exists(LIB_PATH):
        subprocess.check_call([sys.executable, os.path.join(PKG_DIR, "build.py")])
    return LIB_PATH


def oracle_c_lib():
    so = os.path.join(ROOT, "oracle", "libpetit_oracle.so")
    src = os.path.join(ROOT, "oracle", "petit_oracle.c")
    if not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(src):
        subprocess.check_call(["gcc", "-O2", "-fopenmp", "-fPIC", "-shared", "-o", so, src, "-lm"])
    return ctypes.CDLL(so)


def golden(name):
    return np.load(os.path.join(GOLDEN, name))


def bits16(t: torch.Tensor) -> np.ndarray:
    return t.detach().cpu().contiguous().view(torch.int16).numpy().view(np.uint16)


def from_bits16(arr: np.ndarray, dtype) -> torch.Tensor:
    return torch.from_numpy(arr.view(np.int16).copy()).view(dtype)


def pack_nvfp4(pk, q_u8, scales, n, k):
    """repack + process on the GPU through the public Python API."""
    b = pk.repack_nvfp4(q_u8.cuda().contiguous().view(torch.int32), n, k)
    s = pk.process_nvfp4_scales(scales.cuda(), n, k)
    return b, s


def pack_mxfp4(pk, q_u8, scales, n, k):
    b = pk.repack_mxfp4(q_u8.cuda().contiguous().view(torch.int32), n, k)
    s = pk.process_mxfp4_scales(scales.cuda(), n, k)
    return b, s


def stream_k_cuts_fn(lib):
    """cuts_fn for oracle.stream_k_plan: the launcher's range cuts (petit_debug_stream_k_cuts)."""

    def cuts(units, k_tiles, grid, lat, late):
        out = (ctypes.c_uint * (grid + 1))()
        assert lib.petit_debug_stream_k_cuts(units, k_tiles, grid, lat, late, out) == 0
        return list(out)

    return cuts
