"""ctypes binding of libtfem_b200.so (the C ABI declared in include/tfem_b200.h).

There is no CPU fallback: if the library is missing or a call fails, the caller gets an
exception.  The library is loaded lazily so that host-side logic (mesh topology, symbolic CSR)
can be imported and unit-tested on a box without the built library.
"""

from __future__ import annotations

import ctypes
import os
import re
import sys
import threading
from ctypes import POINTER, Structure, c_char_p, c_double, c_int, c_int32, c_int64, c_uint32, c_void_p

import torch

PKG = os.path.dirname(os.path.abspath(__file__))
# TFEM_B200_LIB selects another build of the same ABI (profiling variants); default: the in-tree library
LIB_PATH = os.environ.get("TFEM_B200_LIB") or os.path.join(PKG, "lib", "libtfem_b200.so")
HEADER = os.path.join(os.path.dirname(PKG), "include", "tfem_b200.h")

TFEM_SRC_NONE, TFEM_SRC_SAMPLED, TFEM_SRC_CONST, TFEM_SRC_SINSIN = 0, 1, 2, 3


class TfemError(RuntimeError):
    """A C-ABI call returned a negative tfem_status."""


class Source(Structure):
    """struct tfem_source."""

    _fields_ = [("kind", c_int32), ("p", c_double * 4)]


class Bilinear(Structure):
    """struct tfem_bilinear."""

    _fields_ = [("alpha", c_double), ("beta", c_double)]


class AmgLevel(Structure):
    """struct tfem_amg_level."""

    _fields_ = [("n", c_int64), ("n_coarse", c_int64)] + [
        (name, c_void_p)
        for name in ("a_crow", "a_col", "a_val", "p_crow", "p_col", "p_val", "r_crow", "r_col", "r_val", "wdinv", "x", "rc", "ec")
    ]


class TilePlan(Structure):
    """struct tfem_tile_plan."""

    _fields_ = [
        ("n_tiles", c_int64),
        ("tile_list", c_void_p),
        ("tile_desc", c_void_p),
        ("inst_blob", c_void_p),
        ("tpl_desc", c_void_p),
        ("tpl_blob", c_void_p),
        ("max_vert", c_int32),
        ("max_elem", c_int32),
        ("max_inst_words", c_int32),
        ("max_tb_words", c_int32),
        ("max_tc_words", c_int32),
        ("has_elem_ids", c_int32),
        ("table_bytes", c_int32),
        ("od_base", c_int32 * 3),
        ("consumer_threads", c_int32),
        ("reserve_ctas", c_int32),
        ("n_progress_tiles", c_int32),
        ("progress", c_void_p),
    ]


P = c_void_p
I64 = c_int64
_TYPED = {
    "tfem_tri_p1_geometry": [I64, I64, I64, P, P, c_int, P, P, P, P, P, P, P, P, P],
    "tfem_edge_p1_geometry": [I64, I64, P, c_int, P, P, P, P, P, P, P, P],
    "tfem_quad_reduce": [I64, c_int, c_int, P, I64, I64, P, P, P],
    "tfem_scatter_bilinear": [I64, P, P, P, P, P],
    "tfem_scatter_linear": [I64, P, P, P, P, P],
    "tfem_tri_p1_local_forms": [I64, I64, I64, P, P, c_int, P, P, P, P, POINTER(Bilinear), POINTER(Source), P, P, P, P],
    "tfem_tri_p1_weighted_local_forms": [I64, I64, I64, P, P, c_int, P, P, P, P, POINTER(Bilinear), POINTER(Source), P, P, P, P, P,
                                         P],
    "tfem_tri_p1_assemble_csr": [POINTER(TilePlan), P, c_int, POINTER(Bilinear), POINTER(Source), P, P, P],
    "tfem_tri_p1_assemble_csr_ex": [POINTER(TilePlan), P, c_int, POINTER(Bilinear), POINTER(Source), P, I64, P, P, P, P],
    "tfem_weak_residual_local": [I64, I64, I64, P, P, c_int, P, P, P, P, POINTER(Source), P, P, P, P],
    "tfem_weak_residual_tiled": [POINTER(TilePlan), P, c_int, P, P, I64, P, P, P, P],
    "tfem_weak_residual_bwd": [I64, I64, I64, P, P, P, c_int, P, P, P, P, P, P],
    "tfem_batched_weak_residual": [I64, c_int, c_int, P, P, c_int, POINTER(Source), P, P, P, P],
    "tfem_h1_error": [I64, I64, I64, P, P, c_int, P, c_int, P, P, P, P, P, P],
    "tfem_interp_cells": [I64, P, P, c_int, c_int, P, P, P, P],
    "tfem_interp_edges": [I64, I64, I64, P, P, P, P, c_int, P, c_int, P, P, P, P],
    "tfem_interp_cells_bwd": [I64, P, c_int, c_int, P, P, P, P],
    "tfem_interp_edges_bwd": [I64, I64, I64, P, P, P, c_int, P, c_int, P, P, P, P],
    "tfem_edge_jump": [I64, c_int, c_int, P, P, P, P, P, P],
    "tfem_csr_spmv": [I64, P, P, P, P, P, P, P],
    "tfem_cg_iteration": [I64, P, P, P, P, P, P, P, P, P, P, P, c_int32, P, P],
    "tfem_pcg_iteration": [I64, P, P, P, P, POINTER(AmgLevel), c_int32, P, I64, P, P, P, P, P, P, c_int32, P, P],
    "tfem_amg_vcycle": [POINTER(AmgLevel), c_int32, P, I64, P, P, P],
    "tfem_amg_strength": [I64, P, P, P, c_double, P, P, P],
    "tfem_csr_spgemm": [I64, P, P, P, c_int, P, P, P, I64, I64, I64, P, I64, P, P, P, P, P],
    "tfem_csr_spgemm_numeric": [I64, P, P, P, P, P, P, P, P, P, P, P],
    "tfem_amg_diag": [I64, P, P, P, P, P],
    "tfem_amg_smoother": [I64, P, P, P, P, c_double, P, P, P],
    "tfem_gather": [I64, P, P, c_double, P, P],
    "tfem_mlp_value_grad": [I64, c_int, c_int, c_int, c_int, P, P, P, P, P],
    "tfem_mlp_value_grad_bwd": [I64, c_int, c_int, c_int, c_int, P, P, P, P, P, c_int, P, P],
    "tfem_iface_pack": [I64, P, P, P, P],
    "tfem_iface_pack_after": [I64, P, P, P, P, c_uint32, P],
    "tfem_iface_unpack_add": [I64, P, P, P, P],
}
_UNTYPED = {
    "tfem_coo_keys": ([I64, P, I64, P, P], c_int),
    "tfem_csr_symbolic_workspace": ([I64, I64, POINTER(c_int64)], c_int),
    "tfem_csr_symbolic": ([I64, P, I64, P, I64, P, P, P, P, P, P, P, P, P], c_int),
    "tfem_amg_mis2_round": ([I64, P, P, P, c_int32, c_int, P, P, P, P], c_int),
    "tfem_amg_aggregate_workspace": ([I64, POINTER(c_int64)], c_int),
    "tfem_amg_aggregate": ([I64, P, P, P, P, P, I64, P, P, P], c_int),
    "tfem_csr_spgemm_workspace": ([I64, I64, POINTER(c_int64)], c_int),
    "tfem_half_edges_workspace": ([I64, I64, POINTER(c_int64)], c_int),
    "tfem_half_edges": ([I64, I64, I64, P, POINTER(c_int32), P, I64, P, P, P, P, P, P], c_int),
    "tfem_edge_cells": ([I64, I64, I64, P, c_int, P, P, I64, P, P, P], c_int),
    "tfem_interior_edge_geometry_f64": ([I64, I64, I64, I64, P, P, P, P, P, P, P, P], c_int),
    "tfem_interior_edge_geometry_f32": ([I64, I64, I64, I64, P, P, P, P, P, P, P, P], c_int),
    "tfem_abi_version": ([], c_int),
    "tfem_status_string": ([c_int], c_char_p),
    "tfem_set_device": ([c_int], c_int),
    "tfem_sm_count": ([], c_int),
}


def exported_symbols() -> list[str]:
    """Every symbol the header declares (typed ones in both precisions)."""
    names = [f"{base}_{suf}" for base in _TYPED for suf in ("f64", "f32")]
    return names + list(_UNTYPED)


def header_symbols() -> list[str]:
    """Parse include/tfem_b200.h: the source of truth the tests compare against."""
    with open(HEADER) as fh:
        text = fh.read()
    typed = re.findall(r"int (tfem_\w+)_##SUF\(", text)
    plain = re.findall(r"^(?:int|const char\*) (tfem_\w+)\(", text, flags=re.M)
    return [f"{t}_{s}" for t in typed for s in ("f64", "f32")] + plain


_lib = None


def load() -> ctypes.CDLL:
    """Load the shared library or raise; never falls back to another implementation."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH) and "TFEM_B200_LIB" not in os.environ:
        # a fresh checkout: compile the CUDA library once (nvcc, sm_100a).  This is the product path
        # itself, not a fallback; if it cannot be built the error below stands.
        try:
            from . import build

            build.build()
        except Exception as error:  # noqa: BLE001 - reported, then the hard failure below
            print(f"[tfem] building {LIB_PATH} failed: {error!r}", file=sys.stderr)
    if not os.path.exists(LIB_PATH):
        raise TfemError(
            f"{LIB_PATH} is missing: build it with `python -m pytorch_fem_solver_b200.build` "
            "(there is no CPU fallback for the assembly path)"
        )
    lib = ctypes.CDLL(LIB_PATH)
    for base, argtypes in _TYPED.items():
        for suf in ("f64", "f32"):
            fn = getattr(lib, f"{base}_{suf}")
            fn.argtypes = argtypes
            fn.restype = c_int
    for name, (argtypes, restype) in _UNTYPED.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = restype
    _lib = lib
    return lib


def suffix(dtype: torch.dtype) -> str:
    if dtype == torch.float64:
        return "f64"
    if dtype == torch.float32:
        return "f32"
    raise TfemError(f"unsupported dtype {dtype}: the kernels are instantiated for float64 and float32")


def ptr(t: torch.Tensor | None):
    return None if t is None else t.data_ptr()


def check_cuda(*tensors: torch.Tensor | None) -> torch.device:
    device = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise TfemError(
                "tfem_b200 kernels need CUDA tensors (there is no CPU fallback); got a tensor on " + str(t.device)
            )
        if not t.is_contiguous():
            raise TfemError("tfem_b200 kernels need contiguous tensors")
        if device is None:
            device = t.device
        elif t.device != device:
            raise TfemError(f"tensors on different devices: {device} and {t.device}")
    if device is None:
        raise TfemError("no tensor arguments")
    return device


def call(base: str, dtype: torch.dtype | None, device: torch.device, *args):
    """Invoke `base_{f64|f32}` on the current stream of `device`; raise on a negative status."""
    lib = load()
    index = device.index if device.index is not None else torch.cuda.current_device()
    # every call: the library links the static CUDA runtime but shares the thread's current context with torch,
    # so another `torch.cuda.set_device` / `torch.cuda.device(...)` on this thread would invalidate a cached choice
    if lib.tfem_set_device(index) != 0:
        raise TfemError(f"tfem_set_device({index}) failed")
    name = base if dtype is None else f"{base}_{suffix(dtype)}"
    stream = torch.cuda.current_stream(device).cuda_stream
    status = getattr(lib, name)(*args, stream)
    if status != 0:
        raise TfemError(f"{name} failed: {lib.tfem_status_string(status).decode()} ({status})")
    LAUNCHES[name] = LAUNCHES.get(name, 0) + 1


LAUNCHES: dict[str, int] = {}


def make_source(kind: int = TFEM_SRC_NONE, p=(0.0, 0.0, 0.0, 0.0)) -> Source:
    s = Source()
    s.kind = kind
    for i, v in enumerate(p):
        s.p[i] = float(v)
    return s
