"""ctypes binding of the C-ABI library (include/diffusion_net_b200.h).

The shared object is built IN-TREE (``diffusion-net_b200/libdiffusion_net_b200.so``)
with nvcc for sm_100a and loaded with ctypes -- plain pointers and sizes, no torch
types cross the boundary.  There is no CPU or library fallback: if the library is
missing or a call fails, a RuntimeError is raised.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.path.join(_HERE, "libdiffusion_net_b200.so")
SOURCES = ["dn_simt.cu", "dn_geom.cu", "dn_tc.cu", "dn_chain.cu", "dn_chain16.cu", "dn_capi.cu"]
HEADER = os.path.join(os.path.dirname(_HERE), "include", "diffusion_net_b200.h")

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]

ENGINE_SIMT, ENGINE_TC3X, ENGINE_TC1X, ENGINE_BF16 = 0, 1, 2, 3


def _stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(_CSRC, f) for f in os.listdir(_CSRC)] + [HEADER]
    return any(os.path.getmtime(d) > t for d in deps)


def nvcc() -> str:
    """The nvcc that builds the library: $NVCC, else the CUDA toolkit's default install location."""
    return os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/*.cu into the in-tree shared library (nvcc cross-compiles without a GPU)."""
    if not force and not _stale():
        return LIB_PATH
    cmd = [nvcc()] + NVCC_FLAGS + ["-o", LIB_PATH] + [os.path.join(_CSRC, s) for s in SOURCES]
    if verbose:
        print(" ".join(cmd))
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + r.stdout + r.stderr)
    return LIB_PATH


class dn_patches(C.Structure):
    _fields_ = [("n_patches", C.c_int32), ("max_src", C.c_int32), ("tgt_ptr", C.c_void_p), ("tgt", C.c_void_p),
                ("src_ptr", C.c_void_p), ("src_rows", C.c_void_p), ("ent_ptr", C.c_void_p), ("lcol", C.c_void_p),
                ("vals", C.c_void_p)]


class dn_csr(C.Structure):
    _fields_ = [("rowptr", C.c_void_p), ("colidx", C.c_void_p), ("vals", C.c_void_p), ("nnz", C.c_int64),
                ("patches", C.POINTER(dn_patches))]


class dn_block_params(C.Structure):
    _fields_ = [("diffusion_time", C.c_void_p), ("A_re", C.c_void_p), ("A_im", C.c_void_p),
                ("with_gradient_features", C.c_int), ("with_gradient_rotations", C.c_int),
                ("n_mlp_layers", C.c_int), ("mlp_weight_host", C.POINTER(C.c_void_p)),
                ("mlp_bias_host", C.POINTER(C.c_void_p)), ("mlp_dims_host", C.POINTER(C.c_int))]


class dn_mesh_batch(C.Structure):
    _fields_ = [("n_meshes", C.c_int32), ("n_tb_ctas", C.c_int32), ("tile_mesh", C.c_void_p), ("tb_rows", C.c_void_p),
                ("mesh_cta_begin", C.c_void_p)]


class dn_head(C.Structure):
    _fields_ = [("weight", C.c_void_p), ("bias", C.c_void_p), ("n_out", C.c_int32), ("out", C.c_void_p), ("ld_out", C.c_int64)]


_P, _I, _L = C.c_void_p, C.c_int, C.c_int64
_PP = C.POINTER(C.c_void_p)
_IP = C.POINTER(C.c_int)

# name -> (restype, argtypes): every symbol include/diffusion_net_b200.h declares
SIGNATURES = {
    "dn_abi_version": (_I, []),
    "dn_error_string": (C.c_char_p, [_I]),
    "dn_device_query": (_I, [_I, _IP, _IP, C.POINTER(_L)]),
    "dn_kernel_launch_count": (_L, []),
    "dn_workspace_bytes": (_L, [_L, _I, _I]),
    "dn_csr_from_coo": (_I, [_P, _P, _P, _P, _L, _L, _P, _P, _P, _P]),
    "dn_patch_build": (_L, [_L, _P, _P, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P]),
    "dn_csr_transpose": (_I, [C.POINTER(dn_csr), _L, _P, _P, _P, _P, _L, _P]),
    "dn_compute_hks": (_I, [_P, _P, _P, _L, _I, _I, _P, _P]),
    "dn_to_basis": (_I, [_P, _P, _P, _L, _I, _I, _P, _P, _L, _I, _P]),
    "dn_from_basis": (_I, [_P, _P, _P, _L, _I, _I, _P, _P, _L, _I, _P]),
    "dn_learned_time_diffusion_fwd": (_I, [_P, _P, _P, _P, _P, _L, _I, _I, _P, _P, _P, _L, _I, _P]),
    "dn_learned_time_diffusion_bwd": (_I, [_P, _P, _P, _P, _P, _P, _L, _I, _I, _P, _P, _P, _L, _I, _P]),
    "dn_learned_time_diffusion_fwd_batched": (_I, [_P, _P, _P, _P, _P, C.POINTER(dn_mesh_batch), _L, _I, _I, _P, _P, _P, _L,
                                                   _I, _P]),
    "dn_learned_time_diffusion_bwd_batched": (_I, [_P, _P, _P, _P, _P, _P, C.POINTER(dn_mesh_batch), _L, _I, _I, _P, _P, _P,
                                                   _L, _I, _P]),
    "dn_grad_spmm": (_I, [C.POINTER(dn_csr), _P, _L, _I, _P, _P]),
    "dn_spatial_gradient_features_fwd": (_I, [_P, _P, _P, _I, _L, _I, _P, _P, _L, _I, _P]),
    "dn_gradient_features_fwd": (_I, [C.POINTER(dn_csr), _P, _P, _P, _I, _L, _I, _P, _P, _P, _L, _I, _P]),
    "dn_gradient_features_bwd": (_I, [C.POINTER(dn_csr), C.POINTER(dn_csr), _P, _P, _P, _P, _P, _P, _I, _L, _I,
                                      _P, _P, _P, _P, _L, _I, _P]),
    "dn_mini_mlp_fwd": (_I, [_PP, _IP, _I, _PP, _PP, _IP, _I, _PP, _P, _L, _PP, _P, _P, _L, _I, _P]),
    "dn_mini_mlp_bwd": (_I, [_P, _PP, _IP, _I, _PP, _IP, _I, _PP, _PP, _L, _PP, _PP, _PP, _P, _L, _I, _P]),
    "dn_block_fwd": (_I, [_P, _P, _P, _P, C.POINTER(dn_csr), C.POINTER(dn_block_params), _L, _I, _I, _P, _P, _L,
                          _I, _P]),
    "dn_block_fwd_profile": (_I, [_P, _P, _P, _P, C.POINTER(dn_csr), C.POINTER(dn_block_params), _L, _I, _I, _P, _P, _L,
                                  _I, _P, C.POINTER(C.c_float)]),
    "dn_build_grad": (_I, [_P, _P, _P, _P, _L, _L, _P, _P, _P, _P, _L, _P]),
    "dn_mesh_batch_plan": (_I, [_I, _P, _I, _P, _P, _P, _P]),
    "dn_block_fwd_ex": (_I, [_P, _P, _P, _P, C.POINTER(dn_csr), C.POINTER(dn_block_params), C.POINTER(dn_mesh_batch),
                             C.POINTER(dn_head), _L, _I, _I, _P, _P, _L, _I, _P]),
    "dn_block_fwd_batched": (_I, [_P, _P, _P, _P, C.POINTER(dn_csr), C.POINTER(dn_block_params), C.POINTER(dn_mesh_batch),
                                  _L, _I, _I, _P, _P, _L, _I, _P]),
}

_lib = None


def load():
    """Load (building first if the .so is absent) and type the C-ABI library."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        build()
    try:
        lib = C.CDLL(LIB_PATH)
    except OSError as e:  # fail loudly: there is no fallback path
        raise RuntimeError("diffusion_net_b200: cannot load {}: {}".format(LIB_PATH, e))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if a declared symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.dn_abi_version() != 5:
        raise RuntimeError("diffusion_net_b200: ABI version mismatch")
    _lib = lib
    return lib


def check(code: int, what: str = ""):
    if code != 0:
        msg = load().dn_error_string(code).decode()
        raise RuntimeError("diffusion_net_b200 {} failed ({}): {}".format(what, code, msg))


def ptr_array(ptrs):
    arr = (C.c_void_p * len(ptrs))()
    for i, p in enumerate(ptrs):
        arr[i] = p if p else None
    return arr


def int_array(vals):
    arr = (C.c_int * len(vals))()
    for i, v in enumerate(vals):
        arr[i] = int(v)
    return arr
