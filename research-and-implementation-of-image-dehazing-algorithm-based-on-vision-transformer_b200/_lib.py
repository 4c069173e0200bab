"""ctypes binding of the C ABI declared in include/lewin_b200.h.

There is no CPU or PyTorch fallback: if the shared library is missing or a call returns a
non-zero code, a RuntimeError is raised.  The library is built in-tree by
``__graft_entry__.build()`` (``csrc/liblewin_b200.so``).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "liblewin_b200.so")

c_f32p = C.c_void_p
c_ptr = C.c_void_p


class LewinAttnFwdArgs(C.Structure):
    _fields_ = [
        ("B", C.c_int32), ("H", C.c_int32), ("W", C.c_int32), ("C", C.c_int32), ("nH", C.c_int32),
        ("shift", C.c_int32), ("windowed", C.c_int32), ("use_rpb", C.c_int32),
        ("analytic_shift_mask", C.c_int32), ("nW_mask", C.c_int32), ("save_for_backward", C.c_int32),
        ("reserved", C.c_int32),
        ("x", c_ptr), ("y", c_ptr), ("ln_w", c_ptr), ("ln_b", c_ptr),
        ("w_qkv", c_ptr), ("b_qkv", c_ptr), ("w_out", c_ptr), ("b_out", c_ptr),
        ("rpb_table", c_ptr), ("rpb_dense", c_ptr), ("index_sample", c_ptr), ("mask", c_ptr),
        ("drop_scale", c_ptr),
        ("qkv", c_ptr), ("ctx", c_ptr), ("top", c_ptr),
        ("timing", c_ptr),
        ("w_qkv_bf16", c_ptr), ("w_out_bf16", c_ptr),
        ("band_mode", C.c_int32), ("band_y0", C.c_int32), ("band_Hg", C.c_int32), ("reserved2", C.c_int32),
        ("token_mask", c_ptr), ("Bm", C.c_int32), ("reserved3", C.c_int32),
    ]


class LewinAttnBwdArgs(C.Structure):
    _fields_ = [
        ("fwd", LewinAttnFwdArgs),
        ("dy", c_ptr), ("dx", c_ptr),
        ("d_ln_w", c_ptr), ("d_ln_b", c_ptr), ("d_w_qkv", c_ptr), ("d_b_qkv", c_ptr),
        ("d_w_out", c_ptr), ("d_b_out", c_ptr), ("d_rpb_table", c_ptr), ("d_rpb_dense", c_ptr),
        ("deterministic", C.c_int32), ("reserved", C.c_int32),
    ]


class LewinCoreFwdArgs(C.Structure):
    _fields_ = [
        ("B_", C.c_int32), ("nH", C.c_int32), ("use_rpb", C.c_int32), ("nW_mask", C.c_int32),
        ("head_dim", C.c_int32), ("reserved", C.c_int32),
        ("qkv", c_ptr), ("ctx", c_ptr), ("rpb_table", c_ptr), ("rpb_dense", c_ptr),
        ("index_sample", c_ptr), ("mask", c_ptr), ("top", c_ptr),
    ]


class LewinCoreBwdArgs(C.Structure):
    _fields_ = [
        ("fwd", LewinCoreFwdArgs),
        ("dctx", c_ptr), ("dqkv", c_ptr), ("d_rpb_table", c_ptr), ("d_rpb_dense", c_ptr),
        ("deterministic", C.c_int32), ("reserved", C.c_int32),
    ]


class LewinLeffFwdArgs(C.Structure):
    _fields_ = [
        ("B", C.c_int32), ("H", C.c_int32), ("W", C.c_int32), ("C", C.c_int32), ("hidden", C.c_int32),
        ("fused", C.c_int32), ("save_for_backward", C.c_int32), ("ld_out", C.c_int32),
        ("y", c_ptr), ("out", c_ptr), ("ln_w", c_ptr), ("ln_b", c_ptr),
        ("w1", c_ptr), ("b1", c_ptr), ("w_dw", c_ptr), ("b_dw", c_ptr), ("w2", c_ptr), ("b2", c_ptr),
        ("drop_scale", c_ptr),
        ("h1", c_ptr), ("h2", c_ptr), ("a1", c_ptr), ("a2", c_ptr),
        ("timing", c_ptr),
        ("w1_bf16", c_ptr), ("w2_bf16", c_ptr),
    ]


class LewinLeffBwdArgs(C.Structure):
    _fields_ = [
        ("fwd", LewinLeffFwdArgs),
        ("dout", c_ptr), ("dy", c_ptr),
        ("d_ln_w", c_ptr), ("d_ln_b", c_ptr), ("d_w1", c_ptr), ("d_b1", c_ptr),
        ("d_w_dw", c_ptr), ("d_b_dw", c_ptr), ("d_w2", c_ptr), ("d_b2", c_ptr),
        ("deterministic", C.c_int32), ("reserved", C.c_int32),
    ]


class LewinUpsampleFwdArgs(C.Structure):
    _fields_ = [
        ("B", C.c_int32), ("H", C.c_int32), ("W", C.c_int32), ("Cin", C.c_int32), ("Cout", C.c_int32),
        ("ld_out", C.c_int32), ("reserved0", C.c_int32), ("reserved1", C.c_int32),
        ("x", c_ptr), ("weight", c_ptr), ("bias", c_ptr), ("out", c_ptr),
    ]


class LewinInputProjArgs(C.Structure):
    _fields_ = [
        ("B", C.c_int32), ("H", C.c_int32), ("W", C.c_int32), ("Cin", C.c_int32), ("Cout", C.c_int32),
        ("negative_slope", C.c_float), ("reserved0", C.c_int32), ("reserved1", C.c_int32),
        ("x", c_ptr), ("weight", c_ptr), ("bias", c_ptr), ("out", c_ptr),
    ]


class LewinDownsampleArgs(C.Structure):
    _fields_ = [
        ("B", C.c_int32), ("H", C.c_int32), ("W", C.c_int32), ("Cin", C.c_int32),
        ("ld_x", C.c_int32), ("ld_out", C.c_int32), ("pad_h", C.c_int32), ("reserved", C.c_int32),
        ("x", c_ptr), ("weight", c_ptr), ("bias", c_ptr), ("out", c_ptr),
    ]


class LewinOutputProjArgs(C.Structure):
    _fields_ = [
        ("B", C.c_int32), ("H", C.c_int32), ("W", C.c_int32), ("Cin", C.c_int32), ("Cout", C.c_int32),
        ("ld_x", C.c_int32), ("pad_h", C.c_int32), ("reserved", C.c_int32),
        ("x", c_ptr), ("weight", c_ptr), ("bias", c_ptr), ("residual", c_ptr), ("out", c_ptr),
    ]


class LewinConv3x3Args(C.Structure):
    _fields_ = [
        ("B", C.c_int32), ("H", C.c_int32), ("W", C.c_int32), ("Cin", C.c_int32), ("Cout", C.c_int32),
        ("ld_x", C.c_int32), ("ld_out", C.c_int32), ("relu", C.c_int32),
        ("x", c_ptr), ("weight", c_ptr), ("w_bf16", c_ptr), ("bias", c_ptr), ("out", c_ptr),
    ]


# every symbol include/lewin_b200.h declares (tests check the .so exports all of them)
EXPORTS = (
    "lewin_attn_fwd_f32", "lewin_attn_fwd_bf16", "lewin_attn_bwd_f32", "lewin_attn_bwd_bf16",
    "lewin_leff_fwd_f32", "lewin_leff_fwd_bf16", "lewin_leff_bwd_f32", "lewin_leff_bwd_bf16",
    "lewin_attn_fwd_workspace_bytes", "lewin_attn_bwd_workspace_bytes",
    "lewin_leff_fwd_workspace_bytes", "lewin_leff_bwd_workspace_bytes",
    "lewin_probsparse_core_fwd_f32", "lewin_probsparse_core_fwd_bf16", "lewin_probsparse_core_fwd_workspace_bytes",
    "lewin_probsparse_core_bwd_f32", "lewin_probsparse_core_bwd_bf16", "lewin_probsparse_core_bwd_workspace_bytes",
    "lewin_abi_version", "lewin_build_info", "lewin_error_string", "lewin_launch_count",
    "lewin_attn_fwd_kernel_mask", "lewin_leff_fwd_kernel_mask", "lewin_leff_fwd_supports_ld_out",
    "lewin_upsample_fwd_bf16", "lewin_upsample_fwd_workspace_bytes", "lewin_input_proj_fwd_bf16",
    "lewin_downsample_fwd_bf16", "lewin_downsample_fwd_workspace_bytes",
    "lewin_conv3x3_fwd_bf16", "lewin_conv3x3_fwd_workspace_bytes",
    "lewin_output_proj_fwd_bf16", "lewin_output_proj_fwd_workspace_bytes",
)

ABI_VERSION = 7
DTYPE_TAG = {"f32": 0, "bf16": 1}

_lib = None


def load():
    """Load csrc/liblewin_b200.so (once).  Raises RuntimeError if it is absent — no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise RuntimeError(
            f"lewin_b200: CUDA library {LIB_PATH} not found. Build it with "
            f"`python -c 'import __graft_entry__ as g; g.build()'` (nvcc, sm_100a). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, args_t in (("attn_fwd", LewinAttnFwdArgs), ("attn_bwd", LewinAttnBwdArgs),
                         ("leff_fwd", LewinLeffFwdArgs), ("leff_bwd", LewinLeffBwdArgs),
                         ("probsparse_core_fwd", LewinCoreFwdArgs), ("probsparse_core_bwd", LewinCoreBwdArgs)):
        for dt in ("f32", "bf16"):
            fn = getattr(lib, f"lewin_{name}_{dt}")
            fn.argtypes = [C.POINTER(args_t), C.c_void_p, C.c_size_t, C.c_void_p]
            fn.restype = C.c_int
        ws = getattr(lib, f"lewin_{name}_workspace_bytes")
        ws.argtypes = [C.POINTER(args_t), C.c_int]
        ws.restype = C.c_size_t
    lib.lewin_upsample_fwd_bf16.argtypes = [C.POINTER(LewinUpsampleFwdArgs), C.c_void_p, C.c_size_t, C.c_void_p]
    lib.lewin_upsample_fwd_bf16.restype = C.c_int
    lib.lewin_upsample_fwd_workspace_bytes.argtypes = [C.POINTER(LewinUpsampleFwdArgs), C.c_int]
    lib.lewin_upsample_fwd_workspace_bytes.restype = C.c_size_t
    for nm, at in (("downsample", LewinDownsampleArgs), ("output_proj", LewinOutputProjArgs), ("conv3x3", LewinConv3x3Args)):
        fn = getattr(lib, f"lewin_{nm}_fwd_bf16")
        fn.argtypes = [C.POINTER(at), C.c_void_p, C.c_size_t, C.c_void_p]
        fn.restype = C.c_int
        wsf = getattr(lib, f"lewin_{nm}_fwd_workspace_bytes")
        wsf.argtypes = [C.POINTER(at), C.c_int]
        wsf.restype = C.c_size_t
    lib.lewin_input_proj_fwd_bf16.argtypes = [C.POINTER(LewinInputProjArgs), C.c_void_p]
    lib.lewin_input_proj_fwd_bf16.restype = C.c_int
    lib.lewin_abi_version.restype = C.c_int
    lib.lewin_attn_fwd_kernel_mask.argtypes = [C.POINTER(LewinAttnFwdArgs), C.c_int]
    lib.lewin_attn_fwd_kernel_mask.restype = C.c_int
    lib.lewin_leff_fwd_kernel_mask.argtypes = [C.POINTER(LewinLeffFwdArgs), C.c_int]
    lib.lewin_leff_fwd_kernel_mask.restype = C.c_int
    lib.lewin_leff_fwd_supports_ld_out.argtypes = [C.POINTER(LewinLeffFwdArgs), C.c_int]
    lib.lewin_leff_fwd_supports_ld_out.restype = C.c_int
    lib.lewin_launch_count.restype = C.c_longlong
    lib.lewin_build_info.restype = C.c_char_p
    lib.lewin_error_string.argtypes = [C.c_int]
    lib.lewin_error_string.restype = C.c_char_p
    if lib.lewin_abi_version() != ABI_VERSION:
        raise RuntimeError(f"lewin_b200: ABI version mismatch (library {lib.lewin_abi_version()}, binding {ABI_VERSION})")
    _lib = lib
    return lib


def check(code: int, what: str):
    if code == 0:
        return
    lib = load()
    msg = lib.lewin_error_string(code).decode()
    raise RuntimeError(f"lewin_b200: {what} failed with code {code}: {msg}")
