"""ctypes binding of libadm_b200.so (the C-ABI declared in include/adm_b200.h).

The library is built in-tree by ``adm_b200/csrc/Makefile`` (``__graft_entry__.build()``).  There is no CPU fallback:
if the shared object is missing, importing the ops raises, and every op checks that its tensors live on a CUDA device.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# ADM_B200_LIB: another build of the same library (A/B timing of kernel changes on one box); default = the in-tree build
LIB_PATH = os.environ.get("ADM_B200_LIB") or os.path.join(_HERE, "libadm_b200.so")

_lib = None

c_p = C.c_void_p
c_i = C.c_int
c_ll = C.c_longlong
c_f = C.c_float
c_d = C.c_double
c_ull = C.c_ulonglong


class Operand(C.Structure):
    _fields_ = [("ptr", c_p), ("mn_major", c_i), ("dim0", c_ll), ("dim1", c_ll), ("dim2", c_ll),
                ("stride1", c_ll), ("stride2", c_ll), ("c0", c_i), ("c0_lo", c_i), ("c1", c_i), ("c1_lo", c_i),
                ("bhi", c_i), ("blo", c_i)]


class GemmDesc(C.Structure):
    _fields_ = [("a", Operand), ("b", Operand), ("m", c_i), ("n", c_i), ("k", c_i), ("batches", c_i), ("bdiv", c_i),
                ("splits", c_i), ("c", c_p), ("out_mode", c_i), ("ldc", c_ll), ("c_bhi", c_ll), ("c_blo", c_ll),
                ("c_col_lo", c_i), ("bias", c_p), ("residual", c_p), ("ldr", c_ll), ("alpha", c_f)]


# name -> (restype, argtypes).  Must list every symbol include/adm_b200.h declares (tests/test_abi.py checks this).
SIGNATURES = {
    "adm_last_error": (C.c_char_p, []),
    "adm_device_error": (c_i, []),
    "adm_launch_count": (c_ll, []),
    "adm_version": (c_i, []),
    "adm_qsample": (c_i, [c_p, c_p, c_p, c_p, c_ll, c_ll, c_p]),
    "adm_ddm_loss": (c_i, [c_p, c_p, c_p, c_p, c_p, c_f, c_i, c_i, c_f, c_p, c_p, c_p, c_ll, c_ll, c_p]),
    "adm_sampler_step": (c_i, [c_p, c_p, c_p, c_p, c_d, c_d, c_d, c_i, c_i, c_d, c_i, c_ll, c_p]),
    "adm_sampler_step_stochastic": (c_i, [c_p, c_p, c_p, c_p, c_p, c_d, c_d, c_d, c_i, c_ll, c_p]),
    "adm_unet_input": (c_i, [c_p, c_p, c_i, c_p, c_i, c_i, c_i, c_i, c_i, c_p]),
    "adm_unet_output": (c_i, [c_p, c_p, c_i, c_p, c_p, c_i, c_p, c_p, c_i, c_i, c_i, c_i, c_p]),
    "adm_unet_output_bwd": (c_i, [c_p, c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_i, c_p]),
    "adm_conv_fprop": (c_i, [c_p, c_i, c_ll, c_p, c_i, c_ll, c_i, c_i, c_i, c_p, c_i, c_i, c_p, c_i, c_ll, c_p, c_p,
                             c_ll, c_f, c_p]),
    "adm_conv_dgrad": (c_i, [c_p, c_i, c_ll, c_i, c_i, c_i, c_p, c_i, c_i, c_p, c_i, c_ll, c_p, c_ll, c_f, c_p]),
    "adm_conv_wgrad": (c_i, [c_p, c_i, c_ll, c_p, c_i, c_ll, c_p, c_i, c_ll, c_i, c_i, c_i, c_i, c_p, c_p]),
    "adm_gemm_batched": (c_i, [C.POINTER(GemmDesc), c_p]),
    "adm_augment_warp_smem": (c_ll, [c_i, c_i, c_i]),
    "adm_augment_warp": (c_i, [c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_i, c_i, c_i, c_i, c_p]),
    "adm_pack_conv_weight": (c_i, [c_p, c_p, c_i, c_i, c_i, c_i, c_p, c_p]),
    "adm_unpack_conv_wgrad": (c_i, [c_p, c_p, c_i, c_i, c_i, c_i, c_i, c_p, c_p]),
    "adm_cast_f32_bf16": (c_i, [c_p, c_p, c_ll, c_p]),
    "adm_transpose_weight_tiles": (c_i, [c_p, c_p, c_p, c_i, c_p]),
    "adm_gather_rows": (c_i, [c_p, c_p, c_p, c_ll, c_i, c_p]),
    "adm_conv_wgrad_mapped": (c_i, [c_p, c_i, c_ll, c_p, c_i, c_ll, c_p, c_i, c_ll, c_i, c_i, c_i, c_i, c_p, c_p, c_p]),
    "adm_col_sums_mapped": (c_i, [c_p, c_ll, c_ll, c_i, c_p, c_p, c_p]),
    "adm_gn_stats": (c_i, [c_p, c_i, c_ll, c_p, c_i, c_ll, c_i, c_i, c_i, c_f, c_p, c_p, c_p, c_ll, c_p, c_p, c_p]),
    "adm_gn_apply": (c_i, [c_p, c_i, c_ll, c_p, c_i, c_ll, c_i, c_i, c_i, c_p, c_i, c_f, c_ull, c_p, c_i, c_p, c_ll,
                           c_p]),
    "adm_gn_bwd": (c_i, [c_p, c_ll, c_p, c_i, c_ll, c_p, c_i, c_ll, c_i, c_i, c_i, c_i, c_p, c_p, c_p, c_p, c_ll, c_i,
                         c_f, c_ull, c_p, c_i, c_p, c_p, c_p, c_p, c_p, c_ll, c_p, c_ll, c_i, c_p, c_ll, c_p, c_ll, c_p, c_p,
                         c_i, c_p]),
    "adm_gn_forward": (c_i, [c_p, c_i, c_ll, c_p, c_i, c_ll, c_i, c_i, c_i, c_i, c_f, c_p, c_p, c_p, c_ll, c_p, c_p, c_i,
                             c_f, c_ull, c_p, c_i, c_p, c_ll, c_p]),
    "adm_col_sums": (c_i, [c_p, c_ll, c_ll, c_i, c_p, c_p]),
    "adm_add_bf16": (c_i, [c_p, c_ll, c_p, c_ll, c_p, c_ll, c_p, c_ll, c_ll, c_i, c_p]),
    "adm_resample": (c_i, [c_p, c_ll, c_i, c_i, c_i, c_i, c_i, c_p, c_ll, c_p]),
    "adm_silu": (c_i, [c_p, c_p, c_p, c_ll, c_p]),
    "adm_silu_bwd": (c_i, [c_p, c_p, c_p, c_p, c_ll, c_p]),
    "adm_attn_fwd_fused": (c_i, [c_p, c_i, c_i, c_i, c_f, c_p, c_p, c_p]),
    "adm_attn_bwd_fused": (c_i, [c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_f, c_p, c_p]),
    "adm_attn_long_workspace": (c_ll, [c_i, c_i, c_i, c_i]),
    "adm_attn_fwd_long": (c_i, [c_p, c_i, c_i, c_i, c_f, c_p, c_p, c_p, c_ll, c_p]),
    "adm_attn_bwd_long": (c_i, [c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_f, c_p, c_p, c_ll, c_p]),
    "adm_softmax_fwd": (c_i, [c_p, c_p, c_ll, c_i, c_p]),
    "adm_softmax_bwd": (c_i, [c_p, c_p, c_p, c_f, c_ll, c_i, c_p]),
    "adm_spatial_att_fwd": (c_i, [c_p, c_ll, c_p, c_ll, c_p, c_p, c_i, c_i, c_i, c_p, c_ll, c_p, c_p, c_p]),
    "adm_spatial_att_bwd": (c_i, [c_p, c_ll, c_p, c_ll, c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_p, c_ll, c_p, c_p, c_p]),
    "adm_sq_norm": (c_i, [c_p, c_ll, c_p, c_p]),
    "adm_adamw": (c_i, [c_p, c_p, c_p, c_p, c_ll, c_f, c_f, c_f, c_f, c_f, c_i, c_f, c_f, c_p, c_p, c_p, c_p]),
    "adm_lerp_f32": (c_i, [c_p, c_p, c_ll, c_f, c_p]),
    "adm_ws_pack": (c_i, [c_p, c_p, c_p, c_i, c_i, c_i, c_f, c_p]),
    "adm_ws_pack_bwd": (c_i, [c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_p]),
    "adm_chan_layernorm_ok": (c_i, [c_i]),
    "adm_chan_layernorm_fwd": (c_i, [c_p, c_ll, c_ll, c_i, c_p, c_f, c_p, c_ll, c_p]),
    "adm_chan_layernorm_bwd": (c_i, [c_p, c_ll, c_p, c_ll, c_ll, c_i, c_p, c_f, c_p, c_ll, c_p, c_p]),
    "adm_rel_gn_ok": (c_i, [c_i, c_i, c_i, c_i, c_i]),
    "adm_rel_gn_chunks": (c_i, [c_i, c_i, c_i, c_i]),
    "adm_rel_gn_fwd": (c_i, [c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_i, c_i, c_i, c_p, c_p, c_f, c_p, c_i, c_p, c_p, c_p]),
    "adm_rel_gn_bwd": (c_i, [c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_i, c_p, c_p, c_p, c_p, c_p]),
    "adm_bilinear_fwd": (c_i, [c_p, c_ll, c_i, c_i, c_i, c_i, c_p, c_ll, c_i, c_i, c_i, c_i, c_p]),
    "adm_bilinear_bwd": (c_i, [c_p, c_i, c_i, c_i, c_i, c_i, c_i, c_p, c_p, c_p]),
    "adm_avgpool_fwd": (c_i, [c_p, c_i, c_i, c_i, c_i, c_i, c_i, c_p, c_p]),
    "adm_avgpool_bwd": (c_i, [c_p, c_i, c_i, c_i, c_i, c_i, c_i, c_p, c_p]),
    "adm_linattn_workspace": (c_i, [c_i, c_i, c_i, C.POINTER(c_ll)]),
    "adm_linattn_fwd": (c_i, [c_p, c_ll, c_i, c_i, c_i, c_i, c_f, c_p, c_ll, c_p, c_p, c_p, c_p]),
    "adm_linattn_bwd": (c_i, [c_p, c_ll, c_i, c_i, c_i, c_i, c_f, c_p, c_ll, c_p, c_p, c_p, c_p, c_p, c_p, c_ll, c_p]),
}


def load():
    """Load the shared library (once) and attach argtypes.  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(adm_b200 has no CPU or PyTorch fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class AdmError(RuntimeError):
    pass


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().adm_last_error()
        raise AdmError(f"{what} failed ({rc}): {msg.decode() if msg else ''}")
