"""ctypes binding of libmugd.so (the C ABI in include/mugd.h).

There is no CPU fallback: importing this module without the built library, or creating an engine on a
machine without an sm_100 GPU, raises.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MUGD_LIB") or os.path.join(HERE, "libmugd.so")      # MUGD_LIB: experiment builds (tools/build_variant.py)

# ---- enums (include/mugd.h) ------------------------------------------------------------------------
(OP_GEMM, OP_GROUPNORM, OP_LAYERNORM, OP_ATTENTION, OP_S4CONV, OP_DDIM_UPDATE, OP_TRANSPOSE, OP_COPY2D, OP_STEP_ADVANCE, OP_NOTES, OP_EMBED,
 OP_TF32_SPLIT) = range(1, 13)
CONV_NONE, CONV_SAME, CONV_DOWN, CONV_UP, CONV_TAPS = range(5)
ACT_NONE, ACT_SILU, ACT_GELU = range(3)
GATE_NONE, GATE_GEGLU, GATE_GLU = range(3)
GEMM_AUTO, GEMM_SIMT, GEMM_TC = range(3)
TC_AUTO, TC_N64, TC_N128, TC_N256, TC_N128_2CTA = range(5)
ABI_VERSION = 13

_f = C.c_void_p  # device pointers travel as integers


class Gemm(C.Structure):
    _fields_ = [("A", _f), ("lda", C.c_int64), ("W", _f), ("W_hi", _f), ("W_lo", _f), ("bias", _f), ("rowvec", _f),
                ("rowvec_b_stride", C.c_int64), ("rowvec_step_stride", C.c_int64), ("step", _f),
                ("residual", _f), ("ldr", C.c_int64), ("C", _f), ("ldc", C.c_int64),
                ("M", C.c_int32), ("N", C.c_int32), ("K", C.c_int32),
                ("taps", C.c_int32), ("conv_mode", C.c_int32), ("Lin", C.c_int32), ("Lout", C.c_int32),
                ("act", C.c_int32), ("gate", C.c_int32), ("impl", C.c_int32),
                ("split_k", C.c_int32), ("tap_shift", C.c_int32), ("tap_dilation", C.c_int32),
                ("workspace", _f), ("workspace_bytes", C.c_int64),
                ("A2", _f), ("lda2", C.c_int64), ("K2", C.c_int32), ("tc_variant", C.c_int32),
                ("row_moments", _f),
                ("ln_stats", _f), ("ln_colsum", _f), ("ln_eps", C.c_float), ("reserved2_", C.c_int32)]


class GroupNorm(C.Structure):
    _fields_ = [("x", _f), ("ldx", C.c_int64), ("y", _f), ("ldy", C.c_int64), ("gamma", _f), ("beta", _f),
                ("B", C.c_int32), ("L", C.c_int32), ("C", C.c_int32), ("G", C.c_int32),
                ("eps", C.c_float), ("silu", C.c_int32)]


class LayerNorm(C.Structure):
    _fields_ = [("x", _f), ("ldx", C.c_int64), ("y", _f), ("ldy", C.c_int64), ("gamma", _f), ("beta", _f),
                ("rows", C.c_int32), ("C", C.c_int32), ("eps", C.c_float)]


class Attention(C.Structure):
    _fields_ = [("q", _f), ("ldq", C.c_int64), ("k", _f), ("ldk", C.c_int64), ("v", _f), ("ldv", C.c_int64),
                ("o", _f), ("ldo", C.c_int64), ("relpos", _f), ("cgain", _f),
                ("B", C.c_int32), ("H", C.c_int32), ("D", C.c_int32), ("Lq", C.c_int32), ("Lk", C.c_int32),
                ("pos_max", C.c_int32), ("scale", C.c_float)]


class S4Conv(C.Structure):
    _fields_ = [("u", _f), ("ldu", C.c_int64), ("Kt", _f), ("D", _f), ("y", _f), ("ldy", C.c_int64),
                ("B", C.c_int32), ("L", C.c_int32), ("H", C.c_int32)]


class DdimUpdate(C.Structure):
    _fields_ = [("x", _f), ("x_dup", _f), ("eps", _f), ("noise", _f), ("pred_x0", _f), ("coef", _f), ("step", _f),
                ("S", C.c_int32), ("n", C.c_int32), ("cfg", C.c_int32), ("scale", C.c_float),
                ("temperature", C.c_float)]


class Transpose(C.Structure):
    _fields_ = [("inp", _f), ("out", _f), ("ldi", C.c_int64), ("ldo", C.c_int64),
                ("B", C.c_int32), ("C", C.c_int32), ("L", C.c_int32), ("to_nlc", C.c_int32)]


class Copy2D(C.Structure):
    _fields_ = [("src", _f), ("lds", C.c_int64), ("dst", _f), ("ldd", C.c_int64),
                ("rows", C.c_int32), ("cols", C.c_int32)]


class StepAdvance(C.Structure):
    _fields_ = [("step", _f)]


class Notes(C.Structure):
    _fields_ = [("logits", _f), ("ld", C.c_int64), ("count", _f), ("start_ms", _f), ("end_ms", _f), ("frame_ms", C.c_double),
                ("B", C.c_int32), ("T", C.c_int32), ("K", C.c_int32)]


class Embed(C.Structure):
    _fields_ = [("table", _f), ("ids", _f), ("out", _f), ("B", C.c_int32), ("F", C.c_int32), ("H", C.c_int32), ("n_embed", C.c_int32)]


class Tf32Split(C.Structure):
    _fields_ = [("w_hi", _f), ("lo", _f), ("n", C.c_int64)]


class _OpU(C.Union):
    _fields_ = [("gemm", Gemm), ("gn", GroupNorm), ("ln", LayerNorm), ("attn", Attention), ("s4", S4Conv),
                ("ddim", DdimUpdate), ("tr", Transpose), ("cp", Copy2D), ("adv", StepAdvance), ("notes", Notes), ("embed", Embed),
                ("split", Tf32Split)]


class Op(C.Structure):
    _fields_ = [("kind", C.c_int32), ("tag", C.c_int32), ("u", _OpU)]


_KIND_FIELD = {OP_GEMM: "gemm", OP_GROUPNORM: "gn", OP_LAYERNORM: "ln", OP_ATTENTION: "attn", OP_S4CONV: "s4",
               OP_DDIM_UPDATE: "ddim", OP_TRANSPOSE: "tr", OP_COPY2D: "cp", OP_STEP_ADVANCE: "adv", OP_NOTES: "notes", OP_EMBED: "embed", OP_TF32_SPLIT: "split"}


def make_op(kind: int, desc, tag: int = 0) -> Op:
    op = Op()
    op.kind = kind
    op.tag = tag
    setattr(op.u, _KIND_FIELD[kind], desc)
    return op


class Region(C.Structure):
    _fields_ = [("name", C.c_char_p), ("base", _f), ("bytes", C.c_int64)]


class MugdError(RuntimeError):
    pass


_lib: Optional[C.CDLL] = None


def load() -> C.CDLL:
    """dlopen libmugd.so; raises if it has not been built (python -m mug_diffusion_b200.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MugdError(f"{LIB_PATH} not found: build it with `python -m mug_diffusion_b200.build` "
                        "(there is no CPU/PyTorch fallback for the sampler path)")
    lib = C.CDLL(LIB_PATH)
    lib.mugd_last_error.restype = C.c_char_p
    lib.mugd_abi_version.restype = C.c_int
    lib.mugd_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
    lib.mugd_destroy.argtypes = [C.c_void_p]
    lib.mugd_destroy.restype = None
    lib.mugd_device_info.argtypes = [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
    lib.mugd_set_gemm_impl.argtypes = [C.c_void_p, C.c_int]
    lib.mugd_op_run.argtypes = [C.c_void_p, C.POINTER(Op), C.c_void_p]
    lib.mugd_plan_create.argtypes = [C.c_void_p, C.POINTER(Op), C.c_int32, C.POINTER(C.c_void_p)]
    lib.mugd_plan_run.argtypes = [C.c_void_p, C.c_void_p]
    lib.mugd_plan_capture.argtypes = [C.c_void_p, C.c_void_p]
    lib.mugd_plan_replay.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]
    lib.mugd_plan_launch_count.argtypes = [C.c_void_p]
    lib.mugd_plan_destroy.argtypes = [C.c_void_p]
    lib.mugd_plan_destroy.restype = None
    lib.mugd_s4_kernel_gen.argtypes = [C.c_void_p] + [C.c_void_p] * 7 + [C.c_int32] * 4 + [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
    lib.mugd_gemm_tc_variant.argtypes = [C.POINTER(Gemm), C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
    lib.mugd_gemm_tc_query.argtypes = [C.c_void_p, C.POINTER(Gemm), C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                       C.POINTER(C.c_int64), C.POINTER(C.c_int32)]
    lib.mugd_debug_set_tc_timing.argtypes = [C.c_void_p]
    lib.mugd_fill_i32.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]
    lib.mugd_abi_sizes.argtypes = [C.POINTER(C.c_int32), C.c_int32]
    if lib.mugd_abi_version() != ABI_VERSION:
        raise MugdError(f"libmugd ABI {lib.mugd_abi_version()} != binding {ABI_VERSION}: rebuild the library")
    sizes = (C.c_int32 * 12)()
    lib.mugd_abi_sizes(sizes, 12)
    mine = [C.sizeof(t) for t in (Op, Gemm, GroupNorm, LayerNorm, Attention, S4Conv, DdimUpdate, Transpose, Copy2D, Notes, Embed, Tf32Split)]
    if list(sizes) != mine:
        raise MugdError(f"struct layout mismatch: C {list(sizes)} vs ctypes {mine}")
    lib.mugd_sample.argtypes = [C.c_void_p, C.POINTER(Op), C.c_int32, C.c_int32, C.c_void_p]
    lib.mugd_plan_save.argtypes = [C.c_void_p, C.POINTER(Region), C.c_int32, C.c_char_p]
    lib.mugd_plan_load.argtypes = [C.c_void_p, C.c_char_p, C.POINTER(Region), C.c_int32, C.POINTER(C.c_void_p)]
    lib.mugd_set_tc_single_pass_tf32.argtypes = [C.c_void_p, C.c_int]
    lib.mugd_set_attention_impl.argtypes = [C.c_void_p, C.c_int]
    _lib = lib
    return lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().mugd_last_error().decode(errors="replace")
        if rc == 4:
            import torch
            raise torch.cuda.OutOfMemoryError(f"{what}: {msg}")
        raise MugdError(f"{what} failed (status {rc}): {msg}")


EXPORTED_SYMBOLS = [
    "mugd_abi_version", "mugd_last_error", "mugd_create", "mugd_destroy", "mugd_device_info", "mugd_set_gemm_impl",
    "mugd_op_run", "mugd_plan_create", "mugd_plan_run", "mugd_plan_capture", "mugd_plan_replay",
    "mugd_plan_launch_count", "mugd_plan_destroy", "mugd_s4_kernel_gen", "mugd_fill_i32", "mugd_abi_sizes", "mugd_gemm_tc_query",
    "mugd_set_tc_single_pass_tf32", "mugd_set_attention_impl", "mugd_gemm_tc_variant", "mugd_debug_set_tc_timing", "mugd_sample", "mugd_plan_save", "mugd_plan_load", "mugd_plan_regions", "mugd_plan_ops",
]
