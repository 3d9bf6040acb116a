"""ctypes loader for libsrfrd_b200.so (C ABI declared in include/srfrd_b200.h).

There is no CPU fallback: importing this module without the built library, or calling a kernel
without an sm_100 device, raises.  Build with ``python -c "import __graft_entry__ as g; g.build()"``
or ``make -C srfrd_b200/csrc``.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# SRFRD_B200_LIB: load another build of the same ABI (A/B timing of a kernel change; never a different product path)
LIB_PATH = os.environ.get("SRFRD_B200_LIB") or os.path.join(_HERE, "lib", "libsrfrd_b200.so")

vp, i32, i64, f32, u32, u64 = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_uint32, C.c_uint64


class GemmEpilogue(C.Structure):
    _fields_ = [("bias", vp), ("residual", vp), ("gate", vp), ("row_ids", vp), ("out_bf16", vp), ("out_f32", vp),
                ("ldr", i32), ("ldg", i32), ("ldc", i32), ("relu", i32), ("drop_p", f32), ("drop_stream", u32),
                ("drop_seed", u64), ("drop_step", vp),
                ("ln_out_bf16", vp), ("ln_w", vp), ("ln_b", vp), ("ln_stats", vp), ("ld_ln", i32), ("ln_eps", f32)]


class CastDesc(C.Structure):
    _fields_ = [("src", vp), ("src_ld", i32), ("dst", vp), ("dst_ld", i32), ("dst_t", vp), ("dst_t_ld", i32),
                ("rows", i32), ("cols", i32), ("dst_is_f32", i32)]


class Mlp2Epilogue(C.Structure):
    """srfrd_mlp2_t (include/srfrd_b200.h)."""
    _fields_ = [("bias1", vp), ("bias2", vp), ("gate", vp), ("ldg", i32), ("relu1", i32), ("drop1_p", f32), ("drop2_p", f32),
                ("drop1_stream", u32), ("drop2_stream", u32), ("drop_seed", u64), ("drop_step", vp), ("residual", vp), ("ldr", i32),
                ("residual_is_a", i32), ("row_ids", vp), ("mid_out", vp), ("ldm", i32), ("out", vp), ("ldc", i32),
                ("ln_out", vp), ("ld_ln", i32), ("ln_w", vp), ("ln_b", vp), ("ln_stats", vp), ("ln_eps", f32)]


class PackDesc(C.Structure):
    """srfrd_pack_t: device buffers of the packed token layout (include/srfrd_b200.h)."""
    _fields_ = [("rows", vp), ("cnt", vp), ("seq_first", vp), ("tok_row", vp), ("row_tok", vp), ("row_ids", vp),
                ("row_info", vp), ("tile_row0", vp), ("last_row", vp), ("cap", i64)]


class RepackPart(C.Structure):
    _fields_ = [("src", vp), ("ld_s", i32), ("dst", vp), ("ld_d", i32), ("W", i32), ("mode", i32)]


# name -> argtypes, exactly the prototypes of include/srfrd_b200.h
SIGNATURES = {
    "srfrd_abi_version": [],
    "srfrd_device_check": [],
    "srfrd_embed_ln_fwd": [vp, i64, i32, vp, vp, i64, i32, i32, vp, vp, i64, i32, f32, vp, vp, f32, vp, vp, vp, vp, i32,
                           f32, u64, u32, vp, vp],
    "srfrd_srfu_labels": [vp, i64, i32, i32, vp, vp],
    "srfrd_embed_bwd": [vp, i32, vp, vp, i64, i32, i32, i32, i32, f32, vp, vp, vp],
    "srfrd_layernorm_fwd": [vp, i32, vp, vp, f32, vp, vp, i32, vp, i64, i32, i64, i64, vp],
    "srfrd_layernorm_bwd": [vp, vp, i32, vp, i32, vp, vp, vp, i32, vp, vp, i32, vp, vp, i64, i32, vp],
    "srfrd_gemm_tn": [vp, i32, vp, i32, i32, i32, i32, C.POINTER(GemmEpilogue), vp],
    "srfrd_mlp2_tn": [vp, i32, vp, i32, vp, i32, i32, i32, C.POINTER(Mlp2Epilogue), vp],
    "srfrd_gemm_tn_plan": [i32, i32, i32, i32, i32, i32, vp],
    "srfrd_gemm_debug_read": [vp],
    "srfrd_attn_debug_read": [vp],
    "srfrd_gemm_wgrad": [vp, i32, vp, i32, i64, i32, i32, vp, i32, vp, vp],
    "srfrd_gemm_ref": [vp, i32, vp, i32, vp, i32, i32, i32, i32, i32, i32, vp],
    "srfrd_colsum": [vp, i64, i32, i64, vp, vp],
    "srfrd_add_segments": [vp, i64, i32, i32, vp, vp],
    "srfrd_dropout_apply": [vp, i32, vp, i32, i64, i32, f32, u64, u32, vp, vp],
    "srfrd_cast_weights": [vp, i32, vp],
    "srfrd_f32_to_bf16_split": [vp, i64, vp, vp, vp, i64, i32, i32, vp],
    "srfrd_attention_fwd": [vp, i32, vp, vp, i32, vp, i32, vp, i64, i32, i32, i32, f32, u64, u32, vp, vp],
    "srfrd_attention_bwd": [vp, i32, vp, i32, vp, vp, i32, vp, i32, vp, vp, i32, vp, vp, i32, i64, i32, i32, i32, f32, u64,
                            u32, vp, vp],
    "srfrd_score_fwd": [vp, i32, vp, vp, vp, vp, vp, vp, i64, i32, i32, vp, vp, vp],
    "srfrd_score_bwd": [vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, i64, i32, i32, vp, i32, vp, vp, vp],
    "srfrd_score_loss_fused": [vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, i64, i32, i32, vp, vp, vp, vp, i32, vp, vp, vp],
    "srfrd_weight_sums": [vp, vp, vp, i64, vp, vp],
    "srfrd_loss_finalize": [vp, vp, vp, vp],
    "srfrd_adam_tick": [vp, f32, f32, vp],
    "srfrd_adam_step": [vp, vp, vp, vp, i64, f32, f32, f32, f32, vp, i32, vp],
    "srfrd_adam_step_fused": [vp, vp, vp, vp, i64, f32, f32, f32, f32, vp, i32, vp, vp, vp, vp, vp, i32, vp, vp],
    "srfrd_param_l2_plan": [C.POINTER(i64), i32, C.POINTER(i64)],
    "srfrd_param_l2": [vp, vp, i32, i64, f32, vp, vp, vp, vp],
    "srfrd_catalogue_topk_plan": [i64, i64, i64, i32, i32, C.POINTER(i32), i32],
    "srfrd_catalogue_topk_kmax": [i32, i32, C.POINTER(i32)],
    "srfrd_catalogue_topk": [vp, i64, i64, i32, vp, i64, i64, i64, i32, i32, i32, i32, vp, vp, vp, vp, i32],
    "srfrd_merge_topk_packed": [vp, i64, i32, i32, vp, vp, vp],
    "srfrd_catalogue_rank": [vp, i64, i64, i32, vp, i64, i64, i64, i32, i32, i32, vp, i32, vp, vp, vp, vp],
    "srfrd_catalogue_ce_plan": [i32, C.POINTER(i64), C.POINTER(i32), C.POINTER(i32)],
    "srfrd_catalogue_ce_fwd": [vp, i32, vp, i32, i64, i32, vp, vp, vp, vp, i64, vp, vp, vp],
    "srfrd_catalogue_ce_bwd": [vp, i32, vp, i32, i64, i32, i32, vp, vp, vp, vp, vp, i64, vp, vp, i32, vp, i32, vp],
    "srfrd_attention_live_items": [vp, i64, i32, i32, vp, vp, vp, vp],
    "srfrd_set_attention_live": [vp, vp, vp, vp],
    "srfrd_merge_topk": [vp, vp, i64, i32, i32, vp, vp, vp],
    "srfrd_unpack_rows": [C.POINTER(RepackPart), i32, C.POINTER(PackDesc), i64, i32, vp],
    "srfrd_pack_rows": [C.POINTER(RepackPart), i32, C.POINTER(PackDesc), i64, i32, vp],
    "srfrd_dp_adam_step": [vp, vp, vp, i32, i32, i64, vp, vp, f32, f32, f32, f32, vp, vp, vp, vp, vp, i32, vp, vp],
    "srfrd_pack_plan": [vp, vp, i64, i32, C.POINTER(PackDesc), vp],
    "srfrd_set_row_limit": [vp],
    "srfrd_embed_ln_fwd_packed": [vp, i64, i32, vp, vp, i64, i32, i32, vp, vp, i64, i32, f32, vp, vp, f32, vp, vp, vp, i32,
                                  f32, u64, u32, vp, vp, vp, i64, vp],
    "srfrd_layernorm_fwd_rows": [vp, i32, vp, vp, f32, vp, i32, vp, i64, i32, vp],
    "srfrd_attention_packed_supported": [i32, i32, i32],
    "srfrd_attention_packed_oproj_supported": [i32, i32, i32],
    "srfrd_attention_fwd_packed": [vp, i32, vp, vp, i32, vp, i32, C.POINTER(PackDesc), i32, i32, i32, f32, u64, u32, vp, vp,
                                   vp, i32, vp, vp, i32, vp, vp, f32, vp, vp, i32, vp, i32],
    "srfrd_attention_bwd_packed": [vp, i32, vp, i32, vp, vp, i32, vp, i32, vp, vp, i32, C.POINTER(PackDesc), i32, i32, i32,
                                   f32, u64, u32, vp, vp, vp, i32, vp, i32],
    "srfrd_score_loss_fused_packed": [vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, vp, vp, i32, vp, vp, vp, vp,
                                      i64, vp],
    "srfrd_embed_bwd_packed": [vp, i32, vp, vp, vp, vp, i64, i32, i32, i32, i32, f32, vp, vp, vp, vp],
    "srfrd_sample_candidates": [vp, vp, vp, vp, i64, i32, i32, u64, vp, vp],
    "srfrd_candidate_rank": [vp, i32, vp, i64, i32, vp, i64, i32, vp, i32, vp, vp, i32, vp, vp, vp],
    "srfrd_add_user_term": [vp, i32, i64, i32, vp, i32, vp, vp, i32, vp],
    "srfrd_sample_batch": [vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, u64, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp],
}

_lib = None
_device_ok = False
launch_count = 0   # kernels-launching C calls issued by this process (bench.py reports it)


def load() -> C.CDLL:
    """dlopen the library and bind every prototype; raises if it is missing or incomplete."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"srfrd_b200: {LIB_PATH} is not built. Run `make -C srfrd_b200/csrc` (needs nvcc, sm_100a). "
            "There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    lib.srfrd_last_error.restype = C.c_char_p
    lib.srfrd_last_error.argtypes = []
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)            # AttributeError if the symbol is not exported
        fn.argtypes = argtypes
        fn.restype = C.c_int
    if lib.srfrd_abi_version() != 10:
        raise RuntimeError("srfrd_b200: ABI version mismatch between _lib.py and the built library")
    _lib = lib
    return lib


def require_device() -> None:
    global _device_ok
    if _device_ok:
        return
    lib = load()
    if lib.srfrd_device_check() != 0:
        raise RuntimeError("srfrd_b200: " + lib.srfrd_last_error().decode())
    _device_ok = True


_profile = None    # when a list: (name, args, start_event, end_event) per call (bench.py's per-kernel timing)


def set_profile(records) -> None:
    global _profile
    _profile = records


def call(name: str, *args) -> None:
    """Invoke a kernel entry point; a non-zero return code becomes RuntimeError(srfrd_last_error())."""
    global launch_count
    lib = _lib or load()
    if _profile is not None:
        import torch
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        rc = getattr(lib, name)(*args)
        e1.record()
        _profile.append((name, args, e0, e1))
    else:
        rc = getattr(lib, name)(*args)
    if rc != 0:
        raise RuntimeError(f"{name}: {lib.srfrd_last_error().decode()}")
    launch_count += 1
