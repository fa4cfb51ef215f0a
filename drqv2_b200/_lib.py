"""ctypes binding of libdrqv2_b200.so (include/drqv2_b200.h).

There is no fallback: if the shared library has not been built, importing any compute
entry point raises.  Build it with ``make -C drqv2_b200/csrc`` (or
``python -c "import __graft_entry__ as g; g.build()"``).
"""
from __future__ import annotations

import ctypes as C
import os
import pathlib

_HERE = pathlib.Path(__file__).resolve().parent
LIB_PATH = _HERE / "csrc" / "libdrqv2_b200.so"

P = C.c_void_p
I = C.c_int
L = C.c_int64
U = C.c_uint64
F = C.c_float

# name -> argument ctypes, in header order.  All return int status unless noted.
SIGNATURES = {
    "drq_ring_gather_nstep": [P, P, P, P, L, I, I, I, P, P, I, I, F, P, P, P, P, P, P],
    "drq_ring_sample": [P, P, I, U, P, P, P, I, P],
    "drq_rng_update_draws": [U, P, I, P, P, P, P, I, I, P],
    "drq_ring_sample_step": [P, P, I, U, P, P, P, I, P],
    "drq_update_prologue": [P, I, P, P, U, P, I, P, P, P, P, I, I, P],
    "drq_update_prologue_ring": [P, I, P, P, U, P, I, P, P, P, P, I, I, P, P, P, P, P],
    "drq_update_prologue_ring_part": [P, I, P, P, U, P, I, P, P, P, P, I, I, P, P, P, P, I, P],
    "drq_conv1_fwd_bf16_ring": [P, I, P, P, P, I, I, P],
    "drq_conv1_wgrad_bf16_ring": [P, I, P, P, P, P, P, I, I, P],
    "drq_rng_normal_f32": [U, P, P, I, P],
    "drq_counter_advance": [P, P],
    "drq_scalars_fetch": [P, I, P, P, P],
    "drq_random_shift_f32": [P, P, P, I, I, I, I, I, P],
    "drq_conv1_fwd_f32": [P, P, P, P, P, I, I, I, P],
    "drq_conv1_wgrad_f32": [P, P, P, P, P, P, I, I, I, P],
    "drq_conv1_fwd_f32_from_f32": [P, P, P, P, I, I, P],
    "drq_conv1_wgrad_f32_from_f32": [P, P, P, P, P, I, I, P],
    "drq_conv1_dgrad_f32": [P, P, P, I, I, P],
    "drq_random_shift_bwd_f32": [P, P, P, I, I, I, I, I, P],
    "drq_conv3x3_fwd_f32": [P, P, P, P, I, I, I, P],
    "drq_conv3x3_dgrad_f32": [P, P, P, P, I, I, P],
    "drq_conv3x3_wgrad_f32": [P, P, P, P, P, I, I, P],
    "drq_feature_grad_wide_f32": [P, P, P, I, P],
    "drq_pack_conv_w_bf16": [P, P, P, P],
    "drq_conv3x3_fwd_bf16": [P, P, P, P, I, I, I, L, I, I, P],
    "drq_conv3x3_dgrad_bf16": [P, P, P, I, P, I, I, P],
    "drq_conv3x3_wgrad_bf16": [P, I, P, P, P, P, I, I, P],
    "drq_pack_conv1_w_bf16": [P, P, P, I, P],
    "drq_conv1_fwd_bf16": [P, P, P, P, I, I, I, P],
    "drq_conv1_wgrad_bf16": [P, P, P, P, P, P, I, I, I, P],
    "drq_conv1_fwd_bf16_from_f32": [P, P, P, I, I, P],
    "drq_conv1_wgrad_bf16_from_f32": [P, P, P, P, P, I, I, P],
    "drq_conv1_dgrad_bf16": [P, P, P, I, I, P],
    "drq_gemm_bf16": [P, I, P, I, I, P, L, I, P, P, I, I, I, I, I, I, I, I, P, I, I, P],
    "drq_set_sm_limit": [I],
    "drq_set_gemm_small": [I],
    "drq_set_conv4x1": [I],
    "drq_set_conv1_planes": [I],
    "drq_debug_gemm_stamps": [P],
    "drq_debug_conv_stamps": [P],
    "drq_debug_trap_note": [P],
    "drq_debug_conv4x1_stamps": [P],
    "drq_debug_conv1_stamps": [P],
    "drq_pack_multi": [P, I, P],
    "drq_conv_wgrad_reduce_multi": [P, I, P],
    "drq_colsum_multi": [P, I, P],
    "drq_pack_linear_tb": [P, P, I, I, P],
    "drq_pack_trunk_tb": [P, P, I, P],
    "drq_pack_features_tb": [P, P, I, P],
    "drq_gemm_f32": [P, L, L, P, L, L, P, L, P, P, L, I, I, I, I, I, I, L, L, L, L, L, I, P],
    "drq_colsum_f32": [P, L, P, I, I, I, L, L, P],
    "drq_ln_tanh_fwd": [P, I, L, P, P, P, P, L, P, P, P, L, I, I, F, P],
    "drq_ln_tanh_fwd_multi": [P, I, I, I, F, P],
    "drq_ln_tanh_bwd": [P, L, P, L, P, P, P, P, P, P, P, L, I, I, I, L, P],
    "drq_actor_sample": [P, P, P, F, P, L, P, P, I, I, P],
    "drq_policy_head_fwd_bf16": [P, L, P, P, P, I, I, I, P, I, P, F, P, P],
    "drq_actor_sample_bwd": [P, L, P, P, P, L, I, I, I, L, P],
    "drq_q_head_fwd_bf16": [P, L, L, P, P, P, I, I, I, L, I, L, P],
    "drq_q_head_bwd_loss_bf16": [I, P, P, P, P, P, P, P, L, L, P, P, P, P, I, I, L, P],
    "drq_q_head_bwd_bf16": [P, P, P, L, L, P, P, P, P, I, I, L, P],
    "drq_features_to_ref": [P, I, P, I, P],
    "drq_feature_grad_wide_bf16": [P, P, P, I, P],
    "drq_plane_sum_f32": [P, L, L, I, P, L, I, I, P],
    "drq_critic_loss": [P, P, P, P, P, P, P, P, P, P, I, P],
    "drq_actor_loss": [P, P, P, P, P, I, P],
    "drq_copy2d_f32": [P, L, P, L, I, I, P],
    "drq_adam_step": [P, P, P, P, L, P, P],
    "drq_soft_update": [P, P, L, F, F, P],
    "drq_adam_ema_step": [P, P, P, P, L, P, P, P, L, F, F, P],
    "drq_adam_pack_step": [P, P, P, P, P, P, P, F, F, P, I, P],
}
# entry points with a non-status return
SPECIAL = {
    "drq_abi_version": (I, []),
    "drq_last_error": (C.c_char_p, []),
    "drq_device_sm_count": (I, []),
    "drq_conv_wgrad_ws_floats": (L, [I]),
    "drq_wb_elems": (L, [I]),
    "drq_conv_wgrad_bf16_ws_floats": (L, []),
    "drq_conv1_wgrad_bf16_ws_floats": (L, []),
    "drq_conv1_w_packed_elems": (L, []),
}

EPI_NONE, EPI_RELU, EPI_MASK, EPI_MASK_WIDE = 0, 1, 2, 3
TEPI_F32, TEPI_RELU_BF16, TEPI_MASK_BF16, TEPI_TRUNK_WGRAD, TEPI_TRUNK_DGRAD = 0, 1, 2, 3, 4
IMG, PW, PLANE, CONV_CH, REPR_DIM = 84, 41, 1696, 32, 39200
PLB, GUARD, WB_SLACK = 1776, 88, 128
TB_ACT, TB_W = 128, 64
POLICY_MAX_A, POLICY_MAX_PARTIALS, POLICY_GROUP = 128, 16384, 32   # DRQ_POLICY_MAX_A, DRQ_POLICY_MAX_PARTIALS; heads.cu kPolicyGroup
POLICY_STATIC_SMEM = 1040        # policy_head_fwd_kernel's static shared memory (block-sum buffer + last-block flag)
LN_MAX_F = 256                   # the LayerNorm kernels' feature bound (heads.cu: 32 lanes x kMaxFPerLane)
GEMM_KK, GEMM_KMN, GEMM_MNMN = 0, 1, 2


class DrqError(RuntimeError):
    pass


_lib = None


def lib():
    """The loaded shared library; raises (never falls back) when it is missing."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise ImportError(
                f"{LIB_PATH} is missing: build the CUDA extension first (make -C {LIB_PATH.parent}). "
                "drqv2_b200 has no CPU or PyTorch fallback.")
        h = C.CDLL(str(LIB_PATH))
        for name, args in SIGNATURES.items():
            fn = getattr(h, name)
            fn.argtypes, fn.restype = args, I
        for name, (res, args) in SPECIAL.items():
            fn = getattr(h, name)
            fn.argtypes, fn.restype = args, res
        if h.drq_abi_version() != 2:
            raise ImportError("libdrqv2_b200.so ABI version mismatch")
        if os.environ.get("DRQV2_B200_CONV4X1"):        # A/B: 0 = one-pixel-per-row conv kernels, 1 = default, 2 = four-pixel-column kernels always
            h.drq_set_conv4x1(int(os.environ["DRQV2_B200_CONV4X1"]))
        if os.environ.get("DRQV2_B200_CONV1_PLANES"):   # A/B: 0 = im2col conv1 forward, 1 = parity-plane forward (default)
            h.drq_set_conv1_planes(int(os.environ["DRQV2_B200_CONV1_PLANES"]))
        _lib = h
    return _lib


def exported_symbols():
    return list(SIGNATURES) + list(SPECIAL)


def call(name, *args):
    """Invoke a status-returning entry point; raise DrqError with the library's message."""
    rc = getattr(lib(), name)(*args)
    if rc != 0:
        raise DrqError(f"{name} failed ({rc}): {lib().drq_last_error().decode()}")


def ptr(t):
    """Device (or host) pointer of a torch tensor / None."""
    return None if t is None else t.data_ptr()
