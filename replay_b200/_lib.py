"""ctypes binding of librp_b200.so (C ABI: include/rp_b200.h).  Fails loudly when the library is missing - there is no
CPU or PyTorch fallback for the kernels."""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_float, c_int, c_int32, c_int64, c_size_t, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
# RP_B200_LIB: load another build of the SAME C ABI (A/B timing of kernel variants inside one GPU call, tools/ab_env.sh)
LIB_PATH = os.environ.get("RP_B200_LIB") or os.path.join(_HERE, "librp_b200.so")

_lib = None


class RpError(RuntimeError):
    pass


_ERR = {-1: "RP_EINVAL (null pointer / unsupported flag)", -2: "RP_ESHAPE (unsupported size)",
        -3: "RP_EALIGN (pointer or pitch not 16-byte aligned)", -4: "RP_EDRIVER (driver entry point / tensor map)",
        -5: "RP_EWORKSPACE (workspace too small)"}


def check(rc: int, what: str) -> None:
    if rc == 0:
        return
    if rc < 0:
        raise RpError(f"{what}: {_ERR.get(rc, rc)}")
    raise RpError(f"{what}: cudaError {rc}")


def _sig(fn, restype, argtypes):
    fn.restype = restype
    fn.argtypes = argtypes


def lib():
    """Load (once) and return the ctypes handle.  Raises if the extension has not been built (python -m replay_b200.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RpError(
            f"{LIB_PATH} is missing: build it with `python -m replay_b200.build` (nvcc, sm_100a). "
            "replay_b200 has no CPU fallback."
        )
    L = ctypes.CDLL(LIB_PATH)
    P = c_void_p
    _sig(L.rp_version, c_char_p, [])
    _sig(L.rp_selftest_umma, c_int, [c_int, P, P, P, P])
    _sig(L.rp_seen_prepare, c_int, [P, c_int, c_int, c_int, P, P, P])
    _sig(L.rp_score_topk_workspace, c_size_t, [c_int, c_int, c_int, c_int])
    _sig(L.rp_score_topk, c_int, [P, P, P, P, c_int, c_int, c_int, c_int, c_int, P, P, P, P, c_size_t, P])
    _sig(L.rp_ce_head_workspace, c_size_t, [c_int, c_int, c_int])
    _sig(L.rp_ce_head_fwd, c_int, [P, P, P, P, P, c_int, c_int, c_int, P, P, P, P, c_int, P, c_size_t, P])
    _sig(L.rp_ce_head_fwd_w, c_int, [P, P, P, P, P, c_int, c_int, c_int, P, P, P, P, c_int, P, c_int, c_float, c_float, P, c_size_t, P])
    _sig(L.rp_ce_head_bwd, c_int, [P, P, P, P, P, c_int, c_int, c_int, P, P, P, P, P, c_int, c_int, P, c_size_t, P])
    _sig(L.rp_bce_head_workspace, c_size_t, [c_int, c_int, c_int])
    _sig(L.rp_bce_head_fwd, c_int, [P, P, P, P, P, c_int, c_int, c_int, P, P, c_int, P, c_size_t, P])
    _sig(L.rp_bce_head_bwd, c_int, [P, P, P, P, P, c_int, c_int, c_int, P, P, P, P, c_size_t, P])
    U64, LL = ctypes.c_ulonglong, ctypes.c_longlong
    _sig(L.rp_gemm, c_int, [ctypes.POINTER(GemmDesc), P])
    _sig(L.rp_attn_fwd, c_int, [ctypes.POINTER(AttnDesc), P])
    _sig(L.rp_attn_bwd, c_int, [ctypes.POINTER(AttnBwdDesc), P])
    _sig(L.rp_reduce_splits, c_int, [P, c_int, LL, LL, P, c_int, P])
    _sig(L.rp_attn_softmax_bwd, c_int, [P, P, P, c_int, c_int, c_float, c_float, U64, U64, P, P])
    _sig(L.rp_prepare_batch, c_int, [P, P, P, P, c_int, c_int, c_int, P, P, P, P, P, P])
    _sig(L.rp_embed_fwd, c_int, [P, P, P, P, c_int, c_int, c_int, c_int, c_float, c_int, c_float, U64, U64, P, P, P])
    _sig(L.rp_embed_bwd, c_int, [P, P, P, c_int, c_int, c_int, c_int, c_int, c_float, c_int, c_float, U64, U64, P, P, P, P])
    _sig(L.rp_layernorm_fwd, c_int, [P, P, P, c_float, c_int, c_int, P, P, P, P, P, c_int, P])
    _sig(L.rp_layernorm_bwd, c_int, [P, P, P, P, P, c_int, c_int, P, P, P, P, P, P, c_int, P])
    _sig(L.rp_dropout_bwd, c_int, [P, P, LL, c_int, P, c_float, U64, U64, P, P])
    _sig(L.rp_colsum, c_int, [P, c_int, c_int, LL, P, P])
    _sig(L.rp_adam_step, c_int, [P, P, P, P, P, LL, P, P, c_float, c_float, c_float, c_float, P, c_int, P])
    _sig(L.rp_peer_allreduce_state_bytes, c_size_t, [])
    _sig(L.rp_peer_allreduce, c_int, [P, P, c_int, c_int, LL, P])
    _sig(L.rp_cast_bf16, c_int, [P, P, LL, P])
    _sig(L.rp_counter_add, c_int, [P, U64, P])
    _sig(L.rp_bert_embed_fwd, c_int, [P, P, P, P, P, c_int, c_int, c_int, c_float, U64, U64, P, P, P])
    _sig(L.rp_bert_embed_bwd, c_int, [P, P, P, P, c_int, c_int, c_int, c_float, U64, U64, P, P, P, P, P])
    _sig(L.rp_attn_last, c_int, [P, P, P, LL, LL, c_int, c_int, P, c_int, c_int, c_int, c_int, c_int, P, c_float, P])
    _sig(L.rp_gather_rows, c_int, [P, P, c_int, P, c_int, P, c_int, P])
    _sig(L.rp_sampled_head_workspace, c_size_t, [c_int, c_int, c_int, c_int])
    _sig(L.rp_sampled_head_fwd, c_int, [P, P])
    _sig(L.rp_sampled_head_bwd, c_int, [P, P, P, P])
    _sig(L.rp_selftest_mma_probe, c_int, [c_int, c_int, c_int, P, P])
    _sig(L.rp_selftest_tma_probe, c_int, [P, LL, c_int, c_int, c_int, c_int, c_int, P])
    _sig(L.rp_colsum_multi, c_int, [c_int, P, P, P, P, c_int, P])
    _sig(L.rp_post_attn_fused, c_int, [P, P, P, P, P, P, c_float, P, P, P, P, P, c_int, c_int, P, c_int, P])
    _sig(L.rp_ffn_fused, c_int, [P, P, P, P, P, P, c_int, c_int, P, P])
    _sig(L.rp_build_batch, c_int, [P, P, LL, P, P, c_int, c_int, c_int, c_int, c_float, P, U64, U64, P, P, P, P, P, P, P])
    _sig(L.rp_post_attn_train, c_int, [P, P, P, P, P, P, c_float, P, P, P, P, P, c_int, c_int, c_float, U64, U64, U64, P,
                                       P, P, P, P, P, P, c_int, P])
    _sig(L.rp_post_attn_bwd, c_int, [P, P, P, P, P, P, P, P, P, P, c_int, c_int, c_float, U64, U64, P, P, P, P, P, P, P, c_int, P])
    _sig(L.rp_ln_qkv_fused, c_int, [P, P, P, c_float, P, P, c_int, c_int, P, P, P, P, P, c_int, P])
    _sig(L.rp_pre_attn_bwd, c_int, [P, P, P, P, P, P, P, P, c_int, c_int, P, P, P, c_int, P])
    _sig(L.rp_wgrad_group_workspace, c_size_t, [ctypes.POINTER(WgradPair), c_int])
    _sig(L.rp_wgrad_group, c_int, [ctypes.POINTER(WgradPair), c_int, c_int, c_int, P, c_size_t, P])
    for name, restype, argtypes in _EXTRA_SIGS:
        _sig(getattr(L, name), restype, argtypes)
    _lib = L
    return L


class GemmDesc(ctypes.Structure):
    """Mirror of ``struct rp_gemm_desc`` (include/rp_b200.h)."""

    _fields_ = [
        ("A", c_void_p), ("a_rows", ctypes.c_longlong), ("a_cols", ctypes.c_longlong), ("lda", ctypes.c_longlong), ("a_mn", c_int),
        ("B", c_void_p), ("b_rows", ctypes.c_longlong), ("b_cols", ctypes.c_longlong), ("ldb", ctypes.c_longlong), ("b_mn", c_int),
        ("M", c_int), ("N", c_int), ("K", c_int), ("batch", c_int), ("inner", c_int),
        ("a_r0", c_int), ("a_ro", c_int), ("a_ri", c_int), ("a_c0", c_int), ("a_co", c_int), ("a_ci", c_int),
        ("b_r0", c_int), ("b_ro", c_int), ("b_ri", c_int), ("b_c0", c_int), ("b_co", c_int), ("b_ci", c_int),
        ("C", c_void_p), ("ldc", ctypes.c_longlong), ("c_off0", ctypes.c_longlong), ("c_oo", ctypes.c_longlong),
        ("c_oi", ctypes.c_longlong), ("out_mode", c_int),
        ("alpha", c_float), ("bias", c_void_p), ("act", c_int),
        ("residual", c_void_p), ("rowmask", c_void_p), ("rowmask_off0", ctypes.c_longlong), ("rowmask_oo", ctypes.c_longlong),
        ("drop_p", c_float), ("seed", ctypes.c_ulonglong), ("drop_offset", ctypes.c_ulonglong), ("seed_ptr", c_void_p),
        ("split_k", c_int),
        ("gate", c_void_p), ("gate_scale", c_float),
        ("C2", c_void_p), ("gate_mode", c_int), ("post_drop_p", c_float), ("post_drop_offset", ctypes.c_ulonglong),
        ("c_split_stride", ctypes.c_longlong),
        ("row_exp2_offset", c_void_p), ("m_limit_dev", c_void_p), ("m_limit_base", c_int),
        ("k_limit_dev", c_void_p), ("k_limit_base", c_int),
    ]


class WgradPair(ctypes.Structure):
    """Mirror of ``struct rp_wgrad_pair`` (include/rp_b200.h)."""

    _fields_ = [
        ("dY", c_void_p), ("dy_ld", ctypes.c_longlong), ("n_out", c_int),
        ("X", c_void_p), ("x_ld", ctypes.c_longlong), ("n_in", c_int),
        ("dW", c_void_p), ("dw_ld", ctypes.c_longlong),
        ("db", c_void_p),
    ]


class SampledDesc(ctypes.Structure):
    """Mirror of ``struct rp_sampled_desc`` (include/rp_b200.h)."""

    _fields_ = [
        ("hc", c_void_p), ("table", c_void_p), ("labels", c_void_p), ("valid_idx", c_void_p), ("negatives", c_void_p),
        ("n_valid", c_void_p),
        ("capacity", c_int), ("n_items", c_int), ("d", c_int), ("n_neg", c_int), ("neg_mode", c_int), ("seq_len", c_int),
        ("kind", c_int), ("ignore_index", c_int), ("vocab_size", c_int),
        ("log_eps", c_float), ("clamp", c_float),
        ("loss_out", c_void_p),
        ("workspace", c_void_p), ("workspace_bytes", c_size_t),
    ]


class AttnDesc(ctypes.Structure):
    """Mirror of ``struct rp_attn_desc`` (include/rp_b200.h)."""

    _fields_ = [
        ("q", c_void_p), ("q_rows", ctypes.c_longlong), ("q_cols", ctypes.c_longlong), ("ldq", ctypes.c_longlong), ("q_c0", c_int),
        ("k", c_void_p), ("k_rows", ctypes.c_longlong), ("k_cols", ctypes.c_longlong), ("ldk", ctypes.c_longlong), ("k_c0", c_int),
        ("v", c_void_p), ("v_rows", ctypes.c_longlong), ("v_cols", ctypes.c_longlong), ("ldv", ctypes.c_longlong), ("v_c0", c_int),
        ("B", c_int), ("H", c_int), ("L", c_int), ("head_dim", c_int),
        ("causal", c_int), ("mask_pad_keys", c_int),
        ("pad_mask", c_void_p),
        ("out", c_void_p), ("ldo", c_int),
        ("p_save", c_void_p), ("inv_sum", c_void_p),
        ("drop_p", c_float), ("seed", ctypes.c_ulonglong), ("drop_off", ctypes.c_ulonglong), ("seed_ptr", c_void_p),
        ("m_save", c_void_p),
        ("scale", c_float),
    ]


class AttnBwdDesc(ctypes.Structure):
    """Mirror of ``struct rp_attn_bwd_desc`` (include/rp_b200.h)."""

    _fields_ = [
        ("q", c_void_p), ("q_rows", ctypes.c_longlong), ("q_cols", ctypes.c_longlong), ("ldq", ctypes.c_longlong), ("q_c0", c_int),
        ("k", c_void_p), ("k_rows", ctypes.c_longlong), ("k_cols", ctypes.c_longlong), ("ldk", ctypes.c_longlong), ("k_c0", c_int),
        ("v", c_void_p), ("v_rows", ctypes.c_longlong), ("v_cols", ctypes.c_longlong), ("ldv", ctypes.c_longlong), ("v_c0", c_int),
        ("d_out", c_void_p), ("do_rows", ctypes.c_longlong), ("do_cols", ctypes.c_longlong), ("ld_do", ctypes.c_longlong),
        ("out", c_void_p), ("ldo", c_int),
        ("B", c_int), ("H", c_int), ("L", c_int), ("head_dim", c_int),
        ("causal", c_int), ("mask_pad_keys", c_int),
        ("pad_mask", c_void_p),
        ("m_save", c_void_p), ("inv_sum", c_void_p),
        ("dq", c_void_p), ("ld_dq", c_int), ("dq_c0", c_int),
        ("dk", c_void_p), ("ld_dk", c_int), ("dk_c0", c_int),
        ("dv", c_void_p), ("ld_dv", c_int), ("dv_c0", c_int),
        ("drop_p", c_float), ("seed", ctypes.c_ulonglong), ("drop_off", ctypes.c_ulonglong), ("seed_ptr", c_void_p),
        ("scale", c_float),
    ]


_EXTRA_SIGS: list = []

__all__ = ["GemmDesc", "AttnDesc", "AttnBwdDesc", "WgradPair", "lib", "check", "RpError", "LIB_PATH", "c_float", "c_int", "c_int32", "c_int64", "c_size_t", "c_void_p"]
