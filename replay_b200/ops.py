"""Tensor-level wrappers over the C ABI (include/rp_b200.h).  torch is used for device memory and streams only; every
function launches hand-written sm_100a kernels from librp_b200.so on the current CUDA stream."""
from __future__ import annotations

import torch

import ctypes

from ._lib import GemmDesc, check, lib


def _ptr(t):
    return None if t is None else t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _need(t, dtype, name):
    if t.dtype != dtype or not t.is_cuda or not t.is_contiguous():
        raise ValueError(f"{name}: expected contiguous CUDA tensor of {dtype}, got {t.dtype} on {t.device}")


def selftest_umma(mode: int, a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    _need(a, torch.bfloat16, "a")
    _need(b, torch.bfloat16, "b")
    d = torch.empty(128, 128, device=a.device, dtype=torch.float32)
    check(lib().rp_selftest_umma(mode, _ptr(a), _ptr(b), _ptr(d), _stream()), "rp_selftest_umma")
    return d


def seen_prepare(seen_ids: torch.Tensor, item_count: int, inv_map: torch.Tensor | None = None) -> torch.Tensor:
    """int64 [B,S] seen ids -> int32 [B,S] sorted ascending, padding = INT32_MAX (include/rp_b200.h rp_seen_prepare)."""
    _need(seen_ids, torch.int64, "seen_ids")
    B, S = seen_ids.shape
    out = torch.empty(B, S, device=seen_ids.device, dtype=torch.int32)
    if inv_map is not None:
        _need(inv_map, torch.int32, "inv_map")
    check(lib().rp_seen_prepare(_ptr(seen_ids), B, S, item_count, _ptr(inv_map), _ptr(out), _stream()), "rp_seen_prepare")
    return out


MAX_FUSED_K = 32  # rp_score_topk keeps per-thread sorted lists of K entries (include/rp_b200.h); larger K: logits + torch.topk


def score_topk(hq: torch.Tensor, table: torch.Tensor, k: int, seen_sorted: torch.Tensor | None = None,
               candidates: torch.Tensor | None = None, bias: torch.Tensor | None = None):
    """Fused scores -> seen mask -> top-k.  hq bf16 [B,d], table bf16 [I,d].  Returns (ids int64 [B,k], scores fp32 [B,k])."""
    _need(hq, torch.bfloat16, "hq")
    _need(table, torch.bfloat16, "table")
    B, d = hq.shape
    n_items = table.shape[0]
    S = 0
    if seen_sorted is not None:
        _need(seen_sorted, torch.int32, "seen_sorted")
        S = seen_sorted.shape[1]
    if candidates is not None:
        _need(candidates, torch.int64, "candidates")
    L = lib()
    ws_bytes = L.rp_score_topk_workspace(B, n_items, d, k)
    ws = torch.empty(ws_bytes, device=hq.device, dtype=torch.uint8)
    ids = torch.empty(B, k, device=hq.device, dtype=torch.int64)
    scores = torch.empty(B, k, device=hq.device, dtype=torch.float32)
    check(L.rp_score_topk(_ptr(hq), _ptr(table), _ptr(bias), _ptr(seen_sorted), S, B, n_items, d, k, _ptr(candidates),
                          _ptr(ids), _ptr(scores), _ptr(ws), ws_bytes, _stream()), "rp_score_topk")
    return ids, scores


class CEHeadState:
    """Buffers shared by rp_ce_head_fwd / rp_ce_head_bwd for one (capacity, n_items, d)."""

    def __init__(self, capacity: int, n_items: int, d: int, device):
        L = lib()
        self.capacity, self.n_items, self.d = capacity, n_items, d
        self.ws_bytes = L.rp_ce_head_workspace(capacity, n_items, d)
        self.ws = torch.zeros(self.ws_bytes, device=device, dtype=torch.uint8)
        self.loss = torch.zeros(2, device=device, dtype=torch.float32)
        self.lse = torch.zeros(capacity, device=device, dtype=torch.float32)
        cap128 = (capacity + 127) // 128 * 128
        self.cvec = torch.full((cap128,), float("-inf"), device=device, dtype=torch.float32)


def ce_head_fwd(st: CEHeadState, hc, table, labels, n_valid, bias=None, d_hc=None, n_valid_hint: int = 0, row_weight=None,
                loss_kind: int = 0, log_eps: float = 1e-6, clamp: float = 100.0):
    """hc bf16 [capacity,d] (zero/finite beyond n_valid), table bf16 [I,d], labels int32 [capacity], n_valid int32 [1].
    With ``d_hc`` (bf16 [capacity,d]) the fused forward+dH pass runs and d_hc is final after this call.
    ``row_weight`` fp32 [capacity] (compacted order) / ``loss_kind`` 1 = LogInCE: the per-row variants (rp_ce_head_fwd_w).
    Returns st.loss (fp32 [2]: mean loss, 1/n_valid) - a view that the next call overwrites."""
    _need(hc, torch.bfloat16, "hc")
    _need(table, torch.bfloat16, "table")
    _need(labels, torch.int32, "labels")
    _need(n_valid, torch.int32, "n_valid")
    if d_hc is not None:
        _need(d_hc, torch.bfloat16, "d_hc")
    st.fused = d_hc is not None and st.d <= 256
    if row_weight is not None:
        _need(row_weight, torch.float32, "row_weight")
    check(lib().rp_ce_head_fwd_w(_ptr(hc), _ptr(table), _ptr(bias), _ptr(labels), _ptr(n_valid), st.capacity, st.n_items, st.d,
                                 _ptr(st.loss), _ptr(st.lse), _ptr(st.cvec), _ptr(d_hc), int(n_valid_hint), _ptr(row_weight),
                                 int(loss_kind), float(log_eps), float(clamp), _ptr(st.ws), st.ws_bytes, _stream()),
          "rp_ce_head_fwd_w")
    return st.loss


def ce_head_fused_taken(st: CEHeadState) -> bool:
    """Diagnostic (one device read): did the last fused forward pass run, i.e. did the device-side bound on |logit| hold?
    (workspace layout of csrc/rp_ce_head.cu: the flag follows the partials, the block sums, the ticket and bound[3])"""
    off = st.capacity * 32 * 2 * 8 + 4096 + 16
    return bool(st.ws[off:off + 4].view(torch.int32).item() != 0)


def ce_head_bwd(st: CEHeadState, hc, table, labels, n_valid, d_hc, d_table, bias=None, d_bias=None, n_valid_hint: int = 0):
    """d_hc bf16 [capacity,d] (computed here unless the forward ran fused), d_table fp32 [>=I, d] (rows < I overwritten)."""
    _need(d_hc, torch.bfloat16, "d_hc")
    _need(d_table, torch.float32, "d_table")
    check(lib().rp_ce_head_bwd(_ptr(hc), _ptr(table), _ptr(bias), _ptr(labels), _ptr(n_valid), st.capacity, st.n_items, st.d,
                               _ptr(st.loss), _ptr(st.cvec), _ptr(d_hc), _ptr(d_table), _ptr(d_bias), int(getattr(st, "fused", False)),
                               int(n_valid_hint), _ptr(st.ws), st.ws_bytes, _stream()), "rp_ce_head_bwd")


class BCEHeadState:
    """Buffers shared by rp_bce_head_fwd / rp_bce_head_bwd for one (capacity, n_items, d), d in {64, 128, 256}."""

    def __init__(self, capacity: int, n_items: int, d: int, device, loss=None):
        """``loss``: an fp32 [2] device buffer to write the loss into (the engines share the CE head's), else a new one."""
        if d not in (64, 128, 256):
            raise NotImplementedError(f"the full-catalog BCE head supports hidden sizes 64, 128 and 256 (got {d})")
        self.capacity, self.n_items, self.d = capacity, n_items, d
        self.ws_bytes = lib().rp_bce_head_workspace(capacity, n_items, d)
        self.ws = torch.zeros(self.ws_bytes, device=device, dtype=torch.uint8)
        self.loss = loss if loss is not None else torch.zeros(2, device=device, dtype=torch.float32)


def bce_head_fwd(st: BCEHeadState, hc, table, labels, n_valid, d_hc, bias=None, n_valid_hint: int = 0):
    """Full-catalog BCE: hc bf16 [capacity,d], table bf16 [I,d], labels int32 [capacity], n_valid int32 [1], bias fp32
    [round_up(I,128)] or None.  d_hc (bf16 [capacity,d]) is final after this call.  Returns st.loss (fp32 [2]: mean loss,
    1/n_valid) - a view that the next call overwrites."""
    _need(hc, torch.bfloat16, "hc")
    _need(table, torch.bfloat16, "table")
    _need(labels, torch.int32, "labels")
    _need(n_valid, torch.int32, "n_valid")
    _need(d_hc, torch.bfloat16, "d_hc")
    check(lib().rp_bce_head_fwd(_ptr(hc), _ptr(table), _ptr(bias), _ptr(labels), _ptr(n_valid), st.capacity, st.n_items, st.d,
                                _ptr(st.loss), _ptr(d_hc), int(n_valid_hint), _ptr(st.ws), st.ws_bytes, _stream()),
          "rp_bce_head_fwd")
    return st.loss


def bce_head_bwd(st: BCEHeadState, hc, table, labels, n_valid, d_table, bias=None, d_bias=None):
    """d_table fp32 [>=I, d] (rows < I overwritten), d_bias fp32 [>=I] (iff bias; overwritten) of the last bce_head_fwd."""
    _need(d_table, torch.float32, "d_table")
    check(lib().rp_bce_head_bwd(_ptr(hc), _ptr(table), _ptr(bias), _ptr(labels), _ptr(n_valid), st.capacity, st.n_items, st.d,
                                _ptr(st.loss), _ptr(d_table), _ptr(d_bias), _ptr(st.ws), st.ws_bytes, _stream()),
          "rp_bce_head_bwd")


def gemm(A, B, C, M, N, K, *, a_mn=False, b_mn=False, bias=None, act=0, residual=None, rowmask=None, drop_p=0.0,
         drop_offset=0, seed=0, seed_ptr=None, out_mode=0, split_k=1, gate=None, gate_scale=1.0, gate_mode=0, alpha=1.0,
         batch=1, inner=1, a_off=(0, 0, 0, 0, 0, 0), b_off=(0, 0, 0, 0, 0, 0), c_geom=None, rowmask_oo=0, C2=None,
         post_drop_p=0.0, post_drop_offset=0, c_split_stride=0, row_exp2_offset=None, m_limit=None, m_limit_base=0,
         k_limit=None, k_limit_base=0, L=None):
    """C = epilogue(alpha * A(m,k) . B(n,k)) through rp_gemm (include/rp_b200.h).  A / B are 2-D bf16 tensors (views allowed:
    pointer, shape and row pitch are taken from the tensor); x_mn selects the MN-major reading of an operand."""
    g = GemmDesc()
    g.A, g.a_rows, g.a_cols, g.lda, g.a_mn = A.data_ptr(), A.shape[0], A.shape[1], A.stride(0), int(a_mn)
    g.B, g.b_rows, g.b_cols, g.ldb, g.b_mn = B.data_ptr(), B.shape[0], B.shape[1], B.stride(0), int(b_mn)
    g.M, g.N, g.K, g.batch, g.inner = M, N, K, batch, inner
    g.a_r0, g.a_ro, g.a_ri, g.a_c0, g.a_co, g.a_ci = a_off
    g.b_r0, g.b_ro, g.b_ri, g.b_c0, g.b_co, g.b_ci = b_off
    g.C = C.data_ptr()
    g.ldc, g.c_off0, g.c_oo, g.c_oi = (C.stride(0), 0, 0, 0) if c_geom is None else c_geom
    g.out_mode, g.alpha, g.act = out_mode, alpha, act
    g.bias = _ptr(bias)
    g.residual = _ptr(residual)
    g.rowmask = _ptr(rowmask)
    g.rowmask_off0, g.rowmask_oo = 0, rowmask_oo
    g.drop_p, g.seed, g.drop_offset, g.seed_ptr = drop_p, seed, drop_offset, seed_ptr
    g.split_k = split_k
    g.gate, g.gate_scale, g.gate_mode = _ptr(gate), gate_scale, gate_mode
    g.C2 = _ptr(C2)
    g.post_drop_p, g.post_drop_offset = post_drop_p, post_drop_offset
    g.c_split_stride = c_split_stride
    g.row_exp2_offset = _ptr(row_exp2_offset)
    g.m_limit_dev, g.m_limit_base = _ptr(m_limit), m_limit_base
    g.k_limit_dev, g.k_limit_base = _ptr(k_limit), k_limit_base
    check((L or lib()).rp_gemm(ctypes.byref(g), _stream()), "rp_gemm")
