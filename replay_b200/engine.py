"""Execution engine of the SASRec hot path on B200: owns the flat parameter / gradient / optimizer buffers and the
activation workspace, and sequences the hand-written sm_100a kernels (librp_b200.so, include/rp_b200.h) for

    train step  = batch prep -> embedding -> N x [LN, QKV GEMMs, fused attention, out-proj, LN, FFN] -> final LN with
                  valid-target compaction -> fused CE head  -> full backward -> (gradient all-reduce) -> Adam
    predict     = same body without dropout -> last hidden state -> fused score + seen-mask + top-K head

It is the host-side counterpart of the reference's torch modules (replay/nn/sequential/sasrec/model.py:85-113,258-307 and
replay/models/nn/sequential/sasrec/model.py:159-180); the ``replay_b200.nn`` / ``replay_b200.models`` classes that mirror
the reference API delegate to it.  torch supplies device memory, streams, CUDA graphs and the NCCL process group only.
"""
from __future__ import annotations

import contextlib
import ctypes
import math
import os
from dataclasses import dataclass

import torch

from ._lib import SampledDesc, AttnBwdDesc, AttnDesc, GemmDesc, WgradPair, check, lib


@dataclass
class EncoderConfig:
    n_items: int
    d: int
    n_heads: int
    n_blocks: int
    max_len: int
    dropout: float = 0.0
    variant: str = "new"  # "new": replay.nn.sequential.SasRec ; "legacy": replay.models.nn.sequential.SasRecModel
    lnf_eps: float | None = None

    def __post_init__(self):
        if self.variant not in ("new", "legacy"):
            raise ValueError(f"unknown variant {self.variant}")
        if self.d % self.n_heads:
            raise ValueError("d must be divisible by n_heads")
        if self.d // self.n_heads > 128:
            raise ValueError("head_dim must not exceed 128 (one 128-wide tensor-core feature slot per head)")
        if self.dp not in (64, 128, 256, 512):
            raise ValueError(f"hidden size {self.d} with {self.n_heads} heads needs {self.dp} padded columns; the kernels "
                             "support 64/128/256/512 (= n_heads x 64-wide slots, or 128-wide for head_dim > 64)")
        if self.lnf_eps is None:
            # new: torch.nn.LayerNorm default (nn/sequential/sasrec/model.py:248); legacy: 1e-8 (sasrec/model.py:463)
            self.lnf_eps = 1e-5 if self.variant == "new" else 1e-8

    @property
    def pad_id(self) -> int:
        return self.n_items

    # ---- feature slots: every head occupies one 64-wide (head_dim <= 64) or 128-wide tensor-core slot.  The reference's own
    # defaults (embedding_dim 192 / 4 heads -> head_dim 48; legacy hidden_size 50; examples d 64 / 2 heads -> 32) leave padded
    # columns, which are zero in every activation / weight / gradient (include/rp_b200.h "PADDED FEATURE SLOTS")
    @property
    def head_dim(self) -> int:
        return self.d // self.n_heads

    @property
    def head_slot(self) -> int:
        return 64 if self.head_dim <= 64 else 128

    @property
    def dp(self) -> int:
        """columns of the token-major activations / weights as the kernels see them"""
        return self.n_heads * self.head_slot

    @property
    def hd_valid(self) -> int:
        """the kernels' `hd_valid` argument: real features per slot, 0 when nothing is padded"""
        return 0 if self.head_dim == self.head_slot else self.head_dim

    def feat_index(self, device=None) -> torch.Tensor:
        """padded column of every true feature: (head h, j) -> h * slot + j"""
        h = torch.arange(self.n_heads, device=device).repeat_interleave(self.head_dim)
        j = torch.arange(self.head_dim, device=device).repeat(self.n_heads)
        return h * self.head_slot + j


_BLOCK_PARAMS = ("ln1_w", "ln1_b", "in_w", "in_b", "out_w", "out_b", "ln2_w", "ln2_b", "w1", "b1", "w2", "b2")


def _ru(x, m):
    return (x + m - 1) // m * m


def param_shapes(cfg: EncoderConfig) -> list:
    """(name, padded shape) of every parameter, in the order of the flat buffers."""
    d, I = cfg.dp, cfg.n_items
    shapes = [("item_emb", (I + 1, d)), ("pos_emb", (cfg.max_len, d))]
    for i in range(cfg.n_blocks):
        shapes += [(f"b{i}.ln1_w", (d,)), (f"b{i}.ln1_b", (d,)), (f"b{i}.in_w", (3 * d, d)), (f"b{i}.in_b", (3 * d,)),
                   (f"b{i}.out_w", (d, d)), (f"b{i}.out_b", (d,)), (f"b{i}.ln2_w", (d,)), (f"b{i}.ln2_b", (d,)),
                   (f"b{i}.w1", (d, d)), (f"b{i}.b1", (d,)), (f"b{i}.w2", (d, d)), (f"b{i}.b2", (d,))]
    return shapes + [("lnf_w", (d,)), ("lnf_b", (d,))]


def pad_kind(name: str):
    """(row kind, column kind) of a parameter in the padded layout: 'f' = feature axis (scattered into the head slots),
    'f3' = three stacked feature axes (packed in-projection), None = not a feature axis."""
    leaf = name.split(".")[-1]
    if leaf in ("item_emb", "pos_emb"):
        return (None, "f")
    if leaf == "in_w":
        return ("f3", "f")
    if leaf == "in_b":
        return ("f3", None)
    if leaf in ("out_w", "w1", "w2"):
        return ("f", "f")
    return ("f", None)  # LayerNorm weights / biases, linear biases


def true_shape(cfg: EncoderConfig, name: str, padded_shape) -> tuple:
    """The reference's shape of parameter ``name`` stored with ``padded_shape``: only the axes ``pad_kind`` marks as
    feature axes shrink (a row count such as max_len or n_items + 1 never does, whatever its value)."""
    if not getattr(cfg, "hd_valid", 0):
        return tuple(padded_shape)
    true = {"f": cfg.d, "f3": 3 * cfg.d}
    kinds = pad_kind(name)[:len(padded_shape)]
    return tuple(x if k is None else true[k] for x, k in zip(padded_shape, kinds))


class _CountingLib:
    """Proxy over the ctypes library that counts the sm_100a kernel launches issued through it (bench.py reports them)."""

    KERNELS = {"rp_gemm": 1, "rp_attn_fwd": 1, "rp_attn_bwd": 1, "rp_attn_last": 1, "rp_attn_softmax_bwd": 1, "rp_prepare_batch": 2, "rp_embed_fwd": 1,
               "rp_embed_bwd": 2, "rp_layernorm_fwd": 1, "rp_layernorm_bwd": 1, "rp_dropout_bwd": 1, "rp_colsum": 1, "rp_colsum_multi": 1,
               "rp_adam_step": 2, "rp_cast_bf16": 1, "rp_counter_add": 1, "rp_reduce_splits": 1, "rp_ce_head_fwd": 2, "rp_ce_head_bwd": 3, "rp_bce_head_fwd": 2, "rp_bce_head_bwd": 2,
               "rp_score_topk": 2, "rp_seen_prepare": 1, "rp_sampled_head_fwd": 4, "rp_sampled_head_bwd": 4, "rp_ffn_fused": 1, "rp_post_attn_fused": 1,
               "rp_post_attn_train": 1, "rp_wgrad_group": 2, "rp_ln_qkv_fused": 1, "rp_pre_attn_bwd": 1,
               "rp_post_attn_bwd": 1}

    def __init__(self, L):
        self._L = L
        self.count = 0
        self._cache = {}

    def __getattr__(self, name):
        w = self._cache.get(name)
        if w is None:
            fn, k = getattr(self._L, name), self.KERNELS.get(name, 0)

            def w(*a, _fn=fn, _k=k):
                self.count += _k
                return _fn(*a)

            self._cache[name] = w
        return w


class SasRecEngine:
    def __init__(self, cfg: EncoderConfig, max_batch: int, seq_len: int, device="cuda", seed: int = 0,
                 with_grad: bool = True):
        self.cfg = cfg
        self.dev = torch.device(device)
        self.B, self.L = max_batch, seq_len
        self._check_geometry(seq_len)
        self.T = max_batch * seq_len
        self.Lp = _ru(seq_len, 64)
        self.with_grad = with_grad
        self.lib = _CountingLib(lib())
        d = cfg.dp   # padded width: what buffers and kernels use; cfg.d is the model's true hidden size
        self._feat = cfg.feat_index(self.dev)
        # ---------------------------------------------------------------- flat parameter layout
        self.layout = {}
        off = 0
        for name, shp in param_shapes(cfg):
            n = math.prod(shp)
            self.layout[name] = (off, shp)
            off = _ru(off + n, 64)
        self.n_flat = off
        f32 = dict(device=self.dev, dtype=torch.float32)
        self.p32 = torch.zeros(off, **f32)
        self.p16 = torch.zeros(off, device=self.dev, dtype=torch.bfloat16)
        self.params = {k: self.p32[o:o + math.prod(s)].view(s) for k, (o, s) in self.layout.items()}
        self.params16 = {k: self.p16[o:o + math.prod(s)].view(s) for k, (o, s) in self.layout.items()}
        if with_grad:
            self._alloc_grad_state()
        self.rng_counter = torch.zeros(1, device=self.dev, dtype=torch.int64)
        self.seed = seed & 0xFFFFFFFFFFFF
        self.training = with_grad
        # fused tcgen05 attention backward: head_dim 64, L <= 256; otherwise saved probabilities + batched GEMMs
        self.fused_attn_bwd = cfg.head_slot == 64 and seq_len <= 256
        self.sampled = None       # full-catalog CE unless set_loss() selects a sampled head
        self.bce = None           # ... or the full-catalog BCE head
        self._loss_args = None
        self.fused_ffn_eval = True  # eval / predict: one-pass FFN kernel for d <= 128
        self.fused_post_attn_eval = True  # eval / predict: out-projection + LayerNorm + FFN in one kernel for d <= 128
        # training: out-projection + LayerNorm + FFN (+ dropouts, saved activations) in one pass for d <= 128; all weight / bias
        # gradients of a block in one grouped launch (RP_FUSED_BODY=0 restores round 1's launch-per-GEMM body for A/B runs)
        fused_body = os.environ.get("RP_FUSED_BODY", "1") != "0"
        self.fused_post_attn_train = fused_body
        self.fused_wgrad = fused_body and d <= 256          # rp_wgrad_group: at most 48 output tiles per block
        self.fused_pre_attn = fused_body and d <= 128       # LN1 + Q / KV projections in one pass (forward and backward)
        self.fused_post_attn_bwd = fused_body and d <= 128  # dropout' + FFN + LN2 + out-projection backward in one pass
        self.fused_ce = True      # single-pass CE forward + dH (guarded on the device by a bound on |logit|)
        self.n_valid_hint = 0     # host estimate of the number of valid targets per step (load balance of the CE head only)
        self._alloc_workspace()
        self.init_parameters(seed)

    # ------------------------------------------------------------------------------------------------ state that outlives a batch geometry
    def _alloc_grad_state(self):
        """Flat gradient, Adam moments, learning rate and step counter: sized by the configuration only, allocated once."""
        f32 = dict(device=self.dev, dtype=torch.float32)
        n = self.n_flat
        # data-parallel runs on one NVLink node: the gradient lives in a symmetric (peer-mapped) allocation so that the
        # all-reduce is this repo's own in-graph kernel (replay_b200/peer.py); otherwise a plain buffer (ncclAllReduce)
        from .peer import alloc_peer_grad

        self.peer = alloc_peer_grad(n, self.dev)
        self.g32 = self.peer.g32 if self.peer is not None else torch.zeros(n, **f32)
        self.adam_m = torch.zeros(n, **f32)
        self.adam_v = torch.zeros(n, **f32)
        self.grads = {k: self.g32[o:o + math.prod(s)].view(s) for k, (o, s) in self.layout.items()}
        self.lr = torch.full((1,), 1e-3, **f32)
        self.step_count = torch.zeros(1, device=self.dev, dtype=torch.int32)

    def _check_geometry(self, seq_len: int):
        cfg = self.cfg
        if seq_len > cfg.max_len:
            raise ValueError(f"sequence length {seq_len} exceeds max_len {cfg.max_len}")
        if cfg.variant == "legacy" and seq_len != cfg.max_len:
            raise ValueError("legacy SASRec needs seq_len == max_len (sasrec/model.py:528-529)")
        if seq_len > 512 or (seq_len > 256 and cfg.head_slot != 64):
            raise ValueError("attention kernels support seq_len <= 256 (head_dim 128) / <= 512 (head_dim 64)")

    def resize(self, max_batch: int, seq_len: int, with_grad: bool | None = None):
        """New batch geometry (a larger validation / predict batch, another sequence length): ONLY the activation workspace is
        re-allocated.  Parameters, the bf16 shadow, gradients, Adam moments, the learning rate, the step counter and the
        dropout counter keep their buffers - and their addresses, so an ``nn.Parameter`` / optimizer / CUDA pointer that
        refers to them stays valid."""
        self._check_geometry(seq_len)
        if with_grad and not self.with_grad:
            self.with_grad = True
            self._alloc_grad_state()
        self.B, self.L = max_batch, seq_len
        self.T = max_batch * seq_len
        self.Lp = _ru(seq_len, 64)
        self.fused_attn_bwd = self.cfg.head_slot == 64 and seq_len <= 256
        self._realloc_workspace()
        if self._loss_args is not None and self._loss_args[0] != "ce":  # sampled-head buffers are sized by (B, T)
            self.sampled = None
            if self.with_grad:
                self.set_loss(*self._loss_args[:1], **self._loss_args[1])
        return self

    def _realloc_workspace(self):
        self._alloc_workspace()

    # ------------------------------------------------------------------------------------------------ parameters
    def _pad_kind(self, name: str):
        return pad_kind(name)

    def _axis_index(self, kind):
        if kind == "f":
            return self._feat
        dp = self.cfg.dp
        return torch.cat([self._feat + k * dp for k in range(3)])

    def import_named(self, name: str, value: torch.Tensor, dst=None):
        """Write a TRUE-shape tensor (reference layout) into the padded parameter ``name`` (padded entries become zero)."""
        tgt = (self.params if dst is None else dst)[name]
        v = value.to(self.dev, torch.float32)
        if self._hdv() == 0:
            tgt.copy_(v.reshape(tgt.shape))
            return
        rk, ck = self._pad_kind(name)
        tgt.zero_()
        if tgt.dim() == 1:
            tgt[self._axis_index(rk)] = v
        else:
            rows = self._axis_index(rk) if rk else torch.arange(tgt.shape[0], device=self.dev)
            cols = self._axis_index(ck) if ck else torch.arange(tgt.shape[1], device=self.dev)
            tgt[rows[:, None], cols[None, :]] = v

    def export_named(self, name: str, source=None) -> torch.Tensor:
        """The TRUE-shape view (a copy) of the padded parameter / gradient ``name``."""
        t = (self.params if source is None else source)[name].detach()
        if self._hdv() == 0:
            return t.clone()
        rk, ck = self._pad_kind(name)
        if t.dim() == 1:
            return t[self._axis_index(rk)].clone()
        rows = self._axis_index(rk) if rk else torch.arange(t.shape[0], device=t.device)
        cols = self._axis_index(ck) if ck else torch.arange(t.shape[1], device=t.device)
        return t[rows[:, None], cols[None, :]].clone()

    def true_shape(self, name: str):
        return true_shape(self.cfg, name, self.layout[name][1])

    def init_parameters(self, seed: int = 0):
        """Reference-style init: xavier_normal_ on >=2-D tensors, LN (1, 0), biases zero / U(+-1/sqrt(fan_in)) for the
        conv layers, pad row zero (new path, nn/embedding.py:198-200) - drawn in the model's TRUE shapes, then laid out in the
        head slots.  Weights are normally loaded from a reference state_dict instead (``load_canonical``)."""
        g = torch.Generator(device="cpu").manual_seed(seed)
        d = self.cfg.d
        with torch.no_grad():
            for name in self.layout:
                shp = self.true_shape(name)
                if len(shp) == 2:
                    std = math.sqrt(2.0 / (shp[0] + shp[1]))
                    v = torch.randn(shp, generator=g) * std
                    if name == "item_emb" and self.cfg.variant == "new":
                        v[self.cfg.pad_id].zero_()
                elif name.endswith(("ln1_w", "ln2_w", "lnf_w")):
                    v = torch.ones(shp)
                elif name.endswith((".b1", ".b2")):
                    v = (torch.rand(shp, generator=g) * 2 - 1) / math.sqrt(d)
                else:
                    v = torch.zeros(shp)
                self.import_named(name, v)
        self.refresh_shadow()

    def refresh_shadow(self):
        check(self.lib.rp_cast_bf16(self.p32.data_ptr(), self.p16.data_ptr(), self.n_flat, self._stream()), "rp_cast_bf16")

    def load_canonical(self, P: dict):
        """Copy weights from the canonical dict used by oracle/ (keys item_emb, pos_emb, blocks[i][...], lnf_w, lnf_b)."""
        with torch.no_grad():
            self.import_named("item_emb", P["item_emb"])
            self.import_named("pos_emb", P["pos_emb"])
            for i, blk in enumerate(P["blocks"]):
                for k in _BLOCK_PARAMS:
                    self.import_named(f"b{i}.{k}", blk[k])
            self.import_named("lnf_w", P["lnf_w"])
            self.import_named("lnf_b", P["lnf_b"])
        self.refresh_shadow()

    def export_canonical(self, source=None) -> dict:
        ex = lambda k: self.export_named(k, source).cpu()  # noqa: E731
        P = {"item_emb": ex("item_emb"), "pos_emb": ex("pos_emb"), "blocks": [], "lnf_w": ex("lnf_w"), "lnf_b": ex("lnf_b")}
        for i in range(self.cfg.n_blocks):
            P["blocks"].append({k: ex(f"b{i}.{k}") for k in _BLOCK_PARAMS})
        return P

    def unpad_features(self, t: torch.Tensor) -> torch.Tensor:
        """[..., dp] activations -> [..., d] (the reference's hidden size)"""
        return t if self._hdv() == 0 else t[..., self._feat].contiguous()

    def pad_features(self, t: torch.Tensor) -> torch.Tensor:
        if self._hdv() == 0:
            return t
        out = torch.zeros(*t.shape[:-1], self.cfg.dp, device=t.device, dtype=t.dtype)
        out[..., self._feat] = t
        return out

    # ------------------------------------------------------------------------------------------------ workspace
    def _alloc_workspace(self):
        cfg, T, d, dev = self.cfg, self.T, self.cfg.dp, self.dev
        self._alloc_B, self._alloc_T, self._sub_last_idx = self.B, self.T, {}
        bf = dict(device=dev, dtype=torch.bfloat16)
        f32 = dict(device=dev, dtype=torch.float32)
        i32 = dict(device=dev, dtype=torch.int32)
        BH = self.B * cfg.n_heads
        self.ids32 = torch.zeros(T, **i32)
        self.pad_u8 = torch.zeros(T, device=dev, dtype=torch.uint8)
        self.in_ids = torch.zeros(T, device=dev, dtype=torch.int64)
        self.in_pad = torch.zeros(T, device=dev, dtype=torch.bool)
        self.in_labels = torch.zeros(T, device=dev, dtype=torch.int64)
        self.in_tmask = torch.zeros(T, device=dev, dtype=torch.bool)
        self.valid_idx = torch.zeros(T, **i32)
        self.labels_c = torch.zeros(T, **i32)
        self.n_valid = torch.zeros(1, **i32)
        self.prep_scratch = torch.zeros((T + 1023) // 1024 + 1, **i32)
        nb = cfg.n_blocks
        self.x = [torch.zeros(T, d, **bf) for _ in range(nb + 1)]
        self.act = []
        for _ in range(nb):
            a = {k: torch.zeros(T, d, **bf) for k in ("q_in", "Q", "O", "h", "y", "u")}
            a["KV"] = torch.zeros(T, 2 * d, **bf)
            for k in ("mean1", "rstd1", "mean2", "rstd2"):
                a[k] = torch.zeros(T, **f32)
            if self.with_grad:
                if not self.fused_attn_bwd:
                    a["P"] = torch.zeros(BH, self.Lp, self.Lp, **bf)
                a["inv_sum"] = torch.zeros(BH, self.Lp, **f32)
                a["m2"] = torch.zeros(BH, self.Lp, **f32)
            self.act.append(a)
        self.hc = torch.zeros(T, d, **bf)
        self.meanf = torch.zeros(T, **f32)
        self.rstdf = torch.zeros(T, **f32)
        self.hq = torch.zeros(self.B, d, **bf)
        self.last_idx = (torch.arange(self.B, device=dev, dtype=torch.int32) * self.L + (self.L - 1)).contiguous()
        self.last_buf = {k: torch.zeros(self.B, d, **bf) for k in ("q_in", "Q", "O", "h", "y", "u")}
        self.last_rows = torch.zeros(self.B, d, **bf)
        self.last_pad = torch.zeros(self.B, device=dev, dtype=torch.bool)
        if self.with_grad:
            from .ops import CEHeadState

            self.ce = CEHeadState(T, cfg.n_items, d, dev)
            self.s = {k: torch.zeros(T, d, **bf) for k in ("dhc", "dxa", "dxb", "d_t", "du", "dy", "dh", "d_o", "dQ", "dq_in", "tmp")}
            self.s["dKV"] = torch.zeros(T, 2 * d, **bf)
            if not self.fused_attn_bwd:
                self.s["dpd"] = torch.zeros(BH, self.Lp, self.Lp, **bf)
            self.wg_ws = torch.zeros(148 * 4 * d * d, **f32)  # split-K partials of the weight-gradient GEMMs
            self._wgrad_ws = None  # workspace of rp_wgrad_group, sized on first use

    def _stream(self):
        return torch.cuda.current_stream(self.dev).cuda_stream

    @contextlib.contextmanager
    def sub_geometry(self, batch: int, seq_len: int):
        """Inference only: run a SMALLER [batch, seq_len] problem inside the allocated workspace (every activation buffer is a
        flat [T, ...] array, so a problem with batch * seq_len <= T rows uses a prefix of each).  Used by the length-bucketed
        predict (core.py): users whose whole history fits the last ``seq_len`` positions are evaluated on that window only -
        positions are right-aligned (``pos0 = max_len - L``), so the trimmed window sees the same position embeddings."""
        self._check_geometry(seq_len)
        if batch > self._alloc_B or batch * seq_len > self._alloc_T:
            raise ValueError(f"sub-geometry ({batch}, {seq_len}) exceeds the workspace ({self._alloc_B} x {self._alloc_T // self._alloc_B})")
        saved = (self.B, self.L, self.T, self.Lp, self.last_idx)
        key = (batch, seq_len)
        if key not in self._sub_last_idx:
            self._sub_last_idx[key] = (torch.arange(batch, device=self.dev, dtype=torch.int32) * seq_len + (seq_len - 1)).contiguous()
        self.B, self.L, self.T, self.Lp, self.last_idx = batch, seq_len, batch * seq_len, _ru(seq_len, 64), self._sub_last_idx[key]
        try:
            yield self
        finally:
            self.B, self.L, self.T, self.Lp, self.last_idx = saved

    # ------------------------------------------------------------------------------------------------ kernel helpers
    def _gemm(self, A, B, C, M, N, K, *, a_mn=False, b_mn=False, bias=None, act=0, residual=None, rowmask=None,
              drop_p=0.0, drop_site=0, out_mode=0, split_k=1, gate=None, gate_scale=1.0, alpha=1.0, batch=1, inner=1,
              a_off=(0, 0, 0, 0, 0, 0), b_off=(0, 0, 0, 0, 0, 0), c_geom=None, rowmask_oo=0, C2=None, gate_mode=0,
              post_drop_p=0.0, post_drop_site=0, c_split_stride=0):
        g = GemmDesc()
        g.A, g.a_rows, g.a_cols, g.lda, g.a_mn = A.data_ptr(), A.shape[0], A.shape[1], A.stride(0), int(a_mn)
        g.B, g.b_rows, g.b_cols, g.ldb, g.b_mn = B.data_ptr(), B.shape[0], B.shape[1], B.stride(0), int(b_mn)
        g.M, g.N, g.K, g.batch, g.inner = M, N, K, batch, inner
        g.a_r0, g.a_ro, g.a_ri, g.a_c0, g.a_co, g.a_ci = a_off
        g.b_r0, g.b_ro, g.b_ri, g.b_c0, g.b_co, g.b_ci = b_off
        g.C = C.data_ptr()
        if c_geom is None:
            g.ldc, g.c_off0, g.c_oo, g.c_oi = C.stride(0), 0, 0, 0
        else:
            g.ldc, g.c_off0, g.c_oo, g.c_oi = c_geom
        g.out_mode = out_mode
        g.alpha = alpha
        g.bias = None if bias is None else bias.data_ptr()
        g.act = act
        g.residual = None if residual is None else residual.data_ptr()
        g.rowmask = None if rowmask is None else rowmask.data_ptr()
        g.rowmask_off0, g.rowmask_oo = 0, rowmask_oo
        g.drop_p = drop_p
        g.seed = self.seed
        g.drop_offset = drop_site << 40
        g.seed_ptr = self.rng_counter.data_ptr()
        g.split_k = split_k
        g.gate = None if gate is None else gate.data_ptr()
        g.gate_scale = gate_scale
        g.C2 = None if C2 is None else C2.data_ptr()
        g.gate_mode = gate_mode
        g.post_drop_p = post_drop_p
        g.post_drop_offset = post_drop_site << 40
        g.c_split_stride = c_split_stride
        check(self.lib.rp_gemm(ctypes.byref(g), self._stream()), "rp_gemm")

    def _wgrad(self, dY, X, dW, n_out, n_in):
        """dW[n_out, n_in] += dY[T, n_out]^T . X[T, n_in]: both operands read MN-major in place; split-K over about one wave
        of CTAs, each storing its fp32 partial tile (no atomics: 100+ CTAs hammering the same 16 K addresses serialise in
        L2), then one reduction pass adds the partials into the gradient buffer (deterministic)."""
        tiles = ((n_out + 127) // 128) * ((n_in + 127) // 128 if n_in > 64 else 1)
        chunks = (self.T + 63) // 64
        n = n_out * n_in
        per = int(os.environ.get("RP_WGRAD_CHUNKS", "8"))
        split = max(1, min(chunks // per, (148 + tiles - 1) // tiles, self.wg_ws.numel() // n))
        self._gemm(dY, X, self.wg_ws, n_out, n_in, self.T, a_mn=True, b_mn=True, out_mode=3, split_k=split,
                   c_geom=(n_in, 0, 0, 0), c_split_stride=n)
        check(self.lib.rp_reduce_splits(self.wg_ws.data_ptr(), split, n, n, dW.data_ptr(), 1, self._stream()), "rp_reduce_splits")

    def _wgrad_group(self, pairs):
        """[(dY bf16 [T, n_out], X bf16 [T, n_in], dW fp32 [n_out, n_in], db fp32 [n_out] | None), ...]: every weight and bias
        gradient of a block in one tcgen05 launch + one deterministic reduction launch (csrc/rp_wgrad.cu).  Gradients are
        accumulated (+=) like the un-fused path does."""
        n = len(pairs)
        arr = (WgradPair * n)()
        for k, (dY, X, dW, db) in enumerate(pairs):
            arr[k].dY, arr[k].dy_ld, arr[k].n_out = dY.data_ptr(), dY.stride(0), dW.shape[0]
            arr[k].X, arr[k].x_ld, arr[k].n_in = X.data_ptr(), X.stride(0), dW.shape[1]
            arr[k].dW, arr[k].dw_ld = dW.data_ptr(), dW.stride(0)
            arr[k].db = None if db is None else db.data_ptr()
        need = self.lib.rp_wgrad_group_workspace(arr, n)
        if need == 0:
            raise ValueError("rp_wgrad_group: unsupported gradient shapes")
        if self._wgrad_ws is None or self._wgrad_ws.numel() < need:
            self._wgrad_ws = torch.zeros(need, device=self.dev, dtype=torch.uint8)
        check(self.lib.rp_wgrad_group(arr, n, self.T, 1, self._wgrad_ws.data_ptr(), self._wgrad_ws.numel(), self._stream()),
              "rp_wgrad_group")

    def _colsum(self, dY, db):
        check(self.lib.rp_colsum(dY.data_ptr(), dY.shape[0], dY.shape[1], dY.stride(0), db.data_ptr(), self._stream()),
              "rp_colsum")

    def _colsum_multi(self, pairs):
        """[(dY bf16 [T, cols], db fp32 [cols]), ...] (<= 6) in one launch: the bias gradients of one block."""
        n = len(pairs)
        dy = (ctypes.c_void_p * n)(*[a.data_ptr() for a, _ in pairs])
        db = (ctypes.c_void_p * n)(*[b.data_ptr() for _, b in pairs])
        cols = (ctypes.c_int * n)(*[a.shape[1] for a, _ in pairs])
        ld = (ctypes.c_longlong * n)(*[a.stride(0) for a, _ in pairs])
        check(self.lib.rp_colsum_multi(n, dy, cols, ld, db, pairs[0][0].shape[0], self._stream()), "rp_colsum_multi")

    def _ln_fwd(self, x, w, b, eps, y, mean, rstd, n_rows, gather=None, n_rows_dev=None):
        check(self.lib.rp_layernorm_fwd(x.data_ptr(), w.data_ptr(), b.data_ptr(), eps, n_rows, self._dp(),
                                        None if n_rows_dev is None else n_rows_dev.data_ptr(),
                                        None if gather is None else gather.data_ptr(), y.data_ptr(), mean.data_ptr(),
                                        rstd.data_ptr(), self._hdv(), self._stream()), "rp_layernorm_fwd")

    def _ln_bwd(self, dy, x, w, mean, rstd, dx, dw, db, n_rows, gather=None, n_rows_dev=None, add_to=None):
        check(self.lib.rp_layernorm_bwd(dy.data_ptr(), x.data_ptr(), w.data_ptr(), mean.data_ptr(), rstd.data_ptr(),
                                        n_rows, self._dp(), None if n_rows_dev is None else n_rows_dev.data_ptr(),
                                        None if gather is None else gather.data_ptr(),
                                        None if add_to is None else add_to.data_ptr(), dx.data_ptr(), dw.data_ptr(),
                                        db.data_ptr(), self._hdv(), self._stream()), "rp_layernorm_bwd")

    def _dp(self) -> int:
        return getattr(self.cfg, "dp", self.cfg.d)   # BertConfig has no padded layout

    def _hdv(self) -> int:
        return getattr(self.cfg, "hd_valid", 0)

    def _site(self, blk, k):
        return 1 + blk * 8 + k

    # ------------------------------------------------------------------------------------------------ forward
    def set_batch(self, ids, pad_mask, labels=None, target_mask=None):
        """Stage one batch ([B, L] int64 ids, bool masks) into the engine's static input buffers (device copies)."""
        B, L = ids.shape
        if L != self.L or B > self.B:
            raise ValueError(f"batch shape {tuple(ids.shape)} does not fit engine ({self.B}, {self.L})")
        self.cur_B = B
        n = B * L
        self.in_ids[:n].copy_(ids.reshape(-1), non_blocking=True)
        self.in_pad[:n].copy_(pad_mask.reshape(-1), non_blocking=True)
        if labels is not None:
            self.in_labels[:n].copy_(labels.reshape(-1), non_blocking=True)
            self.in_tmask[:n].copy_(target_mask.reshape(-1), non_blocking=True)
        if n < self.T:
            self.in_pad[n:].zero_()
            self.in_tmask[n:].zero_()

    # ------------------------------------------------------------------------------------------------ sampled heads
    SAMPLED_KINDS = {"ce_sampled": 0, "bce_sampled": 1, "legacy_ce_sampled": 2, "legacy_bce_sampled": 3}

    def set_loss(self, kind: str = "ce", n_neg: int = 0, neg_shape: str = "shared", ignore_index: int = -100,
                 log_eps: float = 1e-6, clamp: float = 100.0):
        """``"ce"`` = full-catalog CE (default).  Sampled heads (SURVEY §8 a9): ``ce_sampled`` / ``bce_sampled`` (new path,
        replay/nn/loss/ce.py:146, bce.py:98) and ``legacy_ce_sampled`` / ``legacy_bce_sampled`` (sasrec/lightning.py:310-376)
        with ``n_neg`` negatives per target, ``neg_shape`` in shared [N] / perseq [B, N] / perpos [B, L, N]."""
        self._loss_args = (kind, dict(n_neg=n_neg, neg_shape=neg_shape, ignore_index=ignore_index, log_eps=log_eps, clamp=clamp))
        # per-row variants of the full-catalog head (rp_ce_head_fwd_w): "ce_weighted" (LogOutCEWeighted / CEWeighted: sample
        # weights staged with set_row_weights) and "login_ce" (LogInCE); "ce" is the plain head
        self.ce_row = None
        self.bce = None
        if kind == "bce":
            # full-catalog BCE (replay/nn/loss/bce.py:10-95, legacy loss_type="BCE" without negatives): rp_bce_head_*
            if self._dp() not in (64, 128, 256):
                raise NotImplementedError(f"the full-catalog BCE head supports padded hidden sizes 64, 128 and 256 (got {self._dp()})")
            self.sampled = None
            if self.with_grad:
                from .ops import BCEHeadState

                self.bce = BCEHeadState(self.T, self.cfg.n_items, self._dp(), self.dev, loss=self.ce.loss)
            return
        if kind in ("ce", "ce_weighted", "login_ce"):
            self.sampled = None
            if kind != "ce":
                self.ce_row = dict(kind=1 if kind == "login_ce" else 0, log_eps=log_eps, clamp=clamp, weighted=(kind == "ce_weighted"))
                if not hasattr(self, "in_roww") or self.in_roww.numel() < self.T:
                    self.in_roww = torch.ones(self.T, device=self.dev, dtype=torch.float32)
                    self.roww_c = torch.ones(self.T, device=self.dev, dtype=torch.float32)
            return
        if kind not in self.SAMPLED_KINDS:
            raise NotImplementedError(f"Not supported loss_type {kind!r}")
        mode = {"shared": 0, "perpos": 1, "perseq": 2}[neg_shape]
        rows = {0: 1, 1: self.T, 2: self.B}[mode]
        ws_bytes = self.lib.rp_sampled_head_workspace(self.T, self._dp(), n_neg, mode)
        self.sampled = dict(kind=self.SAMPLED_KINDS[kind], n_neg=n_neg, mode=mode, ignore_index=ignore_index, log_eps=log_eps,
                            clamp=clamp, neg=torch.zeros(rows, n_neg, device=self.dev, dtype=torch.int64),
                            ws=torch.zeros(ws_bytes, device=self.dev, dtype=torch.uint8), ws_bytes=ws_bytes)

    def set_row_weights(self, weights):
        """Stage the sample weights of the current batch ([B, L] float, one per position; only valid targets are read)."""
        n = weights.numel()
        self.in_roww[:n].copy_(weights.reshape(-1).to(torch.float32), non_blocking=True)

    def set_negatives(self, negative_labels):
        """Stage the negatives of the current batch ([N] | [B, N] | [B, L, N] int64, device copy)."""
        sp = self.sampled
        if sp is None:
            raise RuntimeError("set_loss(<sampled kind>, ...) first")
        neg = negative_labels.reshape(-1, sp["n_neg"])
        if neg.shape[0] > sp["neg"].shape[0]:
            raise ValueError(f"negative_labels {tuple(negative_labels.shape)} do not fit the configured shape")
        sp["neg"][: neg.shape[0]].copy_(neg, non_blocking=True)

    def _sampled_desc(self):
        sp, cfg = self.sampled, self.cfg
        sd = SampledDesc()
        sd.hc, sd.table = self.hc.data_ptr(), self.params16["item_emb"].data_ptr()
        sd.labels, sd.valid_idx, sd.negatives = self.labels_c.data_ptr(), self.valid_idx.data_ptr(), sp["neg"].data_ptr()
        sd.n_valid = self.n_valid.data_ptr()
        sd.capacity, sd.n_items, sd.d, sd.n_neg, sd.neg_mode, sd.seq_len = self.T, cfg.n_items, self._dp(), sp["n_neg"], sp["mode"], self.L
        sd.kind, sd.ignore_index, sd.vocab_size = sp["kind"], sp["ignore_index"], cfg.n_items
        sd.log_eps, sd.clamp = sp["log_eps"], sp["clamp"]
        sd.loss_out = self.ce.loss.data_ptr()
        sd.workspace, sd.workspace_bytes = sp["ws"].data_ptr(), sp["ws_bytes"]
        return sd

    def _prepare(self, with_targets: bool):
        cfg = self.cfg
        check(self.lib.rp_prepare_batch(self.in_ids.data_ptr(), self.in_pad.data_ptr(),
                                        self.in_labels.data_ptr() if with_targets else None,
                                        self.in_tmask.data_ptr() if with_targets else None, self.T, cfg.pad_id, cfg.n_items,
                                        self.ids32.data_ptr(), self.valid_idx.data_ptr(), self.labels_c.data_ptr(),
                                        self.n_valid.data_ptr(), self.prep_scratch.data_ptr(), self._stream()), "rp_prepare_batch")

    def _body_forward(self, training: bool, last_only: bool = False):
        """``last_only`` (predict): the final block is evaluated for the LAST position of every sequence only - LN1, the Q
        projection, one-query attention, out-projection, LN2 and the FFN run on [B, d] rows; only the K/V projection of
        that block still covers all tokens.  Result rows land in ``self.last_rows`` (bf16 [B, d])."""
        cfg, T, d, L = self.cfg, self.T, self.cfg.dp, self.L
        hdv, att_scale = cfg.hd_valid, 1.0 / math.sqrt(cfg.head_dim)
        p16, prm = self.params16, self.params
        legacy = cfg.variant == "legacy"
        drop = cfg.dropout if training else 0.0
        pad = self.in_pad
        pos0 = 0 if legacy else cfg.max_len - L
        check(self.lib.rp_embed_fwd(p16["item_emb"].data_ptr(), prm["pos_emb"].data_ptr(), self.ids32.data_ptr(),
                                    pad.data_ptr(), T, L, d, pos0, math.sqrt(cfg.d), int(legacy), drop, self.seed, 0,
                                    self.rng_counter.data_ptr(), self.x[0].data_ptr(), self._stream()), "rp_embed_fwd")
        H, hd = cfg.n_heads, d // cfg.n_heads
        for i in range(cfg.n_blocks):
            a, x = self.act[i], self.x[i]
            w = lambda k: p16[f"b{i}.{k}"]  # noqa: E731
            f = lambda k: prm[f"b{i}.{k}"]  # noqa: E731
            if last_only and i == cfg.n_blocks - 1:
                Bq, lb = self.B, self.last_buf
                in_w, in_b = w("in_w"), f("in_b")
                self._ln_fwd(x, f("ln1_w"), f("ln1_b"), 1e-8, lb["q_in"], self.meanf, self.rstdf, Bq, gather=self.last_idx)
                self._gemm(lb["q_in"], in_w[:d], lb["Q"], Bq, d, d, bias=in_b[:d])
                if self.fused_pre_attn:
                    # [K | V] of ALL tokens through the fused pre-attention kernel in its K | V-only mode (activations read
                    # once, TMA-store epilogue): 227 -> ~120 us per 4096-user call against the weight-stationary GEMM
                    check(self.lib.rp_ln_qkv_fused(x.data_ptr(), None, None, 1e-8, in_w.data_ptr(), in_b.data_ptr(), T, d, None,
                                                   None, a["KV"].data_ptr(), None, None, hdv, self._stream()), "rp_ln_qkv_fused")
                else:
                    self._gemm(x, in_w[d:], a["KV"], T, 2 * d, d, bias=in_b[d:])
                check(self.lib.rp_attn_last(lb["Q"].data_ptr(), a["KV"].data_ptr(), a["KV"].data_ptr(), 2 * d, 2 * d, 0, d,
                                            pad.data_ptr(), Bq, H, L, hd, int(not legacy), lb["O"].data_ptr(), att_scale,
                                            self._stream()), "rp_attn_last")
                if d <= 128 and self.fused_post_attn_eval:
                    # out-projection + residual + LayerNorm + FFN of the B last rows in the same fused pass the full blocks
                    # use (one launch instead of GEMM, LayerNorm, GEMM, GEMM: ~10 us each on [4096, d] rows)
                    check(self.lib.rp_post_attn_fused(lb["O"].data_ptr(), lb["q_in"].data_ptr(), w("out_w").data_ptr(),
                                                      f("out_b").data_ptr(), f("ln2_w").data_ptr(), f("ln2_b").data_ptr(), 1e-8,
                                                      w("w1").data_ptr(), f("b1").data_ptr(), w("w2").data_ptr(), f("b2").data_ptr(),
                                                      self.last_pad.data_ptr() if legacy else None, Bq, d,
                                                      self.last_rows.data_ptr(), hdv, self._stream()), "rp_post_attn_fused")
                    return
                self._gemm(lb["O"], w("out_w"), lb["h"], Bq, d, d, bias=f("out_b"), residual=lb["q_in"])
                self._ln_fwd(lb["h"], f("ln2_w"), f("ln2_b"), 1e-8, lb["y"], self.meanf, self.rstdf, Bq)
                self._gemm(lb["y"], w("w1"), lb["u"], Bq, d, d, bias=f("b1"), act=1)
                self._gemm(lb["u"], w("w2"), self.last_rows, Bq, d, d, bias=f("b2"), residual=lb["y"],
                           rowmask=self.last_pad if legacy else None)
                return
            in_w, in_b = w("in_w"), f("in_b")
            if self.fused_pre_attn:
                check(self.lib.rp_ln_qkv_fused(x.data_ptr(), f("ln1_w").data_ptr(), f("ln1_b").data_ptr(), 1e-8,
                                               in_w.data_ptr(), in_b.data_ptr(), T, d, a["q_in"].data_ptr(), a["Q"].data_ptr(),
                                               a["KV"].data_ptr(), a["mean1"].data_ptr(), a["rstd1"].data_ptr(), hdv,
                                               self._stream()), "rp_ln_qkv_fused")
            else:
                self._ln_fwd(x, f("ln1_w"), f("ln1_b"), 1e-8, a["q_in"], a["mean1"], a["rstd1"], T)
                self._gemm(a["q_in"], in_w[:d], a["Q"], T, d, d, bias=in_b[:d])
                self._gemm(x, in_w[d:], a["KV"], T, 2 * d, d, bias=in_b[d:])
            ad = AttnDesc()
            ad.q, ad.q_rows, ad.q_cols, ad.ldq, ad.q_c0 = a["Q"].data_ptr(), T, d, d, 0
            ad.k, ad.k_rows, ad.k_cols, ad.ldk, ad.k_c0 = a["KV"].data_ptr(), T, 2 * d, 2 * d, 0
            ad.v, ad.v_rows, ad.v_cols, ad.ldv, ad.v_c0 = a["KV"].data_ptr(), T, 2 * d, 2 * d, d
            ad.B, ad.H, ad.L, ad.head_dim = self.B, H, L, hd
            ad.causal, ad.mask_pad_keys = 1, int(not legacy)
            ad.scale = att_scale
            ad.pad_mask = pad.data_ptr()
            ad.out, ad.ldo = a["O"].data_ptr(), d
            if training and self.with_grad:
                ad.p_save = None if self.fused_attn_bwd else a["P"].data_ptr()
                ad.inv_sum, ad.m_save = a["inv_sum"].data_ptr(), a["m2"].data_ptr()
            else:
                ad.p_save, ad.inv_sum, ad.m_save = None, None, None
            ad.drop_p, ad.seed, ad.drop_off, ad.seed_ptr = drop, self.seed, self._site(i, 0) << 40, self.rng_counter.data_ptr()
            check(self.lib.rp_attn_fwd(ctypes.byref(ad), self._stream()), "rp_attn_fwd")
            if not training and d <= 128 and self.fused_post_attn_eval:
                # inference: out-projection + residual + LayerNorm + FFN in one pass over the tokens (csrc/rp_ffn.cu)
                check(self.lib.rp_post_attn_fused(a["O"].data_ptr(), a["q_in"].data_ptr(), w("out_w").data_ptr(),
                                                  f("out_b").data_ptr(), f("ln2_w").data_ptr(), f("ln2_b").data_ptr(), 1e-8,
                                                  w("w1").data_ptr(), f("b1").data_ptr(), w("w2").data_ptr(), f("b2").data_ptr(),
                                                  pad.data_ptr() if legacy else None, T, d, self.x[i + 1].data_ptr(), hdv,
                                                  self._stream()), "rp_post_attn_fused")
                continue
            if training and d <= 128 and self.fused_post_attn_train:
                # training: the same chain in one pass, saving h / y / u and the LayerNorm statistics for the backward
                check(self.lib.rp_post_attn_train(a["O"].data_ptr(), a["q_in"].data_ptr(), w("out_w").data_ptr(),
                                                  f("out_b").data_ptr(), f("ln2_w").data_ptr(), f("ln2_b").data_ptr(), 1e-8,
                                                  w("w1").data_ptr(), f("b1").data_ptr(), w("w2").data_ptr(), f("b2").data_ptr(),
                                                  pad.data_ptr() if legacy else None, T, d, drop, self.seed,
                                                  self._site(i, 1) << 40, self._site(i, 2) << 40, self.rng_counter.data_ptr(),
                                                  a["h"].data_ptr(), a["y"].data_ptr(), a["u"].data_ptr(),
                                                  a["mean2"].data_ptr(), a["rstd2"].data_ptr(), self.x[i + 1].data_ptr(), hdv,
                                                  self._stream()), "rp_post_attn_train")
                continue
            self._gemm(a["O"], w("out_w"), a["h"], T, d, d, bias=f("out_b"), residual=a["q_in"])
            self._ln_fwd(a["h"], f("ln2_w"), f("ln2_b"), 1e-8, a["y"], a["mean2"], a["rstd2"], T)
            if not training and d <= 128 and self.fused_ffn_eval:
                # inference: both FFN GEMMs in one pass, the hidden activation never leaves the SM (csrc/rp_ffn.cu)
                check(self.lib.rp_ffn_fused(a["y"].data_ptr(), w("w1").data_ptr(), f("b1").data_ptr(), w("w2").data_ptr(),
                                            f("b2").data_ptr(), pad.data_ptr() if legacy else None, T, d,
                                            self.x[i + 1].data_ptr(), self._stream()), "rp_ffn_fused")
                continue
            self._gemm(a["y"], w("w1"), a["u"], T, d, d, bias=f("b1"), act=1, drop_p=drop, drop_site=self._site(i, 1))
            self._gemm(a["u"], w("w2"), self.x[i + 1], T, d, d, bias=f("b2"), drop_p=drop, drop_site=self._site(i, 2),
                       residual=a["y"], rowmask=pad if legacy else None)

    def forward_train(self):
        """Loss of the staged batch (device fp32 [2] view: mean CE over the valid targets, 1/n_valid)."""
        cfg, T = self.cfg, self.T
        self._prepare(True)
        self._body_forward(True)
        self._ln_fwd(self.x[-1], self.params["lnf_w"], self.params["lnf_b"], cfg.lnf_eps, self.hc, self.meanf, self.rstdf, T,
                     gather=self.valid_idx, n_rows_dev=self.n_valid)
        if self.sampled is not None:
            check(self.lib.rp_sampled_head_fwd(ctypes.byref(self._sampled_desc()), self._stream()), "rp_sampled_head_fwd")
            return self.ce.loss
        if self.bce is not None:
            from .ops import bce_head_fwd

            self.lib.count += 2
            return bce_head_fwd(self.bce, self.hc, self.params16["item_emb"][: cfg.n_items], self.labels_c, self.n_valid,
                                self.s["dhc"], n_valid_hint=self.n_valid_hint)
        from .ops import ce_head_fwd

        self.lib.count += 2
        row = getattr(self, "ce_row", None)
        roww = None
        if row is not None and row["weighted"]:   # weights of the valid targets in the head's compacted order
            torch.index_select(self.in_roww, 0, self.valid_idx, out=self.roww_c)
            roww = self.roww_c
        return ce_head_fwd(self.ce, self.hc, self.params16["item_emb"][: cfg.n_items], self.labels_c, self.n_valid,
                           d_hc=self.s["dhc"] if self.fused_ce else None, n_valid_hint=self.n_valid_hint, row_weight=roww,
                           loss_kind=row["kind"] if row else 0, log_eps=row["log_eps"] if row else 1e-6,
                           clamp=row["clamp"] if row else 100.0)

    # ------------------------------------------------------------------------------------------------ backward
    def backward(self):
        cfg, T, d, L = self.cfg, self.T, self.cfg.dp, self.L
        hdv, att_scale = cfg.hd_valid, 1.0 / math.sqrt(cfg.head_dim)
        p16, prm, G, s = self.params16, self.params, self.grads, self.s
        legacy = cfg.variant == "legacy"
        drop = cfg.dropout
        ks = 1.0 / (1.0 - drop) if drop > 0 else 1.0
        H, hd, Lp = cfg.n_heads, d // cfg.n_heads, self.Lp
        BH = self.B * H
        st = self._stream
        from .ops import ce_head_bwd

        if self.sampled is not None:
            G["item_emb"].zero_()  # the sampled head accumulates sparse rows (the full-CE head overwrites the dense table)
            check(self.lib.rp_sampled_head_bwd(ctypes.byref(self._sampled_desc()), s["dhc"].data_ptr(), G["item_emb"].data_ptr(),
                                               st()), "rp_sampled_head_bwd")
        elif self.bce is not None:
            from .ops import bce_head_bwd

            bce_head_bwd(self.bce, self.hc, p16["item_emb"][: cfg.n_items], self.labels_c, self.n_valid, G["item_emb"])
            self.lib.count += 2
        else:
            ce_head_bwd(self.ce, self.hc, p16["item_emb"][: cfg.n_items], self.labels_c, self.n_valid, s["dhc"], G["item_emb"],
                        n_valid_hint=self.n_valid_hint)
            self.lib.count += 3
        dx = s["dxa"]
        dx.zero_()
        self._ln_bwd(s["dhc"], self.x[-1], prm["lnf_w"], self.meanf, self.rstdf, dx, G["lnf_w"], G["lnf_b"], T,
                     gather=self.valid_idx, n_rows_dev=self.n_valid)
        other = s["dxb"]
        for i in reversed(range(cfg.n_blocks)):
            a, x = self.act[i], self.x[i]
            w = lambda k: p16[f"b{i}.{k}"]  # noqa: E731
            f = lambda k: prm[f"b{i}.{k}"]  # noqa: E731
            g = lambda k: G[f"b{i}.{k}"]  # noqa: E731
            dz = dx
            if self.fused_post_attn_bwd:
                # one pass: d_t, du, dh (operands of the grouped weight gradients), d_o (into the attention backward), dLN2
                masked = legacy or drop > 0
                check(self.lib.rp_post_attn_bwd(dz.data_ptr(), a["u"].data_ptr(), a["h"].data_ptr(), a["mean2"].data_ptr(),
                                                a["rstd2"].data_ptr(), f("ln2_w").data_ptr(), w("w2").data_ptr(),
                                                w("w1").data_ptr(), w("out_w").data_ptr(),
                                                self.in_pad.data_ptr() if legacy else None, T, d, drop, self.seed,
                                                self._site(i, 2) << 40, self.rng_counter.data_ptr(),
                                                s["d_t"].data_ptr() if masked else None, s["du"].data_ptr(), s["dh"].data_ptr(),
                                                s["d_o"].data_ptr(), g("ln2_w").data_ptr(), g("ln2_b").data_ptr(), hdv, st()),
                      "rp_post_attn_bwd")
                d_t = s["d_t"] if masked else dz
                fw = self.fused_wgrad
                wpairs = [(d_t, a["u"], g("w2"), g("b2")), (s["du"], a["y"], g("w1"), g("b1")), (s["dh"], a["O"], g("out_w"), g("out_b"))]
                bias_grads = [(d_t, g("b2")), (s["du"], g("b1")), (s["dh"], g("out_b"))]
                if not fw:
                    self._wgrad(d_t, a["u"], g("w2"), d, d)
                    self._wgrad(s["du"], a["y"], g("w1"), d, d)
                    self._wgrad(s["dh"], a["O"], g("out_w"), d, d)
            if not self.fused_post_attn_bwd and legacy:  # x_next = (...) * pad   (sasrec/model.py:441)
                check(self.lib.rp_dropout_bwd(dz.data_ptr(), dz.data_ptr(), T, d, self.in_pad.data_ptr(), 0.0, 0, 0, None, st()),
                      "rp_dropout_bwd")
            if not self.fused_post_attn_bwd:
                if drop > 0:
                    check(self.lib.rp_dropout_bwd(dz.data_ptr(), s["d_t"].data_ptr(), T, d, None, drop, self.seed,
                                                  self._site(i, 2) << 40, self.rng_counter.data_ptr(), st()), "rp_dropout_bwd")
                    d_t = s["d_t"]
                else:
                    d_t = dz
                # ---- FFN backward
                fw = self.fused_wgrad
                wpairs = [(d_t, a["u"], g("w2"), g("b2"))]  # (dY, X, dW, db): weight + bias gradients, one grouped launch per block
                if not fw:
                    self._wgrad(d_t, a["u"], g("w2"), d, d)
                bias_grads = [(d_t, g("b2"))]  # column sums of this block, one launch at the end of its backward
                self._gemm(d_t, w("w2"), s["du"], T, d, d, b_mn=True, gate=a["u"], gate_scale=ks)
                wpairs.append((s["du"], a["y"], g("w1"), g("b1")))
                if not fw:
                    self._wgrad(s["du"], a["y"], g("w1"), d, d)
                bias_grads.append((s["du"], g("b1")))
                self._gemm(s["du"], w("w1"), s["dy"], T, d, d, b_mn=True, residual=dz)
                self._ln_bwd(s["dy"], a["h"], f("ln2_w"), a["mean2"], a["rstd2"], s["dh"], g("ln2_w"), g("ln2_b"), T)
                # ---- out projection
                self._gemm(s["dh"], w("out_w"), s["d_o"], T, d, d, b_mn=True)
                wpairs.append((s["dh"], a["O"], g("out_w"), g("out_b")))
                if not fw:
                    self._wgrad(s["dh"], a["O"], g("out_w"), d, d)
                bias_grads.append((s["dh"], g("out_b")))
            # ---- attention backward
            KV, Q = a["KV"], a["Q"]
            if self.fused_attn_bwd:
                bd = AttnBwdDesc()
                bd.q, bd.q_rows, bd.q_cols, bd.ldq, bd.q_c0 = Q.data_ptr(), T, d, d, 0
                bd.k, bd.k_rows, bd.k_cols, bd.ldk, bd.k_c0 = KV.data_ptr(), T, 2 * d, 2 * d, 0
                bd.v, bd.v_rows, bd.v_cols, bd.ldv, bd.v_c0 = KV.data_ptr(), T, 2 * d, 2 * d, d
                bd.d_out, bd.do_rows, bd.do_cols, bd.ld_do = s["d_o"].data_ptr(), T, d, d
                bd.out, bd.ldo = a["O"].data_ptr(), d
                bd.B, bd.H, bd.L, bd.head_dim = self.B, H, L, hd
                bd.causal, bd.mask_pad_keys = 1, int(not legacy)
                bd.scale = att_scale
                bd.pad_mask = self.in_pad.data_ptr()
                bd.m_save, bd.inv_sum = a["m2"].data_ptr(), a["inv_sum"].data_ptr()
                bd.dq, bd.ld_dq, bd.dq_c0 = s["dQ"].data_ptr(), d, 0
                bd.dk, bd.ld_dk, bd.dk_c0 = s["dKV"].data_ptr(), 2 * d, 0
                bd.dv, bd.ld_dv, bd.dv_c0 = s["dKV"].data_ptr(), 2 * d, d
                bd.drop_p, bd.seed, bd.drop_off, bd.seed_ptr = drop, self.seed, self._site(i, 0) << 40, self.rng_counter.data_ptr()
                check(self.lib.rp_attn_bwd(ctypes.byref(bd), st()), "rp_attn_bwd")
            else:
                P, dpd = a["P"].view(BH * Lp, Lp), s["dpd"].view(BH * Lp, Lp)
                # dPd = dO . V^T
                self._gemm(s["d_o"], KV, dpd, L, L, hd, batch=BH, inner=H, a_off=(0, L, 0, 0, 0, hd), b_off=(0, L, 0, d, 0, hd),
                           c_geom=(Lp, 0, H * Lp * Lp, Lp * Lp))
                check(self.lib.rp_attn_softmax_bwd(P.data_ptr(), dpd.data_ptr(), a["inv_sum"].data_ptr(), BH, L,
                                                   att_scale, drop, self.seed, self._site(i, 0) << 40,
                                                   self.rng_counter.data_ptr(), st()), "rp_attn_softmax_bwd")
                # dQ = dS . K      (A = dS [BH*Lp, Lp] K-major, B = K MN-major)
                self._gemm(dpd, KV, s["dQ"], L, hd, L, b_mn=True, batch=BH, inner=H, a_off=(0, H * Lp, Lp, 0, 0, 0),
                           b_off=(0, L, 0, 0, 0, hd), c_geom=(d, 0, L * d, hd))
                # dK = dS^T . Q    (A = dS MN-major, B = Q MN-major)
                self._gemm(dpd, Q, s["dKV"], L, hd, L, a_mn=True, b_mn=True, batch=BH, inner=H, a_off=(0, H * Lp, Lp, 0, 0, 0),
                           b_off=(0, L, 0, 0, 0, hd), c_geom=(2 * d, 0, L * 2 * d, hd))
                # dV = Pd^T . dO
                self._gemm(P, s["d_o"], s["dKV"], L, hd, L, a_mn=True, b_mn=True, batch=BH, inner=H,
                           a_off=(0, H * Lp, Lp, 0, 0, 0), b_off=(0, L, 0, 0, 0, hd), c_geom=(2 * d, d, L * 2 * d, hd))
            # ---- projections
            in_w = w("in_w")
            if self.fused_pre_attn:
                check(self.lib.rp_pre_attn_bwd(s["dQ"].data_ptr(), s["dKV"].data_ptr(), s["dh"].data_ptr(), x.data_ptr(),
                                               a["mean1"].data_ptr(), a["rstd1"].data_ptr(), f("ln1_w").data_ptr(),
                                               in_w.data_ptr(), T, d, other.data_ptr(), g("ln1_w").data_ptr(),
                                               g("ln1_b").data_ptr(), hdv, st()), "rp_pre_attn_bwd")
            else:
                self._gemm(s["dQ"], in_w[:d], s["dq_in"], T, d, d, b_mn=True, residual=s["dh"])
                self._ln_bwd(s["dq_in"], x, f("ln1_w"), a["mean1"], a["rstd1"], s["tmp"], g("ln1_w"), g("ln1_b"), T)
                self._gemm(s["dKV"], in_w[d:], other, T, d, 2 * d, b_mn=True, residual=s["tmp"])
            wpairs.append((s["dQ"], a["q_in"], g("in_w")[:d], g("in_b")[:d]))
            if not fw:
                self._wgrad(s["dQ"], a["q_in"], g("in_w")[:d], d, d)
            bias_grads.append((s["dQ"], g("in_b")[:d]))
            wpairs.append((s["dKV"], x, g("in_w")[d:], g("in_b")[d:]))
            if fw:
                self._wgrad_group(wpairs)
            else:
                self._wgrad(s["dKV"], x, g("in_w")[d:], 2 * d, d)
                bias_grads.append((s["dKV"], g("in_b")[d:]))
                self._colsum_multi(bias_grads)
            dx, other = other, dx
        pos0 = 0 if legacy else cfg.max_len - L
        check(self.lib.rp_embed_bwd(dx.data_ptr(), self.ids32.data_ptr(), self.in_pad.data_ptr(), self.B, L, d, cfg.pad_id,
                                    pos0, math.sqrt(cfg.d), int(legacy), drop, self.seed, 0, self.rng_counter.data_ptr(),
                                    G["item_emb"].data_ptr(), G["pos_emb"].data_ptr(), st()), "rp_embed_bwd")

    def optimizer_step(self, grad_scale: float = 1.0, beta1=0.9, beta2=0.98, eps=1e-8):
        """torch.optim.Adam(lr, betas=(0.9, 0.98)) (optimizer_factory.py:56-63,79-80) on the flat buffers; also refreshes
        the bf16 shadow weights and zeroes the gradients."""
        check(self.lib.rp_adam_step(self.p32.data_ptr(), self.g32.data_ptr(), self.adam_m.data_ptr(), self.adam_v.data_ptr(),
                                    self.p16.data_ptr(), self.n_flat, self.lr.data_ptr(), self.step_count.data_ptr(), beta1,
                                    beta2, eps, grad_scale, None, 1, self._stream()), "rp_adam_step")

    def tick_rng(self):
        check(self.lib.rp_counter_add(self.rng_counter.data_ptr(), 0x9E3779B97F4A7C15 & 0xFFFFFFFFFFFF, self._stream()),
              "rp_counter_add")

    def train_step(self, all_reduce=None, betas=(0.9, 0.98)):
        """forward + backward + (optional gradient all-reduce callback on the flat fp32 gradient) + Adam."""
        self.tick_rng()
        loss = self.forward_train()
        self.backward()
        scale = 1.0
        if all_reduce is not None:
            scale = all_reduce(self.g32)
        self.optimizer_step(grad_scale=scale, beta1=betas[0], beta2=betas[1])
        return loss

    # ------------------------------------------------------------------------------------------------ inference
    def forward_last_hidden(self):
        """Eval-mode body (no dropout) -> final LayerNorm of the LAST position of every sequence -> self.hq bf16 [B, d]
        (SasRec.forward_inference, nn/sequential/sasrec/model.py:292-307 ; legacy get_query_embeddings, model.py:157)."""
        self._prepare(False)
        if self.cfg.variant == "legacy":
            self.last_pad.copy_(self.in_pad.view(self.B, self.L)[:, -1])
        self._body_forward(False, last_only=True)
        self._ln_fwd(self.last_rows, self.params["lnf_w"], self.params["lnf_b"], self.cfg.lnf_eps, self.hq, self.meanf, self.rstdf,
                     self.B)
        return self.hq

    def forward_hidden_all(self):
        """Eval-mode hidden states of every position, bf16 [T, d] (for parity tests / HiddenStatesCallback)."""
        self._prepare(False)
        self._body_forward(False)
        out = torch.empty(self.T, self.cfg.dp, device=self.dev, dtype=torch.bfloat16)
        self._ln_fwd(self.x[-1], self.params["lnf_w"], self.params["lnf_b"], self.cfg.lnf_eps, out, self.meanf, self.rstdf, self.T)
        return out
