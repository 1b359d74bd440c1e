"""BERT4Rec on the B200 engine (replay/models/nn/sequential/bert4rec/model.py:10-527, lightning.py:332-351):
pre-LN transformer blocks with exact-erf GELU 4d FFN, a single <MASK> embedding, key-padding-only attention, no final
LayerNorm, and an untied ``Linear(d, |I|)`` head with bias (default) or the tied item table + ``out_bias``.  The loss is the
full-catalog CE over the positions that are real AND masked.  Same kernels as SASRec (rp_gemm / rp_attn_fwd / fused CE head),
driven by a different block program."""
from __future__ import annotations

import ctypes
import math
from dataclasses import dataclass

import torch

from ._lib import AttnBwdDesc, AttnDesc, check
from .engine import SasRecEngine, _CountingLib, _ru
from ._lib import lib


@dataclass
class BertConfig:
    n_items: int
    d: int
    n_heads: int
    n_blocks: int
    max_len: int
    dropout: float = 0.0
    tying: bool = False
    pad_id: int = 0  # TensorFeatureInfo.padding_value: a VALID row for BERT4Rec (the table has |I| rows, no pad row)
    variant: str = "bert4rec"
    lnf_eps: float = 1e-5

    def __post_init__(self):
        if self.d not in (64, 128, 256):
            raise ValueError("hidden size must be one of 64/128/256 for BERT4Rec (CE-backward tile constraint)")
        if self.d % self.n_heads or self.d // self.n_heads not in (64, 128):
            raise ValueError("head_dim must be 64 or 128 (tcgen05 128B-swizzle tile constraint)")


    # the shared engine code asks every config for its feature-slot geometry; BERT4Rec has no padded layout (head_dim 64 / 128)
    @property
    def head_dim(self) -> int:
        return self.d // self.n_heads

    @property
    def head_slot(self) -> int:
        return self.head_dim

    @property
    def dp(self) -> int:
        return self.d

    @property
    def hd_valid(self) -> int:
        return 0


_BERT_BLOCK = ("ln1_w", "ln1_b", "in_w", "in_b", "out_w", "out_b", "ln2_w", "ln2_b", "w1", "b1", "w2", "b2")


class Bert4RecEngine(SasRecEngine):
    def __init__(self, cfg: BertConfig, max_batch: int, seq_len: int, device="cuda", seed: int = 0, with_grad: bool = True):
        self.cfg = cfg
        self.dev = torch.device(device)
        self.B, self.L = max_batch, seq_len
        if seq_len != cfg.max_len:
            raise ValueError("BERT4Rec needs seq_len == max_len (bert4rec/model.py:276)")
        if seq_len > 512 or (seq_len > 256 and cfg.d // cfg.n_heads != 64):
            raise ValueError("attention kernels support seq_len <= 256 (head_dim 128) / <= 512 (head_dim 64)")
        self.T = max_batch * seq_len
        self.Lp = _ru(seq_len, 64)
        self.with_grad = with_grad
        self.lib = _CountingLib(lib())
        d, I = cfg.d, cfg.n_items
        self.I128 = _ru(I, 128)
        shapes = [("item_emb", (I, d)), ("mask_emb", (1, d)), ("pos_emb", (cfg.max_len, d))]
        for i in range(cfg.n_blocks):
            shapes += [(f"b{i}.ln1_w", (d,)), (f"b{i}.ln1_b", (d,)), (f"b{i}.in_w", (3 * d, d)), (f"b{i}.in_b", (3 * d,)),
                       (f"b{i}.out_w", (d, d)), (f"b{i}.out_b", (d,)), (f"b{i}.ln2_w", (d,)), (f"b{i}.ln2_b", (d,)),
                       (f"b{i}.w1", (4 * d, d)), (f"b{i}.b1", (4 * d,)), (f"b{i}.w2", (d, 4 * d)), (f"b{i}.b2", (d,))]
        if not cfg.tying:
            shapes += [("head_w", (I, d))]
        shapes += [("head_b", (self.I128,))]  # padded: the kernels read the bias in 128-entry tiles
        self.layout, off = {}, 0
        for name, shp in shapes:
            self.layout[name] = (off, shp)
            off = _ru(off + math.prod(shp), 64)
        self.n_flat = off
        f32 = dict(device=self.dev, dtype=torch.float32)
        self.p32 = torch.zeros(off, **f32)
        self.p16 = torch.zeros(off, device=self.dev, dtype=torch.bfloat16)
        self.params = {k: self.p32[o:o + math.prod(s)].view(s) for k, (o, s) in self.layout.items()}
        self.params16 = {k: self.p16[o:o + math.prod(s)].view(s) for k, (o, s) in self.layout.items()}
        if with_grad:
            self._alloc_grad_state()
        self.sampled, self._loss_args, self.bce = None, None, None
        self.rng_counter = torch.zeros(1, device=self.dev, dtype=torch.int64)
        self.seed = seed & 0xFFFFFFFFFFFF
        self.fused_attn_bwd = (cfg.d // cfg.n_heads) == 64 and seq_len <= 256
        self.fused_ce = True
        self.n_valid_hint = 0
        self._alloc_bert_workspace()
        self.init_parameters(seed)

    # ------------------------------------------------------------------------------------------------ parameters
    def init_parameters(self, seed: int = 0):
        """xavier_normal_ on >=2-D tensors (bert4rec/model.py:167-170), LN (1,0), Linear biases U(+-1/sqrt(fan_in))."""
        g = torch.Generator(device="cpu").manual_seed(seed)
        with torch.no_grad():
            for name, (o, shp) in self.layout.items():
                p = self.params[name]
                if len(shp) == 2:
                    p.copy_((torch.randn(shp, generator=g) * math.sqrt(2.0 / (shp[0] + shp[1]))).to(self.dev))
                elif name.endswith(("ln1_w", "ln2_w")):
                    p.fill_(1.0)
                elif name.endswith((".b1", ".b2")):
                    fan_in = self.cfg.d if name.endswith(".b1") else 4 * self.cfg.d
                    p.copy_(((torch.rand(shp, generator=g) * 2 - 1) / math.sqrt(fan_in)).to(self.dev))
                else:
                    p.zero_()
        self.refresh_shadow()

    def load_canonical(self, P: dict):
        """oracle/bert4rec.py canonical dict -> engine."""
        f = lambda t: t.to(self.dev, torch.float32)  # noqa: E731
        with torch.no_grad():
            self.params["item_emb"].copy_(f(P["item_emb"]))
            self.params["mask_emb"].copy_(f(P["mask_emb"]))
            self.params["pos_emb"].copy_(f(P["pos_emb"]))
            for i, blk in enumerate(P["blocks"]):
                for k in _BERT_BLOCK:
                    self.params[f"b{i}.{k}"].copy_(f(blk[k]))
            if not self.cfg.tying:
                self.params["head_w"].copy_(f(P["head_w"]))
            self.params["head_b"].zero_()
            self.params["head_b"][: self.cfg.n_items].copy_(f(P["head_b"]))
        self.refresh_shadow()

    def export_canonical(self, source=None) -> dict:
        src = self.params if source is None else source
        c = lambda t: t.detach().cpu().clone()  # noqa: E731
        P = {"item_emb": c(src["item_emb"]), "mask_emb": c(src["mask_emb"]), "pos_emb": c(src["pos_emb"]), "blocks": []}
        for i in range(self.cfg.n_blocks):
            P["blocks"].append({k: c(src[f"b{i}.{k}"]) for k in _BERT_BLOCK})
        if not self.cfg.tying:
            P["head_w"] = c(src["head_w"])
        P["head_b"] = c(src["head_b"][: self.cfg.n_items])
        return P

    # ------------------------------------------------------------------------------------------------ workspace
    def _check_geometry(self, seq_len: int):
        if seq_len != self.cfg.max_len:
            raise ValueError("BERT4Rec needs seq_len == max_len (bert4rec/model.py:276)")
        if seq_len > 512 or (seq_len > 256 and self.cfg.d // self.cfg.n_heads != 64):
            raise ValueError("attention kernels support seq_len <= 256 (head_dim 128) / <= 512 (head_dim 64)")

    def _realloc_workspace(self):
        self._alloc_bert_workspace()

    def _alloc_bert_workspace(self):
        cfg, T, d, dev = self.cfg, self.T, self.cfg.d, self.dev
        bf = dict(device=dev, dtype=torch.bfloat16)
        f32 = dict(device=dev, dtype=torch.float32)
        i32 = dict(device=dev, dtype=torch.int32)
        BH = self.B * cfg.n_heads
        self.ids32 = torch.zeros(T, **i32)
        self.in_ids = torch.zeros(T, device=dev, dtype=torch.int64)
        self.in_pad = torch.zeros(T, device=dev, dtype=torch.bool)
        self.in_tok = torch.zeros(T, device=dev, dtype=torch.bool)
        self.in_labels = torch.zeros(T, device=dev, dtype=torch.int64)
        self.in_tmask = torch.zeros(T, device=dev, dtype=torch.bool)
        self.valid_idx = torch.zeros(T, **i32)
        self.labels_c = torch.zeros(T, **i32)
        self.n_valid = torch.zeros(1, **i32)
        self.prep_scratch = torch.zeros((T + 1023) // 1024 + 1, **i32)
        self.x = [torch.zeros(T, d, **bf) for _ in range(cfg.n_blocks + 1)]
        self.act = []
        for _ in range(cfg.n_blocks):
            a = {k: torch.zeros(T, d, **bf) for k in ("xn", "O", "y", "yn")}
            a["QKV"] = torch.zeros(T, 3 * d, **bf)
            a["pre"] = torch.zeros(T, 4 * d, **bf)
            a["u"] = torch.zeros(T, 4 * d, **bf)
            for k in ("mean1", "rstd1", "mean2", "rstd2"):
                a[k] = torch.zeros(T, **f32)
            if self.with_grad:
                if not self.fused_attn_bwd:
                    a["P"] = torch.zeros(BH, self.Lp, self.Lp, **bf)
                a["inv_sum"] = torch.zeros(BH, self.Lp, **f32)
                a["m2"] = torch.zeros(BH, self.Lp, **f32)
            self.act.append(a)
        self.hc = torch.zeros(T, d, **bf)
        self.hq = torch.zeros(self.B, d, **bf)
        self.last_idx = (torch.arange(self.B, device=dev, dtype=torch.int32) * self.L + (self.L - 1)).contiguous()
        if self.with_grad:
            from .ops import CEHeadState

            self.ce = CEHeadState(T, cfg.n_items, d, dev)
            self.s = {k: torch.zeros(T, d, **bf) for k in ("dhc", "dxa", "dxb", "dz", "d_t", "dyn", "dy", "d_ao", "d_o", "dxn")}
            self.s["du"] = torch.zeros(T, 4 * d, **bf)
            self.s["dQKV"] = torch.zeros(T, 3 * d, **bf)
            if not self.fused_attn_bwd:
                self.s["dpd"] = torch.zeros(BH, self.Lp, self.Lp, **bf)
            self.wg_ws = torch.zeros(148 * 4 * d * d, **f32)  # split-K partials of the weight-gradient GEMMs

    # ------------------------------------------------------------------------------------------------ batch
    def set_batch(self, ids, pad_mask, token_mask, labels=None):
        """[B, L] int64 ids, bool pad_mask (True = real), bool token_mask (False = <MASK>; pads are False too)."""
        B, L = ids.shape
        if L != self.L or B > self.B:
            raise ValueError(f"batch shape {tuple(ids.shape)} does not fit engine ({self.B}, {self.L})")
        n = B * L
        self.in_ids[:n].copy_(ids.reshape(-1), non_blocking=True)
        self.in_pad[:n].copy_(pad_mask.reshape(-1), non_blocking=True)
        self.in_tok[:n].copy_(token_mask.reshape(-1), non_blocking=True)
        if n < self.T:
            self.in_pad[n:].zero_()
            self.in_tok[n:].zero_()
        if labels is not None:
            self.in_labels[:n].copy_(labels.reshape(-1), non_blocking=True)
        # loss positions: real AND masked  (bert4rec/lightning.py:344-348)
        torch.logical_and(self.in_pad, torch.logical_not(self.in_tok), out=self.in_tmask)

    def _prepare(self, with_targets: bool):
        cfg = self.cfg
        check(self.lib.rp_prepare_batch(self.in_ids.data_ptr(), self.in_pad.data_ptr(),
                                        self.in_labels.data_ptr() if with_targets else None,
                                        self.in_tmask.data_ptr() if with_targets else None, self.T, cfg.pad_id, cfg.n_items,
                                        self.ids32.data_ptr(), self.valid_idx.data_ptr(), self.labels_c.data_ptr(),
                                        self.n_valid.data_ptr(), self.prep_scratch.data_ptr(), self._stream()), "rp_prepare_batch")

    def _bsite(self, blk, k):
        return 1 + blk * 8 + k

    # ------------------------------------------------------------------------------------------------ forward
    def _body_forward(self, training: bool):
        cfg, T, d, L = self.cfg, self.T, self.cfg.d, self.L
        p16, prm = self.params16, self.params
        drop = cfg.dropout if training else 0.0
        rng = self.rng_counter.data_ptr()
        check(self.lib.rp_bert_embed_fwd(p16["item_emb"].data_ptr(), p16["mask_emb"].data_ptr(), prm["pos_emb"].data_ptr(),
                                         self.ids32.data_ptr(), self.in_tok.data_ptr(), T, L, d, drop, self.seed, 0, rng,
                                         self.x[0].data_ptr(), self._stream()), "rp_bert_embed_fwd")
        H, hd = cfg.n_heads, d // cfg.n_heads
        for i in range(cfg.n_blocks):
            a, x = self.act[i], self.x[i]
            w = lambda k: p16[f"b{i}.{k}"]  # noqa: E731
            f = lambda k: prm[f"b{i}.{k}"]  # noqa: E731
            self._ln_fwd(x, f("ln1_w"), f("ln1_b"), 1e-5, a["xn"], a["mean1"], a["rstd1"], T)
            self._gemm(a["xn"], w("in_w"), a["QKV"], T, 3 * d, d, bias=f("in_b"))
            ad = AttnDesc()
            for nm, c0 in (("q", 0), ("k", d), ("v", 2 * d)):
                setattr(ad, nm, a["QKV"].data_ptr())
                setattr(ad, nm + "_rows", T); setattr(ad, nm + "_cols", 3 * d); setattr(ad, "ld" + nm, 3 * d)
                setattr(ad, nm + "_c0", c0)
            ad.B, ad.H, ad.L, ad.head_dim = self.B, H, L, hd
            ad.causal, ad.mask_pad_keys = 0, 1
            ad.pad_mask = self.in_pad.data_ptr()
            ad.out, ad.ldo = a["O"].data_ptr(), d
            if training and self.with_grad:
                ad.p_save = None if self.fused_attn_bwd else a["P"].data_ptr()
                ad.inv_sum, ad.m_save = a["inv_sum"].data_ptr(), a["m2"].data_ptr()
            else:
                ad.p_save, ad.inv_sum, ad.m_save = None, None, None
            ad.drop_p, ad.seed, ad.drop_off, ad.seed_ptr = drop, self.seed, self._bsite(i, 0) << 40, rng
            check(self.lib.rp_attn_fwd(ctypes.byref(ad), self._stream()), "rp_attn_fwd")
            # y = x + drop(O Wo^T + bo)
            self._gemm(a["O"], w("out_w"), a["y"], T, d, d, bias=f("out_b"), drop_p=drop, drop_site=self._bsite(i, 1), residual=x)
            self._ln_fwd(a["y"], f("ln2_w"), f("ln2_b"), 1e-5, a["yn"], a["mean2"], a["rstd2"], T)
            # u = drop(gelu(yn W1^T + b1)) ; the pre-activation is kept for gelu'
            self._gemm(a["yn"], w("w1"), a["u"], T, 4 * d, d, bias=f("b1"), act=2, drop_p=drop, drop_site=self._bsite(i, 2),
                       C2=a["pre"] if (training and self.with_grad) else None)
            # x_next = drop( y + drop(u W2^T + b2) )
            self._gemm(a["u"], w("w2"), self.x[i + 1], T, d, 4 * d, bias=f("b2"), drop_p=drop, drop_site=self._bsite(i, 3),
                       residual=a["y"], post_drop_p=drop, post_drop_site=self._bsite(i, 4))

    def _head(self):
        cfg = self.cfg
        W16 = self.params16["item_emb"] if cfg.tying else self.params16["head_w"]
        return W16, self.params["head_b"]

    def set_loss(self, kind: str = "ce", **kw):
        """``"ce"`` (default) or ``"bce"``: full-catalog CE / pointwise BCE (bert4rec/lightning.py:273-305) over the biased
        (or tied + out_bias) head.  The sampled losses of the reference's BERT4Rec are not built."""
        if kind not in ("ce", "bce"):
            raise NotImplementedError(f"Not supported loss_type {kind!r}")
        self._loss_args = (kind, kw)
        self.bce = None
        if kind == "bce":
            if self.cfg.d not in (64, 128, 256):
                raise NotImplementedError(f"the full-catalog BCE head supports hidden sizes 64, 128 and 256 (got {self.cfg.d})")
            if self.with_grad:
                from .ops import BCEHeadState

                self.bce = BCEHeadState(self.T, self.cfg.n_items, self.cfg.d, self.dev, loss=self.ce.loss)

    def forward_train(self):
        from .ops import bce_head_fwd, ce_head_fwd

        self._prepare(True)
        self._body_forward(True)
        check(self.lib.rp_gather_rows(self.x[-1].data_ptr(), self.valid_idx.data_ptr(), self.T, self.n_valid.data_ptr(),
                                      self.cfg.d, self.hc.data_ptr(), 0, self._stream()), "rp_gather_rows")
        W16, bias = self._head()
        self.lib.count += 2
        if self.bce is not None:
            return bce_head_fwd(self.bce, self.hc, W16, self.labels_c, self.n_valid, self.s["dhc"], bias=bias,
                                n_valid_hint=self.n_valid_hint)
        return ce_head_fwd(self.ce, self.hc, W16, self.labels_c, self.n_valid, bias=bias,
                           d_hc=self.s["dhc"] if self.fused_ce else None, n_valid_hint=self.n_valid_hint)

    # ------------------------------------------------------------------------------------------------ backward
    def backward(self):
        from .ops import bce_head_bwd, ce_head_bwd

        cfg, T, d, L = self.cfg, self.T, self.cfg.d, self.L
        p16, prm, G, s = self.params16, self.params, self.grads, self.s
        drop = cfg.dropout
        ks = 1.0 / (1.0 - drop) if drop > 0 else 1.0
        H, hd, Lp = cfg.n_heads, d // cfg.n_heads, self.Lp
        BH = self.B * H
        st, rng = self._stream, self.rng_counter.data_ptr()
        W16, bias = self._head()
        dW = G["item_emb"] if cfg.tying else G["head_w"]
        if self.bce is not None:
            bce_head_bwd(self.bce, self.hc, W16, self.labels_c, self.n_valid, dW, bias=bias, d_bias=G["head_b"])
            self.lib.count += 2
        else:
            ce_head_bwd(self.ce, self.hc, W16, self.labels_c, self.n_valid, s["dhc"], dW, bias=bias, d_bias=G["head_b"])
            self.lib.count += 3
        dx = s["dxa"]
        dx.zero_()
        check(self.lib.rp_gather_rows(s["dhc"].data_ptr(), self.valid_idx.data_ptr(), T, self.n_valid.data_ptr(), d,
                                      dx.data_ptr(), 1, st()), "rp_gather_rows")
        other = s["dxb"]

        def dbwd(src, dst, site):
            if drop > 0:
                check(self.lib.rp_dropout_bwd(src.data_ptr(), dst.data_ptr(), T, d, None, drop, self.seed, site << 40, rng, st()),
                      "rp_dropout_bwd")
                return dst
            return src

        for i in reversed(range(cfg.n_blocks)):
            a, x = self.act[i], self.x[i]
            w = lambda k: p16[f"b{i}.{k}"]  # noqa: E731
            f = lambda k: prm[f"b{i}.{k}"]  # noqa: E731
            g = lambda k: G[f"b{i}.{k}"]  # noqa: E731
            dz = dbwd(dx, s["dz"], self._bsite(i, 4))          # x_next = drop(z)
            d_t = dbwd(dz, s["d_t"], self._bsite(i, 3))        # z = y + drop(u W2^T + b2)
            self._wgrad(d_t, a["u"], g("w2"), d, 4 * d)
            self._colsum(d_t, g("b2"))
            # du_pre = (d_t W2) * dropmask/keep * gelu'(pre)
            self._gemm(d_t, w("w2"), s["du"], T, 4 * d, d, b_mn=True, drop_p=drop, drop_site=self._bsite(i, 2), gate=a["pre"],
                       gate_mode=1, gate_scale=1.0)
            self._wgrad(s["du"], a["yn"], g("w1"), 4 * d, d)
            self._colsum(s["du"], g("b1"))
            self._gemm(s["du"], w("w1"), s["dyn"], T, d, 4 * d, b_mn=True)
            # dy = dz (residual) + LN2'(dyn)
            self._ln_bwd(s["dyn"], a["y"], f("ln2_w"), a["mean2"], a["rstd2"], s["dy"], g("ln2_w"), g("ln2_b"), T, add_to=dz)
            d_ao = dbwd(s["dy"], s["d_ao"], self._bsite(i, 1))  # y = x + drop(O Wo^T + bo)
            self._wgrad(d_ao, a["O"], g("out_w"), d, d)
            self._colsum(d_ao, g("out_b"))
            self._gemm(d_ao, w("out_w"), s["d_o"], T, d, d, b_mn=True)
            # ---- attention backward, Q/K/V are column slices of QKV
            QKV, dq = a["QKV"], s["dQKV"]
            if self.fused_attn_bwd:
                bd = AttnBwdDesc()
                for nm, c0 in (("q", 0), ("k", d), ("v", 2 * d)):
                    setattr(bd, nm, QKV.data_ptr())
                    setattr(bd, nm + "_rows", T); setattr(bd, nm + "_cols", 3 * d); setattr(bd, "ld" + nm, 3 * d)
                    setattr(bd, nm + "_c0", c0)
                bd.d_out, bd.do_rows, bd.do_cols, bd.ld_do = s["d_o"].data_ptr(), T, d, d
                bd.out, bd.ldo = a["O"].data_ptr(), d
                bd.B, bd.H, bd.L, bd.head_dim = self.B, H, L, hd
                bd.causal, bd.mask_pad_keys = 0, 1
                bd.pad_mask = self.in_pad.data_ptr()
                bd.m_save, bd.inv_sum = a["m2"].data_ptr(), a["inv_sum"].data_ptr()
                bd.dq, bd.ld_dq, bd.dq_c0 = dq.data_ptr(), 3 * d, 0
                bd.dk, bd.ld_dk, bd.dk_c0 = dq.data_ptr(), 3 * d, d
                bd.dv, bd.ld_dv, bd.dv_c0 = dq.data_ptr(), 3 * d, 2 * d
                bd.drop_p, bd.seed, bd.drop_off, bd.seed_ptr = drop, self.seed, self._bsite(i, 0) << 40, rng
                check(self.lib.rp_attn_bwd(ctypes.byref(bd), st()), "rp_attn_bwd")
            else:
                P, dpd = a["P"].view(BH * Lp, Lp), s["dpd"].view(BH * Lp, Lp)
                self._gemm(s["d_o"], QKV, dpd, L, L, hd, batch=BH, inner=H, a_off=(0, L, 0, 0, 0, hd), b_off=(0, L, 0, 2 * d, 0, hd),
                           c_geom=(Lp, 0, H * Lp * Lp, Lp * Lp))
                check(self.lib.rp_attn_softmax_bwd(P.data_ptr(), dpd.data_ptr(), a["inv_sum"].data_ptr(), BH, L,
                                                   1.0 / math.sqrt(hd), drop, self.seed, self._bsite(i, 0) << 40, rng, st()),
                      "rp_attn_softmax_bwd")
                self._gemm(dpd, QKV, dq, L, hd, L, b_mn=True, batch=BH, inner=H, a_off=(0, H * Lp, Lp, 0, 0, 0),
                           b_off=(0, L, 0, d, 0, hd), c_geom=(3 * d, 0, L * 3 * d, hd))                      # dQ = dS . K
                self._gemm(dpd, QKV, dq, L, hd, L, a_mn=True, b_mn=True, batch=BH, inner=H, a_off=(0, H * Lp, Lp, 0, 0, 0),
                           b_off=(0, L, 0, 0, 0, hd), c_geom=(3 * d, d, L * 3 * d, hd))                      # dK = dS^T . Q
                self._gemm(P, s["d_o"], dq, L, hd, L, a_mn=True, b_mn=True, batch=BH, inner=H, a_off=(0, H * Lp, Lp, 0, 0, 0),
                           b_off=(0, L, 0, 0, 0, hd), c_geom=(3 * d, 2 * d, L * 3 * d, hd))                  # dV = Pd^T . dO
            self._gemm(dq, w("in_w"), s["dxn"], T, d, 3 * d, b_mn=True)
            self._wgrad(dq, a["xn"], g("in_w"), 3 * d, d)
            self._colsum(dq, g("in_b"))
            # dx = dy (residual) + LN1'(dxn)
            self._ln_bwd(s["dxn"], x, f("ln1_w"), a["mean1"], a["rstd1"], other, g("ln1_w"), g("ln1_b"), T, add_to=s["dy"])
            dx, other = other, dx
        check(self.lib.rp_bert_embed_bwd(dx.data_ptr(), self.ids32.data_ptr(), self.in_pad.data_ptr(), self.in_tok.data_ptr(),
                                         self.B, L, d, drop, self.seed, 0, rng, G["item_emb"].data_ptr(),
                                         G["mask_emb"].data_ptr(), G["pos_emb"].data_ptr(), st()), "rp_bert_embed_bwd")

    # ------------------------------------------------------------------------------------------------ inference
    def forward_last_hidden(self):
        """Eval body -> hidden state of the LAST position (the caller has already shifted the window and put <MASK> there,
        bert4rec/dataset.py:322-345) -> self.hq bf16 [B, d]."""
        self._prepare(False)
        self._body_forward(False)
        check(self.lib.rp_gather_rows(self.x[-1].data_ptr(), self.last_idx.data_ptr(), self.B, None, self.cfg.d,
                                      self.hq.data_ptr(), 0, self._stream()), "rp_gather_rows")
        return self.hq

    def forward_hidden_all(self):
        self._prepare(False)
        self._body_forward(False)
        return self.x[-1]

    def head_for_scoring(self):
        """(W bf16 [I, d], bias fp32 [I128]) for rp_score_topk."""
        return self._head()
