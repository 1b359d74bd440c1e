"""``SasRecCore``: torch.nn.Module facade over the CUDA engine, shared by the new-path and legacy API mirrors.

* parameters live in ONE flat fp32 ``nn.Parameter`` (the engine's master buffer); ``state_dict`` / ``load_state_dict`` use the
  REFERENCE's key names (SURVEY.md Appendix B) so checkpoints interchange with RePlay's modules;
* the loss is produced by an ``autograd.Function`` whose backward runs the engine's hand-written backward kernels and
  hands the flat gradient to autograd, so ``loss.backward()`` + any torch optimizer (or Lightning's automatic
  optimization) work unchanged; ``fused_step()`` instead runs forward+backward+Adam entirely in the engine.
"""
from __future__ import annotations

import os

import torch

from .engine import _BLOCK_PARAMS, EncoderConfig, SasRecEngine

_LEAF = {"ln1_w": "attention_layernorms.{i}.weight", "ln1_b": "attention_layernorms.{i}.bias",
         "in_w": "attention_layers.{i}.in_proj_weight", "in_b": "attention_layers.{i}.in_proj_bias",
         "out_w": "attention_layers.{i}.out_proj.weight", "out_b": "attention_layers.{i}.out_proj.bias",
         "ln2_w": "forward_layernorms.{i}.weight", "ln2_b": "forward_layernorms.{i}.bias",
         "w1": "forward_layers.{i}.conv1.weight", "b1": "forward_layers.{i}.conv1.bias",
         "w2": "forward_layers.{i}.conv2.weight", "b2": "forward_layers.{i}.conv2.bias"}


def reference_key_map(variant: str, n_blocks: int, item_feature: str = "item_id") -> dict:
    """engine parameter name -> reference state_dict key (without the Lightning prefix)."""
    if variant == "new":
        m = {"item_emb": f"body.embedder.feature_embedders.{item_feature}.emb.weight",
             "pos_emb": "body.embedding_aggregator.pe.weight",
             "lnf_w": "body.output_normalization.weight", "lnf_b": "body.output_normalization.bias"}
        enc = "body.encoder."
    else:
        m = {"item_emb": "item_embedder.item_emb.weight", "pos_emb": "item_embedder.pos_emb.pe.weight",
             "lnf_w": "output_normalization.last_layernorm.weight", "lnf_b": "output_normalization.last_layernorm.bias"}
        enc = "sasrec_layers."
    for i in range(n_blocks):
        for k in _BLOCK_PARAMS:
            m[f"b{i}.{k}"] = enc + _LEAF[k].format(i=i)
    return m


class _EngineLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, flat, core):
        ctx.core = core
        eng = core.engine
        if core._shadow_dirty:
            eng.refresh_shadow()
            core._shadow_dirty = False
        eng.tick_rng()
        loss = eng.forward_train()
        return loss[0].clone()

    @staticmethod
    def backward(ctx, grad_out):
        eng = ctx.core.engine
        eng.g32.zero_()
        eng.backward()
        ctx.core._shadow_dirty = True  # an optimizer is about to change the fp32 master weights
        return eng.g32 * grad_out, None


def dist_grad_all_reduce():
    """Gradient exchange of the fused training step when ``torch.distributed`` is initialised with more than one rank (what
    Lightning's DDP hooks do for the reference's autograd ``training_step``; here there is no autograd backward for them to
    fire on): returns the ``all_reduce`` callback of ``SasRecEngine.train_step`` - one sum-all-reduce of the flat fp32
    gradient, Adam then applies it scaled by 1/world - or None for a single process."""
    import torch.distributed as dist

    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return None
    world = dist.get_world_size()

    def _all_reduce(g32):
        dist.all_reduce(g32, op=dist.ReduceOp.SUM)
        return 1.0 / world

    return _all_reduce


class SasRecCore(torch.nn.Module):
    def __init__(self, cfg: EncoderConfig, item_feature: str = "item_id", device=None, seed: int = 0):
        super().__init__()
        self.cfg = cfg
        self.item_feature = item_feature
        self._device = torch.device(device) if device is not None else torch.device("cuda")
        self._seed = seed
        self.engine: SasRecEngine | None = None
        self.flat: torch.nn.Parameter | None = None
        self._pending_state = None
        self._shadow_dirty = True
        self.adam_betas = (0.9, 0.98)  # optimizer_factory.py:56-63 / nn/lightning/optimizer.py:44-60
        self._keymap = reference_key_map(cfg.variant, cfg.n_blocks, item_feature)
        self._materialise()

    def _materialise(self):
        """Parameters exist from construction on (their layout depends on the configuration only), so ``parameters()``,
        ``configure_optimizers`` and DDP wrapping work before the first batch.  Skipped where there is no GPU (the CPU-side
        tests construct the mirrors for their key maps and error behaviour only)."""
        if self._device.type == "cuda" and torch.cuda.is_available():
            self.ensure_engine(1, self._initial_seq_len(), with_grad=False)

    def _initial_seq_len(self) -> int:
        return self.cfg.max_len if self.cfg.variant == "legacy" else min(self.cfg.max_len, 64)

    def _make_engine(self, batch: int, seq_len: int, with_grad: bool):
        return SasRecEngine(self.cfg, batch, seq_len, self._device, seed=self._seed, with_grad=with_grad)

    # ---- engine lifetime: the engine (parameters, gradients, Adam state, lr, RNG counter) is created ONCE; a larger batch or
    # another sequence length only re-allocates its activation workspace (SasRecEngine.resize), so ``flat`` keeps its identity
    def ensure_engine(self, batch: int, seq_len: int, with_grad: bool = True) -> SasRecEngine:
        e = self.engine
        if e is None:
            e = self.engine = self._make_engine(batch, seq_len, with_grad)
            if self._pending_state is not None:
                self._import(self._pending_state)
                self._pending_state = None
            self.flat = torch.nn.Parameter(e.p32, requires_grad=True)
            self._shadow_dirty = True
            spec = getattr(self, "_loss_spec", None)
            if spec is not None and spec[0] == "ce":
                e.set_loss("ce")
        elif batch > e.B or seq_len != e.L or (with_grad and not e.with_grad):
            e.resize(max(batch, e.B) if seq_len == e.L else batch, seq_len, with_grad or e.with_grad)
            e._loss_applied = None
            self._drop_graphs()
        return e

    # ---- the fused step replays two CUDA graphs (forward + backward | Adam) around the gradient exchange, exactly like
    # replay_b200.trainer.Trainer: ~40 launches per step would otherwise cost their launch latency on every training_step
    use_cuda_graph = os.environ.get("RP_NO_GRAPH", "0") == "0"

    def _drop_graphs(self):
        tr = getattr(self, "_trainer", None)
        if tr is not None:
            tr.invalidate()
        self._predict_graphs = {}

    def _graph_trainer(self, eng):
        from .trainer import Trainer

        tr = getattr(self, "_trainer", None)
        if tr is None or tr.engine is not eng:
            tr = self._trainer = Trainer(eng, use_graph=self.use_cuda_graph, betas=self.adam_betas)
        if tr.betas != tuple(self.adam_betas):
            tr.betas = tuple(self.adam_betas)
            tr.invalidate()
        return tr

    def _export(self) -> dict:
        # true (reference) shapes: the engine stores every head in its own 64/128-wide feature slot (EncoderConfig.dp)
        return {self._keymap[k]: self._to_ref(k, self.engine.export_named(k)) for k in self.engine.params}

    def _to_ref(self, k, v):
        return v.unsqueeze(-1) if k.endswith((".w1", ".w2")) else v  # Conv1d weight [d, d, 1]

    def _import(self, state: dict):
        inv = {v: k for k, v in self._keymap.items()}
        with torch.no_grad():
            for rk, val in state.items():
                k = inv.get(rk)
                if k is None:
                    continue
                val = val.to(self.engine.dev, torch.float32)
                if k.endswith((".w1", ".w2")) and val.dim() == 3:
                    val = val[:, :, 0]
                self.engine.import_named(k, val)
        self._shadow_dirty = True

    # ---- reference-compatible checkpoints
    def state_dict(self, *args, destination=None, prefix="", keep_vars=False):  # noqa: D102
        out = destination if destination is not None else {}
        src = self._export() if self.engine is not None else (self._pending_state or {})
        for k, v in src.items():
            out[prefix + k] = v
        if self.cfg.variant == "legacy":  # the reference's head registers the embedder again (Appendix B aliases)
            for a, b in (("_head._item_embedder.item_emb.weight", "item_embedder.item_emb.weight"),
                         ("_head._item_embedder.pos_emb.pe.weight", "item_embedder.pos_emb.pe.weight")):
                if b in src:
                    out[prefix + a] = src[b]
        return out

    def load_state_dict(self, state_dict, strict: bool = True, assign: bool = False):  # noqa: D102
        known = set(self._keymap.values())
        sd = {k: v for k, v in state_dict.items() if k in known}
        missing = known - set(sd)
        if strict and missing:
            raise RuntimeError(f"missing keys in state_dict: {sorted(missing)[:5]} ...")
        if self.engine is None:
            self._pending_state = {k: v.detach().clone() for k, v in sd.items()}
        else:
            self._import(sd)
        return torch.nn.modules.module._IncompatibleKeys(sorted(missing), [])

    # ---- loss selection (full-catalog CE by default; sampled heads: SURVEY §8 a9)
    def set_loss(self, kind: str = "ce", **kw):
        """Remembered across engine re-creations; see SasRecEngine.set_loss."""
        if kind == "bce" and self.cfg.dp not in (64, 128, 256):
            raise NotImplementedError(f"the full-catalog BCE head supports padded hidden sizes 64, 128 and 256 (got {self.cfg.dp})")
        self._loss_spec = (kind, kw)
        if self.engine is not None:
            self.engine._loss_applied = None  # re-applied with the negatives' shape when the next batch is staged
            if kind in self._FULL_CATALOG:
                self.engine.set_loss(kind, **kw)

    _FULL_CATALOG = ("ce", "ce_weighted", "login_ce", "bce")   # heads over the whole catalog (no negatives)

    def _stage(self, eng, ids, pad_mask, labels, target_mask, negatives, row_weights=None):
        spec = getattr(self, "_loss_spec", ("ce", {}))
        if spec[0] in self._FULL_CATALOG:
            if eng.sampled is not None or getattr(eng, "_loss_applied", None) != (spec[0], tuple(sorted(spec[1].items()))):
                eng.set_loss(spec[0], **spec[1])
                eng._loss_applied = (spec[0], tuple(sorted(spec[1].items())))
            eng.set_batch(ids, pad_mask, labels, target_mask)
            if spec[0] == "ce_weighted":
                if row_weights is None:
                    raise ValueError("this loss needs the sample weights of the batch")
                eng.set_row_weights(row_weights)
            return
        if spec[0] != "ce":
            shape = {1: "shared", 2: "perseq", 3: "perpos"}[negatives.dim()]
            want = dict(spec[1], n_neg=negatives.shape[-1], neg_shape=shape)
            if eng.sampled is None or getattr(eng, "_loss_applied", None) != (spec[0], tuple(sorted(want.items()))):
                eng.set_loss(spec[0], **want)
                eng._loss_applied = (spec[0], tuple(sorted(want.items())))
        elif eng.sampled is not None:
            eng.set_loss("ce")
        eng.set_batch(ids, pad_mask, labels, target_mask)
        if eng.sampled is not None:
            if negatives is None:
                raise ValueError("this loss needs negative_labels")
            eng.set_negatives(negatives)

    # ---- training / inference on [B, L] batches
    def loss(self, ids, pad_mask, labels, target_mask, negatives=None, row_weights=None) -> torch.Tensor:
        B, L = ids.shape
        eng = self.ensure_engine(B, L, with_grad=True)
        self._stage(eng, ids, pad_mask, labels, target_mask, negatives, row_weights)
        return _EngineLoss.apply(self.flat, self)

    def fused_step(self, ids, pad_mask, labels, target_mask, all_reduce="auto", lr: float | None = None,
                   negatives=None, row_weights=None) -> torch.Tensor:
        """forward + backward + Adam entirely inside the engine (no autograd, no torch optimizer).  ``all_reduce="auto"``
        exchanges the gradient over ``torch.distributed`` whenever a process group with more than one rank is initialised
        (Lightning ``strategy="ddp"``): this path has no autograd backward for DDP's hooks to fire on."""
        B, L = ids.shape
        eng = self.ensure_engine(B, L, with_grad=True)
        if self._shadow_dirty:
            eng.refresh_shadow()
            self._shadow_dirty = False
        self._set_lr(eng, lr)
        loss_before = getattr(eng, "_loss_applied", None), eng.sampled is None
        self._stage(eng, ids, pad_mask, labels, target_mask, negatives, row_weights)
        if (getattr(eng, "_loss_applied", None), eng.sampled is None) != loss_before:
            self._drop_graphs()  # another loss head: different kernels / buffers
        if isinstance(all_reduce, str):  # "auto": torch.distributed when initialised (inside Trainer.run)
            return self._graph_trainer(eng).run()[0]
        return eng.train_step(all_reduce, betas=self.adam_betas)[0]

    def _set_lr(self, eng, lr):
        if lr is not None and lr != getattr(eng, "_lr_host", None):
            eng.lr.fill_(lr)
            eng._lr_host = lr

    def mark_params_updated(self):
        """Call after an external optimizer changed ``flat`` (done automatically by the API mirrors)."""
        self._shadow_dirty = True

    def _eval_engine(self, ids):
        B, L = ids.shape
        eng = self.ensure_engine(B, L, with_grad=self.engine.with_grad if self.engine is not None else False)
        if self._shadow_dirty:
            eng.refresh_shadow()
            self._shadow_dirty = False
        return eng

    @torch.no_grad()
    def query_embeddings(self, ids, pad_mask) -> torch.Tensor:
        """Last-position hidden state, bf16 [B, d] (get_query_embeddings / forward_inference's last_hidden_state)."""
        eng = self._eval_engine(ids)
        return eng.unpad_features(self._last_hidden(eng, ids, pad_mask))

    def _last_hidden_padded(self, eng, ids):
        return eng.forward_last_hidden()[: ids.shape[0]]

    # ---- length-bucketed inference.  The query embedding only depends on the user's real items: pad positions are masked as
    # keys (new path: key_padding_mask, replay/nn/sequential/sasrec/model.py:258-307 with replay/nn/mask.py) and are never read
    # as queries (the last position is real).  With LEFT-padded windows a user with n <= W real items can therefore be
    # evaluated on the last W positions alone - same position embeddings (right-aligned), same result, W / L of the body work.
    # MovieLens-shaped histories at L = 200: ~1/3 of the users fit 64 positions, ~2/3 fit 128: the body of a 4096-user call
    # shrinks by a third.  One host read (bucket sizes + a left-padding check) and one extra pass of launches per bucket per
    # call: measured through predict_step + TopItemsCallback (bench25, r2) it pays for large calls only - 32768 users per
    # call 14.7 -> 12.5 ms, 4096 users 2.08 -> 2.25 ms (launch-bound) - so it engages from ``predict_bucket_min_batch`` users
    # per call.  RP_PREDICT_BUCKETS=0 turns it off.
    predict_buckets = tuple(int(v) for v in os.environ.get("RP_PREDICT_BUCKETS", "64,128").split(",") if v and int(v) > 0)
    predict_bucket_min_users = 1024    # smaller buckets join the next wider one
    predict_bucket_min_batch = 8192    # calls with fewer users take the single full-window pass

    def _last_hidden(self, eng, ids, pad_mask):
        """Padded-width last hidden states bf16 [B, dp] of a batch; stages the batch (or its buckets) itself."""
        B, L = ids.shape
        widths = [w for w in self.predict_buckets if w < L]
        if self.cfg.variant != "new" or not widths or B < self.predict_bucket_min_batch:
            eng.set_batch(ids, pad_mask)
            return self._last_hidden_padded(eng, ids)
        n_real = pad_mask.sum(1)
        bucket = sum((n_real > w).to(torch.int64) for w in widths)            # 0 .. len(widths): index of the narrowest fit
        left_padded = (pad_mask[:, 1:] >= pad_mask[:, :-1]).all()
        info = torch.cat([torch.bincount(bucket, minlength=len(widths) + 1), left_padded.to(torch.int64).view(1)]).tolist()
        counts, ok = info[:-1], bool(info[-1])
        for b in range(len(widths)):                                           # small buckets join the next wider one
            if counts[b] < self.predict_bucket_min_users:
                counts[b + 1] += counts[b]
                counts[b] = 0
        if not ok or counts[-1] == B:
            eng.set_batch(ids, pad_mask)
            return self._last_hidden_padded(eng, ids)
        order = torch.argsort(bucket, stable=True)
        out = torch.empty(B, self.cfg.dp, device=ids.device, dtype=torch.bfloat16)
        start = 0
        for b, w in enumerate(widths + [L]):
            cnt = counts[b]
            if cnt == 0:
                continue
            idx = order[start:start + cnt]
            start += cnt
            with eng.sub_geometry(cnt, w):
                eng.set_batch(ids[idx, L - w:], pad_mask[idx, L - w:])
                out[idx] = eng.forward_last_hidden()[:cnt]
        return out

    @torch.no_grad()
    def hidden_states(self, ids, pad_mask) -> torch.Tensor:
        eng = self._eval_engine(ids)
        eng.set_batch(ids, pad_mask)
        B, L = ids.shape
        return eng.unpad_features(eng.forward_hidden_all().view(eng.B, L, -1)[:B])

    @torch.no_grad()
    def item_table(self, candidates=None) -> torch.Tensor:
        t = self.engine.params16["item_emb"][: self.cfg.n_items]
        return t if candidates is None else t[candidates].contiguous()

    @torch.no_grad()
    def logits(self, ids, pad_mask, candidates=None) -> torch.Tensor:
        """Materialised fp32 scores [B, |I|] or [B, |C|] (API compatibility; the fused top-K path never builds them)."""
        eng = self._eval_engine(ids)
        hq = self._last_hidden(eng, ids, pad_mask)   # padded width: pairs with the padded table
        tab = self.item_table(candidates)
        out = torch.empty(hq.shape[0], tab.shape[0], device=hq.device, dtype=torch.float32)
        self.engine._gemm(hq, tab, out, hq.shape[0], tab.shape[0], self.cfg.dp, out_mode=2)
        return out

    @torch.no_grad()
    def predict_topk(self, ids, pad_mask, k: int, seen_ids=None, candidates=None):
        """Fused predict: body -> last hidden -> scores -> seen filter -> top-k.  Returns (item ids int64 [B,k], scores)."""
        from . import ops

        eng = self._eval_engine(ids)
        n_items = self.cfg.n_items
        B, L = ids.shape
        if (self.use_cuda_graph and candidates is None and seen_ids is not None and seen_ids.dtype == torch.int64
                and (self.cfg.variant != "new" or B < self.predict_bucket_min_batch or not self.predict_buckets)):
            # one CUDA-graph replay per call (body kernels + seen-list sort + fused scoring / top-K, ~20 launches): at 512 .. 4096
            # users per call the eager launches, not the GPU, bound the call through the callbacks (bench r2: 4096 users 1.91 ms
            # on the device, 2.08 ms end to end).  Inputs are staged into static buffers, the result is copied out.
            key = (B, L, int(k), tuple(seen_ids.shape), eng.B, eng.L)
            graphs = self.__dict__.setdefault("_predict_graphs", {})
            st = graphs.get(key)
            if st is None:
                while len(graphs) >= 8:   # a handful of call shapes per deployment; the oldest capture goes first
                    graphs.pop(next(iter(graphs)))
                st = graphs[key] = {"seen": torch.empty_like(seen_ids, memory_format=torch.contiguous_format), "calls": 0}
            st["seen"].copy_(seen_ids, non_blocking=True)
            eng.set_batch(ids, pad_mask)

            def run():
                hq_ = self._last_hidden_padded(eng, ids).contiguous()
                return ops.score_topk(hq_, self.item_table(None), k, ops.seen_prepare(st["seen"], n_items, None), None)

            if "graph" in st:
                st["graph"].replay()
                return st["ids"].clone(), st["scores"].clone()
            st["calls"] += 1
            if st["calls"] < 3:          # eager warm-up (lazy module load, kernel attributes) before the capture
                return run()
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                st["ids"], st["scores"] = run()
            st["graph"] = g
            g.replay()
            return st["ids"].clone(), st["scores"].clone()
        hq = self._last_hidden(eng, ids, pad_mask).contiguous()
        inv = None
        if candidates is not None:
            inv = torch.full((n_items,), -1, device=hq.device, dtype=torch.int32)
            inv[candidates] = torch.arange(candidates.numel(), device=hq.device, dtype=torch.int32)
        seen = None if seen_ids is None else ops.seen_prepare(seen_ids.contiguous(), n_items, inv)
        return ops.score_topk(hq, self.item_table(candidates), k, seen, candidates)
