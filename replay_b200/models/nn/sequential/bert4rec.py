"""Mirror of the legacy ``replay.models.nn.sequential.bert4rec`` modules on the B200 engine: ``Bert4RecModel``
(bert4rec/model.py:10-170) and the Lightning module ``Bert4Rec`` (bert4rec/lightning.py:15-683), plus the host-side
input-layout helpers (uniform masker dataset.py:55-92, predict shift dataset.py:322-345)."""
from __future__ import annotations

import torch

from ....compat import LightningModuleBase
from ....core import SasRecCore, _EngineLoss, dist_grad_all_reduce
from ....engine_bert import _BERT_BLOCK, Bert4RecEngine, BertConfig
from ....schema import item_feature_of

_BLEAF = {"ln1_w": "attention_norm.weight", "ln1_b": "attention_norm.bias", "in_w": "attention.in_proj_weight",
          "in_b": "attention.in_proj_bias", "out_w": "attention.out_proj.weight", "out_b": "attention.out_proj.bias",
          "ln2_w": "pff_norm.weight", "ln2_b": "pff_norm.bias", "w1": "pff.w_1.weight", "b1": "pff.w_1.bias",
          "w2": "pff.w_2.weight", "b2": "pff.w_2.bias"}


def bert_key_map(n_blocks: int, tying: bool, item_feature: str = "item_id") -> dict:
    """engine parameter name -> reference state_dict key (SURVEY.md Appendix B)."""
    m = {"item_emb": f"item_embedder.cat_embeddings.{item_feature}.weight", "mask_emb": "item_embedder.mask_embedding.weight",
         "pos_emb": "item_embedder.position.pe.weight"}
    for i in range(n_blocks):
        for k in _BERT_BLOCK:
            m[f"b{i}.{k}"] = f"transformer_blocks.{i}." + _BLEAF[k]
    if tying:
        m["head_b"] = "_head.out_bias"
    else:
        m["head_w"], m["head_b"] = "_head.linear.weight", "_head.linear.bias"
    return m


def uniform_masker(pad_mask: torch.Tensor, mask_prob: float = 0.15, generator=None) -> torch.Tensor:
    """Bert4RecUniformMasker.mask (dataset.py:71-92), vectorised over rows: token_mask = (rand * pad) >= p (0 = masked);
    a row where NOTHING is masked gets its last position masked, else a row where EVERYTHING is masked gets position -2
    unmasked - literally the reference's corner cases (known answers: tests/.../test_bert4rec_dataset.py:15-41)."""
    pm = pad_mask if pad_mask.dim() == 2 else pad_mask.unsqueeze(0)
    r = torch.rand(pm.shape, dtype=torch.float32, generator=generator, device="cpu").to(pm.device)
    tok = (r * pm) >= mask_prob
    all_kept = tok.all(-1)
    none_kept = ~tok.any(-1) & ~all_kept
    tok[all_kept, -1] = False
    if pm.shape[-1] > 1:
        tok[none_kept, -2] = True
    return tok if pad_mask.dim() == 2 else tok[0]


def shift_features(ids, pad_mask, token_mask, pad_value: int = 0):
    """_shift_features (dataset.py:322-345): roll left by one; the last position becomes <MASK> with pad = True."""
    ids2 = torch.roll(ids, -1, dims=-1); ids2[..., -1] = pad_value
    pm = torch.roll(pad_mask, -1, dims=-1); pm[..., -1] = True
    tm = torch.roll(token_mask, -1, dims=-1); tm[..., -1] = False
    return ids2, pm, tm


class _BertCore(SasRecCore):
    def __init__(self, cfg: BertConfig, item_feature="item_id", device=None, seed=0):
        torch.nn.Module.__init__(self)
        self.cfg, self.item_feature = cfg, item_feature
        self._device = torch.device(device) if device is not None else torch.device("cuda")
        self._seed, self.engine, self.flat, self._pending_state, self._shadow_dirty = seed, None, None, None, True
        self.adam_betas = (0.9, 0.98)
        self._keymap = bert_key_map(cfg.n_blocks, cfg.tying, item_feature)
        self._materialise()

    def _initial_seq_len(self):
        return self.cfg.max_len

    def _make_engine(self, batch, seq_len, with_grad):
        return Bert4RecEngine(self.cfg, batch, seq_len, self._device, seed=self._seed, with_grad=with_grad)

    def _to_ref(self, k, v):
        return v[: self.cfg.n_items] if k == "head_b" else v

    def _import(self, state):
        inv = {v: k for k, v in self._keymap.items()}
        with torch.no_grad():
            for rk, val in state.items():
                k = inv.get(rk)
                if k is None:
                    continue
                val = val.to(self.engine.dev, torch.float32)
                if k == "head_b":
                    self.engine.params[k][: val.numel()].copy_(val)
                else:
                    self.engine.params[k].copy_(val)
        self._shadow_dirty = True

    def state_dict(self, *a, destination=None, prefix="", keep_vars=False):
        src = self._export() if self.engine is not None else (self._pending_state or {})
        out = destination if destination is not None else {}
        for k, v in src.items():
            out[prefix + k] = v
        if self.cfg.tying:  # the tied head registers the embedder again (Appendix B)
            for k, v in list(src.items()):
                if k.startswith("item_embedder."):
                    out[prefix + "_head._item_embedder." + k[len("item_embedder."):]] = v
        return out

    def _apply_loss(self, eng) -> bool:
        """Select the engine's head for the remembered loss ("ce" | "bce"); True when it changed (captured graphs are stale)."""
        spec = getattr(self, "_loss_spec", ("ce", {}))
        key = (spec[0], tuple(sorted(spec[1].items())))
        if getattr(eng, "_loss_applied", None) == key:
            return False
        eng.set_loss(spec[0], **spec[1])
        eng._loss_applied = key
        return True

    def loss(self, ids, pad_mask, token_mask, labels):
        eng = self.ensure_engine(*ids.shape, with_grad=True)
        self._apply_loss(eng)
        eng.set_batch(ids, pad_mask, token_mask, labels)
        return _EngineLoss.apply(self.flat, self)

    def fused_step(self, ids, pad_mask, token_mask, labels, all_reduce="auto", lr=None):
        eng = self.ensure_engine(*ids.shape, with_grad=True)
        if self._shadow_dirty:
            eng.refresh_shadow(); self._shadow_dirty = False
        self._set_lr(eng, lr)
        if self._apply_loss(eng):
            self._drop_graphs()   # another loss head: different kernels / buffers
        eng.set_batch(ids, pad_mask, token_mask, labels)
        if isinstance(all_reduce, str):
            return self._graph_trainer(eng).run()[0]
        return eng.train_step(all_reduce, betas=self.adam_betas)[0]

    @torch.no_grad()
    def query_embeddings(self, ids, pad_mask, token_mask):
        eng = self.ensure_engine(*ids.shape, with_grad=self.engine.with_grad if self.engine is not None else False)
        if self._shadow_dirty:
            eng.refresh_shadow(); self._shadow_dirty = False
        eng.set_batch(ids, pad_mask, token_mask)
        return eng.forward_last_hidden()[: ids.shape[0]]

    @torch.no_grad()
    def logits(self, ids, pad_mask, token_mask, candidates=None):
        hq = self.query_embeddings(ids, pad_mask, token_mask)
        W, b = self.engine.head_for_scoring()
        b = b[: self.cfg.n_items]
        if candidates is not None:
            W, b = W[candidates].contiguous(), b[candidates].contiguous()
        out = torch.empty(hq.shape[0], W.shape[0], device=hq.device, dtype=torch.float32)
        self.engine._gemm(hq, W, out, hq.shape[0], W.shape[0], self.cfg.d, out_mode=2, bias=b)
        return out

    @torch.no_grad()
    def predict_topk(self, ids, pad_mask, token_mask, k, seen_ids=None, candidates=None):
        from .... import ops

        hq = self.query_embeddings(ids, pad_mask, token_mask).contiguous()
        W, b = self.engine.head_for_scoring()
        n_items, inv = self.cfg.n_items, None
        if candidates is not None:
            inv = torch.full((n_items,), -1, device=hq.device, dtype=torch.int32)
            inv[candidates] = torch.arange(candidates.numel(), device=hq.device, dtype=torch.int32)
            W = W[candidates].contiguous()
            bb = torch.zeros((candidates.numel() + 127) // 128 * 128, device=hq.device)
            bb[: candidates.numel()] = b[candidates]
            b = bb
        seen = None if seen_ids is None else ops.seen_prepare(seen_ids.contiguous(), n_items, inv)
        return ops.score_topk(hq, W, k, seen, candidates, bias=b)


class Bert4RecModel(torch.nn.Module):
    def __init__(self, schema, max_len: int = 100, hidden_size: int = 256, num_blocks: int = 2, num_heads: int = 4,
                 num_passes_over_block: int = 1, dropout: float = 0.1, enable_positional_embedding: bool = True,
                 enable_embedding_tying: bool = False, device=None, seed: int = 0):
        super().__init__()
        if num_passes_over_block != 1 or not enable_positional_embedding:
            raise NotImplementedError("only the reference defaults (one pass per block, positional embedding) are built")
        name, card, pad, _ = item_feature_of(schema)
        self.schema, self.item_feature_name, self.item_count, self.max_len = schema, name, card, max_len
        cfg = BertConfig(n_items=card, d=hidden_size, n_heads=num_heads, n_blocks=num_blocks, max_len=max_len, dropout=dropout,
                         tying=enable_embedding_tying, pad_id=pad if 0 <= pad < card else 0)
        self.core = _BertCore(cfg, item_feature=name, device=device, seed=seed)

    def state_dict(self, *a, **k):
        return self.core.state_dict(*a, **k)

    def load_state_dict(self, sd, strict=True, assign=False):
        return self.core.load_state_dict(sd, strict=strict)

    def get_query_embeddings(self, inputs, pad_mask, token_mask):
        return self.core.query_embeddings(inputs[self.item_feature_name], pad_mask, token_mask).float()

    def predict(self, inputs, pad_mask, token_mask, candidates_to_score=None):
        return self.core.logits(inputs[self.item_feature_name], pad_mask, token_mask, candidates_to_score)


class Bert4Rec(LightningModuleBase):
    def __init__(self, tensor_schema, block_count: int = 2, head_count: int = 4, hidden_size: int = 256, max_seq_len: int = 100,
                 dropout_rate: float = 0.1, pass_per_transformer_block_count: int = 1, enable_positional_embedding: bool = True,
                 enable_embedding_tying: bool = False, loss_type: str = "CE", loss_sample_count=None,
                 negative_sampling_strategy: str = "global_uniform", negatives_sharing: bool = False, optimizer_factory=None,
                 lr_scheduler_factory=None, fused_optimizer: bool = True, device=None):
        super().__init__()
        self.save_hyperparameters()
        if loss_type not in ("CE", "BCE") or loss_sample_count is not None:
            raise NotImplementedError("Not supported loss_type")   # sampled losses / CE_restricted: no fused head
        self._model = Bert4RecModel(tensor_schema, max_len=max_seq_len, hidden_size=hidden_size, num_blocks=block_count,
                                    num_heads=head_count, num_passes_over_block=pass_per_transformer_block_count,
                                    dropout=dropout_rate, enable_positional_embedding=enable_positional_embedding,
                                    enable_embedding_tying=enable_embedding_tying, device=device)
        self._schema = tensor_schema
        self._loss_type = loss_type
        if loss_type == "BCE":   # full-catalog BCE (bert4rec/lightning.py:273-305)
            self._model.core.set_loss("bce")
        self._optimizer_factory, self._lr_scheduler_factory = optimizer_factory, lr_scheduler_factory
        self._candidates_to_score = None
        self.fused_optimizer = fused_optimizer
        if fused_optimizer:
            self.automatic_optimization = False
        self._lr = getattr(optimizer_factory, "learning_rate", 1e-3)
        self._model.core.adam_betas = tuple(getattr(optimizer_factory, "betas", (0.9, 0.98)))

    def state_dict(self, *a, prefix="", **k):
        return {prefix + "_model." + key: v for key, v in self._model.state_dict().items()}

    def load_state_dict(self, sd, strict=True, assign=False):
        return self._model.load_state_dict({k[len("_model."):]: v for k, v in sd.items() if k.startswith("_model.")}, strict)

    def training_step(self, batch: dict, batch_idx: int = 0):
        """batch keys (bert4rec/dataset.py:167-173): query_id, pad_mask, inputs, token_mask, positive_labels."""
        ids = batch["inputs"][self._model.item_feature_name]
        args = (ids, batch["pad_mask"], batch["token_mask"], batch["positive_labels"])
        core = self._model.core
        loss = core.fused_step(*args, lr=self._fused_lr()) if self.fused_optimizer else core.loss(*args)
        self.log("train_loss", loss, on_step=True, on_epoch=True, prog_bar=True, sync_dist=True)
        return loss

    def _prepared(self, batch):
        """_prepare_prediction_batch (bert4rec/lightning.py:649-683): a batch of full length is taken AS IS (the prediction
        dataset already shifted it, bert4rec/dataset.py:322-345); a shorter one is left-padded with the padding value and
        then shifted; a longer one is an error."""
        ids, pm, tm = batch["inputs"][self._model.item_feature_name], batch["pad_mask"], batch["token_mask"]
        seq_len, max_len = pm.shape[1], self._model.max_len
        if seq_len > max_len:
            raise ValueError("The length of the submitted sequence must not exceed the maximum length of the sequence. "
                             f"The length of the sequence is given {seq_len}, while the maximum length is {max_len}")
        if seq_len < max_len:
            feats = self._schema.item_id_features
            feat = feats.item() if hasattr(feats, "item") else feats[self._schema.item_id_feature_name]
            ids = torch.nn.functional.pad(ids, (max_len - seq_len, 0), value=int(feat.padding_value))
            pm = torch.nn.functional.pad(pm, (max_len - seq_len, 0), value=0)
            ids, pm, tm = shift_features(ids, pm, pm, int(feat.padding_value))
        return ids, pm, tm

    def _model_predict(self, ids, pm, tm, candidates_to_score=None):
        cands = self._candidates_to_score if candidates_to_score is None else candidates_to_score
        return self._model.core.logits(ids, pm, tm, cands)

    def forward(self, feature_tensors, padding_mask, tokens_mask, candidates_to_score=None):
        return self._model_predict(feature_tensors[self._model.item_feature_name], padding_mask, tokens_mask, candidates_to_score)

    def validation_step(self, batch: dict, batch_idx: int = 0, dataloader_idx: int = 0):
        return self._model_predict(batch["inputs"][self._model.item_feature_name], batch["pad_mask"], batch["token_mask"])

    def predict_step(self, batch: dict, batch_idx: int = 0, dataloader_idx: int = 0):
        return self._model_predict(*self._prepared(batch))

    def predict(self, batch: dict, candidates_to_score=None):
        return self._model_predict(*self._prepared(batch), candidates_to_score)

    def predict_topk(self, batch: dict, k: int, seen_ids=None, candidates_to_score=None):
        ids, pm, tm = self._prepared(batch)
        cands = self._candidates_to_score if candidates_to_score is None else candidates_to_score
        return self._model.core.predict_topk(ids, pm, tm, k, seen_ids, cands)

    def _fused_lr(self) -> float:
        try:
            opt = self.optimizers()
        except Exception:  # noqa: BLE001 - no trainer attached
            opt = None
        if isinstance(opt, (list, tuple)):
            opt = opt[0] if opt else None
        if opt is not None and getattr(opt, "param_groups", None):
            return float(opt.param_groups[0]["lr"])
        return float(self._lr)

    def on_train_epoch_end(self):
        if self.fused_optimizer and self._lr_scheduler_factory is not None:
            try:
                sch = self.lr_schedulers()
            except Exception:  # noqa: BLE001
                sch = None
            for s_ in (sch if isinstance(sch, (list, tuple)) else [sch]):
                if s_ is not None:
                    s_.step()

    def configure_optimizers(self):
        params = [self._model.core.flat]
        opt = self._optimizer_factory.create(params) if self._optimizer_factory is not None else torch.optim.Adam(
            params, lr=1e-3, betas=(0.9, 0.98))
        return opt if self._lr_scheduler_factory is None else ([opt], [self._lr_scheduler_factory.create(opt)])

    @property
    def candidates_to_score(self):
        return self._candidates_to_score

    @candidates_to_score.setter
    def candidates_to_score(self, candidates=None):
        total = self._model.item_count
        if isinstance(candidates, torch.Tensor) and candidates.dtype is torch.long:
            if not (0 < candidates.shape[0] <= total):
                raise ValueError(f"Expected candidates length to be between 1 and total_item_count={total}")
        elif candidates is not None:
            raise ValueError(f"Expected candidates to be of type torch.LongTensor or None, gpt {type(candidates)}")
        self._candidates_to_score = candidates
