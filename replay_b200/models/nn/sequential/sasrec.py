"""Mirror of the legacy ``replay.models.nn.sequential.sasrec`` modules on the B200 engine:
``SasRecModel`` (model.py:15-197) and the Lightning module ``SasRec`` (lightning.py:22-658).  Legacy semantics: causal mask
only (pad keys are NOT masked), pad rows zeroed after the embedding and after every block, final LayerNorm eps 1e-8,
sequence length must equal ``max_len`` (predict batches are left-padded up to it, lightning.py:624-658)."""
from __future__ import annotations

import torch

from ....compat import LightningModuleBase
from ....core import SasRecCore
from ....engine import EncoderConfig
from ....schema import item_feature_of


def _prepare_prediction_batch(schema, max_len: int, batch: dict) -> dict:
    """lightning.py:624-658: raise if longer than max_len, left-pad (ids with 0, mask with False) if shorter."""
    seq_len = batch["padding_mask"].shape[1]
    if seq_len > max_len:
        msg = ("The length of the submitted sequence must not exceed the maximum length of the sequence. "
               f"The length of the sequence is given {seq_len}, while the maximum length is {max_len}")
        raise ValueError(msg)
    if seq_len < max_len:
        pad = (max_len - seq_len, 0)
        batch = dict(batch)
        batch["feature_tensor"] = {k: torch.nn.functional.pad(v, pad, value=0) for k, v in batch["feature_tensor"].items()}
        batch["padding_mask"] = torch.nn.functional.pad(batch["padding_mask"], pad, value=0)
    return batch


class SasRecModel(torch.nn.Module):
    def __init__(self, schema, num_blocks: int = 2, num_heads: int = 1, hidden_size: int = 50, max_len: int = 200,
                 dropout: float = 0.2, ti_modification: bool = False, time_span: int = 256, device=None, seed: int = 0):
        super().__init__()
        if ti_modification:
            raise NotImplementedError("TiSASRec is outside the B200 hot-path scope (SURVEY.md §2)")
        name, card, pad, _ = item_feature_of(schema)
        self.schema = schema
        self.item_feature_name = name
        self.item_count = card
        self.padding_idx = card
        self.max_len = max_len
        self.hidden_size, self.num_blocks, self.num_heads, self.dropout = hidden_size, num_blocks, num_heads, dropout
        cfg = EncoderConfig(n_items=card, d=hidden_size, n_heads=num_heads, n_blocks=num_blocks, max_len=max_len,
                            dropout=dropout, variant="legacy")
        self.core = SasRecCore(cfg, item_feature=name, device=device, seed=seed)

    def state_dict(self, *a, **k):
        return self.core.state_dict(*a, **k)

    def load_state_dict(self, sd, strict=True, assign=False):
        return self.core.load_state_dict(sd, strict=strict)

    def item_table_fp32(self) -> torch.Tensor:
        """fp32 master copy of the item table incl. the padding row, [item_count + 1, hidden]."""
        if self.core.engine is None and not self.core._pending_state:
            self.core.ensure_engine(1, self.max_len, with_grad=False)  # materialise the seeded initial weights
        return self.core.state_dict()["item_embedder.item_emb.weight"].detach().clone()

    def replace_item_table(self, table: torch.Tensor):
        """Swap in a table for a (larger) vocabulary, keeping every other weight (lightning.py:612-621): the engine is rebuilt
        for the new catalog size; optimizer moments restart, as they do for the reference's freshly created Embedding."""
        import dataclasses
        sd = {k: v for k, v in self.state_dict().items() if not k.startswith("_head.")}
        sd["item_embedder.item_emb.weight"] = table.detach().to(torch.float32)
        new_count = table.shape[0] - 1
        spec = getattr(self.core, "_loss_spec", None)
        self.core = SasRecCore(dataclasses.replace(self.core.cfg, n_items=new_count), item_feature=self.item_feature_name,
                               device=self.core._device, seed=self.core._seed)
        if spec is not None:
            self.core.set_loss(spec[0], **spec[1])
        self.core.load_state_dict(sd)
        self.item_count = self.padding_idx = new_count

    def forward_step(self, feature_tensor, padding_mask):
        """Hidden states [B, L, d] (model.py:159-180)."""
        return self.core.hidden_states(feature_tensor[self.item_feature_name], padding_mask).float()

    def get_query_embeddings(self, feature_tensor, padding_mask):
        return self.core.query_embeddings(feature_tensor[self.item_feature_name], padding_mask).float()

    def get_logits(self, out_embeddings, item_ids=None):
        h = out_embeddings.reshape(-1, out_embeddings.shape[-1]).to(torch.bfloat16)
        h = self.core.engine.pad_features(h).contiguous()  # true hidden size -> the engine's feature slots
        tab = self.core.item_table(item_ids)
        out = torch.empty(h.shape[0], tab.shape[0], device=h.device, dtype=torch.float32)
        self.core.engine._gemm(h, tab, out, h.shape[0], tab.shape[0], self.core.cfg.dp, out_mode=2)
        return out.view(*out_embeddings.shape[:-1], tab.shape[0])

    def forward(self, feature_tensor, padding_mask):
        """All-position scores [B, L, |I|] (model.py:111-125) - materialised; use only for small problems."""
        return self.get_logits(self.forward_step(feature_tensor, padding_mask))

    def predict(self, feature_tensor, padding_mask, candidates_to_score=None):
        return self.core.logits(feature_tensor[self.item_feature_name], padding_mask, candidates_to_score)


class SasRec(LightningModuleBase):
    def __init__(self, tensor_schema, block_count: int = 2, head_count: int = 1, hidden_size: int = 50,
                 max_seq_len: int = 200, dropout_rate: float = 0.2, ti_modification: bool = False, time_span: int = 256,
                 loss_type: str = "CE", loss_sample_count=None, negative_sampling_strategy: str = "global_uniform",
                 negatives_sharing: bool = False, optimizer_factory=None, lr_scheduler_factory=None, sce_params=None,
                 fused_optimizer: bool = True, device=None):
        super().__init__()
        self.save_hyperparameters()
        if loss_type not in ("CE", "BCE") or (loss_type == "BCE" and loss_sample_count is None):
            # lightning.py:485 ; SCE has no fused head; full-catalog BCE is selected on the core: _model.core.set_loss("bce")
            raise NotImplementedError("Not supported loss_type")
        if negative_sampling_strategy not in {"global_uniform", "inbatch"}:
            raise AssertionError("negative_sampling_strategy must be 'global_uniform' or 'inbatch'")
        if loss_sample_count is not None and negative_sampling_strategy != "global_uniform":
            raise NotImplementedError("only the 'global_uniform' negative sampling strategy has a fused head")
        self._model = SasRecModel(tensor_schema, num_blocks=block_count, num_heads=head_count, hidden_size=hidden_size,
                                  max_len=max_seq_len, dropout=dropout_rate, ti_modification=ti_modification,
                                  time_span=time_span, device=device)
        self._schema = tensor_schema
        self._loss_type, self._loss_sample_count = loss_type, loss_sample_count
        self._negative_sampling_strategy, self._negatives_sharing = negative_sampling_strategy, negatives_sharing
        self._vocab_size = self._model.item_count
        if loss_sample_count is not None:
            self._model.core.set_loss("legacy_ce_sampled" if loss_type == "CE" else "legacy_bce_sampled")
        self._optimizer_factory = optimizer_factory
        self._lr_scheduler_factory = lr_scheduler_factory
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

    def _sample_negatives(self, ids):
        """lightning.py:394-472, 'global_uniform': one shared draw without replacement (negatives_sharing) or an independent
        uniform draw per position.  Drawn on the device with torch's generator (the reference draws inside the loss too)."""
        n = min(self._loss_sample_count, self._vocab_size)
        if self._negatives_sharing:
            return torch.multinomial(torch.ones(self._vocab_size, device=ids.device), n, replacement=False)
        return torch.randint(0, self._vocab_size, (*ids.shape, n), device=ids.device, dtype=torch.long)

    def training_step(self, batch: dict, batch_idx: int = 0):
        ids = batch["feature_tensor"][self._model.item_feature_name]
        args = (ids, batch["padding_mask"], batch["positive_labels"], batch["target_padding_mask"])
        core = self._model.core
        neg = self._sample_negatives(ids) if self._loss_sample_count is not None else None
        if self.fused_optimizer:
            loss = core.fused_step(*args, lr=self._fused_lr(), negatives=neg)  # all_reduce="auto": DDP exchange inside
        else:
            loss = core.loss(*args, negatives=neg)
        self.log("train_loss", loss, on_step=True, on_epoch=True, prog_bar=True, sync_dist=True)
        return loss

    def forward(self, feature_tensors, padding_mask, candidates_to_score=None):
        return self._model.predict(feature_tensors, padding_mask, candidates_to_score)

    def predict_step(self, batch: dict, batch_idx: int = 0, dataloader_idx: int = 0):
        batch = _prepare_prediction_batch(self._schema, self._model.max_len, batch)
        return self._model.predict(batch["feature_tensor"], batch["padding_mask"], self._candidates_to_score)

    def predict(self, batch: dict, candidates_to_score=None):
        batch = _prepare_prediction_batch(self._schema, self._model.max_len, batch)
        return self._model.predict(batch["feature_tensor"], batch["padding_mask"], candidates_to_score)

    def predict_topk(self, batch: dict, k: int, seen_ids=None, candidates_to_score=None):
        """Fused predict (no [B, |I|] scores): (item ids [B,k] int64, scores [B,k])."""
        batch = _prepare_prediction_batch(self._schema, self._model.max_len, batch)
        ids = batch["feature_tensor"][self._model.item_feature_name]
        return self._model.core.predict_topk(ids, batch["padding_mask"], k, seen_ids, candidates_to_score)

    def _fused_lr(self) -> float:
        """learning rate of this step: the (possibly scheduled) optimizer Lightning holds, else the factory's."""
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
        if self.fused_optimizer and self._lr_scheduler_factory is not None:  # manual optimisation: step the scheduler here
            try:
                sch = self.lr_schedulers()
            except Exception:  # noqa: BLE001
                sch = None
            for s_ in (sch if isinstance(sch, (list, tuple)) else [sch]):
                if s_ is not None:
                    s_.step()

    def configure_optimizers(self):
        params = [self._model.core.flat]
        if self._optimizer_factory is not None:
            opt = self._optimizer_factory.create(params)
        else:
            opt = torch.optim.Adam(params, lr=1e-3, betas=(0.9, 0.98))  # optimizer_factory.py:56-63
        if self._lr_scheduler_factory is None:
            return opt
        return [opt], [self._lr_scheduler_factory.create(opt)]

    def validation_step(self, batch: dict, batch_idx: int = 0, dataloader_idx: int = 0):
        """lightning.py:196-220: scores of the validation batch (same computation as predict)."""
        batch = _prepare_prediction_batch(self._schema, self._model.max_len, batch)
        return self._model.predict(batch["feature_tensor"], batch["padding_mask"])

    # ---- vocabulary growth (lightning.py:493-566, 612-621)
    def _set_new_item_table(self, table: torch.Tensor):
        self._model.replace_item_table(table)
        self._vocab_size = self._model.item_count
        feats = self._schema.item_id_features
        feat = feats.item() if hasattr(feats, "item") else feats[self._schema.item_id_feature_name]
        feat._set_cardinality(self._model.item_count)

    def set_item_embeddings_by_size(self, new_vocab_size: int):
        """Keep the fitted item embeddings and add xavier-normal rows for the new items."""
        old = self._model.item_table_fp32()
        old_vocab, hidden = old.shape[0] - 1, self._model.hidden_size
        if new_vocab_size <= old_vocab:
            raise ValueError("New vocabulary size must be greater then already fitted")
        new = torch.empty(new_vocab_size + 1, hidden)
        torch.nn.init.xavier_normal_(new)
        new[:old_vocab] = old[:-1].cpu()
        self._set_new_item_table(new)

    def set_item_embeddings_by_tensor(self, all_item_embeddings: torch.Tensor):
        """Replace the whole item table (possibly with more items); the padding row is zero."""
        if all_item_embeddings.dim() != 2:
            raise ValueError("Input tensor must have (number of all items, model hidden size) shape")
        old_vocab, hidden = self._model.item_count, self._model.hidden_size
        if all_item_embeddings.shape[0] < old_vocab:
            raise ValueError("New vocabulary size can't be less then already fitted")
        if all_item_embeddings.shape[1] != hidden:
            raise ValueError("Input tensor second dimension doesn't match model hidden size")
        new = torch.zeros(all_item_embeddings.shape[0] + 1, hidden)
        new[:-1] = all_item_embeddings.detach().float().cpu()
        self._set_new_item_table(new)

    def append_item_embeddings(self, item_embeddings: torch.Tensor):
        """Append rows for new items only; the padding row is zero."""
        if item_embeddings.dim() != 2:
            raise ValueError("Input tensor must have (number of new items, model hidden size) shape")
        if item_embeddings.shape[1] != self._model.hidden_size:
            raise ValueError("Input tensor second dimension doesn't match model hidden size")
        old = self._model.item_table_fp32()
        old_vocab = old.shape[0] - 1
        new = torch.zeros(old_vocab + item_embeddings.shape[0] + 1, self._model.hidden_size)
        new[:old_vocab] = old[:-1].cpu()
        new[old_vocab:-1] = item_embeddings.detach().float().cpu()
        self._set_new_item_table(new)

    def get_all_embeddings(self):
        """Copies, with the reference's keys (sasrec/model.py:374-381)."""
        sd = self._model.state_dict() if (self._model.core.engine is not None or self._model.core._pending_state) else None
        if sd is None:
            self._model.item_table_fp32()
            sd = self._model.state_dict()
        return {"item_embedding": sd["item_embedder.item_emb.weight"][:-1].detach().clone(),
                "positional_embedding": sd["item_embedder.pos_emb.pe.weight"].detach().clone()}

    @property
    def optimizer_factory(self):
        return self._optimizer_factory

    @optimizer_factory.setter
    def optimizer_factory(self, optimizer_factory):
        if not hasattr(optimizer_factory, "create"):  # lightning.py:575-585 (isinstance check against OptimizerFactory)
            raise ValueError(f"Expected optimizer_factory of type OptimizerFactory, got {type(optimizer_factory)}")
        self._optimizer_factory = optimizer_factory
        self._lr = getattr(optimizer_factory, "learning_rate", 1e-3)
        self._model.core.adam_betas = tuple(getattr(optimizer_factory, "betas", (0.9, 0.98)))

    @property
    def candidates_to_score(self):
        return self._candidates_to_score

    @candidates_to_score.setter
    def candidates_to_score(self, candidates=None):
        total = self._model.item_count  # lightning.py:594-610
        if isinstance(candidates, torch.Tensor) and candidates.dtype is torch.long:
            if not (0 < candidates.shape[0] <= total):
                raise ValueError(f"Expected candidates length to be between 1 and total_item_count={total}")
        elif candidates is not None:
            raise ValueError(f"Expected candidates to be of type torch.LongTensor or None, gpt {type(candidates)}")
        self._candidates_to_score = candidates
