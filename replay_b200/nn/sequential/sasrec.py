"""Mirror of ``replay.nn.sequential.SasRec`` (replay/nn/sequential/sasrec/model.py:116-378) backed by the B200 engine.

Same construction (``from_params``), same ``forward`` signature and train / inference output contracts, same
``state_dict`` key names (SURVEY.md Appendix B); the computation is the fused CUDA path (``replay_b200.core``)."""
from __future__ import annotations

import warnings

import torch

from ...core import SasRecCore
from ..loss import CE
from ...engine import EncoderConfig
from ...schema import item_feature_of


class _InferenceOutput(dict):
    """``InferenceOutput`` with a lazily evaluated ``hidden_states`` entry."""

    def __init__(self, logits, hidden_fn):
        super().__init__(logits=logits)
        self._hidden_fn = hidden_fn

    def __getitem__(self, k):
        if k == "hidden_states" and not super().__contains__(k):
            super().__setitem__(k, self._hidden_fn())
        return super().__getitem__(k)

    def __contains__(self, k):
        return k == "hidden_states" or super().__contains__(k)


class SasRec(torch.nn.Module):
    def __init__(self, core: SasRecCore, loss=None):
        super().__init__()
        self.core = core
        self.loss = loss if loss is not None else CE(ignore_index=core.cfg.n_items)

    @property
    def loss(self):
        """The reference's ``SasRec.loss`` attribute (model.py:181-197): assign ``CE`` / ``BCE`` / ``CESampled`` / ``BCESampled`` from
        ``replay_b200.nn.loss`` to select the fused head."""
        return self._loss

    @loss.setter
    def loss(self, spec):
        if not hasattr(spec, "kind"):
            raise NotImplementedError(f"loss {type(spec).__name__} has no fused CUDA head (supported: CE, CEWeighted, LogOutCE, "
                                      "LogOutCEWeighted, LogInCE, BCE, CESampled, BCESampled)")
        self._loss = spec
        self.core.set_loss(spec.kind, **spec.engine_kwargs())

    @classmethod
    def from_params(cls, schema, embedding_dim: int = 192, num_heads: int = 4, num_blocks: int = 2,
                    max_sequence_length: int = 50, dropout: float = 0.3, excluded_features=None,
                    categorical_list_feature_aggregation_method: str = "sum", device=None, seed: int = 0) -> "SasRec":
        """replay/nn/sequential/sasrec/model.py:199-253.  Only the item-id feature takes part (SURVEY §2: multi-feature
        embedders are out of the hot-path scope); ReLU FFN, LayerNorm(eps=1e-5) output normalisation, full CE loss."""
        name, card, pad, _ = item_feature_of(schema)
        if pad != card:
            raise ValueError("the item feature's padding_value must equal its cardinality (replay/data/nn/schema.py:89-90)")
        cfg = EncoderConfig(n_items=card, d=embedding_dim, n_heads=num_heads, n_blocks=num_blocks,
                            max_len=max_sequence_length, dropout=dropout, variant="new")
        return cls(SasRecCore(cfg, item_feature=name, device=device, seed=seed))

    # ---- reference surface
    @property
    def item_feature_name(self) -> str:
        return self.core.item_feature

    def state_dict(self, *a, **k):
        return self.core.state_dict(*a, **k)

    def load_state_dict(self, sd, strict=True, assign=False):
        return self.core.load_state_dict(sd, strict=strict)

    def parameters(self, recurse=True):
        if self.core.flat is None:
            raise RuntimeError("no CUDA device: the parameters live in the engine's flat device buffer (replay_b200 has no CPU path)")
        return iter([self.core.flat])

    def warm_up(self, batch_size: int, seq_len: int, with_grad: bool = True):
        self.core.ensure_engine(batch_size, seq_len, with_grad)
        return self

    def get_logits(self, model_embeddings, candidates_to_score=None):
        """model.py:258-265: scores of given hidden states [*, d] against the item table (materialised, fp32)."""
        h = model_embeddings.reshape(-1, model_embeddings.shape[-1]).to(torch.bfloat16)
        h = self.core.engine.pad_features(h).contiguous()  # true hidden size -> the engine's feature slots
        tab = self.core.item_table(candidates_to_score)
        out = torch.empty(h.shape[0], tab.shape[0], device=h.device, dtype=torch.float32)
        self.core.engine._gemm(h, tab, out, h.shape[0], tab.shape[0], self.core.cfg.dp, out_mode=2)
        return out.view(*model_embeddings.shape[:-1], tab.shape[0])

    def forward_train(self, feature_tensors, padding_mask, positive_labels, negative_labels=None, target_padding_mask=None):
        if positive_labels.dim() == 3:
            if positive_labels.size(-1) != 1:
                raise NotImplementedError("The case of multi-positive labels is not supported in the CE loss")
            positive_labels = positive_labels[..., 0]
        if target_padding_mask is not None and target_padding_mask.dim() == 3:
            target_padding_mask = target_padding_mask[..., 0]
        ids = feature_tensors[self.core.item_feature]
        if self._loss.needs_negatives and negative_labels is None:
            raise ValueError(f"{type(self._loss).__name__} needs negative_labels")
        rw = self._loss.row_weights(feature_tensors, target_padding_mask) if hasattr(self._loss, "row_weights") else None
        loss = self.core.loss(ids, padding_mask, positive_labels, target_padding_mask,
                              negatives=negative_labels if self._loss.needs_negatives else None, row_weights=rw)
        return {"loss": loss, "hidden_states": ()}

    def forward_inference(self, feature_tensors, padding_mask, candidates_to_score=None):
        """model.py:292-307: ``logits`` = scores of the LAST position [B, |I|] (or [B, |C|]); ``hidden_states`` = ([B, L, d],).
        The scores come from the last-position shortcut of the engine; the all-position hidden states (a second, full pass over
        the body) are only computed if that key is actually read."""
        ids = feature_tensors[self.core.item_feature]
        logits = self.core.logits(ids, padding_mask, candidates_to_score)
        return _InferenceOutput(logits, lambda: (self.core.hidden_states(ids, padding_mask).float(),))

    def forward(self, feature_tensors, padding_mask, candidates_to_score=None, positive_labels=None, negative_labels=None,
                target_padding_mask=None):
        assert padding_mask.dim() == 2, "padding_mask must be [batch, sequence]"
        if self.training:
            if candidates_to_score is not None:
                warnings.warn("Variable `candidates_to_score` is not None. This will have no effect at the training stage.")
            return self.forward_train(feature_tensors, padding_mask, positive_labels, negative_labels, target_padding_mask)
        return self.forward_inference(feature_tensors, padding_mask, candidates_to_score)

    # ---- fused extras
    def predict_topk(self, feature_tensors, padding_mask, k: int, seen_ids=None, candidates_to_score=None):
        return self.core.predict_topk(feature_tensors[self.core.item_feature], padding_mask, k, seen_ids, candidates_to_score)
