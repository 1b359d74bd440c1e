"""Loss selectors with the reference's names and constructor arguments (replay/nn/loss/{ce,bce}.py).  They carry no
computation: assigning one to ``SasRec.loss`` selects the fused CUDA head that implements it (full-catalog CE:
rp_ce_head_*; full-catalog BCE: rp_bce_head_*; sampled heads: rp_sampled_head_*).  Single positive label per position (multi-positive: NotImplementedError,
as in the reference's CE)."""
from __future__ import annotations

import torch


class _LossSpec:
    kind = "ce"
    needs_negatives = False

    def engine_kwargs(self) -> dict:
        return {}

    # LossProto surface (replay/nn/loss/base.py:9-28): the fused path never calls a logits callback
    @property
    def logits_callback(self):
        return getattr(self, "_logits_callback", None)

    @logits_callback.setter
    def logits_callback(self, func):
        self._logits_callback = func


class CE(_LossSpec):
    """replay/nn/loss/ce.py:10-81: torch CrossEntropyLoss over the whole catalog, ``ignore_index`` = padding value."""

    def __init__(self, ignore_index: int = -100, **kwargs):
        if kwargs:
            raise NotImplementedError(f"CrossEntropyLoss options {sorted(kwargs)} are not supported by the fused head")
        self.ignore_index = ignore_index


class BCE(_LossSpec):
    """replay/nn/loss/bce.py:10-95: ``BCEWithLogitsLoss(reduction="sum")`` over the whole catalog against the one-hot row of
    each valid target, divided by the number of valid targets -> the fused full-catalog BCE head (rp_bce_head_*)."""
    kind = "bce"

    def __init__(self, **kwargs):
        if kwargs:
            raise NotImplementedError(f"BCEWithLogitsLoss options {sorted(kwargs)} are not supported by the fused head")


class CESampled(_LossSpec):
    """replay/nn/loss/ce.py:146-249."""
    kind = "ce_sampled"
    needs_negatives = True

    def __init__(self, negative_labels_ignore_index: int = -100, **kwargs):
        if kwargs:
            raise NotImplementedError(f"CrossEntropyLoss options {sorted(kwargs)} are not supported by the fused head")
        self.negative_labels_ignore_index = negative_labels_ignore_index

    def engine_kwargs(self):
        return {"ignore_index": self.negative_labels_ignore_index}


class BCESampled(_LossSpec):
    """replay/nn/loss/bce.py:98-218."""
    kind = "bce_sampled"
    needs_negatives = True

    def __init__(self, log_epsilon: float = 1e-6, clamp_border: float = 100.0, negative_labels_ignore_index: int = -100):
        self.log_epsilon, self.clamp_border = log_epsilon, clamp_border
        self.negative_labels_ignore_index = negative_labels_ignore_index

    def engine_kwargs(self):
        return {"ignore_index": self.negative_labels_ignore_index, "log_eps": self.log_epsilon, "clamp": self.clamp_border}


class LogOutCE(CE):
    """replay/nn/loss/logout_ce.py:10-145.  With one positive label per position the loss is ``CrossEntropyLoss`` over
    [positive logit | all other logits with the positive's own column masked] - the full-catalog softmax CE itself, so it selects
    the same fused head (checked against the real class: tests/golden/row_losses.npz)."""

    def __init__(self, cardinality: int, negative_labels_ignore_index: int = -100, **kwargs):
        super().__init__(**kwargs)
        self.cardinality, self.negative_labels_ignore_index = cardinality, negative_labels_ignore_index


LogOutCESampled = CE   # replay/nn/loss/__init__.py:6


class _Weighted:
    """Sample weights ride in ``feature_tensors[feature_name]`` ([B, L, 1] or [B, L])."""
    kind = "ce_weighted"
    feature_name: str

    def row_weights(self, feature_tensors, target_mask):
        w = feature_tensors[self.feature_name]
        return w[..., 0] if w.dim() == 3 else w


class LogOutCEWeighted(_Weighted, LogOutCE):
    """replay/nn/loss/logout_ce.py:148-228: ``mean(loss_t * w_t)`` over the valid targets, w = the feature masked by the
    target padding mask -> per-row weights of the fused head (rp_ce_head_fwd_w)."""

    def __init__(self, cardinality: int, feature_name: str, negative_labels_ignore_index: int = -100, **kwargs):
        LogOutCE.__init__(self, cardinality, negative_labels_ignore_index, **kwargs)
        self.feature_name = feature_name


class CEWeighted(_Weighted, CE):
    """replay/nn/loss/ce.py:84-143.  The reference multiplies the [B * L] vector of row losses (zeros at the ignored positions)
    with the UNMASKED weight tensor [B, L, 1] and takes the mean of the broadcast [B, L, B * L] product, i.e.
    ``sum(valid CE) / (B * L) * mean(w over all positions)``: every valid row gets the same weight mean(w) * T_v / (B * L).
    Reproduced as such (known answer of the real class in tests/golden/row_losses.npz)."""

    def __init__(self, feature_name: str, **kwargs):
        CE.__init__(self, **kwargs)
        self.feature_name = feature_name

    def row_weights(self, feature_tensors, target_mask):
        w = feature_tensors[self.feature_name].to(torch.float32)
        return (w.mean() * target_mask.to(torch.float32).mean()).expand(target_mask.shape[0], target_mask.shape[1])


class LogInCE(_LossSpec):
    """replay/nn/loss/login_ce.py:102-239 with the whole catalog as negatives and one positive per position:
    ``-clamp(log(p + log_epsilon), -clamp_border, clamp_border)`` of the positive's softmax probability, mean over the valid
    targets."""
    kind = "login_ce"

    def __init__(self, cardinality: int, log_epsilon: float = 1e-6, clamp_border: float = 100.0,
                 negative_labels_ignore_index: int = -100):
        self.cardinality, self.log_epsilon, self.clamp_border = cardinality, log_epsilon, clamp_border
        self.negative_labels_ignore_index = negative_labels_ignore_index

    def engine_kwargs(self):
        return {"log_eps": self.log_epsilon, "clamp": self.clamp_border}
