"""TEST INFRASTRUCTURE - CPU restatement of the reference's full-catalog pointwise BCE, plain torch autograd.

Follows (one positive label per position)
  * BCE.forward                           replay/nn/loss/bce.py:52-95
  * legacy SasRec._compute_loss_bce       replay/models/nn/sequential/sasrec/lightning.py:278-308
  * legacy Bert4Rec._compute_loss_bce     replay/models/nn/sequential/bert4rec/lightning.py:273-305 (biased / tied head)
BCEWithLogitsLoss(reduction="sum") of the [M, |I|] logits against their one-hot rows, divided by M.  Pinned against the
real classes by oracle/gen_bce_golden.py -> tests/golden/bce_losses.npz.
"""
from __future__ import annotations

import torch


def bce_full(hidden, table, labels, target_mask, bias=None):
    """hidden [B, L, d], table [|I|, d], labels [B, L], target_mask [B, L] bool, bias [|I|] or None."""
    h = hidden[target_mask]
    y = labels[target_mask]
    logits = h @ table.T
    if bias is not None:
        logits = logits + bias
    onehot = torch.zeros_like(logits).scatter_(-1, y.unsqueeze(-1), 1.0)
    return torch.nn.functional.binary_cross_entropy_with_logits(logits, onehot, reduction="sum") / logits.size(0)


def sasrec_loss_and_grads(P, ids, pad_mask, labels, target_mask, n_heads, variant="new"):
    """SASRec body of oracle.sasrec + the full-catalog BCE; returns (loss, gradients in the canonical layout)."""
    from .sasrec import sasrec_body

    Pg = {}
    for k, v in P.items():
        Pg[k] = [{kk: vv.detach().clone().requires_grad_(True) for kk, vv in b.items()} for b in v] if k == "blocks" \
            else v.detach().clone().requires_grad_(True)
    hidden = sasrec_body(Pg, ids, pad_mask, n_heads, variant=variant)
    n_items = Pg["item_emb"].shape[0] - 1
    loss = bce_full(hidden, Pg["item_emb"][:n_items], labels, target_mask)
    loss.backward()
    G = {}
    for k, v in Pg.items():
        if k == "blocks":
            G[k] = [{kk: (vv.grad if vv.grad is not None else torch.zeros_like(vv)) for kk, vv in b.items()} for b in v]
        else:
            G[k] = v.grad if v.grad is not None else torch.zeros_like(v)
    G["item_emb"][-1].zero_()
    return loss.detach(), G


def bert4rec_loss(P, ids, pad_mask, token_mask, labels, n_heads):
    """Full-catalog BCE over the positions that are real and masked (bert4rec/lightning.py:283-305), through the biased (or
    tied + out_bias) head of oracle.bert4rec."""
    from .bert4rec import bert4rec_body, head_weights

    h = bert4rec_body(P, ids, pad_mask, token_mask, n_heads)
    w, b = head_weights(P)
    return bce_full(h, w, labels, pad_mask & ~token_mask, bias=b)
