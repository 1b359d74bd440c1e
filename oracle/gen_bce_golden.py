"""Generate tests/golden/bce_losses.npz FROM THE REAL REFERENCE (run in the build container only; the reference is not on
the GPU box).  TEST INFRASTRUCTURE.

    PYTHONPATH=oracle/shim:/root/reference python oracle/gen_bce_golden.py

Runs the reference's full-catalog BCE on the weights / batches of the tiny golden cases written by oracle/gen_golden.py.
tests/test_bce_cpu.py checks oracle/bce.py against it; tests/test_gpu_bce.py checks the CUDA head through the mirrors.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)

# oracle/gen_golden.py puts the shim and the reference on the path; its schema() and golden directory are reused
from gen_golden import OUT, SasRec, golden, schema  # noqa: E402


def gen_bce_losses():
    """Real reference full-catalog BCE (BCEWithLogitsLoss(reduction="sum") / M against one-hot rows) on the weights / batches
    of the tiny cases: the new-path SasRec with ``loss = BCE()`` (sasrec_new_tiny), legacy SasRec(loss_type="BCE")
    ._compute_loss_bce (sasrec_legacy_tiny) and Bert4Rec(loss_type="BCE")._compute_loss_bce untied / tied (bert4rec_tiny,
    bert4rec_tiny_tied) -> tests/golden/bce_losses.npz: loss, item-table gradient, one block weight's gradient and, for
    BERT4Rec, the head-bias gradient (and, untied, the head weight's)."""
    from replay.models.nn.sequential.bert4rec.lightning import Bert4Rec as LegacyBert4Rec
    from replay.models.nn.sequential.sasrec.lightning import SasRec as LegacySasRec
    from replay.nn.loss import BCE

    out = {}

    def grads(module):
        return {k: p.grad for k, p in module.named_parameters() if p.grad is not None}

    # ---- new path
    z = golden.load(os.path.join(OUT, "sasrec_new_tiny.npz"))
    sd = {k[4:]: torch.from_numpy(z[k]) for k in z if k.startswith("sd::")}
    n_items, d, H, L, nb = int(z["n_items"]), int(z["d"]), int(z["H"]), int(z["L"]), int(z["n_blocks"])
    ids, pm = torch.from_numpy(z["ids"]), torch.from_numpy(z["pad_mask"])
    labels, tm = torch.from_numpy(z["labels"]), torch.from_numpy(z["target_mask"])
    model = SasRec.from_params(schema(n_items, d, n_items), embedding_dim=d, num_heads=H, num_blocks=nb,
                               max_sequence_length=L, dropout=0.0)
    model.load_state_dict(sd)
    model.loss = BCE()
    model.loss.logits_callback = model.get_logits
    model.train()
    res = model(feature_tensors={"item_id": ids}, padding_mask=pm, positive_labels=labels.unsqueeze(-1),
                negative_labels=None, target_padding_mask=tm.unsqueeze(-1).clone())
    res["loss"].backward()
    gr = grads(model)
    ek = [k for k in gr if "item_id" in k or "item_emb" in k]
    wk = [k for k in gr if k.endswith("in_proj_weight")]
    out["new_loss"] = res["loss"].detach().numpy()
    out["new_gE"] = gr[ek[0]].numpy().copy()
    out["new_gW"] = gr[wk[0]].numpy().copy()
    print("bce new", float(res["loss"]), ek[0], wk[0])

    # ---- legacy SASRec
    z = golden.load(os.path.join(OUT, "sasrec_legacy_tiny.npz"))
    sd = {k[4:]: torch.from_numpy(z[k]) for k in z if k.startswith("sd::")}
    n_items, d, H, L, nb = int(z["n_items"]), int(z["d"]), int(z["H"]), int(z["L"]), int(z["n_blocks"])
    ids, pm = torch.from_numpy(z["ids"]), torch.from_numpy(z["pad_mask"])
    labels, tm = torch.from_numpy(z["labels"]), torch.from_numpy(z["target_mask"])
    mod = LegacySasRec(schema(n_items, d, n_items), block_count=nb, head_count=H, hidden_size=d, max_seq_len=L,
                       dropout_rate=0.0, loss_type="BCE")
    mod._model.load_state_dict(sd)
    mod.train()
    loss = mod._compute_loss_bce({"item_id": ids}, labels, pm, tm)
    loss.backward()
    gr = grads(mod._model)
    ek = [k for k in gr if "item_emb" in k]
    wk = [k for k in gr if k.endswith("in_proj_weight")]
    out["legacy_loss"] = loss.detach().numpy()
    out["legacy_gE"] = gr[ek[0]].numpy().copy()
    out["legacy_gW"] = gr[wk[0]].numpy().copy()
    print("bce legacy", float(loss), ek[0], wk[0])

    # ---- legacy BERT4Rec, untied (ClassificationHead: Linear with bias) and tied (item table + out_bias)
    for tag in ("tiny", "tiny_tied"):
        z = golden.load(os.path.join(OUT, f"bert4rec_{tag}.npz"))
        sd = {k[4:]: torch.from_numpy(z[k]) for k in z if k.startswith("sd::")}
        n_items, d, H, L, nb = int(z["n_items"]), int(z["d"]), int(z["H"]), int(z["L"]), int(z["n_blocks"])
        tying = bool(int(z["tying"]))
        ids, pm, tok = (torch.from_numpy(z[k]) for k in ("ids", "pad_mask", "token_mask"))
        labels = torch.from_numpy(z["labels"])
        mod = LegacyBert4Rec(schema(n_items, d, 0), block_count=nb, head_count=H, hidden_size=d, max_seq_len=L,
                             dropout_rate=0.0, enable_embedding_tying=tying, loss_type="BCE")
        mod._model.load_state_dict(sd)
        mod.train()
        loss = mod._compute_loss_bce({"item_id": ids}, labels, pm, tok)
        loss.backward()
        gr = grads(mod._model)
        ek = [k for k in gr if k.endswith("cat_embeddings.item_id.weight")]
        wk = [k for k in gr if k.endswith("in_proj_weight")]
        bk = [k for k in gr if k in ("_head.linear.bias", "_head.out_bias")]
        key = "bert_tied" if tying else "bert"
        out[f"{key}_loss"] = loss.detach().numpy()
        out[f"{key}_gE"] = gr[ek[0]].numpy().copy()
        out[f"{key}_gW"] = gr[wk[0]].numpy().copy()
        out[f"{key}_gb"] = gr[bk[0]].numpy().copy()
        if not tying:
            out[f"{key}_gHW"] = gr["_head.linear.weight"].numpy().copy()
        print("bce", key, float(loss), ek[0], wk[0], bk[0])
    np.savez_compressed(os.path.join(OUT, "bce_losses.npz"), **out)
    print("wrote bce_losses")


if __name__ == "__main__":
    gen_bce_losses()
