"""Generate golden vectors FROM THE REAL REFERENCE (run in the build container only; /root/reference is not on the
GPU box).  TEST INFRASTRUCTURE.

    PYTHONPATH=oracle/shim:/root/reference python oracle/gen_golden.py

Writes tests/golden/*.npz: seeded inputs, the reference modules' weights (state_dict) and the reference's outputs
(hidden states, train loss, gradients, eval logits, SeenItemsFilter + torch.topk result, one Adam step).  The larger
cases store int8-grid weights and a sample of each gradient to stay under 1 MB a file (format: oracle/golden.py).
tests/test_oracle_golden.py checks oracle/ against these; tests/test_parity_gpu.py checks the CUDA path against them.
"""
import os
import sys
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "shim"))
sys.path.insert(1, "/root/reference")
warnings.filterwarnings("ignore")

import golden  # noqa: E402  (oracle/golden.py, next to this script)

from replay.data import FeatureHint, FeatureSource, FeatureType  # noqa: E402
from replay.data.nn import TensorFeatureInfo, TensorFeatureSource, TensorSchema  # noqa: E402
from replay.models.nn.sequential.bert4rec.model import Bert4RecModel  # noqa: E402
from replay.models.nn.sequential.sasrec.model import SasRecModel  # noqa: E402
from replay.nn.lightning.postprocessor import SeenItemsFilter  # noqa: E402
from replay.nn.sequential import SasRec  # noqa: E402

OUT = os.path.join(os.path.dirname(HERE), "tests", "golden")
os.makedirs(OUT, exist_ok=True)


def schema(n_items, d, pad):
    return TensorSchema(
        [
            TensorFeatureInfo(
                name="item_id",
                is_seq=True,
                cardinality=n_items,
                padding_value=pad,
                embedding_dim=d,
                feature_type=FeatureType.CATEGORICAL,
                feature_sources=[TensorFeatureSource(FeatureSource.INTERACTIONS, "item_id")],
                feature_hint=FeatureHint.ITEM_ID,
            )
        ]
    )


def make_batch(g, B, L, n_items, pad, min_len=1):
    """Left-padded windows of L+1 ids -> inputs/labels shifted by one (sasrec/dataset.py:104-126)."""
    lens = torch.randint(min_len, L + 2, (B,), generator=g)
    lens[0] = L + 1  # one full row
    lens[1] = 2  # one nearly empty row
    full = torch.full((B, L + 1), pad, dtype=torch.int64)
    msk = torch.zeros(B, L + 1, dtype=torch.bool)
    for b in range(B):
        n = int(lens[b])
        full[b, L + 1 - n :] = torch.randint(0, n_items, (n,), generator=g)
        msk[b, L + 1 - n :] = True
    return full[:, :-1].contiguous(), msk[:, :-1].contiguous(), full[:, 1:].contiguous(), msk[:, 1:].contiguous()


def randomise_small_params(module, g):
    """xavier leaves biases 0 and LN at (1,0); perturb so the golden vectors exercise them."""
    with torch.no_grad():
        for name, p in module.named_parameters():
            if p.dim() == 1:
                p.add_(torch.randn(p.shape, generator=g) * 0.05)


def gen_new_sasrec(tag, B, L, d, H, n_items, n_blocks, seed, with_adam=True, int8=False, grad_sample=None):
    g = torch.Generator().manual_seed(seed)
    torch.manual_seed(seed)
    pad = n_items
    model = SasRec.from_params(schema(n_items, d, pad), embedding_dim=d, num_heads=H, num_blocks=n_blocks,
                               max_sequence_length=L, dropout=0.0)
    randomise_small_params(model, g)
    if int8:
        golden.snap_to_int8_grid(model)
    sd0 = {k: v.detach().clone() for k, v in model.state_dict().items()}
    ids, pmask, labels, tmask = make_batch(g, B, L, n_items, pad)
    out = golden.state_dict_arrays(model, int8)
    out.update(ids=ids.numpy(), pad_mask=pmask.numpy(), labels=labels.numpy(), target_mask=tmask.numpy(),
               n_items=n_items, d=d, H=H, L=L, n_blocks=n_blocks)
    # --- train mode: loss + grads (dropout 0)
    model.train()
    res = model(feature_tensors={"item_id": ids}, padding_mask=pmask, positive_labels=labels.unsqueeze(-1),
                negative_labels=None, target_padding_mask=tmask.unsqueeze(-1))
    loss = res["loss"]
    loss.backward()
    out["train_hidden"] = res["hidden_states"][0].detach().numpy()
    out["train_loss"] = loss.detach().numpy()
    for k, p in model.named_parameters():
        gr = (p.grad if p.grad is not None else torch.zeros_like(p)).numpy().copy()
        out["grad::" + k] = golden.sample(gr, grad_sample) if grad_sample else gr
    # --- one Adam step with the reference's optimizer settings (optimizer_factory.py:56-63)
    opt = torch.optim.Adam(model.parameters(), lr=1e-3, betas=(0.9, 0.98))
    opt.step()
    if with_adam:
        for k, p in model.named_parameters():
            out["adam1::" + k] = p.detach().numpy().copy()
    # restore weights for the eval leg
    model.load_state_dict(sd0)
    model.eval()
    with torch.no_grad():
        inf = model(feature_tensors={"item_id": ids}, padding_mask=pmask)
        logits = inf["logits"]
        out["eval_logits"] = logits.numpy()
        out["eval_hidden_last"] = inf["hidden_states"][0][:, -1].numpy()
        # SeenItemsFilter + topk (seen = the window ids, padding = n_items which the filter ignores)
        seen = ids.clone()
        filt = SeenItemsFilter(item_count=n_items, seen_items_column="seen_ids")
        fl = filt.on_prediction({"seen_ids": seen}, logits)
        k = 10
        top_s, top_i = torch.topk(fl, k=k, dim=1)
        out.update(seen_ids=seen.numpy(), topk_scores=top_s.numpy(), topk_ids=top_i.numpy())
        cands = torch.randperm(n_items, generator=g)[: max(k + L + 2, n_items // 3)]
        inf_c = model(feature_tensors={"item_id": ids}, padding_mask=pmask, candidates_to_score=cands)
        out.update(candidates=cands.numpy(), cand_logits=inf_c["logits"].numpy())
    np.savez_compressed(os.path.join(OUT, f"sasrec_new_{tag}.npz"), **out)
    print("wrote sasrec_new_" + tag, "loss", float(loss))


def gen_legacy_sasrec(tag, B, L, d, H, n_items, n_blocks, seed):
    g = torch.Generator().manual_seed(seed)
    torch.manual_seed(seed)
    pad = n_items
    model = SasRecModel(schema(n_items, d, pad), num_blocks=n_blocks, num_heads=H, hidden_size=d, max_len=L, dropout=0.0)
    randomise_small_params(model, g)
    ids, pmask, labels, tmask = make_batch(g, B, L, n_items, pad)
    out = golden.state_dict_arrays(model)
    out.update(ids=ids.numpy(), pad_mask=pmask.numpy(), labels=labels.numpy(), target_mask=tmask.numpy(),
               n_items=n_items, d=d, H=H, L=L, n_blocks=n_blocks)
    model.train()
    hidden = model.forward_step({"item_id": ids}, pmask)
    logits = model.get_logits(hidden)
    # sasrec/lightning.py:335-355
    lab = labels.masked_fill(~tmask, -100)
    loss = torch.nn.CrossEntropyLoss()(logits.view(-1, logits.size(-1)), lab.view(-1))
    loss.backward()
    out["train_hidden"] = hidden.detach().numpy()
    out["train_loss"] = loss.detach().numpy()
    for k, p in model.named_parameters():
        out["grad::" + k] = (p.grad if p.grad is not None else torch.zeros_like(p)).numpy().copy()
    model.eval()
    with torch.no_grad():
        out["eval_logits"] = model.predict({"item_id": ids}, pmask).numpy()
        out["eval_hidden_last"] = model.get_query_embeddings({"item_id": ids}, pmask).numpy()
    np.savez_compressed(os.path.join(OUT, f"sasrec_legacy_{tag}.npz"), **out)
    print("wrote sasrec_legacy_" + tag, "loss", float(loss))


def gen_bert4rec(tag, B, L, d, H, n_items, n_blocks, seed, tying, int8=False):
    g = torch.Generator().manual_seed(seed)
    torch.manual_seed(seed)
    model = Bert4RecModel(schema(n_items, d, 0), max_len=L, hidden_size=d, num_blocks=n_blocks, num_heads=H,
                          num_passes_over_block=1, dropout=0.0, enable_positional_embedding=True,
                          enable_embedding_tying=tying)
    randomise_small_params(model, g)
    if int8:
        golden.snap_to_int8_grid(model)
    # left padded inputs, uniform token mask (bert4rec/dataset.py:71-92): tok False = <MASK>; pads are False too
    lens = torch.randint(2, L + 1, (B,), generator=g)
    lens[0] = L
    ids = torch.zeros(B, L, dtype=torch.int64)
    pmask = torch.zeros(B, L, dtype=torch.bool)
    for b in range(B):
        n = int(lens[b])
        ids[b, L - n :] = torch.randint(0, n_items, (n,), generator=g)
        pmask[b, L - n :] = True
    tok = (torch.rand(B, L, generator=g) > 0.3) & pmask
    tok[:, -1] = False  # make sure every row has a masked real position
    labels = ids.clone()
    out = golden.state_dict_arrays(model, int8)
    out.update(ids=ids.numpy(), pad_mask=pmask.numpy(), token_mask=tok.numpy(), labels=labels.numpy(),
               n_items=n_items, d=d, H=H, L=L, n_blocks=n_blocks, tying=int(tying))
    model.train()
    hidden = model.forward_step({"item_id": ids}, pmask, tok)
    logits = model.get_logits(hidden)
    # bert4rec/lightning.py:332-351
    labels_mask = (~pmask) + tok
    masked = ~labels_mask
    loss = torch.nn.CrossEntropyLoss()(logits[masked], labels[masked])
    loss.backward()
    out["train_hidden"] = hidden.detach().numpy()
    out["train_loss"] = loss.detach().numpy()
    for k, p in model.named_parameters():
        out["grad::" + k] = (p.grad if p.grad is not None else torch.zeros_like(p)).numpy().copy()
    model.eval()
    with torch.no_grad():
        out["eval_logits"] = model.predict({"item_id": ids}, pmask, tok).numpy()
    np.savez_compressed(os.path.join(OUT, f"bert4rec_{tag}.npz"), **out)
    print("wrote bert4rec_" + tag, "loss", float(loss))


def gen_seen_filter_known_answers():
    """tests/nn/lightning/postprocessor/conftest.py:7-31 + test_postprocessor.py:7-46, run through the reference."""
    g = torch.Generator().manual_seed(3)
    seen = torch.LongTensor([[5, 5, 0, 1, 1], [1, 2, 4, 0, 3], [5, 5, 5, 5, 5], [0, 1, 2, 2, 2]])
    logits = torch.rand(4, 5, generator=g)
    filt = SeenItemsFilter(item_count=5)
    o1 = filt.on_prediction({"seen_ids": seen}, logits)
    cands = torch.LongTensor([1, 3, 2, 4])
    lc = torch.rand(4, 4, generator=g)
    filt2 = SeenItemsFilter(item_count=5)
    filt2.candidates = cands
    o2 = filt2.on_prediction({"seen_ids": seen}, lc)
    np.savez_compressed(os.path.join(OUT, "seen_filter_known.npz"), seen=seen.numpy(), logits=logits.numpy(),
                        out=o1.numpy(), candidates=cands.numpy(), cand_logits=lc.numpy(), cand_out=o2.numpy())
    print("wrote seen_filter_known")


def gen_dataset_layout():
    """The reference's per-sample dataset classes run on a tiny history store (sliding windows, short / empty-ish /
    over-long histories) -> tests/golden/dataset_layout.npz.  The BERT masker is fed a seeded generator; the same uniform
    draws are regenerated here and stored so the restatement and the device kernel can be checked bit-exactly."""
    from replay.models.nn.sequential.bert4rec.dataset import (Bert4RecPredictionDataset, Bert4RecTrainingDataset,
                                                              Bert4RecUniformMasker)
    from replay.models.nn.sequential.sasrec.dataset import SasRecPredictionDataset, SasRecTrainingDataset

    n_items, L, step, prob = 40, 6, 2, 0.3
    sch = schema(n_items, 8, n_items)
    rng = np.random.default_rng(5)
    lens = [1, 2, 3, 6, 7, 8, 13, 20, 5, 6, 1, 30]
    seqs = [rng.integers(0, n_items, n).astype(np.int64) for n in lens]

    class Store:
        schema = sch

        def __len__(self):
            return len(seqs)

        def get_query_id(self, i):
            return 1000 + 3 * i

        def get_sequence_length(self, i):
            return len(seqs[i])

        def get_sequence(self, i, name):
            return seqs[i]

        def get_max_sequence_length(self):
            return max(lens)

    ds = Store()
    out = {"lengths": np.asarray(lens), "items": np.concatenate(seqs), "L": L, "step": step, "mask_prob": prob,
           "pad": n_items, "query_ids": np.asarray([1000 + 3 * i for i in range(len(seqs))])}

    def stack(samples, path):
        def get(s):
            for k in path:
                s = s[k]
            return s.numpy()
        return np.stack([get(s) for s in samples])

    for tag, st in (("slide", step), ("last", None)):
        t = SasRecTrainingDataset(ds, max_sequence_length=L, sliding_window_step=st)
        smp = [t[i] for i in range(len(t))]
        out[f"sas_{tag}_index"] = np.asarray(t._inner._index2sequence_map)
        out[f"sas_{tag}_query"] = stack(smp, ["query_id"])[:, 0]
        out[f"sas_{tag}_ids"] = stack(smp, ["feature_tensor", "item_id"])
        out[f"sas_{tag}_pad"] = stack(smp, ["padding_mask"])
        out[f"sas_{tag}_labels"] = stack(smp, ["positive_labels"])
        out[f"sas_{tag}_tmask"] = stack(smp, ["target_padding_mask"])
    p = SasRecPredictionDataset(ds, max_sequence_length=L)
    smp = [p[i] for i in range(len(p))]
    out["pred_ids"] = stack(smp, ["feature_tensor", "item_id"])
    out["pred_pad"] = stack(smp, ["padding_mask"])

    for tag, st in (("slide", step), ("last", None)):
        bt = Bert4RecTrainingDataset(ds, L, sliding_window_step=st,
                                     custom_masker=Bert4RecUniformMasker(prob, torch.Generator().manual_seed(21)))
        smp = [bt[i] for i in range(len(bt))]
        g2 = torch.Generator().manual_seed(21)
        out[f"bert_{tag}_uniforms"] = np.stack([torch.rand(L, dtype=torch.float32, generator=g2).numpy() for _ in smp])
        out[f"bert_{tag}_index"] = np.asarray(bt._inner._index2sequence_map)
        out[f"bert_{tag}_ids"] = stack(smp, ["inputs", "item_id"])
        out[f"bert_{tag}_pad"] = stack(smp, ["pad_mask"])
        out[f"bert_{tag}_tok"] = stack(smp, ["token_mask"])
        out[f"bert_{tag}_labels"] = stack(smp, ["positive_labels"])
    # corner cases of the masker: nothing masked (prob 0 -> last token masked), everything masked (prob > 1)
    for tag, pr in (("p0", 0.0), ("p2", 2.0)):
        bt = Bert4RecTrainingDataset(ds, L, custom_masker=Bert4RecUniformMasker(pr, torch.Generator().manual_seed(22)))
        out[f"bert_{tag}_tok"] = stack([bt[i] for i in range(len(bt))], ["token_mask"])
    bp = Bert4RecPredictionDataset(ds, L)
    smp = [bp[i] for i in range(len(bp))]
    out["bertpred_ids"] = stack(smp, ["inputs", "item_id"])
    out["bertpred_pad"] = stack(smp, ["pad_mask"])
    out["bertpred_tok"] = stack(smp, ["token_mask"])
    # ---- new path: Array1DColumn.__getitem__ (left-padded gather of the LAST shape elements from flat values + offsets,
    # replay/data/nn/parquet/impl/array_1d_column.py:70-84, indexing.py:42-78) followed by NextTokenTransform(shift=1)
    from replay.data.nn.parquet.impl.array_1d_column import Array1DColumn
    from replay.nn.transform.next_token import NextTokenTransform
    col = Array1DColumn(data=torch.from_numpy(np.concatenate(seqs)), lengths=torch.tensor(lens, dtype=torch.int64), shape=L + 1,
                        padding=n_items)
    order = torch.tensor([3, 0, 11, 7, 7, 2, 10, 5, 1, 4, 6, 8, 9])
    mask, vals = col[order]
    nt = NextTokenTransform(label_name="item_id", shift=1, ignore="query_id")({"query_id": order.clone(), "item_id": vals,
                                                                               "item_id_mask": mask})
    out.update(newpath_order=order.numpy(), newpath_ids=nt["item_id"].numpy(), newpath_pad=nt["item_id_mask"].numpy(),
               newpath_labels=nt["positive_labels"].numpy(), newpath_tmask=nt["positive_labels_mask"].numpy())
    np.savez_compressed(os.path.join(OUT, "dataset_layout.npz"), **out)
    print("wrote dataset_layout", {k: np.asarray(v).shape for k, v in out.items() if k.endswith("_ids")})


def gen_sampled_losses():
    """Real reference sampled losses on the weights / batch of sasrec_new_tiny (new path: CESampled, BCESampled with the three
    negative shapes incl. collisions with the positive and an ignore index) and of sasrec_legacy_tiny (legacy module's
    _compute_loss_ce_sampled / _compute_loss_bce_sampled with the internally drawn negatives captured)
    -> tests/golden/sampled_losses.npz (losses + gradient of the item table and of one block weight)."""
    from replay.nn.loss import BCESampled, CESampled
    from replay.models.nn.sequential.sasrec.lightning import SasRec as LegacySasRec

    out = {}
    z = np.load(os.path.join(OUT, "sasrec_new_tiny.npz"))
    sd = {k[4:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd::")}
    n_items, d, H, L, nb = int(z["n_items"]), int(z["d"]), int(z["H"]), int(z["L"]), int(z["n_blocks"])
    ids, pm = torch.from_numpy(z["ids"]), torch.from_numpy(z["pad_mask"])
    labels, tm = torch.from_numpy(z["labels"]), torch.from_numpy(z["target_mask"])
    B = ids.shape[0]
    g = torch.Generator().manual_seed(77)
    N = 37
    negs = {"shared": torch.randint(0, n_items, (N,), generator=g),
            "perseq": torch.randint(0, n_items, (B, N), generator=g),
            "perpos": torch.randint(0, n_items, (B, L, N), generator=g)}
    # force collisions with the positive (several per row) and entries equal to the ignore index
    ignore = 5
    negs["shared"][3] = labels[tm][0]
    negs["shared"][7] = ignore
    negs["perseq"][:, 2] = labels[:, -1]
    negs["perseq"][1, 4] = ignore
    negs["perpos"][:, :, 1] = labels.clamp(max=n_items - 1)
    negs["perpos"][:, :, 9] = labels.clamp(max=n_items - 1)
    negs["perpos"][0, -1, 5] = ignore
    for k, v in negs.items():
        out["neg_" + k] = v.numpy()
    out["ignore_index"] = ignore
    for lname, mk in (("ce", lambda: CESampled(negative_labels_ignore_index=ignore)),
                      ("bce", lambda: BCESampled(negative_labels_ignore_index=ignore))):
        for shape, neg in negs.items():
            model = SasRec.from_params(schema(n_items, d, n_items), embedding_dim=d, num_heads=H, num_blocks=nb,
                                       max_sequence_length=L, dropout=0.0)
            model.load_state_dict(sd)
            model.loss = mk()
            model.loss.logits_callback = model.get_logits
            model.train()
            res = model(feature_tensors={"item_id": ids}, padding_mask=pm, positive_labels=labels.unsqueeze(-1),
                        negative_labels=neg, target_padding_mask=tm.unsqueeze(-1))
            res["loss"].backward()
            gr = {k: p.grad for k, p in model.named_parameters() if p.grad is not None}
            ek = [k for k in gr if "item_id" in k or "item_emb" in k]
            wk = [k for k in gr if k.endswith("in_proj_weight")]
            out[f"new_{lname}_{shape}_loss"] = res["loss"].detach().numpy()
            out[f"new_{lname}_{shape}_gE"] = gr[ek[0]].numpy().copy()
            out[f"new_{lname}_{shape}_gW"] = gr[wk[0]].numpy().copy()
            print("new", lname, shape, float(res["loss"]), ek[0], wk[0])

    # ---- legacy module: negatives are drawn inside the loss (torch.randint per valid target); capture them
    zl = np.load(os.path.join(OUT, "sasrec_legacy_tiny.npz"))
    sdl = {k[4:]: torch.from_numpy(zl[k]) for k in zl.files if k.startswith("sd::")}
    n_items, d, H, L, nb = int(zl["n_items"]), int(zl["d"]), int(zl["H"]), int(zl["L"]), int(zl["n_blocks"])
    ids, pm = torch.from_numpy(zl["ids"]), torch.from_numpy(zl["pad_mask"])
    labels, tm = torch.from_numpy(zl["labels"]), torch.from_numpy(zl["target_mask"])
    for lname, ltype in (("ce", "CE"), ("bce", "BCE")):
        mod = LegacySasRec(schema(n_items, d, n_items), block_count=nb, head_count=H, hidden_size=d, max_seq_len=L,
                           dropout_rate=0.0, loss_type=ltype, loss_sample_count=23)
        mod._model.load_state_dict(sdl)
        mod.train()
        rec = {}
        orig = torch.randint

        def wrap(*a, **k):
            r = orig(*a, **k)
            rec["neg"] = r.clone()
            return r

        torch.manual_seed(5)
        torch.randint = wrap
        try:
            fn = mod._compute_loss_ce_sampled if ltype == "CE" else mod._compute_loss_bce_sampled
            loss = fn({"item_id": ids}, labels, pm, tm)
        finally:
            torch.randint = orig
        loss.backward()
        gr = {k: p.grad for k, p in mod._model.named_parameters() if p.grad is not None}
        ek = [k for k in gr if "item_emb" in k]
        wk = [k for k in gr if k.endswith("in_proj_weight")]
        out[f"legacy_{lname}_neg"] = rec["neg"].numpy()          # [M, 23] in valid-target order
        out[f"legacy_{lname}_loss"] = loss.detach().numpy()
        out[f"legacy_{lname}_gE"] = gr[ek[0]].numpy().copy()
        out[f"legacy_{lname}_gW"] = gr[wk[0]].numpy().copy()
        print("legacy", lname, float(loss), rec["neg"].shape, ek[0], wk[0])
    np.savez_compressed(os.path.join(OUT, "sampled_losses.npz"), **out)
    print("wrote sampled_losses")


def gen_row_losses():
    """Real reference full-catalog per-row losses on the weights / batch of sasrec_new_tiny: LogOutCE, LogOutCEWeighted,
    CEWeighted (incl. its broadcast quirk), LogInCE (default eps / clamp and a tight clamp that is active on some rows)
    -> tests/golden/row_losses.npz (losses + gradient of the item table and of one block weight + the sample weights)."""
    from replay.nn.loss import CEWeighted, LogInCE, LogOutCE, LogOutCEWeighted

    out = {}
    z = np.load(os.path.join(OUT, "sasrec_new_tiny.npz"))
    sd = {k[4:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd::")}
    n_items, d, H, L, nb = int(z["n_items"]), int(z["d"]), int(z["H"]), int(z["L"]), int(z["n_blocks"])
    ids, pm = torch.from_numpy(z["ids"]), torch.from_numpy(z["pad_mask"])
    labels, tm = torch.from_numpy(z["labels"]), torch.from_numpy(z["target_mask"])
    B = ids.shape[0]
    g = torch.Generator().manual_seed(91)
    w = torch.rand(B, L, 1, generator=g) * 1.5 + 0.25
    out["weights"] = w.numpy()
    cases = {"logout": lambda: LogOutCE(cardinality=n_items),
             "logout_weighted": lambda: LogOutCEWeighted(cardinality=n_items, feature_name="w"),
             "ce_weighted": lambda: CEWeighted(feature_name="w"),
             "login": lambda: LogInCE(cardinality=n_items),
             "login_clamped": lambda: LogInCE(cardinality=n_items, log_epsilon=1e-3, clamp_border=5.5)}
    for name, mk in cases.items():
        model = SasRec.from_params(schema(n_items, d, n_items), embedding_dim=d, num_heads=H, num_blocks=nb,
                                   max_sequence_length=L, dropout=0.0)
        model.load_state_dict(sd)
        model.loss = mk()
        model.loss.logits_callback = model.get_logits
        model.train()
        res = model(feature_tensors={"item_id": ids, "w": w}, padding_mask=pm, positive_labels=labels.unsqueeze(-1),
                    negative_labels=None, target_padding_mask=tm.unsqueeze(-1).clone())
        res["loss"].backward()
        gr = {k: p.grad for k, p in model.named_parameters() if p.grad is not None}
        ek = [k for k in gr if "item_id" in k or "item_emb" in k]
        wk = [k for k in gr if k.endswith("in_proj_weight")]
        out[f"{name}_loss"] = res["loss"].detach().numpy()
        out[f"{name}_gE"] = gr[ek[0]].numpy().copy()
        out[f"{name}_gW"] = gr[wk[0]].numpy().copy()
        print("row loss", name, float(res["loss"]))
    np.savez_compressed(os.path.join(OUT, "row_losses.npz"), **out)
    print("wrote row_losses")



def gen_metrics_known():
    """TorchMetricsBuilder (replay/metrics/torch_metrics_builder.py) on a seeded case incl. novelty and coverage: pins the
    on-device mirror ``replay_b200.nn.lightning.RankingMetrics``."""
    from replay.metrics.torch_metrics_builder import TorchMetricsBuilder

    g = torch.Generator().manual_seed(77)
    n_items, B, K = 60, 40, 20
    names = ["recall", "precision", "ndcg", "map", "mrr", "novelty", "coverage"]
    b = TorchMetricsBuilder(names, top_k=[1, 5, 10, 20], item_count=n_items)
    out = {}
    for i in range(3):
        pred = torch.stack([torch.randperm(n_items, generator=g)[:K] for _ in range(B)])
        gt = torch.randint(0, n_items, (B, 6), generator=g)
        gt[torch.rand(B, 6, generator=g) < 0.4] = -1
        train = torch.randint(0, n_items, (B, 12), generator=g)
        train[torch.rand(B, 12, generator=g) < 0.3] = -2
        b.add_prediction(pred, gt, train)
        out[f"pred{i}"], out[f"gt{i}"], out[f"train{i}"] = pred.numpy(), gt.numpy(), train.numpy()
    res = b.get_metrics()
    out["names"] = np.array(sorted(res))
    out["values"] = np.array([res[k] for k in sorted(res)], dtype=np.float64)
    out["n_items"] = n_items
    np.savez_compressed(os.path.join(OUT, "metrics_known.npz"), **out)
    print("wrote metrics_known", {k: round(v, 4) for k, v in list(res.items())[:4]})


def gen_reference_default_shapes():
    """The reference's OWN default / example shapes, which are not multiples of the kernels' 64-wide feature slots:
    SasRec.from_params defaults embedding_dim=192, num_heads=4 (head_dim 48; nn/sequential/sasrec/model.py:199-253), the legacy
    module's hidden_size=50, head_count=1 (sasrec/lightning.py:30-47) and SURVEY's config 1 (d=64, H=2: head_dim 32)."""
    gen_new_sasrec("d192h4", B=4, L=12, d=192, H=4, n_items=200, n_blocks=2, seed=21, with_adam=False, int8=True,
                   grad_sample=4096)
    gen_new_sasrec("d64h2", B=4, L=12, d=64, H=2, n_items=200, n_blocks=2, seed=22, with_adam=False)
    gen_legacy_sasrec("d50h1", B=4, L=12, d=50, H=1, n_items=200, n_blocks=2, seed=23)


if __name__ == "__main__":
    import sys as _sys

    if len(_sys.argv) > 1 and _sys.argv[1] == "defaults":
        gen_reference_default_shapes()
        raise SystemExit(0)
    if len(_sys.argv) > 1 and _sys.argv[1] == "row_losses":
        gen_row_losses()
        raise SystemExit(0)
    if len(_sys.argv) > 1 and _sys.argv[1] == "metrics":
        gen_metrics_known()
        raise SystemExit(0)
    # shapes respect the CUDA path's tile constraints: hidden in {64,128,256,512}, head_dim in {64,128}
    gen_new_sasrec("tiny", B=6, L=16, d=64, H=1, n_items=300, n_blocks=2, seed=11)
    gen_new_sasrec("small", B=8, L=50, d=128, H=2, n_items=600, n_blocks=2, seed=12, with_adam=False, int8=True,
                   grad_sample=4096)
    gen_legacy_sasrec("tiny", B=6, L=16, d=64, H=1, n_items=300, n_blocks=2, seed=13)
    gen_bert4rec("tiny", B=6, L=16, d=64, H=1, n_items=300, n_blocks=2, seed=14, tying=False, int8=True)
    gen_bert4rec("tiny_tied", B=6, L=16, d=64, H=1, n_items=300, n_blocks=2, seed=15, tying=True, int8=True)
    gen_seen_filter_known_answers()
    gen_dataset_layout()
    gen_sampled_losses()
    gen_row_losses()
    gen_reference_default_shapes()
    gen_metrics_known()
