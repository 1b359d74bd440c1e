"""The CPU oracle (oracle/) must reproduce the golden vectors that oracle/gen_golden.py produced by running the REAL
reference (sb-ai-lab/RePlay @ b4e051e8) in the build container.  This is what pins the oracle (SURVEY.md §8c)."""
import os

import numpy as np
import pytest
import torch

from oracle import bert4rec as ob
from oracle import golden
from oracle import sasrec as osr

TOL = dict(rtol=2e-5, atol=2e-6)


def load(golden_dir, name):
    z = golden.load(os.path.join(golden_dir, name))
    sd = {k[4:]: torch.from_numpy(z[k]) for k in z if k.startswith("sd::")}
    return z, sd


@pytest.mark.parametrize("name", ["sasrec_new_tiny.npz", "sasrec_new_small.npz", "sasrec_new_d192h4.npz", "sasrec_new_d64h2.npz"])
def test_new_sasrec_matches_reference(golden_dir, name):
    z, sd = load(golden_dir, name)
    P = osr.params_from_new_state_dict(sd)
    ids, pm = torch.from_numpy(z["ids"]), torch.from_numpy(z["pad_mask"])
    labels, tm = torch.from_numpy(z["labels"]), torch.from_numpy(z["target_mask"])
    H, n_items = int(z["H"]), int(z["n_items"])
    h = osr.sasrec_body(P, ids, pm, H, "new")
    torch.testing.assert_close(h, torch.from_numpy(z["train_hidden"]), **TOL)  # all rows incl. pad rows
    loss, G = osr.loss_and_grads(P, ids, pm, labels, tm, H, "new")
    torch.testing.assert_close(loss, torch.from_numpy(z["train_loss"]), rtol=1e-5, atol=1e-6)
    # gradients of every parameter
    gref = {k[6:]: torch.from_numpy(z[k]) for k in z if k.startswith("grad::")}
    Gref = osr.params_from_new_state_dict(gref)
    for a, b in zip(osr.flat_param_list(G), osr.flat_param_list(Gref)):
        kept = ~b.isnan()  # large golden gradients hold a sample of their elements (oracle/golden.py)
        torch.testing.assert_close(a[kept], b[kept], rtol=1e-4, atol=1e-6)
    # eval logits of the last position (real rows identical in eval)
    h_eval = osr.sasrec_body(P, ids, pm, H, "new", mode="eval")  # differs from train only on pad query rows
    real = pm[:, -1]
    torch.testing.assert_close(h_eval[pm], h[pm], rtol=0, atol=0)  # real rows: bit-identical
    h = h_eval
    logits = h[:, -1] @ P["item_emb"][:n_items].T
    torch.testing.assert_close(logits, torch.from_numpy(z["eval_logits"]), **TOL)
    # SeenItemsFilter + topk
    ids_k, sc_k = osr.score_topk(h[:, -1], P["item_emb"][:n_items], torch.from_numpy(z["seen_ids"]), 10,
                                 acc_dtype=torch.float32)
    assert torch.equal(ids_k, torch.from_numpy(z["topk_ids"]))
    torch.testing.assert_close(sc_k, torch.from_numpy(z["topk_scores"]), **TOL)
    # candidates
    c = torch.from_numpy(z["candidates"])
    torch.testing.assert_close(h[:, -1] @ P["item_emb"][:n_items][c].T, torch.from_numpy(z["cand_logits"]), **TOL)
    # one Adam step (optimizer_factory.py:56-63)
    if any(k.startswith("adam1::") for k in z):
        a1 = osr.params_from_new_state_dict({k[7:]: torch.from_numpy(z[k]) for k in z if k.startswith("adam1::")})
        for p, g, ref in zip(osr.flat_param_list(P), osr.flat_param_list(Gref), osr.flat_param_list(a1)):
            p1, _, _ = osr.adam_step(p, g, torch.zeros_like(p), torch.zeros_like(p), 1)
            torch.testing.assert_close(p1, ref, rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("name", ["sasrec_legacy_tiny.npz", "sasrec_legacy_d50h1.npz"])
def test_legacy_sasrec_matches_reference(golden_dir, name):
    z, sd = load(golden_dir, name)
    P = osr.params_from_legacy_state_dict(sd)
    ids, pm = torch.from_numpy(z["ids"]), torch.from_numpy(z["pad_mask"])
    labels, tm = torch.from_numpy(z["labels"]), torch.from_numpy(z["target_mask"])
    H, n_items = int(z["H"]), int(z["n_items"])
    h = osr.sasrec_body(P, ids, pm, H, "legacy")
    torch.testing.assert_close(h, torch.from_numpy(z["train_hidden"]), **TOL)
    loss, G = osr.loss_and_grads(P, ids, pm, labels, tm, H, "legacy")
    torch.testing.assert_close(loss, torch.from_numpy(z["train_loss"]), rtol=1e-5, atol=1e-6)
    gref = osr.params_from_legacy_state_dict({k[6:]: torch.from_numpy(z[k]) for k in z if k.startswith("grad::")})
    for a, b in zip(osr.flat_param_list(G), osr.flat_param_list(gref)):
        torch.testing.assert_close(a, b, rtol=1e-4, atol=1e-6)
    torch.testing.assert_close(h[:, -1] @ P["item_emb"][:n_items].T, torch.from_numpy(z["eval_logits"]), **TOL)


@pytest.mark.parametrize("name", ["bert4rec_tiny.npz", "bert4rec_tiny_tied.npz"])
def test_bert4rec_matches_reference(golden_dir, name):
    z, sd = load(golden_dir, name)
    P = ob.params_from_state_dict(sd)
    ids, pm, tok = (torch.from_numpy(z[k]) for k in ("ids", "pad_mask", "token_mask"))
    H = int(z["H"])
    h = ob.bert4rec_body(P, ids, pm, tok, H)
    torch.testing.assert_close(h, torch.from_numpy(z["train_hidden"]), **TOL)
    loss = ob.train_loss(P, ids, pm, tok, torch.from_numpy(z["labels"]), H)
    torch.testing.assert_close(loss, torch.from_numpy(z["train_loss"]), rtol=1e-5, atol=1e-6)
    w, b = ob.head_weights(P)
    torch.testing.assert_close(h[:, -1] @ w.T + b, torch.from_numpy(z["eval_logits"]), **TOL)


def test_seen_filter_known_answers(golden_dir):
    """tests/nn/lightning/postprocessor/test_postprocessor.py:7-46 (reference), via golden outputs of the reference."""
    z = np.load(os.path.join(golden_dir, "seen_filter_known.npz"))
    out = osr.seen_filter(torch.from_numpy(z["logits"]), torch.from_numpy(z["seen"]), 5)
    assert torch.equal(out, torch.from_numpy(z["out"]))
    expect_mask = torch.tensor([[1, 1, 0, 0, 0], [1, 1, 1, 1, 1], [0, 0, 0, 0, 0], [1, 1, 1, 0, 0]], dtype=torch.bool)
    assert torch.equal(torch.isinf(out), expect_mask)


def test_sasrec_training_example_layout():
    """tests/models/nn/sequential/sasrec/test_sasrec_dataset.py:40-48 known answer (sequence [0, 1], max_len 8)."""
    ids, pm, labels, tm = osr.sasrec_training_example([0, 1], 8, pad_value=-1)
    assert pm.tolist() == [False] * 7 + [True]
    assert tm.tolist() == [False] * 6 + [True, True]
    assert labels.tolist() == [-1] * 6 + [0, 1]


# ------------------------------------------------------------------------------------------------ dataset layout (§8 a15/f.1)
def _layout():
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "dataset_layout.npz"))


def _histories(z):
    off = np.concatenate([[0], np.cumsum(z["lengths"])])
    return [z["items"][off[i]:off[i + 1]] for i in range(len(z["lengths"]))]


def test_dataset_restatement_matches_reference_samples():
    """oracle/dataset.py against samples produced by the reference's own dataset classes (sliding windows, short and
    over-long histories, both BERT masker corner cases)."""
    from oracle import dataset as od
    z = _layout()
    seqs, L, pad, step, prob = _histories(z), int(z["L"]), int(z["pad"]), int(z["step"]), float(z["mask_prob"])
    for tag, st in (("slide", step), ("last", None)):
        idx = od.window_index(z["lengths"], L + 1, st)
        assert np.array_equal(np.asarray(idx), z[f"sas_{tag}_index"])
        smp = [od.sasrec_training_sample(seqs[i], o, L, pad) for i, o in idx]
        assert np.array_equal(np.stack([s["item_id"] for s in smp]), z[f"sas_{tag}_ids"])
        assert np.array_equal(np.stack([s["padding_mask"] for s in smp]), z[f"sas_{tag}_pad"])
        assert np.array_equal(np.stack([s["positive_labels"] for s in smp]), z[f"sas_{tag}_labels"])
        assert np.array_equal(np.stack([s["target_padding_mask"] for s in smp]), z[f"sas_{tag}_tmask"])
        bidx = od.window_index(z["lengths"], L, st)
        assert np.array_equal(np.asarray(bidx), z[f"bert_{tag}_index"])
        u = z[f"bert_{tag}_uniforms"]
        bs = [od.bert_training_sample(seqs[i], o, L, pad, u[r], prob) for r, (i, o) in enumerate(bidx)]
        assert np.array_equal(np.stack([s["item_id"] for s in bs]), z[f"bert_{tag}_ids"])
        assert np.array_equal(np.stack([s["pad_mask"] for s in bs]), z[f"bert_{tag}_pad"])
        assert np.array_equal(np.stack([s["token_mask"] for s in bs]), z[f"bert_{tag}_tok"])
        assert np.array_equal(np.stack([s["positive_labels"] for s in bs]), z[f"bert_{tag}_labels"])
    pr = [od.prediction_sample(s, L, pad) for s in seqs]
    assert np.array_equal(np.stack([s["item_id"] for s in pr]), z["pred_ids"])
    assert np.array_equal(np.stack([s["padding_mask"] for s in pr]), z["pred_pad"])
    bp = [od.bert_prediction_sample(s, L, pad) for s in seqs]
    assert np.array_equal(np.stack([s["item_id"] for s in bp]), z["bertpred_ids"])
    assert np.array_equal(np.stack([s["pad_mask"] for s in bp]), z["bertpred_pad"])
    assert np.array_equal(np.stack([s["token_mask"] for s in bp]), z["bertpred_tok"])
    # masker corner cases are independent of the draws: prob 0 keeps everything -> last token masked;
    # prob > 1 masks everything -> the one before last is un-masked
    for tag, p_ in (("p0", 0.0), ("p2", 2.0)):
        got = np.stack([od.bert_token_mask(z["bert_last_pad"][r], np.full(L, 0.5, np.float32), p_) for r in range(len(seqs))])
        assert np.array_equal(got, z[f"bert_{tag}_tok"])


# ------------------------------------------------------------------------------------------------ sampled losses (§8 a9/f.2)
def _scatter_neg(neg_valid, tm):
    """[M, N] negatives in valid-target order -> [B, L, N] (the layout the restatement / the CUDA path take)."""
    out = torch.zeros(*tm.shape, neg_valid.shape[1], dtype=torch.int64)
    out[tm] = neg_valid
    return out


@pytest.mark.parametrize("loss", ["ce", "bce"])
@pytest.mark.parametrize("shape", ["shared", "perseq", "perpos"])
def test_sampled_losses_new_path_match_reference(golden_dir, loss, shape):
    from oracle import sampled as osm
    z, sd = load(golden_dir, "sasrec_new_tiny.npz")
    zs = np.load(os.path.join(golden_dir, "sampled_losses.npz"))
    P = osr.params_from_new_state_dict(sd)
    ids, pm = torch.from_numpy(z["ids"]), torch.from_numpy(z["pad_mask"])
    labels, tm = torch.from_numpy(z["labels"]), torch.from_numpy(z["target_mask"])
    neg = torch.from_numpy(zs["neg_" + shape])
    l, G = osm.loss_and_grads(P, ids, pm, labels, tm, neg, int(z["H"]), loss, ignore_index=int(zs["ignore_index"]))
    torch.testing.assert_close(l, torch.from_numpy(zs[f"new_{loss}_{shape}_loss"]), rtol=2e-5, atol=2e-6)
    torch.testing.assert_close(G["item_emb"], torch.from_numpy(zs[f"new_{loss}_{shape}_gE"]), rtol=1e-4, atol=2e-6)
    torch.testing.assert_close(G["blocks"][0]["in_w"], torch.from_numpy(zs[f"new_{loss}_{shape}_gW"]), rtol=1e-4, atol=2e-6)


@pytest.mark.parametrize("loss", ["ce", "bce"])
def test_sampled_losses_legacy_match_reference(golden_dir, loss):
    from oracle import sampled as osm
    z, sd = load(golden_dir, "sasrec_legacy_tiny.npz")
    zs = np.load(os.path.join(golden_dir, "sampled_losses.npz"))
    P = osr.params_from_legacy_state_dict(sd)
    ids, pm = torch.from_numpy(z["ids"]), torch.from_numpy(z["pad_mask"])
    labels, tm = torch.from_numpy(z["labels"]), torch.from_numpy(z["target_mask"])
    neg = _scatter_neg(torch.from_numpy(zs[f"legacy_{loss}_neg"]), tm)
    kw = dict(vocab_size=int(z["n_items"])) if loss == "ce" else {}
    l, G = osm.loss_and_grads(P, ids, pm, labels, tm, neg, int(z["H"]), "legacy_" + loss, variant="legacy", **kw)
    torch.testing.assert_close(l, torch.from_numpy(zs[f"legacy_{loss}_loss"]), rtol=2e-5, atol=2e-6)
    torch.testing.assert_close(G["item_emb"], torch.from_numpy(zs[f"legacy_{loss}_gE"]), rtol=1e-4, atol=2e-6)
    torch.testing.assert_close(G["blocks"][0]["in_w"], torch.from_numpy(zs[f"legacy_{loss}_gW"]), rtol=1e-4, atol=2e-6)


# ------------------------------------------------------------------------------------------------ full-catalog per-row losses (§8 f.2)
ROW_CASES = {"logout": ("logout", {}), "logout_weighted": ("logout_weighted", {}), "ce_weighted": ("ce_weighted", {}),
             "login": ("login", {}), "login_clamped": ("login", dict(log_eps=1e-3, clamp=5.5))}


@pytest.mark.parametrize("case", sorted(ROW_CASES))
def test_row_losses_match_reference(golden_dir, case):
    from oracle import sampled as osm
    z, sd = load(golden_dir, "sasrec_new_tiny.npz")
    zr = np.load(os.path.join(golden_dir, "row_losses.npz"))
    P = osr.params_from_new_state_dict(sd)
    ids, pm = torch.from_numpy(z["ids"]), torch.from_numpy(z["pad_mask"])
    labels, tm = torch.from_numpy(z["labels"]), torch.from_numpy(z["target_mask"])
    kind, kw = ROW_CASES[case]
    l, G = osm.row_loss_and_grads(P, ids, pm, labels, tm, int(z["H"]), kind, weights=torch.from_numpy(zr["weights"]), **kw)
    torch.testing.assert_close(l, torch.from_numpy(zr[f"{case}_loss"]), rtol=2e-5, atol=2e-6)
    torch.testing.assert_close(G["item_emb"], torch.from_numpy(zr[f"{case}_gE"]), rtol=2e-4, atol=2e-6)
    torch.testing.assert_close(G["blocks"][0]["in_w"], torch.from_numpy(zr[f"{case}_gW"]), rtol=2e-4, atol=2e-6)
