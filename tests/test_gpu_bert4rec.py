"""GPU parity of the BERT4Rec path (pre-LN blocks, GELU FFN, <MASK> embedding, biased head, masked-position CE) against
the golden vectors of the real reference (tests/golden/bert4rec_*.npz).  Tolerances as in test_gpu_engine.py."""
import os

import pytest
import torch

from oracle import golden

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def cuda():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    return torch.device("cuda")


def _cos(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return float((a @ b) / (a.norm() * b.norm() + 1e-30))


def _flat(P):
    out = [("item_emb", P["item_emb"]), ("mask_emb", P["mask_emb"]), ("pos_emb", P["pos_emb"])]
    for i, b in enumerate(P["blocks"]):
        out += [(f"b{i}.{k}", b[k]) for k in ("ln1_w", "ln1_b", "in_w", "in_b", "out_w", "out_b", "ln2_w", "ln2_b", "w1", "b1", "w2", "b2")]
    if "head_w" in P:
        out.append(("head_w", P["head_w"]))
    out.append(("head_b", P["head_b"]))
    return out


@pytest.mark.parametrize("name", ["bert4rec_tiny.npz", "bert4rec_tiny_tied.npz"])
def test_bert4rec_train_step_matches_reference(golden_dir, cuda, name):
    from oracle import bert4rec as ob
    from replay_b200.engine_bert import Bert4RecEngine, BertConfig

    z = golden.load(os.path.join(golden_dir, name))
    sd = {k[4:]: torch.from_numpy(z[k]) for k in z if k.startswith("sd::")}
    P = ob.params_from_state_dict(sd)
    B, L = z["ids"].shape
    cfg = BertConfig(n_items=int(z["n_items"]), d=int(z["d"]), n_heads=int(z["H"]), n_blocks=int(z["n_blocks"]), max_len=L,
                     dropout=0.0, tying=bool(int(z["tying"])))
    eng = Bert4RecEngine(cfg, B, L, cuda)
    eng.load_canonical(P)
    ids, pm, tok = (torch.from_numpy(z[k]).cuda() for k in ("ids", "pad_mask", "token_mask"))
    labels = torch.from_numpy(z["labels"]).cuda()
    eng.set_batch(ids, pm, tok, labels)
    hid = eng.forward_hidden_all().float().cpu().view(B, L, -1)
    ref_h = torch.from_numpy(z["train_hidden"])
    real = torch.from_numpy(z["pad_mask"])
    assert (hid[real] - ref_h[real]).abs().max() < 6e-2  # pad query rows are never consumed
    loss = eng.forward_train()
    torch.cuda.synchronize()
    ref_loss = float(z["train_loss"])
    assert abs(loss[0].item() - ref_loss) < 5e-3 * ref_loss, (loss[0].item(), ref_loss)
    assert int(eng.n_valid.item()) == int((real & ~torch.from_numpy(z["token_mask"])).sum())
    eng.g32.zero_()
    eng.backward()
    torch.cuda.synchronize()
    Gref = ob.params_from_state_dict({k[6:]: torch.from_numpy(z[k]) for k in z if k.startswith("grad::")})
    G = eng.export_canonical(eng.grads)
    bad = []
    for (nm, a), (_, b) in zip(_flat(G), _flat(Gref)):
        if b.norm() < 1e-12:
            assert a.norm() < 1e-6, nm
            continue
        c, r = _cos(a, b), float(a.double().norm() / b.double().norm())
        if c < 0.995 or abs(r - 1) > 0.03:
            bad.append((nm, round(c, 5), round(r, 4)))
    assert not bad, bad


def test_bert4rec_predict_with_biased_head(golden_dir, cuda):
    from oracle import bert4rec as ob
    from oracle import sasrec as osr
    from replay_b200 import ops
    from replay_b200.engine_bert import Bert4RecEngine, BertConfig

    z = golden.load(os.path.join(golden_dir, "bert4rec_tiny.npz"))
    sd = {k[4:]: torch.from_numpy(z[k]) for k in z if k.startswith("sd::")}
    P = ob.params_from_state_dict(sd)
    B, L = z["ids"].shape
    n_items = int(z["n_items"])
    cfg = BertConfig(n_items=n_items, d=int(z["d"]), n_heads=int(z["H"]), n_blocks=int(z["n_blocks"]), max_len=L)
    eng = Bert4RecEngine(cfg, B, L, cuda, with_grad=False)
    eng.load_canonical(P)
    ids, pm, tok = (torch.from_numpy(z[k]) for k in ("ids", "pad_mask", "token_mask"))
    eng.set_batch(ids.cuda(), pm.cuda(), tok.cuda())
    hq = eng.forward_last_hidden()
    W16, bias = eng.head_for_scoring()
    # materialised logits of the reference's predict() on the same inputs
    ref_logits = torch.from_numpy(z["eval_logits"])
    ids_k, sc_k = ops.score_topk(hq, W16, 10, None, bias=bias)
    logits16 = hq.float().cpu() @ W16.float().cpu().T + bias[:n_items].cpu()
    ids_o = torch.argsort(-logits16.double(), dim=1, stable=True)[:, :10]
    assert torch.equal(ids_k.cpu(), ids_o)
    assert (sc_k.cpu() - torch.gather(ref_logits, 1, ids_k.cpu())).abs().max() < 0.1


def test_bert4rec_lightning_mirror(golden_dir, cuda):
    """Legacy Bert4Rec module: reference checkpoint keys, training_step on the reference batch layout, predict with the
    shifted window, fused top-k with candidates."""
    from replay_b200.models.nn.sequential import Bert4Rec
    from replay_b200.schema import TensorFeatureInfo, TensorSchema

    z = golden.load(os.path.join(golden_dir, "bert4rec_tiny.npz"))
    sd = {"_model." + k[4:]: torch.from_numpy(z[k]) for k in z if k.startswith("sd::")}
    n_items, d, H, L = int(z["n_items"]), int(z["d"]), int(z["H"]), int(z["L"])
    m = Bert4Rec(TensorSchema(TensorFeatureInfo("item_id", n_items, 0, d)), block_count=int(z["n_blocks"]), head_count=H,
                 hidden_size=d, max_seq_len=L, dropout_rate=0.0)
    m.load_state_dict(sd)
    ids, pm, tok = (torch.from_numpy(z[k]).cuda() for k in ("ids", "pad_mask", "token_mask"))
    batch = {"query_id": torch.arange(ids.shape[0]).view(-1, 1), "inputs": {"item_id": ids}, "pad_mask": pm, "token_mask": tok,
             "positive_labels": torch.from_numpy(z["labels"]).cuda()}
    loss = m.training_step(batch, 0)
    assert abs(float(loss) - float(z["train_loss"])) < 5e-3 * float(z["train_loss"])
    sd2 = m.state_dict()
    assert set(sd2) == set(sd)
    # prediction batches arrive already shifted from the reference's Bert4RecPredictionDataset (full length: taken as is)
    from replay_b200.models.nn.sequential.bert4rec import shift_features
    sids, spm, stm = shift_features(ids, pm, pm, 0)
    batch = {"query_id": batch["query_id"], "inputs": {"item_id": sids}, "pad_mask": spm, "token_mask": stm}
    scores = m.predict(batch)
    assert scores.shape == (ids.shape[0], n_items) and torch.isfinite(scores).all()
    torch.testing.assert_close(m.validation_step(batch, 0), scores)
    torch.testing.assert_close(m(batch["inputs"], spm, stm), scores)
    # a shorter (un-shifted) window is left-padded and shifted by the module (bert4rec/lightning.py:660-682)
    short = {"inputs": {"item_id": ids[:, 4:]}, "pad_mask": pm[:, 4:], "token_mask": pm[:, 4:]}
    sc_short = m.predict(short)
    keep = ~pm[:, :4].any(1)                       # rows whose 4 dropped positions were padding anyway
    assert keep.any()
    torch.testing.assert_close(sc_short[keep], scores[keep])
    with pytest.raises(ValueError):
        m.predict({"inputs": {"item_id": torch.cat([ids, ids[:, :1]], 1)}, "pad_mask": torch.cat([pm, pm[:, :1]], 1),
                   "token_mask": torch.cat([pm, pm[:, :1]], 1)})
    cands = torch.arange(5, 200, 3).cuda()
    top_ids, top_sc = m.predict_topk(batch, 7, seen_ids=ids, candidates_to_score=cands)
    assert set(top_ids.flatten().tolist()) <= set(cands.tolist())
    sc_c = m.predict(batch, candidates_to_score=cands)
    seen_mask = torch.zeros(ids.shape[0], n_items, dtype=torch.bool, device="cuda")
    seen_mask.scatter_(1, ids, True)
    sc_c = sc_c.masked_fill(seen_mask[:, cands], float("-inf"))
    ref_top = torch.argsort(-sc_c.double(), dim=1, stable=True)[:, :7]
    assert torch.equal(top_ids, cands[ref_top])
