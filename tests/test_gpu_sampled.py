"""GPU tests of the sampled training heads (rp_sampled_head_*, SURVEY.md §8 a9/f.2) against losses and gradients produced by
the REAL reference classes (tests/golden/sampled_losses.npz) and against the restatement (oracle/sampled.py) at larger sizes."""
import os

import numpy as np
import pytest
import torch

from oracle import golden

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def cuda():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    return torch.device("cuda")


def _load(golden_dir, name):
    z = golden.load(os.path.join(golden_dir, name))
    return z, {k[4:]: torch.from_numpy(z[k]) for k in z if k.startswith("sd::")}


def _cos(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return float((a @ b) / (a.norm() * b.norm() + 1e-30))


def _engine(z, P, variant, cuda):
    from replay_b200.engine import EncoderConfig, SasRecEngine
    B, L = z["ids"].shape
    cfg = EncoderConfig(n_items=int(z["n_items"]), d=int(z["d"]), n_heads=int(z["H"]), n_blocks=int(z["n_blocks"]), max_len=L,
                        dropout=0.0, variant=variant)
    eng = SasRecEngine(cfg, B, L, cuda)
    eng.load_canonical(P)
    return eng


def _run(eng, z, neg):
    ids, pm = torch.from_numpy(z["ids"]).cuda(), torch.from_numpy(z["pad_mask"]).cuda()
    lab, tm = torch.from_numpy(z["labels"]).cuda(), torch.from_numpy(z["target_mask"]).cuda()
    eng.set_batch(ids, pm, lab, tm)
    eng.set_negatives(neg.cuda())
    loss = eng.forward_train()
    eng.g32.zero_()
    eng.grads["item_emb"].fill_(3.0)  # like the full-CE head, the sampled head owns (overwrites) the table gradient
    eng.backward()
    torch.cuda.synchronize()
    return float(loss[0]), eng.export_canonical(eng.grads)


@pytest.mark.parametrize("loss", ["ce", "bce"])
@pytest.mark.parametrize("shape", ["shared", "perseq", "perpos"])
def test_new_path_sampled_heads_match_reference(golden_dir, cuda, loss, shape):
    from oracle import sasrec as osr
    z, sd = _load(golden_dir, "sasrec_new_tiny.npz")
    zs = np.load(os.path.join(golden_dir, "sampled_losses.npz"))
    eng = _engine(z, osr.params_from_new_state_dict(sd), "new", cuda)
    neg = torch.from_numpy(zs["neg_" + shape])
    eng.set_loss(loss + "_sampled", n_neg=neg.shape[-1], neg_shape=shape, ignore_index=int(zs["ignore_index"]))
    l, G = _run(eng, z, neg)
    ref = float(zs[f"new_{loss}_{shape}_loss"])
    assert abs(l - ref) < 5e-3 * abs(ref), (l, ref)
    gE, gW = torch.from_numpy(zs[f"new_{loss}_{shape}_gE"]), torch.from_numpy(zs[f"new_{loss}_{shape}_gW"])
    for nm, a, b in (("item_emb", G["item_emb"].cpu(), gE), ("in_w", G["blocks"][0]["in_w"].cpu(), gW)):
        c, r = _cos(a, b), float(a.double().norm() / b.double().norm())
        assert c > 0.995 and abs(r - 1) < 0.03, (nm, c, r)
    # rows of the table that are neither a positive, a negative nor an input stay exactly zero (sparse gradient)
    touched = torch.zeros(gE.shape[0], dtype=torch.bool)
    touched[gE.abs().sum(1) > 0] = True
    assert (G["item_emb"].cpu()[~touched] == 0).all()


@pytest.mark.parametrize("loss", ["ce", "bce"])
def test_legacy_sampled_heads_match_reference(golden_dir, cuda, loss):
    from oracle import sasrec as osr
    z, sd = _load(golden_dir, "sasrec_legacy_tiny.npz")
    zs = np.load(os.path.join(golden_dir, "sampled_losses.npz"))
    eng = _engine(z, osr.params_from_legacy_state_dict(sd), "legacy", cuda)
    tm = torch.from_numpy(z["target_mask"])
    nv = torch.from_numpy(zs[f"legacy_{loss}_neg"])
    neg = torch.zeros(*tm.shape, nv.shape[1], dtype=torch.int64)
    neg[tm] = nv
    eng.set_loss(f"legacy_{loss}_sampled", n_neg=nv.shape[1], neg_shape="perpos")
    l, G = _run(eng, z, neg)
    ref = float(zs[f"legacy_{loss}_loss"])
    assert abs(l - ref) < 5e-3 * abs(ref), (l, ref)
    for nm, a, b in (("item_emb", G["item_emb"].cpu(), torch.from_numpy(zs[f"legacy_{loss}_gE"])),
                     ("in_w", G["blocks"][0]["in_w"].cpu(), torch.from_numpy(zs[f"legacy_{loss}_gW"]))):
        c, r = _cos(a, b), float(a.double().norm() / b.double().norm())
        assert c > 0.995 and abs(r - 1) < 0.03, (nm, c, r)


@pytest.mark.parametrize("kind,shape,N", [("ce_sampled", "shared", 1000), ("bce_sampled", "shared", 257), ("ce_sampled", "perpos", 64),
                                          ("legacy_ce_sampled", "perseq", 100), ("legacy_bce_sampled", "shared", 512)])
def test_sampled_heads_against_restatement_config2_shape(cuda, kind, shape, N):
    """L = 200, d = 128, H = 2 (config 2 model shape) at a 20K catalog: loss and gradients vs oracle/sampled.py."""
    from oracle import sampled as osm
    from oracle import sasrec as osr
    from replay_b200.engine import EncoderConfig, SasRecEngine
    from replay_b200.synthetic import make_sequences
    B, L, d, H, I = 6, 200, 128, 2, 20_000
    P = osr.random_params(I, d, L, 2, seed=3)
    ids, pm, lab, tm = make_sequences(B, I, L, seed=9)
    g = torch.Generator().manual_seed(N)
    neg = {"shared": lambda: torch.randint(0, I, (N,), generator=g), "perseq": lambda: torch.randint(0, I, (B, N), generator=g),
           "perpos": lambda: torch.randint(0, I, (B, L, N), generator=g)}[shape]()
    if shape == "shared":
        neg[:5] = lab[tm][:5]  # collisions with some positives
    eng = SasRecEngine(EncoderConfig(n_items=I, d=d, n_heads=H, n_blocks=2, max_len=L, dropout=0.0, variant="new"), B, L, cuda)
    eng.load_canonical(P)
    eng.set_loss(kind, n_neg=N, neg_shape=shape)
    eng.set_batch(ids.cuda(), pm.cuda(), lab.cuda(), tm.cuda())
    eng.set_negatives(neg.cuda())
    loss = eng.forward_train()
    eng.backward()
    torch.cuda.synchronize()
    okind = kind.replace("_sampled", "")
    kw = dict(vocab_size=I) if okind == "legacy_ce" else {}
    ref, Gref = osm.loss_and_grads(P, ids, pm, lab, tm, neg, H, okind, **kw)
    assert abs(float(loss[0]) - float(ref)) < 5e-3 * abs(float(ref)), (float(loss[0]), float(ref))
    G = eng.export_canonical(eng.grads)
    bad = []
    for k, (a, b) in enumerate(zip(osr.flat_param_list(G), osr.flat_param_list(Gref))):
        if b.norm() < 1e-12:
            continue
        c, r = _cos(a.cpu(), b), float(a.double().norm().cpu() / b.double().norm())
        if c < 0.99 or abs(r - 1) > 0.04:
            bad.append((k, round(c, 5), round(r, 4)))
    assert not bad, bad


def test_api_mirrors_select_the_sampled_heads(golden_dir, cuda):
    """replay_b200.nn.loss.CESampled on the new-path module (reference key: SasRec.loss) and loss_sample_count on the legacy
    module; a few fused steps must reduce the loss."""
    from replay_b200.models.nn.sequential import SasRec as LegacySasRec
    from replay_b200.nn.loss import BCESampled, CESampled
    from replay_b200.nn.sequential import SasRec
    from replay_b200.schema import TensorFeatureInfo, TensorSchema
    z, sd = _load(golden_dir, "sasrec_new_tiny.npz")
    zs = np.load(os.path.join(golden_dir, "sampled_losses.npz"))
    n_items, d, H, L = int(z["n_items"]), int(z["d"]), int(z["H"]), int(z["L"])
    model = SasRec.from_params(TensorSchema(TensorFeatureInfo("item_id", n_items, n_items, d)), embedding_dim=d, num_heads=H,
                               num_blocks=int(z["n_blocks"]), max_sequence_length=L, dropout=0.0)
    model.load_state_dict(sd)
    ids, pm = torch.from_numpy(z["ids"]).cuda(), torch.from_numpy(z["pad_mask"]).cuda()
    lab, tm = torch.from_numpy(z["labels"]).cuda(), torch.from_numpy(z["target_mask"]).cuda()
    model.train()
    for spec, key in ((CESampled(negative_labels_ignore_index=int(zs["ignore_index"])), "new_ce_perseq_loss"),
                      (BCESampled(negative_labels_ignore_index=int(zs["ignore_index"])), "new_bce_perseq_loss")):
        model.loss = spec
        out = model(feature_tensors={"item_id": ids}, padding_mask=pm, positive_labels=lab.unsqueeze(-1),
                    negative_labels=torch.from_numpy(zs["neg_perseq"]).cuda(), target_padding_mask=tm.unsqueeze(-1))
        ref = float(zs[key])
        assert abs(out["loss"].item() - ref) < 5e-3 * ref
        out["loss"].backward()
        assert model.core.flat.grad is not None and torch.isfinite(model.core.flat.grad).all()
        model.core.flat.grad = None
    with pytest.raises(ValueError):
        model(feature_tensors={"item_id": ids}, padding_mask=pm, positive_labels=lab.unsqueeze(-1), target_padding_mask=tm.unsqueeze(-1))
    # Lightning mirror, fused forward+backward+Adam with per-batch shared negatives
    from replay_b200.nn.lightning import LightningModule, OptimizerFactory
    model.loss = CESampled()
    lm = LightningModule(model, optimizer_factory=OptimizerFactory(learning_rate=3e-3))
    g = torch.Generator().manual_seed(1)
    b = {"feature_tensors": {"item_id": ids}, "padding_mask": pm, "positive_labels": lab.unsqueeze(-1),
         "target_padding_mask": tm.unsqueeze(-1)}
    ls = [float(lm.training_step({**b, "negative_labels": torch.randint(0, n_items, (50,), generator=g).cuda()}, i)) for i in range(40)]
    assert ls[-1] < ls[0] - 0.5, (ls[0], ls[-1])
    with pytest.raises(ValueError):
        lm.training_step(b, 0)
    # legacy module: CE with 64 sampled negatives per position / shared BCE negatives
    for kw in (dict(loss_type="CE", loss_sample_count=64), dict(loss_type="BCE", loss_sample_count=32, negatives_sharing=True)):
        torch.manual_seed(0)
        leg = LegacySasRec(TensorSchema(TensorFeatureInfo("item_id", n_items, 0, d)), block_count=1, head_count=1, hidden_size=d,
                           max_seq_len=L, dropout_rate=0.0, **kw)
        b = {"feature_tensor": {"item_id": ids.clamp(max=n_items - 1)}, "padding_mask": pm, "positive_labels": lab.clamp(max=n_items - 1),
             "target_padding_mask": tm}
        losses = [float(leg.training_step(b, i)) for i in range(30)]
        assert losses[-1] < losses[0] - 0.3, (kw, losses[0], losses[-1])
    with pytest.raises(NotImplementedError):
        LegacySasRec(TensorSchema(TensorFeatureInfo("item_id", n_items, 0, d)), loss_type="CE", loss_sample_count=8,
                     negative_sampling_strategy="inbatch")


# ------------------------------------------------------------------------------------------------ full-catalog per-row losses (§8 f.2)
ROW_CASES = {"logout": ("LogOutCE", {}), "logout_weighted": ("LogOutCEWeighted", dict(feature_name="w")),
             "ce_weighted": ("CEWeighted", dict(feature_name="w")), "login": ("LogInCE", {}),
             "login_clamped": ("LogInCE", dict(log_epsilon=1e-3, clamp_border=5.5))}


@pytest.mark.parametrize("case", sorted(ROW_CASES))
@pytest.mark.parametrize("fused", [True, False])
def test_row_losses_match_reference(golden_dir, cuda, case, fused):
    """LogOutCE / LogOutCEWeighted / CEWeighted / LogInCE through the new-path mirror (SasRec.loss = selector) against loss and
    gradients of the REAL reference classes; ``fused=False`` forces the two-pass head (separate code path for the weights)."""
    from oracle import sasrec as osr
    from replay_b200 import nn as _nn  # noqa: F401
    from replay_b200.nn import loss as L
    from replay_b200.nn.sequential import SasRec
    from replay_b200.schema import TensorFeatureInfo, TensorSchema

    z, sd = _load(golden_dir, "sasrec_new_tiny.npz")
    zr = np.load(os.path.join(golden_dir, "row_losses.npz"))
    n_items, d = int(z["n_items"]), int(z["d"])
    Lmax = z["ids"].shape[1]
    model = SasRec.from_params(TensorSchema(TensorFeatureInfo("item_id", n_items, n_items, d)), embedding_dim=d,
                               num_heads=int(z["H"]), num_blocks=int(z["n_blocks"]), max_sequence_length=Lmax, dropout=0.0,
                               device=cuda)
    model.load_state_dict(sd)
    cls, kw = ROW_CASES[case]
    if cls != "CEWeighted":
        kw = dict(kw, cardinality=n_items)
    model.loss = getattr(L, cls)(**kw)
    model.train()
    ids, pm = torch.from_numpy(z["ids"]).cuda(), torch.from_numpy(z["pad_mask"]).cuda()
    lab, tm = torch.from_numpy(z["labels"]).cuda(), torch.from_numpy(z["target_mask"]).cuda()
    w = torch.from_numpy(zr["weights"]).cuda()
    eng = model.core.ensure_engine(ids.shape[0], Lmax, with_grad=True)
    eng.fused_ce = fused
    out = model(feature_tensors={"item_id": ids, "w": w}, padding_mask=pm, positive_labels=lab.unsqueeze(-1),
                target_padding_mask=tm.unsqueeze(-1))
    out["loss"].backward()
    torch.cuda.synchronize()
    ref = float(zr[f"{case}_loss"])
    assert abs(float(out["loss"]) - ref) < 5e-3 * abs(ref), (float(out["loss"]), ref)
    G = eng.export_canonical(eng.grads)
    gE, gW = torch.from_numpy(zr[f"{case}_gE"]), torch.from_numpy(zr[f"{case}_gW"])
    for nm, a, b in (("item_emb", G["item_emb"].cpu(), gE), ("in_w", G["blocks"][0]["in_w"].cpu(), gW)):
        c, r = _cos(a, b), float(a.double().norm() / b.double().norm())
        assert c > 0.995 and abs(r - 1) < 0.03, (nm, c, r)
