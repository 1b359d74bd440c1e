"""GPU tests of the full-catalog BCE head (rp_bce_head_*): the kernels against fp64 on the same bf16 inputs over the ragged
shapes, run-to-run determinism, the API mirrors against the REAL reference (tests/golden/bce_losses.npz), CUDA-graph replay,
switching CE <-> BCE, training progress, and the config-2 / config-3 shapes without a [T_v, |I|] logits tensor."""
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


def _cos(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return float((a @ b) / (a.norm() * b.norm() + 1e-30))


def _rel(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / (b.norm() + 1e-300))


def _inputs(cap, n_valid, n_items, d, bias, seed, big_row=True):
    """bf16 hc / table, fp32 bias padded to 128 entries (zeros beyond the catalog), int32 labels; the first valid row is
    scaled so that its logits reach |s| ~ 80 (sigmoid / softplus far in saturation, where exp(s) would overflow a bf16 G)."""
    g = torch.Generator().manual_seed(seed)
    hc = torch.randn(cap, d, generator=g) * 0.5
    E = torch.randn(n_items, d, generator=g) * 0.1
    b = None
    if bias:
        b = torch.zeros((n_items + 127) // 128 * 128)
        b[:n_items] = torch.randn(n_items, generator=g) * 0.5
    if big_row:
        s0 = hc[0].bfloat16().float() @ E.bfloat16().float().T
        hc[0] *= 80.0 / float(s0.abs().max())
    labels = torch.randint(0, n_items, (cap,), generator=g, dtype=torch.int32)
    dev = torch.device("cuda")
    return (hc.bfloat16().to(dev), E.bfloat16().to(dev), None if b is None else b.to(dev), labels.to(dev),
            torch.tensor([n_valid], dtype=torch.int32, device=dev))


def _run(hc, E, b, labels, nv, n_valid_hint=0):
    from replay_b200.ops import BCEHeadState, bce_head_bwd, bce_head_fwd

    cap, d = hc.shape
    I = E.shape[0]
    st = BCEHeadState(cap, I, d, hc.device)
    d_hc = torch.full_like(hc, float("nan"))
    dE = torch.full((I, d), float("nan"), device=hc.device)
    db = None if b is None else torch.full((I,), float("nan"), device=hc.device)
    loss = bce_head_fwd(st, hc, E, labels, nv, d_hc, bias=b, n_valid_hint=n_valid_hint).clone()
    bce_head_bwd(st, hc, E, labels, nv, dE, bias=b, d_bias=db)
    torch.cuda.synchronize()
    return loss, d_hc, dE, db


def _reference(hc, E, b, labels, n, chunk=2048):
    """fp64 loss, dH [n, d], dE, db of the mean BCE over the first n rows, chunked over the rows, and the mean of
    sum_i softplus (the scale of the loss's fp32 rounding)."""
    Ed, I = E.double(), E.shape[0]
    bd = None if b is None else b[:I].double()
    loss, sp, dE, db = 0.0, 0.0, torch.zeros_like(Ed), torch.zeros(I, dtype=torch.float64, device=E.device)
    dH = torch.empty(n, E.shape[1], dtype=torch.float64, device=E.device)
    y = labels[:n].long()
    for lo in range(0, n, chunk):
        hi = min(n, lo + chunk)
        h = hc[lo:hi].double()
        s = h @ Ed.T
        if bd is not None:
            s += bd
        r = torch.arange(hi - lo, device=E.device)
        sp += float(torch.nn.functional.softplus(s).sum())
        loss += float(torch.nn.functional.softplus(s).sum() - s[r, y[lo:hi]].sum())
        G = torch.sigmoid(s)
        G[r, y[lo:hi]] -= 1.0
        G /= n
        dH[lo:hi] = G @ Ed
        dE += G.T @ h
        db += G.sum(0)
    return loss / n, dH, dE, db, sp / n


# (capacity, n_valid, n_items, d, bias): T and n_valid across the 128-row tile edges, ragged catalogs, one-tile and
# column-split fused passes (P = 1: a single item tile / a catalog of 129 items at 148 token tiles; P > 1: 50 000 items)
SHAPES = [(1, 1, 1, 64, False), (200, 127, 129, 128, True), (256, 128, 127, 256, False), (300, 129, 1, 128, True),
          (1000, 129, 50_000, 64, True), (5000, 4000, 50_000, 128, False), (4500, 4000, 127, 256, True),
          (20_000, 18_900, 129, 128, False), (5000, 3001, 50_000, 256, True)]


@pytest.mark.parametrize("cap,n_valid,n_items,d,bias", SHAPES)
def test_bce_head_matches_fp64(cuda, cap, n_valid, n_items, d, bias):
    # (a one-item catalog has only the positive: the saturated row's exact gradient there is ~1e-35, below any rounding)
    hc, E, b, labels, nv = _inputs(cap, n_valid, n_items, d, bias, seed=cap + n_items + d, big_row=n_items > 1)
    loss, d_hc, dE, db = _run(hc, E, b, labels, nv, n_valid_hint=n_valid)
    ref_loss, dH_ref, dE_ref, db_ref, sp = _reference(hc, E, b, labels, n_valid)
    assert torch.isfinite(loss).all() and abs(float(loss[0]) - ref_loss) < 2e-4 * sp, (float(loss[0]), ref_loss, sp)
    assert abs(float(loss[1]) - 1.0 / n_valid) < 1e-7 / n_valid
    assert _rel(d_hc[:n_valid], dH_ref) < 1e-2
    assert _rel(dE, dE_ref) < 1e-2
    if bias:
        assert _rel(db, db_ref) < 1e-2
    if n_items > 1:   # the saturated row: its gradient is still right (sigmoid = 1 or e^s, no overflow, no fall-back)
        assert _rel(d_hc[0], dH_ref[0]) < 1e-2


@pytest.mark.parametrize("cap,n_valid,n_items,d,bias", [(300, 200, 2000, 128, True), (5000, 4000, 3000, 64, False),
                                                         (20_000, 18_900, 129, 256, True)])
def test_bce_head_label_term(cuda, cap, n_valid, n_items, d, bias):
    """The loss is dominated by sum softplus; two calls that differ only in the labels isolate the label term: their losses
    differ by -mean(s_y - s_y') in fp64.  Labels: the largest and the smallest logit of each row (a difference of several
    units per row, far above the fp32 rounding of a loss of ~0.7 |I|)."""
    hc, E, b, _, nv = _inputs(cap, n_valid, n_items, d, bias, seed=7 + d, big_row=False)
    hc = (hc.float() * 2).bfloat16()
    s = hc.double() @ E.double().T + (0 if b is None else b[:n_items].double())
    y_hi, y_lo = s.argmax(1).int(), s.argmin(1).int()
    l_hi = _run(hc, E, b, y_hi, nv, n_valid)[0]
    l_lo = _run(hc, E, b, y_lo, nv, n_valid)[0]
    r = torch.arange(n_valid, device=cuda)
    want = -float((s[r, y_hi[:n_valid].long()] - s[r, y_lo[:n_valid].long()]).mean())
    got = float(l_hi[0]) - float(l_lo[0])
    assert abs(want) > 2.0
    assert abs(got - want) < 1e-3 * abs(want) + 1e-6 * abs(float(l_lo[0])), (got, want)


@pytest.mark.parametrize("cap,n_valid,n_items,d,bias", [(5000, 4000, 50_000, 128, True), (20_000, 18_900, 129, 64, False)])
def test_bce_head_run_to_run_determinism(cuda, cap, n_valid, n_items, d, bias):
    """Loss, dH, d_bias and dE bit-identical across repeats.  With distinct labels (first case) that holds for every row; with
    repeated labels (129 items) the one-hot scatter's float atomics add several rows of hc into one row of dE in a scheduling
    dependent order, so those rows agree to rounding and every other row bit for bit."""
    hc, E, b, labels, nv = _inputs(cap, n_valid, n_items, d, bias, seed=3)
    if n_items >= n_valid:
        labels[:n_valid] = torch.randperm(n_items, generator=torch.Generator().manual_seed(6))[:n_valid].int().to(cuda)
    runs = [_run(hc, E, b, labels, nv, n_valid) for _ in range(3)]
    bits = lambda t: t.view(torch.int32) if t.dtype == torch.float32 else t.view(torch.int16)  # noqa: E731
    shared = torch.zeros(n_items, dtype=torch.bool, device=cuda)
    if n_items < n_valid:
        shared[labels[:n_valid].long()] = True
    for r in runs[1:]:
        assert torch.equal(bits(r[0]), bits(runs[0][0])) and torch.equal(bits(r[1][:n_valid]), bits(runs[0][1][:n_valid]))
        if bias:
            assert torch.equal(bits(r[3]), bits(runs[0][3]))
        assert torch.equal(bits(r[2][~shared]), bits(runs[0][2][~shared]))
        torch.testing.assert_close(r[2][shared], runs[0][2][shared], rtol=1e-5, atol=1e-9)


# ------------------------------------------------------------------------------------------------ goldens through the mirrors
def _load(golden_dir, name):
    z = golden.load(os.path.join(golden_dir, name))
    return z, {k[4:]: torch.from_numpy(z[k]) for k in z if k.startswith("sd::")}


def _check_grads(pairs):
    for nm, a, b in pairs:
        c, r = _cos(a, b), float(a.double().norm() / b.double().norm())
        assert c > 0.995 and abs(r - 1) < 0.03, (nm, c, r)


def test_new_path_sasrec_bce_matches_reference(golden_dir, cuda):
    from replay_b200.nn.loss import BCE
    from replay_b200.nn.sequential import SasRec
    from replay_b200.schema import TensorFeatureInfo, TensorSchema

    z, sd = _load(golden_dir, "sasrec_new_tiny.npz")
    zb = np.load(os.path.join(golden_dir, "bce_losses.npz"))
    n_items, d, L = int(z["n_items"]), int(z["d"]), z["ids"].shape[1]
    model = SasRec.from_params(TensorSchema(TensorFeatureInfo("item_id", n_items, n_items, d)), embedding_dim=d,
                               num_heads=int(z["H"]), num_blocks=int(z["n_blocks"]), max_sequence_length=L, dropout=0.0,
                               device=cuda)
    model.load_state_dict(sd)
    model.loss = BCE()
    model.train()
    ids, pm = torch.from_numpy(z["ids"]).cuda(), torch.from_numpy(z["pad_mask"]).cuda()
    lab, tm = torch.from_numpy(z["labels"]).cuda(), torch.from_numpy(z["target_mask"]).cuda()
    out = model(feature_tensors={"item_id": ids}, padding_mask=pm, positive_labels=lab.unsqueeze(-1),
                target_padding_mask=tm.unsqueeze(-1))
    out["loss"].backward()
    torch.cuda.synchronize()
    ref = float(zb["new_loss"])
    assert abs(float(out["loss"]) - ref) < 5e-3 * abs(ref), (float(out["loss"]), ref)
    G = model.core.engine.export_canonical(model.core.engine.grads)
    _check_grads([("item_emb", G["item_emb"].cpu(), torch.from_numpy(zb["new_gE"])),
                  ("in_w", G["blocks"][0]["in_w"].cpu(), torch.from_numpy(zb["new_gW"]))])


def test_legacy_sasrec_bce_matches_reference(golden_dir, cuda):
    from replay_b200.models.nn.sequential import SasRec as LegacySasRec
    from replay_b200.schema import TensorFeatureInfo, TensorSchema

    z, sd = _load(golden_dir, "sasrec_legacy_tiny.npz")
    zb = np.load(os.path.join(golden_dir, "bce_losses.npz"))
    n_items, d, L = int(z["n_items"]), int(z["d"]), z["ids"].shape[1]
    # the legacy module's constructor keeps refusing loss_type="BCE" without a sample count; its core selects the head
    mod = LegacySasRec(TensorSchema(TensorFeatureInfo("item_id", n_items, n_items, d)), block_count=int(z["n_blocks"]),
                       head_count=int(z["H"]), hidden_size=d, max_seq_len=L, dropout_rate=0.0, fused_optimizer=False)
    mod._model.core.set_loss("bce")
    mod._model.load_state_dict(sd)
    batch = {"feature_tensor": {"item_id": torch.from_numpy(z["ids"]).cuda()}, "padding_mask": torch.from_numpy(z["pad_mask"]).cuda(),
             "positive_labels": torch.from_numpy(z["labels"]).cuda(), "target_padding_mask": torch.from_numpy(z["target_mask"]).cuda()}
    loss = mod.training_step(batch, 0)
    loss.backward()
    torch.cuda.synchronize()
    ref = float(zb["legacy_loss"])
    assert abs(float(loss) - ref) < 5e-3 * abs(ref), (float(loss), ref)
    eng = mod._model.core.engine
    G = eng.export_canonical(eng.grads)
    _check_grads([("item_emb", G["item_emb"].cpu(), torch.from_numpy(zb["legacy_gE"])),
                  ("in_w", G["blocks"][0]["in_w"].cpu(), torch.from_numpy(zb["legacy_gW"]))])


@pytest.mark.parametrize("name,key", [("bert4rec_tiny.npz", "bert"), ("bert4rec_tiny_tied.npz", "bert_tied")])
def test_bert4rec_bce_matches_reference(golden_dir, cuda, name, key):
    from replay_b200.models.nn.sequential import Bert4Rec
    from replay_b200.schema import TensorFeatureInfo, TensorSchema

    z, sd = _load(golden_dir, name)
    zb = np.load(os.path.join(golden_dir, "bce_losses.npz"))
    n_items, d, L = int(z["n_items"]), int(z["d"]), z["ids"].shape[1]
    tying = bool(int(z["tying"]))
    mod = Bert4Rec(TensorSchema(TensorFeatureInfo("item_id", n_items, 0, d)), block_count=int(z["n_blocks"]), head_count=int(z["H"]),
                   hidden_size=d, max_seq_len=L, dropout_rate=0.0, enable_embedding_tying=tying, loss_type="BCE",
                   fused_optimizer=False)
    mod._model.load_state_dict(sd)
    batch = {"inputs": {"item_id": torch.from_numpy(z["ids"]).cuda()}, "pad_mask": torch.from_numpy(z["pad_mask"]).cuda(),
             "token_mask": torch.from_numpy(z["token_mask"]).cuda(), "positive_labels": torch.from_numpy(z["labels"]).cuda()}
    loss = mod.training_step(batch, 0)
    loss.backward()
    torch.cuda.synchronize()
    ref = float(zb[f"{key}_loss"])
    assert abs(float(loss) - ref) < 5e-3 * abs(ref), (float(loss), ref)
    eng = mod._model.core.engine
    G = eng.export_canonical(eng.grads)
    pairs = [("item_emb", G["item_emb"].cpu(), torch.from_numpy(zb[f"{key}_gE"])),
             ("in_w", G["blocks"][0]["in_w"].cpu(), torch.from_numpy(zb[f"{key}_gW"])),
             ("head_b", G["head_b"].cpu(), torch.from_numpy(zb[f"{key}_gb"]))]
    if not tying:
        pairs.append(("head_w", G["head_w"].cpu(), torch.from_numpy(zb[f"{key}_gHW"])))
    _check_grads(pairs)


# ------------------------------------------------------------------------------------------------ training paths
def _core(cuda, seed=4, I=500, d=64, L=32):
    from replay_b200.core import SasRecCore
    from replay_b200.engine import EncoderConfig

    return SasRecCore(EncoderConfig(n_items=I, d=d, n_heads=1, n_blocks=2, max_len=L, dropout=0.0, variant="new"),
                      device=cuda, seed=seed)


def _batch(seed, B=8, I=500, L=32):
    from replay_b200.synthetic import make_sequences

    return [t.cuda() for t in make_sequences(B, I, L, seed=seed)]


def test_bce_graph_replay_matches_eager_steps(cuda):
    """fused_step captured in a CUDA graph (two eager warm-up steps, capture, replay) against eager steps: 4 steps."""
    cores = [_core(cuda), _core(cuda)]
    cores[1].use_cuda_graph = False
    losses = [[], []]
    for k, core in enumerate(cores):
        core.set_loss("bce")
        for step in range(4):
            losses[k].append(float(core.fused_step(*_batch(100 + step), lr=2e-3)))
    torch.cuda.synchronize()
    np.testing.assert_allclose(losses[0], losses[1], rtol=1e-5)
    assert cores[0]._trainer._g_fb is not None   # the graph path really ran
    torch.testing.assert_close(cores[0].flat.detach(), cores[1].flat.detach(), rtol=0, atol=2e-5)


def test_switching_ce_bce_ce_matches_fresh_models(cuda):
    """CE -> BCE -> CE on one model (the captured graphs are dropped at each switch) gives the losses of fresh models;
    lr = 0 keeps the parameters fixed across the steps."""
    b = _batch(7)
    fresh = {}
    for kind in ("ce", "bce"):
        core = _core(cuda)
        core.set_loss(kind)
        fresh[kind] = [float(core.fused_step(*b, lr=0.0)) for _ in range(3)]
    core = _core(cuda)
    got = []
    for kind in ("ce", "bce", "ce"):
        core.set_loss(kind)
        got.append((kind, [float(core.fused_step(*b, lr=0.0)) for _ in range(3)]))
    torch.cuda.synchronize()
    assert fresh["bce"][0] > 10 * fresh["ce"][0]   # really two different losses (BCE sums over the catalog)
    for kind, ls in got:
        np.testing.assert_allclose(ls, fresh[kind], rtol=1e-6, err_msg=kind)


def test_bce_training_makes_progress(cuda):
    """30 training_step calls of the Lightning mirror with BCE() (fused forward + backward + Adam) reduce the loss."""
    from replay_b200.nn.lightning import LightningModule, OptimizerFactory
    from replay_b200.nn.loss import BCE
    from replay_b200.nn.sequential import SasRec
    from replay_b200.schema import TensorFeatureInfo, TensorSchema

    I, L = 400, 32
    model = SasRec.from_params(TensorSchema(TensorFeatureInfo("item_id", I, I, 64)), embedding_dim=64, num_heads=1,
                               num_blocks=2, max_sequence_length=L, dropout=0.0, device=cuda)
    model.loss = BCE()
    lm = LightningModule(model, optimizer_factory=OptimizerFactory(learning_rate=3e-3))
    ids, pm, lab, tm = _batch(11, B=16, I=I, L=L)
    b = {"feature_tensors": {"item_id": ids}, "padding_mask": pm, "positive_labels": lab.unsqueeze(-1),
         "target_padding_mask": tm.unsqueeze(-1)}
    ls = [float(lm.training_step(b, i)) for i in range(30)]
    assert all(np.isfinite(ls)) and ls[-1] < 0.7 * ls[0], (ls[0], ls[-1])


# ------------------------------------------------------------------------------------------------ full shapes
def test_c2_bce_train_step_full_shape(cuda):
    """Config 2 (512 sequences x 200, d = 128, 50 K items) through the SASRec engine with the BCE head: the loss of all valid
    targets against a chunked fp64 restatement on the engine's own bf16 head inputs, dH on a token subsample, dE on an item
    subsample; the head allocates far less than one [T_v, |I|] fp32 logits tensor."""
    from oracle import sasrec as osr
    from replay_b200.engine import EncoderConfig, SasRecEngine
    from replay_b200.ops import bce_head_bwd, bce_head_fwd
    from replay_b200.synthetic import make_sequences

    B, L, d, H, I = 512, 200, 128, 2, 50_000
    eng = SasRecEngine(EncoderConfig(n_items=I, d=d, n_heads=H, n_blocks=2, max_len=L, dropout=0.0, variant="new"), B, L, cuda)
    eng.load_canonical(osr.random_params(I, d, L, 2, seed=3))
    eng.set_loss("bce")
    ids, pm, lab, tm = make_sequences(B, I, L, seed=1234)
    eng.set_batch(ids.cuda(), pm.cuda(), lab.cuda(), tm.cuda())
    eng.n_valid_hint = int(tm.sum())
    loss = eng.forward_train()
    eng.g32.zero_()
    eng.backward()
    torch.cuda.synchronize()
    n = int(eng.n_valid.item())
    assert n == int(tm.sum())
    tb = eng.params16["item_emb"][:I]
    hcd, y = eng.hc[:n].double(), eng.labels_c[:n].long()
    Ed = tb.double()
    tot = 0.0
    for lo in range(0, n, 4096):
        s = hcd[lo:lo + 4096] @ Ed.T
        tot += float(torch.nn.functional.softplus(s).sum() - s.gather(1, y[lo:lo + 4096, None]).sum())
    ref_loss = tot / n
    assert abs(float(loss[0]) - ref_loss) < 2e-4 * abs(ref_loss), (float(loss[0]), ref_loss)
    # dH on a token subsample
    tsel = torch.arange(0, n, 53, device=cuda)
    G = torch.sigmoid(hcd[tsel] @ Ed.T)
    G[torch.arange(tsel.numel(), device=cuda), y[tsel]] -= 1.0
    assert _rel(eng.s["dhc"][tsel], (G @ Ed) / n) < 1e-2
    # dE on an item subsample (every kind of tile position + the most popular labels), the head alone into a scratch table
    isel = torch.unique(torch.cat([torch.arange(0, I, 997, device=cuda), torch.tensor([0, 127, 128, I - 1], device=cuda),
                                   torch.bincount(y, minlength=I).topk(16).indices]))
    acc = torch.zeros(isel.numel(), d, device=cuda, dtype=torch.float64)
    for lo in range(0, n, 8192):
        pp = torch.sigmoid(hcd[lo:lo + 8192] @ Ed[isel].T)
        pp -= (y[lo:lo + 8192, None] == isel[None, :]).double()
        acc += pp.T @ hcd[lo:lo + 8192]
    scratch = torch.zeros(I, d, device=cuda)
    d_hc2 = torch.zeros_like(eng.s["dhc"])
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    bce_head_fwd(eng.bce, eng.hc, tb, eng.labels_c, eng.n_valid, d_hc2, n_valid_hint=n)
    bce_head_bwd(eng.bce, eng.hc, tb, eng.labels_c, eng.n_valid, scratch)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    assert peak < 0.01 * n * I * 4, (peak, n * I * 4)
    assert eng.bce.ws_bytes < 0.1 * n * I * 4, (eng.bce.ws_bytes, n * I * 4)   # the preallocated workspace, all included
    assert _rel(scratch[isel], acc / n) < 1e-2


def test_c3_bce_head_with_bias_full_shape(cuda):
    """Config 3 head shape with a bias (BERT4Rec's untied head): |I| = 100 K, d = 256, ~4 K masked targets."""
    I, d, cap, n = 100_000, 256, 4608, 4100
    hc, E, b, labels, nv = _inputs(cap, n, I, d, True, seed=33, big_row=False)
    loss, d_hc, dE, db = _run(hc, E, b, labels, nv, n_valid_hint=n)
    hcd, Ed, y = hc[:n].double(), E.double(), labels[:n].long()
    bd = b[:I].double()
    tot = 0.0
    for lo in range(0, n, 1024):
        s = hcd[lo:lo + 1024] @ Ed.T + bd
        tot += float(torch.nn.functional.softplus(s).sum() - s.gather(1, y[lo:lo + 1024, None]).sum())
    assert abs(float(loss[0]) - tot / n) < 2e-4 * abs(tot / n)
    tsel = torch.arange(0, n, 37, device=cuda)
    G = torch.sigmoid(hcd[tsel] @ Ed.T + bd)
    G[torch.arange(tsel.numel(), device=cuda), y[tsel]] -= 1.0
    assert _rel(d_hc[tsel], (G @ Ed) / n) < 1e-2
    isel = torch.unique(torch.cat([torch.arange(0, I, 1999, device=cuda), torch.tensor([0, 127, 128, I - 1], device=cuda), y[:8]]))
    P = torch.sigmoid(hcd @ Ed[isel].T + bd[isel])
    P -= (y[:, None] == isel[None, :]).double()
    assert _rel(dE[isel], (P.T @ hcd) / n) < 1e-2
    assert _rel(db[isel], P.sum(0) / n) < 1e-2
