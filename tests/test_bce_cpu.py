"""CPU tests of the full-catalog BCE head: the plain-torch restatement (oracle/bce.py) against the REAL reference classes
(tests/golden/bce_losses.npz), the C-ABI argument errors of rp_bce_head_*, and how the loss selectors and the legacy modules
choose the head.  No kernel is launched here."""
import ctypes
import os

import numpy as np
import pytest
import torch

from oracle import bce as obce
from oracle import bert4rec as ob
from oracle import golden
from oracle import sasrec as osr
from replay_b200.schema import TensorFeatureInfo, TensorSchema


def _schema(n=300, d=64, pad=None):
    return TensorSchema(TensorFeatureInfo("item_id", n, n if pad is None else pad, d))


def _load(golden_dir, name):
    z = golden.load(os.path.join(golden_dir, name))
    return z, {k[4:]: torch.from_numpy(z[k]) for k in z if k.startswith("sd::")}


# ------------------------------------------------------------------------------------------------ restatement vs reference
@pytest.mark.parametrize("variant", ["new", "legacy"])
def test_sasrec_bce_restatement_matches_reference(golden_dir, variant):
    """New path ``SasRec.loss = BCE()`` and legacy ``SasRec(loss_type="BCE")._compute_loss_bce``."""
    z, sd = _load(golden_dir, f"sasrec_{variant}_tiny.npz")
    zb = np.load(os.path.join(golden_dir, "bce_losses.npz"))
    P = osr.params_from_new_state_dict(sd) if variant == "new" else osr.params_from_legacy_state_dict(sd)
    ids, pm = torch.from_numpy(z["ids"]), torch.from_numpy(z["pad_mask"])
    labels, tm = torch.from_numpy(z["labels"]), torch.from_numpy(z["target_mask"])
    loss, G = obce.sasrec_loss_and_grads(P, ids, pm, labels, tm, int(z["H"]), variant)
    torch.testing.assert_close(loss, torch.from_numpy(zb[f"{variant}_loss"]), rtol=2e-5, atol=2e-6)
    torch.testing.assert_close(G["item_emb"], torch.from_numpy(zb[f"{variant}_gE"]), rtol=2e-4, atol=2e-6)
    torch.testing.assert_close(G["blocks"][0]["in_w"], torch.from_numpy(zb[f"{variant}_gW"]), rtol=2e-4, atol=2e-6)


@pytest.mark.parametrize("name,key", [("bert4rec_tiny.npz", "bert"), ("bert4rec_tiny_tied.npz", "bert_tied")])
def test_bert4rec_bce_restatement_matches_reference(golden_dir, name, key):
    """``Bert4Rec(loss_type="BCE")._compute_loss_bce``, untied (Linear with bias) and tied (item table + out_bias)."""
    z, sd = _load(golden_dir, name)
    zb = np.load(os.path.join(golden_dir, "bce_losses.npz"))
    P = ob.params_from_state_dict(sd)
    leaves = [P["item_emb"], P["head_b"], P["blocks"][0]["in_w"]] + ([P["head_w"]] if "head_w" in P else [])
    for t in leaves:
        t.requires_grad_(True)
    ids, pm, tok = (torch.from_numpy(z[k]) for k in ("ids", "pad_mask", "token_mask"))
    loss = obce.bert4rec_loss(P, ids, pm, tok, torch.from_numpy(z["labels"]), int(z["H"]))
    loss.backward()
    torch.testing.assert_close(loss.detach(), torch.from_numpy(zb[f"{key}_loss"]), rtol=2e-5, atol=2e-6)
    torch.testing.assert_close(P["item_emb"].grad, torch.from_numpy(zb[f"{key}_gE"]), rtol=2e-4, atol=2e-6)
    torch.testing.assert_close(P["head_b"].grad, torch.from_numpy(zb[f"{key}_gb"]), rtol=2e-4, atol=2e-6)
    torch.testing.assert_close(P["blocks"][0]["in_w"].grad, torch.from_numpy(zb[f"{key}_gW"]), rtol=2e-4, atol=2e-6)
    if "head_w" in P:
        torch.testing.assert_close(P["head_w"].grad, torch.from_numpy(zb[f"{key}_gHW"]), rtol=2e-4, atol=2e-6)


def test_bce_restatement_is_softplus_minus_label_logit():
    """The closed form the kernels compute: (1/M) sum_t [ sum_i softplus(s_ti) - s_t,y_t ], incl. |s| far beyond exp's range."""
    g = torch.Generator().manual_seed(0)
    h = torch.randn(2, 5, 8, generator=g, dtype=torch.float64) * 4
    E = torch.randn(40, 8, generator=g, dtype=torch.float64) * 4
    y = torch.randint(0, 40, (2, 5), generator=g)
    tm = torch.rand(2, 5, generator=g) > 0.3
    s = h[tm] @ E.T
    want = (torch.nn.functional.softplus(s).sum(-1) - s.gather(1, y[tm][:, None])[:, 0]).mean()
    got = obce.bce_full(h, E, y, tm)
    assert float(s.abs().max()) > 80
    torch.testing.assert_close(got, want, rtol=1e-10, atol=0.0)


# ------------------------------------------------------------------------------------------------ C ABI
def test_bce_head_c_abi_argument_errors_without_a_gpu():
    """rp_bce_head_* follow include/rp_b200.h's error convention; every check is decided before any CUDA call."""
    from replay_b200._lib import lib

    L = lib()
    EINVAL, ESHAPE, EWORKSPACE = -1, -2, -5
    ws = L.rp_bce_head_workspace(1024, 5000, 128)
    assert 0 < ws < L.rp_bce_head_workspace(2048, 5000, 128)
    assert L.rp_bce_head_workspace(1024, 5000, 64) < ws < L.rp_bce_head_workspace(1024, 5000, 256)
    assert L.rp_bce_head_workspace(0, 5000, 128) == 0 and L.rp_bce_head_workspace(1024, 0, 128) == 0
    assert L.rp_bce_head_workspace(1024, 5000, 512) == 0
    buf = ctypes.create_string_buffer(64)
    p = ctypes.cast(buf, ctypes.c_void_p)
    big = 1 << 40
    # NULL pointers (d_hc is required: the forward is one fused forward + dH pass)
    assert L.rp_bce_head_fwd(None, None, None, None, None, 1, 1, 128, None, None, 0, None, 0, None) == EINVAL
    assert L.rp_bce_head_fwd(p, p, None, p, p, 128, 100, 128, p, None, 0, p, big, None) == EINVAL
    assert L.rp_bce_head_fwd(p, p, None, p, p, 128, 100, 128, p, p, 0, None, big, None) == EINVAL
    assert L.rp_bce_head_bwd(None, None, None, None, None, 1, 1, 128, None, None, None, None, 0, None) == EINVAL
    assert L.rp_bce_head_bwd(p, p, p, p, p, 128, 100, 128, p, p, None, p, big, None) == EINVAL    # bias without d_bias
    assert L.rp_bce_head_bwd(p, p, None, p, p, 128, 100, 128, p, p, p, p, big, None) == EINVAL    # d_bias without bias
    # shapes: d in {64, 128, 256}; d = 512 is not built
    for d in (96, 512):
        assert L.rp_bce_head_fwd(p, p, None, p, p, 128, 100, d, p, p, 0, p, big, None) == ESHAPE
        assert L.rp_bce_head_bwd(p, p, None, p, p, 128, 100, d, p, p, None, p, big, None) == ESHAPE
    assert L.rp_bce_head_fwd(p, p, None, p, p, 0, 100, 128, p, p, 0, p, big, None) == ESHAPE
    assert L.rp_bce_head_fwd(p, p, None, p, p, 128, 0, 128, p, p, 0, p, big, None) == ESHAPE
    # a workspace one byte short
    need = L.rp_bce_head_workspace(128, 100, 128)
    assert L.rp_bce_head_fwd(p, p, None, p, p, 128, 100, 128, p, p, 0, p, need - 1, None) == EWORKSPACE
    assert L.rp_bce_head_bwd(p, p, None, p, p, 128, 100, 128, p, p, None, p, need - 1, None) == EWORKSPACE


# ------------------------------------------------------------------------------------------------ selectors and modules
def test_bce_selector_constructor():
    from replay_b200.nn.loss import BCE

    spec = BCE()
    assert spec.kind == "bce" and not spec.needs_negatives and spec.engine_kwargs() == {}
    spec.logits_callback = len   # the LossProto surface: assignable, never called by the fused path
    assert spec.logits_callback is len
    for kw in (dict(weight=torch.ones(3)), dict(pos_weight=torch.ones(3)), dict(reduction="mean")):
        with pytest.raises(NotImplementedError):
            BCE(**kw)


def test_new_path_sasrec_selects_the_bce_head():
    from replay_b200.nn.loss import BCE, CE
    from replay_b200.nn.sequential import SasRec

    m = SasRec.from_params(_schema(), embedding_dim=64, num_heads=1)
    m.loss = BCE()
    assert m.core._loss_spec == ("bce", {}) and "bce" in m.core._FULL_CATALOG
    m.loss = CE()
    assert m.core._loss_spec == ("ce", {})
    # padded hidden size 512 (4 heads of 128): no BCE head - refused when the loss is selected, not at the first step
    big = SasRec.from_params(_schema(d=512), embedding_dim=512, num_heads=4)
    assert big.core.cfg.dp == 512
    with pytest.raises(NotImplementedError):
        big.loss = BCE()
    # multi-positive labels still raise
    m.loss = BCE()
    m.train()
    ids = torch.zeros(2, 8, dtype=torch.long)
    with pytest.raises(NotImplementedError):
        m(feature_tensors={"item_id": ids}, padding_mask=torch.ones(2, 8, dtype=torch.bool),
          positive_labels=torch.zeros(2, 8, 2, dtype=torch.long), target_padding_mask=torch.ones(2, 8, 2, dtype=torch.bool))
    # the setter names what is supported
    with pytest.raises(NotImplementedError, match="BCE, CESampled"):
        m.loss = object()


def test_legacy_sasrec_bce_runs_on_the_core():
    """The legacy SASRec module keeps its constructor contract (``loss_type="BCE"`` without a sample count is refused, the
    sampled BCE head is selected with one); its core selects the full-catalog BCE head like the new path's."""
    from replay_b200.models.nn.sequential import SasRec

    with pytest.raises(NotImplementedError):
        SasRec(_schema(), hidden_size=64, head_count=1, max_seq_len=8, loss_type="BCE")
    sampled = SasRec(_schema(), hidden_size=64, head_count=1, max_seq_len=8, loss_type="BCE", loss_sample_count=8)
    assert sampled._model.core._loss_spec[0] == "legacy_bce_sampled"
    m = SasRec(_schema(), hidden_size=64, head_count=1, max_seq_len=8)
    m._model.core.set_loss("bce")
    assert m._model.core._loss_spec == ("bce", {})


def test_legacy_bert4rec_loss_type_bce_selects_the_head():
    from replay_b200.models.nn.sequential import Bert4Rec

    sch = _schema(pad=0)
    for tying in (False, True):
        m = Bert4Rec(sch, block_count=1, head_count=1, hidden_size=64, max_seq_len=8, loss_type="BCE",
                     enable_embedding_tying=tying)
        assert m._model.core._loss_spec == ("bce", {})
    assert getattr(Bert4Rec(sch, block_count=1, head_count=1, hidden_size=64, max_seq_len=8)._model.core, "_loss_spec",
                   ("ce", {}))[0] == "ce"
    # BERT4Rec's sampled losses and CE_restricted stay unsupported
    for kw in (dict(loss_type="BCE", loss_sample_count=10), dict(loss_type="CE", loss_sample_count=10),
               dict(loss_type="CE_restricted")):
        with pytest.raises(NotImplementedError):
            Bert4Rec(sch, block_count=1, head_count=1, hidden_size=64, max_seq_len=8, **kw)
