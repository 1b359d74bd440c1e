"""CPU tests of the host-side mirror of the reference interface: no kernel is launched here."""
import os

import numpy as np
import pytest
import torch

from replay_b200.core import reference_key_map
from replay_b200.data import left_pad, sasrec_prediction_batch, sasrec_training_batch, to_new_path_batch
from replay_b200.schema import TensorFeatureInfo, TensorSchema


def _schema(n=300, d=64):
    return TensorSchema(TensorFeatureInfo("item_id", n, n, d))


def test_state_dict_keys_match_reference_new(golden_dir):
    z = np.load(os.path.join(golden_dir, "sasrec_new_tiny.npz"))
    ref_keys = {k[4:] for k in z.files if k.startswith("sd::")}
    assert set(reference_key_map("new", int(z["n_blocks"])).values()) == ref_keys


def test_state_dict_keys_match_reference_legacy(golden_dir):
    z = np.load(os.path.join(golden_dir, "sasrec_legacy_tiny.npz"))
    ref_keys = {k[4:] for k in z.files if k.startswith("sd::")}
    ours = set(reference_key_map("legacy", int(z["n_blocks"])).values())
    aliases = {"_head._item_embedder.item_emb.weight", "_head._item_embedder.pos_emb.pe.weight"}
    assert ours | aliases == ref_keys


def test_training_batch_layout_known_answer():
    """tests/models/nn/sequential/sasrec/test_sasrec_dataset.py:40-48 of the reference (sequence [0, 1], max_len 8)."""
    b = sasrec_training_batch([[0, 1]], 8, pad_value=-1)
    assert b["padding_mask"][0].tolist() == [False] * 7 + [True]
    assert b["target_padding_mask"][0].tolist() == [False] * 6 + [True, True]
    assert b["positive_labels"][0].tolist() == [-1] * 6 + [0, 1]
    p = sasrec_prediction_batch([[0, 1, 2]], 8, pad_value=5)
    assert p["padding_mask"][0].tolist() == [False] * 5 + [True] * 3
    n = to_new_path_batch(b)
    assert n["positive_labels"].shape == (1, 8, 1) and n["seen_ids"].shape == (1, 8)


def test_left_pad_truncates_to_last_items_and_handles_empty():
    ids, m = left_pad([list(range(10)), []], 4, 99)
    assert ids[0].tolist() == [6, 7, 8, 9] and m[0].all()
    assert ids[1].tolist() == [99] * 4 and not m[1].any()


def test_new_path_from_params_validation():
    from replay_b200.nn.sequential import SasRec

    # the reference's own defaults (embedding_dim 192, 4 heads -> head_dim 48) are laid out in padded 64-wide head slots
    m = SasRec.from_params(_schema())
    assert (m.core.cfg.d, m.core.cfg.n_heads, m.core.cfg.head_dim, m.core.cfg.dp, m.core.cfg.hd_valid) == (192, 4, 48, 256, 48)
    m = SasRec.from_params(_schema(), embedding_dim=64, num_heads=2)  # SURVEY config 1 / examples/09: head_dim 32
    assert (m.core.cfg.dp, m.core.cfg.hd_valid) == (128, 32)
    assert m.core.cfg.feat_index().tolist() == list(range(32)) + list(range(64, 96))
    with pytest.raises(ValueError):  # head_dim 150 does not fit one 128-wide slot
        SasRec.from_params(_schema(), embedding_dim=300, num_heads=2)
    with pytest.raises(ValueError):  # 8 heads x 128-wide slots = 1024 padded columns: beyond the kernels
        SasRec.from_params(_schema(), embedding_dim=640, num_heads=8)
    with pytest.raises(ValueError):
        SasRec.from_params(TensorSchema(TensorFeatureInfo("item_id", 300, 0, 64)), embedding_dim=64, num_heads=1)
    m = SasRec.from_params(_schema(), embedding_dim=128, num_heads=2, max_sequence_length=50, dropout=0.1)
    assert m.core.cfg.lnf_eps == 1e-5 and m.core.cfg.variant == "new"


def test_lightning_module_candidates_validation():
    from replay_b200.nn.lightning import LightningModule
    from replay_b200.nn.sequential import SasRec

    lm = LightningModule(SasRec.from_params(_schema(), embedding_dim=64, num_heads=1))
    with pytest.raises(ValueError):
        lm.candidates_to_score = torch.tensor([1, 1, 2])
    with pytest.raises(ValueError):
        lm.candidates_to_score = torch.tensor([1.0, 2.0])
    lm.candidates_to_score = torch.tensor([3, 1, 2])
    assert lm.candidates_to_score.tolist() == [3, 1, 2]


def test_legacy_module_error_conventions():
    from replay_b200.models.nn.sequential import SasRec
    from replay_b200.models.nn.sequential.sasrec import _prepare_prediction_batch

    with pytest.raises(NotImplementedError):
        SasRec(_schema(), hidden_size=64, loss_type="BCE")
    m = SasRec(_schema(), hidden_size=64, head_count=1, max_seq_len=8)
    with pytest.raises(ValueError):
        m.candidates_to_score = torch.arange(301)
    with pytest.raises(ValueError):
        m.candidates_to_score = [1, 2]
    b = {"feature_tensor": {"item_id": torch.ones(2, 9, dtype=torch.long)}, "padding_mask": torch.ones(2, 9, dtype=torch.bool)}
    with pytest.raises(ValueError):
        _prepare_prediction_batch(None, 8, b)
    b = {"feature_tensor": {"item_id": torch.ones(2, 5, dtype=torch.long)}, "padding_mask": torch.ones(2, 5, dtype=torch.bool)}
    out = _prepare_prediction_batch(None, 8, b)
    assert out["padding_mask"].shape == (2, 8) and not out["padding_mask"][:, :3].any()


def test_seen_items_filter_known_answers(golden_dir):
    """reference tests/nn/lightning/postprocessor/test_postprocessor.py:7-46 on the mirror class."""
    from replay_b200.nn.lightning import SeenItemsFilter

    z = np.load(os.path.join(golden_dir, "seen_filter_known.npz"))
    f = SeenItemsFilter(item_count=5)
    out = f.on_prediction({"seen_ids": torch.from_numpy(z["seen"])}, torch.from_numpy(z["logits"]))
    assert torch.equal(out, torch.from_numpy(z["out"]))
    f.candidates = torch.from_numpy(z["candidates"])
    out = f.on_prediction({"seen_ids": torch.from_numpy(z["seen"])}, torch.from_numpy(z["cand_logits"]))
    assert torch.equal(out, torch.from_numpy(z["cand_out"]))


def test_library_exports_every_declared_symbol():
    """The C-ABI library loads and exports every entry point include/rp_b200.h declares (no compute call)."""
    import ctypes
    import re

    from replay_b200 import _lib

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    hdr = open(os.path.join(root, "include", "rp_b200.h")).read()
    names = set(re.findall(r"\b(rp_[a-z0-9_]+)\s*\(", hdr))
    assert len(names) >= 15
    if not os.path.exists(_lib.LIB_PATH):
        from replay_b200.build import build

        build(verbose=False)
    h = ctypes.CDLL(_lib.LIB_PATH)
    for n in names:
        assert hasattr(h, n), n


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    from replay_b200 import _lib

    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(_lib.RpError):
        _lib.lib()


@pytest.mark.parametrize("mask_prob,padding,result", [
    (0.0, [0, 0, 0, 0, 0, 1, 1, 1], [1, 1, 1, 1, 1, 1, 1, 0]),
    (1.0, [0, 0, 0, 0, 0, 1, 1, 1], [0, 0, 0, 0, 0, 0, 1, 0]),
    (1e-6, [0, 1, 1, 1, 1, 1, 1, 1], [0, 1, 1, 1, 1, 1, 1, 1]),
])
def test_uniform_bert_masking_corner_cases(mask_prob, padding, result):
    """reference tests/models/nn/sequential/bert4rec/test_bert4rec_dataset.py:15-41 (known answers) on the mirror."""
    from replay_b200.models.nn.sequential import uniform_masker

    tok = uniform_masker(torch.tensor(padding, dtype=torch.bool), mask_prob)
    assert tok.tolist() == [bool(v) for v in result]
    tok2 = uniform_masker(torch.tensor([padding, padding], dtype=torch.bool), mask_prob)
    assert tok2.tolist() == [[bool(v) for v in result]] * 2


def test_bert_shift_features_known_answer():
    """_shift_features (bert4rec/dataset.py:322-345): roll left, last position = <MASK>, pad = True."""
    from replay_b200.models.nn.sequential import shift_features

    ids = torch.tensor([[0, 0, 5, 6, 7]]); pm = torch.tensor([[0, 0, 1, 1, 1]], dtype=torch.bool); tm = pm.clone()
    i2, p2, t2 = shift_features(ids, pm, tm, pad_value=0)
    assert i2.tolist() == [[0, 5, 6, 7, 0]]
    assert p2.tolist() == [[False, True, True, True, True]]
    assert t2.tolist() == [[False, True, True, True, False]]


def test_bert_state_dict_keys_match_reference(golden_dir):
    from replay_b200.models.nn.sequential.bert4rec import bert_key_map

    for name, tying in (("bert4rec_tiny.npz", False), ("bert4rec_tiny_tied.npz", True)):
        z = np.load(os.path.join(golden_dir, name))
        ref = {k[4:] for k in z.files if k.startswith("sd::")}
        ours = set(bert_key_map(int(z["n_blocks"]), tying).values())
        if tying:
            ours |= {"_head._item_embedder." + k[len("item_embedder."):] for k in ours if k.startswith("item_embedder.")}
        assert ours == ref, (ours ^ ref)


def test_ranking_metrics_match_reference_definitions():
    """RankingMetrics vs a direct evaluation of TorchMetricsBuilder's formulas (torch_metrics_builder.py:305-393) on a
    hand-checkable case."""
    import math

    from replay_b200.nn.lightning import RankingMetrics

    pred = torch.tensor([[5, 3, 9, 1], [7, 8, 2, 0]])
    gt = torch.tensor([[3, 1, -1], [4, -1, -1]])
    m = RankingMetrics(("recall", "precision", "ndcg", "map", "mrr"), (2, 4))
    m.add_prediction(pred, gt)
    r = m.get_metrics()
    # user 0: hits at ranks 2 and 4 (|gt| = 2); user 1: no hit
    assert abs(r["recall@2"] - (0.5 + 0) / 2) < 1e-6 and abs(r["recall@4"] - (1.0 + 0) / 2) < 1e-6
    assert abs(r["precision@4"] - (0.5 + 0) / 2) < 1e-6
    dcg4 = 1 / math.log2(3) + 1 / math.log2(5)
    idcg2 = 1 / math.log2(2) + 1 / math.log2(3)
    assert abs(r["ndcg@4"] - (dcg4 / idcg2) / 2) < 1e-6
    assert abs(r["mrr@4"] - (0.5 + 0) / 2) < 1e-6
    assert abs(r["map@4"] - ((1 / 2 + 2 / 4) / 2) / 2) < 1e-6


def test_window_index_vectorised_matches_reference_order():
    """replay_b200.device_data.window_index (numpy, no GPU needed) against the loop restatement and the reference's own
    index maps stored in the golden fixture."""
    import os
    from oracle import dataset as od
    from replay_b200.device_data import window_index
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "dataset_layout.npz"))
    L, step = int(z["L"]), int(z["step"])
    for window, st, key in ((L + 1, step, "sas_slide_index"), (L + 1, None, "sas_last_index"), (L, step, "bert_slide_index")):
        s, o = window_index(z["lengths"], window, st)
        assert np.array_equal(np.stack([s, o], 1), z[key])
    rng = np.random.default_rng(0)
    lens = rng.integers(0, 60, 500)
    for window in (1, 7, 33):
        for st in (None, 1, 3, 50):
            s, o = window_index(lens, window, st)
            ref = np.asarray(od.window_index(lens, window, st)).reshape(-1, 2)
            assert np.array_equal(np.stack([s, o], 1), ref)


def test_parquet_to_csr_store(tmp_path):
    """DeviceSequenceStore.from_parquet: list<int> column -> offsets / flat values without a Python loop (multiple files,
    empty and null lists, int32 / int64 item types); no kernel is involved, so this runs on the CPU."""
    import pyarrow as pa
    import pyarrow.parquet as pq
    from replay_b200.device_data import DeviceSequenceStore
    seqs = [[3, 1, 2], [], [7], None, [5, 5, 5, 9]]
    t1 = pa.table({"user": pa.array([10, 11, 12, 13, 14], pa.int64()), "item_id": pa.array(seqs, pa.list_(pa.int64()))})
    t2 = pa.table({"user": pa.array([20, 21], pa.int64()), "item_id": pa.array([[4, 4], [0]], pa.list_(pa.int64()))})
    p1, p2 = str(tmp_path / "a.parquet"), str(tmp_path / "b.parquet")
    pq.write_table(t1, p1, row_group_size=2)
    pq.write_table(t2, p2)
    st = DeviceSequenceStore.from_parquet([p1, p2], "item_id", query_column="user", device="cpu")
    assert st.offsets.tolist() == [0, 3, 3, 4, 4, 8, 10, 11]
    assert st.items.tolist() == [3, 1, 2, 7, 5, 5, 5, 9, 4, 4, 0] and st.items.dtype == torch.int32
    assert st.query_ids.tolist() == [10, 11, 12, 13, 14, 20, 21] and len(st) == 7
    st32 = DeviceSequenceStore.from_parquet(pa.table({"item_id": pa.array([[1, 2], [3]], pa.list_(pa.int32()))}), device="cpu")
    assert st32.offsets.tolist() == [0, 2, 3] and st32.query_ids is None
    with pytest.raises(ValueError):
        DeviceSequenceStore.from_parquet(pa.table({"item_id": pa.array([1, 2, 3])}), device="cpu")
    with pytest.raises(ValueError):
        DeviceSequenceStore(offsets=[0, 2, 1], items=[1, 2], device="cpu")


def test_c_abi_argument_errors_without_a_gpu():
    """include/rp_b200.h error convention: < 0 for argument / shape errors, decided before any CUDA call - so it can be checked
    on a machine without a GPU (no kernel is launched here).  Workspace queries are pure host functions."""
    import ctypes
    from replay_b200._lib import AttnBwdDesc, AttnDesc, GemmDesc, SampledDesc, lib
    L = lib()
    EINVAL, ESHAPE = -1, -2
    assert L.rp_version().decode().startswith("rp_b200")
    # workspace sizes: positive, monotone in the problem size, 0 for nonsense
    a, b = L.rp_score_topk_workspace(4096, 500_000, 128, 10), L.rp_score_topk_workspace(8192, 500_000, 128, 10)
    assert 0 < a < b and L.rp_score_topk_workspace(0, 10, 128, 10) == 0
    assert 0 < L.rp_ce_head_workspace(1024, 5000, 128) < L.rp_ce_head_workspace(2048, 5000, 128)
    assert L.rp_ce_head_workspace(1024, 5000, 512) > L.rp_ce_head_workspace(1024, 5000, 256)      # d = 512 holds a G chunk
    assert 0 < L.rp_sampled_head_workspace(1024, 128, 100, 1) < L.rp_sampled_head_workspace(1024, 128, 100, 0)
    assert L.rp_sampled_head_workspace(0, 128, 100, 0) == 0
    # NULL / malformed arguments
    assert L.rp_gemm(None, None) == EINVAL
    g = GemmDesc()
    assert L.rp_gemm(ctypes.byref(g), None) == EINVAL                      # NULL operands
    assert L.rp_attn_fwd(None, None) == EINVAL and L.rp_attn_fwd(ctypes.byref(AttnDesc()), None) == EINVAL
    assert L.rp_attn_bwd(None, None) == EINVAL and L.rp_attn_bwd(ctypes.byref(AttnBwdDesc()), None) == EINVAL
    assert L.rp_sampled_head_fwd(None, None) == EINVAL and L.rp_sampled_head_fwd(ctypes.byref(SampledDesc()), None) == EINVAL
    assert L.rp_sampled_head_bwd(ctypes.byref(SampledDesc()), None, None, None) == EINVAL
    assert L.rp_seen_prepare(None, 1, 1, 1, None, None, None) == EINVAL
    assert L.rp_score_topk(None, None, None, None, 0, 1, 1, 128, 10, None, None, None, None, 0, None) == EINVAL
    assert L.rp_ce_head_fwd(None, None, None, None, None, 1, 1, 128, None, None, None, None, 0, None, 0, None) == EINVAL
    assert L.rp_ce_head_bwd(None, None, None, None, None, 1, 1, 128, None, None, None, None, None, 0, 0, None, 0, None) == EINVAL
    assert L.rp_ffn_fused(None, None, None, None, None, None, 1, 128, None, None) == EINVAL
    assert L.rp_post_attn_fused(None, None, None, None, None, None, 1e-8, None, None, None, None, None, 1, 128, None, 0, None) == EINVAL
    assert L.rp_post_attn_train(None, None, None, None, None, None, 1e-8, None, None, None, None, None, 1, 128, 0.0, 0, 0, 0, None,
                                None, None, None, None, None, None, 0, None) == EINVAL
    assert L.rp_post_attn_bwd(None, None, None, None, None, None, None, None, None, None, 1, 128, 0.0, 0, 0, None, None, None, None,
                              None, None, None, 0, None) == EINVAL
    assert L.rp_ln_qkv_fused(None, None, None, 1e-8, None, None, 1, 128, None, None, None, None, None, 0, None) == EINVAL
    assert L.rp_pre_attn_bwd(None, None, None, None, None, None, None, None, 1, 128, None, None, None, 0, None) == EINVAL
    assert L.rp_wgrad_group(None, 0, 1, 1, None, 0, None) == EINVAL and L.rp_wgrad_group_workspace(None, 0) == 0
    assert L.rp_build_batch(None, None, 1, None, None, 1, 1, 0, 0, 0.0, None, 0, 0, None, None, None, None, None, None, None) == EINVAL
    assert L.rp_reduce_splits(None, 1, 4, 4, None, 0, None) == EINVAL
    assert L.rp_colsum(None, 1, 4, 4, None, None) == EINVAL
    assert L.rp_colsum_multi(0, None, None, None, None, 1, None) == EINVAL
    assert L.rp_adam_step(None, None, None, None, None, 4, None, None, 0.9, 0.98, 1e-8, 1.0, None, 1, None) == EINVAL
    assert L.rp_selftest_mma_probe(99, 1, 1, None, None) == EINVAL
    # shape errors with non-NULL dummies (no memory is touched before the shape check)
    buf = ctypes.create_string_buffer(64)
    p = ctypes.cast(buf, ctypes.c_void_p)
    assert L.rp_ffn_fused(p, p, p, p, p, None, 10, 96, ctypes.cast(ctypes.create_string_buffer(8), ctypes.c_void_p), None) == ESHAPE
    assert L.rp_ce_head_fwd(p, p, None, p, p, 128, 100, 96, p, p, p, None, 0, p, 1 << 40, None) == ESHAPE


def test_device_loader_sharding_covers_every_window_once():
    """Host-side index logic of DeviceBatchLoader (no kernel involved: the store may live on the CPU for this): for every world
    size the ranks' shards are disjoint up to the wrap-around padding and cover all windows; every epoch reshuffles."""
    from replay_b200.device_data import DeviceBatchLoader, DeviceSequenceStore
    rng = np.random.default_rng(0)
    seqs = [rng.integers(0, 50, n) for n in rng.integers(1, 40, 101)]
    st = DeviceSequenceStore(seqs, device="cpu")
    for world in (1, 2, 3, 8):
        loaders = [DeviceBatchLoader(st, 8, 16, 50, sliding_window_step=3, seed=5, rank=r, world_size=world) for r in range(world)]
        n = loaders[0].n
        shards = [ld.epoch_indices() for ld in loaders]
        assert all(len(s) == -(-n // world) for s in shards)
        allidx = torch.cat(shards)
        assert set(allidx.tolist()) == set(range(n)) and len(allidx) - n < world      # only the wrap-around duplicates
        assert len(loaders[0]) == -(-len(shards[0]) // 16)
        loaders[0].set_epoch(1)
        assert not torch.equal(loaders[0].epoch_indices(), shards[0])
    fixed = DeviceBatchLoader(st, 8, 16, 50, shuffle=False)
    assert torch.equal(fixed.epoch_indices(), torch.arange(fixed.n))


def test_ranking_metrics_match_reference_builder_incl_novelty_and_coverage(golden_dir):
    """tests/golden/metrics_known.npz holds the output of the REAL TorchMetricsBuilder (oracle/gen_golden.py metrics) over three
    batches: recall / precision / ndcg / map / mrr / novelty @ {1,5,10,20} and coverage."""
    import numpy as np

    from replay_b200.nn.lightning import RankingMetrics

    z = np.load(os.path.join(golden_dir, "metrics_known.npz"))
    m = RankingMetrics(("recall", "precision", "ndcg", "map", "mrr", "novelty", "coverage"), (1, 5, 10, 20), item_count=int(z["n_items"]))
    for i in range(3):
        m.add_prediction(torch.from_numpy(z[f"pred{i}"]), torch.from_numpy(z[f"gt{i}"]), torch.from_numpy(z[f"train{i}"]))
    r = m.get_metrics()
    ref = dict(zip([str(n) for n in z["names"]], z["values"]))
    assert set(r) == set(ref)
    for k, v in ref.items():
        assert abs(r[k] - v) < 1e-6, (k, r[k], v)


def test_compute_metrics_callback_history_and_state_dict():
    """metrics_callback.py:72-100,147-163: per-epoch history for validation and test stages, state_dict round trip."""
    from replay_b200.nn.lightning import ComputeMetricsCallback

    class _PL:  # a module without an engine: the callback takes the logits path
        candidates_to_score = None
        logged = {}

        def log_dict(self, d, **k):
            self.logged.update(d)

    cb = ComputeMetricsCallback(metrics=("recall", "ndcg"), ks=(1, 2))
    logits = torch.tensor([[0.1, 0.9, 0.3], [0.8, 0.2, 0.5]])
    batch = {"ground_truth": torch.tensor([[1, -1], [2, -1]])}
    for stage in ("validation", "test"):
        getattr(cb, f"on_{stage}_epoch_start")(None, _PL())
        getattr(cb, f"on_{stage}_batch_end")(None, _PL(), {"logits": logits}, batch, 0)
        res = getattr(cb, f"on_{stage}_epoch_end")(None, _PL())
        assert abs(res["recall@1"] - 0.5) < 1e-6 and abs(res["recall@2"] - 1.0) < 1e-6
    assert cb.get_metrics("validate")[0]["recall@2"] == 1.0 and cb.get_metrics("test")[0]["recall@1"] == 0.5
    sd = cb.state_dict()
    cb2 = ComputeMetricsCallback(metrics=("recall", "ndcg"), ks=(1, 2))
    cb2.load_state_dict({k: {str(e): m for e, m in v.items()} for k, v in sd.items()})  # keys come back as strings from json
    assert cb2.get_metrics("validate") == cb.get_metrics("validate") and cb2.get_metrics("test") == cb.get_metrics("test")


def test_prediction_side_callbacks_without_an_engine():
    """predictions_callback.py:124-163,282-325 and callbacks/{prediction_callbacks,validation_callback}.py: the frame-building,
    hidden-state, query-embedding and legacy validation callbacks on plain tensors (the dense-scores path every callback
    keeps for modules without an engine)."""
    from replay_b200.models.nn.sequential import (PandasPredictionCallback, QueryEmbeddingsPredictionCallback,
                                                  ValidationMetricsCallback)
    from replay_b200.nn.lightning import HiddenStatesCallback, PandasTopItemsCallback, RankingMetrics

    class _PL:
        candidates_to_score = None
        logged = {}

        def log_dict(self, d, **k):
            self.logged.update(d)

    logits = torch.tensor([[0.1, 0.9, 0.3, 0.0], [0.8, 0.2, 0.5, 0.6]])
    # new-path pandas frame: one row per (query, item, rating), best first
    cb = PandasTopItemsCallback(top_k=2, query_column="user", item_column="item", rating_column="score")
    cb.on_predict_epoch_start(None, _PL())
    cb.on_predict_batch_end(None, _PL(), {"logits": logits}, {"user": torch.tensor([7, 9])}, 0)
    df = cb.get_result()
    assert df["user"].tolist() == [7, 7, 9, 9] and df["item"].tolist() == [1, 2, 0, 3]
    assert np.allclose(df["score"].to_numpy(), [0.9, 0.3, 0.8, 0.6])
    # legacy pandas frame (outputs are the scores themselves)
    lcb = PandasPredictionCallback(top_k=1, query_column="user", item_column="item")
    lcb.on_predict_epoch_start(None, _PL())
    lcb.on_predict_batch_end(None, _PL(), logits, {"query_id": torch.tensor([[7], [9]])}, 0)
    assert lcb.get_result()["item"].tolist() == [1, 0]
    # hidden states: the chosen element of outputs["hidden_states"], concatenated over batches
    h = HiddenStatesCallback(hidden_state_index=1)
    h.on_predict_epoch_start(None, None)
    for k in range(2):
        h.on_predict_batch_end(None, None, {"hidden_states": (torch.zeros(2, 3), torch.full((2, 3), float(k)))}, {}, k)
    assert h.get_result().shape == (4, 3) and h.get_result()[2:].eq(1).all()

    # query embeddings: batch entries are matched to the signature of _model.get_query_embeddings
    class _M:
        @staticmethod
        def get_query_embeddings(feature_tensor, padding_mask):
            return feature_tensor["item_id"].float() * padding_mask

    class _PLQ:
        _model = _M()

    q = QueryEmbeddingsPredictionCallback()
    q.on_predict_epoch_start(None, _PLQ())
    q.on_predict_batch_end(None, _PLQ(), None, {"query_id": torch.tensor([1]), "feature_tensor": {"item_id": torch.tensor([[2, 3]])},
                                               "padding_mask": torch.tensor([[0, 1]])}, 0)
    assert q.get_result().tolist() == [[0.0, 3.0]]
    # legacy validation callback == the metric builder on top-k of the scores
    v = ValidationMetricsCallback(metrics=("recall", "ndcg", "map"), ks=(1, 2))
    v.on_validation_epoch_start(None, _PL())
    gt = torch.tensor([[1, -1], [3, 2]])
    v.on_validation_batch_end(None, _PL(), logits, {"query_id": torch.tensor([7, 9]), "ground_truth": gt}, 0)
    res = v.on_validation_epoch_end(None, _PL())
    ref = RankingMetrics(("recall", "ndcg", "map"), (1, 2))
    ref.add_prediction(torch.topk(logits, 2, dim=1).indices, gt)
    assert res == ref.get_metrics() and abs(res["recall@1"] - 0.5) < 1e-6


def test_balanced_rank_shards_deals_equal_counts_and_near_equal_work():
    """replay_b200.data.balanced_rank_shards: a partition, equal sample counts, per-rank work within one sample of the mean."""
    import torch

    from replay_b200.data import balanced_rank_shards

    g = torch.Generator().manual_seed(0)
    work = torch.randint(1, 200, (4096,), generator=g)
    sh = balanced_rank_shards(work, 8)
    assert sh.shape == (8, 512)
    assert torch.equal(torch.sort(sh.reshape(-1)).values, torch.arange(4096))
    tot = work[sh].sum(1).float()
    assert float(tot.max() - tot.min()) <= 200
    import pytest

    with pytest.raises(ValueError):
        balanced_rank_shards(work[:4095], 8)


def test_replica_partition_reproduces_reference_known_answers(golden_dir):
    """replay_b200.data.replica_partition against outputs of the real ``Partitioning.generate`` (tests/golden/partitioning_known.npz,
    produced in the build container; the generator variant was checked there element by element against the reference)."""
    import numpy as np
    import pytest
    import torch

    from replay_b200.data import replica_partition

    z = np.load(os.path.join(golden_dir, "partitioning_known.npz"))
    assert len(z.files) == 14
    for key in z.files:
        _, n, w, r = key.split("_")
        got = replica_partition(int(n), int(r), int(w))
        assert torch.equal(got, torch.from_numpy(z[key])), key
    # every row is covered, padding wraps around (5 rows over 7 replicas: every replica one row, two of them repeats)
    allrows = torch.cat([replica_partition(5, r, 7) for r in range(7)])
    assert set(allrows.tolist()) == set(range(5)) and allrows.numel() == 7
    for bad in ((0, 0, 1), (4, 2, 2), (4, 0, 0)):
        with pytest.raises(ValueError):
            replica_partition(*bad)


def test_row_loss_selectors_weights_and_kinds():
    """replay_b200.nn.loss selectors of the per-row heads: which fused head they select and the per-position weights they hand
    to it (CEWeighted reproduces the reference's broadcast: every valid row gets mean(w) * T_v / (B * L))."""
    import torch

    from replay_b200.nn import loss as L

    tm = torch.tensor([[False, True, True], [True, True, True]])
    w = torch.tensor([[[2.0], [1.0], [0.5]], [[1.5], [1.0], [3.0]]])
    lo = L.LogOutCE(cardinality=10)
    assert lo.kind == "ce" and not lo.needs_negatives and not hasattr(lo, "row_weights")
    low = L.LogOutCEWeighted(cardinality=10, feature_name="w")
    assert low.kind == "ce_weighted"
    assert torch.equal(low.row_weights({"w": w}, tm), w[..., 0])
    cw = L.CEWeighted(feature_name="w")
    got = cw.row_weights({"w": w}, tm)
    assert got.shape == (2, 3) and torch.allclose(got, torch.full((2, 3), float(w.mean()) * 5 / 6))
    li = L.LogInCE(cardinality=10, log_epsilon=1e-3, clamp_border=5.0)
    assert li.kind == "login_ce" and li.engine_kwargs() == {"log_eps": 1e-3, "clamp": 5.0}
    assert L.LogOutCESampled is L.CE


def test_peer_gradient_buffer_needs_an_nccl_group():
    """replay_b200.peer.alloc_peer_grad: no process group (or a non-NCCL one) -> None, the trainer keeps ncclAllReduce / gloo."""
    from replay_b200.peer import alloc_peer_grad

    assert alloc_peer_grad(1024, "cpu") is None


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the reference algorithm - oracle port - on the host cores; what the driver runs next to
    the GPU arm): ONE JSON line with the contract's keys, same metric / unit as the GPU arm, e2e == value, no GPU needed."""
    import json
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=root)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    j = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "dtype",
              "data", "config", "cpu_baseline", "e2e"):
        assert k in j, k
    assert j["impl"] == "reference" and j["metric"] == "sasrec_train_seq_per_s" and j["unit"] == "seq/s"
    assert j["value"] > 0 and j["higher_is_better"] is True
    assert j["e2e"]["value"] == j["value"] and j["e2e"]["h2d_bytes_per_step"] == 0 and j["e2e"]["d2h_bytes_per_step"] == 0
    assert j["cpu_baseline"]["kind"] == "port" and j["cpu_baseline"]["cores"] >= 1


def test_bench_dump_outputs_are_reproducible_and_follow_steps(tmp_path):
    """`bench.py --dump-outputs DIR` writes what the last timed step computed as float32 / float64 .npy files (< 64 MB in
    all); the same arguments give the same outputs (up to the order of multithreaded CPU sums), and one more timed step
    moves the parameters by about Adam's learning rate."""
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

    def run(steps, name):
        out = tmp_path / name
        r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--no-scoring", "--steps",
                            str(steps), "--warmup", "0", "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600,
                           cwd=root)
        assert r.returncode == 0, r.stderr[-2000:]
        return {p.stem: np.load(p) for p in out.glob("*.npy")}

    a, b, c = run(1, "a"), run(1, "b"), run(2, "c")
    assert set(a) == {"train_loss", "train_params"}
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    for k in a:
        np.testing.assert_allclose(a[k], b[k], rtol=1e-5, atol=1e-7, err_msg=k)
    assert np.abs(a["train_params"] - c["train_params"]).max() > 1e-4


@pytest.mark.parametrize("d,H,L,n_items", [(192, 4, 256, 1000), (192, 4, 512, 1000), (192, 4, 768, 1000), (64, 2, 128, 1000),
                                           (50, 1, 128, 1000), (50, 1, 64, 127), (192, 4, 50, 255), (64, 2, 64, 383)])
def test_true_shape_shrinks_feature_axes_only(d, H, L, n_items):
    """The reference shape of every padded parameter: only feature axes shrink.  A row count equal to a padded width
    (max_len or n_items + 1 in {dp, 2 dp, 3 dp}) stays what it is."""
    from replay_b200.engine import EncoderConfig, param_shapes, true_shape

    cfg = EncoderConfig(n_items=n_items, d=d, n_heads=H, n_blocks=2, max_len=L)
    assert cfg.hd_valid > 0 and L in (cfg.dp, 2 * cfg.dp, 3 * cfg.dp) or n_items + 1 in (cfg.dp, 2 * cfg.dp, 3 * cfg.dp)
    want = {"item_emb": (n_items + 1, d), "pos_emb": (L, d), "in_w": (3 * d, d), "in_b": (3 * d,), "out_w": (d, d),
            "w1": (d, d), "w2": (d, d)}
    shapes = param_shapes(cfg)
    assert len(shapes) == 2 + 12 * 2 + 2
    for name, padded in shapes:
        assert true_shape(cfg, name, padded) == want.get(name.split(".")[-1], (d,)), name
