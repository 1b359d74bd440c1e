#!/usr/bin/env python
"""bench.py - headline benchmark of the B200-native RePlay sequential-recommender hot path.

    python bench.py --gpus N --steps K --warmup W [--config 2|3|5]     # this repo's CUDA path (torchrun launches N>1)
    python bench.py --impl reference --gpus N --steps K ... [--config]  # the reference's CPU algorithm (oracle port), host cores

--config 2 (default, BASELINE.json configs[1]): SASRec seq_len=200 d=128 H=2 2 blocks |items|=50 000, full-catalog CE, Adam,
  dropout 0.2, bf16 compute / fp32 master, MovieLens-shaped synthetic sequences (replay_b200/synthetic.py, seed 1234), data
  parallel over N GPUs (weak scaling: 512 sequences per GPU per step).  The same JSON line carries the scoring leg of
  BASELINE's metric (configs[3]: top-K@10 with seen-item filter, |items| = 500 000, >= 1 M users per GPU, per-call user
  batches {512, 4096, 32768}) under "scoring".
--config 3 (configs[2]): BERT4Rec seq_len=200 d=256 H=4 |items|=100 000, untied biased head, mask_prob 0.15, 256 seq / GPU.
--config 5 (configs[4]): SASRec seq_len=512 d=512 H=8 |items|=1 000 000, 32 seq / GPU (2 GB fp32 gradient all-reduce).

One step = forward + backward + gradient all-reduce + Adam over one batch.  `value`: inputs resident in HBM, CUDA-graph
replays (replay_b200.trainer.Trainer).  `e2e`: the same step through the reference-facing Lightning mirror
(`LightningModule.training_step` / legacy `Bert4Rec.training_step`) with PINNED HOST batches, host->device copies and a
device->host read of the loss inside the timed region.  Timing: CUDA events on the launching stream, barrier + synchronize on
both sides, max over ranks; every step works on > L2 of activations (no L2 flush needed; stated in `config`).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    2: dict(kind="sasrec", name="BASELINE configs[1]", seq_len=200, d=128, heads=2, blocks=2, n_items=50_000, dropout=0.2,
            per_gpu_batch=512, cpu_batch=8),
    3: dict(kind="bert", name="BASELINE configs[2]", seq_len=200, d=256, heads=4, blocks=2, n_items=100_000, dropout=0.1,
            per_gpu_batch=256, mask_prob=0.15, cpu_batch=4),
    5: dict(kind="sasrec", name="BASELINE configs[4]", seq_len=512, d=512, heads=8, blocks=2, n_items=1_000_000, dropout=0.2,
            per_gpu_batch=32, cpu_batch=1),
}
SCORE_CFG = dict(n_items=500_000, d=128, seq_len=200, k=10, users_per_call=4096, sweep=(512, 4096, 32768),
                 users_per_gpu=1_048_576, distinct_histories=65_536)
DUMP_PARAM_ELEMENTS = 1 << 23  # --dump-outputs: the fp32 parameters take at most 32 MB of its 64 MB


def param_sample(flat):
    """The flat parameter vector itself when it fits DUMP_PARAM_ELEMENTS, else that many elements at fixed seeded
    positions (the same positions for the same configuration), fp32 on the host."""
    flat = flat.detach().reshape(-1)
    if flat.numel() > DUMP_PARAM_ELEMENTS:
        idx = torch.randint(0, flat.numel(), (DUMP_PARAM_ELEMENTS,), generator=torch.Generator().manual_seed(0)).sort().values
        flat = flat[idx.to(flat.device)]
    return flat.float().cpu()


def write_outputs(out_dir, arrays):
    """--dump-outputs: one DIR/<name>.npy per array, float32 (float64 for integer ids: exact below 2**53)."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach().cpu()
        t = t.double() if not t.is_floating_point() or t.dtype == torch.float64 else t.float()
        np.save(os.path.join(out_dir, name + ".npy"), t.numpy())


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as fh:
            z = json.load(fh)
        return dict(hbm=z["hbm_gbs"], tc_burst=z["bf16_tflops"], tc_sustained=z["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tc_burst=1590.0, tc_sustained=1400.0, src="fallback")


def measured_traffic(key: str):
    """dram__bytes_read + dram__bytes_write per launch of the named kernel from the committed ncu capture of THIS shape
    (profiles/r2_traffic.json, written by tools/extract_traffic.py from the .ncu-rep); None if no capture exists for it."""
    p = os.path.join(ROOT, "profiles", "r2_traffic.json")
    if not os.path.exists(p):
        return None
    with open(p) as fh:
        return json.load(fh).get(key)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index: int):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        pw = sorted(float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "", 1).isdigit())
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        mx = int(self.rows[0][1]) if self.rows and self.rows[0][1].isdigit() else None
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": pw[-1] if pw else None}


def train_flops_per_seq(c, n_valid_per_seq):
    """SURVEY.md §8d: body per token N_b(12 d^2 + 4 d L) (SASRec) / N_b(24 d^2 + 4 d L) (BERT4Rec, 4d FFN), head 2 d |I| per
    VALID target (+ |I| bias adds for the biased head, not counted), x3 for training."""
    L, d, nb, I = c["seq_len"], c["d"], c["blocks"], c["n_items"]
    per_tok = nb * ((24 if c["kind"] == "bert" else 12) * d * d + 4 * d * L)
    return 3.0 * (L * per_tok + n_valid_per_seq * 2 * d * I)


def workload_string(c):
    if c["kind"] == "bert":
        return (f"{c['name']}: BERT4Rec L={c['seq_len']} d={c['d']} H={c['heads']} blocks={c['blocks']} |I|={c['n_items']}, untied biased head, "
                f"mask_prob {c['mask_prob']}, full-catalog CE over masked positions + Adam, dropout {c['dropout']}, synthetic windows "
                "(activations per step > L2)")
    return (f"{c['name']}: SASRec L={c['seq_len']} d={c['d']} H={c['heads']} blocks={c['blocks']} |I|={c['n_items']}, full-catalog CE + Adam, "
            f"dropout {c['dropout']}, MovieLens-shaped synthetic windows (inputs > L2: activations per step exceed the 126 MB L2)")


# ----------------------------------------------------------------------------------------------------------------------
# synthetic batches
# ----------------------------------------------------------------------------------------------------------------------
def make_batches(c, n_seq, seed):
    """CPU tensors of n_seq training windows in the layout of the reference datasets (sasrec/dataset.py:104-126,
    bert4rec/dataset.py:163-177): SASRec (ids, pad_mask, labels, target_mask); BERT4Rec (ids, pad_mask, token_mask, labels)."""
    from replay_b200.synthetic import make_sequences

    if c["kind"] == "bert":
        from replay_b200.models.nn.sequential import uniform_masker

        ids, pm, _, _ = make_sequences(n_seq, c["n_items"], c["seq_len"], seed=seed, pad_value=0)
        tok = uniform_masker(pm, c["mask_prob"], torch.Generator().manual_seed(seed))
        return ids, pm, tok, ids.clone()
    return make_sequences(n_seq, c["n_items"], c["seq_len"], seed=seed)


def valid_targets(c, batch):
    if c["kind"] == "bert":
        return float((batch[1] & ~batch[2]).sum()) / batch[0].shape[0]
    return float(batch[3].sum()) / batch[0].shape[0]


# ----------------------------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port (plain torch fp32 on the host cores)
# ----------------------------------------------------------------------------------------------------------------------
def cpu_train_seq_per_s(c, steps=3, warmup=1):
    torch.set_num_threads(min(os.cpu_count() or 1, 32))  # torch CPU GEMMs stop scaling (and regress) past ~32 threads
    batch = c["cpu_batch"]
    data = make_batches(c, batch * (steps + warmup), seed=1234)
    if c["kind"] == "bert":
        from oracle import bert4rec as ob

        g = torch.Generator().manual_seed(0)
        d, I, L = c["d"], c["n_items"], c["seq_len"]
        rn = lambda *s: torch.randn(*s, generator=g) * 0.05  # noqa: E731
        P = {"item_emb": rn(I, d), "mask_emb": rn(1, d), "pos_emb": rn(L, d), "head_w": rn(I, d), "head_b": torch.zeros(I),
             "blocks": [{"ln1_w": torch.ones(d), "ln1_b": torch.zeros(d), "in_w": rn(3 * d, d), "in_b": torch.zeros(3 * d),
                         "out_w": rn(d, d), "out_b": torch.zeros(d), "ln2_w": torch.ones(d), "ln2_b": torch.zeros(d),
                         "w1": rn(4 * d, d), "b1": torch.zeros(4 * d), "w2": rn(d, 4 * d), "b2": torch.zeros(d)}
                        for _ in range(c["blocks"])]}
        flat = [P[k] for k in ("item_emb", "mask_emb", "pos_emb", "head_w", "head_b")] + [v for b in P["blocks"] for v in b.values()]
        for p in flat:
            p.requires_grad_(True)
        loss_fn = lambda sl: ob.train_loss(P, data[0][sl], data[1][sl], data[2][sl], data[3][sl], c["heads"])  # noqa: E731
    else:
        from oracle import sasrec as osr

        P = osr.random_params(c["n_items"], c["d"], c["seq_len"], c["blocks"], seed=0)
        flat = [p.requires_grad_(True) for p in osr.flat_param_list(P)]
        loss_fn = lambda sl: osr.train_loss(P, data[0][sl], data[1][sl], data[2][sl], data[3][sl], c["heads"], "new")  # noqa: E731
    opt = torch.optim.Adam(flat, lr=1e-3, betas=(0.9, 0.98))
    ts = []
    for s in range(steps + warmup):
        sl = slice(s * batch, (s + 1) * batch)
        t0 = time.perf_counter()
        opt.zero_grad(set_to_none=True)
        loss = loss_fn(sl)
        loss.backward()
        opt.step()
        ts.append(time.perf_counter() - t0)
    ts = sorted(ts[warmup:])
    med = ts[len(ts) // 2]
    return batch / med, med, loss.detach(), torch.cat([p.detach().reshape(-1) for p in flat])


def cpu_predict_users_per_s(users=64, reps=3):
    """Reference predict path on the host cores (oracle port): body forward (eval) -> last hidden -> [U, |I|] logits ->
    SeenItemsFilter (clone + scatter -inf) -> torch.topk(10), fp32, at the scoring leg's shape (|I| = 500K, L = 200, d = 128)."""
    from oracle import sasrec as osr
    from replay_b200.synthetic import make_sequences

    torch.set_num_threads(min(os.cpu_count() or 1, 32))
    sc = SCORE_CFG
    P = osr.random_params(sc["n_items"], sc["d"], sc["seq_len"], 2, seed=7)
    ids, pm, _, _ = make_sequences(users, sc["n_items"], sc["seq_len"], seed=7)
    ts = []
    with torch.no_grad():
        for _ in range(reps + 1):
            t0 = time.perf_counter()
            h = osr.sasrec_body(P, ids, pm, 2, "new", mode="eval")[:, -1]
            scores = h @ P["item_emb"][: sc["n_items"]].T
            scores = osr.seen_filter(scores, ids, sc["n_items"])
            torch.topk(scores, sc["k"], dim=1)
            ts.append(time.perf_counter() - t0)
    ts = sorted(ts[1:])
    return users / ts[len(ts) // 2]


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    c = CONFIGS[args.config]
    v, med, loss, flat = cpu_train_seq_per_s(c, steps=args.steps, warmup=args.warmup)
    if args.dump_outputs:
        write_outputs(args.dump_outputs, {"train_loss": loss.reshape(1), "train_params": param_sample(flat)})
    cores = torch.get_num_threads()
    metric = "bert4rec_train_seq_per_s" if c["kind"] == "bert" else "sasrec_train_seq_per_s"
    line = {
        "impl": "reference", "metric": metric, "value": v, "unit": "seq/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": med * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_string(c) + " - CPU oracle port of the reference algorithm",
                   **{k: c[k] for k in ("seq_len", "d", "heads", "blocks", "n_items")}, "global_batch": c["cpu_batch"]},
        "cpu_baseline": {"value": v, "unit": "seq/s", "cores": cores, "kind": "port",
                         "sample": f"{args.steps} timed steps of batch {c['cpu_batch']} (fwd+bwd+Adam, dropout off), torch fp32, {cores} threads"},
        "e2e": {"value": v, "unit": "seq/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if args.config == 2 and not args.no_scoring:
        line["scoring"] = {"metric": "sasrec_predict_topk10_users_per_s", "value": cpu_predict_users_per_s(), "unit": "users/s",
                           "cores": cores, "kind": "port",
                           "sample": "64 users, 3 timed calls: oracle body + full logits + seen filter + torch.topk, torch fp32 CPU"}
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------------------------------
# this repo's arm
# ----------------------------------------------------------------------------------------------------------------------
def build_module(c, dev):
    """The reference-facing module of this config (what a RePlay user constructs) and the batch-dict maker for its
    training_step.  SASRec: new-path ``SasRec.from_params`` wrapped in ``LightningModule`` (replay/nn/lightning/module.py);
    BERT4Rec: the legacy Lightning module ``Bert4Rec`` (replay/models/nn/sequential/bert4rec/lightning.py)."""
    from replay_b200.schema import TensorFeatureInfo, TensorSchema

    I, d, L = c["n_items"], c["d"], c["seq_len"]
    if c["kind"] == "bert":
        from replay_b200.models.nn.sequential import Bert4Rec

        schema = TensorSchema(TensorFeatureInfo("item_id", I, 0, d))
        mod = Bert4Rec(schema, block_count=c["blocks"], head_count=c["heads"], hidden_size=d, max_seq_len=L,
                       dropout_rate=c["dropout"], device=dev)
        core = mod._model.core
        to_batch = lambda b: {"inputs": {"item_id": b[0]}, "pad_mask": b[1], "token_mask": b[2], "positive_labels": b[3]}  # noqa: E731
    else:
        from replay_b200.nn.lightning import LightningModule
        from replay_b200.nn.sequential import SasRec

        schema = TensorSchema(TensorFeatureInfo("item_id", I, I, d))
        model = SasRec.from_params(schema, embedding_dim=d, num_heads=c["heads"], num_blocks=c["blocks"], max_sequence_length=L,
                                   dropout=c["dropout"], device=dev, seed=1234)
        mod = LightningModule(model)
        core = model.core
        to_batch = lambda b: {"feature_tensors": {"item_id": b[0]}, "padding_mask": b[1],  # noqa: E731
                              "positive_labels": b[2].unsqueeze(-1), "target_padding_mask": b[3].unsqueeze(-1)}
    return mod, core, to_batch


def run_ours(args):
    import torch.distributed as dist

    from replay_b200 import ops
    from replay_b200.trainer import Trainer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU: replay_b200 has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    c = dict(CONFIGS[args.config])
    if args.dropout is not None:
        c["dropout"] = args.dropout
    if args.batch is not None:
        c["per_gpu_batch"] = args.batch
    B, L, d, I = c["per_gpu_batch"], c["seq_len"], c["d"], c["n_items"]
    mod, core, to_batch = build_module(c, dev)
    eng = core.ensure_engine(B, L, with_grad=True)
    tr = Trainer(eng, use_graph=not args.no_graph)
    n_batches = 6
    data = make_batches(c, B * n_batches * world, seed=1234)
    if world > 1 and not args.no_balance:
        # global batch j = windows [j * world * B, (j + 1) * world * B) of the pool, dealt to the ranks by their number of valid
        # targets (replay_b200.data.balanced_rank_shards): the gradient exchange is a barrier, so every step runs at the pace
        # of the rank with the most targets - 3.7 % above the mean with index sharding at 8 ranks
        from replay_b200.data import balanced_rank_shards

        work = (data[3] if c["kind"] == "sasrec" else (data[1] & ~data[2])).reshape(n_batches, world * B, L).sum(-1)
        pick = torch.stack([balanced_rank_shards(work[j], world)[rank] + j * world * B for j in range(n_batches)])  # [n_batches, B]
        host = [t[pick.reshape(-1)].reshape(n_batches, B, L).pin_memory() for t in data]
    else:
        sh = slice(rank * B * n_batches, (rank + 1) * B * n_batches)
        host = [t[sh].reshape(n_batches, B, L).pin_memory() for t in data]
    devb = [t.to(dev) for t in host]
    valid_per_seq = valid_targets(c, data)
    eng.n_valid_hint = int(valid_per_seq * B)  # the data loader knows how many targets a batch holds (load balance only)
    PK = peaks()

    def step_dev(i):
        j = i % n_batches
        return tr.step(*(t[j] for t in devb))

    def step_e2e(i):  # pinned host batch -> device inside the module call, loss read back to the host, every step
        j = i % n_batches
        loss = mod.training_step(to_batch([h[j].to(dev, non_blocking=True) for h in host]), i)
        return float(loss.item())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = None
        for i in range(n):
            out = fn(i)
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), out

    W, K = max(args.warmup, 3), args.steps
    for i in range(W + 3):  # +3: two eager steps and the graph capture
        step_dev(i)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms, loss = timed(step_dev, K)
    clocks = sampler.stop() if rank == 0 else None
    final_loss = float(loss[0].item())
    # what the last timed step returned (loss buffer: mean CE, 1 / n_valid) and the parameters it left, before later legs
    # overwrite both
    outputs = {"train_loss": loss.cpu(), "train_params": param_sample(eng.p32)} if args.dump_outputs else None
    # ---- (N > 1) the gradient exchange alone: 20 back-to-back calls on the staged gradient, ranks in lock step
    exchange = None
    if world > 1:
        def xchg(_i):
            tr._all_reduce()
        xchg(0)
        ms_x, _ = timed(xchg, 20)
        exchange = {"kind": "rp_peer_allreduce (in-graph NVLink kernel)" if tr.peer is not None else "ncclAllReduce (eager, between two graphs)",
                    "ms": ms_x / 20, "bytes": int(eng.g32.numel() * 4), "balanced_batches": not args.no_balance}
        eng.g32.zero_()
    # ---- sustained: the same step for >= 2 s (power / thermal steady state), clocks sampled over the whole window
    sustained = None
    if not args.no_sustained:
        n_sus = max(K, int(2500.0 / (ms / K)))
        s2 = ClockSampler(local)
        if rank == 0:
            s2.start()
        ms_sus, _ = timed(step_dev, n_sus)
        sustained = {"value": world * B * n_sus / ms_sus * 1e3, "unit": "seq/s", "steps": n_sus, "seconds": ms_sus / 1e3,
                     "ms_per_step": ms_sus / n_sus, "clocks": s2.stop() if rank == 0 else None}
    # ---- e2e: the same step through the Lightning mirror's training_step with pinned host batches
    for i in range(4):  # the module's own warm-up + graph capture
        step_e2e(i)
    ms_e2e, _ = timed(step_e2e, K)
    h2d = sum(h[0].numel() * h[0].element_size() for h in host)
    # ---- same step fed by device-side batch construction (SASRec): histories resident in HBM as CSR, one rp_build_batch launch
    # per step cuts / left-pads / shifts the windows of B randomly drawn users (SURVEY 8 f.1), loss read back every step
    dev_batches = None
    if not args.no_device_batches and c["kind"] == "sasrec":
        from replay_b200.device_data import DeviceSequenceStore
        from replay_b200.synthetic import make_histories

        n_hist = 65536
        off_h, items_h = make_histories(n_hist, I, seed=1234 + rank)
        store = DeviceSequenceStore(offsets=off_h.numpy(), items=items_h.numpy(), device=dev)
        picks = torch.randint(0, n_hist, (n_batches, B), generator=torch.Generator().manual_seed(rank), dtype=torch.int32).to(dev)

        def step_store(i):
            b = store.sasrec_training_batch(picks[i % n_batches], L, I)
            loss = tr.step(b["feature_tensor"]["item_id"], b["padding_mask"], b["positive_labels"], b["target_padding_mask"])
            return float(loss[0].item())

        for i in range(2):
            step_store(i)
        ms_st, _ = timed(step_store, K)
        dev_batches = {"value": world * B * K / ms_st * 1e3, "unit": "seq/s", "ms_per_step": ms_st / K,
                       "histories_per_gpu": n_hist, "store_bytes": int(items_h.numel() * 4 + off_h.numel() * 8),
                       "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 4,
                       "note": "batches cut on the GPU from the HBM-resident CSR history store (rp_build_batch), no host input"}
        del store

    def time_kernel(fn, iters=10):
        fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / iters

    # ---- roofline of the dominant kernels: the tcgen05 CE-head kernels, timed live with CUDA events (standalone, same
    # buffers as the last step; each launch streams > L2 worth of operands through TMEM/SMEM)
    step_dev(0)
    torch.cuda.synchronize()
    n_valid = int(eng.n_valid.item())
    if c["kind"] == "bert":
        W16, bias = eng._head()
        dW, dbias = (eng.grads["item_emb"] if eng.cfg.tying else eng.grads["head_w"]), eng.grads["head_b"]
    else:
        W16, bias, dW, dbias = eng.params16["item_emb"][:I], None, eng.grads["item_emb"], None
    t_fwd = time_kernel(lambda: ops.ce_head_fwd(eng.ce, eng.hc, W16, eng.labels_c, eng.n_valid, bias=bias,
                                                d_hc=eng.s["dhc"] if eng.fused_ce else None, n_valid_hint=eng.n_valid_hint))
    t_bwd = time_kernel(lambda: ops.ce_head_bwd(eng.ce, eng.hc, W16, eng.labels_c, eng.n_valid, eng.s["dhc"], dW, bias=bias,
                                                d_bias=dbias, n_valid_hint=eng.n_valid_hint))
    fused_taken = bool(ops.ce_head_fused_taken(eng.ce)) if (eng.fused_ce and d <= 256) else False
    eng.g32.zero_()
    gemm_flops = 2.0 * n_valid * I * d
    ce_ms = t_fwd + t_bwd
    fused = bool(eng.fused_ce and d <= 256)
    n_exec = 4 if fused else 5  # GEMM-equivalents executed: fused fwd+dH (S, dH) + dE pass (S, dE); un-fused: S twice more
    traffic = measured_traffic(f"ce_head_c{args.config}_b{B}")
    roof = {
        "bound": "tensor",
        "kernel": ("ce_bwd_kernel<FUSED> (fwd+dH) + ce_bwd_kernel<COL> (dE)" if fused else "ce_fwd_kernel + materialised-G GEMMs (d = 512)")
                  + ": logits GEMM + softmax-CE, fwd+bwd",
        "achieved": 3 * gemm_flops / (ce_ms * 1e-3) / 1e12, "peak": PK["tc_burst"], "unit": "TFLOP/s",
        "frac": 3 * gemm_flops / (ce_ms * 1e-3) / 1e12 / PK["tc_burst"],
        # dram__bytes_read + dram__bytes_write per launch of the two passes (committed ncu capture of THIS shape), else null
        "traffic": traffic,
        "algorithmic_bytes": 2 * (I * d * 2 + n_valid * d * 2) + I * d * 4 + n_valid * d * 2,
        "peak_source": PK["src"] + " burst (kernels timed alone)",
        "detail": {"ce_fwd_ms": t_fwd, "ce_bwd_ms": t_bwd, "n_valid_targets": n_valid,
                   "algorithmic_flops_per_launch_pair": 3 * gemm_flops,
                   "executed_tflops": n_exec * gemm_flops / (ce_ms * 1e-3) / 1e12, "fused_fwd_dh": fused,
                   "fused_path_taken": fused_taken,  # False: the device-side bound on |logit| failed, the two-pass kernels ran
                   "share_of_step": ce_ms / (ms / K)},
    }
    launches = (tr.launches_per_step or 0) * K
    del tr

    # ---- scoring leg (config 2 only; every rank scores its own contiguous shard of the users, no collective: SURVEY 8e)
    scoring = None
    if args.config == 2 and not args.no_scoring:
        del mod, core, eng, devb
        torch.cuda.empty_cache()
        scoring = run_scoring(args, dev, rank, world, PK, barrier, time_kernel, outputs)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    seq_s = world * B * K / ms * 1e3
    fl_seq = train_flops_per_seq(c, valid_per_seq)
    step_tflops = seq_s / world * fl_seq / 1e12
    cpu = None
    if not args.no_cpu:
        v, med, _, _ = cpu_train_seq_per_s(c, steps=3 if args.config == 2 else 1, warmup=1)
        cpu = {"value": v, "unit": "seq/s", "cores": torch.get_num_threads(), "kind": "port",
               "sample": f"timed steps of batch {c['cpu_batch']} (fwd+bwd+Adam, dropout off) of the oracle port, torch fp32 CPU"}
    line = {
        "metric": "bert4rec_train_seq_per_s" if c["kind"] == "bert" else "sasrec_train_seq_per_s",
        "value": seq_s, "unit": "seq/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic",
        "config": {"workload": workload_string(c), "global_batch": world * B, "per_gpu_batch": B, "seq_len": L, "d": d, "n_items": I,
                   "parallelism": f"dp{world}", "valid_targets_per_seq": valid_per_seq, "cuda_graph": not args.no_graph,
                   "batch_sharding": ("one rank" if world == 1 else
                                      ("index" if args.no_balance else "global batch dealt to the ranks by valid-target count")),
                   "l2": "no flush: every step streams > 126 MB of activations / table"},
        "e2e": {"value": world * B * K / ms_e2e * 1e3, "unit": "seq/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                "ms_per_step": ms_e2e / K,
                "path": ("LightningModule(SasRec).training_step" if c["kind"] == "sasrec" else "Bert4Rec.training_step")
                        + " on pinned host batches (fused step: CUDA-graph replay, gradient exchange inside the module)"},
        "e2e_device_batches": dev_batches,
        "sustained": sustained, "gradient_exchange": exchange,
        "gpu_launches": launches,
        "clocks": clocks,
        "roofline": roof,
        "step_roofline": {"credited_flops_per_seq": fl_seq, "achieved_tflops_per_gpu": step_tflops,
                          "peak": PK["tc_sustained"], "frac": step_tflops / PK["tc_sustained"],
                          "note": "whole step vs sustained bf16 peak; FLOPs per SURVEY 8d (valid targets only, x3 for train)"},
        "cpu_baseline": cpu,
        "scoring": scoring,
        "final_loss": final_loss,
    }
    if outputs is not None:
        write_outputs(args.dump_outputs, outputs)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def run_scoring(args, dev, rank, world, PK, barrier, time_kernel, outputs=None):
    """BASELINE configs[3]: SASRec predict() top-K@10 over |I| = 500 000 with filter_seen_items, >= 1 M users per GPU.
    `value`: ids resident in HBM, engine calls (body, last-position shortcut, fused score + seen mask + top-K).
    `e2e`: pinned host ids -> ``LightningModule.predict_step`` + ``TorchTopItemsCallback(postprocessors=[SeenItemsFilter])`` ->
    top-K ids / scores copied back to pinned host memory, every call, inside the timed region.  ``outputs`` (a dict, or
    None) receives the top-K ids and scores of the last device-resident call at the headline call size."""
    import torch.distributed as dist

    from replay_b200 import ops
    from replay_b200.nn.lightning import LightningModule, SeenItemsFilter, TorchTopItemsCallback
    from replay_b200.nn.sequential import SasRec
    from replay_b200.schema import TensorFeatureInfo, TensorSchema
    from replay_b200.synthetic import make_sequences

    sc = SCORE_CFG
    I, d, L, K = sc["n_items"], sc["d"], sc["seq_len"], sc["k"]
    n_users = sc["users_per_gpu"] if not args.quick_scoring else 65_536
    distinct = min(sc["distinct_histories"], n_users)
    model = SasRec.from_params(TensorSchema(TensorFeatureInfo("item_id", I, I, d)), embedding_dim=d, num_heads=2, num_blocks=2,
                               max_sequence_length=L, dropout=0.0, device=dev, seed=7)
    model.eval()
    lm = LightningModule(model)
    uid, upm, _, _ = make_sequences(distinct, I, L, seed=7 + rank)  # this rank's shard of the users (exact partition)
    uid_h, upm_h = uid.pin_memory(), upm.pin_memory()
    uid_d, upm_d = uid.to(dev), upm.to(dev)
    core = model.core

    def maxr(x):
        t = torch.tensor([x], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def leg(Bu):
        n_calls = max(1, n_users // Bu)
        eng = core.ensure_engine(Bu, L, with_grad=False)
        if eng.B != Bu:  # exactly this call size (a larger workspace would make every call process its padding rows too)
            eng.resize(Bu, L)
        tab = core.item_table()
        per = distinct // Bu if distinct >= Bu else 0

        def sl(i):
            if per == 0:
                return slice(0, distinct)
            j = i % per
            return slice(j * Bu, (j + 1) * Bu)

        # device-resident inputs, through the model's fused predict (what the callbacks call): one graph replay per call
        # below 8192 users, the length-bucketed body above
        def call_dev(i):
            s = sl(i)
            return core.predict_topk(uid_d[s], upm_d[s], K, seen_ids=uid_d[s])

        for i in range(3):
            call_dev(i)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n_calls):
            top = call_dev(i)
        e1.record()
        barrier()
        ms_dev = maxr(e0.elapsed_time(e1))
        if outputs is not None and Bu == sc["users_per_call"]:
            outputs["score_topk_ids"], outputs["score_topk_scores"] = (t.cpu() for t in top)
        # end to end through the reference-facing callback
        cb = TorchTopItemsCallback(top_k=K, query_column="query_id", item_column="item_id",
                                   postprocessors=[SeenItemsFilter(item_count=I, seen_items_column="seen_ids")])
        out_ids = torch.empty(Bu, K, dtype=torch.int64).pin_memory()
        out_sc = torch.empty(Bu, K, dtype=torch.float32).pin_memory()
        qid = torch.arange(Bu, device=dev)

        def call_e2e(i):
            s = sl(i)
            ids = uid_h[s].to(dev, non_blocking=True)
            pm = upm_h[s].to(dev, non_blocking=True)
            batch = {"query_id": qid[: ids.shape[0]], "feature_tensors": {"item_id": ids}, "padding_mask": pm, "seen_ids": ids}
            cb._query_batches.clear(); cb._item_batches.clear(); cb._item_scores.clear()
            cb.on_predict_batch_end(None, lm, lm.predict_step(batch, i), batch, i)
            out_ids[: ids.shape[0]].copy_(cb._item_batches[0], non_blocking=True)
            out_sc[: ids.shape[0]].copy_(cb._item_scores[0], non_blocking=True)

        cb.on_predict_epoch_start(None, lm)
        for i in range(3):
            call_e2e(i)
        barrier()
        e0.record()
        for i in range(n_calls):
            call_e2e(i)
        e1.record()
        barrier()
        ms_e2e = maxr(e0.elapsed_time(e1))
        users = n_calls * min(Bu, distinct)
        return {"users_per_call": Bu, "calls": n_calls, "users_per_gpu": users,
                "value": world * users / ms_dev * 1e3, "ms_per_call": ms_dev / n_calls,
                "e2e": {"value": world * users / ms_e2e * 1e3, "unit": "users/s", "ms_per_call": ms_e2e / n_calls,
                        "h2d_bytes_per_call": min(Bu, distinct) * L * 9, "d2h_bytes_per_call": min(Bu, distinct) * K * 12}}

    sweep = {}
    sizes = [sc["users_per_call"]] if args.quick_scoring else list(sc["sweep"])
    for Bu in sizes:
        sweep[str(Bu)] = leg(Bu)
        torch.cuda.empty_cache()
    head = sweep[str(sc["users_per_call"])]
    if rank != 0:
        return None
    # roofline of the head kernel alone at the headline call size
    Bu = sc["users_per_call"]
    eng = core.ensure_engine(Bu, L, with_grad=False)
    if eng.B != Bu:
        eng.resize(Bu, L)
    eng.set_batch(uid_d[:Bu], upm_d[:Bu])
    hq = eng.forward_last_hidden()
    tab = core.item_table()
    seen = ops.seen_prepare(uid_d[:Bu], I)
    t_head = time_kernel(lambda: ops.score_topk(hq, tab, K, seen))
    head_flops = 2.0 * Bu * I * d
    return {
        "metric": "sasrec_predict_topk10_users_per_s", "value": head["value"], "unit": "users/s", "n_gpus": world,
        "config": {"workload": "BASELINE configs[3]: SASRec predict() top-K@10, body fwd (last-position shortcut) + fused score + "
                               "seen-item filter + top-10, users sharded contiguously over the GPUs (no collective); "
                               f"{n_users} users per GPU per sweep point, inputs cycle over {distinct} distinct synthetic histories per GPU",
                   "n_items": I, "d": d, "seq_len": L, "k": K, "users_per_call": Bu},
        "ms_per_call": head["ms_per_call"],
        "e2e": {**head["e2e"], "h2d_bytes_per_step": head["e2e"]["h2d_bytes_per_call"], "d2h_bytes_per_step": head["e2e"]["d2h_bytes_per_call"],
                "path": "pinned host ids -> LightningModule.predict_step -> TorchTopItemsCallback(SeenItemsFilter) -> top-K ids + scores -> pinned host"},
        "sweep": sweep,
        "cpu_baseline": None if args.no_cpu else {
            "value": cpu_predict_users_per_s(), "unit": "users/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": "64 users, 3 timed calls: oracle body + full logits + seen filter + torch.topk, torch fp32 CPU"},
        "roofline": {"bound": "tensor", "kernel": "score_topk_kernel", "achieved": head_flops / (t_head * 1e-3) / 1e12,
                     "peak": PK["tc_burst"], "unit": "TFLOP/s", "frac": head_flops / (t_head * 1e-3) / 1e12 / PK["tc_burst"],
                     "head_ms": t_head, "head_users_per_s": Bu / t_head * 1e3, "traffic": measured_traffic(f"score_topk_b{Bu}"),
                     "algorithmic_bytes": I * d * 2 + Bu * d * 2 + Bu * L * 4 + Bu * K * 12},
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS), help="BASELINE config: 2 (default), 3 (BERT4Rec), 5 (SASRec d=512 |I|=1M)")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-scoring", action="store_true")
    ap.add_argument("--quick-scoring", action="store_true", help="scoring leg on 65 536 users at 4096 users per call only")
    ap.add_argument("--no-sustained", action="store_true", help="skip the >= 2 s sustained window")
    ap.add_argument("--no-balance", action="store_true", help="N > 1: shard the global batch by index instead of dealing it by valid-target count")
    ap.add_argument("--no-device-batches", action="store_true", help="skip the device-side batch construction leg")
    ap.add_argument("--batch", type=int, default=None, help="sequences per GPU and step (SURVEY 8d sweeps {128, 256, 512} at config 2)")
    ap.add_argument("--dropout", type=float, default=None, help="diagnostic override of the workload's dropout; "
                    "a run with this flag is not the benchmark configuration")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed to DIR/<name>.npy (float32 / "
                         "float64, < 64 MB in all): train_loss, train_params (the updated fp32 parameters, a fixed seeded "
                         "sample of 8 Mi elements when larger) and, with the scoring leg, score_topk_ids / score_topk_scores "
                         "of its last call at the headline call size; the inputs are the same from run to run")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
