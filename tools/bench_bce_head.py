"""Time the full-catalog BCE head against the CE head (forward + backward each, same process, alternating) at the config-2
and config-3 head shapes.

    python tools/bench_bce_head.py [--reps 7] [--iters 10] [--out results.json]

config 2: SASRec, 512 x 200 positions, 55 574 valid targets, |I| = 50 000, d = 128, tied head (no bias)
config 3: BERT4Rec, 256 x 200 positions, 3 997 masked targets, |I| = 100 000, d = 256, biased head
Each timed call runs on one of four independent input sets in turn (hidden rows, item table, labels; > 126 MB together at
both shapes), so the operands do not stay in L2 between calls.  Times come from CUDA events around `iters` calls; the median
over `reps` alternating BCE / CE rounds is reported, with the credited rate 3 * 2 * d * |I| FLOP per valid target (the
logits GEMM, dH and dE) and the card's name and power limit.  Needs a GPU: without one it exits with an error.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

SHAPES = {"config2": dict(T=102_400, n_valid=55_574, I=50_000, d=128, bias=False),
          "config3": dict(T=51_200, n_valid=3_997, I=100_000, d=256, bias=True)}
N_SETS = 4


def card():
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        power, sm_clock = [x.strip() for x in q[torch.cuda.current_device()].split(",")]
    except Exception as e:  # noqa: BLE001 - the numbers are still worth printing, flagged
        power, sm_clock = f"unknown ({type(e).__name__})", "unknown"
    return dict(name=name, power_limit=power, max_sm_clock=sm_clock)


def bench_shape(T, n_valid, I, d, bias, reps, iters):
    from replay_b200.ops import BCEHeadState, CEHeadState, bce_head_bwd, bce_head_fwd, ce_head_bwd, ce_head_fwd

    dev = torch.device("cuda")
    g = torch.Generator(device="cuda").manual_seed(0)
    sets = []
    for _ in range(N_SETS):
        hc = (torch.randn(T, d, device=dev, generator=g) * 0.5).bfloat16()
        hc[n_valid:] = 0
        table = (torch.randn(I, d, device=dev, generator=g) * 0.1).bfloat16()
        labels = torch.randint(0, I, (T,), device=dev, generator=g, dtype=torch.int32)
        b = None
        if bias:
            b = torch.zeros((I + 127) // 128 * 128, device=dev)
            b[:I] = torch.randn(I, device=dev, generator=g) * 0.5
        sets.append((hc, table, labels, b))
    nv = torch.tensor([n_valid], dtype=torch.int32, device=dev)
    d_hc = torch.zeros(T, d, device=dev, dtype=torch.bfloat16)
    d_tab = torch.zeros(I, d, device=dev)
    d_b = torch.zeros((I + 127) // 128 * 128, device=dev) if bias else None
    ce, bce = CEHeadState(T, I, d, dev), BCEHeadState(T, I, d, dev)

    def ce_step(k):
        hc, table, labels, b = sets[k % N_SETS]
        ce_head_fwd(ce, hc, table, labels, nv, bias=b, d_hc=d_hc, n_valid_hint=n_valid)
        ce_head_bwd(ce, hc, table, labels, nv, d_hc, d_tab, bias=b, d_bias=d_b, n_valid_hint=n_valid)

    def bce_step(k):
        hc, table, labels, b = sets[k % N_SETS]
        bce_head_fwd(bce, hc, table, labels, nv, d_hc, bias=b, n_valid_hint=n_valid)
        bce_head_bwd(bce, hc, table, labels, nv, d_tab, bias=b, d_bias=d_b)

    def timed(step):
        a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for k in range(iters):
            step(k)
        e.record()
        torch.cuda.synchronize()
        return a.elapsed_time(e) / iters

    for step in (ce_step, bce_step):   # warm-up: module load, function attributes, every input set once
        for k in range(2 * N_SETS):
            step(k)
    torch.cuda.synchronize()
    t_ce, t_bce = [], []
    for _ in range(reps):
        t_ce.append(timed(ce_step))
        t_bce.append(timed(bce_step))
    med = lambda v: sorted(v)[len(v) // 2]  # noqa: E731
    flop = 3 * 2 * d * I * n_valid
    ms_ce, ms_bce = med(t_ce), med(t_bce)
    return dict(T=T, n_valid=n_valid, n_items=I, d=d, bias=bias, ce_ms=round(ms_ce, 4), bce_ms=round(ms_bce, 4),
                ce_tflops=round(flop / ms_ce / 1e9, 1), bce_tflops=round(flop / ms_bce / 1e9, 1),
                bce_over_ce=round(ms_bce / ms_ce, 3), ce_ms_all=[round(x, 4) for x in t_ce],
                bce_ms_all=[round(x, 4) for x in t_bce], bce_loss=float(bce.loss[0]), ce_loss=float(ce.loss[0]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--shapes", default="config2,config3")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_bce_head: no CUDA device - these numbers are only measured on the GPU")
    res = dict(card=card(), shapes={})
    for name in a.shapes.split(","):
        r = bench_shape(**SHAPES[name], reps=a.reps, iters=a.iters)
        res["shapes"][name] = r
        print(f"{name}: CE {r['ce_ms']:.3f} ms ({r['ce_tflops']} TFLOP/s credited)  BCE {r['bce_ms']:.3f} ms "
              f"({r['bce_tflops']} TFLOP/s)  BCE/CE {r['bce_over_ce']}", flush=True)
    print(f"card: {res['card']}")
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
