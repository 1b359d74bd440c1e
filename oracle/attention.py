"""fp64 restatement of the attention kernels (replay_b200/csrc/rp_attention.cu, rp_attention_bwd.cu).

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).  It starts from the same bf16 Q / K / V the kernels read, widened to
fp64, and restates what the kernels compute - not what the reference model computes - so that a kernel can be held to a
bf16-rounding tolerance instead of a model-level one:

* Visibility (rp_attention.cu:163,179-183; rp_attention_bwd.cu:90,205): key j is visible to query i iff j < L, j <= i
  when causal, and pad[b, j] when mask_pad_keys.  Any pad mask is allowed, not only left padding.
* A query row with no visible key has O = 0, inv_sum = 0, m_save = 0 and contributes nothing to dK / dV
  (rp_attention.cu:9,217,301; DESIGN.md section 4: torch >= 2.5 safe-softmax semantics).
* Scale 1/sqrt(head_dim) of the TRUE head dim: a head of 48 or 50 features inside a 64-wide slot (100 inside 128) has zero
  padded columns and is scaled by 1/sqrt(48) (include/rp_b200.h "PADDED FEATURE SLOTS"; engine.py passes the scale).
* Saved statistics (AttnParams, rp_attention.cu:23-25): m_save = row max * scale * log2 e (0 for a fully masked row),
  inv_sum = 1 / sum_j exp(s - max) (0 for a fully masked row), p_save = exp(s - max) BEFORE dropout, 0 where masked.
* Probability dropout (rp_philox.cuh drop_row_key / drop_col_key / drop_mix, restated below in uint32 arithmetic): the draw
  of (query i, key j) is drop_mix(drop_row_key(seed + *seed_ptr, drop_off, (b*H + h)*Lp + i), drop_col_key(j)) with
  Lp = round_up(L, 64); keep <=> draw >= floor(p * 2^32); kept probabilities are scaled by 1/(1 - p)
  (rp_attention.cu:170-173,281; rp_attention_bwd.cu:83-88,207,213).
* Backward (rp_attention_bwd.cu:9-17, rp_attention.cu:336-338): with Pd = P * mask / keep, dV = Pd^T dO,
  dP = (dO V^T) * mask / keep, delta_i = sum_c dO[i, c] O[i, c], dS = P * (dP - delta) * scale, dQ = dS K, dK = dS^T Q.

``mutate`` injects one plausible kernel bug into the restatement (tests/test_attention_oracle.py proves that every such bug
moves the outputs by more than four times the tolerance tests/test_gpu_attention.py allows).
"""
from __future__ import annotations

import math

import numpy as np
import torch

_M32 = 0xFFFFFFFF

# Tolerances of tests/test_gpu_attention.py (argument in its module docstring): max |x - x_ref| <= TOL[x] * scale(x), with
# scale(O) = max |V| and scale(dQ / dK / dV) = max |dQ_ref| / max |dK_ref| / max |dV_ref|.
TOL = {"O": 6e-3, "dQ": 1.5e-2, "dK": 1.5e-2, "dV": 1.5e-2}


def tol_scale(name: str, ref: dict, inputs: dict) -> float:
    """What TOL[name] is relative to.  dQ and dK vanish identically at L = 1 (one key: dS = P (dP - delta) = 0); there the
    kernels' round-off of delta against dP is compared with 1e-3."""
    if name == "O":
        return float(inputs["v"].double().abs().max())
    return max(float(ref[name].abs().max()), 1e-3)


MODES = {  # mask mode -> (causal, mask_pad_keys)
    "sasrec": (1, 1),   # replay/nn/sequential/sasrec: causal + key padding
    "legacy": (1, 0),   # replay/models/nn/sequential/sasrec: causal only (pad rows zeroed after the block)
    "bert": (0, 1),     # BERT4Rec: key padding only
}


# ------------------------------------------------------------------------------------------------ dropout draws (uint32)
def _fmix32_int(h: int) -> int:
    h ^= h >> 16
    h = (h * 0x85EBCA6B) & _M32
    h ^= h >> 13
    h = (h * 0xC2B2AE35) & _M32
    h ^= h >> 16
    return h


def _fmix32(h: np.ndarray) -> np.ndarray:
    h = h.astype(np.uint32)
    h ^= h >> np.uint32(16)
    h *= np.uint32(0x85EBCA6B)
    h ^= h >> np.uint32(13)
    h *= np.uint32(0xC2B2AE35)
    h ^= h >> np.uint32(16)
    return h


def drop_row_key(seed: int, off: int, rows: np.ndarray) -> np.ndarray:
    """rp_philox.cuh drop_row_key for an array of (64-bit) row indices."""
    seed &= (1 << 64) - 1
    off &= (1 << 64) - 1
    s = _fmix32_int((seed & _M32) ^ (((seed >> 32) * 0x85EBCA77) & _M32) ^ (((off >> 32) * 0xC2B2AE3D) & _M32)
                    ^ (((off & _M32) * 0x27D4EB2F) & _M32))
    r = np.asarray(rows).astype(np.uint64)
    lo = (r & np.uint64(_M32)).astype(np.uint32)
    hi = (r >> np.uint64(32)).astype(np.uint32)
    return _fmix32(np.uint32(s) + lo * np.uint32(0x9E3779B1) + hi * np.uint32(0x165667B1))


def drop_col_key(j: np.ndarray) -> np.ndarray:
    return _fmix32(np.asarray(j).astype(np.uint32) * np.uint32(0x9E3779B1) + np.uint32(0x27D4EB2F))


def drop_mix(row_key: np.ndarray, col_key: np.ndarray) -> np.ndarray:
    x = (row_key ^ col_key) * np.uint32(0x9E3779B1)
    x ^= x >> np.uint32(15)
    return x * np.uint32(0x85EBCA77)


def drop_threshold(p: float) -> int:
    """(uint32_t)(drop_p * 4294967296.0) with drop_p a float32 (the kernels' argument type)."""
    return int(float(np.float32(p)) * 4294967296.0)


def keep_mask(B: int, H: int, L: int, p: float, seed: int, drop_off: int, seed_counter: int = 0, *, row_shift: int = 0,
              pitch: int | None = None, invert: bool = False) -> torch.Tensor:
    """bool [B, H, L, L]: True where probability (i, j) of head (b, h) is kept.  ``row_shift`` / ``pitch`` / ``invert`` are
    the mutations of the row key and the threshold."""
    Lp = -(-L // 64) * 64 if pitch is None else pitch
    bz = np.arange(B * H, dtype=np.int64)[:, None]
    i = np.arange(L, dtype=np.int64)[None, :]
    rows = (bz * Lp + i + row_shift).astype(np.uint64)          # negative rows wrap like the kernels' unsigned arithmetic
    rk = drop_row_key(seed + seed_counter, drop_off, rows)      # [BH, L]
    ck = drop_col_key(np.arange(L))                              # [L]
    draw = drop_mix(rk[:, :, None], ck[None, None, :])          # [BH, L, L]
    keep = draw >= np.uint32(drop_threshold(p))
    if invert:
        keep = ~keep
    return torch.from_numpy(keep.reshape(B, H, L, L))


# ------------------------------------------------------------------------------------------------ reference
def attention(q, k, v, pad, *, causal: int, mask_pad_keys: int, head_dim: int, drop_p: float = 0.0, seed: int = 0,
              seed_counter: int = 0, drop_off: int = 0, d_out=None, mutate: str | None = None) -> dict:
    """q, k, v, d_out: [B, L, H, slot] (any float dtype, widened to fp64); pad: [B, L] bool (True = real token).

    Returns fp64 tensors: O [B, L, H, slot]; m_save, inv_sum [B, H, L]; p_save [B, H, L, L]; keep [B, H, L, L] (the
    dropout multiplier mask / keep, 1 without dropout); and, when d_out is given, dQ / dK / dV [B, L, H, slot]."""
    B, L, H, slot = q.shape
    qd, kd, vd = (t.to(torch.float64).permute(0, 2, 1, 3) for t in (q, k, v))   # [B, H, L, slot]
    pad = pad.to(torch.bool)
    scale = 1.0 / math.sqrt(slot if mutate == "slot_scale" else head_dim)
    ii = torch.arange(L)[:, None]
    jj = torch.arange(L)[None, :]
    vis = torch.ones(B, L, L, dtype=torch.bool)
    if causal:
        shift = {"diag+1": 1, "diag-1": -1}.get(mutate, 0)
        vis &= jj <= ii + shift
    if mask_pad_keys and mutate != "ignore_pad":
        src = torch.roll(pad, -1, 0) if mutate == "pad_neighbour" else pad
        vis &= src[:, None, :]
    if mutate is not None and mutate.startswith("drop_key:"):
        j = int(mutate.split(":")[1])
        if j < L:
            vis[:, :, j] = False
    vis = vis[:, None].expand(B, H, L, L)
    s = (qd @ kd.transpose(-1, -2)) * scale
    any_vis = vis.any(-1)
    mx = torch.where(vis, s, torch.full_like(s, -math.inf)).amax(-1)
    mx0 = torch.where(any_vis, mx, torch.zeros_like(mx))
    e = torch.where(vis, torch.exp(s - mx0[..., None]), torch.zeros_like(s))
    ssum = e.sum(-1)
    inv = torch.where(any_vis, 1.0 / torch.where(any_vis, ssum, torch.ones_like(ssum)), torch.zeros_like(ssum))
    P = e * inv[..., None]
    if mutate == "masked_uniform":   # a fully masked row spreads uniformly over its window instead of giving zero
        window = (jj <= ii) if causal else torch.ones(L, L, dtype=torch.bool)
        uni = window.double() / window.double().sum(-1, keepdim=True)
        P = torch.where(any_vis[..., None], P, uni.expand_as(P))
    keep = torch.ones_like(P)
    if drop_p > 0:
        km = keep_mask(B, H, L, drop_p, seed, drop_off, seed_counter,
                       row_shift={"rowkey+1": 1, "rowkey-1": -1}.get(mutate, 0),
                       pitch=L if mutate == "pitch_L" else None, invert=mutate == "thr_inv")
        ks = 1.0 if mutate == "no_rescale" else 1.0 / (1.0 - float(np.float32(drop_p)))
        keep = km.double() * ks
    Pd = P * keep
    O = Pd @ vd
    out = {"O": O.permute(0, 2, 1, 3).contiguous(), "m_save": mx0 * math.log2(math.e), "inv_sum": inv, "p_save": e,
           "keep": keep, "vis": vis, "scale": scale}
    if d_out is not None:
        g = d_out.to(torch.float64).permute(0, 2, 1, 3)
        dV = Pd.transpose(-1, -2) @ g
        dP = (g @ vd.transpose(-1, -2)) * keep
        delta = (g * O).sum(-1, keepdim=True)
        dS = P * (dP - delta) * scale
        dQ = dS @ kd
        dK = dS.transpose(-1, -2) @ qd
        for name, t in (("dQ", dQ), ("dK", dK), ("dV", dV)):
            out[name] = t.permute(0, 2, 1, 3).contiguous()
    return out


# ------------------------------------------------------------------------------------------------ test cases
def make_pad(B: int, L: int, mode: str, gen: torch.Generator) -> torch.Tensor:
    """[B, L] bool: sequence 0 all padding, sequence 1 full, the rest random left padding; BERT4Rec masks (key padding
    only) also get random holes inside the history."""
    pad = torch.zeros(B, L, dtype=torch.bool)
    pad[1] = True
    for b in range(2, B):
        n = int(torch.randint(1, L + 1, (1,), generator=gen))
        pad[b, L - n:] = True
        if mode == "bert" and L > 2:
            holes = torch.rand(L, generator=gen) < 0.15
            pad[b] &= ~holes
            pad[b, L - 1] = True
    return pad


def make_inputs(B: int, H: int, L: int, slot: int, head_dim: int, mode: str, seed: int) -> dict:
    """bf16 Q / K / V / dO [B, L, H, slot] with zero padded-slot columns and a peaked attention pattern: every query leans
    towards its own key (logit ~ 0.6 * head_dim / sqrt(head_dim) above a N(0, 1.2^2) background), so a single key - the
    last one, one at a 32- / 128- / 256-column boundary, the diagonal - carries a large share of some row.  V has a
    per-column mean so that a fully masked row spread uniformly is far from zero."""
    gen = torch.Generator().manual_seed(seed)
    shape = (B, L, H, slot)
    kk = torch.randn(shape, generator=gen)
    qq = torch.randn(shape, generator=gen) + 0.6 * kk
    vv = torch.randn(shape, generator=gen) + (torch.rand(1, 1, H, slot, generator=gen) * 2 - 1)
    do = torch.randn(shape, generator=gen) * 0.5
    out = {}
    for name, t in (("q", qq), ("k", kk), ("v", vv), ("d_out", do)):
        t = t.clone()
        t[..., head_dim:] = 0
        out[name] = t.to(torch.bfloat16)
    out["pad"] = make_pad(B, L, mode, gen)
    return out


FWD_LENGTHS = {  # (slot, resident 256-key blocks) -> lengths: every 32 / 64 / 128 / 256-key boundary and both sides of it
    (64, 1): [1, 2, 31, 33, 63, 64, 65, 127, 128, 129, 200, 255, 256],
    (64, 2): [257, 300, 384, 385, 511, 512],
    (128, 1): [1, 65, 128, 129, 200, 256],
}
# fused backward (head_dim 64, L <= 256): weight on L mod 128 in [1, 64], where one 64-query half of the last tile is live
BWD_LENGTHS = [1, 2, 31, 33, 63, 64, 65, 100, 127, 128, 129, 160, 192, 200, 255, 256]
_PAD_HD = {64: (48, 50), 128: (100, 100)}


def _case(k: int, L: int, slot: int, modes, drops) -> dict:
    mode = modes[k % len(modes)]
    drop = drops[(k // len(modes)) % len(drops)]
    H = (1, 2, 4, 8)[k % 4]
    head_dim = slot
    if mode != "bert" and k % 5 in (1, 3):     # BERT4Rec has no padded layout (head_dim 64 / 128 only)
        head_dim = _PAD_HD[slot][(k // 5) % 2]
    return dict(L=L, slot=slot, head_dim=head_dim, mode=mode, H=H, B=4, drop=drop, seed=1000 + 37 * k + L)


def fwd_cases() -> list[dict]:
    cases, k = [], 0
    for (slot, _kb), lengths in FWD_LENGTHS.items():
        for L in lengths:
            cases.append(_case(k, L, slot, ("sasrec", "legacy", "bert"), (0.0, 0.2)))
            k += 1
    return cases


def bwd_cases() -> list[dict]:
    return [_case(k, L, 64, ("sasrec", "bert"), (0.0, 0.2)) for k, L in enumerate(BWD_LENGTHS)]


def case_id(c: dict) -> str:
    return f"L{c['L']}-hd{c['head_dim']}of{c['slot']}-{c['mode']}-H{c['H']}-p{c['drop']}"


SEED, SEED_COUNTER, DROP_OFF = 0x5EED1234ABCD, 0x9E3779B97F4A, 3 << 40


def reference_for(c: dict, inputs: dict, with_grad: bool = False, mutate: str | None = None) -> dict:
    causal, mpk = MODES[c["mode"]]
    return attention(inputs["q"], inputs["k"], inputs["v"], inputs["pad"], causal=causal, mask_pad_keys=mpk,
                     head_dim=c["head_dim"], drop_p=c["drop"], seed=SEED, seed_counter=SEED_COUNTER, drop_off=DROP_OFF,
                     d_out=inputs["d_out"] if with_grad else None, mutate=mutate)


def mutations_for(c: dict) -> list[str]:
    """The bugs the restatement can inject that are reachable in case ``c`` (a mutation that cannot change anything at
    this shape - a diagonal shifted up at L = 1, dropout keys without dropout - is left out)."""
    causal, mpk = MODES[c["mode"]]
    L = c["L"]
    m = []
    if causal and L >= 2:
        m.append("diag+1")
    if causal:
        m.append("diag-1")
    if mpk:
        m += ["ignore_pad", "pad_neighbour"]
    m.append(f"drop_key:{L - 1}")
    m += [f"drop_key:{j}" for j in (255, 256) if j < L - 1]
    if c["head_dim"] != c["slot"]:
        m.append("slot_scale")
    if c["drop"] > 0:
        m += ["rowkey+1", "rowkey-1", "thr_inv", "no_rescale"]
        if L % 64:
            m.append("pitch_L")
    if mpk:   # sequence 0 is all padding: its rows see no key
        m.append("masked_uniform")
    return m
