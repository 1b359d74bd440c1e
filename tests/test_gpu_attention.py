"""Kernel-level parity of every attention route against the fp64 restatement in oracle/attention.py, through the C ABI:
rp_attn_fwd (attn_fwd_kernel<64,1>, <64,2>, <128,1>), the fused rp_attn_bwd, rp_attn_softmax_bwd (both templates) and
rp_attn_last (64 and 128), in the engines' own layouts (SASRec: Q [T, dp] + packed KV [T, 2 dp]; BERT4Rec: packed
QKV [T, 3 d]).  Inputs are peaked (oracle.attention.make_inputs) so that a single key carries a large share of some row.

Tolerances (oracle.attention.TOL; tests/test_attention_oracle.py proves every modelled kernel bug exceeds them 4x):
* O: max |O - O_ref| <= 6e-3 * max |V|.  S = Q K^T is exact products of bf16 values summed in fp32 (relative error ~1e-6);
  the only coarse roundings are P -> bf16 before the P.V MMA (at most 2^-9 of each term, so at most 2^-9 * sum_j P_j |V_j|
  <= 2^-9 / (1 - p) * max |V|) and the bf16 output (2^-9 * |O| <= 2^-9 / (1 - p) * max |V|): at p = 0.2 together 4.9e-3.
* dQ / dK / dV: max error <= 1.5e-2 * max |ref| (1e-3 floor: dQ and dK vanish at L = 1).  dS and Pd are rounded to bf16
  (2^-9 each) and the outputs are bf16, but the dominant term is delta = sum_c dO O taken from the bf16 O: dS = P (dP -
  delta) cancels, most at short rows, so dQ / dK carry an error of 2^-9 |dO| |O| against a small result.  Measured on a
  B200 (1000 W limit) the largest error is 0.66 of this tolerance (dK, L = 2, two keys per row).
* m_save: 2e-4 * max(1, max |m_ref|); inv_sum: relative 1e-3; p_save (bf16 of values in [0, 1]): 3e-3.
* Dropout masks are compared EXACTLY: through V = I (forward) and through dpd = 0 (softmax backward, bit for bit).
"""
import ctypes
import math

import numpy as np
import pytest
import torch

from oracle import attention as oa

pytestmark = pytest.mark.gpu

RP_ESHAPE = -2


@pytest.fixture(scope="module")
def rp():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    from replay_b200._lib import lib

    return lib()


def _st():
    return torch.cuda.current_stream().cuda_stream


def _inputs(c):
    return oa.make_inputs(c["B"], c["H"], c["L"], c["slot"], c["head_dim"], c["mode"], c["seed"])


class _Case:
    """Device buffers of one case in the engine layout of its mask mode."""

    def __init__(self, c, inputs):
        self.c = c
        B, L, H, slot = inputs["q"].shape
        self.B, self.L, self.H, self.slot, self.T, self.dp = B, L, H, slot, B * L, H * slot
        self.causal, self.mpk = oa.MODES[c["mode"]]
        T, dp = self.T, self.dp
        q, k, v = (inputs[n].reshape(T, dp) for n in ("q", "k", "v"))
        if c["mode"] == "bert":   # packed QKV [T, 3d]
            self.Q = self.K = self.V = torch.cat([q, k, v], 1).cuda()
            self.c0 = (0, dp, 2 * dp)
        else:                     # Q [T, dp] + packed KV [T, 2 dp]
            self.Q = q.cuda()
            self.K = self.V = torch.cat([k, v], 1).cuda()
            self.c0 = (0, 0, dp)
        self.pad = inputs["pad"].reshape(-1).to(torch.uint8).cuda()
        self.d_out = inputs["d_out"].reshape(T, dp).cuda()
        self.ctr = torch.tensor([oa.SEED_COUNTER], dtype=torch.int64, device="cuda")
        self.Lp = -(-L // 64) * 64

    def fwd(self, stats=True, p_save=True, O=None):
        c = self.c
        B, L, H, T, dp, Lp = self.B, self.L, self.H, self.T, self.dp, self.Lp
        from replay_b200._lib import AttnDesc, check, lib

        ad = AttnDesc()
        for nm, t, c0 in (("q", self.Q, self.c0[0]), ("k", self.K, self.c0[1]), ("v", self.V, self.c0[2])):
            setattr(ad, nm, t.data_ptr())
            setattr(ad, nm + "_rows", t.shape[0]); setattr(ad, nm + "_cols", t.shape[1]); setattr(ad, "ld" + nm, t.stride(0))
            setattr(ad, nm + "_c0", c0)
        ad.B, ad.H, ad.L, ad.head_dim = B, H, L, self.slot
        ad.causal, ad.mask_pad_keys = self.causal, self.mpk
        ad.scale = 1.0 / math.sqrt(c["head_dim"])
        ad.pad_mask = self.pad.data_ptr()
        out = {"O": torch.full((T, dp), float("nan"), dtype=torch.bfloat16, device="cuda") if O is None else O}
        ad.out, ad.ldo = out["O"].data_ptr(), dp
        if stats:
            out["m_save"] = torch.zeros(B * H, Lp, device="cuda")
            out["inv_sum"] = torch.zeros(B * H, Lp, device="cuda")
            ad.m_save, ad.inv_sum = out["m_save"].data_ptr(), out["inv_sum"].data_ptr()
            if p_save:
                out["p_save"] = torch.zeros(B * H, Lp, Lp, dtype=torch.bfloat16, device="cuda")
                ad.p_save = out["p_save"].data_ptr()
        ad.drop_p, ad.seed, ad.drop_off, ad.seed_ptr = c["drop"], oa.SEED, oa.DROP_OFF, self.ctr.data_ptr()
        check(lib().rp_attn_fwd(ctypes.byref(ad), _st()), "rp_attn_fwd")
        torch.cuda.synchronize()
        return out

    def bwd(self, f):
        c = self.c
        B, L, H, T, dp = self.B, self.L, self.H, self.T, self.dp
        from replay_b200._lib import AttnBwdDesc, check, lib

        bd = AttnBwdDesc()
        for nm, t, c0 in (("q", self.Q, self.c0[0]), ("k", self.K, self.c0[1]), ("v", self.V, self.c0[2])):
            setattr(bd, nm, t.data_ptr())
            setattr(bd, nm + "_rows", t.shape[0]); setattr(bd, nm + "_cols", t.shape[1]); setattr(bd, "ld" + nm, t.stride(0))
            setattr(bd, nm + "_c0", c0)
        bd.d_out, bd.do_rows, bd.do_cols, bd.ld_do = self.d_out.data_ptr(), T, dp, dp
        bd.out, bd.ldo = f["O"].data_ptr(), dp
        bd.B, bd.H, bd.L, bd.head_dim = B, H, L, self.slot
        bd.causal, bd.mask_pad_keys = self.causal, self.mpk
        bd.scale = 1.0 / math.sqrt(c["head_dim"])
        bd.pad_mask = self.pad.data_ptr()
        bd.m_save, bd.inv_sum = f["m_save"].data_ptr(), f["inv_sum"].data_ptr()
        nan = float("nan")
        if c["mode"] == "bert":
            g = torch.full((T, 3 * dp), nan, dtype=torch.bfloat16, device="cuda")
            outs = (g, g, g)
        else:
            gq = torch.full((T, dp), nan, dtype=torch.bfloat16, device="cuda")
            gkv = torch.full((T, 2 * dp), nan, dtype=torch.bfloat16, device="cuda")
            outs = (gq, gkv, gkv)
        for nm, t, c0 in (("dq", outs[0], self.c0[0]), ("dk", outs[1], self.c0[1]), ("dv", outs[2], self.c0[2])):
            setattr(bd, nm, t.data_ptr()); setattr(bd, "ld_" + nm, t.stride(0)); setattr(bd, nm + "_c0", c0)
        bd.drop_p, bd.seed, bd.drop_off, bd.seed_ptr = c["drop"], oa.SEED, oa.DROP_OFF, self.ctr.data_ptr()
        check(lib().rp_attn_bwd(ctypes.byref(bd), _st()), "rp_attn_bwd")
        torch.cuda.synchronize()
        cols = lambda t, c0: t[:, c0:c0 + dp].float().cpu().view(B, L, H, self.slot)  # noqa: E731
        return {"dQ": cols(outs[0], self.c0[0]), "dK": cols(outs[1], self.c0[1]), "dV": cols(outs[2], self.c0[2])}


def _err(got, ref, name, ref_all, inputs):
    """error in units of the tolerance"""
    return float((got.double() - ref).abs().max()) / (oa.TOL[name] * oa.tol_scale(name, ref_all, inputs))


def _check_stats(cs, f, ref):
    B, H, L = cs.B, cs.H, cs.L
    m = f["m_save"].cpu().double().view(B, H, -1)[..., :L]
    inv = f["inv_sum"].cpu().double().view(B, H, -1)[..., :L]
    assert float((m - ref["m_save"]).abs().max()) <= 2e-4 * max(1.0, float(ref["m_save"].abs().max()))
    assert torch.equal(inv == 0, ref["inv_sum"] == 0)
    rel = ((inv - ref["inv_sum"]).abs() / ref["inv_sum"].clamp_min(1e-30))[ref["inv_sum"] > 0]
    assert rel.numel() == 0 or float(rel.max()) <= 1e-3
    if "p_save" in f:
        ps = f["p_save"].cpu().double().view(B, H, cs.Lp, cs.Lp)
        assert float((ps[:, :, :L, :L] - ref["p_save"]).abs().max()) <= 3e-3
        assert (ps[:, :, :L, :L][ref["p_save"] == 0] == 0).all()   # masked entries are exactly zero
        assert (ps[:, :, L:, :] == 0).all() and (ps[:, :, :, L:] == 0).all()


# ------------------------------------------------------------------------------------------------ forward
@pytest.mark.parametrize("c", oa.fwd_cases(), ids=oa.case_id)
def test_attn_fwd_matches_fp64(rp, c, record_property):
    inputs = _inputs(c)
    ref = oa.reference_for(c, inputs)
    cs = _Case(c, inputs)
    f = cs.fwd()
    O = f["O"].float().cpu().view(cs.B, cs.L, cs.H, cs.slot)
    e = _err(O, ref["O"], "O", ref, inputs)
    record_property("err_O", e)
    assert e <= 1.0, f"O error {e:.3f} x tolerance"
    assert (O[..., c["head_dim"]:] == 0).all()          # padded-slot columns stay exactly zero
    none = ~ref["vis"].any(-1)                          # [B, H, L] rows without a visible key
    assert (O.permute(0, 2, 1, 3)[none] == 0).all()
    _check_stats(cs, f, ref)
    # inference call (no saved statistics): live query tiles bit-identical, all-pad query tiles written as zeros
    g = cs.fwd(stats=False)["O"].cpu().view(cs.B, cs.L, -1)
    f16 = f["O"].cpu().view(cs.B, cs.L, -1)
    tiles = -(-cs.L // 128)
    padt = torch.nn.functional.pad(inputs["pad"], (0, tiles * 128 - cs.L)).view(cs.B, tiles, 128).any(-1)
    live = padt.repeat_interleave(128, 1)[:, :cs.L]
    assert torch.equal(g[live].view(torch.int16), f16[live].view(torch.int16))
    assert (g[~live] == 0).all()


@pytest.mark.parametrize("L,mode", [(1, "sasrec"), (33, "bert"), (50, "legacy"), (64, "sasrec"), (64, "bert")])
def test_attn_fwd_dropout_mask_exact(rp, L, mode):
    """V = I_64 (rows of every sequence): O[i, j] = P[i, j] * mask / keep, so the forward's dropout mask reads out
    element by element and must equal the restatement of rp_philox.cuh exactly."""
    c = dict(L=L, slot=64, head_dim=64, mode=mode, H=2, B=4, drop=0.2, seed=77 + L)
    inputs = _inputs(c)
    eye = torch.zeros(c["B"], L, c["H"], 64)
    eye[:, torch.arange(L), :, torch.arange(L)] = 1.0
    inputs["v"] = eye.to(torch.bfloat16)
    ref = oa.reference_for(c, inputs)
    cs = _Case(c, inputs)
    O = cs.fwd()["O"].float().cpu().view(c["B"], L, c["H"], 64).permute(0, 2, 1, 3)   # [B, H, i, j]
    want = ref["vis"] & (ref["keep"] > 0)
    assert ref["p_save"][ref["vis"]].min() > 1e-30          # every visible probability is representable
    assert torch.equal(O[..., :L] != 0, want), int(((O[..., :L] != 0) != want).sum())
    assert (O[..., L:] == 0).all()
    assert float((O[..., :L].double() - ref["O"].permute(0, 2, 1, 3)[..., :L]).abs().max()) <= oa.TOL["O"] * 1.25


# ------------------------------------------------------------------------------------------------ fused backward
@pytest.mark.parametrize("c", oa.bwd_cases(), ids=oa.case_id)
def test_attn_bwd_fused_matches_fp64(rp, c, record_property):
    inputs = _inputs(c)
    ref = oa.reference_for(c, inputs, with_grad=True)
    cs = _Case(c, inputs)
    f = cs.fwd(p_save=False)
    g = cs.bwd(f)
    errs = {k: _err(g[k], ref[k], k, ref, inputs) for k in ("dQ", "dK", "dV")}
    for k, v in errs.items():
        record_property("err_" + k, v)
    assert max(errs.values()) <= 1.0, errs
    hd = c["head_dim"]
    for k in ("dQ", "dK", "dV"):
        assert (g[k][..., hd:] == 0).all(), k               # padded-slot columns exactly zero
    none = ~ref["vis"].any(-1)                               # fully masked queries: dQ row exactly zero
    assert (g["dQ"].permute(0, 2, 1, 3)[none] == 0).all()


# ------------------------------------------------------------------------------------------------ softmax backward
@pytest.mark.parametrize("L,drop", [(1, 0.2), (63, 0.0), (64, 0.2), (65, 0.2), (200, 0.0), (256, 0.2),
                                    (257, 0.2), (300, 0.0), (384, 0.2), (511, 0.2), (512, 0.0)])
def test_attn_softmax_bwd_contract(rp, L, drop):
    """rp_attn_softmax_bwd: dpd := P (dP - sum_j P_j dP_j) scale and p_save := P mask / keep with P = p_save inv_sum,
    dP = dpd mask / keep (rp_attention.cu:336-338).  With dpd = 0 the second output exposes the dropout mask: bit for bit."""
    from replay_b200._lib import check

    BH, Lp, scale = 6, -(-L // 64) * 64, 1 / math.sqrt(48)
    gen = torch.Generator().manual_seed(L)
    p = torch.zeros(BH, Lp, Lp)
    p[:, :L, :L] = torch.rand(BH, L, L, generator=gen) ** 3
    p = p.to(torch.bfloat16)
    inv = torch.rand(BH, Lp, generator=gen) * 0.5 + 0.01
    dpd = torch.zeros(BH, Lp, Lp)
    dpd[:, :L, :L] = torch.randn(BH, L, L, generator=gen)
    dpd = dpd.to(torch.bfloat16)
    keep = oa.keep_mask(BH, 1, L, drop, oa.SEED, oa.DROP_OFF, oa.SEED_COUNTER).view(BH, L, L) if drop > 0 else \
        torch.ones(BH, L, L, dtype=torch.bool)
    ks32 = np.float32(1) / (np.float32(1) - np.float32(drop)) if drop > 0 else np.float32(1)
    P32 = p[:, :L, :L].float() * inv[:, :L, None]            # the kernel's two fp32 roundings: (p * inv) * (1 / (1 - p))
    pd_want = torch.where(keep, P32 * float(ks32), torch.zeros_like(P32)).to(torch.bfloat16)
    ctr = torch.tensor([oa.SEED_COUNTER], dtype=torch.int64, device="cuda")
    for zero in (True, False):
        ps_d, dpd_d, inv_d = p.cuda(), (torch.zeros_like(dpd) if zero else dpd).cuda(), inv.cuda()
        check(rp.rp_attn_softmax_bwd(ps_d.data_ptr(), dpd_d.data_ptr(), inv_d.data_ptr(), BH, L, scale, drop, oa.SEED,
                                     oa.DROP_OFF, ctr.data_ptr(), _st()), "rp_attn_softmax_bwd")
        torch.cuda.synchronize()
        ps_o, ds_o = ps_d.cpu(), dpd_d.cpu()
        assert torch.equal(ps_o[:, :L, :L].view(torch.int16), pd_want.view(torch.int16))
        assert torch.equal(ps_o[:, L:], p[:, L:]) and torch.equal(ps_o[:, :, L:], p[:, :, L:])   # outside [L, L]: untouched
        Pd = p[:, :L, :L].double() * inv[:, :L, None].double()
        dP = (dpd[:, :L, :L].double() if not zero else torch.zeros_like(Pd)) * keep.double() / (1 - drop)
        ds_ref = Pd * (dP - (Pd * dP).sum(-1, keepdim=True)) * scale
        if zero:
            assert (ds_o[:, :L, :L] == 0).all()
        else:
            assert float((ds_o[:, :L, :L].double() - ds_ref).abs().max()) <= 1e-2 * float(ds_ref.abs().max())
        assert torch.equal(ds_o[:, L:], (torch.zeros_like(dpd) if zero else dpd)[:, L:])


# ------------------------------------------------------------------------------------------------ last-position attention
_LAST = [(64, 64, L) for L in (1, 31, 33, 64, 65, 128, 129, 256, 257, 300, 511, 512)] + \
        [(128, 128, L) for L in (1, 65, 129, 256, 300, 512)] + [(64, 48, 200), (128, 100, 384)]


@pytest.mark.parametrize("slot,hd,L", _LAST)
@pytest.mark.parametrize("mode", ["sasrec", "legacy"])
def test_attn_last_matches_fp64(rp, slot, hd, L, mode, record_property):
    """rp_attn_last (predict: one query per sequence, the last position) == row L - 1 of the reference; an all-pad
    sequence with key padding gives a zero row."""
    from replay_b200._lib import check

    c = dict(L=L, slot=slot, head_dim=hd, mode=mode, H=2 if slot == 64 else 1, B=4, drop=0.0, seed=5 * L + slot)
    inputs = _inputs(c)
    ref = oa.reference_for(c, inputs)
    cs = _Case(c, inputs)
    B, H, dp = cs.B, cs.H, cs.dp
    q_last = cs.Q.view(B, L, dp)[:, -1].contiguous()
    out = torch.full((B, dp), float("nan"), dtype=torch.bfloat16, device="cuda")
    check(rp.rp_attn_last(q_last.data_ptr(), cs.K.data_ptr(), cs.V.data_ptr(), 2 * dp, 2 * dp, 0, dp, cs.pad.data_ptr(), B, H, L,
                          slot, cs.mpk, out.data_ptr(), 1.0 / math.sqrt(hd), _st()), "rp_attn_last")
    torch.cuda.synchronize()
    o = out.float().cpu().view(B, H, slot)
    e = _err(o, ref["O"][:, -1], "O", ref, inputs)
    record_property("err_O", e)
    assert e <= 1.0, f"O error {e:.3f} x tolerance"
    assert (o[..., hd:] == 0).all()
    if cs.mpk:
        assert (o[0] == 0).all()     # sequence 0 is all padding


# ------------------------------------------------------------------------------------------------ invariance
_INV = [dict(L=33, slot=64, head_dim=48, mode="sasrec", H=2, B=4, drop=0.2, seed=11),
        dict(L=200, slot=64, head_dim=64, mode="bert", H=2, B=4, drop=0.2, seed=12),
        dict(L=100, slot=64, head_dim=50, mode="legacy", H=1, B=4, drop=0.0, seed=13),
        dict(L=300, slot=64, head_dim=64, mode="sasrec", H=2, B=4, drop=0.2, seed=14),
        dict(L=129, slot=128, head_dim=100, mode="sasrec", H=1, B=4, drop=0.0, seed=15),
        dict(L=129, slot=128, head_dim=128, mode="bert", H=2, B=4, drop=0.2, seed=16)]


def _run(c, inputs):
    cs = _Case(c, inputs)
    f = cs.fwd(p_save=False)
    out = {"O": f["O"].cpu().view(cs.B, cs.L, cs.H, cs.slot), "m_save": f["m_save"].cpu(), "inv_sum": f["inv_sum"].cpu()}
    if c["slot"] == 64 and c["L"] <= 256:
        out.update(cs.bwd(f))
    return out


def _bits(t):
    return t.view(torch.int16) if t.dtype == torch.bfloat16 else t.view(torch.int32)


@pytest.mark.parametrize("c", _INV, ids=oa.case_id)
def test_attn_outputs_ignore_masked_inputs_bitwise(rp, c):
    """Large finite values (+-1e4) in the rows of masked keys and pad queries and in the padded-slot columns of Q and V, or
    a different neighbouring sequence, leave every unaffected output bit-identical; so does repeating the call."""
    inputs = _inputs(c)
    base = _run(c, inputs)
    again = _run(c, inputs)
    for k in base:
        assert torch.equal(_bits(base[k]), _bits(again[k])), f"{k} not reproducible"
    B, L, H, slot, hd = c["B"], c["L"], c["H"], c["slot"], c["head_dim"]
    causal, mpk = oa.MODES[c["mode"]]
    gen = torch.Generator().manual_seed(99)
    big = lambda *s: ((torch.randint(0, 2, s, generator=gen) * 2 - 1) * 1e4).to(torch.bfloat16)  # noqa: E731
    pad = inputs["pad"]
    # (1) masked keys / pad queries (only masked when key padding is on) and padded-slot columns
    mod = {k: v.clone() for k, v in inputs.items()}
    if mpk:
        for n in ("q", "k", "v"):
            mod[n][~pad] = big(int((~pad).sum()), H, slot)
    if hd < slot:
        mod["q"][..., hd:] = big(B, L, H, slot - hd)
        mod["v"][..., hd:] = big(B, L, H, slot - hd)
    got = _run(c, mod)
    rows = pad if mpk else torch.ones_like(pad)              # pad-query rows are affected when they see real keys
    assert torch.equal(_bits(got["O"][rows][..., :hd]), _bits(base["O"][rows][..., :hd]))
    srows = rows[:, None, :].expand(B, H, L)
    for k in ("m_save", "inv_sum"):
        assert torch.equal(_bits(got[k].view(B, H, -1)[..., :L][srows]), _bits(base[k].view(B, H, -1)[..., :L][srows])), k
    if "dV" in base:
        # dQ of the real queries; dK / dV of the real keys too unless a pad query sees them (BERT4Rec: no causal mask)
        grads = ("dQ", "dK", "dV") if causal else ("dQ",)
        for k in grads:
            assert torch.equal(_bits(got[k][rows][..., :hd]), _bits(base[k][rows][..., :hd])), k
    # (2) a different neighbouring sequence (2): the 128-row tiles of sequence 1 read into its rows
    mod = {k: v.clone() for k, v in inputs.items()}
    for n in ("q", "k", "v", "d_out"):
        mod[n][2, :, :, :hd] = big(L, H, hd)
    got = _run(c, mod)
    keep_b = torch.tensor([b != 2 for b in range(B)])
    for k in base:
        if k in ("m_save", "inv_sum"):
            a, b_ = got[k].view(B, H, -1)[keep_b], base[k].view(B, H, -1)[keep_b]
        else:
            a, b_ = got[k][keep_b], base[k][keep_b]
        assert torch.equal(_bits(a), _bits(b_)), k


# ------------------------------------------------------------------------------------------------ rejections
def test_attn_rejects_unsupported_shapes(rp):
    """Shapes outside the kernels' resident-key / head-dim limits return RP_ESHAPE.  Buffers are allocated for the rejected
    shape, so a missing check computes a wrong answer instead of reading out of bounds."""
    from replay_b200._lib import AttnBwdDesc, AttnDesc

    def fwd_rc(L, hd):
        B, dp = 2, hd
        Q = torch.zeros(B * L, dp, dtype=torch.bfloat16, device="cuda")
        KV = torch.zeros(B * L, 2 * dp, dtype=torch.bfloat16, device="cuda")
        O = torch.zeros(B * L, dp, dtype=torch.bfloat16, device="cuda")
        pad = torch.ones(B * L, dtype=torch.uint8, device="cuda")
        Lp = -(-L // 64) * 64
        st = torch.zeros(B * Lp, device="cuda")
        ad = AttnDesc()
        ad.q, ad.q_rows, ad.q_cols, ad.ldq = Q.data_ptr(), B * L, dp, dp
        ad.k, ad.k_rows, ad.k_cols, ad.ldk = KV.data_ptr(), B * L, 2 * dp, 2 * dp
        ad.v, ad.v_rows, ad.v_cols, ad.ldv, ad.v_c0 = KV.data_ptr(), B * L, 2 * dp, 2 * dp, dp
        ad.B, ad.H, ad.L, ad.head_dim, ad.causal, ad.mask_pad_keys = B, 1, L, hd, 1, 1
        ad.pad_mask, ad.out, ad.ldo, ad.m_save, ad.inv_sum = pad.data_ptr(), O.data_ptr(), dp, st.data_ptr(), st.data_ptr()
        rc = rp.rp_attn_fwd(ctypes.byref(ad), _st())
        bd = AttnBwdDesc()
        dq, dkv = torch.zeros_like(Q), torch.zeros_like(KV)
        bd.q, bd.q_rows, bd.q_cols, bd.ldq = Q.data_ptr(), B * L, dp, dp
        bd.k, bd.k_rows, bd.k_cols, bd.ldk = KV.data_ptr(), B * L, 2 * dp, 2 * dp
        bd.v, bd.v_rows, bd.v_cols, bd.ldv, bd.v_c0 = KV.data_ptr(), B * L, 2 * dp, 2 * dp, dp
        bd.d_out, bd.do_rows, bd.do_cols, bd.ld_do = O.data_ptr(), B * L, dp, dp
        bd.out, bd.ldo = O.data_ptr(), dp
        bd.B, bd.H, bd.L, bd.head_dim, bd.causal, bd.mask_pad_keys = B, 1, L, hd, 1, 1
        bd.pad_mask, bd.m_save, bd.inv_sum = pad.data_ptr(), st.data_ptr(), st.data_ptr()
        bd.dq, bd.ld_dq = dq.data_ptr(), dp
        bd.dk, bd.ld_dk = dkv.data_ptr(), 2 * dp
        bd.dv, bd.ld_dv, bd.dv_c0 = dkv.data_ptr(), 2 * dp, dp
        brc = rp.rp_attn_bwd(ctypes.byref(bd), _st())
        lrc = rp.rp_attn_last(Q.data_ptr(), KV.data_ptr(), KV.data_ptr(), 2 * dp, 2 * dp, 0, dp, pad.data_ptr(), B, 1, L, hd, 1,
                              O.data_ptr(), 0.0, _st())
        torch.cuda.synchronize()
        return rc, brc, lrc

    assert fwd_rc(513, 64) == (RP_ESHAPE, RP_ESHAPE, RP_ESHAPE)
    assert fwd_rc(64, 96) == (RP_ESHAPE, RP_ESHAPE, RP_ESHAPE)
    assert fwd_rc(257, 128)[:2] == (RP_ESHAPE, RP_ESHAPE)
    assert fwd_rc(257, 64)[1] == RP_ESHAPE          # fused backward: L <= 256
    assert fwd_rc(128, 128)[1] == RP_ESHAPE         # fused backward: head_dim 64 only


# ------------------------------------------------------------------------------------------------ engines
_ENG = [("sasrec", 64, 1, 200, 0.1, False), ("sasrec", 64, 1, 200, 0.1, True), ("sasrec", 64, 1, 300, 0.0, False),
        ("sasrec", 128, 1, 200, 0.1, False), ("legacy", 100, 1, 128, 0.0, False), ("sasrec", 192, 4, 256, 0.0, False),
        ("sasrec", 192, 4, 256, 0.0, True), ("sasrec", 64, 2, 128, 0.1, False),
        ("bert", 128, 1, 200, 0.1, False), ("bert", 128, 2, 200, 0.0, False), ("bert", 128, 2, 200, 0.1, True),
        ("bert", 64, 1, 300, 0.0, False)]


@pytest.mark.parametrize("mode,d,H,L,drop,unfused", _ENG)
def test_engine_attention_buffers_match_fp64(rp, mode, d, H, L, drop, unfused, record_property):
    """The engines' own attention forward and backward - the fused kernel or the un-fused softmax backward between the
    batched rp_gemm calls (engine.py / engine_bert.py backward) - at kernel-level tolerance: after backward() of a 1-block
    engine, O, dQ, dK and dV equal the fp64 restatement evaluated on the engine's own Q / K / V and dO.  Nothing writes
    these buffers after block 0's attention backward (only the projections' backward and weight gradients read them)."""
    from replay_b200.synthetic import make_sequences

    B, I = 6, 700
    ids, pm, lab, tm = make_sequences(B, I, L, seed=L + d)
    if mode == "bert":
        from replay_b200.engine_bert import BertConfig, Bert4RecEngine

        cfg = BertConfig(n_items=I, d=d, n_heads=H, n_blocks=1, max_len=L, dropout=drop)
        eng = Bert4RecEngine(cfg, B, L, "cuda", seed=5)
    else:
        from replay_b200.engine import EncoderConfig, SasRecEngine

        cfg = EncoderConfig(n_items=I, d=d, n_heads=H, n_blocks=1, max_len=L, dropout=drop,
                            variant="legacy" if mode == "legacy" else "new")
        eng = SasRecEngine(cfg, B, L, "cuda", seed=5)
    if unfused:
        assert eng.fused_attn_bwd
        eng.fused_attn_bwd = False
        eng._realloc_workspace()
    if mode == "bert":
        gen = torch.Generator().manual_seed(L)
        tok = pm & (torch.rand(B, L, generator=gen) > 0.2)
        ids = torch.where(pm, ids, torch.zeros_like(ids))
        eng.set_batch(ids.cuda(), pm.cuda(), tok.cuda(), ids.cuda())
    else:
        eng.set_batch(ids.cuda(), pm.cuda(), lab.cuda(), tm.cuda())
    eng.tick_rng()
    eng.forward_train()
    eng.g32.zero_()
    eng.backward()
    torch.cuda.synchronize()
    dp, hd = cfg.d if mode == "bert" else cfg.dp, cfg.d // H
    slot = dp // H
    a, s = eng.act[0], eng.s
    view = lambda t: t.float().cpu().view(B, L, H, slot)  # noqa: E731
    if mode == "bert":
        qkv, g = a["QKV"], s["dQKV"]
        q, k, v = view(qkv[:, :dp]), view(qkv[:, dp:2 * dp]), view(qkv[:, 2 * dp:])
        got = {"dQ": view(g[:, :dp]), "dK": view(g[:, dp:2 * dp]), "dV": view(g[:, 2 * dp:])}
        site = eng._bsite(0, 0)
    else:
        q, k, v = view(a["Q"]), view(a["KV"][:, :dp]), view(a["KV"][:, dp:])
        got = {"dQ": view(s["dQ"]), "dK": view(s["dKV"][:, :dp]), "dV": view(s["dKV"][:, dp:])}
        site = eng._site(0, 0)
    got["O"] = view(a["O"])
    causal, mpk = oa.MODES[mode]
    ref = oa.attention(q, k, v, pm, causal=causal, mask_pad_keys=mpk, head_dim=hd, drop_p=drop, seed=eng.seed,
                       seed_counter=int(eng.rng_counter.item()), drop_off=site << 40, d_out=view(s["d_o"]))
    inputs = {"v": v}
    errs = {n: _err(got[n], ref[n], n, ref, inputs) for n in ("O", "dQ", "dK", "dV")}
    for k, v in errs.items():
        record_property("err_" + k, v)
    assert max(errs.values()) <= 1.0, errs
