"""The fp64 attention restatement (oracle/attention.py) is sharp enough to hold the kernels to: on the inputs of every case
tests/test_gpu_attention.py runs, each injected kernel bug moves O - and, for the backward cases, dQ / dK / dV - by more
than four times the tolerance the GPU test allows.  Also pins the numpy restatement of the dropout hash."""
import numpy as np
import pytest
import torch

from oracle import attention as oa

MARGIN = 4.0


def _excess(ref: dict, mut: dict, inputs: dict, with_grad: bool) -> dict:
    """How many tolerances each quantity moved by under the mutation."""
    names = ("O", "dQ", "dK", "dV") if with_grad else ("O",)
    return {k: float((mut[k] - ref[k]).abs().max()) / (oa.TOL[k] * oa.tol_scale(k, ref, inputs)) for k in names}


@pytest.mark.parametrize("c", oa.fwd_cases(), ids=oa.case_id)
def test_forward_mutations_exceed_tolerance(c):
    inputs = oa.make_inputs(c["B"], c["H"], c["L"], c["slot"], c["head_dim"], c["mode"], c["seed"])
    ref = oa.reference_for(c, inputs)
    weak = {}
    for m in oa.mutations_for(c):
        x = _excess(ref, oa.reference_for(c, inputs, mutate=m), inputs, False)
        if x["O"] <= MARGIN:
            weak[m] = round(x["O"], 2)
    assert not weak, f"mutations within {MARGIN}x the O tolerance: {weak}"


@pytest.mark.parametrize("c", oa.bwd_cases(), ids=oa.case_id)
def test_backward_mutations_exceed_tolerance(c):
    inputs = oa.make_inputs(c["B"], c["H"], c["L"], c["slot"], c["head_dim"], c["mode"], c["seed"])
    ref = oa.reference_for(c, inputs, with_grad=True)
    weak = {}
    for m in oa.mutations_for(c):
        x = _excess(ref, oa.reference_for(c, inputs, with_grad=True, mutate=m), inputs, True)
        # O must move in every case; of the gradients, at least the one the bug reaches
        if x["O"] <= MARGIN or max(x["dQ"], x["dK"], x["dV"]) <= MARGIN:
            weak[m] = {k: round(v, 2) for k, v in x.items()}
    assert not weak, f"mutations within {MARGIN}x the tolerance: {weak}"


def test_reference_matches_autograd_softmax():
    """Closed-form backward == autograd through a plain masked softmax (no dropout, a fully masked row included)."""
    c = dict(L=70, slot=64, head_dim=48, mode="sasrec", H=2, B=4, drop=0.0, seed=3)
    inputs = oa.make_inputs(c["B"], c["H"], c["L"], c["slot"], c["head_dim"], c["mode"], c["seed"])
    ref = oa.reference_for(c, inputs, with_grad=True)
    q, k, v = (inputs[n].double().permute(0, 2, 1, 3).requires_grad_() for n in ("q", "k", "v"))
    s = q @ k.transpose(-1, -2) / np.sqrt(48)
    vis = ref["vis"]
    p = torch.softmax(s.masked_fill(~vis, -torch.inf), -1).nan_to_num(0.0)
    o = p @ v
    o.backward(inputs["d_out"].double().permute(0, 2, 1, 3))
    torch.testing.assert_close(o.detach().permute(0, 2, 1, 3), ref["O"], rtol=1e-12, atol=1e-12)
    for name, t in (("dQ", q), ("dK", k), ("dV", v)):
        torch.testing.assert_close(t.grad.permute(0, 2, 1, 3), ref[name], rtol=1e-10, atol=1e-10)
    assert (ref["O"][0] == 0).all()      # sequence 0 is all padding: no visible key in any row
    assert (ref["inv_sum"][0] == 0).all() and (ref["m_save"][0] == 0).all()


def test_dropout_hash_restatement():
    """The vectorised uint32 hash agrees with a Python-integer restatement of rp_philox.cuh, and has the statistics the
    header promises."""
    assert oa._fmix32_int(0) == 0 and int(oa._fmix32(np.array([0]))[0]) == 0
    assert int(oa._fmix32(np.array([1]))[0]) == oa._fmix32_int(1) == 0x514E28B7
    rk = oa.drop_row_key(7, 5 << 40, np.arange(4096))
    ck = oa.drop_col_key(np.arange(256))
    keep = oa.drop_mix(rk[:, None], ck[None, :]) >= np.uint32(oa.drop_threshold(0.2))
    assert abs(keep.mean() - 0.8) < 3e-3
    assert oa.drop_threshold(0.2) == int(np.float64(np.float32(0.2)) * 2 ** 32)
    # the row key depends on every input: seed, site offset and row
    a = oa.drop_row_key(7, 5 << 40, np.array([3]))
    assert a != oa.drop_row_key(8, 5 << 40, np.array([3])) and a != oa.drop_row_key(7, 6 << 40, np.array([3]))
    assert a != oa.drop_row_key(7, 5 << 40, np.array([3 + (1 << 32)]))
