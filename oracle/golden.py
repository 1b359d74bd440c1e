"""Storage format of tests/golden/*.npz (written by oracle/gen_golden.py, read by the tests through ``load``).

Each golden file stays under 1 MB.  The larger cases use two compact forms:

- weights ``sd::<key>`` as int8 with a power-of-two scale ``sdscale::<key>``.  The generator snaps the reference module's
  initial weights to that grid (``snap_to_int8_grid``) before running it, so the decoded fp32 weights are exactly the
  ones the reference computed with;
- gradients ``grad::<key>`` as a fixed, seeded sample of at most ``n`` elements, NaN elsewhere (``sample``).  Compare
  them where they are not NaN.
"""
from __future__ import annotations

import math

import numpy as np
import torch


def _grid_scale(absmax: float) -> float:
    """Smallest power of two that maps ``absmax`` into [-127, 127]."""
    return 2.0 ** math.ceil(math.log2(absmax / 127)) if absmax > 0 else 1.0


def snap_to_int8_grid(module: torch.nn.Module) -> None:
    """Round every floating weight of ``module`` in place to q * scale, |q| <= 127, one power-of-two scale per tensor."""
    with torch.no_grad():
        for v in module.state_dict().values():
            if v.is_floating_point():
                s = _grid_scale(float(v.abs().max()))
                v.copy_(torch.round(v / s) * s)


def state_dict_arrays(module: torch.nn.Module, int8: bool = False) -> dict:
    """``sd::<key>`` arrays of the module's state_dict; with ``int8`` the weights (already snapped) as int8 + scale."""
    out = {}
    for k, v in module.state_dict().items():
        v = v.detach().cpu().numpy().copy()
        if int8 and v.dtype == np.float32:
            s = np.float32(_grid_scale(float(np.abs(v).max())))
            q = np.rint(v / s)
            assert np.abs(q).max() <= 127 and np.array_equal(q * s, v), f"{k} is not on the int8 grid"
            out["sd::" + k], out["sdscale::" + k] = q.astype(np.int8), s
        else:
            out["sd::" + k] = v
    return out


def sample(x: np.ndarray, n: int, seed: int = 0) -> np.ndarray:
    """``x`` itself if it has at most ``n`` elements, else a copy holding ``n`` seeded positions of it and NaN elsewhere."""
    if x.size <= n:
        return x
    keep = np.random.RandomState(seed).choice(x.size, n, replace=False)
    out = np.full(x.size, np.nan, dtype=x.dtype)
    out[keep] = x.reshape(-1)[keep]
    return out.reshape(x.shape)


def load(path: str) -> dict:
    """The arrays of a golden file by key, int8 weights decoded to the fp32 values the reference ran with."""
    z = np.load(path)
    out = {}
    for k in z.files:
        if k.startswith("sdscale::"):
            continue
        v = z[k]
        if k.startswith("sd::") and v.dtype == np.int8:
            v = v.astype(np.float32) * z["sdscale::" + k[4:]]
        out[k] = v
    return out
