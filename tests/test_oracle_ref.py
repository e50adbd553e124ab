"""The reference's own ABMIL (model/dim1/ABMIL.py, run unmodified in float64 by tests/golden/make_golden.py, outputs stored
in tests/golden/abmil_L96_N37.npz) against the oracle's restatements, forward and backward."""
import numpy as np
import torch

from oracle import fusion_oracle as fo
from oracle import mil_oracle as mo
from tests.helpers import load_golden, rnd


def test_reference_abmil_module_equals_both_oracles():
    fx = load_golden("abmil_L96_N37")
    L, N, seed = int(fx["L"]), int(fx["N"]), int(fx["seed"])
    p = mo.procedural_state(mo.abmil_shapes(L), seed)
    x = rnd(seed + 100, 1, N, L)
    dM = torch.from_numpy(rnd(seed + 200, 1, L)).double()
    f = mo.abmil_forward(p, x[0])
    assert np.abs(fx["M"] - f["M"]).max() <= 1e-5 * np.abs(f["M"]).max()
    sd = {"a." + k: torch.from_numpy(v).double().requires_grad_(True) for k, v in p.items()}
    xd = torch.from_numpy(x).double().requires_grad_(True)
    Mo = fo.abmil(sd, "a", xd)
    (Mo * dM).sum().backward()
    Mo = Mo.detach()
    assert float((torch.from_numpy(fx["M"]) - Mo).abs().max()) <= 1e-5 * float(Mo.abs().max())
    assert float((torch.from_numpy(fx["dx"]) - xd.grad[0]).abs().max()) <= 1e-5 * float(xd.grad.abs().max())
    for k in p:
        if k == "attention_weights.bias":
            continue
        g = sd["a." + k].grad
        assert float((torch.from_numpy(fx["g:" + k]) - g).abs().max()) <= 2e-5 * float(g.abs().max()), k
