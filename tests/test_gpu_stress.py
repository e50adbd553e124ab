"""Randomised stress of the persistent tensor-core / pooling kernels (their mbarrier pipelines, tile tails and slab
splits depend on the instance count, the bag layout and L): many random packed batches through the trainer step, each
checked three ways — (1) bitwise repeatability (the reductions are fixed-order, so a second run must give the same
bits: a race or a stale pipeline stage shows up here), (2) pooled vectors and scores against plain fp32 torch ops on the
same bf16 operands (<= 1e-2), (3) the weight gradient against torch autograd of that reference (<= 1e-2)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _torch_reference(X, off, Wv, Wu, bv, bu, ww, bw, dM):
    Wv = Wv.clone().requires_grad_(True)
    Wu = Wu.clone().requires_grad_(True)
    Xf = X.float()
    s = (torch.tanh(Xf @ Wv.t() + bv) * torch.sigmoid(Xf @ Wu.t() + bu)) @ ww + bw
    Ms = []
    for b in range(len(off) - 1):
        a = torch.softmax(s[off[b]:off[b + 1]], 0)
        Ms.append(a @ Xf[off[b]:off[b + 1]])
    M = torch.stack(Ms)
    (M * dM).sum().backward()
    return M.detach(), s.detach(), Wv.grad, Wu.grad


@pytest.mark.parametrize("recompute_gate", ["0", "1"])
@pytest.mark.parametrize("seed", list(range(24)))
def test_random_batches_are_repeatable_and_correct(seed, recompute_gate):
    # recompute_gate = "1": no saved gate activations (save_gate=False): score GEMM without the V,U stores, and the
    # backward recomputes V,U (EpiDz) before the dW GEMM
    import mil_b200
    from mil_b200.dp import AbmilTrainer
    rng = np.random.default_rng(1000 + seed)
    L = int(rng.choice([256, 512, 768, 1024]))
    B = int(rng.integers(1, 40))
    hi = int(rng.choice([8, 300, 3000, 12000]))
    lens = rng.integers(1, hi + 1, size=B)
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    n = int(off[-1])
    g = torch.Generator(device="cuda").manual_seed(seed)
    X = torch.randn(n, L, device="cuda", generator=g).to(torch.bfloat16)
    dM = torch.randn(B, L, device="cuda", generator=g)
    torch.manual_seed(seed)
    m = mil_b200.ABMIL(None, L=L).cuda()
    offt = torch.from_numpy(off).cuda()
    outs = []
    for rep in range(2):
        tr = AbmilTrainer(L, 192, torch.bfloat16, device="cuda", save_gate=recompute_gate == "0")
        tr.load_from(m)
        M, _ = tr.forward_backward(X, offt, dM)
        torch.cuda.synchronize()
        outs.append((M.clone(), tr.last_scores.clone(), tr.grads.clone()))
    for a, b in zip(outs[0], outs[1]):
        assert torch.equal(a, b)                                           # (1) same bits
    assert bool(torch.isfinite(outs[0][0]).all()) and bool(torch.isfinite(outs[0][2]).all())
    q = lambda w: w.detach().to(torch.bfloat16).float()                    # the operands the kernels see
    Mr, sr, gWv, gWu = _torch_reference(X, off, q(m.attention_V[0].weight), q(m.attention_U[0].weight),
                                        m.attention_V[0].bias.detach(), m.attention_U[0].bias.detach(),
                                        m.attention_weights.weight.detach().reshape(-1), m.attention_weights.bias.detach(), dM)
    rel = lambda a, b: float((a - b).norm() / b.norm().clamp_min(1e-30))
    assert rel(outs[0][0], Mr) <= 1e-2                                     # (2)
    assert rel(outs[0][1], sr) <= 1e-2
    gv = tr.grad_views()
    if float(gWv.norm()) > 1e-12:                                          # (3) (all-singleton batches have zero gradient)
        assert rel(gv["Wcat"][:192], gWv) <= 1e-2
        assert rel(gv["Wcat"][192:], gWu) <= 1e-2
    else:
        assert float(gv["Wcat"].abs().max()) <= 1e-5
