"""GPU tests at BASELINE.json's full config-2 size (64 ragged bags of 100..20000 x 1024, bf16, ~0.6 M instances):
the oracle cannot run that in seconds, so parity is checked through size-independent properties of the pool plus
an oracle check on sampled bags."""
import numpy as np
import pytest
import torch

from oracle import mil_oracle as mo
from tests.helpers import rel_err

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def big():
    import mil_b200
    g = torch.Generator().manual_seed(1234)
    lens = torch.randint(100, 20001, (64,), generator=g).numpy()
    off = mo.offsets_from_lengths(lens)
    gen = torch.Generator(device="cuda").manual_seed(1)
    X = torch.randn(int(off[-1]), 1024, device="cuda", generator=gen).bfloat16()
    p = mo.procedural_state(mo.abmil_shapes(1024), 1234)
    m = mil_b200.ABMIL(None, L=1024).cuda().eval()
    m.load_state_dict({k: torch.from_numpy(v) for k, v in p.items()})
    return m, p, X, off, lens


def test_fullsize_sampled_bags_match_oracle(big):
    m, p, X, off, lens = big
    offt = torch.from_numpy(off).cuda()
    M = m.forward_csr(X, offt).detach().float().cpu().numpy()
    s = m.last_scores.detach().cpu().numpy()
    am = m.last_argmax.detach().cpu().numpy()
    pq = {k: (torch.from_numpy(v).bfloat16().float().numpy() if k.endswith("0.weight") else v) for k, v in p.items()}
    for b in (0, 17, 63, int(np.argmin(lens)), int(np.argmax(lens))):
        xb = X[off[b]:off[b + 1]].float().cpu().numpy()
        f = mo.abmil_forward(pq, xb)
        assert rel_err(M[b], f["M"][0]) <= 1e-2
        assert rel_err(s[off[b]:off[b + 1]], f["s"]) <= 1e-2
        srt = np.sort(f["s"])
        if srt[-1] - srt[-2] > 1e-3:
            assert int(am[b]) == f["argmax"]


def test_fullsize_properties(big):
    m, p, X, off, lens = big
    from mil_b200 import functional as F
    offt = torch.from_numpy(off).cuda()
    M = m.forward_csr(X, offt).float()
    s = m.last_scores
    # (1) attention weights of every bag sum to one: pooling a constant bag returns the constant
    ones = torch.ones_like(X)
    Mc, _, _, lse = F.segment_softmax_pool(ones, s, offt)
    assert torch.allclose(Mc, torch.ones_like(Mc), atol=1e-5)
    # (2) shift invariance: adding a constant to every score leaves M unchanged, moves lse by the constant
    M1, _, am1, lse1 = F.segment_softmax_pool(X, s, offt)
    M2, _, am2, lse2 = F.segment_softmax_pool(X, s + 3.0, offt)
    assert torch.allclose(M1, M2, rtol=1e-4, atol=1e-5)
    assert torch.allclose(lse2 - lse1, torch.full_like(lse1, 3.0), atol=1e-4)
    assert torch.equal(am1, am2)
    # (3) argmax indexes the largest score of its bag
    sc = s.detach().cpu().numpy()
    for b in (0, 5, 31, 63):
        seg = sc[off[b]:off[b + 1]]
        assert seg[int(am1[b])] == seg.max()
    # (4) batch composition independence: a bag pooled alone equals the bag pooled inside the batch
    for b in (3, 40):
        xb = X[off[b]:off[b + 1]].contiguous()
        Mb = m.forward_csr(xb, torch.tensor([0, xb.shape[0]], dtype=torch.int32, device="cuda")).float()
        assert torch.allclose(Mb[0], M[b], rtol=2e-2, atol=1e-3)
    # (5) linearity of the backward in dM: grads(dM1 + dM2) == grads(dM1) + grads(dM2)
    Mf = M1
    dA, dB = torch.randn_like(Mf), torch.randn_like(Mf)
    dsA, _ = F.segment_softmax_pool_bwd(X, s, offt, dA, Mf, False)
    dsB, _ = F.segment_softmax_pool_bwd(X, s, offt, dB, Mf, False)
    dsAB, _ = F.segment_softmax_pool_bwd(X, s, offt, dA + dB, Mf, False)
    assert rel_err((dsA + dsB).detach().cpu().numpy(), dsAB.detach().cpu().numpy()) <= 1e-4
    # (6) d(scores) sums to zero inside every bag (softmax Jacobian annihilates constants)
    tot = torch.zeros(64, device="cuda", dtype=torch.float64)
    bag = torch.bucketize(torch.arange(X.shape[0], device="cuda"), offt[1:].long(), right=True)
    tot.index_add_(0, bag, dsA.double())
    scale = torch.zeros(64, device="cuda", dtype=torch.float64).index_add_(0, bag, dsA.double().abs())
    assert float((tot.abs() / scale.clamp_min(1e-30)).max()) < 1e-3


def test_fullsize_trainer_step_matches_module_autograd(big):
    """The bench's fused trainer step (flat gradient buffer) produces the same gradients as the nn.Module path."""
    m, p, X, off, lens = big
    from mil_b200.dp import AbmilTrainer
    offt = torch.from_numpy(off).cuda()
    for prm in m.parameters():
        prm.grad = None
    M = m.forward_csr(X, offt)
    M.float().sum().backward()
    tr = AbmilTrainer(1024, 192, torch.bfloat16, device="cuda")
    tr.load_from(m)
    Mt, _ = tr.forward_backward(X, offt)
    gv = tr.grad_views()
    assert rel_err(Mt.detach().cpu().numpy(), M.detach().float().cpu().numpy()) <= 1e-2
    assert rel_err(gv["Wcat"][:192].detach().cpu().numpy(), m.attention_V[0].weight.grad.detach().cpu().numpy()) <= 1e-4
    assert rel_err(gv["Wcat"][192:].detach().cpu().numpy(), m.attention_U[0].weight.grad.detach().cpu().numpy()) <= 1e-4
    assert rel_err(gv["ww"].detach().cpu().numpy(), m.attention_weights.weight.grad.detach().cpu().numpy().reshape(-1)) <= 1e-4


@pytest.mark.parametrize("optimizer", ["adam", "sgd"])
def test_trainer_update_matches_optimizer_oracle(optimizer):
    """Three update steps of the fused optimiser kernels (Adam: train_ddp.py:113-116; SGD: train_ddp.py:105-108)
    over the flat buffer against the float64 restatement (itself pinned to torch.optim in the CPU suite)."""
    from mil_b200.dp import AbmilTrainer
    lr = 1e-5 if optimizer == "adam" else 1e-3
    tr = AbmilTrainer(96, 192, torch.float32, device="cuda", lr=lr, optimizer=optimizer)
    g = torch.Generator().manual_seed(5)
    p0 = torch.randn(tr.numel, generator=g) * 0.05
    tr.params.copy_(p0)
    pn = p0.double().numpy()
    m = np.zeros_like(pn)
    v = np.zeros_like(pn)
    for step in (1, 2, 3):
        grad = torch.randn(tr.numel, generator=g)
        tr.grads.copy_(grad)
        tr.reduce_and_update()
        if optimizer == "adam":
            pn, m, v = mo.adam_step(pn, grad.double().numpy(), m, v, step, lr=lr)
        else:
            pn = mo.sgd_step(pn, grad.double().numpy(), lr=lr)
    got = tr.params.detach().cpu().numpy()
    assert np.abs(got - pn).max() <= 1e-6 * np.abs(pn).max()
    assert rel_err(got - p0.numpy(), pn - p0.double().numpy()) <= 1e-3      # the update itself, not just the parameters


@pytest.mark.parametrize("total_n,L", [(n, 1024) for n in (1, 2, 127, 128, 129, 255, 256, 257, 383, 385, 512, 513, 1025,
                                                            148 * 256 + 1)] +
                         [(2500, 768), (2500, 512), (777, 256), (3001, 320), (40000, 768)])
@pytest.mark.parametrize("recompute_gate", ["0", "1"])
def test_tile_boundaries_of_the_tensor_core_step(total_n, L, recompute_gate):
    """The bench's trainer step (CTA-pair score GEMM with saved V,U, persistent pools, fused dW) at instance counts that
    straddle the 128-row CTA tile, the 256-row pair tile and one full wave of pairs (+1), split into 1-3 ragged bags:
    pooled vectors, scores, argmax and every parameter gradient against the float64 oracle on the same bf16 operands.
    recompute_gate = "1": the trainer saves no gate activations (save_gate=False), so the score GEMM runs without the V,U
    stores and the backward recomputes them (EpiDz)."""
    from mil_b200.dp import AbmilTrainer
    import mil_b200
    p = mo.procedural_state(mo.abmil_shapes(L), 7)
    m = mil_b200.ABMIL(None, L=L).cuda().eval()
    m.load_state_dict({k: torch.from_numpy(v) for k, v in p.items()})
    cuts = sorted({0, total_n // 3, (2 * total_n) // 3 + (1 if total_n > 2 else 0), total_n})
    off = np.asarray(cuts, dtype=np.int32)
    off = off[np.concatenate([[True], np.diff(off) > 0])]          # no empty bags
    g = torch.Generator().manual_seed(total_n)
    X = torch.randn(total_n, L, generator=g).to(torch.bfloat16)
    dM = torch.randn(len(off) - 1, L, generator=g)
    tr = AbmilTrainer(L, 192, torch.bfloat16, device="cuda", save_gate=recompute_gate == "0")
    tr.load_from(m)
    Mt, _ = tr.forward_backward(X.cuda(), torch.from_numpy(off).cuda(), dM.cuda())
    torch.cuda.synchronize()
    pq = {k: (torch.from_numpy(v).to(torch.bfloat16).float().numpy() if k.endswith("0.weight") else v) for k, v in p.items()}
    Xq = X.float().numpy()
    Mr, sr, amr = mo.abmil_forward_csr(pq, Xq, off)
    gr = mo.abmil_backward_csr(pq, Xq, off, dM.numpy())
    assert rel_err(Mt.detach().cpu().numpy(), Mr) <= 1e-2
    assert rel_err(tr.last_scores.detach().cpu().numpy(), sr) <= 1e-2
    if mo.score_margin(sr, off) > 1e-3:
        assert tr.last_argmax.detach().cpu().numpy().tolist() == amr.tolist()
    gv = tr.grad_views()
    got = {"attention_V.0.weight": gv["Wcat"][:192], "attention_U.0.weight": gv["Wcat"][192:],
           "attention_V.0.bias": gv["bcat"][:192], "attention_U.0.bias": gv["bcat"][192:], "attention_weights.weight": gv["ww"]}
    scale = max(float(np.abs(gr[k]).max()) for k in got)
    for k, v in got.items():
        a, b = v.detach().cpu().numpy().reshape(-1), np.asarray(gr[k]).reshape(-1)
        if total_n <= 2:
            # one-instance bags: softmax weight exactly 1, every attention gradient exactly 0 in exact arithmetic; the
            # kernels leave float noise from g_i - dM.M (same bound as tests/test_gpu_abmil.py uses for N = 1)
            assert float(np.abs(a - b).max()) <= 1e-5, k
        elif float(np.abs(b).max()) < 1e-6 * max(scale, 1e-30):
            assert float(np.abs(a - b).max()) <= 1e-2 * max(scale, 1e-6), k      # (near-)zero true gradient
        else:
            assert rel_err(a, b) <= 1e-2, k


@pytest.mark.parametrize("recompute_gate", ["0", "1"])
@pytest.mark.parametrize("case", ["many_tiny_bags", "one_huge_bag", "huge_then_tiny"])
def test_extreme_bag_shapes(case, recompute_gate):
    """Edge cases of the CSR machinery: 3000 bags of 1-3 instances (every CTA slab holds hundreds of bag pieces),
    one bag spread over every CTA of the persistent pools, and a huge bag followed by tiny ones.  recompute_gate = "1":
    the trainer saves no gate activations and the backward recomputes them."""
    from mil_b200.dp import AbmilTrainer
    import mil_b200
    L = 512
    rng = np.random.default_rng(11)
    if case == "many_tiny_bags":
        lens = rng.integers(1, 4, size=3000)
    elif case == "one_huge_bag":
        lens = np.asarray([80_001])
    else:
        lens = np.concatenate([[50_000], rng.integers(1, 5, size=500)])
    off = mo.offsets_from_lengths(lens)
    n = int(off[-1])
    p = mo.procedural_state(mo.abmil_shapes(L), 3)
    m = mil_b200.ABMIL(None, L=L).cuda().eval()
    m.load_state_dict({k: torch.from_numpy(v) for k, v in p.items()})
    g = torch.Generator().manual_seed(99)
    X = torch.randn(n, L, generator=g).to(torch.bfloat16)
    dM = torch.randn(len(lens), L, generator=g)
    tr = AbmilTrainer(L, 192, torch.bfloat16, device="cuda", save_gate=recompute_gate == "0")
    tr.load_from(m)
    Mt, _ = tr.forward_backward(X.cuda(), torch.from_numpy(off).cuda(), dM.cuda())
    torch.cuda.synchronize()
    pq = {k: (torch.from_numpy(v).to(torch.bfloat16).float().numpy() if k.endswith("0.weight") else v) for k, v in p.items()}
    Xq = X.float().numpy()
    Mr, sr, amr = mo.abmil_forward_csr(pq, Xq, off)
    gr = mo.abmil_backward_csr(pq, Xq, off, dM.numpy())
    assert rel_err(Mt.detach().cpu().numpy(), Mr) <= 1e-2
    assert rel_err(tr.last_scores.detach().cpu().numpy(), sr) <= 1e-2
    am = tr.last_argmax.detach().cpu().numpy()
    assert am.shape == amr.shape and np.all((am >= 0) & (am < lens))          # index within the bag
    for b in np.nonzero(am != amr)[0]:       # bf16 near-ties may pick another instance: its score must be the maximum too
        seg = sr[off[b]:off[b + 1]]
        assert seg[am[b]] >= seg.max() - 1e-2 * max(1.0, abs(seg.max())), b
    gv = tr.grad_views()
    got = {"attention_V.0.weight": gv["Wcat"][:192], "attention_U.0.weight": gv["Wcat"][192:],
           "attention_V.0.bias": gv["bcat"][:192], "attention_U.0.bias": gv["bcat"][192:], "attention_weights.weight": gv["ww"]}
    for k, v in got.items():
        assert rel_err(v.detach().cpu().numpy().reshape(-1), np.asarray(gr[k]).reshape(-1)) <= 1e-2, k


def test_trainer_train_mode_dropout_matches_the_module_on_the_same_mask():
    """AbmilTrainer(dropout_p=0.5) = ABMIL.forward in train mode (ABMIL.py:49): with the generator seeded identically both
    draw the same Philox seed, hence the same mask, and must produce the same pooled vectors and weight gradients."""
    import mil_b200
    from mil_b200.dp import AbmilTrainer
    L = 512
    torch.manual_seed(3)
    m = mil_b200.ABMIL(None, L=L).cuda().train()
    lens = np.asarray([700, 33, 1500, 260])
    off = torch.from_numpy(mo.offsets_from_lengths(lens)).cuda()
    X = torch.randn(int(lens.sum()), L, device="cuda").to(torch.bfloat16)
    dM = torch.randn(len(lens), L, device="cuda")
    torch.manual_seed(77)
    M_mod = m.forward_csr(X, off)
    (M_mod.float() * dM).sum().backward()
    tr = AbmilTrainer(L, 192, torch.bfloat16, device="cuda", dropout_p=m.dropout1.p)
    tr.load_from(m)
    torch.manual_seed(77)
    M_tr, _ = tr.forward_backward(X, off, dM)
    assert rel_err(M_tr.detach().cpu().numpy(), M_mod.detach().float().cpu().numpy()) <= 1e-2
    gv = tr.grad_views()
    assert rel_err(gv["Wcat"][:192].detach().cpu().numpy(), m.attention_V[0].weight.grad.detach().cpu().numpy()) <= 1e-2
    # and it is dropout: about half of the instances' features are zeroed, the rest doubled
    tr0 = AbmilTrainer(L, 192, torch.bfloat16, device="cuda")
    tr0.load_from(m)
    M0, _ = tr0.forward_backward(X, off, dM)
    assert rel_err(M_tr.detach().cpu().numpy(), M0.detach().cpu().numpy()) > 0.05
