"""Round-2 parity additions (run with -m gpu on a B200): the gaps the round-1 review named.

  * cfg 4 (BASELINE configs[3]): EVERY gradient of `aggregator_wMask.forward_padded` + survival head + BCE against the
    float64 oracle (reference: model/aggregator_wMask.py:67-70,114 over model/dim1/ABMIL.py:47-64 on each unpadded bag),
    fp32 (<= 1e-5) and bf16 (<= 1e-2);
  * cfg 2 at full bag sizes: weight gradients of an 8-bag subset of the 100..20 000 draw against the float64 oracle;
  * the argmax tie rule (first index, as torch.argmax / the reference's softmax-argmax give for equal scores), pinned on
    EXACT ties (duplicated instances) across CTA tiles and bag pieces;
  * train-mode trainer: dL/dX passes through the dropout's own backward (same Philox mask).
"""
import numpy as np
import pytest
import torch
from argparse import Namespace

from oracle import fusion_oracle as fo
from oracle import mil_oracle as mo
from tests.helpers import rel_err, rnd
from tests.test_oracle_golden import wmask_shapes

pytestmark = pytest.mark.gpu


# ---------------------------------------------------------------------------------------------------------------
# cfg 4: masked/padded CT-slice bags + survival head + BCE: all gradients vs the oracle
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype,tol", [(torch.float32, 1e-5), (torch.bfloat16, 1e-2)])
def test_cfg4_padded_bags_head_bce_all_gradients_vs_oracle(dtype, tol):
    import mil_b200
    args = Namespace(modality=["CT", "pathology"], model_CT="resnetMC3_18_wMask", model_pathology="ABMIL", num_classes=2,
                     clinical_features=list("abcdefghi"))
    m = mil_b200.get_model(args).cuda().eval()
    sdn = mo.procedural_state(wmask_shapes(), 81)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in sdn.items()})
    B, Nmax, L = 32, 160, 768                                    # SURVEY 8(d) cfg 4: (B=32, 160, 768), len in [40, 160]
    Xpad = rnd(43, B, Nmax, L)
    lens = mo.ragged_lengths(B, 40, 160, 44)
    path_feat = rnd(45, B, 768)
    target_np = (np.arange(B * 2).reshape(B, 2) % 3 == 0).astype(np.float32)
    pool = m.extractor_pathology
    xpad_t = torch.from_numpy(Xpad).cuda().to(dtype).requires_grad_(True)
    pf_t = torch.from_numpy(path_feat).cuda().to(dtype).requires_grad_(True)
    prob = m.forward_padded(pool, xpad_t, torch.from_numpy(lens).cuda(), other_feats=(pf_t,))
    loss = torch.nn.BCELoss()(prob.float(), torch.from_numpy(target_np).cuda())
    loss.backward()
    torch.cuda.synchronize()

    # oracle: the reference pool on each UNPADDED bag, the reference head, BCELoss; float64, on the operands the kernels saw
    quant = (lambda t: t.to(dtype).double()) if dtype != torch.float32 else (lambda t: t.double())
    sd = {}
    for k, v in sdn.items():
        t = torch.from_numpy(v)
        # bf16 mode quantises what the tensor-core kernels consume: the gate weights; the small head stays fp32
        sd[k] = (quant(t) if (t.dim() == 2 and "attention_" in k and k.endswith("0.weight")) else t.double()).requires_grad_(True)
    xd = xpad_t.detach().double().cpu().requires_grad_(True)
    pfd = pf_t.detach().double().cpu().requires_grad_(True)
    pooled = torch.cat([fo.abmil(sd, "extractor_pathology", xd[b, :int(n)]) for b, n in enumerate(lens)], dim=0)
    pr = fo.wmask_head_forward(sd, [pooled, pfd])
    lr = torch.nn.BCELoss()(pr, torch.from_numpy(target_np).double())
    lr.backward()

    assert rel_err(prob.detach().float().cpu().numpy(), pr.detach().numpy()) <= tol
    assert abs(float(loss) - float(lr)) <= tol * max(1.0, abs(float(lr)))
    g = xpad_t.grad.detach().float().cpu().numpy()
    for b_, n_ in enumerate(lens):
        assert float(np.abs(g[b_, int(n_):]).max(initial=0.0)) == 0.0          # padding rows never get gradient
    assert rel_err(g, xd.grad.numpy()) <= tol
    assert rel_err(pf_t.grad.detach().float().cpu().numpy(), pfd.grad.numpy()) <= tol
    checked = 0
    for name, p in m.named_parameters():
        ref = sd[name].grad
        if ref is None or float(ref.abs().max()) == 0.0:
            assert p.grad is None or float(p.grad.abs().max()) == 0.0, name    # parameters off this path
            continue
        if name.endswith("attention_weights.bias"):                            # exactly-zero true gradient (softmax shift)
            assert float(p.grad.abs().max()) <= 1e-6
            continue
        assert p.grad is not None, name
        assert rel_err(p.grad.detach().float().cpu().numpy(), ref.numpy()) <= tol, name
        checked += 1
    assert checked >= 9          # pool: Wv, bv, Wu, bu, ww; head: fc.1.{weight,bias}, fc.4.{weight,bias}


# ---------------------------------------------------------------------------------------------------------------
# cfg 2 at full bag sizes: an 8-bag subset of the 100..20 000 draw, every parameter gradient vs the float64 oracle
# ---------------------------------------------------------------------------------------------------------------
def test_cfg2_fullsize_8bag_subset_gradients_vs_oracle():
    import mil_b200
    from mil_b200.dp import AbmilTrainer
    g = torch.Generator().manual_seed(1234)
    lens_all = torch.randint(100, 20001, (64,), generator=g).numpy()           # the bench's draw (bench.py, cfg 2)
    pick = [int(np.argmin(lens_all)), int(np.argmax(lens_all)), 0, 9, 17, 31, 42, 63]
    lens = lens_all[pick]
    off = mo.offsets_from_lengths(lens)
    n = int(off[-1])
    gen = torch.Generator().manual_seed(7)
    X = torch.randn(n, 1024, generator=gen).to(torch.bfloat16)
    dM = torch.randn(len(lens), 1024, generator=gen)
    p = mo.procedural_state(mo.abmil_shapes(1024), 1234)
    m = mil_b200.ABMIL(None, L=1024).cuda().eval()
    m.load_state_dict({k: torch.from_numpy(v) for k, v in p.items()})
    tr = AbmilTrainer(1024, 192, torch.bfloat16, device="cuda")
    tr.load_from(m)
    Mt, _ = tr.forward_backward(X.cuda(), torch.from_numpy(off).cuda(), dM.cuda())
    torch.cuda.synchronize()
    pq = {k: (torch.from_numpy(v).to(torch.bfloat16).float().numpy() if k.endswith("0.weight") else v) for k, v in p.items()}
    Xq = X.float().numpy()
    Mr, sr, amr = mo.abmil_forward_csr(pq, Xq, off)
    gr = mo.abmil_backward_csr(pq, Xq, off, dM.numpy(), need_dx=False)
    assert rel_err(Mt.detach().cpu().numpy(), Mr) <= 1e-2
    assert rel_err(tr.last_scores.detach().cpu().numpy(), sr) <= 1e-2
    am = tr.last_argmax.detach().cpu().numpy()
    for b in range(len(lens)):                 # bit-exact where the oracle's own top-2 margin exceeds the bf16 score noise
        seg = np.sort(sr[off[b]:off[b + 1]])
        if seg[-1] - seg[-2] > 1e-3:
            assert int(am[b]) == int(amr[b]), b
    gv = tr.grad_views()
    got = {"attention_V.0.weight": gv["Wcat"][:192], "attention_U.0.weight": gv["Wcat"][192:],
           "attention_V.0.bias": gv["bcat"][:192], "attention_U.0.bias": gv["bcat"][192:], "attention_weights.weight": gv["ww"]}
    for k, v in got.items():
        assert rel_err(v.detach().cpu().numpy().reshape(-1), np.asarray(gr[k]).reshape(-1)) <= 1e-2, k


# ---------------------------------------------------------------------------------------------------------------
# argmax tie rule on EXACT ties
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("recompute_gate", ["0", "1"])
def test_argmax_exact_ties_pick_the_first_index(dtype, recompute_gate, monkeypatch):
    """Duplicated instances have bit-identical scores.  torch.argmax (what the reference's users apply to the attention
    row, and what the float64 oracle restates) returns the FIRST maximal index; the pooling kernel must do the same no
    matter which warp, CTA slab or bag piece holds the copies.  recompute_gate = "1": the forward keeps no gate
    activations (the other instantiation of the score kernel)."""
    monkeypatch.setenv("MILB200_RECOMPUTE_GATE", recompute_gate)
    import mil_b200
    L = 1024 if dtype == torch.bfloat16 else 512
    p = mo.procedural_state(mo.abmil_shapes(L), 5)
    m = mil_b200.ABMIL(None, L=L).cuda().eval()
    m.load_state_dict({k: torch.from_numpy(v) for k, v in p.items()})
    lens = np.asarray([700, 3, 40_000, 129, 5000])
    off = mo.offsets_from_lengths(lens)
    g = torch.Generator().manual_seed(21)
    X = torch.randn(int(off[-1]), L, generator=g).to(dtype).cuda()
    offt = torch.from_numpy(off).cuda()
    m.forward_csr(X, offt)
    am0 = m.last_argmax.cpu().numpy()
    # plant copies of every bag's winning instance: before it, after it, and far away (other tiles / slabs / pieces)
    expect = []
    for b, n in enumerate(lens):
        w = int(am0[b])
        spots = sorted({max(0, w - 1), min(int(n) - 1, w + 1), int(n) // 7, int(n) - 1, (int(n) * 5) // 6} - {w})
        for s_ in spots:
            X[off[b] + s_] = X[off[b] + w]
        expect.append(min(spots + [w]))
    m.forward_csr(X, offt)
    s = m.last_scores.cpu().numpy()
    am = m.last_argmax.cpu().numpy()
    for b, n in enumerate(lens):
        seg = s[off[b]:off[b + 1]]
        ties = np.nonzero(seg == seg.max())[0]
        assert len(ties) >= 2 or n < 3, (b, ties)                   # the copies really tie bit-for-bit
        assert int(am[b]) == int(ties[0]) == int(np.argmax(seg)), (b, am[b], ties[:4])
        assert int(am[b]) == expect[b]


# ---------------------------------------------------------------------------------------------------------------
# AbmilTrainer in train mode: dX goes through the dropout backward
# ---------------------------------------------------------------------------------------------------------------
def test_trainer_train_mode_input_gradient_matches_module_autograd():
    import mil_b200
    from mil_b200.dp import AbmilTrainer
    L = 512
    torch.manual_seed(3)
    m = mil_b200.ABMIL(None, L=L).cuda().train()
    lens = np.asarray([300, 17, 900])
    off = torch.from_numpy(mo.offsets_from_lengths(lens)).cuda()
    X = torch.randn(int(lens.sum()), L, device="cuda").to(torch.bfloat16).requires_grad_(True)
    dM = torch.randn(len(lens), L, device="cuda")
    torch.manual_seed(77)
    M_mod = m.forward_csr(X, off)
    (M_mod.float() * dM).sum().backward()
    tr = AbmilTrainer(L, 192, torch.bfloat16, device="cuda", dropout_p=m.dropout1.p, need_input_grad=True)
    tr.load_from(m)
    torch.manual_seed(77)
    M_tr, dX = tr.forward_backward(X.detach(), off, dM)
    ref = X.grad.detach().float()
    got = dX.detach().float()
    assert torch.equal(got == 0, ref == 0)                         # the same elements were dropped
    assert float((got == 0).float().mean()) > 0.4                  # ... and about half of them are (p = 0.5)
    assert rel_err(got.cpu().numpy(), ref.cpu().numpy()) <= 1e-2


def test_graphed_trainer_step_equals_eager_steps():
    """AbmilTrainer.step_graphed (the whole step as one replayed CUDA graph, Adam step number in device memory) against
    the eager step on the same data: same pooled vectors, same parameters after 6 optimiser steps."""
    import mil_b200
    from mil_b200.dp import AbmilTrainer
    L = 1024
    torch.manual_seed(5)
    m = mil_b200.ABMIL(None, L=L).cuda()
    lens = np.asarray([900, 40, 2100, 333, 1500])
    off = torch.from_numpy(mo.offsets_from_lengths(lens)).cuda()
    X = torch.randn(int(lens.sum()), L, device="cuda").to(torch.bfloat16)
    a = AbmilTrainer(L, 192, torch.bfloat16, device="cuda", lr=1e-3)
    b = AbmilTrainer(L, 192, torch.bfloat16, device="cuda", lr=1e-3)
    a.load_from(m)
    b.load_from(m)
    p0 = a.params.clone()
    for _ in range(6):
        Ma = a.step(X, off).clone()
        Mb = b.step_graphed(X, off).clone()
    torch.cuda.synchronize()
    assert a.step_count == b.step_count == 6 and int(b._step_dev.item()) == 6
    assert rel_err(Mb.cpu().numpy(), Ma.cpu().numpy()) <= 1e-5
    # Adam normalises each element's update to ~lr: compare the updates, elementwise, where the gradient is not noise
    live = a.grads.abs() > 1e-4 * a.grads.abs().max()
    ua, ub = (a.params - p0)[live], (b.params - p0)[live]
    assert float((ua - ub).abs().max()) <= 1e-3 * float(ua.abs().max())
    assert torch.equal(a.last_argmax, b.last_argmax)
