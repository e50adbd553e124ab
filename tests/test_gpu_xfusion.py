"""GPU parity tests of the collapsed cross-modal fusion path (csrc/xfusion.cu; run with -m gpu on a B200).

The CT+pathology branch of `aggregator.forward` (model/aggregator.py:134-203 over model/sam/transformer.py:58-120,278-309)
with ONE clinical-text token runs as a segmented program whose image side never projects the image tokens (the key / value
projections are folded into the token side — exact algebra, see csrc/xfusion.cu).  Checked here against the float64
oracle (oracle/fusion_oracle.py, pinned to the reference's fixtures by the CPU suite):

  * fp32: outputs, input gradients and EVERY parameter gradient <= 1e-5 (max-norm relative), with the two documented
    classes of exception (exactly-zero gradients; softmax-Jacobian cancellation gradients, 2e-4);
  * bf16 (bf16 storage of the bags / key stream, bf16 tensor-core GEMMs for fc_pathology and the gated pool, fp32 token
    side): outputs, input gradients and EVERY parameter gradient <= 1e-2 — the north-star bound, max-norm relative, no
    Frobenius relaxation, MLP and q/k projections included;
  * B patients in one launch set == B single calls; collapsed program == projected-keys program (round-1 path).
"""
from argparse import Namespace

import numpy as np
import pytest
import torch

from oracle import fusion_oracle as fo
from oracle import mil_oracle as mo
from tests.test_oracle_golden import aggregator_shapes

pytestmark = pytest.mark.gpu

ARGS = Namespace(modality=["CT", "pathology"], model_CT="resnetMC3_18", model_pathology="ABMIL", model_CI="none",
                 aggregator="ABMIL", num_classes=2, alignment_base="none", clinical_features=list("abcdefghi"))
# weights the bf16 program consumes in bf16 (tensor-core operands); everything else stays fp32 in both modes
BF16_WEIGHTS = ("fc_pathology.0.weight", "aggregator.attention_V.0.weight", "aggregator.attention_U.0.weight")


def _rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def _model(seed=7):
    import mil_b200
    m = mil_b200.get_model(ARGS).cuda().eval()
    sdn = mo.procedural_state(aggregator_shapes(), seed)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in sdn.items()})
    return m, sdn


def _oracle_sd(sdn, dtype):
    sd = {}
    for k, v in sdn.items():
        t = torch.from_numpy(v)
        if dtype == torch.bfloat16 and k in BF16_WEIGHTS:
            t = t.to(dtype)
        sd[k] = t.double().requires_grad_(True)
    return sd


def _inputs(dtype, Np, Nc=160, seed=0, text_scale=0.05):
    g = torch.Generator(device="cuda").manual_seed(1000 + Np + seed)
    x_ct = torch.randn(1, 512, Nc, 1, 2, device="cuda", generator=g).to(dtype).requires_grad_(True)
    x_p = torch.randn(1, Np, 768, device="cuda", generator=g).to(dtype).requires_grad_(True)
    x_t = (torch.randn(1, 1, 512, device="cuda", generator=g) * text_scale).to(dtype).requires_grad_(True)
    return x_ct, x_p, x_t


def _loss(prob, a, b, label):
    import mil_b200
    return torch.nn.BCELoss()(prob.float(), label) + mil_b200.clip_loss.cosine_embedding_loss(a.squeeze(0), b.squeeze(0)).float()


def _oracle_run(sdn, dtype, x_ct, x_p, x_t, label):
    sd = _oracle_sd(sdn, dtype)
    xc, xp, xt = (t.detach().double().cpu().requires_grad_(True) for t in (x_ct, x_p, x_t))
    # the position table is fp32 in both modes (built in fp32 upstream too, aggregator.py:100-106)
    prob, a, b = fo.aggregator_fusion_forward(sd, xc, xp, xt, pe_fn=lambda n, E: fo.sinusoid_pe(n, E, torch.float32).double())
    loss = torch.nn.BCELoss()(prob, label.double().cpu()) + (1 - torch.nn.functional.cosine_similarity(a[0], b[0])).mean()
    loss.backward()
    return sd, (prob, a, b, loss), (xc, xp, xt)


@pytest.mark.parametrize("dtype,tol", [(torch.float32, 1e-5), (torch.bfloat16, 1e-2)])
@pytest.mark.parametrize("Np", [70, 1501, 6000])
def test_collapsed_fusion_all_outputs_and_gradients_vs_oracle(dtype, tol, Np):
    m, sdn = _model()
    x_ct, x_p, x_t = _inputs(dtype, Np)
    label = torch.tensor([[0.0, 1.0]], device="cuda")
    prob, a, b = m([x_ct, x_p], x_t)
    assert tuple(prob.shape) == (1, 2) and tuple(a.shape) == (1, 1, 512) and tuple(b.shape) == (1, 1, 512)
    loss = _loss(prob, a, b, label)
    loss.backward()
    torch.cuda.synchronize()
    sd, (rprob, ra, rb, rloss), (xc, xp, xt) = _oracle_run(sdn, dtype, x_ct, x_p, x_t, label)
    assert _rel(prob, rprob) <= tol and _rel(a, ra) <= tol and _rel(b, rb) <= tol
    assert abs(float(loss) - float(rloss)) <= tol * max(1.0, abs(float(rloss)))
    assert _rel(x_p.grad, xp.grad) <= tol and _rel(x_ct.grad, xc.grad) <= tol and _rel(x_t.grad, xt.grad) <= tol
    live = 0
    worst = (0.0, None)
    for name, p in m.named_parameters():
        ref = sd[name].grad
        if ref is None or float(ref.abs().max()) == 0.0:
            assert p.grad is None or float(p.grad.abs().max()) == 0.0, name        # dead modules / exactly-zero gradients
            continue
        assert p.grad is not None, name
        if name.endswith("k_proj.bias") or name.endswith("attention_weights.bias"):
            # true gradient exactly 0 (softmax shift invariance): float noise upstream, 0 or noise here
            assert float(p.grad.abs().max()) <= max(1e-6, 10 * float(ref.abs().max())), name
            continue
        qk = (".q_proj" in name or ".k_proj" in name) and dtype == torch.float32
        e = _rel(p.grad, ref)
        if e > worst[0]:
            worst = (e, name)
        assert e <= (2e-4 if qk else tol), (name, e)
        live += 1
    assert live > 60, live


def test_forward_bags_equals_single_calls():
    m, sdn = _model(seed=9)
    import mil_b200
    lens = [700, 33, 2500]
    Nc = 160
    g = torch.Generator(device="cuda").manual_seed(5)
    ct = torch.randn(3, Nc, 512, device="cuda", generator=g).requires_grad_(True)
    xp = torch.randn(sum(lens), 768, device="cuda", generator=g).requires_grad_(True)
    xt = (torch.randn(3, 1, 512, device="cuda", generator=g) * 0.05).requires_grad_(True)
    w = torch.randn(3, 2, device="cuda", generator=g)
    wa, wb = torch.randn(3, 1, 512, device="cuda", generator=g), torch.randn(3, 1, 512, device="cuda", generator=g)
    prob, a, b = m.forward_bags(ct, xp, lens, xt)
    ((prob * w).sum() + (a * wa).sum() + (b * wb).sum()).backward()
    got = {n: p.grad.clone() for n, p in m.named_parameters() if p.grad is not None}
    gin = (ct.grad.clone(), xp.grad.clone(), xt.grad.clone())
    for p in m.parameters():
        p.grad = None
    ct.grad = xp.grad = xt.grad = None
    off = np.concatenate([[0], np.cumsum(lens)])
    total = 0
    for i in range(3):
        # the module interface takes the CT encoder's feature map (1, 512, c, h, w): one (h, w) = (1, 1) cell per slice
        fmap = ct[i].t().reshape(1, 512, Nc, 1, 1)
        pi, ai, bi = m([fmap, xp[off[i]:off[i + 1]].unsqueeze(0)], xt[i:i + 1])
        assert _rel(prob[i:i + 1], pi) <= 1e-5 and _rel(a[i], ai[0]) <= 1e-5 and _rel(b[i], bi[0]) <= 1e-5
        total = total + (pi * w[i:i + 1]).sum() + (ai[0] * wa[i]).sum() + (bi[0] * wb[i]).sum()
    total.backward()
    assert _rel(gin[0], ct.grad) <= 1e-5 and _rel(gin[1], xp.grad) <= 1e-5 and _rel(gin[2], xt.grad) <= 1e-5
    for n, p in m.named_parameters():
        if p.grad is None or float(p.grad.abs().max()) == 0.0 or n.endswith("k_proj.bias") or n.endswith("attention_weights.bias"):
            continue        # dead / exactly-zero true gradient (float noise)
        assert _rel(got[n], p.grad) <= (2e-4 if (".q_proj" in n or ".k_proj" in n) else 2e-5), n


def test_collapsed_program_equals_projected_keys_program(monkeypatch):
    """MILB200_FUSION_COLLAPSED=0 runs the round-1 program (projected K, V; generic attention kernels): two independent
    implementations of transformer.py:278-309 must agree."""
    m, sdn = _model(seed=11)
    x_ct, x_p, x_t = _inputs(torch.float32, 900, seed=3)
    label = torch.tensor([[1.0, 0.0]], device="cuda")
    out = {}
    for flag in ("1", "0"):
        monkeypatch.setenv("MILB200_FUSION_COLLAPSED", flag)
        for t in (x_ct, x_p, x_t):
            t.grad = None
        for p in m.parameters():
            p.grad = None
        prob, a, b = m([x_ct, x_p], x_t)
        _loss(prob, a, b, label).backward()
        out[flag] = (prob.detach().clone(), a.detach().clone(), b.detach().clone(), x_p.grad.clone(),
                     {n: p.grad.clone() for n, p in m.named_parameters() if p.grad is not None})
    for i in range(4):
        assert _rel(out["1"][i], out["0"][i]) <= 2e-5
    for n, g in out["0"][4].items():
        if float(g.abs().max()) == 0.0 or n.endswith("k_proj.bias") or n.endswith("attention_weights.bias"):
            continue
        assert _rel(out["1"][4][n], g) <= (4e-4 if (".q_proj" in n or ".k_proj" in n) else 2e-5), n


def test_collapsed_launch_count_and_determinism():
    """<= 100 library launches per patient forward+backward at B = 4 (the review's bar), and bit-identical repeats."""
    import mil_b200
    m, sdn = _model(seed=13)
    lens = [1200, 900, 2000, 450]
    g = torch.Generator(device="cuda").manual_seed(8)
    ct = torch.randn(4, 160, 512, device="cuda", generator=g).bfloat16()
    xp = torch.randn(sum(lens), 768, device="cuda", generator=g).bfloat16()
    xt = (torch.randn(4, 1, 512, device="cuda", generator=g) * 0.05).bfloat16()
    outs = []
    for it in range(3):
        for p in m.parameters():
            p.grad = None
        l0 = mil_b200.launch_count()
        prob, a, b = m.forward_bags(ct, xp, lens, xt)
        (prob.sum() + a.float().sum() + b.float().sum()).backward()
        torch.cuda.synchronize()
        n = mil_b200.launch_count() - l0
        outs.append((prob.clone(), m.fc_pathology[0].weight.grad.clone(),
                     m.TwoWayTransformer_Both.layers[1].mlp.lin1.weight.grad.clone()))
    assert n / 4 <= 100, n
    for o in outs[1:]:
        assert all(torch.equal(x, y) for x, y in zip(o, outs[0]))


# ---------------------------------------------------------------------------------------------------------------------
# FusionTrainer on the collapsed program: B patients per step, no autograd graph
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype,tol", [(torch.float32, 1e-5), (torch.bfloat16, 1e-2)])
def test_fusion_trainer_bags_all_gradients_vs_oracle(dtype, tol):
    """forward_backward_bags (B = 3 patients, one launch set) against the float64 oracle run patient by patient:
    loss = mean over patients of BCE + cosine loss (the default reductions over a batch), every parameter gradient."""
    import mil_b200
    m, sdn = _model(seed=17)
    lens, Nc, B = [900, 64, 3100], 160, 3
    g = torch.Generator(device="cuda").manual_seed(12)
    ct = torch.randn(B, Nc, 512, device="cuda", generator=g).to(dtype)
    xp = torch.randn(sum(lens), 768, device="cuda", generator=g).to(dtype)
    xt = (torch.randn(B, 512, device="cuda", generator=g) * 0.05).to(dtype)
    labels = torch.tensor([[0.0, 1.0], [1.0, 0.0], [0.0, 1.0]], device="cuda")
    tr = mil_b200.FusionTrainer(m, n_text_tokens=1, compute_dtype=dtype)
    loss, prob = tr.forward_backward_bags(ct, xp, lens, xt, labels)
    torch.cuda.synchronize()
    sd = _oracle_sd(sdn, dtype)
    off = np.concatenate([[0], np.cumsum(lens)])
    probs, cos = [], []
    for i in range(B):
        fmap = ct[i].double().cpu().t().reshape(1, 512, Nc, 1, 1)
        p_, a_, b_ = fo.aggregator_fusion_forward(sd, fmap, xp[off[i]:off[i + 1]].double().cpu().unsqueeze(0),
                                                  xt[i].double().cpu().reshape(1, 1, 512),
                                                  pe_fn=lambda n, E: fo.sinusoid_pe(n, E, torch.float32).double())
        probs.append(p_)
        cos.append(1 - torch.nn.functional.cosine_similarity(a_[0], b_[0]))
    rprob = torch.cat(probs, dim=0)
    rbce = torch.nn.BCELoss()(rprob, labels.double().cpu())
    rcos = torch.cat(cos).mean()
    (rbce + rcos).backward()
    assert _rel(prob, rprob) <= tol
    assert abs(float(loss[0]) - float(rbce)) <= tol * max(1.0, float(rbce))
    assert abs(float(loss[1]) - float(rcos)) <= tol * max(1.0, float(rcos))
    got = tr.named_grads()
    live = 0
    for name, ref in ((k, v.grad) for k, v in sd.items()):
        if ref is None or float(ref.abs().max()) == 0.0 or name not in got:
            continue
        if name.endswith("k_proj.bias") or name.endswith("attention_weights.bias"):
            assert float(got[name].abs().max()) <= max(1e-6, 10 * float(ref.abs().max())), name
            continue
        qk = (".q_proj" in name or ".k_proj" in name) and dtype == torch.float32
        assert _rel(got[name], ref) <= (2e-4 if qk else tol), name
        live += 1
    assert live > 60, live


def test_fusion_trainer_train_mode_matches_module_train_mode_on_the_same_masks():
    """train_mode=True = the reference's train-mode arithmetic (ABMIL.py:49 Dropout(0.5) on the bag, aggregator.py:128-131
    Dropout(0.25) before the head).  Module and trainer draw their Philox seeds from torch's generator in the same order,
    so with the generator seeded identically they drop the same elements and must agree; and the result differs from
    eval mode."""
    import mil_b200
    from mil_b200 import functional as F
    m, sdn = _model(seed=19)
    x_ct, x_p, x_t = _inputs(torch.float32, 800, seed=4)
    label = torch.tensor([[0.0, 1.0]], device="cuda")
    m.train()
    torch.manual_seed(123)
    prob, a, b = m([x_ct, x_p], x_t)
    _loss(prob, a, b, label).backward()
    ref = {k: v.grad.detach().clone() for k, v in m.named_parameters() if v.grad is not None}
    tr = mil_b200.FusionTrainer(m, n_text_tokens=1, compute_dtype=torch.float32, train_mode=True)
    torch.manual_seed(123)
    loss, p2 = tr.forward_backward(F.ct_tokens(x_ct.detach())[0], x_p.detach()[0], x_t.detach()[0], label[0])
    assert _rel(p2, prob) <= 1e-5
    got = tr.named_grads()
    n = 0
    for k, g in ref.items():
        if float(g.abs().max()) == 0.0 or k.endswith("k_proj.bias") or k.endswith("attention_weights.bias"):
            continue
        assert _rel(got[k], g) <= (4e-4 if (".q_proj" in k or ".k_proj" in k) else 2e-5), k
        n += 1
    assert n > 60
    tr_eval = mil_b200.FusionTrainer(m, n_text_tokens=1, compute_dtype=torch.float32)
    _, p3 = tr_eval.forward_backward(F.ct_tokens(x_ct.detach())[0], x_p.detach()[0], x_t.detach()[0], label[0])
    assert _rel(p3, prob) > 1e-3                      # dropout really changed the result
    m.eval()


@pytest.mark.parametrize("T", [1, 10])
def test_fusion_trainer_pool_head_bce_is_the_labelled_step(T):
    """The pool, head and BCE of a FusionTrainer step (collapsed program with B = 3 patients, projected-keys program with
    T = 10) are the pool trainer's labelled step: the head's row dots come from the pooling pass, so the backward makes no
    pass over the packed bag; its loss and prob equal the two-pass route's (forward, head + BCE, backward(dM)) on the same
    bag bit for bit, and the bag's gradient differs by reassociation only."""
    import mil_b200
    from mil_b200.dp import AbmilTrainer
    from tests.test_gpu_labelled_step import _two_pass
    m, _ = _model(seed=37)
    tr = mil_b200.FusionTrainer(m, n_text_tokens=T, compute_dtype=torch.float32)
    seen, names = {}, []
    step = tr.pool.forward_backward_labels

    def spy(X, offsets, labels, loss=None):
        seen.update(X=X.clone(), offsets=offsets.clone(), labels=labels.clone())
        out = step(X, offsets, labels, loss=loss)
        seen["dX"] = tr.pool.last_dX.clone()          # the program's backward then adds the cosine loss's rows in place
        return out

    tr.pool.forward_backward_labels = spy
    tr.pool.phase_hook = names.append
    g = torch.Generator(device="cuda").manual_seed(14)
    if T == 1:
        lens, B = [900, 64, 3100], 3
        ct = torch.randn(B, 160, 512, device="cuda", generator=g)
        xp = torch.randn(sum(lens), 768, device="cuda", generator=g)
        xt = torch.randn(B, 512, device="cuda", generator=g) * 0.05
        labels = torch.tensor([[0.0, 1.0], [1.0, 0.0], [0.0, 1.0]], device="cuda")
        loss, prob = tr.forward_backward_bags(ct, xp, lens, xt, labels)
    else:
        ct = torch.randn(160, 512, device="cuda", generator=g)
        xp = torch.randn(1203, 768, device="cuda", generator=g)
        xt = torch.randn(T, 512, device="cuda", generator=g) * 0.05
        loss, prob = tr.forward_backward(ct, xp, xt, torch.tensor([1.0, 0.0], device="cuda"))
    torch.cuda.synchronize()
    assert "pool_bwd_headdot" in names and "segment_softmax_pool_bwd" not in names
    assert tuple(loss.shape) == (2,) and float(loss[1]) > 0.0
    ref = AbmilTrainer(512, tr.pool.D, torch.float32, device="cuda", need_input_grad=True, head_classes=2)
    ref.params.copy_(tr.pool.params)
    l2, p2, dX2 = _two_pass(ref, seen["X"], seen["offsets"], seen["labels"])
    torch.cuda.synchronize()
    assert torch.equal(loss[0:1], l2) and torch.equal(prob, p2)
    assert _rel(seen["dX"], dX2) <= 1e-5


@pytest.mark.parametrize("case", ["tiny_bags", "sixteen_segments", "one_huge_bag"])
def test_collapsed_fusion_edge_shapes_vs_oracle(case):
    """Segment machinery at its edges: 2-row bags (fewer rows than warps), 8 patients = 16 segments with lengths that are
    not multiples of the row-item size, and one bag far above the per-item row cap next to a 3-row one; fp32 vs float64."""
    import mil_b200
    m, sdn = _model(seed=23)
    if case == "tiny_bags":
        lens, Nc = [2, 3, 2], 2
    elif case == "sixteen_segments":
        lens, Nc = [37, 1, 513, 64, 7, 1290, 255, 33], 160
        lens = [max(2, n) for n in lens]
    else:
        lens, Nc = [41_003, 3], 5
    B = len(lens)
    g = torch.Generator(device="cuda").manual_seed(len(lens) * 7 + Nc)
    ct = torch.randn(B, Nc, 512, device="cuda", generator=g).requires_grad_(True)
    xp = torch.randn(sum(lens), 768, device="cuda", generator=g).requires_grad_(True)
    xt = (torch.randn(B, 1, 512, device="cuda", generator=g) * 0.05).requires_grad_(True)
    w = torch.randn(B, 2, device="cuda", generator=g)
    wa = torch.randn(B, 1, 512, device="cuda", generator=g)
    prob, a, b = m.forward_bags(ct, xp, lens, xt)
    ((prob * w).sum() + (a * wa).sum() + (b * wa).sum()).backward()
    torch.cuda.synchronize()
    sd = _oracle_sd(sdn, torch.float32)
    off = np.concatenate([[0], np.cumsum(lens)])
    ctd, xpd, xtd = (t.detach().double().cpu().requires_grad_(True) for t in (ct, xp, xt))
    total = 0
    for i in range(B):
        fmap = ctd[i].t().reshape(1, 512, Nc, 1, 1)
        p_, a_, b_ = fo.aggregator_fusion_forward(sd, fmap, xpd[off[i]:off[i + 1]].unsqueeze(0), xtd[i:i + 1],
                                                  pe_fn=lambda n, E: fo.sinusoid_pe(n, E, torch.float32).double())
        assert _rel(prob[i:i + 1], p_) <= 1e-5 and _rel(a[i], a_[0]) <= 1e-5 and _rel(b[i], b_[0]) <= 1e-5, (case, i)
        total = total + (p_ * w[i:i + 1].double().cpu()).sum() + (a_[0] * wa[i].double().cpu()).sum() + (b_[0] * wa[i].double().cpu()).sum()
    total.backward()
    assert _rel(xp.grad, xpd.grad) <= 2e-5 and _rel(ct.grad, ctd.grad) <= 2e-5 and _rel(xt.grad, xtd.grad) <= 2e-5
    n = 0
    for name, p in m.named_parameters():
        ref = sd[name].grad
        if ref is None or float(ref.abs().max()) == 0.0 or name.endswith("k_proj.bias") or name.endswith("attention_weights.bias"):
            continue
        qk = ".q_proj" in name or ".k_proj" in name
        assert _rel(p.grad, ref) <= (4e-4 if qk else 2e-5), (case, name, _rel(p.grad, ref))
        n += 1
    assert n > 60


def test_forward_bags_rejects_bad_arguments():
    import mil_b200
    m, _ = _model(seed=29)
    ct = torch.randn(2, 160, 512, device="cuda")
    xp = torch.randn(100, 768, device="cuda")
    xt = torch.randn(2, 1, 512, device="cuda")
    with pytest.raises(mil_b200.MilB200Error):
        m.forward_bags(ct, xp, [60, 30], xt)              # lengths do not add up to the packed rows
    with pytest.raises(mil_b200.MilB200Error):
        m.forward_bags(ct, xp, [99, 1], xt)               # a 1-row bag (the one-key shortcut needs >= 2 rows)
    with pytest.raises(mil_b200.MilB200Error):
        m.forward_bags(torch.randn(9, 4, 512, device="cuda"), torch.randn(90, 768, device="cuda"), [10] * 9,
                       torch.randn(9, 1, 512, device="cuda"))       # more than 8 patients = 16 segments


def test_fusion_trainer_varying_shapes_share_buffers_and_stay_correct():
    """Real cohorts have a different row count per patient: consecutive steps with different shapes (same capacity bucket,
    then a larger one, then a repeat that replays its CUDA graph) must each equal a fresh trainer's result."""
    import mil_b200
    m, sdn = _model(seed=31)
    tr = mil_b200.FusionTrainer(m, n_text_tokens=1, compute_dtype=torch.float32)
    g = torch.Generator(device="cuda").manual_seed(3)
    shapes = [[700, 90], [650, 301], [5000, 40], [700, 90], [700, 90]]
    for lens in shapes:
        B = len(lens)
        ct = torch.randn(B, 160, 512, device="cuda", generator=g)
        xp = torch.randn(sum(lens), 768, device="cuda", generator=g)
        xt = torch.randn(B, 512, device="cuda", generator=g) * 0.05
        lab = torch.tensor([[0.0, 1.0], [1.0, 0.0]], device="cuda")
        loss, prob = tr.forward_backward_bags(ct, xp, lens, xt, lab)
        got = (loss.clone(), prob.clone(), tr.grads.clone())
        fresh = mil_b200.FusionTrainer(m, n_text_tokens=1, compute_dtype=torch.float32)
        l2, p2 = fresh.forward_backward_bags(ct, xp, lens, xt, lab)
        assert torch.equal(got[0], l2) and torch.equal(got[1], p2), lens
        assert torch.equal(got[2], fresh.grads), lens
    assert len(tr._buf) == 2          # two capacity buckets: (4096 rows) and (8192 rows)
