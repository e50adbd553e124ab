"""Tests of the labelled training step: the gated pool with a linear classifier head and sigmoid + BCE, trained through
AbmilTrainer(head_classes=C).forward_backward_labels / step_labels / step_graphed(X, offsets, labels), and of the pooling
pair it runs on (milb200_segment_softmax_pool_fwd_headdot / _bwd_headdot), whose forward takes the head's C row dots
(W_c * s_b) . x_i so that the backward does not read X again.

The headdot forward must return the plain forward's M, M_lowp, argmax and lse bit for bit, and its row dots and the
backward's score gradients must match float64 at every vector width and dot bucket the kernels are instantiated for.  The
trainer must match the float64 oracle (pool, head, BCE, Adam), the two-pass route (forward + head + backward(dM)) and the
reference model's golden outputs."""
import ctypes as Cty
from argparse import Namespace

import numpy as np
import pytest
import torch

from oracle import mil_oracle as mo
from tests.helpers import load_golden, rel_err, rnd
from tests.test_gpu_pool_rowdot import CASES, _csr, _expect_rejected, _layout
from tests.test_oracle_golden import clip_agg_shapes

D = 192


@pytest.fixture(scope="module")
def F():
    from mil_b200 import functional
    return functional


def _refused(dtype, L, C):
    """Shapes the headdot forward refuses: more than 4 dots on a bf16 row of more than 1536 elements."""
    return dtype == torch.bfloat16 and L > 1536 and C > 4


# ---------------------------------------------------------------------------------------------------------------------
# the kernel pair
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("C", [1, 2, 3, 5, 8])
@pytest.mark.parametrize("dtype,L,layout", CASES)
def test_headdot_pool_pair(F, dtype, L, layout, C):
    lens = _layout(layout)
    offt = _csr(lens)
    n, B = int(sum(lens)), len(lens)
    g = torch.Generator(device="cuda").manual_seed(L * 7 + len(layout) + 100 * C)
    X = torch.randn(n, L, device="cuda", generator=g).to(dtype)
    s = torch.randn(n, device="cuda", generator=g) * 2
    W = torch.randn(C, L, device="cuda", generator=g) * 0.05
    dz = torch.randn(B, C, device="cuda", generator=g)
    keep = (torch.rand(B, L, device="cuda", generator=g) >= 0.25).float() / 0.75
    lowp = dtype != torch.float32
    if _refused(dtype, L, C):
        _expect_rejected(F, lambda: F.segment_softmax_pool_headdot(X, s, offt, W))
        return
    M, Ml, am, lse = F.segment_softmax_pool(X, s, offt, want_lowp=lowp)
    bag = torch.repeat_interleave(torch.arange(B, device="cuda"), (offt[1:] - offt[:-1]).long())
    Xd = X.double()
    # float64 softmax weights and pooled vectors for the backward's reference
    sd = s.double()
    mx = torch.full((B,), -float("inf"), dtype=torch.float64, device="cuda").scatter_reduce(0, bag, sd, "amax")
    e = torch.exp(sd - mx[bag])
    a64 = e / torch.zeros(B, dtype=torch.float64, device="cuda").index_add(0, bag, e)[bag]
    M64 = torch.zeros(B, L, dtype=torch.float64, device="cuda").index_add(0, bag, a64[:, None] * Xd)
    for cs in (None, keep):
        M2, Ml2, am2, lse2, hdot = F.segment_softmax_pool_headdot(X, s, offt, W, cs, want_lowp=lowp)
        torch.cuda.synchronize()
        assert torch.equal(M2, M) and torch.equal(am2, am) and torch.equal(lse2, lse)
        if lowp:
            assert torch.equal(Ml2, Ml)
        scale = torch.ones(B, L, dtype=torch.float64, device="cuda") if cs is None else cs.double()
        V = W.double()[None] * scale[:, None, :]                       # [B, C, L]
        want = torch.einsum("il,icl->ic", Xd, V[bag]) if n * C * L < (1 << 26) else torch.cat(
            [Xd[int(offt[b]):int(offt[b + 1])] @ V[b].T for b in range(B)])
        assert rel_err(hdot.double().cpu().numpy(), want.cpu().numpy()) <= 1e-5, f"hdot (col_scale={cs is not None})"
        dM = (scale * (dz.double() @ W.double())).float()              # the head's gradient of M: s_b * (W^T dz_b)
        ds, attn = F.segment_softmax_pool_bwd_headdot(s, offt, dz, dM, M2, hdot, want_attn=True)
        ds_only, none = F.segment_softmax_pool_bwd_headdot(s, offt, dz, dM, M2, hdot, want_attn=False)
        dMd = dM.double()
        g64, c64 = (Xd * dMd[bag]).sum(1), (dMd * M64).sum(1)[bag]
        ds64 = a64 * (g64 - c64)
        torch.cuda.synchronize()
        # relative to the terms the formula subtracts: a one-row bag has ds = 0 exactly (M = x), and fp32 leaves the
        # rounding of dM . x - dM . M there, larger than the other bags' ds in a batch with a 7000-row bag
        scale = float((a64 * (g64.abs() + c64.abs())).max())
        err = float((ds.double() - ds64).abs().max()) / scale
        assert err <= 1e-5, f"ds (col_scale={cs is not None}): {err:.3e}"
        assert rel_err(attn.double().cpu().numpy(), a64.cpu().numpy()) <= 1e-5
        assert torch.equal(ds_only, ds) and none is None


@pytest.mark.gpu
def test_headdot_pool_rejects_bad_arguments(F):
    L, lens, C = 1024, [300, 0, 257], 2
    offt = _csr(lens)
    n, B = int(sum(lens)), len(lens)
    X = torch.randn(n, L, device="cuda").bfloat16()
    s = torch.randn(n, device="cuda")
    W = torch.randn(8 + 1, L, device="cuda")
    dz = torch.randn(B * 9 + 1, device="cuda")
    dM = torch.randn(B, L, device="cuda")
    M = torch.empty(B, L, device="cuda")
    am = torch.empty(B, dtype=torch.int32, device="cuda")
    lse = torch.empty(B, device="cuda")
    hdot = torch.empty(n * 9 + 1, device="cuda")
    ds = torch.empty(n + 1, device="cuda")
    attn = torch.empty(n + 1, device="cuda")
    lib, p = F.L.lib(), F.L.ptr
    nb = lib.milb200_pool_workspace_bytes(n, B, L)
    ws = F.L.workspace(nb, X.device)

    def off2(t):
        return Cty.c_void_p(t.data_ptr() + 2)

    def fwd(w, c, hd, x=X, Lx=L, code=F.L.BF16):
        return lambda: F.L.check(lib.milb200_segment_softmax_pool_fwd_headdot(
            p(x), p(s), p(offt), B, n, Lx, code, w, c, None, p(M), None, p(am), p(lse), hd, p(ws), ws.numel(),
            F.L.stream_ptr()), "segment_softmax_pool_fwd_headdot")

    def bwd(c, z, hd):
        return lambda: F.L.check(lib.milb200_segment_softmax_pool_bwd_headdot(
            p(s), p(offt), B, n, L, c, z, p(dM), p(M), hd, p(ds), p(attn), p(ws), ws.numel(), F.L.stream_ptr()),
            "segment_softmax_pool_bwd_headdot")

    torch.cuda.synchronize()
    fwd(p(W), C, p(hdot))()                      # the well-formed calls run
    bwd(C, p(dz), p(hdot))()
    torch.cuda.synchronize()
    _expect_rejected(F, fwd(None, C, p(hdot)))
    _expect_rejected(F, fwd(p(W), C, None))
    _expect_rejected(F, fwd(off2(W), C, p(hdot)))
    _expect_rejected(F, fwd(p(W), C, off2(hdot)))
    _expect_rejected(F, fwd(p(W), 0, p(hdot)))
    _expect_rejected(F, fwd(p(W), 9, p(hdot)))
    _expect_rejected(F, bwd(C, None, p(hdot)))
    _expect_rejected(F, bwd(C, off2(dz), p(hdot)))
    _expect_rejected(F, bwd(C, p(dz), None))
    _expect_rejected(F, bwd(C, p(dz), off2(hdot)))
    _expect_rejected(F, bwd(0, p(dz), p(hdot)))
    _expect_rejected(F, bwd(9, p(dz), p(hdot)))
    # staged vectors past the shared memory (and the register budget) of one CTA: bf16 L = 4096 with 8 dots per row
    Xw = torch.randn(n, 4096, device="cuda").bfloat16()
    Ww = torch.randn(8, 4096, device="cuda")
    _expect_rejected(F, lambda: F.segment_softmax_pool_headdot(Xw, s, offt, Ww))
    _expect_rejected(F, fwd(p(Ww), 8, p(hdot), x=Xw, Lx=4096))


# ---------------------------------------------------------------------------------------------------------------------
# the trainer
# ---------------------------------------------------------------------------------------------------------------------
def _head_trainer(dtype, L, C, seed=5, **kw):
    from mil_b200.dp import AbmilTrainer
    tr = AbmilTrainer(L, D, dtype, device="cuda", head_classes=C, **kw)
    p = mo.procedural_state(mo.abmil_shapes(L), seed)
    lay = _layout_of(tr)
    rs = np.random.RandomState(seed + 1)
    full = np.zeros(tr.numel, dtype=np.float32)
    for k, v in p.items():
        a, b = lay[k]
        full[a:b] = v.reshape(-1)
    a, b = lay["head.weight"]
    full[a:b] = rs.uniform(-1, 1, b - a) / np.sqrt(L)
    a, b = lay["head.bias"]
    full[a:b] = rs.uniform(-1, 1, b - a) / np.sqrt(L)
    tr.params.copy_(torch.from_numpy(full))
    return tr


def _layout_of(tr):
    from mil_b200.dp import flat_layout
    return flat_layout(tr.L, tr.D, tr.C)


def _labels(B, C, seed):
    rs = np.random.RandomState(seed)
    return torch.from_numpy(np.eye(C, dtype=np.float32)[rs.randint(0, C, B)] if C > 1 else
                            rs.randint(0, 2, (B, 1)).astype(np.float32)).cuda()


def _oracle(tr, X, off, labels, dtype):
    """float64 oracle of the labelled step at the trainer's current parameters (the gate weights rounded to the compute
    dtype, as the kernels use them): (loss, prob, {flat-layout name: gradient})."""
    lay = _layout_of(tr)
    flat = tr.params.detach().cpu().numpy().astype(np.float64)
    pq = {}
    for k, shp in mo.abmil_shapes(tr.L).items():
        a, b = lay[k]
        v = flat[a:b].reshape(shp)
        if k.endswith("0.weight"):
            v = torch.from_numpy(v).float().to(dtype).double().numpy()
        pq[k] = v
    Xq = X.double().cpu().numpy()
    Mr, _, _ = mo.abmil_forward_csr(pq, Xq, off)
    a, b = lay["head.weight"]
    Wh = flat[a:b].reshape(tr.C, tr.L)
    a, b = lay["head.bias"]
    loss, prob, dM, dW, db = mo.sigmoid_head_bce(Mr, Wh, flat[a:b], labels.cpu().numpy())
    gr = mo.abmil_backward_csr(pq, Xq, off, dM, need_dx=False)
    gr.pop("ds")
    gr["head.weight"], gr["head.bias"] = dW, db
    return loss, prob, gr


def _grads(tr):
    return {k: tr.grads[a:b].detach().cpu().numpy() for k, (a, b) in _layout_of(tr).items()}


def _two_pass(tr, X, offt, labels, seed_h=None):
    """The labelled step's forward and backward without row dots: forward, head + BCE through the same library kernels
    (with the head's dropout drawn from `seed_h`), backward(dM).  Returns (loss, prob, dX)."""
    from mil_b200 import _lib as L
    from mil_b200 import functional as Fn
    lib, B, C, Lf = L.lib(), offt.numel() - 1, tr.C, tr.L
    M = tr.forward(X, offt)
    if tr.head_p > 0.0:
        seed_h = int(torch.randint(0, 2 ** 62, (1,), dtype=torch.int64).item())
    Mh = M if seed_h is None else Fn._dropout_raw(M, tr.head_p, seed_h, 0)
    v, g = tr._views(tr.params), tr._views(tr.grads)
    f32 = dict(dtype=torch.float32, device="cuda")
    z, prob, dz, loss, dMh = (torch.empty(B, C, **f32), torch.empty(B, C, **f32), torch.empty(B, C, **f32),
                              torch.empty(1, **f32), torch.empty(B, Lf, **f32))
    lws = L.workspace(lib.milb200_linear_workspace_bytes(B, C, Lf, L.F32, 1), X.device)
    L.check(lib.milb200_linear_fwd(L.ptr(Mh), None, L.ptr(v["head_w"]), L.ptr(v["head_b"]), L.ptr(z), B, C, Lf,
                                   L.ACT_NONE, L.F32, L.ptr(lws), lws.numel(), L.stream_ptr()), "linear_fwd")
    L.check(lib.milb200_sigmoid_bce_fwd_bwd(L.ptr(z), L.ptr(labels), L.ptr(prob), L.ptr(loss), L.ptr(dz), B * C,
                                            L.stream_ptr()), "sigmoid_bce")
    L.check(lib.milb200_linear_bwd(L.ptr(Mh), None, L.ptr(v["head_w"]), L.ptr(z), L.ptr(dz), L.ptr(dMh), L.ptr(g["head_w"]),
                                   L.ptr(g["head_b"]), B, C, Lf, L.ACT_NONE, L.F32, 0, L.ptr(lws), lws.numel(),
                                   L.stream_ptr()), "linear_bwd")
    dM = dMh if seed_h is None else Fn._dropout_raw(dMh, tr.head_p, seed_h, 0)
    return loss, prob, tr.backward(dM)


LENS = [300, 17, 900, 1, 257, 64]


@pytest.mark.gpu
@pytest.mark.parametrize("C", [1, 2])
@pytest.mark.parametrize("L", [768, 1024])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_labelled_step_matches_oracle(dtype, L, C):
    off = mo.offsets_from_lengths(np.asarray(LENS))
    offt = torch.from_numpy(off).cuda()
    X = torch.from_numpy(rnd(31, int(off[-1]), L)).cuda().to(dtype)
    labels = _labels(len(LENS), C, 8)
    tr = _head_trainer(dtype, L, C)
    loss, prob = tr.forward_backward_labels(X, offt, labels)
    torch.cuda.synchronize()
    lr, pr, gr = _oracle(tr, X, off, labels, dtype)
    tol = 1e-5 if dtype == torch.float32 else 1e-2
    assert abs(float(loss) - lr) <= tol * abs(lr)
    assert rel_err(prob.cpu().numpy(), pr) <= tol
    got = _grads(tr)
    for k, want in gr.items():
        if k == "attention_weights.bias":       # analytically 0 (softmax is shift invariant): both sides are rounding noise
            continue
        assert rel_err(got[k], np.asarray(want).reshape(-1)) <= tol, k


@pytest.mark.gpu
@pytest.mark.parametrize("head_dropout", [0.0, 0.25])
def test_labelled_step_equals_two_pass_route(head_dropout):
    """forward_backward_labels (head row dots in the pooling pass) against forward + head + backward(dM) in fp32, with
    dX, and in train mode with the head's dropout drawn from the same seed."""
    L, C = 1024, 2
    off = mo.offsets_from_lengths(np.asarray(LENS))
    offt = torch.from_numpy(off).cuda()
    X = torch.from_numpy(rnd(32, int(off[-1]), L)).cuda()
    labels = _labels(len(LENS), C, 9)
    a = _head_trainer(torch.float32, L, C, need_input_grad=True, head_dropout=head_dropout)
    b = _head_trainer(torch.float32, L, C, need_input_grad=True, head_dropout=head_dropout)
    names = []
    a.phase_hook = names.append
    torch.manual_seed(41)
    la, pa = a.forward_backward_labels(X, offt, labels)
    dXa = a.last_dX
    torch.manual_seed(41)
    lb, pb, dXb = _two_pass(b, X, offt, labels)
    torch.cuda.synchronize()
    assert "pool_bwd_headdot" in names and "segment_softmax_pool_bwd" not in names
    assert ("head_mask" in names) == (head_dropout > 0)
    assert torch.equal(a.last_argmax, b.last_argmax) and torch.equal(a.last_scores, b.last_scores)
    assert rel_err(la.cpu().numpy(), lb.cpu().numpy()) <= 1e-5 and rel_err(pa.cpu().numpy(), pb.cpu().numpy()) <= 1e-5
    ga, gb = _grads(a), _grads(b)
    for k in ga:
        if k != "attention_weights.bias":
            assert rel_err(ga[k], gb[k]) <= 1e-5, k
    assert rel_err(dXa.cpu().numpy(), dXb.cpu().numpy()) <= 1e-5


@pytest.mark.gpu
def test_reference_pathology_aggregator_pin():
    """The pathology-only aggregator_clip of the reference (golden state, seed 72) loaded into the trainer: prob and the
    pooled vector match the golden outputs; store_to writes the same state_dict back."""
    from mil_b200.dp import AbmilTrainer
    from mil_b200.model import utils_clip
    fx = load_golden("aggregator_clip_path")
    args = Namespace(modality=["pathology"], model_pathology="ABMIL", num_classes=2)
    m = utils_clip.get_model(args).cuda().eval()
    sd = {k: torch.from_numpy(v) for k, v in mo.procedural_state(clip_agg_shapes(False), 72).items()}
    m.load_state_dict(sd)
    tr = AbmilTrainer(768, 192, torch.float32, device="cuda", head_classes=2)
    tr.load_from(m.extractor_pathology, head=m.fc[1])
    X = torch.from_numpy(rnd(272, 1, 64, 768)[0]).cuda()
    offt = torch.tensor([0, 64], dtype=torch.int32, device="cuda")
    labels = torch.tensor([[0.0, 1.0]], device="cuda")
    loss, prob = tr.forward_backward_labels(X, offt, labels)
    torch.cuda.synchronize()
    assert rel_err(prob.cpu().numpy(), fx["prob"]) <= 1e-5
    assert rel_err(tr.last_pooled.cpu().numpy(), fx["pooled"]) <= 1e-5
    m2 = utils_clip.get_model(args).cuda().eval()
    tr.store_to(m2.extractor_pathology, head=m2.fc[1])
    for k, v in m2.state_dict().items():
        assert torch.equal(v.cpu(), sd[k]), k


@pytest.mark.gpu
def test_step_labels_adam_matches_float64():
    """Three step_labels calls (Adam) against float64 Adam on the oracle's gradients, at the reference's learning rate
    (train_ddp.py:113-116)."""
    L, C, lr = 768, 2, 1e-5
    off = mo.offsets_from_lengths(np.asarray(LENS))
    offt = torch.from_numpy(off).cuda()
    X = torch.from_numpy(rnd(33, int(off[-1]), L)).cuda()
    labels = _labels(len(LENS), C, 10)
    tr = _head_trainer(torch.float32, L, C, lr=lr)
    ref = _head_trainer(torch.float32, L, C)              # parameters of the float64 run, one step at a time
    lay = _layout_of(tr)
    p = tr.params.double().cpu().numpy()
    ref0 = p.copy()
    m, v = np.zeros_like(p), np.zeros_like(p)
    live = np.zeros(p.size, dtype=bool)
    for step in range(1, 4):
        ref.params.copy_(torch.from_numpy(p).float())
        _, _, gr = _oracle(ref, X, off, labels, torch.float32)
        g = np.zeros_like(p)
        for k, (a, b) in lay.items():
            g[a:b] = np.asarray(gr[k]).reshape(-1)
        a, b = lay["attention_weights.bias"]
        g[a:b] = 0.0
        live |= np.abs(g) > 1e-3 * np.abs(g).max()
        p, m, v = mo.adam_step(p, g, m, v, step, lr=lr)
        tr.step_labels(X, offt, labels)
    torch.cuda.synchronize()
    got = tr.params.double().cpu().numpy()
    assert tr.step_count == 3
    assert np.abs(got - p)[live].max() <= 1e-5 * np.abs(p).max()
    # the updates themselves: Adam's m / sqrt(v) amplifies the gradients' fp32 rounding where a gradient changes sign
    # between steps, so the bound is looser than the parameters'
    p0 = ref0.astype(np.float64)
    assert np.abs((got - p0) - (p - p0))[live].max() <= 1e-2 * np.abs(p - p0)[live].max()


@pytest.mark.gpu
def test_graphed_labelled_step_equals_eager_steps():
    """Three step_graphed(X, offsets, labels) replays against three eager step_labels calls, bit for bit, with the labels
    rewritten in place between steps (a replay reads the values the buffer holds then)."""
    L, C = 1024, 2
    lens = [900, 40, 0, 2100, 333, 1500]
    offt = _csr(lens)
    X = torch.from_numpy(rnd(34, sum(lens), L)).cuda().bfloat16()
    a = _head_trainer(torch.bfloat16, L, C, lr=1e-3)
    b = _head_trainer(torch.bfloat16, L, C, lr=1e-3)
    la, lb = _labels(len(lens), C, 11), _labels(len(lens), C, 11)
    for step in range(3):
        new = _labels(len(lens), C, 12 + step)
        la.copy_(new)
        lb.copy_(new)
        loss_a, prob_a = a.step_labels(X, offt, la)
        loss_b, prob_b = b.step_graphed(X, offt, lb)
        torch.cuda.synchronize()
        assert torch.equal(loss_a, loss_b) and torch.equal(prob_a, prob_b), step
    assert a.step_count == b.step_count == 3
    assert torch.equal(a.params, b.params) and torch.equal(a.exp_avg, b.exp_avg) and torch.equal(a.exp_avg_sq, b.exp_avg_sq)


# ---------------------------------------------------------------------------------------------------------------------
# host side (no GPU)
# ---------------------------------------------------------------------------------------------------------------------
def test_flat_layout_with_head():
    from mil_b200.dp import AbmilTrainer, flat_layout
    for Lf, C in ((768, 2), (1024, 1), (96, 8)):
        base = flat_layout(Lf, D)
        lay = flat_layout(Lf, D, C)
        assert flat_layout(Lf, D, 0) == base and {k: lay[k] for k in base} == base
        h0, h1 = lay["head.weight"]
        assert h0 % 8 == 0 and h0 >= base["attention_weights.bias"][1] and h1 - h0 == C * Lf
        assert lay["head.bias"] == (h1, h1 + C)
        tr = AbmilTrainer(Lf, D, torch.float32, device="cpu", head_classes=C)
        assert tr.numel == h1 + C and tr.n_pool == 2 * D * Lf + 3 * D + 1
        assert AbmilTrainer(Lf, D, torch.float32, device="cpu").numel == 2 * D * Lf + 3 * D + 1
    with pytest.raises(ValueError):
        AbmilTrainer(64, 8, torch.float32, device="cpu", head_classes=9)


def test_load_from_store_to_round_trip_with_head():
    import mil_b200
    from mil_b200.dp import AbmilTrainer
    torch.manual_seed(0)
    src, dst = mil_b200.ABMIL(None, L=96), mil_b200.ABMIL(None, L=96)
    h_src, h_dst = torch.nn.Linear(96, 3), torch.nn.Linear(96, 3)
    tr = AbmilTrainer(96, 192, torch.float32, device="cpu", head_classes=3)
    tr.load_from(src, head=h_src)
    tr.store_to(dst, head=h_dst)
    for (k, x), (_, y) in zip(src.state_dict().items(), dst.state_dict().items()):
        assert torch.equal(x, y), k
    assert torch.equal(h_src.weight, h_dst.weight) and torch.equal(h_src.bias, h_dst.bias)
    with pytest.raises(ValueError):
        tr.load_from(src, head=torch.nn.Linear(96, 2))
    with pytest.raises(ValueError):
        AbmilTrainer(96, 192, torch.float32, device="cpu").load_from(src, head=h_src)
