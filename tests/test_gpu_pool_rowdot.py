"""GPU tests of the pooling pair that takes the backward's row dots in the forward (milb200_segment_softmax_pool_fwd_rowdot
/ _bwd_rowdot) and of AbmilTrainer.forward_backward, which uses it.

The row-dot forward must return the plain forward's M, M_lowp, argmax and lse, and the row-dot backward the plain
backward's ds and attn, bit for bit, at every vector width the pool kernels are instantiated for and on bag layouts that
straddle their row slabs or hold empty bags; empty bags change no output or gradient of the other bags.
forward_backward(X, offsets, dM) must give the same gradients, dX, scores and argmax as forward() followed by
backward(dM), which keeps the two-pass backward."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import mil_oracle as mo
from tests.test_gpu_shape_edges import _layout as shape_edges_layout

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def F():
    from mil_b200 import functional
    return functional


def _csr(lens):
    return torch.from_numpy(mo.offsets_from_lengths(np.asarray(lens))).cuda()


def _layout(name):
    """The bag layouts of the shape-edges tests, plus empty bags first, mid-batch (inside and at slab edges) and last."""
    if name == "empty":
        return [0, 5, 0, 300, 0, 0, 257, 1, 511, 0, 3, 0]
    return shape_edges_layout(name)


# Every NV bucket of both dtypes (NV = ceil(L * elem / 16 / 32)): bf16 L = 8 / 264 / 768 / 1000, 1024 / 1280, 1536 /
# 2048 / 4096 run NV = 1 / 2 / 3 / 4 / 6 / 8 / 16; fp32 L = 4 / 132 / 384 / 512, 1000 / 768 / 1024 / 1028, 1536, 2048 the
# same.  264, 1000, 132 and 1028 leave lanes with a partial last vector.
CASES = [(torch.bfloat16, 8, "tiny"), (torch.bfloat16, 264, "slabs"), (torch.bfloat16, 768, "empty"),
         (torch.bfloat16, 1000, "wide"), (torch.bfloat16, 1024, "slabs"), (torch.bfloat16, 1024, "empty"),
         (torch.bfloat16, 1280, "one"), (torch.bfloat16, 1536, "mixed"), (torch.bfloat16, 1536, "empty"),
         (torch.bfloat16, 2048, "slabs"), (torch.bfloat16, 4096, "mixed"),
         (torch.float32, 4, "slabs"), (torch.float32, 132, "tiny"), (torch.float32, 384, "empty"),
         (torch.float32, 512, "one"), (torch.float32, 768, "mixed"), (torch.float32, 1024, "slabs"),
         (torch.float32, 1024, "empty"), (torch.float32, 1028, "wide"), (torch.float32, 1536, "slabs"),
         (torch.float32, 1536, "empty"), (torch.float32, 2048, "mixed")]


@pytest.mark.parametrize("dtype,L,layout", CASES)
def test_rowdot_pool_pair_equals_plain_pool_pair(F, dtype, L, layout):
    lens = _layout(layout)
    offt = _csr(lens)
    n, B = int(sum(lens)), len(lens)
    g = torch.Generator(device="cuda").manual_seed(L * 7 + len(layout))
    X = torch.randn(n, L, device="cuda", generator=g).to(dtype)
    s = torch.randn(n, device="cuda", generator=g) * 2
    dM = torch.randn(B, L, device="cuda", generator=g)
    lowp = dtype != torch.float32
    M, Ml, am, lse = F.segment_softmax_pool(X, s, offt, want_lowp=lowp)
    ds, attn = F.segment_softmax_pool_bwd(X, s, offt, dM, M, want_attn=True)
    M2, Ml2, am2, lse2, rowdot = F.segment_softmax_pool_rowdot(X, s, offt, dM, want_lowp=lowp)
    ds2, attn2 = F.segment_softmax_pool_bwd_rowdot(s, offt, dM, M2, rowdot, want_attn=True)
    ds3, none = F.segment_softmax_pool_bwd_rowdot(s, offt, dM, M2, rowdot, want_attn=False)
    torch.cuda.synchronize()
    assert torch.equal(M2, M) and torch.equal(am2, am) and torch.equal(lse2, lse)
    if lowp:
        assert torch.equal(Ml2, Ml)
    assert torch.equal(ds2, ds) and torch.equal(attn2, attn) and torch.equal(ds3, ds) and none is None
    # the row dots themselves against float64
    bag = torch.repeat_interleave(torch.arange(B, device="cuda"), (offt[1:] - offt[:-1]).long())
    want = (X.double() * dM.double()[bag]).sum(1)
    err = float((rowdot.double() - want).abs().max() / want.abs().max().clamp_min(1e-30))
    assert err <= 1e-5, f"rowdot: max-norm relative error {err:.3e}"


def _expect_rejected(F, fn):
    n0 = F.L.launch_count()
    with pytest.raises(F.L.MilB200Error):
        fn()
    torch.cuda.synchronize()
    assert F.L.launch_count() == n0, "a call whose argument check failed launched a kernel"


def test_rowdot_pool_rejects_null_and_misaligned_pointers(F):
    L, lens = 1024, [300, 0, 257]
    offt = _csr(lens)
    n, B = int(sum(lens)), len(lens)
    X = torch.randn(n, L, device="cuda").bfloat16()
    s = torch.randn(n, device="cuda")
    dM = torch.randn(B, L, device="cuda")
    M = torch.empty(B, L, device="cuda")
    am = torch.empty(B, dtype=torch.int32, device="cuda")
    lse = torch.empty(B, device="cuda")
    rowdot = torch.empty(n + 1, device="cuda")
    ds = torch.empty(n + 1, device="cuda")
    attn = torch.empty(n + 1, device="cuda")
    lib, p = F.L.lib(), F.L.ptr
    nb = lib.milb200_pool_workspace_bytes(n, B, L)
    ws = F.L.workspace(nb, X.device)

    def off2(t):
        return C.c_void_p(t.data_ptr() + 2)

    def fwd(dm, rd, ws_bytes=ws.numel()):
        return lambda: F.L.check(lib.milb200_segment_softmax_pool_fwd_rowdot(
            p(X), p(s), p(offt), B, n, L, F.L.BF16, dm, p(M), None, p(am), p(lse), rd, p(ws), ws_bytes,
            F.L.stream_ptr()), "segment_softmax_pool_fwd_rowdot")

    def bwd(rd, d, a, ws_bytes=ws.numel()):
        return lambda: F.L.check(lib.milb200_segment_softmax_pool_bwd_rowdot(
            p(s), p(offt), B, n, L, p(dM), p(M), rd, d, a, p(ws), ws_bytes, F.L.stream_ptr()),
            "segment_softmax_pool_bwd_rowdot")

    torch.cuda.synchronize()
    fwd(p(dM), p(rowdot))()                      # the well-formed calls run
    bwd(p(rowdot), p(ds), p(attn))()
    torch.cuda.synchronize()
    _expect_rejected(F, fwd(None, p(rowdot)))
    _expect_rejected(F, fwd(p(dM), None))
    _expect_rejected(F, fwd(off2(dM), p(rowdot)))
    _expect_rejected(F, fwd(p(dM), off2(rowdot)))
    _expect_rejected(F, fwd(p(dM), p(rowdot), nb - 1))
    _expect_rejected(F, bwd(None, p(ds), p(attn)))
    _expect_rejected(F, bwd(p(rowdot), None, p(attn)))
    _expect_rejected(F, bwd(off2(rowdot), p(ds), p(attn)))
    _expect_rejected(F, bwd(p(rowdot), off2(ds), p(attn)))
    _expect_rejected(F, bwd(p(rowdot), p(ds), off2(attn)))
    _expect_rejected(F, bwd(p(rowdot), p(ds), p(attn), nb - 1))
    # rows past the widest instantiation, as for the plain forward
    Xw = torch.randn(n, 4104, device="cuda").bfloat16()
    _expect_rejected(F, lambda: F.segment_softmax_pool_rowdot(Xw, s, offt, torch.randn(B, 4104, device="cuda")))


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_empty_bags_have_defined_outputs_and_zero_gradient_share(F, dtype):
    """Zero-length bags at the start, in the middle (also exactly on a slab boundary of the persistent pool kernel) and at
    the end of a packed batch: pooled vector 0, argmax -1, lse -inf; the other bags and every gradient are what the batch
    without the empty bags gives, through the pooling backward and the gate backward (with and without dX)."""
    L, D = 1024, 192
    lens_full = [0, 0, 700, 0, 4096, 0, 33, 0]
    lens = [l for l in lens_full if l > 0]
    off_full = _csr(lens_full)
    off = _csr(lens)
    gen = torch.Generator(device="cuda").manual_seed(13)
    X = torch.randn(sum(lens), L, device="cuda", generator=gen).to(dtype)
    Wv = torch.randn(D, L, device="cuda", generator=gen) * 0.03
    Wu = torch.randn(D, L, device="cuda", generator=gen) * 0.03
    bv = torch.zeros(D, device="cuda")
    ww = torch.randn(D, device="cuda", generator=gen) * 0.3
    bw = torch.zeros(1, device="cuda")
    Wcat, bcat = F.pack_gate_weights(Wv, bv, Wu, bv, dtype)
    s, act = F.gated_scores(X, Wcat, bcat, ww, bw, save=True)
    M, _, am, lse = F.segment_softmax_pool(X, s, off)
    Mf, _, amf, lsef = F.segment_softmax_pool(X, s, off_full)
    keep = torch.tensor([i for i, l in enumerate(lens_full) if l > 0], device="cuda")
    gone = torch.tensor([i for i, l in enumerate(lens_full) if l == 0], device="cuda")
    assert torch.equal(Mf[keep], M) and torch.equal(amf[keep], am) and torch.equal(lsef[keep], lse)
    assert float(Mf[gone].abs().max()) == 0.0 and bool((amf[gone] == -1).all()) and bool(torch.isinf(lsef[gone]).all())
    dMf = torch.randn(len(lens_full), L, device="cuda", generator=gen)
    dM = dMf[keep].contiguous()
    ds, attn = F.segment_softmax_pool_bwd(X, s, off, dM, M, want_attn=True)
    dsf, attnf = F.segment_softmax_pool_bwd(X, s, off_full, dMf, Mf, want_attn=True)
    assert torch.equal(ds, dsf) and torch.equal(attn, attnf)
    for need_dx in (False, True):
        a = F.gated_scores_bwd(X, Wcat, bcat, ww, bw, ds, attn, dM, off, need_dx, gate_act=act)
        b = F.gated_scores_bwd(X, Wcat, bcat, ww, bw, dsf, attnf, dMf, off_full, need_dx, gate_act=act)
        assert (a[0] is None) == (b[0] is None) == (not need_dx)
        for name, x, y in zip(("dX", "dWcat", "dbcat", "dww", "dbw"), a, b):
            assert x is None or torch.equal(x, y), (name, need_dx)


# ---------------------------------------------------------------------------------------------------------------------
# AbmilTrainer: forward_backward (row dots) against forward + backward (two passes)
# ---------------------------------------------------------------------------------------------------------------------
def _trainer(dtype, L, **kw):
    from mil_b200.dp import AbmilTrainer
    tr = AbmilTrainer(L, 192, dtype, device="cuda", **kw)
    g = torch.Generator(device="cuda").manual_seed(21)
    tr.params.copy_(torch.randn(tr.numel, device="cuda", generator=g) * 0.03)
    return tr


def _phases(tr):
    names = []
    tr.phase_hook = names.append
    return names


@pytest.mark.parametrize("dtype,L", [(torch.bfloat16, 1024), (torch.float32, 512)])
@pytest.mark.parametrize("save_gate", [True, False])
@pytest.mark.parametrize("need_input_grad", [False, True])
@pytest.mark.parametrize("dropout_p", [0.0, 0.5])
@pytest.mark.parametrize("random_dM", [True, False])
def test_forward_backward_equals_forward_then_backward(dtype, L, save_gate, need_input_grad, dropout_p, random_dM):
    lens = [300, 0, 17, 900, 1, 257, 0]
    offt = _csr(lens)
    n, B = int(sum(lens)), len(lens)
    g = torch.Generator(device="cuda").manual_seed(3)
    X = torch.randn(n, L, device="cuda", generator=g).to(dtype)
    dM = torch.randn(B, L, device="cuda", generator=g) if random_dM else None
    kw = dict(save_gate=save_gate, need_input_grad=need_input_grad, dropout_p=dropout_p)
    a, b = _trainer(dtype, L, **kw), _trainer(dtype, L, **kw)
    pa, pb = _phases(a), _phases(b)
    torch.manual_seed(77)                                     # the dropout seed comes from torch's generator
    Ma, dXa = a.forward_backward(X, offt, dM)
    torch.manual_seed(77)
    Mb = b.forward(X, offt)
    dXb = b.backward(dM if random_dM else torch.ones(B, L, device="cuda"))
    torch.cuda.synchronize()
    assert "pool_bwd_rowdot" in pa and "segment_softmax_pool_bwd" not in pa
    assert "segment_softmax_pool_bwd" in pb and "pool_bwd_rowdot" not in pb
    assert torch.equal(Ma, Mb)
    assert torch.equal(a.last_scores, b.last_scores) and torch.equal(a.last_argmax, b.last_argmax)
    assert torch.equal(a.grads, b.grads)
    assert float(a.grads.abs().max()) > 0
    if need_input_grad:
        assert torch.equal(dXa, dXb)
    else:
        assert dXa is None and dXb is None


def test_graphed_step_equals_eager_step():
    """step_graphed (one replayed CUDA graph, row-dot pooling inside) against the eager step: the first step's pooled
    vectors and gradients bit for bit, then three steps' parameters (the graph's Adam reads its step number from device
    memory, so the updates are compared with a tolerance, as in test_gpu_parity_r2)."""
    L, lens = 1024, [900, 40, 0, 2100, 333, 1500]
    offt = _csr(lens)
    X = torch.randn(sum(lens), L, device="cuda").bfloat16()
    a, b = _trainer(torch.bfloat16, L, lr=1e-3), _trainer(torch.bfloat16, L, lr=1e-3)
    p0 = a.params.clone()
    Ma = a.step(X, offt).clone()
    Mb = b.step_graphed(X, offt).clone()
    torch.cuda.synchronize()
    assert torch.equal(Ma, Mb) and torch.equal(a.grads, b.grads) and torch.equal(a.last_argmax, b.last_argmax)
    for _ in range(2):
        Ma = a.step(X, offt).clone()
        Mb = b.step_graphed(X, offt).clone()
    torch.cuda.synchronize()
    assert a.step_count == b.step_count == 3
    assert float((Ma - Mb).abs().max()) <= 1e-5 * float(Ma.abs().max())
    live = a.grads.abs() > 1e-4 * a.grads.abs().max()
    ua, ub = (a.params - p0)[live], (b.params - p0)[live]
    assert float((ua - ub).abs().max()) <= 1e-3 * float(ua.abs().max())
    assert torch.equal(a.last_argmax, b.last_argmax)
