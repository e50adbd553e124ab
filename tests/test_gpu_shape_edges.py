"""GPU tests of the kernels at the edges of the shapes their argument checks accept, each against a float64 reference
evaluated on the operands the kernel saw (bf16 inputs and weights quantised as the kernel reads them):

  A. the gated pool at any L (K tails of the tensor-core GEMMs, the last partial 512-column tile of the TN GEMM, odd
     m-tile counts that leave the second CTA of a pair without rows) and any D <= 256 on the FFMA path;
  B. the segmented softmax pool, segment sum and bag broadcast at every vector width the kernels are instantiated for,
     on bag layouts that straddle their row slabs;
  C. the dense linear layer (bf16 tensor cores, the small-m kernel, FFMA, 3xTF32) at N / M / K tails, every activation,
     with and without the fused add and the bias, and on both sides of every routing boundary;
  D. LayerNorm with a broadcast residual row and the column sum (the additions to LayerNorm and attention sit with their
     existing tests in test_gpu_fusion.py).

Tolerances as in the rest of the suite: max-norm relative error fp32 <= 1e-5, bf16 <= 1e-2; argmax bit-exact; exactly
zero true gradients (the score bias) get an absolute bound.  Shapes just outside each check must raise MilB200Error
without launching anything (the C ABI promises that nothing is launched when a check fails)."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from oracle import mil_oracle as mo

pytestmark = pytest.mark.gpu

TOL = {torch.float32: 1e-5, torch.bfloat16: 1e-2}
F64 = torch.float64


@pytest.fixture(scope="module")
def F():
    from mil_b200 import functional
    return functional


def _rel(a, b):
    a, b = a.detach().to(F64), b.detach().to(F64).to(a.device)
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def _close(name, got, want, tol):
    e = _rel(got, want)
    assert e <= tol, f"{name}: max-norm relative error {e:.3e} > {tol:g}"


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _lens(n, pattern=(31, 1, 33, 2, 64, 5, 97, 129, 7, 255, 3, 40)):
    """Bag lengths summing to n whose boundaries fall inside the 128-row tiles and 32-row k-blocks."""
    out, tot, i = [], 0, 0
    while tot < n:
        out.append(min(pattern[i % len(pattern)], n - tot))
        tot += out[-1]
        i += 1
    return out


def _csr(lens):
    off = mo.offsets_from_lengths(np.asarray(lens))
    return torch.from_numpy(off).cuda()


def _bag_of_row(offt):
    lens = (offt[1:] - offt[:-1]).long()
    return torch.repeat_interleave(torch.arange(lens.numel(), device=offt.device), lens)


def _expect_rejected(F, fn):
    """fn must raise MilB200Error and launch no kernel."""
    n0 = F.L.launch_count()
    with pytest.raises(F.L.MilB200Error):
        fn()
    torch.cuda.synchronize()
    assert F.L.launch_count() == n0, "a call whose argument check failed launched a kernel"


# ---------------------------------------------------------------------------------------------------------------------
# float64 references
# ---------------------------------------------------------------------------------------------------------------------
def _first_argmax(s, offt, bag):
    """Index within the bag of the largest score, the first one on ties; plus the gap to the runner-up (inf for
    single-row bags)."""
    B = offt.numel() - 1
    mx = torch.full((B,), -math.inf, dtype=s.dtype, device=s.device).scatter_reduce(0, bag, s, "amax")
    local = torch.arange(s.numel(), device=s.device) - offt[:-1].long()[bag]
    big = torch.iinfo(torch.int64).max
    cand = torch.where(s == mx[bag], local, torch.full_like(local, big))
    am = torch.full((B,), big, dtype=torch.int64, device=s.device).scatter_reduce(0, bag, cand, "amin")
    s2 = s.clone()
    s2[offt[:-1].long() + am] = -math.inf
    mx2 = torch.full((B,), -math.inf, dtype=s.dtype, device=s.device).scatter_reduce(0, bag, s2, "amax")
    return am, mx - mx2


def _pool_ref(Xd, sd, offt, bag):
    B = offt.numel() - 1
    mx = torch.full((B,), -math.inf, dtype=F64, device=Xd.device).scatter_reduce(0, bag, sd, "amax")
    e = torch.exp(sd - mx[bag])
    den = torch.zeros(B, dtype=F64, device=Xd.device).index_add_(0, bag, e)
    a = e / den[bag]
    M = torch.zeros(B, Xd.shape[1], dtype=F64, device=Xd.device).index_add_(0, bag, a[:, None] * Xd)
    return M, a, mx + torch.log(den)


def _pool_bwd_ref(Xd, a, M, dM, bag):
    """ds_i = a_i (dM_b . x_i - dM_b . M_b), and the size of the terms before that difference: a one-row bag has ds = 0
    exactly, but the kernel forms it from two fp32 dot products of size |dM| |x| taken in different orders, so ds is
    compared relative to max_i a_i (|dM_b . x_i| + |dM_b . M_b|)."""
    dMd = dM.to(F64)
    g = (Xd * dMd[bag]).sum(1)
    c = (dMd * M.to(F64)).sum(1)[bag]
    return a * (g - c), float((a * (g.abs() + c.abs())).max())


def _close_ds(name, got, want, scale, tol):
    e = float((got.to(F64) - want).abs().max()) / max(scale, 1e-30)
    assert e <= tol, f"{name}: error {e:.3e} of the dot-product scale > {tol:g}"


def _check_argmax(am, s, sr, offt, bag):
    """Bit-exact: the kernel's argmax is the first maximum of the kernel's own scores, and equals the float64 argmax in
    every bag whose top two float64 scores are further apart than the kernel's score error (mo.score_margin per bag)."""
    am = am.long()
    own, _ = _first_argmax(s.to(F64), offt, bag)
    assert torch.equal(am, own), "argmax is not the first maximum of the scores"
    ref, margin = _first_argmax(sr, offt, bag)
    err = float((s.to(F64) - sr).abs().max())
    ok = margin > 4 * err + 1e-7
    assert torch.equal(am[ok], ref[ok]), "argmax differs from the float64 argmax in a well-separated bag"
    assert float(ok.double().mean()) >= 0.5, "too few well-separated bags for the argmax check"


# ---------------------------------------------------------------------------------------------------------------------
# A. gated pool at any L and D
# ---------------------------------------------------------------------------------------------------------------------
def _gate_params(L, D, seed):
    g = _gen(seed)
    Wv = torch.randn(D, L, device="cuda", generator=g) / math.sqrt(L)
    Wu = torch.randn(D, L, device="cuda", generator=g) / math.sqrt(L)
    bv = torch.randn(D, device="cuda", generator=g) * 0.1
    bu = torch.randn(D, device="cuda", generator=g) * 0.1
    ww = torch.randn(D, device="cuda", generator=g) * 0.3
    bw = torch.randn(1, device="cuda", generator=g) * 0.1
    return g, (Wv, bv, Wu, bu, ww, bw)


def _gated_pool(F, dtype, L, D, lens, seed):
    """Forward through functional, every backward variant the shape supports; returns (got, reference)."""
    offt = _csr(lens)
    n, B = int(sum(lens)), len(lens)
    g, (Wv, bv, Wu, bu, ww, bw) = _gate_params(L, D, seed)
    X = torch.randn(n, L, device="cuda", generator=g).to(dtype)
    dM = torch.randn(B, L, device="cuda", generator=g)
    Wcat, bcat = F.pack_gate_weights(Wv, bv, Wu, bu, dtype)
    s, act = F.gated_scores(X, Wcat, bcat, ww, bw, save=True)
    M, Ml, am, lse = F.segment_softmax_pool(X, s, offt, want_lowp=dtype != torch.float32)
    ds, attn = F.segment_softmax_pool_bwd(X, s, offt, dM, M, want_attn=True)
    got = {"s": s, "M": M, "M_lowp": Ml, "argmax": am, "lse": lse, "ds": ds, "attn": attn, "act": act}
    runs = {"saved+dX": (act, True), "saved": (act, False), "recompute+dX": (None, True), "recompute": (None, False)}
    seen = set()
    for name, (ga, need_dx) in runs.items():
        if (ga is None, need_dx) in seen:
            continue             # the FFMA paths save nothing: "saved" is "recompute" there
        seen.add((ga is None, need_dx))
        dX, dWcat, dbcat, dww, dbw = F.gated_scores_bwd(X, Wcat, bcat, ww, bw, ds, attn, dM, offt, need_dx, gate_act=ga)
        got[name] = [t.clone() if t is not None else None for t in (dX, dWcat, dbcat, dww, dbw)]
    torch.cuda.synchronize()

    q = (lambda t: t.to(dtype).to(F64))
    Xd = X.to(F64)
    Wvd, Wud = q(Wv), q(Wu)
    V = torch.tanh(Xd @ Wvd.t() + bv.to(F64))
    U = torch.sigmoid(Xd @ Wud.t() + bu.to(F64))
    wwd = ww.to(F64)
    sr = (V * U) @ wwd + bw.to(F64)
    bag = _bag_of_row(offt)
    Mr, a, lser = _pool_ref(Xd, sr, offt, bag)
    dsr, ds_scale = _pool_bwd_ref(Xd, a, M, dM, bag)    # M: the forward result the backward is handed
    dG = dsr[:, None] * wwd[None, :]
    dVp, dUp = dG * U * (1 - V * V), dG * V * U * (1 - U)
    ref = {"s": sr, "M": Mr, "lse": lser, "ds": dsr, "ds_scale": ds_scale, "attn": a,
           "dX": a[:, None] * dM.to(F64)[bag] + dVp @ Wvd + dUp @ Wud,
           "dWcat": torch.cat([dVp.t() @ Xd, dUp.t() @ Xd]), "dbcat": torch.cat([dVp.sum(0), dUp.sum(0)]),
           "dww": dsr @ (V * U), "dbw": dsr.sum()}
    return got, ref, offt, bag


def _check_gated_pool(got, ref, offt, bag, dtype, lens):
    tol = TOL[dtype]
    singles = max(lens) == 1        # every softmax weight is 1: ds and all parameter gradients are 0 in exact arithmetic
    for k in ("s", "M", "lse", "attn"):
        _close(k, got[k], ref[k], tol)
    if got["M_lowp"] is not None:
        _close("M_lowp", got["M_lowp"], ref["M"], tol)
    _check_argmax(got["argmax"], got["s"], ref["s"], offt, bag)
    dscale = float(ref["ds"].abs().max()) if not singles else 1.0
    n = int(sum(lens))
    for run in ("saved+dX", "saved", "recompute+dX", "recompute"):
        if run not in got:
            continue
        dX, dWcat, dbcat, dww, dbw = got[run]
        if dX is not None:
            _close(f"{run} dX", dX, ref["dX"], tol)
        for k, t in (("dWcat", dWcat), ("dbcat", dbcat), ("dww", dww)):
            if singles:
                assert float(t.abs().max()) <= 1e-4, (run, k)
            else:
                _close(f"{run} {k}", t, ref[k], tol)
        assert abs(float(dbw) - float(ref["dbw"])) <= 2e-5 * math.sqrt(n) * dscale + 1e-6, (run, "dbw", float(dbw))
    _close_ds("ds", got["ds"], ref["ds"], ref["ds_scale"], tol)


# bf16, D = 192, L % 16 == 0: the tensor-core path.  L = 64 is one K block, 80 / 144 / 208 / 1008 end in a partial K block,
# 1040 gives the TN GEMM a third 512-column tile with 16 valid columns, 1536 / 2048 run the pool's NV = 6 / 8.  Row counts: 1, one short m-tile,
# +-1 around the 128-row tile and the 256-row CTA pair, an odd tile count (385 = 3 tiles + 1 row), and a batch past a
# full wave of 74 CTA pairs (2 x 18944 + 129 rows).
# The saved-activation dW kernel (k_gemm_tn_gate) splits the 32-row k-blocks over 49 / 24 / 6 splits (L <= 512 / <= 1024
# / 4096 on 148 SMs) and stages ds eight k-blocks at a time in a 32-block ring: splits of exactly 8 and 9 k-blocks
# (512 x 49*8*32, 512 x 49*9*32), a ring that wraps once or twice (1024 x 24*33*32, 768 x 24*64*32 + 5), a last split
# shorter than one ds chunk (1024 x 24*8*32 + 1) and fewer than 8 rows (256 x 7).  L = 96 / 112 end the accumulator
# epilogue in a full / half 32-column chunk, 528 puts 16 columns in a second 512-column tile at L <= 1024, and 4096 runs
# eight 512-column tiles with the pool's NV = 16.
TC_CASES = [(64, 1), (80, 31), (144, 127), (208, 128), (1008, 129), (1040, 256), (1536, 257), (2048, 385),
            (80, 2 * 18944 + 129), (1040, 2 * 18944 + 129),
            (512, 49 * 8 * 32), (512, 49 * 9 * 32), (1024, 24 * 33 * 32), (768, 24 * 64 * 32 + 5), (1024, 24 * 8 * 32 + 1),
            (256, 7), (96, 2), (112, 33), (528, 300), (4096, 40)]


@pytest.mark.parametrize("L,n", TC_CASES)
def test_gated_pool_tensor_core_path_any_L(F, L, n):
    lens = _lens(n)
    got, ref, offt, bag = _gated_pool(F, torch.bfloat16, L, 192, lens, seed=L + n)
    assert got["saved"][1] is not None
    assert got["act"] is not None, "the tensor-core forward must save the gate activations"
    _check_gated_pool(got, ref, offt, bag, torch.bfloat16, lens)


# FFMA path: any D <= 256 (D = 100 leaves lanes with a partial last group of gate units), bf16 with L < 64 or L % 16 == 8,
# and fp32 shapes below the 3xTF32 row threshold.
FFMA_CASES = [(torch.float32, 64, 56), (torch.float32, 100, 96), (torch.float32, 128, 1000), (torch.float32, 256, 96),
              (torch.bfloat16, 64, 1000), (torch.bfloat16, 100, 56), (torch.bfloat16, 128, 96),
              (torch.bfloat16, 256, 8), (torch.bfloat16, 192, 56), (torch.bfloat16, 192, 8),
              (torch.bfloat16, 192, 72), (torch.bfloat16, 192, 1000)]


@pytest.mark.parametrize("dtype,D,L", FFMA_CASES)
def test_gated_pool_ffma_path_any_D(F, dtype, D, L):
    lens = _lens(700)
    got, ref, offt, bag = _gated_pool(F, dtype, L, D, lens, seed=D * 7 + L)
    if dtype == torch.bfloat16:
        assert got["act"] is None, "bf16 gate activations are saved by the tensor-core forward only"
    _check_gated_pool(got, ref, offt, bag, dtype, lens)


@pytest.mark.parametrize("dtype,L,D", [(torch.bfloat16, 1008, 192), (torch.bfloat16, 1000, 192), (torch.bfloat16, 200, 100),
                                         (torch.float32, 96, 100)])
def test_abmil_module_at_other_L_and_D_matches_oracle(dtype, L, D):
    """nn.Module route (ABMIL(None, L, D).forward_csr, autograd) on each gate path against the float64 oracle."""
    import mil_b200
    lens = [1, 40, 129, 7, 300]
    off = mo.offsets_from_lengths(np.asarray(lens))
    p = mo.procedural_state(mo.abmil_shapes(L, D), 31)
    m = mil_b200.ABMIL(None, L=L, D=D).cuda().eval()
    m.load_state_dict({k: torch.from_numpy(v) for k, v in p.items()})
    g = _gen(L + D)
    X = torch.randn(int(off[-1]), L, device="cuda", generator=g).to(dtype).requires_grad_(True)
    dM = torch.randn(len(lens), L, device="cuda", generator=g)
    M = m.forward_csr(X, torch.from_numpy(off).cuda())
    (M.float() * dM).sum().backward()
    torch.cuda.synchronize()
    pq = {k: (torch.from_numpy(v).to(dtype).float().numpy() if k.endswith("0.weight") else v) for k, v in p.items()}
    Xq = X.detach().double().cpu().numpy()
    Mr, sr, amr = mo.abmil_forward_csr(pq, Xq, off)
    gr = mo.abmil_backward_csr(pq, Xq, off, dM.double().cpu().numpy())
    tol = TOL[dtype]
    assert mo.score_margin(sr, off) > 1e-4, "seed gives a near-tie; argmax would not be well-posed"
    assert m.last_argmax.cpu().numpy().tolist() == amr.tolist()
    _close("M", M, torch.from_numpy(Mr), tol)
    _close("scores", m.last_scores, torch.from_numpy(sr), tol)
    _close("dX", X.grad, torch.from_numpy(gr["x"]), tol)
    for k, prm in m.state_dict(keep_vars=True).items():
        if k == "attention_weights.bias":
            assert abs(float(prm.grad) - float(gr[k][0])) <= 1e-4
        else:
            _close(k, prm.grad, torch.from_numpy(np.asarray(gr[k])), tol)


def test_gated_pool_tail_shape_is_repeatable(F):
    """Every output of the tensor-core forward and of each backward variant twice, bit for bit, at a K tail and a partial
    TN tile with an odd number of m-tiles (a race or a stale pipeline stage at a tail shows up here first)."""
    lens = _lens(2 * 18944 + 129)
    a, _, _, _ = _gated_pool(F, torch.bfloat16, 1040, 192, lens, seed=5)
    b, _, _, _ = _gated_pool(F, torch.bfloat16, 1040, 192, lens, seed=5)
    for k in a:
        xs, ys = (a[k], b[k]) if isinstance(a[k], list) else ([a[k]], [b[k]])
        for x, y in zip(xs, ys):
            assert (x is None and y is None) or torch.equal(x, y), k


def test_gated_scores_reject_unsupported_shapes(F):
    _, (Wv, bv, Wu, bu, ww, bw) = _gate_params(1000, 257, 3)
    for dtype in (torch.float32, torch.bfloat16):
        X = torch.randn(300, 1000, device="cuda").to(dtype)
        offt = _csr([100, 200])
        Wcat, bcat = F.pack_gate_weights(Wv, bv, Wu, bu, dtype)
        ds = torch.randn(300, device="cuda")
        dM = torch.randn(2, 1000, device="cuda")
        torch.cuda.synchronize()
        # D = 257 > 256 is outside the FFMA backward (8 gate units per lane)
        _expect_rejected(F, lambda: F.gated_scores_bwd(X, Wcat, bcat, ww, bw, ds, None, dM, offt, False))
    # bf16 rows of 60 elements are 120 bytes: not a multiple of 16
    _, (Wv, bv, Wu, bu, ww, bw) = _gate_params(60, 192, 3)
    X = torch.randn(300, 60, device="cuda").bfloat16()
    Wcat, bcat = F.pack_gate_weights(Wv, bv, Wu, bu, torch.bfloat16)
    torch.cuda.synchronize()
    _expect_rejected(F, lambda: F.gated_scores(X, Wcat, bcat, ww, bw))


# ---------------------------------------------------------------------------------------------------------------------
# B. pool, segment sum and bag broadcast at every vector width
# ---------------------------------------------------------------------------------------------------------------------
def _layout(name):
    if name == "slabs":          # straddle the 256-row forward slab and the 128-row backward slab
        return [255, 256, 257, 513, 1, 255, 256, 257]
    if name == "one":            # one bag over ~28 slabs, between two one-row bags
        return [1, 7001, 1]
    if name == "tiny":           # 20 000 bags of 1..3 rows
        return mo.ragged_lengths(20000, 1, 3, 7).tolist()
    if name == "wide":           # > 2 x 148 x 256 rows: the slab grows past its minimum
        return [1300] * 58 + [1, 1400]
    return [1, 2, 17, 255, 256, 257, 513, 1000, 3]


# bf16 L = 8 is one 16-byte vector per row, 264 a partial nv = 2, 1000 a partial nv = 4, 1280 / 2048 / 4096 run NV = 6 /
# 8 / 16; fp32 L = 4 is one vector, 132 and 1028 leave lanes with a partial last vector, 2048 runs NV = 16.
POOL_CASES = [(torch.bfloat16, 8, "tiny"), (torch.bfloat16, 264, "slabs"), (torch.bfloat16, 1000, "wide"),
              (torch.bfloat16, 1280, "one"), (torch.bfloat16, 2048, "slabs"), (torch.bfloat16, 4096, "mixed"),
              (torch.float32, 4, "slabs"), (torch.float32, 132, "tiny"), (torch.float32, 1000, "one"),
              (torch.float32, 1028, "wide"), (torch.float32, 2048, "mixed")]


def _pool_all(F, X, s, offt, dM, w):
    lib, code = F.L.lib(), F.L.dtype_code(X)
    n, L = X.shape
    B = offt.numel() - 1
    M, Ml, am, lse = F.segment_softmax_pool(X, s, offt, want_lowp=X.dtype != torch.float32)
    ds, attn = F.segment_softmax_pool_bwd(X, s, offt, dM, M, want_attn=True)
    ds2, _ = F.segment_softmax_pool_bwd(X, s, offt, dM, M, want_attn=False)
    S = torch.empty(B, L, device="cuda")
    Sl = torch.empty(B, L, device="cuda", dtype=X.dtype)
    ws = F.L.workspace(lib.milb200_pool_workspace_bytes(n, B, L), X.device)
    F.L.check(lib.milb200_segment_sum_fwd(F.L.ptr(X), F.L.ptr(offt), B, n, L, code, F.L.ptr(S), F.L.ptr(Sl), F.L.ptr(ws),
                                          ws.numel(), F.L.stream_ptr()), "segment_sum_fwd")
    bc = torch.empty_like(X)
    bcw = torch.empty_like(X)
    F.L.check(lib.milb200_bag_broadcast(F.L.ptr(dM), None, F.L.ptr(offt), B, n, L, code, F.L.ptr(bc), F.L.stream_ptr()),
              "bag_broadcast")
    F.L.check(lib.milb200_bag_broadcast(F.L.ptr(dM), F.L.ptr(w), F.L.ptr(offt), B, n, L, code, F.L.ptr(bcw),
                                        F.L.stream_ptr()), "bag_broadcast")
    torch.cuda.synchronize()
    return dict(M=M, M_lowp=Ml, argmax=am, lse=lse, ds=ds, ds_noattn=ds2, attn=attn, S=S, S_lowp=Sl, bc=bc, bcw=bcw)


@pytest.mark.parametrize("dtype,L,layout", POOL_CASES)
def test_pool_sum_and_broadcast_every_vector_width(F, dtype, L, layout):
    lens = _layout(layout)
    offt = _csr(lens)
    n, B = int(sum(lens)), len(lens)
    g = _gen(L * 3 + len(layout))
    X = torch.randn(n, L, device="cuda", generator=g).to(dtype)
    s = torch.randn(n, device="cuda", generator=g) * 2
    dM = torch.randn(B, L, device="cuda", generator=g)
    w = torch.randn(n, device="cuda", generator=g)
    got = _pool_all(F, X, s, offt, dM, w)
    tol = TOL[dtype]
    bag = _bag_of_row(offt)
    Xd = X.to(F64)
    Mr, a, lser = _pool_ref(Xd, s.to(F64), offt, bag)
    _close("M", got["M"], Mr, tol)
    if got["M_lowp"] is not None:
        _close("M_lowp", got["M_lowp"], Mr, tol)
    _close("lse", got["lse"], lser, tol)
    _check_argmax(got["argmax"], s, s.to(F64), offt, bag)
    dsr, ds_scale = _pool_bwd_ref(Xd, a, got["M"], dM, bag)   # got["M"]: the forward result the backward is handed
    _close_ds("ds", got["ds"], dsr, ds_scale, tol)
    assert torch.equal(got["ds"], got["ds_noattn"])
    _close("attn", got["attn"], a, tol)
    Sr = torch.zeros(B, L, dtype=F64, device="cuda").index_add_(0, bag, Xd)
    _close("segment sum", got["S"], Sr, tol)
    _close("segment sum (lowp)", got["S_lowp"], Sr, tol)
    bcr = dM.to(F64)[bag]
    _close("bag broadcast", got["bc"], bcr, tol)
    _close("weighted bag broadcast", got["bcw"], w.to(F64)[:, None] * bcr, tol)


def test_pool_tail_width_is_repeatable(F):
    lens = _layout("wide")
    offt = _csr(lens)
    n, B = int(sum(lens)), len(lens)
    g = _gen(17)
    X = torch.randn(n, 1000, device="cuda", generator=g).bfloat16()
    s = torch.randn(n, device="cuda", generator=g) * 2
    dM = torch.randn(B, 1000, device="cuda", generator=g)
    w = torch.randn(n, device="cuda", generator=g)
    a = _pool_all(F, X, s, offt, dM, w)
    b = _pool_all(F, X, s, offt, dM, w)
    for k in a:
        assert torch.equal(a[k], b[k]), k


@pytest.mark.parametrize("dtype,L", [(torch.bfloat16, 264), (torch.float32, 132)])
def test_pool_argmax_ties_pick_the_first_index_at_partial_lanes(F, dtype, L):
    """Scores drawn from {0, 1, 2}: almost every bag holds exact ties for its maximum, spread over slab boundaries."""
    lens = _layout("slabs") + _layout("mixed") + [3] * 50
    offt = _csr(lens)
    n = int(sum(lens))
    g = _gen(L)
    X = torch.randn(n, L, device="cuda", generator=g).to(dtype)
    s = torch.randint(0, 3, (n,), device="cuda", generator=g).float()
    M, _, am, lse = F.segment_softmax_pool(X, s, offt)
    torch.cuda.synchronize()
    bag = _bag_of_row(offt)
    want, _ = _first_argmax(s.to(F64), offt, bag)
    assert torch.equal(am.long(), want)
    Mr, _, lser = _pool_ref(X.to(F64), s.to(F64), offt, bag)
    _close("M", M, Mr, TOL[dtype])
    _close("lse", lse, lser, TOL[dtype])


@pytest.mark.parametrize("dtype,L", [(torch.bfloat16, 4104), (torch.float32, 2052)])
def test_pool_rejects_rows_past_the_widest_instantiation(F, dtype, L):
    offt = _csr([3, 5])
    X = torch.randn(8, L, device="cuda").to(dtype)
    s = torch.randn(8, device="cuda")
    dM = torch.randn(2, L, device="cuda")
    M = torch.randn(2, L, device="cuda")
    lib = F.L.lib()
    ws = F.L.workspace(lib.milb200_pool_workspace_bytes(8, 2, L), X.device)
    S = torch.empty(2, L, device="cuda")
    torch.cuda.synchronize()
    _expect_rejected(F, lambda: F.segment_softmax_pool(X, s, offt))
    _expect_rejected(F, lambda: F.segment_softmax_pool_bwd(X, s, offt, dM, M, want_attn=True))
    _expect_rejected(F, lambda: F.L.check(lib.milb200_segment_sum_fwd(
        F.L.ptr(X), F.L.ptr(offt), 2, 8, L, F.L.dtype_code(X), F.L.ptr(S), None, F.L.ptr(ws), ws.numel(),
        F.L.stream_ptr()), "segment_sum_fwd"))


# ---------------------------------------------------------------------------------------------------------------------
# C. dense linear layer against float64
# ---------------------------------------------------------------------------------------------------------------------
def _bias(kind, n, g):
    if kind is None:
        return None
    if kind == "offset":         # a slice 4 bytes into a larger buffer: not 16-byte aligned (scalar bias loads)
        return (torch.randn(n + 1, device="cuda", generator=g) * 0.1)[1:]
    return torch.randn(n, device="cuda", generator=g) * 0.1


def _act64(act, pre, y_kernel):
    """Forward activation in float64; for ReLU the active set is the kernel's own (a pre-activation within rounding of
    zero may land on either side)."""
    if act == "relu":
        return pre * (y_kernel > 0).to(F64)
    if act == "tanh":
        return torch.tanh(pre)
    if act == "sigmoid":
        return torch.sigmoid(pre)
    return pre


def _dact64(act, y_kernel):
    """d act / d pre as the backward defines it: a function of the forward output Y the caller hands back."""
    y = y_kernel.to(F64)
    if act == "relu":
        return (y > 0).to(F64)
    if act == "tanh":
        return 1 - y * y
    if act == "sigmoid":
        return y * (1 - y)
    return torch.ones_like(y)


def _linear_check(F, dtype, m, n, k, act, use_add, bias, seed, tol=None):
    g = _gen(seed)
    x = torch.randn(m, k, device="cuda", generator=g).to(dtype).requires_grad_(True)
    add = torch.randn(m, k, device="cuda", generator=g).to(dtype).requires_grad_(True) if use_add else None
    W = (torch.randn(n, k, device="cuda", generator=g) / math.sqrt(k)).requires_grad_(True)
    b = _bias(bias, n, g)
    if b is not None:
        b.requires_grad_(True)
    dy = torch.randn(m, n, device="cuda", generator=g).to(dtype)
    y = F.linear(x, W, b, act=act, add=add)
    y.backward(dy)
    torch.cuda.synchronize()
    tol = tol or TOL[dtype]
    xin = x.detach().to(F64)
    if use_add:
        # the small-m kernel adds in fp32 registers; the other paths stage X + add in the workspace in the input dtype
        xsum = x.detach().float() + add.detach().float()
        xin = (xsum if m <= 16 else xsum.to(dtype)).to(F64)
    Wd = W.detach().to(dtype).to(F64)
    pre = xin @ Wd.t() + (b.detach().to(F64) if b is not None else 0)
    _close("Y", y, _act64(act, pre, y.detach()), tol)
    dpre = dy.to(F64) * _dact64(act, y.detach())
    dX = dpre @ Wd
    _close("dX", x.grad, dX, tol)
    if use_add:
        _close("d add", add.grad, dX, tol)
    _close("dW", W.grad, dpre.t() @ xin, tol)
    if b is not None:
        _close("dbias", b.grad, dpre.sum(0), tol)
    return y.detach(), x.grad, W.grad


# Pairwise grid: every m / n / k / act / add value and each bias variant, each next to a tail on another axis.
#   m: 17..33 take the direct stores (no TMA store below 32 rows), 128 x 148 + 1 is a full wave of tiles plus one row;
#   n: 16 / 48 / 144 / 272 / 1040 / 2064 leave a partial 128- or 256-column tile, 1040 and 2064 are past the 1024-float
#      bias cache; k: 72 / 200 / 520 end in a partial 64-wide K block.
LINEAR_CASES = [  # m, n, k, act, add, bias
    (17, 2064, 72, "sigmoid", False, "vec"),
    (31, 16, 2048, None, True, None),
    (32, 272, 64, "relu", False, "offset"),
    (33, 144, 520, "tanh", True, "vec"),
    (127, 1040, 200, None, False, "offset"),
    (129, 48, 64, "relu", True, "vec"),
    (1000, 256, 72, "sigmoid", True, None),
    (128 * 148 + 1, 128, 200, "tanh", False, "vec"),
    (1000, 272, 2048, "relu", False, "vec"),
    (128 * 148 + 1, 2064, 520, None, True, "offset"),
    (33, 1040, 64, "sigmoid", False, None),
    (129, 128, 72, None, False, "vec"),
]


@pytest.mark.parametrize("m,n,k,act,use_add,bias", LINEAR_CASES)
def test_bf16_linear_vs_float64(F, m, n, k, act, use_add, bias):
    _linear_check(F, torch.bfloat16, m, n, k, act, use_add, bias, seed=m + 3 * n + 7 * k)


def test_bf16_linear_tail_shape_is_repeatable(F):
    a = _linear_check(F, torch.bfloat16, 129, 1040, 72, "tanh", True, "offset", seed=3)
    b = _linear_check(F, torch.bfloat16, 129, 1040, 72, "tanh", True, "offset", seed=3)
    for x, y in zip(a, b):
        assert torch.equal(x, y)


# Both sides of every routing boundary, in both dtypes: m = 16 | 17 (small-m kernel | tensor cores / FFMA), n = 16 | 24
# and k = 56 | 64 (tensor cores | FFMA), n = 48 (tensor-core forward, FFMA backward), fp32 m = 4095 | 4096 (FFMA |
# 3xTF32).
ROUTE_CASES = [(dt, m, n, k) for dt in (torch.float32, torch.bfloat16)
               for (m, n, k) in ((16, 128, 64), (17, 128, 64), (1000, 16, 64), (1000, 24, 64), (1000, 128, 56),
                                 (1000, 128, 64), (1000, 48, 200))] + \
              [(torch.float32, 4095, 128, 64), (torch.float32, 4096, 128, 64)]


@pytest.mark.parametrize("dtype,m,n,k", ROUTE_CASES)
def test_linear_routing_boundaries_vs_float64(F, dtype, m, n, k):
    _linear_check(F, dtype, m, n, k, "tanh", True, "vec", seed=m * 5 + n + k)


def _raw_linear_bwd(F, x, W, Y, dY, dX, dW, db, act, accumulate):
    lib = F.L.lib()
    m, k = x.shape
    n = W.shape[0]
    code = F.L.dtype_code(x)
    ws = F.L.workspace(lib.milb200_linear_workspace_bytes(m, n, k, code, 1), x.device)
    F.L.check(lib.milb200_linear_bwd(F.L.ptr(x), None, F.L.ptr(W), F.L.ptr(Y), F.L.ptr(dY), F.L.ptr(dX), F.L.ptr(dW),
                                     F.L.ptr(db), m, n, k, act, code, accumulate, F.L.ptr(ws), ws.numel(),
                                     F.L.stream_ptr()), "linear_bwd")


@pytest.mark.parametrize("dtype,m,n,k", [(torch.bfloat16, 1000, 272, 200), (torch.bfloat16, 16, 128, 64),
                                         (torch.bfloat16, 1000, 48, 200), (torch.float32, 16, 128, 64),
                                         (torch.float32, 1000, 272, 200), (torch.float32, 4096, 128, 64)])
def test_linear_bwd_accumulates_and_allows_no_bias_gradient(F, dtype, m, n, k):
    """milb200_linear_bwd with accumulate = 1 adds dW / dbias to what the buffers hold; dbias = NULL and dX = NULL skip
    those outputs without disturbing dW."""
    g = _gen(m + n + k)
    x = torch.randn(m, k, device="cuda", generator=g).to(dtype)
    W = (torch.randn(n, k, device="cuda", generator=g) / math.sqrt(k)).to(dtype)
    Y = torch.tanh(x.float() @ W.float().t()).to(dtype)       # any forward output: the backward only reads it
    dY = torch.randn(m, n, device="cuda", generator=g).to(dtype)
    dW0 = torch.randn(n, k, device="cuda", generator=g)
    db0 = torch.randn(n, device="cuda", generator=g)
    dX = torch.empty_like(x)
    dW, db = dW0.clone(), db0.clone()
    _raw_linear_bwd(F, x, W, Y, dY, dX, dW, db, F.L.ACT_TANH, 1)
    dW2 = dW0.clone()
    _raw_linear_bwd(F, x, W, Y, dY, None, dW2, None, F.L.ACT_TANH, 1)
    torch.cuda.synchronize()
    dpre = dY.to(F64) * _dact64("tanh", Y)
    dWr = dpre.t() @ x.to(F64)
    tol = TOL[dtype]
    assert float((dW.to(F64) - dW0.to(F64) - dWr).abs().max()) <= tol * float(dWr.abs().max())
    assert float((db.to(F64) - db0.to(F64) - dpre.sum(0)).abs().max()) <= tol * float(dpre.sum(0).abs().max())
    assert float((dW2.to(F64) - dW0.to(F64) - dWr).abs().max()) <= tol * float(dWr.abs().max())
    _close("dX", dX, dpre @ W.to(F64), tol)


@pytest.mark.parametrize("m,n,k,act", [(33, 272, 80, "relu"), (1000, 144, 528, None), (129, 1040, 64, "tanh"),
                                       (17, 2064, 208, "sigmoid"), (31, 48, 72, "tanh")])
def test_linear_f32out_vs_float64(F, m, n, k, act):
    """The mixed linear of the fusion path's key stream: bf16 operands on the tensor cores, fp32 result and gradients.
    The backward needs n >= 64 and k % 16 == 0 (its dX GEMM has N = k): other shapes get the forward only and a refused
    backward."""
    lib = F.L.lib()
    g = _gen(m + n)
    x = torch.randn(m, k, device="cuda", generator=g).bfloat16()
    W = (torch.randn(n, k, device="cuda", generator=g) / math.sqrt(k)).bfloat16()
    b = _bias("offset" if n > 1024 else "vec", n, g)
    a = F._ACT[act]
    Y = torch.empty(m, n, device="cuda")
    F.L.check(lib.milb200_linear_f32out_fwd(F.L.ptr(x), F.L.ptr(W), F.L.ptr(b), F.L.ptr(Y), m, n, k, a, F.L.stream_ptr()),
              "linear_f32out_fwd")
    dY = torch.randn(m, n, device="cuda", generator=g)
    dX = torch.empty_like(x)
    dW = torch.empty(n, k, device="cuda")
    db = torch.empty(n, device="cuda")
    ws = F.L.workspace(lib.milb200_linear_workspace_bytes(m, n, k, F.L.BF16, 1), x.device)
    torch.cuda.synchronize()
    xd, Wd = x.to(F64), W.to(F64)
    tol = TOL[torch.bfloat16]
    _close("Y", Y, _act64(act, xd @ Wd.t() + b.to(F64), Y), tol)

    def bwd():
        F.L.check(lib.milb200_linear_f32out_bwd(F.L.ptr(x), F.L.ptr(W), F.L.ptr(Y), F.L.ptr(dY), F.L.ptr(dX), F.L.ptr(dW),
                                                F.L.ptr(db), m, n, k, a, 0, F.L.ptr(ws), ws.numel(), F.L.stream_ptr()),
                  "linear_f32out_bwd")
    if n < 64 or k % 16:
        _expect_rejected(F, bwd)
        return
    bwd()
    torch.cuda.synchronize()
    dpre = dY.to(F64) * _dact64(act, Y)
    _close("dX", dX, dpre @ Wd, tol)
    _close("dW", dW, dpre.t() @ xd, tol)
    _close("dbias", db, dpre.sum(0), tol)


# ---------------------------------------------------------------------------------------------------------------------
# D. LayerNorm with a broadcast residual row, column sums, LayerNorm width limit, attention head-dim limit
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("m,n", [(1, 512), (37, 200), (5000, 1024)])
def test_layernorm_broadcast_residual_row_vs_float64(F, dtype, m, n):
    """Y = LN(X + r) with one residual row r for every row of X (r_broadcast = 1); dgamma / dbeta overwritten, then added
    to (accumulate = 1); the gradient of r is the column sum of dXR (milb200_colsum, overwritten and added to)."""
    lib = F.L.lib()
    code = F.L.dtype_code(torch.empty(0, dtype=dtype))
    g = _gen(m + n)
    x = torch.randn(m, n, device="cuda", generator=g).to(dtype)
    r = torch.randn(n, device="cuda", generator=g).to(dtype)
    ga = torch.rand(n, device="cuda", generator=g) + 0.5
    be = torch.randn(n, device="cuda", generator=g)
    dy = torch.randn(m, n, device="cuda", generator=g).to(dtype)
    y = torch.empty_like(x)
    mean = torch.empty(m, device="cuda")
    rstd = torch.empty(m, device="cuda")
    st = F.L.stream_ptr()
    F.L.check(lib.milb200_layernorm_fwd(F.L.ptr(x), F.L.ptr(r), F.L.ptr(ga), F.L.ptr(be), F.L.ptr(y), F.L.ptr(mean),
                                        F.L.ptr(rstd), m, n, code, 1, st), "layernorm_fwd")
    dxr = torch.empty_like(x)
    dg, db = torch.empty(n, device="cuda"), torch.empty(n, device="cuda")
    ws = F.L.workspace(lib.milb200_layernorm_workspace_bytes(m, n), x.device)

    def bwd(acc):
        F.L.check(lib.milb200_layernorm_bwd(F.L.ptr(x), F.L.ptr(r), F.L.ptr(ga), F.L.ptr(mean), F.L.ptr(rstd), F.L.ptr(dy),
                                            F.L.ptr(dxr), F.L.ptr(dg), F.L.ptr(db), m, n, code, acc, 1, F.L.ptr(ws),
                                            ws.numel(), st), "layernorm_bwd")
    bwd(0)
    dg1, db1 = dg.clone(), db.clone()
    bwd(1)
    dr = torch.empty(n, device="cuda")
    F.L.check(lib.milb200_colsum(F.L.ptr(dxr), m, n, F.L.ptr(dr), code, 0, st), "colsum")
    dr1 = dr.clone()
    F.L.check(lib.milb200_colsum(F.L.ptr(dxr), m, n, F.L.ptr(dr), code, 1, st), "colsum")
    torch.cuda.synchronize()
    xd = x.to(F64).requires_grad_(True)
    rd = r.to(F64).requires_grad_(True)
    gd, bd = ga.to(F64).requires_grad_(True), be.to(F64).requires_grad_(True)
    yr = torch.nn.functional.layer_norm(xd + rd[None, :], (n,), gd, bd, 1e-5)
    (yr * dy.to(F64)).sum().backward()
    tol = TOL[dtype]
    _close("Y", y, yr, tol)
    _close("mean", mean, (xd + rd).mean(1), tol)
    _close("dXR", dxr, xd.grad, tol)
    _close("dgamma", dg1, gd.grad, max(tol, 1e-5))
    _close("dbeta", db1, bd.grad, max(tol, 1e-5))
    _close("dgamma (accumulated)", dg, 2 * gd.grad, max(tol, 1e-5))
    _close("dbeta (accumulated)", db, 2 * bd.grad, max(tol, 1e-5))
    # dr sums the kernel's own dXR: compare with the float64 column sum of that matrix (and with the true gradient)
    _close("colsum", dr1, dxr.to(F64).sum(0), 1e-5)
    _close("colsum (accumulated)", dr, 2 * dxr.to(F64).sum(0), 1e-5)
    _close("d r", dr1, rd.grad, tol)


@pytest.mark.parametrize("dtype,rows,cols,offset", [(torch.float32, 1, 4, 0), (torch.float32, 5000, 1030, 1),
                                                    (torch.float32, 33, 2064, 0), (torch.bfloat16, 37, 200, 0),
                                                    (torch.bfloat16, 20000, 1031, 0), (torch.bfloat16, 3, 1024, 3)])
def test_colsum_vs_float64(F, dtype, rows, cols, offset):
    """out[c] (+)= sum_r A[r, c]: the vectorised kernel (cols a multiple of the 16-byte vector, aligned) and the scalar one
    (odd widths, a matrix starting off a 16-byte boundary)."""
    lib = F.L.lib()
    g = _gen(rows + cols)
    A = torch.randn(rows * cols + offset, device="cuda", generator=g).to(dtype)[offset:]
    out0 = torch.randn(cols, device="cuda", generator=g)
    out = torch.empty(cols, device="cuda")
    code = F.L.dtype_code(A)
    F.L.check(lib.milb200_colsum(C.c_void_p(A.data_ptr()), rows, cols, F.L.ptr(out), code, 0, F.L.stream_ptr()), "colsum")
    acc = out0.clone()
    F.L.check(lib.milb200_colsum(C.c_void_p(A.data_ptr()), rows, cols, F.L.ptr(acc), code, 1, F.L.stream_ptr()), "colsum")
    torch.cuda.synchronize()
    want = A.to(F64).view(rows, cols).sum(0)
    _close("colsum", out, want, 1e-5)
    assert float((acc.to(F64) - out0.to(F64) - want).abs().max()) <= 1e-5 * float(want.abs().max()) + 1e-6


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_layernorm_rejects_rows_wider_than_1024(F, dtype):
    lib = F.L.lib()
    m, n = 4, 1032
    code = F.L.dtype_code(torch.empty(0, dtype=dtype))
    x = torch.randn(m, n, device="cuda").to(dtype)
    ga, be = torch.ones(n, device="cuda"), torch.zeros(n, device="cuda")
    y, dxr = torch.empty_like(x), torch.empty_like(x)
    mean, rstd = torch.zeros(m, device="cuda"), torch.ones(m, device="cuda")
    dg, db = torch.empty(n, device="cuda"), torch.empty(n, device="cuda")
    ws = F.L.workspace(lib.milb200_layernorm_workspace_bytes(m, n), x.device)
    torch.cuda.synchronize()
    _expect_rejected(F, lambda: F.layernorm(x, ga, be))
    _expect_rejected(F, lambda: F.L.check(lib.milb200_layernorm_bwd(
        F.L.ptr(x), None, F.L.ptr(ga), F.L.ptr(mean), F.L.ptr(rstd), F.L.ptr(x), F.L.ptr(dxr), F.L.ptr(dg), F.L.ptr(db),
        m, n, code, 0, 0, F.L.ptr(ws), ws.numel(), F.L.stream_ptr()), "layernorm_bwd"))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_attention_rejects_many_keys_with_head_dim_64(F, dtype):
    """Many-key attention (more than 16 keys) is built for head dim 32 only: forward and backward must refuse c = 64."""
    lib = F.L.lib()
    nq, nk, H, c = 4, 100, 2, 64
    code = F.L.dtype_code(torch.empty(0, dtype=dtype))
    q = torch.randn(nq, H * c, device="cuda").to(dtype)
    k = torch.randn(nk, H * c, device="cuda").to(dtype)
    v = torch.randn(nk, H * c, device="cuda").to(dtype)
    o, do, dq = torch.zeros_like(q), torch.randn_like(q), torch.empty_like(q)
    dk, dv = torch.empty_like(k), torch.empty_like(v)
    lse = torch.zeros(H, nq, device="cuda")
    ws = F.L.workspace(lib.milb200_attention_workspace_bytes(nq, nk, H, c, 1), q.device)
    torch.cuda.synchronize()
    _expect_rejected(F, lambda: F.attention_core(q, k, v, H))
    _expect_rejected(F, lambda: F.L.check(lib.milb200_attention_bwd(
        F.L.ptr(q), F.L.ptr(k), F.L.ptr(v), F.L.ptr(o), F.L.ptr(lse), F.L.ptr(do), F.L.ptr(dq), F.L.ptr(dk), F.L.ptr(dv),
        nq, nk, H, c, code, F.L.ptr(ws), ws.numel(), F.L.stream_ptr()), "attention_bwd"))
