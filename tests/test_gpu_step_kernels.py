"""GPU tests of the kernels that close each training step, each against a float64 reference evaluated on the operands
the kernel saw (bf16 inputs quantised, fp32 hyperparameters rounded to fp32), at the shapes and values where they can go
wrong:

  A. the optimisers: Adam (eager and graphed), the step counter and SGD, over the grid-stride tail, weight decay,
     grad_scale, eps-dominated and exactly zero gradients, and late steps;
  B. the CLIP cosine logits and their backward at d tails, one- and many-row sides, every omitted output;
  C. CLIPloss_v1 past one CTA's reductions, with logits large enough to need the max subtraction, and at the edge of its
     shared memory;
  D. the cosine embedding loss (zero rows, parallel and antiparallel rows) and sigmoid + BCE over the whole fp32 range;
  E. the elementwise glue: dropout (its mask against a host Philox4x32-10, on the vector and scalar paths), cast,
     axpby / add, transpose, the sinusoid table and the CT token mean;
  F. the launch counter against the kernels the profiler sees, for every entry point above.

Tolerances as in the rest of the suite, max-norm relative: fp32 1e-5, bf16 1e-2.  Where a quantity is a difference of
larger terms, the bound is taken relative to those terms, and the comment at the check says why.  The C ABI is called
directly where the Python wrapper hides an argument (NULL outputs, offset, grad_scale, the device step counter)."""
import json
import math

import numpy as np
import pytest
import torch

from oracle import fusion_oracle as fo
from oracle import mil_oracle as mo

pytestmark = pytest.mark.gpu

TOL = {torch.float32: 1e-5, torch.bfloat16: 1e-2}
F64, F32, BF16 = torch.float64, torch.float32, torch.bfloat16
DTYPES = [F32, BF16]
U32 = 2.0 ** -24          # unit roundoff of fp32


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


def _close_scaled(name, got, want, scale, tol):
    got = got.detach().to(F64)
    e = float((got - want.to(F64).to(got.device)).abs().max()) / max(float(scale), 1e-30)
    assert e <= tol, f"{name}: error {e:.3e} of the term scale > {tol:g}"


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _expect_rejected(F, fn):
    """fn must raise MilB200Error and launch no kernel."""
    n0 = F.L.launch_count()
    with pytest.raises(F.L.MilB200Error):
        fn()
    torch.cuda.synchronize()
    assert F.L.launch_count() == n0, "a call whose argument check failed launched a kernel"


def _f32(x):
    return float(np.float32(x))


def _misaligned(t):
    """A copy of 1-D t that starts one element past a 16-byte boundary (the scalar paths of the vector kernels)."""
    buf = torch.empty(t.numel() + 8, dtype=t.dtype, device=t.device)
    out = buf[1:1 + t.numel()]
    out.copy_(t)
    return out


# ---------------------------------------------------------------------------------------------------------------------
# A. optimisers
# ---------------------------------------------------------------------------------------------------------------------
ADAM_N = [1, 3, 255, 257, 303104, 303105, 1000003]     # 148 * 8 * 256 = 303104: one pass of the capped grid
B1, B2, EPS = 0.9, 0.999, 1e-8
# name: (lr, weight decay, grad_scale, gradients)
ADAM_HP = {
    "defaults": (1e-5, 1e-7, 1.0, "normal"),          # mo.adam_step's defaults (train_ddp.py's Adam)
    "wd": (1e-3, 1e-2, 1.0, "normal"),
    "gscale": (1e-3, 0.0, 0.125, "normal"),
    "wd_gscale": (1e-3, 1e-2, 0.125, "normal"),
    "tiny": (1e-3, 0.0, 1.0, "tiny"),                 # |g| in [1e-9, 1e-6]: eps decides the step
    "zeros": (1e-3, 0.0, 0.125, "zeros"),             # every third gradient exactly 0
}


def _adam64(p, g, m, v, step, lr, wd, gs, b1=B1, b2=B2, eps=EPS):
    """mo.adam_step restated on device tensors, applied to grad * grad_scale, with the hyperparameters as the fp32 values
    the kernel receives (pinned to mo.adam_step by test_adam_reference_is_the_oracle)."""
    lr, wd, gs, b1, b2, eps = map(_f32, (lr, wd, gs, b1, b2, eps))
    p, g, m, v = (t.to(F64) for t in (p, g, m, v))
    g = g * gs + wd * p
    m = b1 * m + (1 - b1) * g
    v = b2 * v + (1 - b2) * g * g
    mhat = m / (1 - b1 ** step)
    vhat = v / (1 - b2 ** step)
    return p - lr * mhat / (vhat.sqrt() + eps), m, v


def test_adam_reference_is_the_oracle():
    rs = np.random.RandomState(0)
    p, g, m, v = rs.randn(4, 50)
    v = np.abs(v)
    for step in (1, 7):
        want = mo.adam_step(p, g * _f32(0.125), m, v, step, lr=_f32(1e-3), b1=_f32(B1), b2=_f32(B2), eps=_f32(EPS),
                            wd=_f32(1e-2))
        got = _adam64(*(torch.from_numpy(a) for a in (p, g, m, v)), step, 1e-3, 1e-2, 0.125)
        for w, x in zip(want, got):
            np.testing.assert_allclose(x.numpy(), w, rtol=1e-14, atol=0)


def _grads(kind, n, g):
    x = torch.randn(n, device="cuda", generator=g)
    if kind == "tiny":
        mag = 10.0 ** (-9 + 3 * torch.rand(n, device="cuda", generator=g))
        x = torch.where(x < 0, -mag, mag)
    elif kind == "zeros":
        x[::3] = 0.0
    return x


def _adam_call(F, p, g, m, v, step, lr, wd, gs):
    L = F.L
    L.check(L.lib().milb200_adam_step(L.ptr(p), L.ptr(g), L.ptr(m), L.ptr(v), p.numel(), lr, B1, B2, EPS, wd, gs, step,
                                      L.stream_ptr()), "adam_step")


def _check_update(name, p_new, p0, want_p):
    """The update p - p0 on its own.  The kernel stores fl(p0 - u): besides u's own error (relative, 1e-5) the stored
    parameter carries one rounding, at most 2^-24 |p|, which is absolute for u."""
    du, du_ref = p_new.to(F64) - p0.to(F64), want_p - p0.to(F64)
    err = float((du - du_ref).abs().max())
    bound = 1e-5 * float(du_ref.abs().max()) + U32 * float(p_new.abs().max())
    assert err <= bound, f"{name}: update error {err:.3e} > {bound:.3e}"


@pytest.mark.parametrize("n", ADAM_N)
@pytest.mark.parametrize("hp", list(ADAM_HP))
def test_adam_step_vs_float64(F, hp, n):
    lr, wd, gs, kind = ADAM_HP[hp]
    g = _gen(1000 + n + len(hp))
    p = torch.randn(n, device="cuda", generator=g) * 0.05
    m = torch.zeros(n, device="cuda")
    v = torch.zeros(n, device="cuda")
    zero_rows = None
    for step in (1, 2, 3):
        grad = _grads(kind, n, g)
        p0, m0, v0 = p.clone(), m.clone(), v.clone()
        want_p, want_m, want_v = _adam64(p0, grad, m0, v0, step, lr, wd, gs)
        _adam_call(F, p, grad, m, v, step, lr, wd, gs)
        _close(f"{hp} n={n} step {step} exp_avg", m, want_m, 1e-5)
        _close(f"{hp} n={n} step {step} exp_avg_sq", v, want_v, 1e-5)
        _close(f"{hp} n={n} step {step} param", p, want_p, 1e-5)
        _check_update(f"{hp} n={n} step {step}", p, p0, want_p)
        if kind == "zeros":
            zero_rows = torch.arange(0, n, 3, device="cuda")
            # with no weight decay a zero gradient from a zero state must leave everything exactly as it was
            assert torch.equal(p[zero_rows], p0[zero_rows]) and not m[zero_rows].any() and not v[zero_rows].any()
    for step in (1000, 100000):
        grad = _grads(kind, n, g)
        scale = 1e-7 if kind == "tiny" else 0.1
        m = torch.randn(n, device="cuda", generator=g) * scale
        v = torch.rand(n, device="cuda", generator=g) * scale * scale
        p0, m0, v0 = p.clone(), m.clone(), v.clone()
        want_p, want_m, want_v = _adam64(p0, grad, m0, v0, step, lr, wd, gs)
        _adam_call(F, p, grad, m, v, step, lr, wd, gs)
        _close(f"{hp} n={n} step {step} exp_avg", m, want_m, 1e-5)
        _close(f"{hp} n={n} step {step} exp_avg_sq", v, want_v, 1e-5)
        _close(f"{hp} n={n} step {step} param", p, want_p, 1e-5)
        _check_update(f"{hp} n={n} step {step}", p, p0, want_p)


@pytest.mark.parametrize("s", [1, 2, 3, 10, 1000, 100000])
def test_adam_step_dev_equals_eager(F, s):
    """The graphed update (step number in device memory, advanced by step_counter_inc) is bit-identical to the eager one."""
    L = F.L
    n = 303105
    g = _gen(77 + s)
    p = torch.randn(n, device="cuda", generator=g) * 0.05
    grad = torch.randn(n, device="cuda", generator=g)
    m = torch.randn(n, device="cuda", generator=g) * 0.1
    v = torch.rand(n, device="cuda", generator=g) * 0.01
    pe, me, ve = p.clone(), m.clone(), v.clone()
    _adam_call(F, pe, grad, me, ve, s, 1e-3, 1e-2, 0.125)
    ctr = torch.tensor([s - 1], dtype=torch.int32, device="cuda")
    L.check(L.lib().milb200_step_counter_inc(L.ptr(ctr), L.stream_ptr()), "step_counter_inc")
    L.check(L.lib().milb200_adam_step_dev(L.ptr(p), L.ptr(grad), L.ptr(m), L.ptr(v), n, 1e-3, B1, B2, EPS, 1e-2, 0.125,
                                          L.ptr(ctr), L.stream_ptr()), "adam_step_dev")
    assert int(ctr.item()) == s
    assert torch.equal(p, pe) and torch.equal(m, me) and torch.equal(v, ve), f"adam_step_dev differs from adam_step at {s}"


def test_step_counter_inc(F):
    L = F.L
    ctr = torch.tensor([0, 12345], dtype=torch.int32, device="cuda")
    for _ in range(3):
        L.check(L.lib().milb200_step_counter_inc(L.ptr(ctr), L.stream_ptr()), "step_counter_inc")
    assert ctr.tolist() == [3, 12345]


@pytest.mark.parametrize("n", ADAM_N)
@pytest.mark.parametrize("wd,gs", [(0.0, 1.0), (1e-2, 0.125)])
def test_sgd_step_vs_float64(F, n, wd, gs):
    L = F.L
    g = _gen(500 + n)
    p = torch.randn(n, device="cuda", generator=g) * 0.05
    grad = torch.randn(n, device="cuda", generator=g)
    grad[::5] = 0.0
    p0 = p.clone()
    want = torch.from_numpy(mo.sgd_step(p0.cpu().numpy(), (grad.to(F64) * _f32(gs)).cpu().numpy(), lr=_f32(1e-3),
                                        wd=_f32(wd))).cuda()
    L.check(L.lib().milb200_sgd_step(L.ptr(p), L.ptr(grad), n, 1e-3, wd, gs, L.stream_ptr()), "sgd_step")
    _close(f"sgd n={n}", p, want, 1e-5)
    _check_update(f"sgd n={n}", p, p0, want)


def test_optimizer_refusals(F):
    L = F.L
    lib, S = L.lib(), L.stream_ptr()
    t = [torch.zeros(8, device="cuda") for _ in range(4)]
    P = [L.ptr(x) for x in t]
    ctr = torch.ones(1, dtype=torch.int32, device="cuda")

    def adam(p, g, m, v, n, step):
        return lambda: L.check(lib.milb200_adam_step(p, g, m, v, n, 1e-3, B1, B2, EPS, 0.0, 1.0, step, S), "adam")

    def adam_dev(p, g, m, v, n, c):
        return lambda: L.check(lib.milb200_adam_step_dev(p, g, m, v, n, 1e-3, B1, B2, EPS, 0.0, 1.0, c, S), "adam_dev")

    _expect_rejected(F, adam(*P, 8, 0))
    _expect_rejected(F, adam(*P, -1, 1))
    for k in range(4):
        q = list(P)
        q[k] = None
        _expect_rejected(F, adam(*q, 8, 1))
        _expect_rejected(F, adam_dev(*q, 8, L.ptr(ctr)))
    _expect_rejected(F, adam_dev(*P, 8, None))
    _expect_rejected(F, adam_dev(*P, -1, L.ptr(ctr)))
    _expect_rejected(F, lambda: L.check(lib.milb200_sgd_step(None, P[1], 8, 1e-3, 0.0, 1.0, S), "sgd"))
    _expect_rejected(F, lambda: L.check(lib.milb200_sgd_step(P[0], None, 8, 1e-3, 0.0, 1.0, S), "sgd"))
    _expect_rejected(F, lambda: L.check(lib.milb200_sgd_step(P[0], P[1], -1, 1e-3, 0.0, 1.0, S), "sgd"))
    _expect_rejected(F, lambda: L.check(lib.milb200_step_counter_inc(None, S), "step_counter_inc"))
    n0 = L.launch_count()
    assert lib.milb200_adam_step(*P, 0, 1e-3, B1, B2, EPS, 0.0, 1.0, 1, S) == 0
    assert lib.milb200_adam_step_dev(*P, 0, 1e-3, B1, B2, EPS, 0.0, 1.0, L.ptr(ctr), S) == 0
    assert lib.milb200_sgd_step(P[0], P[1], 0, 1e-3, 0.0, 1.0, S) == 0
    torch.cuda.synchronize()
    assert L.launch_count() == n0, "an empty optimiser step launched a kernel"


# ---------------------------------------------------------------------------------------------------------------------
# B. CLIP cosine logits
# ---------------------------------------------------------------------------------------------------------------------
CLIP_SHAPES = [(1, 1), (1, 24), (24, 1), (7, 300), (300, 7), (129, 65)]
CLIP_D = [1, 31, 32, 33, 255, 256, 257, 512, 1000, 1024]
CLIP_LS = [0.0, math.log(1 / 0.07), math.log(100.0)]
# pairwise: every (shape, d) pair; logit_scale cycles so that every (shape, scale) and (d, scale) pair occurs too
CLIP_CASES = [(s, d, CLIP_LS[(i + j) % 3]) for i, s in enumerate(CLIP_SHAPES) for j, d in enumerate(CLIP_D)]
SENTINEL = 1234.5


def _clip_fwd(F, I, T, ls):
    L = F.L
    bi, d = I.shape
    bt = T.shape[0]
    li = torch.empty(bi, bt, device="cuda")
    ni, nt = torch.empty(bi, device="cuda"), torch.empty(bt, device="cuda")
    L.check(L.lib().milb200_clip_logits_fwd(L.ptr(I), L.ptr(T), L.ptr(ls), L.ptr(li), L.ptr(ni), L.ptr(nt), bi, bt, d,
                                            L.dtype_code(I), L.stream_ptr()), "clip_logits_fwd")
    return li, ni, nt


def _clip_bwd(F, I, T, ls, li, ni, nt, dli, dlt, want):
    """want: subset of {"dI", "dT", "ds"}; omitted outputs are sentinel-filled buffers the call does not receive."""
    L = F.L
    bi, d = I.shape
    bt = T.shape[0]
    out = {"dI": torch.full_like(I, SENTINEL), "dT": torch.full_like(T, SENTINEL),
           "ds": torch.full((1,), SENTINEL, device="cuda")}
    arg = {k: (L.ptr(v) if k in want else None) for k, v in out.items()}
    L.check(L.lib().milb200_clip_logits_bwd(L.ptr(I), L.ptr(T), L.ptr(ls), L.ptr(li), L.ptr(ni), L.ptr(nt), L.ptr(dli),
                                            L.ptr(dlt), arg["dI"], arg["dT"], arg["ds"], bi, bt, d, L.dtype_code(I),
                                            L.stream_ptr()), "clip_logits_bwd")
    for k, v in out.items():
        if k not in want:
            assert bool((v == SENTINEL).all()), f"clip_logits_bwd wrote the omitted output {k}"
    return out


@pytest.mark.parametrize("shape,d,ls", CLIP_CASES)
@pytest.mark.parametrize("dt", DTYPES)
def test_clip_logits_vs_float64(F, dt, shape, d, ls):
    bi, bt = shape
    tol = TOL[dt]
    g = _gen(bi * 7919 + bt * 31 + d)
    I = torch.randn(bi, d, device="cuda", generator=g).to(dt)
    T = torch.randn(bt, d, device="cuda", generator=g).to(dt)
    lsv = torch.tensor([ls], dtype=F32, device="cuda")
    li, ni, nt = _clip_fwd(F, I, T, lsv)
    Id, Td = I.to(F64).cpu().numpy(), T.to(F64).cpu().numpy()
    lsf = float(lsv.item())
    li_ref, _ = mo.clip_cosine_logits(Id, Td, lsf)
    _close("logits", li, torch.from_numpy(li_ref), tol)
    _close("inv_norm_i", ni, torch.from_numpy(1 / np.linalg.norm(Id, axis=1)), tol)
    _close("inv_norm_t", nt, torch.from_numpy(1 / np.linalg.norm(Td, axis=1)), tol)

    dli = torch.randn(bi, bt, device="cuda", generator=g)
    dlt = torch.randn(bt, bi, device="cuda", generator=g)
    sc = math.exp(lsf)
    ih, th = Id / np.linalg.norm(Id, axis=1, keepdims=True), Td / np.linalg.norm(Td, axis=1, keepdims=True)
    for tag, a, b in (("image side", dli, None), ("text side", None, dlt), ("both", dli, dlt)):
        G = (a.to(F64).cpu().numpy() if a is not None else 0) + (b.to(F64).cpu().numpy().T if b is not None else 0)
        G = np.broadcast_to(G, (bi, bt))
        dI_ref, dT_ref, ds_ref = mo.clip_cosine_logits_bwd(Id, Td, lsf, G, np.zeros((bt, bi)))
        full = _clip_bwd(F, I, T, lsv, li, ni, nt, a, b, {"dI", "dT", "ds"})
        # dI = (g - ihat (g . ihat)) / |I|: the projection cancels (exactly, at d = 1), so the error is measured against
        # the pre-projection gradient g / |I|, the size of the terms the kernel subtracts
        gI = np.abs(sc * (G @ th) / np.linalg.norm(Id, axis=1, keepdims=True)).max()
        gT = np.abs(sc * (G.T @ ih) / np.linalg.norm(Td, axis=1, keepdims=True)).max()
        _close_scaled(f"{tag} dI", full["dI"], torch.from_numpy(dI_ref), gI, tol)
        _close_scaled(f"{tag} dT", full["dT"], torch.from_numpy(dT_ref), gT, tol)
        # dscale = sum G * logits: a sum of signed terms, bounded against the sum of their magnitudes
        _close_scaled(f"{tag} dscale", full["ds"], torch.tensor([ds_ref]), np.abs(G * li_ref).sum(), tol)
        if tag == "both":
            for only in ("dI", "dT", "ds"):
                one = _clip_bwd(F, I, T, lsv, li, ni, nt, a, b, {only})
                assert torch.equal(one[only], full[only]), f"{only} alone differs from {only} with every output"


@pytest.mark.parametrize("dt", DTYPES)
def test_clip_logits_refuse_d_past_backward(F, dt):
    """d = 1025: the backward cannot take it, so the forward refuses it too, before launching anything."""
    L = F.L
    I = torch.randn(3, 1025, device="cuda").to(dt)
    T = torch.randn(4, 1025, device="cuda").to(dt)
    ls = torch.zeros(1, device="cuda")
    li, ni, nt = torch.empty(3, 4, device="cuda"), torch.empty(3, device="cuda"), torch.empty(4, device="cuda")
    _expect_rejected(F, lambda: _clip_fwd(F, I, T, ls))
    dli = torch.randn(3, 4, device="cuda")
    _expect_rejected(F, lambda: L.check(L.lib().milb200_clip_logits_bwd(
        L.ptr(I), L.ptr(T), L.ptr(ls), L.ptr(li), L.ptr(ni), L.ptr(nt), L.ptr(dli), None, L.ptr(torch.empty_like(I)),
        None, None, 3, 4, 1025, L.dtype_code(I), L.stream_ptr()), "clip_logits_bwd"))
    _expect_rejected(F, lambda: F.clip_logits(I, T, ls))


# ---------------------------------------------------------------------------------------------------------------------
# C. CLIPloss_v1
# ---------------------------------------------------------------------------------------------------------------------
CL_B = [1, 2, 8, 9, 255, 256, 257, 700]
CL_I = [1, 9, 33]
CL_D = [1, 33, 512, 1024]
# pairwise over (b, d) with n_info cycling; every other case scales the inputs so that the largest logit is ~100,
# past fp32 exp's overflow at 88.7: only the max subtraction keeps those columns finite
CL_CASES = [(b, CL_I[(i + j) % 3], d, (i + j) % 2 == 1) for i, b in enumerate(CL_B) for j, d in enumerate(CL_D)]
CL_MAX_BD = (48 * 1024 - 32) // 4       # feature row + logits column in 48 KB, next to the kernel's 32-byte red[8]


def _cliploss64(out, feat):
    """mo.cliploss_v1 / mo.cliploss_v1_bwd restated on device tensors (pinned by test_cliploss_reference_is_the_oracle).
    Returns (loss, logits [I, b, b], dout)."""
    out, feat = out.to(F64), feat.to(F64)
    lg = torch.einsum("rd,cid->irc", out, feat)
    z = lg - lg.amax(dim=1, keepdim=True)
    lsm = z - z.exp().sum(dim=1, keepdim=True).log()
    n_info, b = lg.shape[0], lg.shape[1]
    loss = -lsm.diagonal(dim1=1, dim2=2).sum() / (n_info * b)
    dlog = (lsm.exp() - torch.eye(b, dtype=F64, device=lg.device)) / (n_info * b)
    return float(loss), lg, torch.einsum("irc,cid->rd", dlog, feat)


def test_cliploss_reference_is_the_oracle():
    rs = np.random.RandomState(1)
    out, feat = rs.randn(5, 7), rs.randn(5, 3, 7)
    loss, lg = mo.cliploss_v1(out, feat)
    dout = mo.cliploss_v1_bwd(out, feat)
    l2, lg2, d2 = _cliploss64(torch.from_numpy(out), torch.from_numpy(feat))
    assert abs(l2 - loss) <= 1e-13 * abs(loss)
    np.testing.assert_allclose(lg2.numpy(), lg, rtol=1e-13)
    np.testing.assert_allclose(d2.numpy(), dout, rtol=1e-12, atol=1e-15)


def _cliploss_call(F, out, feat, with_dout=True):
    L = F.L
    b, d = out.shape
    n_info = feat.shape[1]
    logits = torch.empty(n_info, b, b, device="cuda")
    ws = torch.empty(2 * n_info * b, device="cuda")
    loss = torch.empty(1, device="cuda")
    dout = torch.empty(b, d, device="cuda") if with_dout else None
    L.check(L.lib().milb200_cliploss_fwd_bwd(L.ptr(out), L.ptr(feat), L.ptr(logits), L.ptr(ws), L.ptr(loss), L.ptr(dout),
                                             b, n_info, d, L.dtype_code(out), L.stream_ptr()), "cliploss_fwd_bwd")
    return loss, logits, dout


def _cliploss_check(F, out, feat, tol, tag):
    loss, logits, dout = _cliploss_call(F, out, feat)
    l_ref, lg_ref, d_ref = _cliploss64(out, feat)
    big = float(lg_ref.abs().max())
    _close(f"{tag} logits", logits, lg_ref, tol)
    # loss = mean(lse - diagonal logit): the two terms are as large as the logits
    _close_scaled(f"{tag} loss", loss, torch.tensor([l_ref]), max(abs(l_ref), big), tol)
    # dout sums softmax weights exp(l - lse); l - lse carries a few ulps of the largest logit as absolute error, which
    # each weight carries as relative error: at logits ~100 that is 8 * 2^-24 * 100 = 4.8e-5 on top of the tolerance
    _close(f"{tag} dout", dout, d_ref, tol + 8 * U32 * big)
    return loss, logits, dout


@pytest.mark.parametrize("b,n_info,d,large", CL_CASES)
@pytest.mark.parametrize("dt", DTYPES)
def test_cliploss_vs_float64(F, dt, b, n_info, d, large):
    g = _gen(b * 131 + n_info * 17 + d)
    out = (torch.randn(b, d, device="cuda", generator=g) / d ** 0.25).to(dt)
    feat = (torch.randn(b, n_info, d, device="cuda", generator=g) / d ** 0.25).to(dt)
    if large:
        _, lg, _ = _cliploss64(out, feat)
        out = (out.to(F32) * (100.0 / float(lg.abs().max()))).to(dt)
    tag = f"b={b} I={n_info} d={d}{' large' if large else ''}"
    loss, logits, dout = _cliploss_check(F, out, feat, TOL[dt], tag)
    loss2, logits2, none = _cliploss_call(F, out, feat, with_dout=False)
    assert none is None and torch.equal(loss2, loss) and torch.equal(logits2, logits), "dout = NULL changed the loss"
    if b == 1:
        assert float(loss.item()) == 0.0 and not dout.any(), "b = 1: loss and dout must be exactly 0"


@pytest.mark.parametrize("dt", DTYPES)
def test_cliploss_shared_memory_edge(F, dt):
    """The last b + d the kernel's shared memory takes runs and is right; the next one is refused before any launch."""
    d, b = 16, CL_MAX_BD - 16
    g = _gen(4242)
    out = (torch.randn(b, d, device="cuda", generator=g) / 2).to(dt)
    feat = (torch.randn(b, 1, d, device="cuda", generator=g) / 2).to(dt)
    _cliploss_check(F, out, feat, TOL[dt], f"b={b} d={d}")
    out1 = torch.zeros(b + 1, d, device="cuda", dtype=dt)
    feat1 = torch.zeros(b + 1, 1, d, device="cuda", dtype=dt)
    _expect_rejected(F, lambda: _cliploss_call(F, out1, feat1))


# ---------------------------------------------------------------------------------------------------------------------
# D. cosine embedding loss, sigmoid + BCE
# ---------------------------------------------------------------------------------------------------------------------
COS_N = [1, 7, 8, 9, 1000]
COS_D = [1, 31, 33, 512, 1030, 4096]


def _cos_inputs(n, d, dt, g, first):
    """Rows cycle through a = 0 (the 1e-12 path), a = b, a = -b, a = 1e3 b and random, starting at `first`."""
    a = torch.randn(n, d, device="cuda", generator=g)
    b = torch.randn(n, d, device="cuda", generator=g).to(dt)
    kind = (torch.arange(n, device="cuda") + first) % 5
    bf = b.to(F32)
    a = torch.where((kind == 0)[:, None], torch.zeros_like(a), a)
    a = torch.where((kind == 1)[:, None], bf, a)
    a = torch.where((kind == 2)[:, None], -bf, a)
    a = torch.where((kind == 3)[:, None], 1e3 * bf, a)
    return a.to(dt), b


def _cos_call(F, a, b, da=True, db=True):
    L = F.L
    n, d = a.shape
    loss, rows = torch.empty(1, device="cuda"), torch.empty(n, device="cuda")
    ga = torch.empty_like(a) if da else None
    gb = torch.empty_like(b) if db else None
    L.check(L.lib().milb200_cosine_embedding_fwd_bwd(L.ptr(a), L.ptr(b), L.ptr(loss), L.ptr(rows), L.ptr(ga), L.ptr(gb), n,
                                                     d, L.dtype_code(a), L.stream_ptr()), "cosine_embedding")
    return loss, ga, gb


@pytest.mark.parametrize("d", COS_D)
@pytest.mark.parametrize("n", COS_N)
@pytest.mark.parametrize("dt", DTYPES)
def test_cosine_embedding_vs_float64(F, dt, n, d):
    g = _gen(n * 9973 + d)
    a, b = _cos_inputs(n, d, dt, g, first=COS_D.index(d))
    loss, da, db = _cos_call(F, a, b)
    a64 = a.to(F64).requires_grad_()
    b64 = b.to(F64).requires_grad_()
    ref = torch.nn.functional.cosine_embedding_loss(a64, b64, torch.ones(n, dtype=F64, device="cuda"))
    ref.backward()
    # 1 - cos is computed to a few fp32 ulps of 1, whatever the size of the mean
    _close_scaled("loss", loss, ref.detach().reshape(1), max(abs(float(ref)), 1.0), TOL[dt])
    # per row, da = -(b/sqrt(AB) - cos a/A)/n: the difference vanishes at a = +-b and a = 1e3 b, so each row is measured
    # against the size of its two terms
    with torch.no_grad():
        A = (a64 * a64).sum(1, keepdim=True) + 1e-12
        B = (b64 * b64).sum(1, keepdim=True) + 1e-12
        cs = (a64 * b64).sum(1, keepdim=True) / (A * B).sqrt()
        ta = (b64.abs().amax(1, keepdim=True) / (A * B).sqrt() + cs.abs() * a64.abs().amax(1, keepdim=True) / A) / n
        tb = (a64.abs().amax(1, keepdim=True) / (A * B).sqrt() + cs.abs() * b64.abs().amax(1, keepdim=True) / B) / n
        # (db of an a = 0 row has no terms at all: it must be exactly 0)
        ea = float(((da.to(F64) - a64.grad).abs().amax(1, keepdim=True) / ta.clamp_min(1e-300)).max())
        eb = float(((db.to(F64) - b64.grad).abs().amax(1, keepdim=True) / tb.clamp_min(1e-300)).max())
    assert ea <= TOL[dt] and eb <= TOL[dt], f"da / db error {ea:.3e} / {eb:.3e} of the row term scale > {TOL[dt]}"
    l1, ga, none = _cos_call(F, a, b, db=False)
    assert none is None and torch.equal(ga, da) and torch.equal(l1, loss)
    l2, none, gb = _cos_call(F, a, b, da=False)
    assert none is None and torch.equal(gb, db) and torch.equal(l2, loss)


BCE_N = [1, 2, 255, 256, 257, 4096]
BCE_PLANTED = [0.0, 16.6, -16.6, 27.6, -27.6, 15.0, -15.0, 120.0, -120.0, 95.0, -95.0]


def _bce_call(F, z, t, prob=True, loss=True, dz=True):
    L = F.L
    n = z.numel()
    o = {"prob": torch.empty_like(z) if prob else None, "loss": torch.empty(1, device="cuda") if loss else None,
         "dz": torch.empty_like(z) if dz else None}
    L.check(L.lib().milb200_sigmoid_bce_fwd_bwd(L.ptr(z), L.ptr(t), L.ptr(o["prob"]), L.ptr(o["loss"]), L.ptr(o["dz"]), n,
                                                L.stream_ptr()), "sigmoid_bce")
    return o


@pytest.mark.parametrize("n", BCE_N)
def test_sigmoid_bce_vs_float64(F, n):
    g = _gen(31 * n)
    z = torch.rand(n, device="cuda", generator=g) * 240 - 120
    k = min(n, len(BCE_PLANTED))
    z[:k] = torch.tensor(BCE_PLANTED[:k], device="cuda")
    t = torch.rand(n, device="cuda", generator=g)
    t[1::7] = 0.0
    t[2::7] = 1.0
    o = _bce_call(F, z, t)
    z64, t64 = z.to(F64), t.to(F64)
    p64 = torch.sigmoid(z64)
    # 1 / (1 + exp(-z)) in fp32 (here and in torch) is 0 once exp(-z) overflows (z < -88.7, sigmoid < 2^-126): below
    # the smallest normal float the probability is held to an absolute bound
    err = (o["prob"].to(F64) - p64).abs()
    assert bool((err <= 1e-5 * p64 + 2.0 ** -126).all()), "prob is not sigmoid(z) to 1e-5 relative"
    # The loss is that of the fp32 model: BCE of its fp32 probability, with torch's -100 clamps.  Where that probability
    # rounds to 1 (z > 16.6) log(1 - p) is decided by the rounding (torch's fp32 reference rounds the same way), so the
    # float64 BCE is taken of the probability the kernel formed, which was checked against float64 just above.
    pk = o["prob"].to(F64)
    l_ref = torch.nn.functional.binary_cross_entropy(pk, t64)
    _close("loss", o["loss"], l_ref.reshape(1), 1e-5)
    assert bool(((pk == 1) & (t64 < 1)).any()) or n < 4, "no element reached the clamp of log(1 - p)"
    # dz against torch's fp32 autograd where torch's gradient is the derivative (|z| <= 15) ...
    zt = z.clone().requires_grad_()
    torch.nn.functional.binary_cross_entropy(torch.sigmoid(zt), t).backward()
    inner = z.abs() <= 15
    _close("dz, |z| <= 15", o["dz"][inner], zt.grad[inner], 1e-5)
    # ... and beyond it the documented (p - t) / n, which torch's clamps do not give (include/milb200.h)
    _close("dz = (p - t)/n", o["dz"], (pk - t64) / n, 1e-5)
    sat = (pk == 1) & (t64 < 1)
    assert bool((o["dz"][sat] > 0).all()), "dz vanished where p rounds to 1"
    for drop in ("prob", "loss", "dz"):
        part = _bce_call(F, z, t, **{drop: False})
        for key, v in part.items():
            if key != drop:
                assert torch.equal(v, o[key]), f"{key} changed when {drop} was NULL"


def test_small_loss_refusals(F):
    L = F.L
    lib, S = L.lib(), L.stream_ptr()
    z = torch.zeros(4, device="cuda")
    _expect_rejected(F, lambda: L.check(lib.milb200_sigmoid_bce_fwd_bwd(L.ptr(z), L.ptr(z), None, None, None, 0, S), "bce"))
    _expect_rejected(F, lambda: L.check(lib.milb200_sigmoid_bce_fwd_bwd(None, L.ptr(z), None, None, None, 4, S), "bce"))
    a = torch.zeros(2, 8, device="cuda")
    _expect_rejected(F, lambda: L.check(lib.milb200_cosine_embedding_fwd_bwd(L.ptr(a), L.ptr(a), None, L.ptr(z), None, None,
                                                                             2, 8, L.F32, S), "cosine"))
    _expect_rejected(F, lambda: L.check(lib.milb200_cliploss_fwd_bwd(L.ptr(a), L.ptr(a), L.ptr(z), L.ptr(z), L.ptr(z),
                                                                     None, 2, 1, 1025, L.F32, S), "cliploss"))


# ---------------------------------------------------------------------------------------------------------------------
# E. elementwise glue
# ---------------------------------------------------------------------------------------------------------------------
def _philox_u16(seed, offset, ngroups):
    """Host Philox4x32-10: the sixteen 16-bit draws of each 8-element group, element j of group c from word j // 2,
    half j % 2 of the block at counter c + offset, key = (seed low, seed high)."""
    M = np.uint64(0xFFFFFFFF)
    c = np.arange(ngroups, dtype=np.uint64) + np.uint64(offset)
    x, y = c & M, c >> np.uint64(32)
    z = np.zeros_like(x)
    w = np.zeros_like(x)
    k0, k1 = np.uint64(seed & 0xFFFFFFFF), np.uint64(seed >> 32)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * x
        p1 = np.uint64(0xCD9E8D57) * z
        x, y, z, w = (p1 >> np.uint64(32)) ^ y ^ k0, p1 & M, (p0 >> np.uint64(32)) ^ w ^ k1, p0 & M
        k0 = (k0 + np.uint64(0x9E3779B9)) & M
        k1 = (k1 + np.uint64(0xBB67AE85)) & M
    words = np.stack([x, y, z, w], 1)
    return np.stack([words & np.uint64(0xFFFF), words >> np.uint64(16)], 2).reshape(ngroups * 8)


def _keep_mask(seed, offset, n, p):
    thr = int(np.float32(min(max(p, 0.0), 1.0)) * np.float32(65536.0))
    return torch.from_numpy(_philox_u16(seed, offset, (n + 7) // 8)[:n] >= thr).cuda()


def _dropout_call(F, x, p, seed, offset=0, out=None):
    L = F.L
    out = torch.empty_like(x) if out is None else out
    L.check(L.lib().milb200_dropout(L.ptr(x), L.ptr(out), x.numel(), p, seed, offset, L.dtype_code(x), L.stream_ptr()),
            "dropout")
    return out


DROP_N = [1, 7, 8, 9, 4095, 2 ** 20 + 3]
DROP_P = [0.0, 0.25, 0.5, 0.9]
SEED = 0x0123456789ABCDEF


@pytest.mark.parametrize("p", DROP_P)
@pytest.mark.parametrize("n", DROP_N)
@pytest.mark.parametrize("dt", DTYPES)
def test_dropout_mask_and_values(F, dt, n, p):
    g = _gen(n + int(100 * p))
    x = (torch.rand(n, device="cuda", generator=g) + 0.5).to(dt)          # nonzero, so a zero output is a drop
    out = _dropout_call(F, x, p, SEED)
    if p == 0.0:
        assert torch.equal(out, x), "p = 0 must be a bit-exact copy"
    keep = _keep_mask(SEED, 0, n, p)
    scale = np.float32(1.0) / (np.float32(1.0) - np.float32(p))
    want = torch.where(keep, (x.to(F32) * float(scale)).to(dt), torch.zeros_like(x))
    assert torch.equal(out, want), "dropout differs from x * fp32(1/(1-p)) under the Philox mask"
    # the scalar path (misaligned x / out) and a gradient through the same call draw the same mask
    xs = _misaligned(x)
    outs = _dropout_call(F, xs, p, SEED, out=_misaligned(torch.empty_like(x)))
    assert torch.equal(outs, out), "the scalar path picked a different mask or value"
    gr = (torch.rand(n, device="cuda", generator=g) - 2.0).to(dt)
    dg = _dropout_call(F, gr, p, SEED)
    assert torch.equal(dg != 0, keep), "the gradient's mask differs from the forward's"


@pytest.mark.parametrize("dt", DTYPES)
def test_dropout_offset_and_seed_bits(F, dt):
    n, k = 4096 + 8 * 5, 5
    x = torch.ones(n, device="cuda", dtype=dt)
    base = _dropout_call(F, x, 0.5, SEED) != 0
    shifted = _dropout_call(F, x[: n - 8 * k].contiguous(), 0.5, SEED, offset=k) != 0
    assert torch.equal(shifted, base[8 * k:]), "offset = k must shift the mask by 8k elements"
    hi = _dropout_call(F, x, 0.5, SEED ^ (1 << 40)) != 0
    assert not torch.equal(hi, base), "seeds that differ in bits 32-63 gave the same mask"
    assert torch.equal(hi, _keep_mask(SEED ^ (1 << 40), 0, n, 0.5))


@pytest.mark.parametrize("p", [0.25, 0.5, 0.9])
def test_dropout_keep_rate(F, p):
    n = 2 ** 22
    out = _dropout_call(F, torch.ones(n, device="cuda"), p, 0xDEADBEEF12345)
    q = 1 - math.floor(65536 * p) / 65536
    rate = float((out != 0).double().mean())
    assert abs(rate - q) <= 5 * math.sqrt(q * (1 - q) / n), f"keep rate {rate} vs {q}"


def test_dropout_refusals(F):
    L = F.L
    x = torch.ones(16, device="cuda")
    for p in (1.0, -0.1, float("nan")):
        _expect_rejected(F, lambda: _dropout_call(F, x, p, 1))
    _expect_rejected(F, lambda: L.check(L.lib().milb200_dropout(None, L.ptr(x), 16, 0.5, 1, 0, L.F32, L.stream_ptr()), "d"))


CAST_N = [1, 255, 606208, 606209]       # 148 * 16 * 256 = 606208: the grid cap
FLT_MAX = float(np.finfo(np.float32).max)
CAST_SPECIALS = [0.0, -0.0, 2.0 ** -149, -2.0 ** -149, 2.0 ** -126 - 2.0 ** -149, 2.0 ** -126, math.inf, -math.inf,
                 math.nan, FLT_MAX, -FLT_MAX, 1 + 2.0 ** -8, 1 + 3 * 2.0 ** -8, -(1 + 2.0 ** -8), 2.0 ** -130 * 1.5]


def _cast_call(F, x, dst):
    L = F.L
    out = torch.empty(x.shape, dtype=dst, device="cuda")
    L.check(L.lib().milb200_cast(L.ptr(x), L.dtype_code(x), L.ptr(out), L.dtype_code(out), x.numel(), L.stream_ptr()),
            "cast")
    return out


def _same_bits(got, want):
    nan = torch.isnan(want)
    assert torch.equal(torch.isnan(got), nan), "NaN-ness differs"
    ib = torch.int16 if got.dtype == BF16 else torch.int32
    assert torch.equal(got.view(ib)[~nan], want.view(ib)[~nan]), "bits differ"


@pytest.mark.parametrize("n", CAST_N)
def test_cast_bits(F, n):
    g = _gen(n)
    bits = torch.randint(-2 ** 31, 2 ** 31, (n,), dtype=torch.int32, device="cuda", generator=g)
    bits[1::4] = (bits[1::4] & -65536) | 0x8000                                         # exact halfway values
    x = bits.view(F32)
    k = min(n, len(CAST_SPECIALS))
    x[:k] = torch.tensor(CAST_SPECIALS[:k], dtype=F32, device="cuda")
    _same_bits(_cast_call(F, x, BF16), x.to(BF16))
    hb = torch.randint(-2 ** 15, 2 ** 15, (n,), dtype=torch.int16, device="cuda", generator=g).view(BF16)
    _same_bits(_cast_call(F, hb, F32), hb.to(F32))


AX_N = [1, 2, 3, 4, 5, 6, 7, 8, 9, 17, 1212419, 2424839]   # tails mod 4 and 8; past the grid cap of fp32 and of bf16


def _ulp(x, dt):
    mant, lo = (23, -149) if dt == F32 else (7, -133)
    e = torch.frexp(x)[1]
    return torch.ldexp(torch.ones_like(x), (e - 1 - mant).clamp_min(lo))


@pytest.mark.parametrize("n", AX_N)
@pytest.mark.parametrize("dt", DTYPES)
def test_axpby_add_rounding(F, dt, n):
    """The result is the float64 value rounded once, to within one ulp of the output type; axpby's fp32 products
    alpha a and beta b add one fp32 rounding each, 2^-24 of their size."""
    L = F.L
    lib, S, code = L.lib(), L.stream_ptr(), L.dtype_code(torch.empty(0, dtype=dt))
    g = _gen(n)
    a = torch.randn(n, device="cuda", generator=g).to(dt)
    b = torch.randn(n, device="cuda", generator=g).to(dt)
    al, be = 0.3, -1.7
    alf, bef = _f32(al), _f32(be)
    a64, b64 = a.to(F64), b.to(F64)

    def check(name, got, want, prod):
        err = (got.to(F64) - want).abs()
        bound = _ulp(want, dt) + 2 * U32 * prod
        assert bool((err <= bound).all()), f"{name}: error {float((err - bound).max()):.3e} past one rounding"

    out = torch.empty_like(a)
    L.check(lib.milb200_axpby(L.ptr(a), L.ptr(b), L.ptr(out), n, al, be, code, S), "axpby")
    check("axpby", out, alf * a64 + bef * b64, (alf * a64).abs() + (bef * b64).abs())
    L.check(lib.milb200_axpby(L.ptr(a), None, L.ptr(out), n, al, be, code, S), "axpby b=NULL")
    check("axpby b=NULL", out, alf * a64, (alf * a64).abs())
    L.check(lib.milb200_add(L.ptr(a), L.ptr(b), L.ptr(out), n, code, S), "add")
    check("add", out, a64 + b64, torch.zeros_like(a64))
    ai = a.clone()
    L.check(lib.milb200_axpby(L.ptr(ai), L.ptr(b), L.ptr(ai), n, al, be, code, S), "axpby in place")
    check("axpby in place", ai, alf * a64 + bef * b64, (alf * a64).abs() + (bef * b64).abs())
    if n > 1:
        am = _misaligned(a)[: n - 1]
        bm = b[: n - 1]
        _expect_rejected(F, lambda: L.check(lib.milb200_axpby(L.ptr(am), L.ptr(bm), L.ptr(out), n - 1, al, be, code, S),
                                            "axpby"))
        _expect_rejected(F, lambda: L.check(lib.milb200_add(L.ptr(bm), L.ptr(am), L.ptr(out), n - 1, code, S), "add"))
        _expect_rejected(F, lambda: L.check(lib.milb200_axpby(L.ptr(bm), None, L.ptr(am), n - 1, al, be, code, S),
                                            "axpby"))


@pytest.mark.parametrize("rows,cols", [(1, 1), (1, 33), (33, 1), (31, 32), (32, 31), (1000, 77)])
@pytest.mark.parametrize("dt", DTYPES)
def test_transpose_exact(F, dt, rows, cols):
    L = F.L
    x = torch.randn(rows, cols, device="cuda").to(dt)
    out = torch.full((cols, rows), SENTINEL, device="cuda", dtype=dt)
    L.check(L.lib().milb200_transpose(L.ptr(x), L.ptr(out), rows, cols, L.dtype_code(x), L.stream_ptr()), "transpose")
    assert torch.equal(out, x.t())


@pytest.mark.parametrize("dim", [2, 512, 768])
@pytest.mark.parametrize("n_pos", [1, 300, 15592, 41003])
def test_sinusoid_pe_bound(F, n_pos, dim):
    """fp32 angles p * w_i carry about two ulps of p (the rounded frequency and the product), and sin / cos a couple of
    ulps of 1: |pe - exact| <= 2 p 2^-23 + 2^-22.  The reference's own fp32 table (fo.sinusoid_pe) meets the same bound
    and no tighter one (its largest error is ~3e-3 at 41 003 rows), so the kernel is held to what the reference does."""
    exact = torch.from_numpy(mo.sinusoid_pe(n_pos, dim)[0]).cuda()
    bound = (2 * torch.arange(n_pos, dtype=F64, device="cuda") * 2.0 ** -23 + 2.0 ** -22)[:, None]
    pe = F.sinusoid_pe(n_pos, dim, F32, "cuda")[0]
    assert bool(((pe.to(F64) - exact).abs() <= bound).all()), "sinusoid_pe past its bound"
    ref = fo.sinusoid_pe(n_pos, dim)[0].cuda()
    assert bool(((ref.to(F64) - exact).abs() <= bound).all()), "the reference's table is past the bound"
    assert torch.equal(F.sinusoid_pe(n_pos, dim, BF16, "cuda")[0], pe.to(BF16)), "bf16 table is not the rounded fp32 one"


@pytest.mark.parametrize("c,t,hw", [(512, 1, 1), (512, 160, 2), (3, 7, 1000)])
@pytest.mark.parametrize("dt", DTYPES)
def test_ct_tokens_vs_float64(F, dt, c, t, hw):
    L = F.L
    g = _gen(c + t + hw)
    fmap = torch.randn(c, t, hw, device="cuda", generator=g).to(dt)
    tok = torch.empty(t, c, device="cuda", dtype=dt)
    L.check(L.lib().milb200_ct_tokens_fwd(L.ptr(fmap), L.ptr(tok), c, t, hw, L.dtype_code(fmap), L.stream_ptr()), "ct")
    _close("ct_tokens", tok, fmap.to(F64).mean(-1).t(), TOL[dt])
    dtok = torch.randn(t, c, device="cuda", generator=g).to(dt)
    dfm = torch.empty_like(fmap)
    L.check(L.lib().milb200_ct_tokens_bwd(L.ptr(dtok), L.ptr(dfm), c, t, hw, L.dtype_code(fmap), L.stream_ptr()), "ct")
    _close("ct_tokens bwd", dfm, (dtok.to(F64).t() / hw)[:, :, None].expand(c, t, hw), TOL[dt])


# ---------------------------------------------------------------------------------------------------------------------
# F. launch accounting
# ---------------------------------------------------------------------------------------------------------------------
def _kernels_recorded(fn, tmp_path, tag):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    path = tmp_path / f"{tag}.json"
    prof.export_chrome_trace(str(path))
    with open(path) as fh:
        ev = json.load(fh)
    ev = ev["traceEvents"] if isinstance(ev, dict) else ev
    return [e.get("name") for e in ev if e.get("cat") == "kernel"]


def test_launch_count_matches_profiler(F, tmp_path):
    """For every entry point of this file, the launch counter moves by the number of kernels the profiler records."""
    L = F.L
    lib, S = L.lib(), L.stream_ptr()
    P = L.ptr
    n = 5000
    p, gr, m, v = (torch.rand(n, device="cuda") for _ in range(4))
    ctr = torch.ones(1, dtype=torch.int32, device="cuda")
    I, T = torch.randn(7, 33, device="cuda"), torch.randn(5, 33, device="cuda")
    ls = torch.zeros(1, device="cuda")
    li, ni, nt = torch.empty(7, 5, device="cuda"), torch.empty(7, device="cuda"), torch.empty(5, device="cuda")
    dli, dlt = torch.randn(7, 5, device="cuda"), torch.randn(5, 7, device="cuda")
    dI, dT, ds = torch.empty_like(I), torch.empty_like(T), torch.empty(1, device="cuda")
    out, feat = torch.randn(9, 33, device="cuda"), torch.randn(9, 3, 33, device="cuda")
    lg, ws, loss, dout = (torch.empty(3, 9, 9, device="cuda"), torch.empty(54, device="cuda"), torch.empty(1, device="cuda"),
                          torch.empty(9, 33, device="cuda"))
    ca, cb, rows = torch.randn(9, 33, device="cuda"), torch.randn(9, 33, device="cuda"), torch.empty(9, device="cuda")
    cg = torch.empty_like(ca)
    z, tg, pz = torch.randn(300, device="cuda"), torch.rand(300, device="cuda"), torch.empty(300, device="cuda")
    xb = torch.empty(n, dtype=BF16, device="cuda")
    fm, tok = torch.randn(6, 4, 10, device="cuda"), torch.empty(4, 6, device="cuda")
    pe = torch.empty(300, 64, device="cuda")
    calls = {
        "adam_step": lambda: lib.milb200_adam_step(P(p), P(gr), P(m), P(v), n, 1e-3, B1, B2, EPS, 0.0, 1.0, 3, S),
        "adam_step n=0": lambda: lib.milb200_adam_step(P(p), P(gr), P(m), P(v), 0, 1e-3, B1, B2, EPS, 0.0, 1.0, 3, S),
        "adam_step_dev": lambda: lib.milb200_adam_step_dev(P(p), P(gr), P(m), P(v), n, 1e-3, B1, B2, EPS, 0.0, 1.0, P(ctr), S),
        "step_counter_inc": lambda: lib.milb200_step_counter_inc(P(ctr), S),
        "sgd_step": lambda: lib.milb200_sgd_step(P(p), P(gr), n, 1e-3, 0.0, 1.0, S),
        "clip_logits_fwd": lambda: lib.milb200_clip_logits_fwd(P(I), P(T), P(ls), P(li), P(ni), P(nt), 7, 5, 33, L.F32, S),
        "cliploss": lambda: lib.milb200_cliploss_fwd_bwd(P(out), P(feat), P(lg), P(ws), P(loss), P(dout), 9, 3, 33, L.F32, S),
        "cliploss dout=NULL": lambda: lib.milb200_cliploss_fwd_bwd(P(out), P(feat), P(lg), P(ws), P(loss), None, 9, 3, 33,
                                                                   L.F32, S),
        "cosine": lambda: lib.milb200_cosine_embedding_fwd_bwd(P(ca), P(cb), P(loss), P(rows), P(cg), None, 9, 33, L.F32, S),
        "sigmoid_bce": lambda: lib.milb200_sigmoid_bce_fwd_bwd(P(z), P(tg), P(pz), P(loss), None, 300, S),
        "dropout": lambda: lib.milb200_dropout(P(p), P(m), n, 0.5, 7, 0, L.F32, S),
        "cast": lambda: lib.milb200_cast(P(p), L.F32, P(xb), L.BF16, n, S),
        "axpby": lambda: lib.milb200_axpby(P(p), None, P(m), n, 2.0, 0.0, L.F32, S),
        "add": lambda: lib.milb200_add(P(p), P(gr), P(m), n, L.F32, S),
        "transpose": lambda: lib.milb200_transpose(P(I), P(dI.view(33, 7)), 7, 33, L.F32, S),
        "sinusoid_pe": lambda: lib.milb200_sinusoid_pe(P(pe), 300, 64, L.F32, S),
        "ct_tokens_fwd": lambda: lib.milb200_ct_tokens_fwd(P(fm), P(tok), 6, 4, 10, L.F32, S),
        "ct_tokens_bwd": lambda: lib.milb200_ct_tokens_bwd(P(tok), P(fm), 6, 4, 10, L.F32, S),
    }
    for up in ("image", "text", "both"):
        a, b = (dli if up != "text" else None), (dlt if up != "image" else None)
        for mask in range(8):
            o = [x if mask >> k & 1 else None for k, x in enumerate((dI, dT, ds))]
            calls[f"clip_logits_bwd {up} dI={o[0] is not None} dT={o[1] is not None} ds={o[2] is not None}"] = (
                lambda a=a, b=b, o=o: lib.milb200_clip_logits_bwd(P(I), P(T), P(ls), P(li), P(ni), P(nt), P(a), P(b),
                                                                  P(o[0]), P(o[1]), P(o[2]), 7, 5, 33, L.F32, S))
    wrong = []
    for i, (name, fn) in enumerate(calls.items()):
        res = {}

        def run(fn=fn, res=res):
            n0 = L.launch_count()
            res["rc"] = fn()
            res["count"] = L.launch_count() - n0
        kernels = _kernels_recorded(run, tmp_path, f"call{i}")
        assert res["rc"] == 0, f"{name}: {lib.milb200_last_error()}"
        if res["count"] != len(kernels):
            wrong.append(f"{name}: counted {res['count']}, profiler saw {len(kernels)} {kernels}")
    assert not wrong, "launch counter disagrees with the profiler:\n" + "\n".join(wrong)
