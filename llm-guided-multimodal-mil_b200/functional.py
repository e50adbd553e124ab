"""autograd.Functions over the C ABI.  Every forward/backward here is a sequence of libmilb200 kernel
launches on the current CUDA stream; nothing is computed with eager PyTorch ops except dtype casts of
tiny parameter vectors and views/slices of the gradient buffers."""
from __future__ import annotations

import torch

from . import _lib as L

# --------------------------------------------------------------------------------------------------
# gated-attention MIL pool over a CSR batch of bags           (reference: model/dim1/ABMIL.py:47-64)
# --------------------------------------------------------------------------------------------------


def _f32(t):
    return t if t.dtype == torch.float32 else t.float()


def _recompute_gate():
    import os
    return os.environ.get("MILB200_RECOMPUTE_GATE", "0") == "1"


def pack_gate_weights(Wv, bv, Wu, bu, dtype):
    """[Wv; Wu] -> Wcat (2D, L) in `dtype`, [bv; bu] -> bcat fp32 (one kernel)."""
    D, Lf = Wv.shape
    Wcat = torch.empty((2 * D, Lf), dtype=dtype, device=Wv.device)
    bcat = torch.empty((2 * D,), dtype=torch.float32, device=Wv.device)
    Wv, Wu, bv, bu = (t.contiguous() for t in (Wv, Wu, bv, bu))
    if not (Wv.dtype == Wu.dtype == bv.dtype == bu.dtype):
        raise L.MilB200Error("gate parameters must share one dtype")
    L.check(L.lib().milb200_pack_gate_weights(L.ptr(Wv), L.ptr(Wu), L.ptr(bv), L.ptr(bu), L.dtype_code(Wv),
                                              Lf, D, L.ptr(Wcat), L.dtype_code(Wcat), L.ptr(bcat),
                                              L.stream_ptr()), "pack_gate_weights")
    return Wcat, bcat


def gated_scores(X, Wcat, bcat, ww, bw, save=False):
    """s[i] = (tanh(x_i Wv^T + bv) * sigmoid(x_i Wu^T + bu)) . ww + bw   -> fp32 [total_n].
    save=True additionally returns the gate activations [total_n, 2D] (or None when the kernel path in use recomputes
    them in backward anyway) to hand to gated_scores_bwd."""
    n, Lf = X.shape
    D = Wcat.shape[0] // 2
    s = torch.empty((n,), dtype=torch.float32, device=X.device)
    code = L.dtype_code(X)
    act = None
    if save and L.lib().milb200_gated_score_saves_activations(Lf, D, code):
        act = torch.empty((n, 2 * D), dtype=X.dtype, device=X.device)
    nb = L.lib().milb200_gated_score_workspace_bytes(n, Lf, D, code, 0)
    ws = L.workspace(nb, X.device)
    L.check(L.lib().milb200_gated_score_fwd(L.ptr(X), L.ptr(Wcat), L.ptr(bcat), L.ptr(ww), L.ptr(bw), L.ptr(s),
                                            L.ptr(act), n, Lf, D, code, L.ptr(ws), ws.numel(), L.stream_ptr()),
            "gated_score_fwd")
    return (s, act) if save else s


def segment_softmax_pool(X, s, offsets, want_lowp=False):
    """M[b] = sum_i softmax_b(s)_i x_i over CSR offsets.  Returns (M fp32 [B,L], M_lowp|None, argmax int32 [B],
    lse fp32 [B])."""
    n, Lf = X.shape
    B = offsets.numel() - 1
    M = torch.empty((B, Lf), dtype=torch.float32, device=X.device)
    Ml = torch.empty((B, Lf), dtype=X.dtype, device=X.device) if want_lowp else None
    am = torch.empty((B,), dtype=torch.int32, device=X.device)
    lse = torch.empty((B,), dtype=torch.float32, device=X.device)
    nb = L.lib().milb200_pool_workspace_bytes(n, B, Lf)
    ws = L.workspace(nb, X.device)
    L.check(L.lib().milb200_segment_softmax_pool_fwd(L.ptr(X), L.ptr(s), L.ptr(offsets), B, n, Lf,
                                                     L.dtype_code(X), L.ptr(M), L.ptr(Ml), L.ptr(am), L.ptr(lse),
                                                     L.ptr(ws), ws.numel(), L.stream_ptr()),
            "segment_softmax_pool_fwd")
    return M, Ml, am, lse


def segment_softmax_pool_bwd(X, s, offsets, dM, M, want_attn):
    n, Lf = X.shape
    B = offsets.numel() - 1
    ds = torch.empty((n,), dtype=torch.float32, device=X.device)
    attn = torch.empty((n,), dtype=torch.float32, device=X.device) if want_attn else None
    nb = L.lib().milb200_pool_workspace_bytes(n, B, Lf)
    ws = L.workspace(nb, X.device)
    L.check(L.lib().milb200_segment_softmax_pool_bwd(L.ptr(X), L.ptr(s), L.ptr(offsets), B, n, Lf,
                                                     L.dtype_code(X), L.ptr(dM), L.ptr(M), L.ptr(ds), L.ptr(attn),
                                                     L.ptr(ws), ws.numel(), L.stream_ptr()),
            "segment_softmax_pool_bwd")
    return ds, attn


def _check_dM(dM, B, Lf):
    if dM.dtype != torch.float32 or tuple(dM.shape) != (B, Lf):
        raise L.MilB200Error(f"dM must be fp32 [{B}, {Lf}], got {dM.dtype} {list(dM.shape)}")


def segment_softmax_pool_rowdot(X, s, offsets, dM, want_lowp=False):
    """segment_softmax_pool for a caller that already has dL/dM: the same pass over X also returns
    rowdot[i] = dM_b . x_i (fp32 [total_n]), which lets segment_softmax_pool_bwd_rowdot skip X.
    Returns (M, M_lowp|None, argmax, lse, rowdot); the first four equal segment_softmax_pool's bit for bit."""
    n, Lf = X.shape
    B = offsets.numel() - 1
    _check_dM(dM, B, Lf)
    M = torch.empty((B, Lf), dtype=torch.float32, device=X.device)
    Ml = torch.empty((B, Lf), dtype=X.dtype, device=X.device) if want_lowp else None
    am = torch.empty((B,), dtype=torch.int32, device=X.device)
    lse = torch.empty((B,), dtype=torch.float32, device=X.device)
    rowdot = torch.empty((n,), dtype=torch.float32, device=X.device)
    ws = L.workspace(L.lib().milb200_pool_workspace_bytes(n, B, Lf), X.device)
    L.check(L.lib().milb200_segment_softmax_pool_fwd_rowdot(L.ptr(X), L.ptr(s), L.ptr(offsets), B, n, Lf,
                                                            L.dtype_code(X), L.ptr(dM), L.ptr(M), L.ptr(Ml), L.ptr(am),
                                                            L.ptr(lse), L.ptr(rowdot), L.ptr(ws), ws.numel(),
                                                            L.stream_ptr()),
            "segment_softmax_pool_fwd_rowdot")
    return M, Ml, am, lse, rowdot


def segment_softmax_pool_bwd_rowdot(s, offsets, dM, M, rowdot, want_attn):
    """segment_softmax_pool_bwd from the row dots of segment_softmax_pool_rowdot (same dM): no pass over X.
    Returns (ds, attn|None), equal to segment_softmax_pool_bwd's bit for bit."""
    n = s.numel()
    B, Lf = M.shape
    _check_dM(dM, B, Lf)
    ds = torch.empty((n,), dtype=torch.float32, device=s.device)
    attn = torch.empty((n,), dtype=torch.float32, device=s.device) if want_attn else None
    ws = L.workspace(L.lib().milb200_pool_workspace_bytes(n, B, Lf), s.device)
    L.check(L.lib().milb200_segment_softmax_pool_bwd_rowdot(L.ptr(s), L.ptr(offsets), B, n, Lf, L.ptr(dM), L.ptr(M),
                                                            L.ptr(rowdot), L.ptr(ds), L.ptr(attn), L.ptr(ws), ws.numel(),
                                                            L.stream_ptr()),
            "segment_softmax_pool_bwd_rowdot")
    return ds, attn


def gated_scores_bwd(X, Wcat, bcat, ww, bw, ds, attn, dM, offsets, need_dx, grad_out=None, gate_act=None):
    """Backward of gated_scores (+ the pooling term of dX).  `grad_out`, if given, is a flat fp32 buffer of
    2D*L + 2D + D + 1 elements (laid out dWcat | dbcat | dww | dbw) that the kernels write in place — the
    data-parallel trainer passes a slice of its flat gradient buffer."""
    n, Lf = X.shape
    D = Wcat.shape[0] // 2
    B = offsets.numel() - 1
    need = 2 * D * Lf + 2 * D + D + 1
    if grad_out is None:
        grad_out = torch.empty((need,), dtype=torch.float32, device=X.device)
    elif grad_out.numel() != need or grad_out.dtype != torch.float32:
        raise L.MilB200Error("gated_scores_bwd: grad_out must be fp32 with 2D*L+3D+1 elements")
    dWcat = grad_out[:2 * D * Lf].view(2 * D, Lf)
    dbcat = grad_out[2 * D * Lf:2 * D * Lf + 2 * D]
    dww = grad_out[2 * D * Lf + 2 * D:2 * D * Lf + 3 * D]
    dbw = grad_out[2 * D * Lf + 3 * D:]
    dX = torch.empty_like(X) if need_dx else None
    code = L.dtype_code(X)
    nb = L.lib().milb200_gated_score_workspace_bytes(n, Lf, D, code, 1)
    ws = L.workspace(nb, X.device)
    L.check(L.lib().milb200_gated_score_bwd(L.ptr(X), L.ptr(Wcat), L.ptr(bcat), L.ptr(ww), L.ptr(bw), L.ptr(ds),
                                            L.ptr(gate_act), L.ptr(attn) if need_dx else None, L.ptr(dM) if need_dx else None,
                                            L.ptr(offsets), B, n, Lf, D, code, L.ptr(dWcat), L.ptr(dbcat),
                                            L.ptr(dww), L.ptr(dbw), L.ptr(dX), L.ptr(ws), ws.numel(),
                                            L.stream_ptr()), "gated_score_bwd")
    return dX, dWcat, dbcat, dww, dbw


class _AbmilPoolCSR(torch.autograd.Function):
    """M[b] = ABMIL(x[offsets[b]:offsets[b+1]]) for every bag of a packed batch, eval-mode semantics
    (ABMIL.py:47-64 applied bag by bag, which is how train_ddp.py:75 / test_ddp.py:73 run it)."""

    @staticmethod
    def forward(ctx, X, offsets, Wv, bv, Wu, bu, ww, bw, out_fp32=False):
        X = X.contiguous()
        Wcat, bcat = pack_gate_weights(Wv, bv, Wu, bu, X.dtype)
        wwf = _f32(ww).reshape(-1).contiguous()
        bwf = _f32(bw).reshape(-1).contiguous()
        # training: keep the gate activations (0.77 KB/instance in bf16) so that backward skips the recompute GEMM;
        # MILB200_RECOMPUTE_GATE=1 trades that memory back for time
        need_grad = any(ctx.needs_input_grad) and not _recompute_gate()
        s, act = gated_scores(X, Wcat, bcat, wwf, bwf, save=True) if need_grad else (gated_scores(X, Wcat, bcat, wwf, bwf), None)
        M, Ml, am, lse = segment_softmax_pool(X, s, offsets, want_lowp=(X.dtype != torch.float32 and not out_fp32))
        ctx.save_for_backward(X, offsets, Wcat, bcat, wwf, bwf, s, M, act)
        ctx.param_dtypes = (Wv.dtype, bv.dtype, Wu.dtype, bu.dtype, ww.dtype, bw.dtype)
        ctx.D = Wv.shape[0]
        ctx.mark_non_differentiable(am, s)
        return (M if Ml is None else Ml), am, s

    @staticmethod
    def backward(ctx, dM_out, _dam, _ds):
        X, offsets, Wcat, bcat, wwf, bwf, s, M, act = ctx.saved_tensors
        D = ctx.D
        need_dx = ctx.needs_input_grad[0]
        dM = _f32(dM_out).contiguous()
        ds, attn = segment_softmax_pool_bwd(X, s, offsets, dM, M, want_attn=need_dx)
        dX, dWcat, dbcat, dww, dbw = gated_scores_bwd(X, Wcat, bcat, wwf, bwf, ds, attn, dM, offsets, need_dx,
                                                      gate_act=act)
        dt = ctx.param_dtypes
        return (dX, None, dWcat[:D].to(dt[0]), dbcat[:D].to(dt[1]), dWcat[D:].to(dt[2]), dbcat[D:].to(dt[3]),
                dww.view(1, D).to(dt[4]), dbw.view(1).to(dt[5]), None)


def abmil_pool_csr(X, offsets, Wv, bv, Wu, bu, ww, bw, out_fp32=False):
    """Returns (M [B,L], argmax int32 [B] (index within the bag), scores fp32 [total_n]).  M is in X.dtype, or — with
    out_fp32 — the fp32 accumulator itself (B x L values: callers that feed a small head keep it in fp32 so that the
    bf16 storage of the instances is the only reduced-precision step on the path)."""
    if offsets.dtype != torch.int32:
        raise L.MilB200Error("offsets must be int32 CSR offsets on the device")
    return _AbmilPoolCSR.apply(X, offsets, Wv, bv, Wu, bu, ww, bw, out_fp32)


# --------------------------------------------------------------------------------------------------
# dropout (train mode only) and the dense-batch sum pool quirk
# --------------------------------------------------------------------------------------------------
def _dropout_raw(x, p, seed, offset):
    out = torch.empty_like(x)
    L.check(L.lib().milb200_dropout(L.ptr(x), L.ptr(out), x.numel(), float(p), int(seed), int(offset),
                                    L.dtype_code(x), L.stream_ptr()), "dropout")
    return out


class _Dropout(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, p):
        x = x.contiguous()
        # one 63-bit seed per call from torch's CPU generator (so torch.manual_seed controls it)
        ctx.seed = int(torch.randint(0, 2 ** 62, (1,), dtype=torch.int64).item())
        ctx.p = p
        return _dropout_raw(x, p, ctx.seed, 0)

    @staticmethod
    def backward(ctx, g):
        return _dropout_raw(g.contiguous(), ctx.p, ctx.seed, 0), None


def dropout(x, p):
    """nn.Dropout(p) in train mode; Philox mask regenerated (not stored) in backward."""
    if p <= 0.0:
        return x
    return _Dropout.apply(x, p)


class _DenseSumPool(torch.autograd.Function):
    """x (B,N,L) -> (B,1,L) = sum over N: the reference's behaviour for dense batches B>1 (SURVEY F2)."""

    @staticmethod
    def forward(ctx, x):
        B, N, Lf = x.shape
        X = x.contiguous().view(B * N, Lf)
        off = torch.arange(0, (B + 1) * N, N, dtype=torch.int32, device=x.device)
        M = torch.empty((B, Lf), dtype=torch.float32, device=x.device)
        Ml = torch.empty((B, Lf), dtype=x.dtype, device=x.device) if x.dtype != torch.float32 else None
        nb = L.lib().milb200_pool_workspace_bytes(B * N, B, Lf)
        ws = L.workspace(nb, x.device)
        L.check(L.lib().milb200_segment_sum_fwd(L.ptr(X), L.ptr(off), B, B * N, Lf, L.dtype_code(X), L.ptr(M),
                                                L.ptr(Ml), L.ptr(ws), ws.numel(), L.stream_ptr()),
                "segment_sum_fwd")
        ctx.save_for_backward(off)
        ctx.shape = (B, N, Lf)
        ctx.dtype = x.dtype
        return (M if Ml is None else Ml).view(B, 1, Lf)

    @staticmethod
    def backward(ctx, g):
        (off,) = ctx.saved_tensors
        B, N, Lf = ctx.shape
        gf = _f32(g).contiguous().view(B, Lf)
        out = torch.empty((B * N, Lf), dtype=ctx.dtype, device=g.device)
        L.check(L.lib().milb200_bag_broadcast(L.ptr(gf), None, L.ptr(off), B, B * N, Lf, L.dtype_code(out),
                                              L.ptr(out), L.stream_ptr()), "bag_broadcast")
        return out.view(B, N, Lf)


def dense_sum_pool(x):
    return _DenseSumPool.apply(x)


# --------------------------------------------------------------------------------------------------
# dense layers, LayerNorm, attention core                    (reference: model/sam/transformer.py)
# --------------------------------------------------------------------------------------------------
_ACT = {None: L.ACT_NONE, "none": L.ACT_NONE, "tanh": L.ACT_TANH, "relu": L.ACT_RELU, "sigmoid": L.ACT_SIGMOID}


def cast(t, dtype):
    """dtype conversion through the library's cast kernel (fp32 <-> bf16)."""
    if t.dtype == dtype:
        return t
    t = t.contiguous()
    out = torch.empty_like(t, dtype=dtype)
    L.check(L.lib().milb200_cast(L.ptr(t), L.dtype_code(t), L.ptr(out), L.dtype_code(out), t.numel(),
                                 L.stream_ptr()), "cast")
    return out


class _Linear(torch.autograd.Function):
    """y = act((x [+ add]) W^T + b): nn.Linear (+Tanh/ReLU) sites of aggregator.py:44,47,66 and
    transformer.py:430-432,448 / common.py:26.  `add` fuses the `keys + key_pe` / `queries + query_pe` sums."""

    @staticmethod
    def forward(ctx, x, W, b, act, add):
        shp = x.shape
        k = shp[-1]
        n = W.shape[0]
        x2 = x.contiguous().view(-1, k)
        a2 = add.contiguous().view(-1, k) if add is not None else None
        if a2 is not None and a2.shape != x2.shape:
            raise L.MilB200Error("linear: `add` must have the shape of x")
        m = x2.shape[0]
        Wc = cast(W, x2.dtype)
        bf = _f32(b).contiguous() if b is not None else None
        y = torch.empty((m, n), dtype=x2.dtype, device=x2.device)
        code = L.dtype_code(x2)
        nb = L.lib().milb200_linear_workspace_bytes(m, n, k, code, 0)
        ws = L.workspace(nb, x2.device)
        L.check(L.lib().milb200_linear_fwd(L.ptr(x2), L.ptr(a2), L.ptr(Wc), L.ptr(bf), L.ptr(y), m, n, k, act, code,
                                           L.ptr(ws), ws.numel(), L.stream_ptr()), "linear_fwd")
        ctx.save_for_backward(x2, a2, Wc, y)
        ctx.meta = (shp, m, n, k, act, W.dtype, b.dtype if b is not None else None, add is not None,
                    add.shape if add is not None else None)
        return y.view(*shp[:-1], n)

    @staticmethod
    def backward(ctx, dy):
        x2, a2, Wc, y = ctx.saved_tensors
        shp, m, n, k, act, wdt, bdt, has_add, ashp = ctx.meta
        need_dx = ctx.needs_input_grad[0] or (has_add and ctx.needs_input_grad[4])
        need_dw = ctx.needs_input_grad[1]
        need_db = bdt is not None and ctx.needs_input_grad[2]
        dy2 = dy.contiguous().view(m, n)
        if dy2.dtype != x2.dtype:
            dy2 = cast(dy2, x2.dtype)
        dX = torch.empty_like(x2) if need_dx else None
        dW = torch.empty((n, k), dtype=torch.float32, device=x2.device) if need_dw else None
        db = torch.empty((n,), dtype=torch.float32, device=x2.device) if need_db else None
        code = L.dtype_code(x2)
        nb = L.lib().milb200_linear_workspace_bytes(m, n, k, code, 1)
        ws = L.workspace(nb, x2.device)
        L.check(L.lib().milb200_linear_bwd(L.ptr(x2), L.ptr(a2), L.ptr(Wc), L.ptr(y), L.ptr(dy2), L.ptr(dX), L.ptr(dW),
                                           L.ptr(db), m, n, k, act, code, 0, L.ptr(ws), ws.numel(), L.stream_ptr()),
                "linear_bwd")
        gx = dX.view(shp) if (dX is not None and ctx.needs_input_grad[0]) else None
        ga = dX.view(ashp) if (dX is not None and has_add and ctx.needs_input_grad[4]) else None
        gw = cast(dW, wdt) if dW is not None else None
        gb = cast(db, bdt) if db is not None else None
        return gx, gw, gb, None, ga


def linear(x, W, b=None, act=None, add=None):
    return _Linear.apply(x, W, b, _ACT[act] if not isinstance(act, int) else act, add)


class _LayerNorm(torch.autograd.Function):
    """y = LayerNorm(x [+ r]) * gamma + beta, eps 1e-5 (transformer.py:288,295,300,307,118; the residual adds of
    :286,294,299,306 are fused in)."""

    @staticmethod
    def forward(ctx, x, r, gamma, beta):
        shp = x.shape
        n = shp[-1]
        x2 = x.contiguous().view(-1, n)
        r2 = r.contiguous().view(-1, n) if r is not None else None
        m = x2.shape[0]
        g, b = _f32(gamma).contiguous(), _f32(beta).contiguous()
        y = torch.empty_like(x2)
        mean = torch.empty((m,), dtype=torch.float32, device=x2.device)
        rstd = torch.empty((m,), dtype=torch.float32, device=x2.device)
        L.check(L.lib().milb200_layernorm_fwd(L.ptr(x2), L.ptr(r2), L.ptr(g), L.ptr(b), L.ptr(y), L.ptr(mean),
                                              L.ptr(rstd), m, n, L.dtype_code(x2), 0, L.stream_ptr()), "layernorm_fwd")
        ctx.save_for_backward(x2, r2, g, mean, rstd)
        ctx.meta = (shp, m, n, gamma.dtype, beta.dtype, r is not None)
        return y.view(shp)

    @staticmethod
    def backward(ctx, dy):
        x2, r2, g, mean, rstd = ctx.saved_tensors
        shp, m, n, gdt, bdt, has_r = ctx.meta
        dy2 = dy.contiguous().view(m, n)
        if dy2.dtype != x2.dtype:
            dy2 = cast(dy2, x2.dtype)
        dxr = torch.empty_like(x2)
        dg = torch.empty((n,), dtype=torch.float32, device=x2.device)
        db = torch.empty((n,), dtype=torch.float32, device=x2.device)
        nb = L.lib().milb200_layernorm_workspace_bytes(m, n)
        ws = L.workspace(nb, x2.device)
        L.check(L.lib().milb200_layernorm_bwd(L.ptr(x2), L.ptr(r2), L.ptr(g), L.ptr(mean), L.ptr(rstd), L.ptr(dy2),
                                              L.ptr(dxr), L.ptr(dg), L.ptr(db), m, n, L.dtype_code(x2), 0, 0, L.ptr(ws),
                                              ws.numel(), L.stream_ptr()), "layernorm_bwd")
        gx = dxr.view(shp)
        return gx, (gx if has_r else None), cast(dg, gdt), cast(db, bdt)


def layernorm(x, gamma, beta, residual=None):
    return _LayerNorm.apply(x, residual, gamma, beta)


class _AttentionCore(torch.autograd.Function):
    """O = softmax(Q K^T / sqrt(c)) V per head (transformer.py:434-446). q [nq, H*c], k/v [nk, H*c]."""

    @staticmethod
    def forward(ctx, q, k, v, heads):
        q, k, v = q.contiguous(), k.contiguous(), v.contiguous()
        nq, C = q.shape
        nk = k.shape[0]
        c = C // heads
        o = torch.empty_like(q)
        lse = torch.empty((heads, nq), dtype=torch.float32, device=q.device)
        nb = L.lib().milb200_attention_workspace_bytes(nq, nk, heads, c, 0)
        ws = L.workspace(nb, q.device)
        L.check(L.lib().milb200_attention_fwd(L.ptr(q), L.ptr(k), L.ptr(v), L.ptr(o), L.ptr(lse), nq, nk, heads, c,
                                              L.dtype_code(q), L.ptr(ws), ws.numel(), L.stream_ptr()), "attention_fwd")
        ctx.save_for_backward(q, k, v, o, lse)
        ctx.heads = heads
        return o

    @staticmethod
    def backward(ctx, do):
        q, k, v, o, lse = ctx.saved_tensors
        heads = ctx.heads
        nq, C = q.shape
        nk = k.shape[0]
        c = C // heads
        do = do.contiguous()
        dq, dk, dv = torch.empty_like(q), torch.empty_like(k), torch.empty_like(v)
        nb = L.lib().milb200_attention_workspace_bytes(nq, nk, heads, c, 1)
        ws = L.workspace(nb, q.device)
        L.check(L.lib().milb200_attention_bwd(L.ptr(q), L.ptr(k), L.ptr(v), L.ptr(o), L.ptr(lse), L.ptr(do), L.ptr(dq),
                                              L.ptr(dk), L.ptr(dv), nq, nk, heads, c, L.dtype_code(q), L.ptr(ws),
                                              ws.numel(), L.stream_ptr()), "attention_bwd")
        return dq, dk, dv, None


def attention_core(q, k, v, heads):
    return _AttentionCore.apply(q, k, v, heads)


class _Add(torch.autograd.Function):
    @staticmethod
    def forward(ctx, a, b):
        a, b = a.contiguous(), b.contiguous()
        out = torch.empty_like(a)
        L.check(L.lib().milb200_add(L.ptr(a), L.ptr(b), L.ptr(out), a.numel(), L.dtype_code(a), L.stream_ptr()), "add")
        return out

    @staticmethod
    def backward(ctx, g):
        return g, g


def add(a, b):
    """a + b for same-shape tensors through the library's vectorised add kernel."""
    if a.shape != b.shape or a.dtype != b.dtype:
        raise L.MilB200Error("add: operands must share shape and dtype")
    return _Add.apply(a, b)


class _Axpby(torch.autograd.Function):
    @staticmethod
    def forward(ctx, a, b, alpha, beta):
        a = a.contiguous()
        b = b.contiguous() if b is not None else None
        out = torch.empty_like(a)
        L.check(L.lib().milb200_axpby(L.ptr(a), L.ptr(b), L.ptr(out), a.numel(), float(alpha), float(beta),
                                      L.dtype_code(a), L.stream_ptr()), "axpby")
        ctx.ab = (float(alpha), float(beta), b is not None)
        return out

    @staticmethod
    def backward(ctx, g):
        alpha, beta, has_b = ctx.ab
        g = g.contiguous()
        ga = _Axpby.apply(g, None, alpha, 0.0) if ctx.needs_input_grad[0] else None
        gb = _Axpby.apply(g, None, beta, 0.0) if (has_b and ctx.needs_input_grad[1]) else None
        return ga, gb, None, None


def axpby(a, b, alpha, beta):
    """alpha * a + beta * b (b may be None) — e.g. (x_CT + x_pathology) / 2 of aggregator_clip.py:94."""
    if b is not None and (a.shape != b.shape or a.dtype != b.dtype):
        raise L.MilB200Error("axpby: operands must share shape and dtype")
    return _Axpby.apply(a, b, alpha, beta)


class _CtTokens(torch.autograd.Function):
    """(1, C, T, h, w) CT feature map -> (1, T, C) tokens: mean over (h, w) then permute (transformer.py:93)."""

    @staticmethod
    def forward(ctx, fmap):
        b, c, t, h, w = fmap.shape
        if b != 1:
            raise L.MilB200Error("ct_tokens: the reference runs one bag per call (batch 1)")
        fmap = fmap.contiguous()
        out = torch.empty((1, t, c), dtype=fmap.dtype, device=fmap.device)
        L.check(L.lib().milb200_ct_tokens_fwd(L.ptr(fmap), L.ptr(out), c, t, h * w, L.dtype_code(fmap), L.stream_ptr()),
                "ct_tokens_fwd")
        ctx.shape = (b, c, t, h, w)
        return out

    @staticmethod
    def backward(ctx, g):
        b, c, t, h, w = ctx.shape
        g = g.contiguous()
        out = torch.empty((b, c, t, h, w), dtype=g.dtype, device=g.device)
        L.check(L.lib().milb200_ct_tokens_bwd(L.ptr(g), L.ptr(out), c, t, h * w, L.dtype_code(g), L.stream_ptr()),
                "ct_tokens_bwd")
        return out


def ct_tokens(fmap):
    return _CtTokens.apply(fmap)


def sinusoid_pe(n_pos, dim, dtype, device):
    """On-device sinusoidal table (aggregator.py:99-106), shape (1, n_pos, dim)."""
    pe = torch.empty((1, n_pos, dim), dtype=dtype, device=device)
    L.check(L.lib().milb200_sinusoid_pe(L.ptr(pe), n_pos, dim, L.dtype_code(pe), L.stream_ptr()), "sinusoid_pe")
    return pe


# --------------------------------------------------------------------------------------------------
# CLIP logits and the small losses
# --------------------------------------------------------------------------------------------------
class _ClipLogits(torch.autograd.Function):
    """clip/model.py:359-368: (logits_per_image, logits_per_text) = exp(logit_scale) * cos(I, T) and transpose."""

    @staticmethod
    def forward(ctx, img, txt, logit_scale):
        img, txt = img.contiguous(), txt.contiguous()
        bi, d = img.shape
        bt = txt.shape[0]
        ls = _f32(logit_scale).reshape(1).contiguous()
        li = torch.empty((bi, bt), dtype=torch.float32, device=img.device)
        ni = torch.empty((bi,), dtype=torch.float32, device=img.device)
        nt = torch.empty((bt,), dtype=torch.float32, device=img.device)
        L.check(L.lib().milb200_clip_logits_fwd(L.ptr(img), L.ptr(txt), L.ptr(ls), L.ptr(li), L.ptr(ni), L.ptr(nt), bi,
                                                bt, d, L.dtype_code(img), L.stream_ptr()), "clip_logits_fwd")
        lt = torch.empty((bt, bi), dtype=torch.float32, device=img.device)
        L.check(L.lib().milb200_transpose(L.ptr(li), L.ptr(lt), bi, bt, L.F32, L.stream_ptr()), "transpose")
        ctx.save_for_backward(img, txt, ls, li, ni, nt)
        ctx.ls_meta = (logit_scale.dtype, logit_scale.shape)
        return li, lt

    @staticmethod
    def backward(ctx, dli, dlt):
        img, txt, ls, li, ni, nt = ctx.saved_tensors
        bi, d = img.shape
        bt = txt.shape[0]
        dli = _f32(dli).contiguous() if dli is not None else None
        dlt = _f32(dlt).contiguous() if dlt is not None else None
        dI = torch.empty_like(img) if ctx.needs_input_grad[0] else None
        dT = torch.empty_like(txt) if ctx.needs_input_grad[1] else None
        dsc = torch.empty((1,), dtype=torch.float32, device=img.device) if ctx.needs_input_grad[2] else None
        L.check(L.lib().milb200_clip_logits_bwd(L.ptr(img), L.ptr(txt), L.ptr(ls), L.ptr(li), L.ptr(ni), L.ptr(nt),
                                                L.ptr(dli), L.ptr(dlt), L.ptr(dI), L.ptr(dT), L.ptr(dsc), bi, bt, d,
                                                L.dtype_code(img), L.stream_ptr()), "clip_logits_bwd")
        if dsc is not None:
            dt, shp = ctx.ls_meta
            dsc = cast(dsc, dt).view(shp)
        return dI, dT, dsc


def clip_logits(image_features, text_features, logit_scale):
    return _ClipLogits.apply(image_features, text_features, logit_scale)


class _ClipLossV1(torch.autograd.Function):
    """utils.py:277-282 given the frozen text features feat [b, I, d]: returns (loss, logits [I,b,b])."""

    @staticmethod
    def forward(ctx, out, feat):
        out, feat = out.contiguous(), feat.contiguous()
        b, d = out.shape
        n_info = feat.shape[1]
        if feat.dtype != out.dtype:
            feat = cast(feat, out.dtype)
        logits = torch.empty((n_info, b, b), dtype=torch.float32, device=out.device)
        wsb = torch.empty((2 * n_info * b,), dtype=torch.float32, device=out.device)
        loss = torch.empty((1,), dtype=torch.float32, device=out.device)
        dout = torch.empty((b, d), dtype=torch.float32, device=out.device)
        L.check(L.lib().milb200_cliploss_fwd_bwd(L.ptr(out), L.ptr(feat), L.ptr(logits), L.ptr(wsb), L.ptr(loss),
                                                 L.ptr(dout), b, n_info, d, L.dtype_code(out), L.stream_ptr()),
                "cliploss_fwd_bwd")
        ctx.save_for_backward(dout)
        ctx.odt = out.dtype
        ctx.mark_non_differentiable(logits)
        return loss.view(()), logits

    @staticmethod
    def backward(ctx, g, _gl):
        (dout,) = ctx.saved_tensors
        return cast((dout * g).contiguous(), ctx.odt) if dout.dtype != ctx.odt else dout * g, None


def cliploss_v1(output, text_features):
    return _ClipLossV1.apply(output, text_features)


class _SigmoidBCE(torch.autograd.Function):
    """prob = sigmoid(z); loss = BCELoss(prob, target) (mean) — aggregator.py:200 + train_ddp.py:99,319."""

    @staticmethod
    def forward(ctx, z, target):
        zf, tf = _f32(z).contiguous(), _f32(target).contiguous()
        n = zf.numel()
        prob = torch.empty_like(zf)
        loss = torch.empty((1,), dtype=torch.float32, device=z.device)
        dz = torch.empty_like(zf)
        L.check(L.lib().milb200_sigmoid_bce_fwd_bwd(L.ptr(zf), L.ptr(tf), L.ptr(prob), L.ptr(loss), L.ptr(dz), n,
                                                    L.stream_ptr()), "sigmoid_bce")
        ctx.save_for_backward(dz)
        ctx.zdt = z.dtype
        ctx.mark_non_differentiable(prob)
        return loss.view(()), prob

    @staticmethod
    def backward(ctx, g, _gp):
        (dz,) = ctx.saved_tensors
        out = dz * g
        return (out if ctx.zdt == torch.float32 else cast(out.contiguous(), ctx.zdt)), None


def sigmoid_bce(logits, target):
    """Returns (loss, prob)."""
    return _SigmoidBCE.apply(logits, target)


class _CosineEmbeddingLoss(torch.autograd.Function):
    """nn.CosineEmbeddingLoss(a, b, target=+1) = mean(1 - cos(a_i, b_i)) (train_ddp.py:102,326)."""

    @staticmethod
    def forward(ctx, a, b):
        a, b = a.contiguous(), b.contiguous()
        n, d = a.shape
        loss = torch.empty((1,), dtype=torch.float32, device=a.device)
        rows = torch.empty((n,), dtype=torch.float32, device=a.device)
        da, db = torch.empty_like(a), torch.empty_like(b)
        L.check(L.lib().milb200_cosine_embedding_fwd_bwd(L.ptr(a), L.ptr(b), L.ptr(loss), L.ptr(rows), L.ptr(da),
                                                         L.ptr(db), n, d, L.dtype_code(a), L.stream_ptr()),
                "cosine_embedding")
        ctx.save_for_backward(da, db)
        return loss.view(())

    @staticmethod
    def backward(ctx, g):
        da, db = ctx.saved_tensors
        return da * g.to(da.dtype), db * g.to(db.dtype)


def cosine_embedding_loss(a, b):
    return _CosineEmbeddingLoss.apply(a, b)
