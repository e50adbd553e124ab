"""Data-parallel training step for the gated-attention MIL pool (train_ddp.py:79,346-348 shape):
bags shard across ranks, parameters are replicated, and the ONLY exchange is one all-reduce of a flat
fp32 gradient buffer per step, followed by a fused Adam kernel (the 1/world scaling of DDP's gradient
average is folded into it).  The backward kernels write straight into the flat buffer, so there are no
gradient buckets, hooks or unused-parameter bitmaps.

Flat layout (fp32), chosen so that [Wv; Wu] is the contiguous Wcat operand the kernels want:
    Wv (D*L) | Wu (D*L) | bv (D) | bu (D) | ww (D) | bw (1)
"""
from __future__ import annotations

import torch

from . import _lib as L
from . import functional as F


def shard_bags(lengths, rank, world, balance=True):
    """Indices of the bags rank `rank` owns.  balance=False is DistributedSampler's stride (train_ddp.py:191:
    rank, rank+world, ...).  balance=True assigns bags longest-first to the rank with the fewest instances so far
    (bag sizes span 200x, so equal bag COUNTS would leave ranks idle at the all-reduce); ties go to the lowest rank,
    which makes the assignment a pure function of `lengths` — every rank computes the same partition locally."""
    n = len(lengths)
    if not balance:
        return list(range(rank, n, world))
    order = sorted(range(n), key=lambda i: (-int(lengths[i]), i))
    load = [0] * world
    owner = [0] * n
    for i in order:
        r = min(range(world), key=lambda q: (load[q], q))
        owner[i] = r
        load[r] += int(lengths[i])
    return [i for i in range(n) if owner[i] == rank]


def flat_layout(L_feat, D):
    """Element ranges of the flat fp32 parameter/gradient buffer, keyed by the reference's state_dict names."""
    o = 2 * D * L_feat
    return {"attention_V.0.weight": (0, D * L_feat), "attention_U.0.weight": (D * L_feat, o),
            "attention_V.0.bias": (o, o + D), "attention_U.0.bias": (o + D, o + 2 * D),
            "attention_weights.weight": (o + 2 * D, o + 3 * D), "attention_weights.bias": (o + 3 * D, o + 3 * D + 1)}


class AbmilTrainer:
    def __init__(self, L_feat=1024, D=192, compute_dtype=torch.bfloat16, lr=1e-5, betas=(0.9, 0.999), eps=1e-8,
                 weight_decay=1e-7, device="cuda", process_group=None, world_size=1, need_input_grad=False,
                 save_gate=True, optimizer="adam", dropout_p=0.0):
        self.L, self.D = L_feat, D
        self.dtype = compute_dtype
        self.device = torch.device(device)
        self.lr, self.betas, self.eps, self.wd = lr, betas, eps, weight_decay
        self.pg, self.world = process_group, world_size
        self.need_input_grad = need_input_grad
        if optimizer not in ("adam", "sgd"):
            raise ValueError("optimizer must be 'adam' (train_ddp.py:113-116) or 'sgd' (train_ddp.py:105-108)")
        self.optimizer = optimizer
        # train-mode semantics of ABMIL.forward (ABMIL.py:49: Dropout(p=0.5) on the INSTANCES before both GEMMs and the
        # pool): the masked copy of X has to exist in memory because TMA feeds the GEMMs straight from it, so it costs
        # one elementwise pass (Philox mask, seed drawn from torch's generator per step).  0 = eval-mode semantics.
        self.dropout_p = float(dropout_p)
        self.phase_hook = None
        self.save_gate = save_gate     # keep V,U from the forward (memory) instead of re-running the GEMM (time)
        n = 2 * D * L_feat + 3 * D + 1
        self.numel = n
        self.params = torch.zeros(n, dtype=torch.float32, device=self.device)
        self.grads = torch.zeros(n, dtype=torch.float32, device=self.device)
        self.exp_avg = torch.zeros(n, dtype=torch.float32, device=self.device)
        self.exp_avg_sq = torch.zeros(n, dtype=torch.float32, device=self.device)
        self.step_count = 0
        self._wcat_c = torch.empty((2 * D, L_feat), dtype=compute_dtype, device=self.device)
        self._bcat_c = torch.empty((2 * D,), dtype=torch.float32, device=self.device)

    # ---- views into the flat buffers -----------------------------------------------------------
    def _views(self, flat):
        D, Lf = self.D, self.L
        o = 2 * D * Lf
        return dict(Wcat=flat[:o].view(2 * D, Lf), bcat=flat[o:o + 2 * D], ww=flat[o + 2 * D:o + 3 * D],
                    bw=flat[o + 3 * D:o + 3 * D + 1])

    def load_from(self, module):
        """Copy an ABMIL module's parameters (reference state_dict names) into the flat buffer."""
        v = self._views(self.params)
        D = self.D
        with torch.no_grad():
            v["Wcat"][:D].copy_(module.attention_V[0].weight)
            v["Wcat"][D:].copy_(module.attention_U[0].weight)
            v["bcat"][:D].copy_(module.attention_V[0].bias)
            v["bcat"][D:].copy_(module.attention_U[0].bias)
            v["ww"].copy_(module.attention_weights.weight.reshape(-1))
            v["bw"].copy_(module.attention_weights.bias.reshape(-1))

    def store_to(self, module):
        v = self._views(self.params)
        D = self.D
        with torch.no_grad():
            module.attention_V[0].weight.copy_(v["Wcat"][:D])
            module.attention_U[0].weight.copy_(v["Wcat"][D:])
            module.attention_V[0].bias.copy_(v["bcat"][:D])
            module.attention_U[0].bias.copy_(v["bcat"][D:])
            module.attention_weights.weight.copy_(v["ww"].view(1, D))
            module.attention_weights.bias.copy_(v["bw"])

    def grad_views(self):
        return self._views(self.grads)

    def broadcast_params(self):
        """DDP's constructor broadcast (rank 0 -> all), once."""
        if self.world > 1:
            torch.distributed.broadcast(self.params, src=0, group=self.pg)

    # ---- one training step ---------------------------------------------------------------------
    def forward(self, X, offsets):
        """Forward of the pool over one packed CSR batch; keeps what `backward` needs.  Returns M fp32 [B, L]."""
        return self._forward(X, offsets, None)

    def _forward(self, X, offsets, dM):
        """`forward`; with the upstream gradient dM already known (forward_backward), the pooling pass also takes the
        backward's row dots dM_b . x_i from the rows it streams, so that the backward does not read X again."""
        v = self._views(self.params)
        # fp32 master -> compute-dtype operand in the row order the kernels expect (one tiny kernel)
        D = self.D
        L.check(L.lib().milb200_pack_gate_weights(L.ptr(v["Wcat"][:D]), L.ptr(v["Wcat"][D:]), L.ptr(v["bcat"][:D]),
                                                  L.ptr(v["bcat"][D:]), L.F32, self.L, D, L.ptr(self._wcat_c),
                                                  L.dtype_code(self._wcat_c), L.ptr(self._bcat_c), L.stream_ptr()),
                "pack_gate_weights")
        Wcat, bcat = self._wcat_c, self._bcat_c
        mark = self.phase_hook or (lambda name: None)     # measurement only: bench.py records a CUDA event per phase
        mark("pack")
        seed = None
        if self.dropout_p > 0.0:
            seed = int(torch.randint(0, 2 ** 62, (1,), dtype=torch.int64).item())
            X = F._dropout_raw(X.contiguous(), self.dropout_p, seed, 0)
            mark("dropout")
        if self.save_gate:
            s, act = F.gated_scores(X, Wcat, bcat, v["ww"], v["bw"], save=True)
        else:
            s, act = F.gated_scores(X, Wcat, bcat, v["ww"], v["bw"]), None
        mark("gated_score_fwd")
        if dM is None:
            M, _, am, _ = F.segment_softmax_pool(X, s, offsets)
            rowdot = None
        else:
            M, _, am, _, rowdot = F.segment_softmax_pool_rowdot(X, s, offsets, dM)
        mark("segment_softmax_pool_fwd")
        self._saved = (X, offsets, s, act, M, v, seed, rowdot)
        self.last_argmax, self.last_scores = am, s
        return M

    def backward(self, dM):
        """Backward of the last `forward` given dL/dM [B, L] fp32: parameter gradients go to the flat buffer; returns
        dL/dX (or None when the trainer was built without need_input_grad)."""
        X, offsets, s, act, M, v, seed, rowdot = self._saved
        self._saved = None
        mark = self.phase_hook or (lambda name: None)
        if rowdot is not None:
            # ds_i = a_i (dM_b . x_i - dM_b . M_b) from the forward's row dots: no pass over X
            ds, attn = F.segment_softmax_pool_bwd_rowdot(s, offsets, dM, M, rowdot, want_attn=self.need_input_grad)
            mark("pool_bwd_rowdot")
        else:
            ds, attn = F.segment_softmax_pool_bwd(X, s, offsets, dM, M, want_attn=self.need_input_grad)
            mark("segment_softmax_pool_bwd")
        dX, *_ = F.gated_scores_bwd(X, self._wcat_c, self._bcat_c, v["ww"], v["bw"], ds, attn, dM, offsets,
                                    self.need_input_grad, grad_out=self.grads, gate_act=act)
        mark("gate_bwd")
        if dX is not None and seed is not None:
            # dX above is the gradient w.r.t. the DROPPED instances; the dropout's own backward is the same Philox mask
            # and 1/(1-p) scale applied to it (nothing was stored: the mask is a function of the step's seed)
            dX = F._dropout_raw(dX, self.dropout_p, seed, 0)
            mark("dropout_bwd")
        return dX

    def forward_backward(self, X, offsets, dM=None):
        """Forward + backward of the pool over one packed CSR batch.  Upstream gradient dM defaults to ones
        (loss = sum of the pooled vectors).  Returns (M fp32 [B, L], dX or None).
        dM is known before the forward here, so the forward takes the pooling backward's row dots and the backward
        never re-reads X (one pass over X fewer than `forward` + `backward`, same results bit for bit)."""
        if dM is None:
            shape = (offsets.numel() - 1, self.L)
            if getattr(self, "_ones", None) is None or tuple(self._ones.shape) != shape:
                self._ones = torch.ones(shape, dtype=torch.float32, device=X.device)
            dM = self._ones
        M = self._forward(X, offsets, dM)
        return M, self.backward(dM)

    # ---- latency-optimal exchange: symmetric memory + one kernel (csrc/exchange.cu) ------------------------------------
    def enable_symmetric_exchange(self):
        """Move the flat gradient buffer into symmetric memory (one allocation mapped on every rank of the node, with a
        multicast mapping through the NVSwitch) so that `reduce_and_update` becomes ONE kernel: in-switch reduction +
        broadcast of the gradients and the fused optimiser step (csrc/exchange.cu), instead of an NCCL all-reduce launch
        followed by the optimiser launch.  torch.distributed's symmetric memory is the plumbing (allocation, handle
        exchange, signal pads); returns False — and leaves the NCCL path in place — when the node has no multicast
        support.  Collective: every rank of the group must call it."""
        if self.world <= 1:
            return False
        try:
            import torch.distributed._symmetric_memory as symm
            group = self.pg if self.pg is not None else torch.distributed.group.WORLD
            pad = 4 * self.world
            n_alloc = (self.numel + pad - 1) // pad * pad
            buf = symm.empty(n_alloc, dtype=torch.float32, device=self.device)
            buf.zero_()
            hdl = symm.rendezvous(buf, group.group_name)
            mc = int(getattr(hdl, "multicast_ptr", 0) or 0)
            ok = torch.tensor([1 if mc else 0], device=self.device)
        except Exception:
            buf = hdl = None
            mc = 0
            ok = torch.tensor([0], device=self.device)
        torch.distributed.all_reduce(ok, op=torch.distributed.ReduceOp.MIN, group=self.pg)     # all ranks or none
        if int(ok.item()) == 0:
            return False
        buf[:self.numel].copy_(self.grads)
        self.grads = buf[:self.numel]
        pads = torch.tensor([int(p) for p in hdl.signal_pad_ptrs], dtype=torch.int64, device=self.device)
        self._symm = dict(hdl=hdl, buf=buf, pads=pads, mc=mc, rank=int(hdl.rank))
        torch.cuda.synchronize()
        torch.distributed.barrier(group=self.pg)       # every rank's buffer is zeroed and mapped before the first exchange
        return True

    def allreduce_grads(self):
        """The path's only exchange: ONE all-reduce(sum) of the flat gradient buffer (NCCL on GPUs; any backend)."""
        if self.world > 1:
            torch.distributed.all_reduce(self.grads, group=self.pg)

    def reduce_and_update(self):
        """all-reduce(sum) of the flat gradient over NCCL, then the fused optimiser step with grad_scale = 1/world."""
        sm = getattr(self, "_symm", None)
        sd = getattr(self, "_step_dev", None)        # device-resident step counter (graphed steps), else None
        if sd is not None:
            L.check(L.lib().milb200_step_counter_inc(L.ptr(sd), L.stream_ptr()), "step_counter_inc")
        if sm is not None:
            self.step_count += 1
            L.check(L.lib().milb200_allreduce_update_symm(
                L.ptr(self.params), L.ptr(self.grads), sm["mc"], L.ptr(sm["pads"]), 0, sm["rank"], self.world,
                L.ptr(self.exp_avg), L.ptr(self.exp_avg_sq), self.numel, 1 if self.optimizer == "sgd" else 0, self.lr,
                self.betas[0], self.betas[1], self.eps, self.wd, 1.0 / self.world, self.step_count, L.ptr(sd),
                L.stream_ptr()), "allreduce_update_symm")
            return
        self.allreduce_grads()
        self.step_count += 1
        if self.optimizer == "adam" and sd is not None:
            L.check(L.lib().milb200_adam_step_dev(L.ptr(self.params), L.ptr(self.grads), L.ptr(self.exp_avg),
                                                  L.ptr(self.exp_avg_sq), self.numel, self.lr, self.betas[0], self.betas[1],
                                                  self.eps, self.wd, 1.0 / self.world, L.ptr(sd), L.stream_ptr()),
                    "adam_step_dev")
            return
        if self.optimizer == "sgd":
            L.check(L.lib().milb200_sgd_step(L.ptr(self.params), L.ptr(self.grads), self.numel, self.lr, self.wd,
                                             1.0 / self.world, L.stream_ptr()), "sgd_step")
            return
        L.check(L.lib().milb200_adam_step(L.ptr(self.params), L.ptr(self.grads), L.ptr(self.exp_avg),
                                          L.ptr(self.exp_avg_sq), self.numel, self.lr, self.betas[0], self.betas[1],
                                          self.eps, self.wd, 1.0 / self.world, self.step_count, L.stream_ptr()),
                "adam_step")

    def step(self, X, offsets, dM=None):
        M, dX = self.forward_backward(X, offsets, dM)
        self.reduce_and_update()
        return M

    def step_graphed(self, X, offsets):
        """`step(X, offsets)` replayed as ONE CUDA graph (forward, backward, exchange, optimiser: ~10 kernels, no host work
        between them).  A graph is captured per (X, offsets) address and shape — the bench's device-resident loop and its
        two rotating end-to-end buffers; data loaders that hand out fresh addresses should stage into fixed buffers first.
        The Adam step number moves to device memory (the graph must not bake the bias corrections in).  Falls back to the
        eager step for train-mode dropout (host-drawn seeds) and for an NCCL exchange (captured collectives are left to
        the caller's NCCL settings).  The first call for an address additionally runs two eager warm-up steps whose effect on the
        parameters, the optimiser state and the step counters is undone before the capture: every call is ONE step."""
        if self.dropout_p > 0.0 or self.phase_hook is not None or (self.world > 1 and getattr(self, "_symm", None) is None):
            return self.step(X, offsets)
        if getattr(self, "_step_dev", None) is None:
            self._step_dev = torch.full((1,), self.step_count, dtype=torch.int32, device=self.device)
            self._graphs = {}
        key = (X.data_ptr(), offsets.data_ptr(), tuple(X.shape), int(offsets.numel()))
        ent = self._graphs.get(key)
        first = ent is None
        if first:
            if len(self._graphs) >= 4:
                self._graphs.pop(next(iter(self._graphs)))
            # two eager steps on a side stream create every lazily allocated buffer; they must not count as training:
            # parameters, optimiser state and both step counters are restored before the capture
            state = [t.clone() for t in (self.params, self.exp_avg, self.exp_avg_sq, self._step_dev)]
            count = self.step_count
            side = torch.cuda.Stream(device=self.device)
            side.wait_stream(torch.cuda.current_stream(self.device))
            with torch.cuda.stream(side):
                for _ in range(2):
                    self.step(X, offsets)
                for dst, src in zip((self.params, self.exp_avg, self.exp_avg_sq, self._step_dev), state):
                    dst.copy_(src)
            torch.cuda.current_stream(self.device).wait_stream(side)
            l0 = L.launch_count()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                M = self.step(X, offsets)
            self.step_count = count                             # nothing has run yet
            ent = self._graphs[key] = (g, M, self.last_argmax, self.last_scores, L.launch_count() - l0)
        g, M, am, s, n_kernels = ent
        g.replay()
        if not first:
            L.lib().milb200_count_launches(n_kernels)           # (the capture itself counted the first replay's kernels)
        self.step_count += 1
        self.last_argmax, self.last_scores = am, s
        return M
