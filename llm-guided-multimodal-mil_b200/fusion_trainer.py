"""Native training step of the CT + pathology `aggregator` (BASELINE configs[2]; train_ddp.py:297-348):

    prob, x_CT2CI, x_Pth2CI = model([x_ct, x_path], x_text)
    loss = BCELoss(prob, label) + CosineEmbeddingLoss(x_CT2CI, x_Pth2CI, +1)
    loss.backward(); all-reduce(grads); Adam / SGD

without the autograd graph: every parameter of the branch lives in ONE flat fp32 buffer (fusion-program parameters |
gated pool | head), the backward kernels write into ONE flat gradient buffer, DDP's exchange is ONE all-reduce and the
optimiser ONE kernel — the same design as `dp.AbmilTrainer`, which this class embeds for the gated pool, the head and
the BCE: the program's packed bag goes through `AbmilTrainer.forward_backward_labels`, whose pooling pass takes the
head's row dots, so the pool's backward does not read the bag again.  `load_from` / `store_to` move parameters from /
to the reference-shaped module, so checkpoints keep the reference's state_dict.  The head takes 1..8 classes.

With one clinical-text token per patient (the reference's active prompt configuration) the step runs the COLLAPSED
program (csrc/xfusion.cu: no projected image tokens, the CT bag and the pathology bag as segments of one launch set,
fp32 token side / key stream, bf16 only for the patch features, the packed bag and the tensor-core GEMMs) and takes
B <= 8 patients per step (`step_bags`): the reference is batch-1 per rank (train_ddp.py:75); several patients per launch
set amortise the ~150 small token-side launches.  The loss of a B-patient step is the mean over patients of the
per-patient loss (BCELoss / CosineEmbeddingLoss with their default mean reduction over the batch).  With T > 1 tokens
the projected-keys program of round 1 is used (one patient per step).

train_mode=True applies the reference's two regularisers (ABMIL.py:49 Dropout(0.5) on the packed bag, aggregator.py:
128-131 Dropout(0.25) on the pooled vector) with Philox masks regenerated in the backward; the default reproduces
model.eval() arithmetic (what the parity tests and the bench's headline compare).
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib as L
from .dp import AbmilTrainer, flat_layout
from .model.sam.transformer import _use_collapsed


def _ptrs(n):
    return (C.c_void_p * n)()


class FusionTrainer:
    def __init__(self, model, n_text_tokens=1, compute_dtype=torch.bfloat16, lr=1e-5, betas=(0.9, 0.999), eps=1e-8,
                 weight_decay=1e-7, optimizer="adam", process_group=None, world_size=1, cosine_loss=True, train_mode=False):
        if not hasattr(model, "_fusion_tape") or not hasattr(model, "aggregator"):
            raise L.MilB200Error("FusionTrainer needs the CT+pathology `aggregator` with a gated-attention pool")
        if optimizer not in ("adam", "sgd"):
            raise ValueError("optimizer must be 'adam' or 'sgd'")
        self.model, self.T = model, int(n_text_tokens)
        self.dtype = compute_dtype
        self.device = model.fc[1].weight.device
        self.lr, self.betas, self.eps, self.wd, self.optimizer = lr, betas, eps, weight_decay, optimizer
        self.pg, self.world = process_group, world_size
        self.cosine_loss = cosine_loss
        self.train_mode = bool(train_mode)
        self.E = model.embedding_dim
        self.C = model.fc[1].weight.shape[0]
        if not 1 <= self.C <= 8:
            raise ValueError(f"FusionTrainer trains 1..8 classes (the pooling pass takes up to 8 head row dots per row), "
                             f"got num_classes = {self.C}")
        self.collapsed = self.T == 1 and _use_collapsed()
        self.tape = model._fusion_tape_v2() if self.collapsed else model._fusion_tape(single_token=(self.T == 1))
        c = self.tape._freeze()
        self.n_tape = c["total"]
        # the gated pool, the head and the BCE run through AbmilTrainer's labelled step on views of the same flat buffers
        # (its instances are the program's output, so it also gives the gradient of the packed bag)
        self.pool = AbmilTrainer(self.E, model.aggregator.attention_V[0].weight.shape[0], compute_dtype, device=self.device,
                                 need_input_grad=True, head_classes=self.C,
                                 dropout_p=(model.aggregator.dropout1.p if self.train_mode else 0.0),
                                 head_dropout=(model.fc[0].p if self.train_mode else 0.0))
        up8 = lambda n: (n + 7) // 8 * 8
        self.o_pool = up8(self.n_tape)
        self.numel = up8(self.o_pool + self.pool.numel)
        z = lambda: torch.zeros(self.numel, dtype=torch.float32, device=self.device)
        self.params, self.grads, self.exp_avg, self.exp_avg_sq = z(), z(), z(), z()
        sl = slice(self.o_pool, self.o_pool + self.pool.numel)
        self.pool.params, self.pool.grads = self.params[sl], self.grads[sl]
        self.wc = torch.empty(self.n_tape, dtype=compute_dtype, device=self.device) if compute_dtype != torch.float32 else None
        self.step_count = 0
        self._buf = {}
        self.load_from(model)

    # ---- parameters <-> module ----------------------------------------------------------------------------------
    def _module_tensors(self):
        """(flat offset, tensor) for every parameter of the fusion program, in flat-buffer order."""
        c = self.tape._freeze()
        return [(off, p) for p, off in zip(self.tape.params, c["offsets"])]

    @torch.no_grad()
    def load_from(self, model=None):
        for off, p in self._module_tensors():
            self.params[off:off + p.numel()].copy_(p.detach().reshape(-1))
        self.pool.load_from(self.model.aggregator, head=self.model.fc[1])
        self._refresh_compute_copy()

    @torch.no_grad()
    def store_to(self, model=None):
        for off, p in self._module_tensors():
            p.copy_(self.params[off:off + p.numel()].view(p.shape))
        self.pool.store_to(self.model.aggregator, head=self.model.fc[1])

    def named_grads(self):
        """{state_dict name: gradient view} for the tests (program parameters by module name, the pool under aggregator.*,
        the head under fc.1.*)."""
        params = dict(self.model.named_parameters())
        names = {id(p): n for n, p in params.items()}
        out = {names[id(p)]: self.grads[off:off + p.numel()].view(p.shape) for off, p in self._module_tensors()}
        for k, (a, b) in flat_layout(self.E, self.pool.D, self.C).items():
            name = "fc.1." + k[len("head."):] if k.startswith("head.") else "aggregator." + k
            out[name] = self.pool.grads[a:b].view(params[name].shape)
        return out

    def _refresh_compute_copy(self):
        if self.wc is not None:
            L.check(L.lib().milb200_cast(L.ptr(self.params), L.F32, L.ptr(self.wc), L.dtype_code(self.wc), self.n_tape,
                                         L.stream_ptr()), "cast")

    def broadcast_params(self):
        if self.world > 1:
            torch.distributed.broadcast(self.params, src=0, group=self.pg)
            self._refresh_compute_copy()

    # ---- buffers (pointer-stable, so a repeated step shape replays as a CUDA graph) ------------------------------------
    CAP_ROWS = 4096        # pathology rows are rounded up to this granule when sizing buffers

    def _buffers(self, key, rows, segs, n_bags, bag_off):
        """Buffers for a step.  Sized by CAPACITY (the packed pathology rows rounded up to CAP_ROWS), not by the exact shape:
        real cohorts have a different row count per patient, and a fresh multi-hundred-MB arena per new shape would turn
        every step into an allocation.  Steps whose shapes fall into the same capacity share one set of buffers (the
        kernels get exact row counts and pointers to the heads of the buffers); exact repeats replay as CUDA graphs."""
        b = self._buf.get(key)
        if b is None:
            if len(self._buf) >= 4:
                self._buf.pop(next(iter(self._buf)))
            t, c, lib = self.tape, self.tape._freeze(), L.lib()
            code = L.BF16 if self.dtype == torch.bfloat16 else L.F32
            dev = self.device
            cap = dict(rows)
            if self.collapsed:          # capacity image of the row counts: every slot at least as large as any shape of the bucket
                extra = key[2] - rows["NP"]
                for k in ("NP", "NK", "NBAG"):
                    cap[k] = rows[k] + extra
            slots_cap = t._slots(cap)
            segp = t._segments(segs)
            mk = lambda r, cc, dt=None: torch.empty((int(r), int(cc)), dtype=dt or self.dtype, device=dev)
            sdt = lambda s: torch.float32 if t.slot_f32[s] else self.dtype
            B, T, E = n_bags, self.T, self.E
            f32 = torch.float32
            b = dict(code=code,
                     arena=torch.empty(lib.milb200_tape_arena_bytes(c["ops"], c["n_ops"], slots_cap, c["n_slots"], code, segp),
                                       dtype=torch.uint8, device=dev),
                     out=[mk(fn(cap), cols, t.buffer_dtype(i, self.dtype)) for i, (fn, cols) in enumerate(t.buffers)],
                     # (the cached position tables are used in place: no staging buffer for them)
                     stage=[None if j in ((2,) if self.collapsed else (1, 3)) else mk(slots_cap[s].rows, slots_cap[s].cols, sdt(s))
                            for j, s in enumerate(t.inputs)],
                     loss=torch.zeros(2, dtype=f32, device=dev),
                     cos_rows=torch.empty(max(B * T, 1), dtype=f32, device=dev),
                     da=mk(B * T, E), db=mk(B * T, E), offsets={})
            if self.collapsed:      # gradient of the fp32 token rows [CT segments | pathology segments]: the cosine loss's
                b["dtok"] = torch.zeros((2 * B * T, E), dtype=f32, device=dev)
            self._buf[key] = b
        off_key = tuple(bag_off)
        if off_key not in b["offsets"]:
            if len(b["offsets"]) > 256:
                b["offsets"].clear()
            b["offsets"][off_key] = torch.tensor(bag_off, dtype=torch.int32, device=self.device)
        return b, self.tape._slots(rows), self.tape._segments(segs), b["offsets"][off_key]

    # ---- forward + backward ------------------------------------------------------------------------------------------
    def forward_backward(self, ct_tokens, x_path, x_text, label):
        """One patient: ct_tokens (Nc, E) per-slice CT tokens (F.ct_tokens of the encoder's feature map); x_path (Np, 768)
        patch features; x_text (T, E) clinical-text embeddings; label (C,) one-hot float.  All on the device, compute dtype.
        Leaves the gradients in `self.grads`; returns (loss tensor [2] = (BCE, cosine), prob (1, C))."""
        if self.collapsed:
            return self.forward_backward_bags(ct_tokens.unsqueeze(0), x_path, [x_path.shape[0]], x_text.reshape(1, self.E),
                                              label.reshape(1, self.C))
        return self._forward_backward_projected(ct_tokens, x_path, x_text, label)

    def forward_backward_bags(self, ct_tokens, x_path, path_lens, x_text, labels):
        """B <= 8 patients in one launch set (collapsed program, T = 1): ct_tokens (B, Nc, E); x_path (sum Np, 768) packed
        row-wise; path_lens host ints; x_text (B, E); labels (B, C) one-hot float.  Returns (loss [2], prob (B, C))."""
        if not self.collapsed:
            raise L.MilB200Error("forward_backward_bags needs the collapsed program (one text token per patient)")
        m, t, lib = self.model, self.tape, L.lib()
        B, Nc = int(ct_tokens.shape[0]), int(ct_tokens.shape[1])
        path_lens = [int(n) for n in path_lens]
        if len(path_lens) != B or 2 * B > L.MAX_SEGMENTS or x_path.shape[0] != sum(path_lens) or min(path_lens) < 2 or Nc < 2:
            raise L.MilB200Error("forward_backward_bags: 1..8 patients, x_path packed (sum Np, 768), bags of >= 2 rows")
        rows, segs, bag_off = m.fusion_layout(Nc, path_lens, 1)
        pe = m._pe_table(max(Nc, max(path_lens)), self.device)
        rows["NPE"] = pe.shape[0]
        n_p = rows["NP"]
        key = (B, Nc, (n_p + self.CAP_ROWS - 1) // self.CAP_ROWS * self.CAP_ROWS)
        b, slots, segp, offsets = self._buffers(key, rows, segs, B, bag_off)
        c = t._freeze()
        code, n_slots = b["code"], c["n_slots"]
        E, Cn = self.E, self.C
        # inputs -> pointer-stable staging (program order: patch features, CT tokens fp32, position table, text fp32)
        st_xp, st_ct, _, st_txt = b["stage"]
        st_xp = st_xp[:n_p]
        st_xp.copy_(x_path)
        for src, dst in ((ct_tokens.reshape(B * Nc, E), st_ct), (x_text.reshape(B, E), st_txt)):
            src = src.contiguous()
            if src.dtype == torch.float32:
                dst.copy_(src)
            else:
                L.check(lib.milb200_cast(L.ptr(src), L.dtype_code(src), L.ptr(dst), L.F32, src.numel(), L.stream_ptr()), "cast")
        inputs = [st_xp, st_ct, pe, st_txt]
        wcomp = self.wc if self.wc is not None else self.params
        ext = _ptrs(n_slots)
        for s, x in zip(t.inputs, inputs):
            ext[s] = x.data_ptr()
        bag, tok = b["out"][0][:rows["NBAG"]], b["out"][1]
        for s, bi, fn in t.outputs:
            ext[s] = b["out"][bi].data_ptr()
        ws = L.workspace(lib.milb200_tape_workspace_bytes(c["ops"], c["n_ops"], slots, n_slots, code, 0, segp), self.device)
        L.check(lib.milb200_tape_forward(c["ops"], c["n_ops"], slots, n_slots, c["params"], c["n_params"], ext, L.ptr(wcomp),
                                         L.ptr(self.params), L.ptr(b["arena"]), b["arena"].numel(), L.ptr(ws), ws.numel(),
                                         code, segp, L.stream_ptr()), "tape_forward")
        _, prob = self.pool.forward_backward_labels(bag, offsets, labels.reshape(B, Cn).to(torch.float32).contiguous(),
                                                    loss=b["loss"][0:1])
        # the program's backward replays as a CUDA graph keyed by its pointers: without the pool trainer's reference the
        # next step's gradient of the packed bag reuses this block instead of alternating between two addresses
        dbag, self.pool.last_dX = self.pool.last_dX, None
        dtok = b["dtok"]
        if not self.cosine_loss:
            dtok.zero_()                  # the backward accumulates into the seeded buffers in place
        else:
            # x_CT2CI = token rows [0, B), x_Pth2CI = rows [B, 2B) of the fp32 token output (aggregator.py:160,168); the
            # loss and its gradients stay fp32 and seed the token rows directly
            L.check(lib.milb200_cosine_embedding_fwd_bwd(L.ptr(tok[:B]), L.ptr(tok[B:]), L.ptr(b["loss"][1:2]),
                                                         L.ptr(b["cos_rows"]), L.ptr(dtok[:B]), L.ptr(dtok[B:]), B, E, L.F32,
                                                         L.stream_ptr()), "cosine_embedding")
        # backward of the fusion program: the gradients of the packed bag and of the token rows are seeded IN PLACE
        ext2, gext, seeds = _ptrs(n_slots), _ptrs(n_slots), _ptrs(n_slots)
        for s, x in zip(t.inputs, inputs):
            ext2[s] = x.data_ptr()
        for s, bi, fn in t.outputs:
            ext2[s] = b["out"][bi].data_ptr()
            seeds[s] = gext[s] = (dbag if bi == 0 else dtok).data_ptr()
        ws = L.workspace(lib.milb200_tape_workspace_bytes(c["ops"], c["n_ops"], slots, n_slots, code, 1, segp), self.device)
        L.check(lib.milb200_tape_backward(c["ops"], c["n_ops"], slots, n_slots, c["params"], c["n_params"], ext2, gext, seeds,
                                          L.ptr(wcomp), L.ptr(self.params), L.ptr(self.grads), L.ptr(b["arena"]),
                                          b["arena"].numel(), L.ptr(ws), ws.numel(), code, segp, L.stream_ptr()),
                "tape_backward")
        return b["loss"], prob

    # ---- the projected-keys program of round 1 (T > 1, or MILB200_FUSION_COLLAPSED=0): one patient per step -------------
    def _forward_backward_projected(self, ct_tokens, x_path, x_text, label):
        m, t, lib = self.model, self.tape, L.lib()
        T, Nc, Np = x_text.shape[0], ct_tokens.shape[0], x_path.shape[0]
        if T != self.T:
            raise L.MilB200Error(f"FusionTrainer was built for {self.T} text token(s), got {T}")
        rows = {"T": T, "Nc": Nc, "Np": Np}
        b, slots, _, offsets = self._buffers(tuple(sorted(rows.items())), rows, None, 1, [0, 2 * T + Nc + Np])
        c = t._freeze()
        code, n_slots = b["code"], c["n_slots"]
        like = x_text
        srcs = [ct_tokens, m._pe(Nc, like)[0], x_path, m._pe(Np, like)[0], x_text]
        inputs = []
        for j, (src, st) in enumerate(zip(srcs, b["stage"])):
            if j in (1, 3):                      # cached position tables: stable address, used in place
                inputs.append(src.contiguous())
            else:
                st.copy_(src)
                inputs.append(st)
        wcomp = self.wc if self.wc is not None else self.params
        esz = inputs[0].element_size()
        ext = _ptrs(n_slots)
        for s, x in zip(t.inputs, inputs):
            ext[s] = x.data_ptr()
        for s, bi, fn in t.outputs:
            ext[s] = b["out"][bi].data_ptr() + int(fn(rows)) * t.slot_cols[s] * esz
        ws = L.workspace(lib.milb200_tape_workspace_bytes(c["ops"], c["n_ops"], slots, n_slots, code, 0, None), self.device)
        L.check(lib.milb200_tape_forward(c["ops"], c["n_ops"], slots, n_slots, c["params"], c["n_params"], ext, L.ptr(wcomp),
                                         L.ptr(self.params), L.ptr(b["arena"]), b["arena"].numel(), L.ptr(ws), ws.numel(),
                                         code, None, L.stream_ptr()), "tape_forward")
        bag = b["out"][0]                                                     # aggregator.py:173 row order
        _, prob = self.pool.forward_backward_labels(bag, offsets, label.reshape(1, self.C).to(torch.float32).contiguous(),
                                                    loss=b["loss"][0:1])
        dbag, self.pool.last_dX = self.pool.last_dX, None                    # (see forward_backward_bags)
        if self.cosine_loss:
            a_rows, b_rows = bag[0:T], bag[T + Nc:2 * T + Nc]                 # x_CT2CI, x_Pth2CI (aggregator.py:160,168)
            L.check(lib.milb200_cosine_embedding_fwd_bwd(L.ptr(a_rows), L.ptr(b_rows), L.ptr(b["loss"][1:2]),
                                                         L.ptr(b["cos_rows"]), L.ptr(b["da"]), L.ptr(b["db"]), T, self.E,
                                                         code, L.stream_ptr()), "cosine_embedding")
            for rows_view, g in ((dbag[0:T], b["da"]), (dbag[T + Nc:2 * T + Nc], b["db"])):     # both losses reach these rows
                L.check(lib.milb200_add(L.ptr(rows_view), L.ptr(g), L.ptr(rows_view), T * self.E, code, L.stream_ptr()), "add")
        # backward of the fusion program, seeded in place with the gradient of the packed bag
        ext2, gext, seeds = _ptrs(n_slots), _ptrs(n_slots), _ptrs(n_slots)
        for s, x in zip(t.inputs, inputs):
            ext2[s] = x.data_ptr()
        for i, (s, bi, fn) in enumerate(t.outputs):
            off = int(fn(rows)) * t.slot_cols[s] * esz
            ext2[s] = b["out"][bi].data_ptr() + off
            seeds[s] = gext[s] = dbag.data_ptr() + off
        ws = L.workspace(lib.milb200_tape_workspace_bytes(c["ops"], c["n_ops"], slots, n_slots, code, 1, None), self.device)
        L.check(lib.milb200_tape_backward(c["ops"], c["n_ops"], slots, n_slots, c["params"], c["n_params"], ext2, gext, seeds,
                                          L.ptr(wcomp), L.ptr(self.params), L.ptr(self.grads), L.ptr(b["arena"]),
                                          b["arena"].numel(), L.ptr(ws), ws.numel(), code, None, L.stream_ptr()), "tape_backward")
        return b["loss"], prob

    # ---- exchange + optimiser -------------------------------------------------------------------------------------------
    def enable_symmetric_exchange(self):
        """The flat gradient buffer moves into symmetric memory and the exchange becomes the in-switch reduce + broadcast
        kernel of csrc/exchange.cu (see dp.AbmilTrainer.enable_symmetric_exchange); the 40 MB buffer keeps its own
        full-width optimiser kernel.  Collective; returns False (NCCL stays) without multicast support."""
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
        torch.distributed.all_reduce(ok, op=torch.distributed.ReduceOp.MIN, group=self.pg)
        if int(ok.item()) == 0:
            return False
        buf[:self.numel].copy_(self.grads)
        self.grads = buf[:self.numel]
        self.pool.grads = self.grads[self.o_pool:self.o_pool + self.pool.numel]    # the embedded pool trainer's view
        pads = torch.tensor([int(p) for p in hdl.signal_pad_ptrs], dtype=torch.int64, device=self.device)
        self._symm = dict(hdl=hdl, buf=buf, pads=pads, mc=mc, rank=int(hdl.rank))
        torch.cuda.synchronize()
        torch.distributed.barrier(group=self.pg)
        return True

    def reduce_and_update(self):
        """ONE exchange (sum) of the flat gradient, then the fused optimiser step with grad_scale = 1/world."""
        sm = getattr(self, "_symm", None)
        if sm is not None:
            L.check(L.lib().milb200_allreduce_update_symm(
                L.ptr(self.params), L.ptr(self.grads), sm["mc"], L.ptr(sm["pads"]), 0, sm["rank"], self.world, None, None,
                self.numel, -1, 0.0, 0.0, 0.0, 0.0, 0.0, 1.0, 1, None, L.stream_ptr()), "allreduce_update_symm")
        elif self.world > 1:
            torch.distributed.all_reduce(self.grads, group=self.pg)
        self.step_count += 1
        if self.optimizer == "sgd":
            L.check(L.lib().milb200_sgd_step(L.ptr(self.params), L.ptr(self.grads), self.numel, self.lr, self.wd,
                                             1.0 / self.world, L.stream_ptr()), "sgd_step")
        else:
            L.check(L.lib().milb200_adam_step(L.ptr(self.params), L.ptr(self.grads), L.ptr(self.exp_avg),
                                              L.ptr(self.exp_avg_sq), self.numel, self.lr, self.betas[0], self.betas[1],
                                              self.eps, self.wd, 1.0 / self.world, self.step_count, L.stream_ptr()),
                    "adam_step")
        self._refresh_compute_copy()

    def step(self, ct_tokens, x_path, x_text, label):
        out = self.forward_backward(ct_tokens, x_path, x_text, label)
        self.reduce_and_update()
        return out

    def step_bags(self, ct_tokens, x_path, path_lens, x_text, labels):
        out = self.forward_backward_bags(ct_tokens, x_path, path_lens, x_text, labels)
        self.reduce_and_update()
        return out
