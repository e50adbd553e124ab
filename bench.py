#!/usr/bin/env python
"""bench.py — bags/s forward+backward of the gated-attention MIL pool on ragged WSI-scale bags
(BASELINE.json configs[1]: 1 B200, bf16, bags of 100..20000 instances x 1024-dim).

One "step" = one packed CSR batch of `--bags` synthetic bags per rank through
  gated-score GEMM (tcgen05) -> segmented softmax pool -> pool backward -> gate backward (dZ recompute,
  split-K dW GEMM) -> [NCCL all-reduce of the flat gradient if N>1] -> fused Adam.
`value` has the inputs resident in HBM; `e2e` goes through the same public call with HOST (pinned) inputs,
H2D copy of the bags and D2H read of the pooled vectors inside the timed region.

  python bench.py --gpus N --steps K --warmup W            (N>1: launched by torch.distributed.run)
  python bench.py --impl reference ...                      (CPU arm: the oracle's torch fp32 restatement)
  python bench.py ... --dump-outputs DIR                    (also write the last timed step's outputs as DIR/*.npy)
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

L_FEAT, D_GATE = 1024, 192
LEN_LO, LEN_HI = 100, 20000
FALLBACK_PEAKS = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}
DUMP_BUDGET_BYTES = 64 << 20


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return d, "measured"
        except Exception:
            pass
    return dict(FALLBACK_PEAKS), "fallback"


def dump_outputs(dirname, arrays):
    """--dump-outputs: the {name: tensor} the timed path produced in its last step, one DIR/<name>.npy each, so that two
    builds can be compared output for output on the same seeded inputs.  Integer and float64 tensors are written as
    float64 (exact), every other tensor as float32.  A tensor larger than its equal share of the 64 MB budget is written
    as a fixed sample of its elements: flat indices drawn without replacement from numpy's default_rng(0), in increasing
    order, so the same shape always gives the same sample."""
    import numpy as np
    import torch
    os.makedirs(dirname, exist_ok=True)
    share = DUMP_BUDGET_BYTES // len(arrays)
    for name, t in arrays.items():
        t = t.detach()
        wide = t.dtype == torch.float64 or not t.dtype.is_floating_point
        a = t.to(torch.float64 if wide else torch.float32).cpu().numpy()
        if a.nbytes > share:
            keep = share // a.itemsize
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
        np.save(os.path.join(dirname, name + ".npy"), a)
    print(f"[bench] last timed step's outputs: {', '.join(sorted(arrays))} -> {dirname}", file=sys.stderr)


def bag_lengths(n_bags, seed):
    import torch
    g = torch.Generator().manual_seed(seed)
    return torch.randint(LEN_LO, LEN_HI + 1, (n_bags,), generator=g)


def bag_lengths_loguniform(n_bags, seed):
    """SURVEY §8d cfg 2 variant: real slides are skewed (biopsy << resection, dataset.py:376-381)."""
    import math
    import torch
    g = torch.Generator().manual_seed(seed)
    u = torch.rand(n_bags, generator=g)
    return torch.exp(u * (math.log(LEN_HI) - math.log(LEN_LO)) + math.log(LEN_LO)).round().long().clamp(LEN_LO, LEN_HI)


def torch_eager_gpu(X, lengths, dtype, steps=2):
    """BASELINE ONLY (SURVEY §8d "reference eager PyTorch on the same B200"): the reference's ABMIL maths
    (model/dim1/ABMIL.py:47-64, eval mode) written with stock torch.nn ops, bag at a time as train_ddp.py feeds it,
    autograd backward, torch.optim.Adam once per batch of bags.  cuBLAS/ATen kernels, none of ours."""
    import torch
    import torch.nn as nn
    dev = X.device
    torch.manual_seed(1234)
    V = nn.Sequential(nn.Linear(L_FEAT, D_GATE), nn.Tanh()).to(dev, dtype)
    U = nn.Sequential(nn.Linear(L_FEAT, D_GATE), nn.Sigmoid()).to(dev, dtype)
    w = nn.Linear(D_GATE, 1).to(dev, dtype)
    params = list(V.parameters()) + list(U.parameters()) + list(w.parameters())
    opt = torch.optim.Adam(params, lr=1e-5, betas=(0.9, 0.999), weight_decay=1e-7)
    offs = [0] + lengths.cumsum(0).tolist()
    Xd = X if X.dtype == dtype else None       # fp32 copies are made per bag (a 2.7 GB fp32 batch is not kept)

    def one_step():
        opt.zero_grad(set_to_none=True)
        for b in range(len(lengths)):
            xb = (Xd if Xd is not None else X)[offs[b]:offs[b + 1]]
            if xb.dtype != dtype:
                xb = xb.to(dtype)
            A = w(V(xb) * U(xb)).transpose(1, 0)
            M = torch.softmax(A, dim=1) @ xb
            M.float().sum().backward()
        opt.step()

    one_step()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        one_step()
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / steps
    return {"bags_per_s": len(lengths) / (ms / 1e3), "ms_per_step": ms, "dtype": str(dtype).replace("torch.", ""),
            "what": "stock torch.nn eager on the same GPU, bag at a time, fwd+bwd+Adam (baseline, not the product)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.idx)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        busy = [s for s in sm if s > 0]
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------
# CPU arm: the oracle's torch restatement of ABMIL.forward (fp32, autograd backward), bag at a time
# ----------------------------------------------------------------------------------------------------
def cpu_reference(lengths, steps, warmup, budget_s=20.0, per_step=4):
    import torch
    from oracle import fusion_oracle as fo
    from oracle import mil_oracle as mo
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    p = mo.procedural_state(mo.abmil_shapes(L_FEAT, D_GATE), 1234)
    g = torch.Generator().manual_seed(1234)
    pool_rows = max(int(v) for v in lengths) + 4096
    big = torch.randn(1, pool_rows, L_FEAT, generator=g)      # one host buffer; each bag is a window of it (not timed)
    cursor = [0]
    # the reference's own module when oracle/_ref holds it (oracle/make_ref.py copies model/dim1/ABMIL.py there, unmodified,
    # at build time); otherwise the oracle's op-for-op restatement
    from oracle import make_ref
    RefABMIL = make_ref.load_reference_abmil()
    if RefABMIL is not None:
        kind = "reference"
        ref = RefABMIL(None, L=L_FEAT, D=D_GATE).eval()       # eval(): dropout off, the semantics our headline step runs
        ref.load_state_dict({k: torch.from_numpy(v) for k, v in p.items()})
        params = list(ref.parameters())

        def fwd_bwd(x):
            for t in params:
                t.grad = None
            ref(x).sum().backward()
    else:
        kind = "port"
        sd = {"a." + k: torch.from_numpy(v).clone().requires_grad_(True) for k, v in p.items()}

        def fwd_bwd(x):
            for t in sd.values():
                t.grad = None
            fo.abmil(sd, "a", x).sum().backward()

    def one_bag(n):
        start = cursor[0] % (pool_rows - n + 1)
        cursor[0] += 997
        x = big[:, start:start + n]
        t0 = time.perf_counter()
        fwd_bwd(x)
        return time.perf_counter() - t0

    lens = [int(v) for v in lengths]
    for i in range(min(warmup, 2)):
        one_bag(lens[i % len(lens)])
    # bounded sample: each "step" is a fixed subset of the workload's bags; stop inside the budget
    per_step = max(1, min(len(lens), per_step))
    times, done_bags, t_begin = [], 0, time.perf_counter()
    for s in range(max(1, steps)):
        t = 0.0
        for j in range(per_step):
            t += one_bag(lens[(s * per_step + j) % len(lens)])
        times.append(t)
        done_bags += per_step
        if time.perf_counter() - t_begin > budget_s:
            break
    total = sum(times)
    what = ("the reference's own model/dim1/ABMIL.py (oracle/_ref, unmodified) in eval() mode" if kind == "reference"
            else "the oracle's restatement of ABMIL.forward (eval-mode arithmetic)")
    return {"value": done_bags / total, "unit": "bags/s", "cores": cores, "kind": kind,
            "sample": f"{done_bags} bags cycling through the workload's {len(lens)} bag lengths ({per_step} bags per step, "
                      f"{len(times)} steps, {total:.1f} s of CPU work), fp32, bag-at-a-time fwd+bwd (M.sum().backward()) as the "
                      f"reference trains, {what}; no dropout and NO optimiser step in the CPU figure (the GPU step includes "
                      f"fused Adam), torch {torch.__version__} with {cores} threads",
            "ms_per_step": 1e3 * total / len(times), "steps": len(times), "bags_per_step": per_step}


def torch_eager_fusion_gpu(model, x_ct_tok, x_p, x_t, label, dtype, steps=5):
    """BASELINE ONLY (the "real bar" for BASELINE configs[2]): the reference's CT+pathology `aggregator.forward`
    (model/aggregator.py:134-203 over model/sam/transformer.py:58-120,278-309,418-450, eval mode) written with STOCK torch
    ops on the same GPU — nn.functional.linear / layer_norm / softmax, projected K and V for every image token as upstream,
    autograd backward, torch.optim.Adam — one patient per step as train_ddp.py:75 feeds it.  None of our kernels."""
    import math
    import torch
    import torch.nn.functional as Fn
    sd = {k: v.detach().to(dtype).clone().requires_grad_(True) for k, v in model.state_dict().items()
          if v.is_floating_point() and not k.startswith(("TwoWayTransformer_CT", "TwoWayTransformer_Pth", "extractor_pathology",
                                                         "fc_CI.", "prompt_embedding"))}
    opt = torch.optim.Adam(list(sd.values()), lr=1e-5, betas=(0.9, 0.999), weight_decay=1e-7)
    lin = lambda pre, x: Fn.linear(x, sd[pre + ".weight"], sd[pre + ".bias"])
    ln = lambda pre, x: Fn.layer_norm(x, (x.shape[-1],), sd[pre + ".weight"], sd[pre + ".bias"], 1e-5)

    def attn(pre, q, k, v, heads=8):
        q, k, v = lin(pre + ".q_proj", q), lin(pre + ".k_proj", k), lin(pre + ".v_proj", v)
        c = q.shape[-1] // heads
        sp = lambda t: t.reshape(t.shape[0], heads, c).transpose(0, 1)
        a = torch.softmax(sp(q) @ sp(k).transpose(1, 2) / math.sqrt(c), dim=-1)
        return lin(pre + ".out_proj", (a @ sp(v)).transpose(0, 1).reshape(q.shape[0], heads * c))

    def twoway(img, pe, pts):
        pre = "TwoWayTransformer_Both"
        qs, ks = pts, img
        for i in range(2):
            lp = f"{pre}.layers.{i}"
            qs = ln(lp + ".norm1", attn(lp + ".self_attn", qs, qs, qs) if i == 0 else
                    qs + attn(lp + ".self_attn", qs + pts, qs + pts, qs))
            qs = ln(lp + ".norm2", qs + attn(lp + ".cross_attn_token_to_image", qs + pts, ks + pe, ks))
            qs = ln(lp + ".norm3", qs + lin(lp + ".mlp.lin2", torch.relu(lin(lp + ".mlp.lin1", qs))))
            ks = ln(lp + ".norm4", ks + attn(lp + ".cross_attn_image_to_token", ks + pe, qs + pts, qs))
        qs = ln(pre + ".norm_final_attn", qs + attn(pre + ".final_attn_token_to_image", qs + pts, ks + pe, ks))
        return qs, ks

    pe_tab = model._pe_table(max(x_ct_tok.shape[0], x_p.shape[0]), x_p.device).to(dtype)
    ct, xp, xt = x_ct_tok.to(dtype), x_p.to(dtype), x_t.to(dtype)

    def one_step():
        opt.zero_grad(set_to_none=True)
        xin = torch.tanh(lin("fc_pathology.0", xp))
        q1, k1 = twoway(ct, pe_tab[:ct.shape[0]], torch.tanh(lin("fc_CI2CT.0", xt)))
        q2, k2 = twoway(xin, pe_tab[:xin.shape[0]], torch.tanh(lin("fc_CI2Pth.0", xt)))
        bag = torch.cat([q1, k1, q2, k2], dim=0)
        A = lin("aggregator.attention_weights", torch.tanh(lin("aggregator.attention_V.0", bag)) *
                torch.sigmoid(lin("aggregator.attention_U.0", bag)))
        M = torch.softmax(A.transpose(1, 0), dim=1) @ bag
        prob = torch.sigmoid(lin("fc.1", M))
        loss = Fn.binary_cross_entropy(prob.float(), label) + (1 - Fn.cosine_similarity(q1.float(), q2.float())).mean()
        loss.backward()
        opt.step()

    one_step()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        one_step()
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / steps
    return {"ms_per_bag": ms, "bags_per_s": 1e3 / ms, "dtype": str(dtype).replace("torch.", ""),
            "what": "stock torch eager on the same GPU, one patient per step, fwd+bwd+Adam (baseline, not the product)"}


# Work per patient of the CT+pathology fusion step, N pathology rows, 160 CT tokens, one text token (DESIGN.md §5b):
#  * what the REFERENCE formulation executes (fc_pathology fwd + dW, 6 image-side K/V projection GEMMs fwd + dW + dX,
#    gated pool L = 512 fwd + dW + dX): the figure the round-1 review used for "useful work"
#  * HBM bytes of the COLLAPSED formulation (csrc/xfusion.cu; fp32 key stream, bf16 patch features and packed bag):
#    every pass listed in DESIGN.md §5b, read + write
def fusion_work_per_patient(n_path, n_ct=160):
    n = n_path + n_ct
    ref_flops = 2.0 * n_path * 768 * 512 * 2 + 6 * 2.0 * n * 512 * 256 * 3 + 12.0 * (n + 2) * 512 * 192
    fwd = n_path * 768 * 2 + n_path * 512 * 4 + 2 * (n * 512 * 8) + (n * 512 * 8) + (n * 512 * 6) + (n * 512 * 6) + 2 * n * 512 * 2
    bwd = (3 * n * 512 * 2) + (n * 512 * 10) + (n * 512 * 10) + (n * 512 * 16) + (n * 512 * 12) + (n * 512 * 16) + \
          (n_path * 512 * 10) + n_path * 512 * 2 + n_path * 768 * 2
    return ref_flops, float(fwd + bwd)


def secondary_fusion(dev):
    """BASELINE configs[2]: the multimodal aggregator (fc_pathology -> two TwoWayTransformer calls -> packed bag -> gated
    pool -> head) forward+backward on ONE WSI-scale bag per call, as the reference trains (train_ddp.py:75), bf16, through
    the public nn.Module; plus the CPU port of the same step on a smaller bag.  Informational."""
    import torch
    from argparse import Namespace
    import mil_b200
    ns = Namespace(modality=["CT", "pathology"], model_CT="resnetMC3_18", model_pathology="ABMIL", model_CI="none",
                   aggregator="ABMIL", num_classes=2, alignment_base="none", clinical_features=list("abcdefghi"))
    torch.manual_seed(1234)
    out = []
    # fp32 (the reference's own arithmetic): same module, fp32 operands — the big GEMMs run as 3xTF32 on the tensor cores
    m32 = mil_b200.get_model(ns).to(dev).train(False)
    p32 = list(m32.parameters())
    for T, N in ((1, 15592),):
        x_ct = torch.randn(1, 512, 160, 1, 1, device=dev)
        x_p = torch.randn(1, N, 768, device=dev)
        x_t = torch.randn(1, T, 512, device=dev) * 0.05
        label = torch.tensor([[0.0, 1.0]], device=dev)

        def step32():
            for p in p32:
                p.grad = None
            prob, a, b = m32([x_ct, x_p], x_t)
            loss = torch.nn.functional.binary_cross_entropy(prob.float(), label) + \
                mil_b200.clip_loss.cosine_embedding_loss(a.squeeze(0), b.squeeze(0)).float()
            loss.backward()

        for _ in range(4):
            step32()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            step32()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 10
        out.append({"workload": f"aggregator CT+pathology fwd+bwd, 1 bag, N={N} x 768 + 160 CT tokens, T={T}, fp32 (3xTF32 GEMMs)",
                    "ms_per_bag": ms, "bags_per_s": 1e3 / ms, "api": "nn.Module + torch.autograd (no optimiser step in the figure)"})
    del m32, p32
    m = mil_b200.get_model(ns).to(dev).to(torch.bfloat16).train(False)
    plist = list(m.parameters())
    for T, N in ((1, 15592), (10, 15592)):
        x_ct = torch.randn(1, 512, 160, 1, 1, device=dev, dtype=torch.bfloat16)
        x_p = torch.randn(1, N, 768, device=dev, dtype=torch.bfloat16)
        x_t = (torch.randn(1, T, 512, device=dev) * 0.05).to(torch.bfloat16)
        label = torch.tensor([[0.0, 1.0]], device=dev)

        def step():
            for p in plist:
                p.grad = None
            prob, a, b = m([x_ct, x_p], x_t)
            loss = torch.nn.functional.binary_cross_entropy(prob.float(), label) + \
                mil_b200.clip_loss.cosine_embedding_loss(a.squeeze(0), b.squeeze(0)).float()
            loss.backward()

        for _ in range(4):
            step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = mil_b200.launch_count()
        e0.record()
        for _ in range(10):
            step()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 10
        out.append({"workload": f"aggregator CT+pathology fwd+bwd, 1 bag, N={N} x 768 + 160 CT tokens, T={T}, bf16",
                    "ms_per_bag": ms, "bags_per_s": 1e3 / ms, "kernels_per_bag": (mil_b200.launch_count() - l0) / 10,
                    "api": "nn.Module + torch.autograd (no optimiser step in the figure)"})
        # the same bag through the native training step: flat buffers, no autograd graph, fused Adam INSIDE the figure
        tr = mil_b200.FusionTrainer(m, n_text_tokens=T, compute_dtype=torch.bfloat16)
        tok = mil_b200.functional.ct_tokens(x_ct)[0].detach()
        for _ in range(4):
            tr.step(tok, x_p[0], x_t[0], label[0])
        torch.cuda.synchronize()
        l0 = mil_b200.launch_count()
        e0.record()
        for _ in range(10):
            tr.step(tok, x_p[0], x_t[0], label[0])
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 10
        out.append({"workload": f"aggregator CT+pathology fwd+bwd+Adam, 1 bag, N={N} x 768 + 160 CT tokens, T={T}, bf16",
                    "ms_per_bag": ms, "bags_per_s": 1e3 / ms, "kernels_per_bag": (mil_b200.launch_count() - l0) / 10,
                    "api": "FusionTrainer.step (flat parameter/gradient buffers, BCE + cosine loss, fused Adam)"})
        del tr
        if T == 1:
            # B patients per launch set (FusionTrainer.step_bags, collapsed program): the token side (~150 small launches) is
            # shared by the B patients; roofline = HBM bytes of the collapsed formulation / time against the measured peak
            peaks, _ = load_peaks()
            hbm_peak = float(peaks.get("hbm_gbs", FALLBACK_PEAKS["hbm_gbs"]))
            tf_sus = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", FALLBACK_PEAKS["bf16_tflops"])))
            ref_flops, hbm_bytes = fusion_work_per_patient(N)
            for Bp in (1, 4, 8):
                trb = mil_b200.FusionTrainer(m, n_text_tokens=1, compute_dtype=torch.bfloat16)
                ctb = tok.unsqueeze(0).repeat(Bp, 1, 1).contiguous()
                xpb = x_p[0].repeat(Bp, 1).contiguous()
                xtb = x_t[0].repeat(Bp, 1).contiguous()
                lab = label.repeat(Bp, 1).contiguous()
                lens_b = [N] * Bp
                for _ in range(4):
                    trb.step_bags(ctb, xpb, lens_b, xtb, lab)
                torch.cuda.synchronize()
                l0 = mil_b200.launch_count()
                e0.record()
                for _ in range(10):
                    trb.step_bags(ctb, xpb, lens_b, xtb, lab)
                e1.record()
                torch.cuda.synchronize()
                ms = e0.elapsed_time(e1) / 10
                out.append({"workload": f"aggregator CT+pathology fwd+bwd+Adam, {Bp} patient(s) per step, N={N} x 768 + 160 CT "
                                        f"tokens each, T=1, bf16 (fp32 key stream / token side)",
                            "ms_per_step": ms, "ms_per_bag": ms / Bp, "bags_per_s": Bp * 1e3 / ms,
                            "kernels_per_bag": (mil_b200.launch_count() - l0) / 10 / Bp,
                            "api": "FusionTrainer.step_bags (collapsed program, csrc/xfusion.cu)",
                            "roofline": {"bound": "hbm", "achieved": hbm_bytes * Bp / ms / 1e6, "peak": hbm_peak, "unit": "GB/s",
                                         "frac": hbm_bytes * Bp / ms / 1e6 / hbm_peak,
                                         "algorithmic": "HBM bytes of the collapsed formulation per patient (DESIGN 5b)",
                                         "reference_formulation_tflops": ref_flops * Bp / ms / 1e9,
                                         "reference_formulation_frac_of_sustained_tensor_peak": ref_flops * Bp / ms / 1e9 / tf_sus}})
                del trb, xpb
            try:
                out.append(dict(torch_eager_fusion_gpu(m, tok, x_p[0], x_t[0], label, torch.float32),
                                workload=f"same step, stock torch eager, fp32, N={N}"))
                out.append(dict(torch_eager_fusion_gpu(m, tok, x_p[0], x_t[0], label, torch.bfloat16),
                                workload=f"same step, stock torch eager, bf16, N={N}"))
            except Exception as e:
                out.append({"workload": "stock torch eager fusion step", "error": repr(e)[:200]})

    def timed(fn, reps=10):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    # configs[2], second half: aggregator_clip (CT + pathology) on a packed CSR batch + CLIPloss_v1 + CLIP cosine logits
    ns = Namespace(modality=["CT", "pathology"], model_CT="resnetMC3_18", model_pathology="ABMIL", num_classes=2)
    mc = mil_b200.model.utils_clip.get_model(ns).to(dev).to(torch.bfloat16).train(False)
    g = torch.Generator().manual_seed(1234)
    lens = torch.randint(100, 15593, (64,), generator=g)
    off = torch.zeros(65, dtype=torch.int32)
    off[1:] = lens.cumsum(0)
    X = torch.randn(int(off[-1]), 768, device=dev, dtype=torch.bfloat16)
    offd = off.to(dev)
    x_ct = torch.randn(64, 512, device=dev, dtype=torch.bfloat16)
    feats = (torch.randn(64, 9, 512, device=dev) * 0.3).to(torch.bfloat16)
    crit = mil_b200.CLIPloss_v1(Namespace(clinical_features=list("abcdefghi")))
    head = mil_b200.CLIPLogits().to(dev)
    pl_c = list(mc.parameters())

    def step_clip():
        for p in pl_c:
            p.grad = None
        a, b, prob = mc.forward_csr(x_ct, X, offd)
        li, lt = head(a, b)
        (crit(b, feats) + li.diagonal().mean() * 1e-3 + prob.float().mean()).backward()

    ms = timed(step_clip)
    out.append({"workload": "aggregator_clip forward_csr (64 ragged bags 100..15592 x 768) + CLIPloss_v1 (I=9) + CLIP logits, "
                            "fwd+bwd, bf16", "ms_per_step": ms, "bags_per_s": 64e3 / ms, "instances": int(off[-1])})

    # configs[3]: masked MIL over padded CT-slice bags (B, 160, 768) with valid lengths + late-fusion head + BCE, fwd+bwd
    ns = Namespace(modality=["CT", "pathology"], model_CT="resnetMC3_18_wMask", model_pathology="ABMIL", num_classes=2,
                   clinical_features=list("abcdefghi"))
    mw = mil_b200.get_model(ns).to(dev).to(torch.bfloat16).train(False)
    Bw = 32
    xpad = torch.randn(Bw, 160, 768, device=dev, dtype=torch.bfloat16)
    lw = torch.randint(40, 161, (Bw,), generator=g).to(dev)
    pfeat = torch.randn(Bw, 768, device=dev, dtype=torch.bfloat16)
    tgt = torch.randint(0, 2, (Bw, 2), generator=g).float().to(dev)
    pl_w = list(mw.parameters())

    def step_wmask():
        for p in pl_w:
            p.grad = None
        prob = mw.forward_padded(mw.extractor_pathology, xpad, lw, other_feats=(pfeat,))
        torch.nn.functional.binary_cross_entropy(prob.float(), tgt).backward()

    ms = timed(step_wmask)
    out.append({"workload": "aggregator_wMask masked MIL: 32 padded CT bags (160 x 768, valid 40..160) + head + BCE, fwd+bwd, bf16",
                "ms_per_step": ms, "bags_per_s": Bw * 1e3 / ms})
    return out


def dp_equivalence_check(tr, module, X, offsets_h, lengths, rank, world, dev, pg):
    """N > 1 correctness signal in every bench run (train_ddp.py:79): on a small verification batch (the first rows of two
    bags per rank) the gradients after the exchange must equal those of ONE process over the union of all ranks' bags.
    Uses fresh trainers with the bench's parameters; the exchange is the one the timed run uses."""
    import torch
    import torch.distributed as dist
    from mil_b200.dp import AbmilTrainer
    rows = 1500
    offs = offsets_h.tolist()
    picks = [b for b in range(len(lengths)) if int(lengths[b]) >= rows][:2]
    mineX = torch.stack([X[offs[b]:offs[b] + rows] for b in picks])                        # [2, rows, L]
    gathered = [torch.empty_like(mineX) for _ in range(world)]
    dist.all_gather(gathered, mineX, group=pg)
    off_local = torch.tensor([0, rows, 2 * rows], dtype=torch.int32, device=dev)
    dpt = AbmilTrainer(tr.L, tr.D, tr.dtype, device=dev, process_group=pg, world_size=world)
    dpt.params.copy_(tr.params)
    symm = getattr(tr, "_symm", None) is not None and dpt.enable_symmetric_exchange()
    dpt.forward_backward(mineX.reshape(2 * rows, tr.L), off_local)
    if symm:
        dpt.lr = 0.0                       # exchange kernel = reduce + update: a zero-step update leaves the summed gradients
        dpt.wd = 0.0
        dpt.reduce_and_update()
    else:
        dpt.allreduce_grads()
    one = AbmilTrainer(tr.L, tr.D, tr.dtype, device=dev)
    one.params.copy_(tr.params)
    Xu = torch.cat([g.reshape(2 * rows, tr.L) for g in gathered])
    offu = torch.arange(0, 2 * world + 1, dtype=torch.int32, device=dev) * rows
    one.forward_backward(Xu, offu)
    err = float((dpt.grads.double() - one.grads.double()).abs().max() / one.grads.double().abs().max())
    hi, lo = dpt.grads.clone(), dpt.grads.clone()
    dist.all_reduce(hi, op=dist.ReduceOp.MAX, group=pg)
    dist.all_reduce(lo, op=dist.ReduceOp.MIN, group=pg)
    same = bool(torch.equal(hi, lo))
    if err > 2e-3 or not same:
        raise SystemExit(f"bench: data-parallel check failed: exchanged gradients vs single-process union rel err {err:.3e}, "
                         f"identical across ranks: {same}")
    return {"exchanged_grads_vs_single_process_union_rel_err": err, "grads_identical_across_ranks": same,
            "batch": f"{2 * world} bags x {rows} rows (two per rank)", "exchange": "symmetric-memory kernel" if symm else "nccl"}


def fusion_main(args, out):
    """BASELINE configs[2] / configs[4]: data-parallel training step of the CT+pathology aggregator — FusionTrainer.step_bags,
    `--patients` patients per rank per step (WSI-scale: 15 592 pathology rows x 768 + 160 CT tokens + one clinical-text
    token each), bf16 storage, BCE + cosine loss, gradient exchange, fused Adam inside the timed region.  One JSON line."""
    import torch
    import torch.distributed as dist
    from argparse import Namespace
    import mil_b200
    warmup = max(args.warmup, 3)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (B200); there is no CPU fallback for the product path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    pg = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        pg = dist.group.WORLD
    N, Nc, Bp = 15592, 160, max(1, min(8, args.patients))
    ns = Namespace(modality=["CT", "pathology"], model_CT="resnetMC3_18", model_pathology="ABMIL", model_CI="none",
                   aggregator="ABMIL", num_classes=2, alignment_base="none", clinical_features=list("abcdefghi"))
    torch.manual_seed(1234)
    m = mil_b200.get_model(ns).to(dev).eval()
    tr = mil_b200.FusionTrainer(m, n_text_tokens=1, compute_dtype=torch.bfloat16, process_group=pg, world_size=world)
    tr.broadcast_params()
    symm_on = world > 1 and os.environ.get("MILB200_SYMM", "1") != "0" and tr.enable_symmetric_exchange()
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    ct = torch.randn(Bp, Nc, 512, device=dev, generator=gen).to(torch.bfloat16)
    xp = torch.randn(Bp * N, 768, device=dev, generator=gen).to(torch.bfloat16)
    xt = (torch.randn(Bp, 512, device=dev, generator=gen) * 0.05).to(torch.bfloat16)
    labels = torch.tensor([[0.0, 1.0], [1.0, 0.0]] * Bp, device=dev)[:Bp].contiguous()
    lens = [N] * Bp

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(warmup):
        tr.step_bags(ct, xp, lens, xt, labels)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    barrier()
    l0 = mil_b200.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        loss, prob = tr.step_bags(ct, xp, lens, xt, labels)
    e1.record()
    barrier()
    launches = mil_b200.launch_count() - l0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"loss": loss, "prob": prob, "params": tr.params, "grads": tr.grads})
    t = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = Bp * world * args.steps / (ms_max / 1e3)
    # the exchange + optimiser part of the step alone (CUDA events around reduce_and_update, max over ranks)
    ex_ms = []
    for _ in range(5):
        tr.forward_backward_bags(ct, xp, lens, xt, labels)
        if world > 1:
            dist.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        tr.reduce_and_update()
        b.record()
        torch.cuda.synchronize()
        ex_ms.append(a.elapsed_time(b))
    ex_ms.sort()
    t = torch.tensor([ex_ms[len(ex_ms) // 2]], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    exchange_update_ms = float(t.item())
    # end to end: host (pinned) patient data, H2D inside the timed region, loss/prob read back every step
    xp_h = torch.empty_like(xp, device="cpu").pin_memory()
    xp_h.copy_(xp)
    ct_h, xt_h = ct.cpu().pin_memory(), xt.cpu().pin_memory()
    xp_d, ct_d, xt_d = torch.empty_like(xp), torch.empty_like(ct), torch.empty_like(xt)
    res_h = torch.empty(2 + Bp * 2, dtype=torch.float32).pin_memory()
    e2e_steps = max(3, min(args.steps, 10))

    def e2e_run(n):
        s = 0.0
        for _ in range(n):
            xp_d.copy_(xp_h, non_blocking=True)
            ct_d.copy_(ct_h, non_blocking=True)
            xt_d.copy_(xt_h, non_blocking=True)
            loss, prob = tr.step_bags(ct_d, xp_d, lens, xt_d, labels)
            res_h[:2].copy_(loss, non_blocking=True)
            res_h[2:].copy_(prob.reshape(-1), non_blocking=True)
            torch.cuda.current_stream().synchronize()
            s += float(res_h[0])
        return s
    e2e_run(2)
    barrier()
    e0.record()
    e2e_run(e2e_steps)
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = float(t.item())
    clocks = sampler.stop() if rank == 0 else None
    params_same = None
    if world > 1:
        hi, lo = tr.params.clone(), tr.params.clone()
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        params_same = bool(torch.equal(hi, lo))
        if not params_same:
            raise SystemExit("bench: parameters differ across ranks after the run — the gradient exchange is broken")
    if rank == 0:
        peaks, peak_src = load_peaks()
        hbm_peak = float(peaks.get("hbm_gbs", FALLBACK_PEAKS["hbm_gbs"]))
        ref_flops, hbm_bytes = fusion_work_per_patient(N, Nc)
        ms_step = ms_max / args.steps
        line = {"metric": "bags/sec fwd+bwd", "value": value, "unit": "bags/s", "n_gpus": world, "steps": args.steps,
                "warmup": warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "bf16", "data": "synthetic",
                "config": {"workload": f"data-parallel training step of the CT+pathology aggregator (BASELINE configs[2]/[4]): "
                                       f"{Bp} patients per rank per step, {N} pathology rows x 768 + {Nc} CT tokens + 1 clinical-"
                                       f"text token each, BCE + cosine loss, one all-reduce of the {tr.numel * 4 / 1e6:.0f} MB flat "
                                       f"gradient buffer, fused Adam; FusionTrainer.step_bags (collapsed program, csrc/xfusion.cu)",
                           "patients_per_rank": Bp, "parallelism": f"dp{world}",
                           "exchange": ("none (single GPU)" if world == 1 else
                                        "multimem.ld_reduce/st over NVSwitch symmetric memory (csrc/exchange.cu) + fused Adam kernel"
                                        if symm_on else "ncclAllReduce of the flat fp32 gradient buffer + fused Adam kernel"),
                           "storage": "bf16 patch features / packed bag / tensor-core operands, fp32 key stream and token side",
                           "cache": "patient data (~96 MB/patient) cycles through HBM; parameters + optimiser state 160 MB > L2"},
                "gpu_launches": int(launches), "kernels_per_bag": launches / args.steps / Bp,
                "exchange_plus_optimizer_ms": exchange_update_ms,
                "e2e": {"value": Bp * world * e2e_steps / (e2e_ms / 1e3), "unit": "bags/s",
                        "h2d_bytes_per_step": int(xp_h.numel() * 2 + ct_h.numel() * 2 + xt_h.numel() * 2),
                        "d2h_bytes_per_step": int(res_h.numel() * 4), "steps": e2e_steps, "ms_per_step": e2e_ms / e2e_steps},
                "roofline": {"bound": "hbm", "achieved": hbm_bytes * Bp / ms_step / 1e6, "peak": hbm_peak, "unit": "GB/s",
                             "frac": hbm_bytes * Bp / ms_step / 1e6 / hbm_peak, "traffic": None, "peak_source": peak_src,
                             "kernel": "whole step (HBM bytes of the collapsed formulation per patient, DESIGN 5b)",
                             "reference_formulation_tflops": ref_flops * Bp / ms_step / 1e9},
                "cpu_baseline": None, "clocks": clocks, "params_identical_across_ranks_after_run": params_same}
        out.write(json.dumps(line) + "\n")
        out.flush()
    if world > 1:
        dist.destroy_process_group()
    return 0


def _claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries (NCCL prints its version banner to stdout) must not add
    to it: point fd 1 at stderr for the whole run and return a writer on the original stdout for the final line."""
    sys.stdout.flush()
    keep = os.dup(1)
    os.dup2(2, 1)
    return os.fdopen(keep, "w")


def main():
    out = _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--bags", type=int, default=64, help="bags per rank per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--input-grad", action="store_true", help="also produce dX (instances are trainable upstream)")
    ap.add_argument("--no-secondary", action="store_true", help="skip the fusion-path (cfg 3) side measurement")
    ap.add_argument("--recompute-gate", action="store_true",
                    help="backward re-runs the gate GEMM instead of reading the V,U activations saved by the forward")
    ap.add_argument("--workload", default="abmil", choices=["abmil", "fusion"],
                    help="abmil: BASELINE configs[1] (the headline metric); fusion: BASELINE configs[2]/[4], the data-parallel "
                         "training step of the CT+pathology aggregator (FusionTrainer.step_bags)")
    ap.add_argument("--deal-bags", action="store_true",
                    help="abmil, world > 1: deal ONE draw of bags x world lengths to the ranks longest-first (dp.shard_bags) "
                         "instead of giving every rank the lengths of the single-GPU workload")
    ap.add_argument("--patients", type=int, default=8, help="fusion: patients per rank per step (<= 8)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (float32 or "
                         "float64, at most 64 MB in all; rank 0)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.steps < 1):
        ap.error("--dump-outputs needs --impl ours and --steps >= 1")
    if args.workload == "fusion" and args.impl == "ours":
        return fusion_main(args, out)
    warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    config = {"workload": f"gated-attention MIL fwd+bwd, ragged bags {LEN_LO}-{LEN_HI} instances x {L_FEAT}-dim "
                          f"(BASELINE configs[1]), {args.bags} bags per rank per step, packed CSR, D={D_GATE}; " +
                          (f"the step's {args.bags} x world bags (lengths randint seed 1234) are dealt to the ranks longest-first "
                           f"by instance count (dp.shard_bags, SURVEY 8e)" if args.deal_bags else
                           f"every rank runs the bag LENGTHS of the single-GPU workload (randint seed 1234, its own data): "
                           f"per-GPU work is identical at every N, so the scaling efficiency measures the exchange alone"),
              "bags_per_rank": args.bags, "L": L_FEAT, "D": D_GATE, "parallelism": f"dp{world}",
              "input_grad": bool(args.input_grad),
              "cache": "inputs (~1.3 GB/rank) exceed the 126 MB L2, no flush needed",
              "gate_backward": "recompute GEMM" if args.recompute_gate else "saved V,U (bf16, 768 B/instance)",
              "mode": "eval-mode semantics (no dropout), dM = ones, optimizer = fused Adam in the timed region"}

    if args.impl == "reference":
        if rank != 0:
            return 0
        lengths = bag_lengths(args.bags, 1234)
        cb = cpu_reference(lengths, args.steps, args.warmup, budget_s=60.0, per_step=16)
        line = {"impl": "reference", "metric": "bags/sec fwd+bwd", "value": cb["value"], "unit": "bags/s",
                "n_gpus": args.gpus, "steps": cb["steps"], "warmup": args.warmup, "ms_per_step": cb["ms_per_step"],
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": config,
                "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
                "e2e": {"value": cb["value"], "unit": "bags/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        out.write(json.dumps(line) + "\n")
        out.flush()
        return 0

    import torch
    import torch.distributed as dist
    import mil_b200
    from mil_b200 import _lib as Lb
    from mil_b200.dp import AbmilTrainer

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (B200); there is no CPU fallback for the product path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    pg = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        pg = dist.group.WORLD

    peaks, peak_src = load_peaks()
    from mil_b200.dp import shard_bags
    if args.deal_bags:
        all_lengths = bag_lengths(args.bags * world, 1234)
        mine = shard_bags(all_lengths.tolist(), rank, world, balance=True)
        lengths = all_lengths[mine]
    else:
        lengths = bag_lengths(args.bags, 1234)                    # the 64 bags of the single-GPU workload, on every rank
        all_lengths = lengths.repeat(world)
    n_bags = len(lengths)
    offsets_h = torch.zeros(n_bags + 1, dtype=torch.int32)
    offsets_h[1:] = lengths.cumsum(0).to(torch.int32)
    total_n = int(offsets_h[-1])
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    X = torch.randn(total_n, L_FEAT, device=dev, generator=gen).to(torch.bfloat16)
    offsets = offsets_h.to(dev)

    # parameters: reference default init (nn.Linear), seed 1234 (config.py:103), replicated via broadcast
    torch.manual_seed(1234)
    module = mil_b200.ABMIL(None, L=L_FEAT, D=D_GATE).to(dev)
    tr = AbmilTrainer(L_FEAT, D_GATE, torch.bfloat16, lr=1e-5, weight_decay=1e-7, device=dev, process_group=pg,
                      world_size=world, need_input_grad=args.input_grad, save_gate=not args.recompute_gate)
    tr.load_from(module)
    tr.broadcast_params()
    exchange = "none (single GPU)"
    if world > 1:
        symm_on = os.environ.get("MILB200_SYMM", "1") != "0" and tr.enable_symmetric_exchange()
        exchange = ("one kernel: multimem.ld_reduce/st over NVSwitch symmetric memory + fused Adam (csrc/exchange.cu)" if symm_on
                    else "ncclAllReduce of the flat fp32 gradient buffer + fused Adam kernel")
    config["exchange"] = exchange

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    dp_check = dp_equivalence_check(tr, module, X, offsets_h, lengths, rank, world, dev, pg) if world > 1 else None

    # ---- device-resident timing ----
    # the whole step (forward, backward, exchange, optimiser) replays as ONE CUDA graph per input address
    # (AbmilTrainer.step_graphed; MILB200_STEP_GRAPH=0 runs the ~10 launches eagerly)
    use_graph = os.environ.get("MILB200_STEP_GRAPH", "1") != "0" and not args.input_grad
    run_step = tr.step_graphed if use_graph else tr.step
    graphed = use_graph and (world == 1 or getattr(tr, "_symm", None) is not None)     # an NCCL exchange keeps the step eager
    config["step_launch"] = "one CUDA graph per step (AbmilTrainer.step_graphed)" if graphed else "eager launches"
    for _ in range(warmup):
        run_step(X, offsets)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    barrier()
    l0 = mil_b200.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        M = run_step(X, offsets)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = mil_b200.launch_count() - l0
    if args.dump_outputs and rank == 0:
        # the pooled vectors the step returns, the per-instance attention scores and per-bag argmax, and the trainer's
        # parameters (after the Adam update) and gradients
        dump_outputs(args.dump_outputs, {"M": M, "scores": tr.last_scores, "argmax": tr.last_argmax, "params": tr.params,
                                         "grads": tr.grads})
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    total_bags = args.bags * world * args.steps
    value = total_bags / (ms_max / 1e3)

    # ---- N > 1: where the gap to N x single-GPU goes — the same ranks, same data, WITHOUT the exchange (forward +
    # backward + a local optimiser step, no cross-rank synchronisation): fastest and slowest rank ----------------------
    no_exchange = None
    if world > 1:
        solo = AbmilTrainer(L_FEAT, D_GATE, torch.bfloat16, lr=1e-5, weight_decay=1e-7, device=dev,
                            need_input_grad=args.input_grad, save_gate=not args.recompute_gate)
        solo.params.copy_(tr.params)
        solo_step = solo.step_graphed if use_graph else solo.step
        for _ in range(warmup):
            solo_step(X, offsets)
        barrier()
        e0.record()
        for _ in range(args.steps):
            solo_step(X, offsets)
        e1.record()
        torch.cuda.synchronize()
        t_solo = torch.tensor([e0.elapsed_time(e1) / args.steps], device=dev)
        hi, lo = t_solo.clone(), t_solo.clone()
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        no_exchange = {"ms_per_step_slowest_rank": float(hi.item()), "ms_per_step_fastest_rank": float(lo.item()),
                       "what": "the same step on every rank without the gradient exchange (no cross-rank synchronisation): "
                               "ms_per_step minus the slowest rank's figure is what the exchange and its barriers cost"}
        del solo
        barrier()

    # ---- the same steps again with a CUDA event between phases: per-kernel durations IN the step -------------------
    # every rank runs them (the step contains the all-reduce); rank 0 records the events
    phase_ms = {}
    marks = []

    def hook(name):
        ev = torch.cuda.Event(enable_timing=True)
        ev.record()
        marks.append((name, ev))
    if rank == 0:
        tr.phase_hook = hook
    n_ph = max(3, min(args.steps, 10))
    for _ in range(n_ph):
        tr.step(X, offsets)
    torch.cuda.synchronize()
    tr.phase_hook = None
    per_phase = {}
    for (n0, a), (n1, b) in zip(marks[:-1], marks[1:]):
        if n1 != "pack":
            per_phase.setdefault(n1, []).append(a.elapsed_time(b))
    for name, vals in per_phase.items():      # median over the steps: one host hiccup must not colour a kernel's duration
        vals.sort()
        phase_ms[name] = vals[len(vals) // 2] if len(vals) % 2 else 0.5 * (vals[len(vals) // 2 - 1] + vals[len(vals) // 2])
    barrier()

    # ---- end to end: host (pinned) inputs, H2D + D2H inside the timed region -----------------------------------
    # Every step copies ITS bags host->device (pinned memory, copy stream), runs the public step and reads the pooled
    # vectors back.  Two device buffers: the copy of step k+1 overlaps the kernels of step k (the copy engine and the
    # SMs are independent), and the host consumes the result of step k-1 while step k runs.
    X_h = torch.empty((total_n, L_FEAT), dtype=torch.bfloat16).pin_memory()
    X_h.copy_(X)
    off_pin = offsets_h.pin_memory()
    M_h = [torch.empty((n_bags, L_FEAT), dtype=torch.float32).pin_memory() for _ in range(2)]
    X_d = [torch.empty_like(X) for _ in range(2)]
    off_d = [torch.empty_like(offsets) for _ in range(2)]
    copy_stream = torch.cuda.Stream(device=dev)
    main_stream = torch.cuda.current_stream()
    copied = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    read_back = [torch.cuda.Event() for _ in range(2)]

    def e2e_run(n_steps):
        checksum = 0.0
        for k in range(n_steps):
            b = k & 1
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(consumed[b])            # the kernels that read this buffer two steps ago are done
                X_d[b].copy_(X_h, non_blocking=True)
                off_d[b].copy_(off_pin, non_blocking=True)
                copied[b].record(copy_stream)
            main_stream.wait_event(copied[b])
            M = run_step(X_d[b], off_d[b])
            consumed[b].record(main_stream)
            M_h[b].copy_(M, non_blocking=True)
            read_back[b].record(main_stream)
            if k > 0:                                          # the caller consumes step k-1's pooled vectors
                read_back[b ^ 1].synchronize()
                checksum += float(M_h[b ^ 1][0, 0])
        read_back[(n_steps - 1) & 1].synchronize()
        return checksum + float(M_h[(n_steps - 1) & 1][0, 0])

    for ev in consumed:
        ev.record(main_stream)
    e2e_steps = max(3, min(args.steps, 10))
    e2e_run(2)
    barrier()
    e0.record()
    e2e_run(e2e_steps)
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = float(t.item())
    e2e_value = args.bags * world * e2e_steps / (e2e_ms / 1e3)
    h2d = X_h.numel() * 2 + off_pin.numel() * 4
    d2h = M_h[0].numel() * 4
    del X_d
    clocks = sampler.stop() if rank == 0 else None     # sampled across both timed regions (device-resident and end-to-end)

    # ---- per-kernel roofline (timed alone, CUDA events on the launch stream, same inputs) ----
    kernels = []
    if rank == 0:
        from mil_b200 import functional as F
        v = tr._views(tr.params)
        Wcat, bcat_c = tr._wcat_c, tr._bcat_c
        hbm_peak = float(peaks.get("hbm_gbs", FALLBACK_PEAKS["hbm_gbs"]))
        tf_peak = float(peaks.get("bf16_tflops", FALLBACK_PEAKS["bf16_tflops"]))
        s, act = F.gated_scores(X, Wcat, bcat_c, v["ww"], v["bw"], save=True)
        M, _, _, _ = F.segment_softmax_pool(X, s, offsets)
        dM = torch.ones_like(M)
        ds, _ = F.segment_softmax_pool_bwd(X, s, offsets, dM, M, False)

        def timeit(fn, reps=10):
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(reps):
                fn()
            b.record()
            torch.cuda.synchronize()
            return a.elapsed_time(b) / reps

        n, Lf, D, B = total_n, L_FEAT, D_GATE, n_bags
        gemm_flops = 2.0 * n * Lf * 2 * D
        save = tr.save_gate and act is not None
        t_score = timeit(lambda: F.gated_scores(X, Wcat, bcat_c, v["ww"], v["bw"], save=save))
        kernels.append({"name": "gated_score_fwd (k_gemm_kmajor_2sm<192x2,EpiScore%s>, CTA pairs)" % ("+save V,U" if save else ""),
                        "ms": t_score, "bound": "tensor",
                        "achieved": gemm_flops / t_score / 1e9, "peak": tf_peak, "unit": "TFLOP/s",
                        "algorithmic": "2*n*L*2D flop",
                        "hbm_gbs": (n * Lf * 2 + n * 4 + (n * 2 * D * 2 if save else 0)) / t_score / 1e6})
        t_pool = timeit(lambda: F.segment_softmax_pool(X, s, offsets))
        pool_bytes = n * (Lf * 2 + 4) + B * Lf * 4 + (B + 1) * 4
        kernels.append({"name": "segment_softmax_pool_fwd (k_pool_fwd)", "ms": t_pool, "bound": "hbm",
                        "achieved": pool_bytes / t_pool / 1e6, "peak": hbm_peak, "unit": "GB/s",
                        "algorithmic": "n*(L*2+4) + B*L*4 + (B+1)*4 bytes"})
        t_pbwd = timeit(lambda: F.segment_softmax_pool_bwd(X, s, offsets, dM, M, False))
        pbwd_bytes = n * (Lf * 2 + 4 + 4) + 2 * B * Lf * 4 + (B + 1) * 4
        kernels.append({"name": "segment_softmax_pool_bwd (k_pool_bwd)", "ms": t_pbwd, "bound": "hbm",
                        "achieved": pbwd_bytes / t_pbwd / 1e6, "peak": hbm_peak, "unit": "GB/s",
                        "algorithmic": "n*(L*2+8) + 2*B*L*4 + (B+1)*4 bytes"})
        Lb.lib().milb200_profile_enable(1)
        acc = [0.0] * 4
        reps = 10
        for i in range(reps + 3):
            F.gated_scores_bwd(X, Wcat, bcat_c, v["ww"], v["bw"], ds, None, dM, offsets, False, grad_out=tr.grads,
                               gate_act=act if save else None)     # need_dx=False here; --input-grad changes the trainer only
            buf = (ctypes.c_float * 8)()
            k = Lb.lib().milb200_profile_read(buf, 8)
            if i >= 3:
                for j in range(min(k, 4)):
                    acc[j] += buf[j] / reps
        Lb.lib().milb200_profile_enable(0)
        fused = save
        if fused:
            # one kernel: dW = dZ^T X with dZ built on the fly from the saved V,U; interval 1 = column-sum fold + split-K reduce
            kernels.append({"name": "gate_bwd dW fused (k_gemm_tn_gate: dZ from saved V,U on the fly)", "ms": acc[0],
                            "bound": "tensor", "achieved": gemm_flops / acc[0] / 1e9, "peak": tf_peak, "unit": "TFLOP/s",
                            "algorithmic": "2*n*L*2D flop", "hbm_gbs": (n * Lf * 2 + n * 2 * D * 2 + n * 4) / acc[0] / 1e6})
            kernels.append({"name": "split-K reduce + column-sum fold", "ms": acc[1], "bound": "hbm", "achieved": None,
                            "peak": hbm_peak, "unit": "GB/s"})
        elif save:
            dz_bytes = n * (2 * 2 * D * 2 + 4)
            kernels.append({"name": "gate_bwd dZ from saved V,U (k_gate_dz_saved)", "ms": acc[0], "bound": "hbm",
                            "achieved": dz_bytes / acc[0] / 1e6, "peak": hbm_peak, "unit": "GB/s",
                            "algorithmic": "n*(2*2D*2 + 4) bytes"})
        else:
            kernels.append({"name": "gate_bwd dZ recompute (k_gemm_kmajor<192x2,EpiDz>)", "ms": acc[0], "bound": "tensor",
                            "achieved": gemm_flops / acc[0] / 1e9, "peak": tf_peak, "unit": "TFLOP/s",
                            "algorithmic": "2*n*L*2D flop", "hbm_gbs": (n * Lf * 2 + n * 2 * D * 2) / acc[0] / 1e6})
        if not fused:
            kernels.append({"name": "gate_bwd dW split-K (k_gemm_tn)", "ms": acc[1], "bound": "tensor",
                            "achieved": gemm_flops / acc[1] / 1e9, "peak": tf_peak, "unit": "TFLOP/s",
                            "algorithmic": "2*n*L*2D flop", "hbm_gbs": (n * Lf * 2 + n * 2 * D * 2) / acc[1] / 1e6})
            kernels.append({"name": "split-K reduce (k_splitk_reduce)", "ms": acc[2], "bound": "hbm", "achieved": None,
                            "peak": hbm_peak, "unit": "GB/s"})
        # The opt-in mirrored single-pass backward (MILB200_FUSED_BWD=1): pooling backward inside the dW kernel.  Timed
        # here for the record (alone, same inputs); it is not in the default step, so it never becomes the dominant kernel.
        if save and Lb.lib().milb200_gated_pool_bwd_supported(Lf, D, Lb.dtype_code(X)):
            t_fb = timeit(lambda: F.gated_pool_bwd(X, s, offsets, dM, M, v["ww"], act, grad_out=tr.grads))
            kernels.append({"name": "gated_pool_bwd, opt-in (k_gemm_tn_gate with the pooling backward in g warps + reduce)",
                            "ms": t_fb, "bound": "tensor", "achieved": (gemm_flops + 2.0 * n * Lf) / t_fb / 1e9,
                            "peak": tf_peak, "unit": "TFLOP/s", "algorithmic": "2*n*L*2D + 2*n*L flop",
                            "in_step": bool(phase_ms.get("gated_pool_bwd")),
                            "replaces_ms": t_pbwd + acc[0] + acc[1],
                            "hbm_gbs": (n * Lf * 2 + n * 2 * D * 2 + n * 8) / t_fb / 1e6})
        # DRAM traffic per launch (dram__bytes_read.sum + dram__bytes_write.sum) from the committed ncu --set full
        # capture of this same workload (tools/ncu_summary.py -> profiles/kernel_traffic.json); null if absent
        try:
            ncu_traffic = json.load(open(os.path.join(ROOT, "profiles", "kernel_traffic.json")))
        except Exception:
            ncu_traffic = {}
        ncu_keys = {"gated_score_fwd": "k_gemm_kmajor_2sm<192, tc::EpiScoreT<%d>>" % (1 if save else 0),
                    "segment_softmax_pool_fwd": "k_pool_fwd<__nv_bfloat16, 4>",
                    "segment_softmax_pool_bwd": "k_pool_bwd<__nv_bfloat16, 4>",
                    "gate_bwd dZ from saved": "k_gate_dz_saved", "gate_bwd dZ recompute": "k_gemm_kmajor<192, tc::EpiDz>",
                    "gate_bwd dW fused": "k_gemm_tn_gate", "gate_bwd dW split-K": "k_gemm_tn"}
        # Durations above are each kernel looped ALONE back to back (10 launches); `ms_in_step` is the same kernel between
        # CUDA events inside the training step.  The roofline uses the in-step duration (the contract's "over the timed
        # region") against the BURST peak (the conservative denominator); the alone-loop figures stay beside it.
        in_step = {"gated_score_fwd": phase_ms.get("gated_score_fwd"),
                   "segment_softmax_pool_fwd": phase_ms.get("segment_softmax_pool_fwd"),
                   "segment_softmax_pool_bwd": phase_ms.get("segment_softmax_pool_bwd"),
                   "gated_pool_bwd": phase_ms.get("gated_pool_bwd")}
        if fused and phase_ms.get("gate_bwd"):
            in_step["gate_bwd dW fused"] = phase_ms["gate_bwd"] - acc[1]
        for kinfo in kernels:
            kinfo["ms_alone"] = kinfo["ms"]
            kinfo["achieved_alone"] = kinfo.get("achieved")
            for prefix, t_in in in_step.items():
                if kinfo["name"].startswith(prefix) and t_in and kinfo.get("achieved"):
                    if prefix == "segment_softmax_pool_bwd":
                        t_in -= 0.0                      # includes the 12 us per-bag statistics kernel; left in (conservative)
                    kinfo["ms_in_step"] = t_in
                    kinfo["achieved"] = kinfo["achieved"] * kinfo["ms"] / t_in
                    kinfo["ms"] = t_in
        # Denominators (the bench contract): a kernel timed INSIDE the long step is measured against the SUSTAINED tensor
        # peak (cuBLAS bf16 back to back for seconds: the chip is power-limited there, ~1335 MHz at ~1 kW), a kernel timed
        # alone against the BURST figure.  Both fractions are kept; HBM has one measured figure.
        sustained = float(peaks["bf16_tflops_sustained"]) if peaks.get("bf16_tflops_sustained") else None
        for kinfo in kernels:
            burst_peak = kinfo["peak"]
            kinfo["frac_alone"] = (kinfo["achieved_alone"] / burst_peak) if kinfo.get("achieved_alone") else None
            if kinfo["bound"] == "tensor" and kinfo.get("achieved") and sustained:
                kinfo["frac_of_sustained_peak"] = kinfo["achieved"] / sustained
                kinfo["frac_of_burst_peak"] = kinfo["achieved"] / burst_peak
                if kinfo.get("ms_in_step"):
                    kinfo["peak"] = sustained
                    kinfo["peak_kind"] = "sustained (kernel timed inside the step); burst %.1f" % burst_peak
            kinfo["frac"] = (kinfo["achieved"] / kinfo["peak"]) if kinfo.get("achieved") else None
            kinfo["traffic"] = None
            for prefix, key in ncu_keys.items():
                if kinfo["name"].startswith(prefix) and key in ncu_traffic:
                    kinfo["traffic"] = ncu_traffic[key]["dram_bytes"]
                    kinfo["traffic_source"] = ncu_traffic[key].get("source")

    # ---- secondary rows of SURVEY §8 (not the headline metric): the cross-modal fusion path, one bag per call -------------
    secondary = None
    if rank == 0 and world == 1 and not args.no_secondary:
        try:
            secondary = {"fusion": secondary_fusion(dev)}
        except Exception as e:  # never let a secondary measurement break the contract line
            secondary = {"fusion": {"error": repr(e)[:200]}}
        try:    # cfg 2 with log-uniform bag lengths (skewed slide sizes), same trainer, device-resident
            ll = bag_lengths_loguniform(args.bags, 1234)
            off_l = torch.zeros(args.bags + 1, dtype=torch.int32)
            off_l[1:] = ll.cumsum(0).to(torch.int32)
            n_l = int(off_l[-1])
            X_l, off_ld = X[:n_l], off_l.to(dev)
            for _ in range(3):
                tr.step(X_l, off_ld)
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(20):
                tr.step(X_l, off_ld)
            b.record()
            torch.cuda.synchronize()
            secondary["cfg2_loguniform_lengths"] = {"bags_per_s": args.bags * 20 / (a.elapsed_time(b) / 1e3),
                                                    "ms_per_step": a.elapsed_time(b) / 20, "instances": n_l,
                                                    "instances_per_s": n_l * 20 / (a.elapsed_time(b) / 1e3)}
        except Exception as e:
            secondary["cfg2_loguniform_lengths"] = {"error": repr(e)[:200]}
        try:    # cfg 2 with train-mode semantics: Dropout(p=0.5) on the instances (ABMIL.py:49), one extra pass over X
            trd = AbmilTrainer(L_FEAT, D_GATE, torch.bfloat16, lr=1e-5, weight_decay=1e-7, device=dev, dropout_p=0.5)
            trd.load_from(module)
            for _ in range(3):
                trd.step(X, offsets)
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(20):
                trd.step(X, offsets)
            b.record()
            torch.cuda.synchronize()
            secondary["cfg2_train_mode_dropout"] = {"bags_per_s": n_bags * 20 / (a.elapsed_time(b) / 1e3),
                                                    "ms_per_step": a.elapsed_time(b) / 20,
                                                    "what": "same step with Dropout(0.5) on the instances as the reference "
                                                            "trains (masked copy of X: +2.7 GB of traffic per step)"}
            del trd
        except Exception as e:
            secondary["cfg2_train_mode_dropout"] = {"error": repr(e)[:200]}
        try:    # BASELINE configs[0] (the reference's CPU-runnable case): 32 bags x 512 instances x 1024, fp32, fwd+bwd
            B1, N1 = 32, 512
            tr1 = AbmilTrainer(L_FEAT, D_GATE, torch.float32, device=dev)
            tr1.load_from(module)
            g1 = torch.Generator(device=dev).manual_seed(1234)
            X1 = torch.randn(B1 * N1, L_FEAT, device=dev, generator=g1)
            off1 = (torch.arange(B1 + 1, device=dev, dtype=torch.int32) * N1).contiguous()
            for _ in range(3):
                tr1.step(X1, off1)
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(20):
                tr1.step(X1, off1)
            b.record()
            torch.cuda.synchronize()
            cfg1 = {"gpu_bags_per_s": B1 * 20 / (a.elapsed_time(b) / 1e3), "gpu_ms_per_step": a.elapsed_time(b) / 20,
                    "gpu_dtype": "f32 operands, 3xTF32 tcgen05 GEMMs (kind::tf32 over hi/lo splits; the <=1e-5 parity path), "
                                 "32 bags packed in one CSR batch"}
            if not args.no_cpu_baseline:
                c1 = cpu_reference(torch.full((B1,), N1), steps=3, warmup=2, budget_s=6.0, per_step=B1)
                cfg1.update({"cpu_bags_per_s": c1["value"], "cpu_cores": c1["cores"], "cpu_sample": c1["sample"]})
            secondary["cfg1_32x512x1024_fp32"] = cfg1
            del tr1, X1
        except Exception as e:
            secondary["cfg1_32x512x1024_fp32"] = {"error": repr(e)[:200]}
        try:    # §8f rank 4: the same step fed from per-slide fp32 host matrices through the native packer + copy stream
            from mil_b200 import feeder as fd
            offs_l = [0] + lengths.cumsum(0).tolist()
            n_src = min(args.bags, 32)                       # 32 slides (~1.3 GB fp32 on the host), cycled
            src = [X[offs_l[b]:offs_l[b + 1]].float().cpu().numpy() for b in range(n_src)]
            fdr = fd.PackedBagFeeder(src * 6, batch_bags=n_src, L_feat=L_FEAT, device=dev, dtype=torch.bfloat16)
            rows = sum(a.shape[0] for a in src)
            stage = torch.empty((rows, L_FEAT), dtype=torch.bfloat16).pin_memory()
            offh = torch.zeros(n_src + 1, dtype=torch.int32)
            fd.pack_bags_host(src, stage, offh)
            t0 = time.perf_counter()
            for _ in range(3):
                fd.pack_bags_host(src, stage, offh)
            t_pack = (time.perf_counter() - t0) / 3
            it = iter(fdr)
            Xb, ob, _ = next(it)
            tr.step(Xb, ob)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            nb = 0
            for Xb, ob, ids in it:
                tr.step(Xb, ob)
                nb += len(ids)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            secondary["feeder_fp32_slides_to_bf16_csr"] = {
                "bags_per_s": nb / dt, "host_pack_ms_per_batch": t_pack * 1e3,
                "host_pack_read_gbs": rows * L_FEAT * 4 / t_pack / 1e9, "host_threads": os.cpu_count(),
                "what": "per-slide fp32 matrices (host) -> native threaded pack to pinned bf16 CSR -> H2D on a copy "
                        "stream -> trainer step; wall clock over 5 batches of %d bags" % n_src}
            del src, stage, fdr
        except Exception as e:
            secondary["feeder_fp32_slides_to_bf16_csr"] = {"error": repr(e)[:200]}
        try:    # the "real bar" of SURVEY F1: stock eager PyTorch on this same GPU
            secondary["torch_eager_same_gpu"] = [torch_eager_gpu(X, lengths, torch.float32),
                                                 torch_eager_gpu(X, lengths, torch.bfloat16)]
        except Exception as e:
            secondary["torch_eager_same_gpu"] = {"error": repr(e)[:200]}

    params_same = None
    if world > 1:      # the replicas must still be bit-identical after every timed step (a broken exchange would not be)
        hi, lo = tr.params.clone(), tr.params.clone()
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        params_same = bool(torch.equal(hi, lo))
        if not params_same:
            raise SystemExit("bench: parameters differ across ranks after the run — the gradient exchange is broken")

    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_base = cpu_reference(lengths, steps=10 ** 6, warmup=1, budget_s=12.0)   # ~12 s of CPU work over the same bags
        cpu_base = {k: cpu_base[k] for k in ("value", "unit", "cores", "kind", "sample")}

    if rank == 0:
        dom = max((k for k in kernels if k.get("in_step", True)), key=lambda k: k["ms"])
        roof = {"kernel": dom["name"], "bound": dom["bound"], "achieved": dom["achieved"], "peak": dom["peak"],
                "unit": dom["unit"], "frac": dom["frac"], "traffic": dom.get("traffic"),
                "traffic_source": dom.get("traffic_source"), "peak_source": peak_src,
                "ms_per_launch": dom["ms"], "algorithmic": dom.get("algorithmic"),
                "timing": "CUDA events around the kernel inside the training step (median over steps)" if dom.get("ms_in_step")
                          else "kernel looped alone, CUDA events",
                "ms_alone_back_to_back": dom.get("ms_alone"), "frac_alone_back_to_back": dom.get("frac_alone"),
                "frac_of_sustained_peak": dom.get("frac_of_sustained_peak"), "frac_of_burst_peak": dom.get("frac_of_burst_peak"),
                "peak_kind": dom.get("peak_kind", "measured burst / copy peak"), "phase_ms_in_step": phase_ms}
        line = {"metric": "bags/sec fwd+bwd", "value": value, "unit": "bags/s", "n_gpus": world, "steps": args.steps,
                "warmup": warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": config,
                "instances_per_step_per_rank": total_n, "bags_this_rank": n_bags,
                "instances_per_s": int(all_lengths.sum()) * args.steps / (ms_max / 1e3),
                "gpu_launches": int(launches),
                "e2e": {"value": e2e_value, "unit": "bags/s", "h2d_bytes_per_step": int(h2d),
                        "d2h_bytes_per_step": int(d2h), "steps": e2e_steps, "ms_per_step": e2e_ms / e2e_steps},
                "roofline": roof, "kernels": kernels, "cpu_baseline": cpu_base, "clocks": clocks, "secondary": secondary,
                "dp_check": dp_check, "params_identical_across_ranks_after_run": params_same,
                "step_without_exchange": no_exchange}
        out.write(json.dumps(line) + "\n")
        out.flush()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
