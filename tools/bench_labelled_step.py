"""Times a labelled training step of the gated-attention pool with a linear classifier head and BCE (the pathology-only
aggregator_clip: pool -> Linear(L, C) -> sigmoid -> BCE) at the cfg-2 shapes of bench.py: 64 bags of 100..20 000 rows,
L = 1024, bf16, C = 2, eval-mode semantics.  X is 1.37 GB, past the 126 MB L2.

  (a) headdot:   AbmilTrainer.step_graphed(X, offsets, labels): the pooling pass takes the head's C row dots, so the
                 step reads X three times (score GEMM, pooling pass, dW GEMM)
  (b) two-pass:  forward + head + BCE + backward(dM) + update, the pooling backward re-reading X, one CUDA graph
  (c) synthetic: AbmilTrainer.step_graphed(X, offsets) with dM = ones (bench.py's step)

The three are timed with CUDA events, alternating rep by rep, and reported as mean, standard deviation, median and min.
Then the pool forward alone (CUDA events, alternating) for the plain kernel, the one-dot _rowdot kernel and the _headdot
kernel at C = 1, 2, 4, 8.  Prints one JSON line with the GPU's name and power limit.

  python tools/bench_labelled_step.py [--reps 30]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import mil_b200  # noqa: E402,F401
from mil_b200 import _lib as L  # noqa: E402
from mil_b200 import functional as F  # noqa: E402
from mil_b200.dp import AbmilTrainer  # noqa: E402


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0), "power_limit_w": None}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit_w"] = float(r.stdout.strip().splitlines()[0])
    except Exception:
        pass
    return info


def two_pass_step(tr, X, offt, labels, buf):
    """The labelled step without row dots: forward, head + BCE through the same library kernels, backward(dM), update."""
    lib, B, C, Lf = L.lib(), offt.numel() - 1, tr.C, tr.L
    M = tr.forward(X, offt)
    v, g = tr._views(tr.params), tr._views(tr.grads)
    lws = L.workspace(lib.milb200_linear_workspace_bytes(B, C, Lf, L.F32, 1), X.device)
    L.check(lib.milb200_linear_fwd(L.ptr(M), None, L.ptr(v["head_w"]), L.ptr(v["head_b"]), L.ptr(buf["z"]), B, C, Lf,
                                   L.ACT_NONE, L.F32, L.ptr(lws), lws.numel(), L.stream_ptr()), "linear_fwd")
    L.check(lib.milb200_sigmoid_bce_fwd_bwd(L.ptr(buf["z"]), L.ptr(labels), L.ptr(buf["prob"]), L.ptr(buf["loss"]),
                                            L.ptr(buf["dz"]), B * C, L.stream_ptr()), "sigmoid_bce")
    L.check(lib.milb200_linear_bwd(L.ptr(M), None, L.ptr(v["head_w"]), L.ptr(buf["z"]), L.ptr(buf["dz"]), L.ptr(buf["dM"]),
                                   L.ptr(g["head_w"]), L.ptr(g["head_b"]), B, C, Lf, L.ACT_NONE, L.F32, 0, L.ptr(lws),
                                   lws.numel(), L.stream_ptr()), "linear_bwd")
    tr.backward(buf["dM"])
    tr.reduce_and_update()
    return buf["loss"], buf["prob"]


def graphed(fn):
    """fn captured as one CUDA graph after two eager warm-up calls on a side stream."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    return g.replay


def stats(ts):
    ts = np.asarray(ts)
    return {"ms_mean": float(ts.mean()), "ms_std": float(ts.std()), "ms_median": float(np.median(ts)),
            "ms_min": float(ts.min()), "n": int(ts.size)}


def time_alternating(fns, reps):
    times = {k: [] for k in fns}
    for _ in range(reps):
        for k, fn in fns.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            times[k].append(a.elapsed_time(b))
    return {k: stats(v) for k, v in times.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    args = ap.parse_args()
    g = torch.Generator().manual_seed(1234)                      # bench.py's bag_lengths(64, 1234)
    lens = torch.randint(100, 20001, (64,), generator=g).numpy()
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    n, B, Lf, C, D = int(off[-1]), len(lens), 1024, 2, 192
    gen = torch.Generator(device="cuda").manual_seed(1)
    X = torch.randn(n, Lf, device="cuda", generator=gen).bfloat16()
    offt = torch.from_numpy(off).cuda()
    labels = torch.nn.functional.one_hot(torch.randint(0, C, (B,), device="cuda", generator=gen), C).float()

    def trainer(C_):
        tr = AbmilTrainer(Lf, D, torch.bfloat16, device="cuda", head_classes=C_)
        tr.params.copy_(torch.randn(tr.numel, device="cuda", generator=torch.Generator(device="cuda").manual_seed(2)) * 0.03)
        return tr

    ta, tb, tc = trainer(C), trainer(C), trainer(0)
    f32 = dict(dtype=torch.float32, device="cuda")
    buf = dict(z=torch.empty(B, C, **f32), prob=torch.empty(B, C, **f32), dz=torch.empty(B, C, **f32),
               loss=torch.empty(1, **f32), dM=torch.empty(B, Lf, **f32))
    # the same step arithmetic on both routes: one step from the same parameters gives the same loss
    la, _ = ta.forward_backward_labels(X, offt, labels)
    ta_grads = ta.grads.clone()
    lb = two_pass_step(tb, X, offt, labels, buf)[0].clone()
    torch.cuda.synchronize()
    grad_err = float((ta_grads - tb.grads).abs().max() / tb.grads.abs().max())
    loss_err = float((la - lb).abs().max() / lb.abs().max())
    replay_b = graphed(lambda: two_pass_step(tb, X, offt, labels, buf))
    steps = {"a_headdot": lambda: ta.step_graphed(X, offt, labels), "b_two_pass": replay_b,
             "c_synthetic": lambda: tc.step_graphed(X, offt)}
    for fn in steps.values():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    step_t = time_alternating(steps, args.reps)

    # pool forward kernels alone
    s = torch.randn(n, device="cuda", generator=gen) * 2
    dM = torch.randn(B, Lf, device="cuda", generator=gen)
    W8 = torch.randn(8, Lf, device="cuda", generator=gen) * 0.03
    pools = {"plain": lambda: F.segment_softmax_pool(X, s, offt),
             "rowdot": lambda: F.segment_softmax_pool_rowdot(X, s, offt, dM)}
    for c in (1, 2, 4, 8):
        pools[f"headdot_C{c}"] = (lambda W: lambda: F.segment_softmax_pool_headdot(X, s, offt, W))(W8[:c].contiguous())
    for fn in pools.values():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    pool_t = time_alternating(pools, args.reps)
    x_bytes = n * Lf * 2
    for k, r in pool_t.items():
        r["x_gbs_median"] = x_bytes / r["ms_median"] / 1e6

    res = {"config": {"bags": B, "rows": n, "L": Lf, "C": C, "dtype": "bf16", "semantics": "eval", "reps": args.reps,
                      "x_bytes": x_bytes},
           "gpu": gpu_info(), "check": {"grad_rel_err_a_vs_b": grad_err, "loss_rel_err_a_vs_b": loss_err},
           "step": step_t, "pool_fwd": pool_t}
    for k, r in step_t.items():
        print(f"step {k:12s} {r['ms_mean']:7.3f} ms mean  {r['ms_std']:6.3f} std  {r['ms_median']:7.3f} median",
              file=sys.stderr)
    for k, r in pool_t.items():
        print(f"pool_fwd {k:11s} {r['ms_median'] * 1e3:8.1f} us  {r['x_gbs_median']:7.0f} GB/s of X", file=sys.stderr)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
