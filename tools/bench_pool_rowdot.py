"""Times the segmented softmax pool's two ways of forming the score gradients at the cfg-2 shapes of bench.py (64 bags of
100..20 000 rows, L = 1024, bf16; X is 1.37 GB, past the 126 MB L2):

  plain:  segment_softmax_pool (k_pool_fwd)  +  segment_softmax_pool_bwd (k_pool_bwd_stats, k_pool_bwd: re-reads X)
  rowdot: segment_softmax_pool_rowdot (k_pool_fwd<..., ROWDOT>: also writes dM_b . x_i)
          +  segment_softmax_pool_bwd_rowdot (k_pool_bwd_stats with the per-bag sweep: no pass over X)

Each phase is timed with CUDA events, the two variants alternating rep by rep, and reported as the median with the
achieved rate against the bytes the algorithm must move.  Prints one JSON line, with the GPU's name and power limit.

  python tools/bench_pool_rowdot.py [--reps 30]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import mil_b200  # noqa: E402,F401
from mil_b200 import functional as F  # noqa: E402


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0), "power_limit_w": None}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit_w"] = float(r.stdout.strip().splitlines()[0])
    except Exception:
        pass
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    args = ap.parse_args()
    g = torch.Generator().manual_seed(1234)                      # bench.py's bag_lengths(64, 1234)
    lens = torch.randint(100, 20001, (64,), generator=g).numpy()
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    n, B, L = int(off[-1]), len(lens), 1024
    gen = torch.Generator(device="cuda").manual_seed(1)
    X = torch.randn(n, L, device="cuda", generator=gen).bfloat16()
    s = torch.randn(n, device="cuda", generator=gen) * 2
    dM = torch.randn(B, L, device="cuda", generator=gen)
    offt = torch.from_numpy(off).cuda()

    state = {}

    def plain_fwd():
        state["M"] = F.segment_softmax_pool(X, s, offt)[0]

    def plain_bwd():
        state["ds"] = F.segment_softmax_pool_bwd(X, s, offt, dM, state["M"], want_attn=False)[0]

    def rowdot_fwd():
        state["M2"], _, _, _, state["rowdot"] = F.segment_softmax_pool_rowdot(X, s, offt, dM)

    def rowdot_bwd():
        state["ds2"] = F.segment_softmax_pool_bwd_rowdot(s, offt, dM, state["M2"], state["rowdot"], want_attn=False)[0]

    phases = {"plain_fwd": plain_fwd, "plain_bwd": plain_bwd, "rowdot_fwd": rowdot_fwd, "rowdot_bwd": rowdot_bwd}
    for fn in phases.values():                                    # warm-up: module load, workspace growth
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    assert torch.equal(state["M"], state["M2"]) and torch.equal(state["ds"], state["ds2"]), "the two variants differ"

    times = {k: [] for k in phases}
    for _ in range(args.reps):
        for variant in ("plain", "rowdot"):                       # alternate the variants; each phase has its own events
            for ph in ("fwd", "bwd"):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                phases[f"{variant}_{ph}"]()
                b.record()
                b.synchronize()
                times[f"{variant}_{ph}"].append(a.elapsed_time(b))

    small = 2 * B * L * 4 + (B + 1) * 4                           # dM and M (or dM twice), offsets
    algo_bytes = {"plain_fwd": n * (L * 2 + 4) + B * L * 4 + (B + 1) * 4,
                  "plain_bwd": n * (L * 2 + 4 + 4) + small,
                  "rowdot_fwd": n * (L * 2 + 4 + 4) + 2 * B * L * 4 + (B + 1) * 4,
                  "rowdot_bwd": n * (4 + 4 + 4) + small}
    res = {"config": {"bags": B, "rows": n, "L": L, "dtype": "bf16", "reps": args.reps}, "gpu": gpu_info(), "phases": {}}
    for k, ts in times.items():
        med = float(np.median(ts))
        res["phases"][k] = {"ms_median": med, "ms_min": float(np.min(ts)), "bytes": algo_bytes[k],
                            "gbs": algo_bytes[k] / med / 1e6}
    res["pair_ms"] = {v: res["phases"][v + "_fwd"]["ms_median"] + res["phases"][v + "_bwd"]["ms_median"]
                      for v in ("plain", "rowdot")}
    for k, r in res["phases"].items():
        print(f"{k:11s} {r['ms_median'] * 1e3:8.1f} us  {r['gbs']:7.0f} GB/s", file=sys.stderr)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
