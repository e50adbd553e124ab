"""Measures the resident feeder (feeder.ResidentBagFeeder: slide set in device memory, batches sampled and packed on the
device) against the host feeder (feeder.PackedBagFeeder) and a fixed device-resident batch, at cfg-2 shapes: slides of
100..20 000 rows (bench.py's cfg-2 lengths), L = 1024, bf16 compute, 64 bags per batch.

  upload:   construction of the resident store from fp32 numpy slides (native packer -> pinned staging -> H2D)
  kernels:  per cfg-2 batch, CUDA-event time of select_rows (augmentation subsets) and gather_rows, and the gather's
            GB/s (read + write bytes) next to a Tensor.copy_ of the same bytes in the same run; the batch (~1.3 GB) and
            its source rows are far past the 126 MB L2
  epochs:   wall-clock bags/s over whole epochs (256 slides, 4 batches an epoch), augmentation off and on, for
            ResidentBagFeeder + AbmilTrainer.step, PackedBagFeeder + step on the same slides, and one fixed device
            batch of the same shape + step
  scale:    ResidentBagFeeder alone on a >= 20 GB store built from CUDA sources (device-to-device upload, ten epochs)

Prints one JSON line with the GPU's name and power limit (and writes it to --out when given).

  python tools/bench_resident_feeder.py [--slides 256] [--epochs 2] [--device-epochs 30] [--out <json>]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import mil_b200  # noqa: E402
from mil_b200 import feeder  # noqa: E402
from mil_b200 import functional as F  # noqa: E402
from mil_b200.dp import AbmilTrainer  # noqa: E402

LEN_LO, LEN_HI, L_FEAT, B = 100, 20000, 1024, 64


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0), "power_limit_w": None}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit_w"] = float(r.stdout.strip().splitlines()[0])
    except Exception:
        pass
    return info


def lengths(n, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randint(LEN_LO, LEN_HI + 1, (n,), generator=g).tolist()


def types_for(n):
    return ["Biopsy" if i % 2 == 0 else "Resection" for i in range(n)]


def event_ms(fns, reps):
    """CUDA-event time (ms) of each fn, alternating fn by fn, rep by rep; returns per-fn median and min."""
    times = [[] for _ in fns]
    for _ in range(reps):
        for j, fn in enumerate(fns):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            times[j].append(a.elapsed_time(b))
    return [{"median_ms": float(np.median(t)), "min_ms": float(np.min(t))} for t in times]


def run_epochs(make_iter, trainer, epochs):
    """Wall-clock bags/s of `epochs` epochs (after one warm-up epoch) of trainer.step over make_iter(epoch)."""
    def one(epoch):
        bags = 0
        for X, off, ids in make_iter(epoch):
            trainer.step(X, off)
            bags += len(ids)
        return bags
    one(0)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    bags = sum(one(1 + e) for e in range(epochs))
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return {"bags": bags, "seconds": dt, "bags_per_s": bags / dt}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--slides", type=int, default=256)
    ap.add_argument("--epochs", type=int, default=2, help="timed epochs of the PackedBagFeeder route (seconds each)")
    ap.add_argument("--device-epochs", type=int, default=30, help="timed epochs of the resident and fixed-batch routes")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--scale-gb", type=float, default=20.5)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_resident_feeder.py measures the GPU and needs one")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res = {"gpu": gpu_info(), "slides": args.slides, "L": L_FEAT, "batch_bags": B, "dtype": "bf16"}

    lens = lengths(args.slides, 7)
    rng = np.random.default_rng(1)
    slides = [rng.random((n, L_FEAT), dtype=np.float32) - 0.5 for n in lens]
    types = types_for(args.slides)
    src_bytes = sum(s.nbytes for s in slides)

    # ---- upload --------------------------------------------------------------------------------------------------
    feeders = {}
    for aug in (False, True):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        feeders[aug] = feeder.ResidentBagFeeder(slides, B, L_FEAT, slide_types=types, augment=aug, shuffle=True, seed=3)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if aug:
            res["upload"] = {"source_fp32_GB": src_bytes / 1e9, "store_bf16_GB": feeders[aug].store.numel() * 2 / 1e9,
                             "seconds": dt, "source_GB_per_s": src_bytes / dt / 1e9}
    fa = feeders[True]

    # ---- kernels at one cfg-2 batch ------------------------------------------------------------------------------
    ids = list(range(B))
    counts = [fa.counts[i] for i in ids]
    off_h = np.zeros(B + 1, dtype=np.int32)
    np.cumsum(counts, out=off_h[1:])
    n = int(off_h[-1])
    ids_d = torch.tensor(ids, dtype=torch.int32, device=dev)
    off_d = torch.from_numpy(off_h).to(dev)
    src = torch.empty(n, dtype=torch.int64, device=dev)
    out = torch.empty((n, L_FEAT), dtype=torch.bfloat16, device=dev)
    cp_src = torch.empty_like(out).normal_()
    cp_dst = torch.empty_like(out)
    sel = lambda: F.select_rows(fa.slide_start, ids_d, off_d, n, 3, 0, 0, out=src)        # noqa: E731
    F.select_rows(fa.slide_start, ids_d, off_d, n, 3, 0, 0, out=src)
    gat = lambda: F.gather_rows(fa.store, src, out=out)                                    # noqa: E731
    cpy = lambda: cp_dst.copy_(cp_src)                                                     # noqa: E731
    for fn in (sel, gat, cpy):
        fn()
    t_sel, t_gat, t_cpy = event_ms([sel, gat, cpy], args.reps)
    nbytes = 2 * n * L_FEAT * 2                      # read + write
    res["kernels"] = {"rows": n, "batch_GB": n * L_FEAT * 2 / 1e9,
                      "select_rows": t_sel, "gather_rows": t_gat, "copy_": t_cpy,
                      "gather_GB_per_s": nbytes / (t_gat["median_ms"] * 1e-3) / 1e9,
                      "copy_GB_per_s": nbytes / (t_cpy["median_ms"] * 1e-3) / 1e9,
                      "gather_over_copy": t_cpy["median_ms"] / t_gat["median_ms"]}
    del cp_src, cp_dst, out, src

    # ---- epochs ---------------------------------------------------------------------------------------------------
    torch.manual_seed(0)
    module = mil_b200.ABMIL(None, L=L_FEAT).to(dev)
    tr = AbmilTrainer(L_FEAT, 192, torch.bfloat16, device=dev)
    tr.load_from(module)
    epochs = {}
    for aug in (False, True):
        fr = feeders[aug]

        def resident_iter(epoch, fr=fr):
            fr.set_epoch(epoch)
            return iter(fr)
        r_res = run_epochs(resident_iter, tr, args.device_epochs)
        fp = feeder.PackedBagFeeder(slides, B, L_FEAT, device=dev, slide_types=types, augment=aug, shuffle=True, seed=3)

        def packed_iter(epoch, fp=fp):
            fp.set_epoch(epoch)
            return iter(fp)
        r_pack = run_epochs(packed_iter, tr, args.epochs)
        del fp
        fr.set_epoch(0)
        X0, off0, ids0 = next(iter(fr))
        X0, off0 = X0.clone(), off0.clone()
        n_batches = len(fr)

        def fixed_iter(epoch):
            return ((X0, off0, ids0) for _ in range(n_batches))
        r_fix = run_epochs(fixed_iter, tr, args.device_epochs)
        epochs["augment" if aug else "no_augment"] = {
            "resident": r_res, "packed": r_pack, "fixed_device_batch": r_fix,
            "resident_over_packed": r_res["bags_per_s"] / r_pack["bags_per_s"]}
        torch.cuda.empty_cache()
    res["epochs"] = epochs
    res["epochs"]["batches_per_epoch"] = len(fa)
    del feeders, fa, slides
    torch.cuda.empty_cache()

    # ---- dataset scale from CUDA sources ---------------------------------------------------------------------------
    row_bytes = L_FEAT * 2
    big_lens = []
    g_lens = lengths(100_000, 11)
    while sum(big_lens) * row_bytes < args.scale_gb * 1e9:
        big_lens.append(g_lens[len(big_lens)])
    total = sum(big_lens)
    base = torch.empty((total, L_FEAT), dtype=torch.bfloat16, device=dev).uniform_(-1, 1)
    starts = np.concatenate([[0], np.cumsum(big_lens)])
    cuda_slides = [base[starts[i]:starts[i + 1]] for i in range(len(big_lens))]
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fb = feeder.ResidentBagFeeder(cuda_slides, B, L_FEAT, slide_types=types_for(len(big_lens)), augment=True,
                                  shuffle=True, seed=5)
    torch.cuda.synchronize()
    t_up = time.perf_counter() - t0
    del cuda_slides, base
    torch.cuda.empty_cache()
    for X, off, ids in fb:                          # warm-up epoch
        pass
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    bags = rows = 0
    for epoch in range(1, 11):
        fb.set_epoch(epoch)
        for X, off, ids in fb:
            bags += len(ids)
            rows += X.shape[0]
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    res["scale"] = {"slides": len(big_lens), "store_GB": total * row_bytes / 1e9, "upload_seconds": t_up,
                    "upload_GB_per_s": total * row_bytes / t_up / 1e9, "epochs": 10, "batches_per_epoch": len(fb), "bags": bags,
                    "seconds": dt, "feeder_bags_per_s": bags / dt,
                    "feeder_GB_per_s_read_plus_write": 2 * rows * row_bytes / dt / 1e9}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
