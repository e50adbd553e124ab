import os, sys, torch, numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import mil_b200
from mil_b200.dp import AbmilTrainer
B1, N1 = 32, 512
gen = torch.Generator(device="cuda").manual_seed(1)
X1 = torch.randn(B1 * N1, 1024, device="cuda", generator=gen)
off1 = torch.arange(0, B1 * N1 + 1, N1, dtype=torch.int32, device="cuda")
for flag in ("1", "0"):
    os.environ["MILB200_TF32X3"] = flag
    tr = AbmilTrainer(L_feat=1024, D=192, compute_dtype=torch.float32)
    for _ in range(5): tr.step(X1, off1)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(20): tr.step(X1, off1)
    b.record(); torch.cuda.synchronize()
    print("TF32X3=%s: %.3f ms/step, %.0f bags/s" % (flag, a.elapsed_time(b)/20, B1*20/(a.elapsed_time(b)/1e3)))
