"""Where does the o_proj-shaped GEMM (M = 147 456, N = K = 768: the slowest K = 768 group of the cfg2 step) lose its time?
Times tcavp_gemm on that shape with the epilogue terms switched on one at a time (device events, ~0.3 s per variant, A-B-A order so a
clock drift shows up as a difference between the two passes of the same variant), next to the QKV / gate-up shapes of the same step.
    python tools/oproj_ablate.py"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import tcavp_b200.lib as L  # noqa: E402

L.build()
from tcavp_b200 import ops  # noqa: E402

dev = torch.device("cuda:0")
M, H, Kx = 147456, 768, 784
a = (torch.randn(M, H, device=dev) * 0.5).bfloat16()
w = (torch.randn(H, H, device=dev) * 0.05).bfloat16()
res = (torch.randn(M, Kx, device=dev) * 0.5).bfloat16()
out_c = torch.empty(M, H, device=dev, dtype=torch.bfloat16)
out_s = torch.empty(M, Kx, device=dev, dtype=torch.bfloat16)
ss = torch.zeros(M, dtype=torch.int64, device=dev)
bias = torch.randn(H, device=dev)
wq = (torch.randn(2304, Kx, device=dev) * 0.05).bfloat16()
outq = torch.empty(M, 2304, device=dev, dtype=torch.bfloat16)
wg = (torch.randn(6144, H, device=dev) * 0.05).bfloat16()
outg = torch.empty(M, 3072, device=dev, dtype=torch.bfloat16)

VARIANTS = [
    ("plain, contiguous out", lambda: ops.gemm(a, w, out_c)),
    ("plain, out row stride 784", lambda: ops.gemm(a, w, out_s, ldo=Kx)),
    ("+ bias", lambda: ops.gemm(a, w, out_c, bias=bias)),
    ("+ residual (row stride 784), contiguous out", lambda: ops.gemm(a, w, out_c, residual=res, ldr=Kx)),
    ("+ residual in place (the step's form, no statistics)", lambda: ops.gemm(a, w, res, ldo=Kx, residual=res, ldr=Kx)),
    ("+ residual in place + row statistics (the step's o_proj)", lambda: ops.gemm(a, w, res, ldo=Kx, residual=res, ldr=Kx, sumsq_out=ss)),
    ("QKV shape N 2304 K 784 plain", lambda: ops.gemm(res, wq, outq, K=Kx)),
    ("gate/up shape N 6144 K 768 SwiGLU", lambda: ops.gemm(a, wg, outg, act=ops.ACT_SWIGLU)),
]


def timed(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


for name, fn in VARIANTS:
    for _ in range(3):
        fn()
torch.cuda.synchronize()
rows = {name: [] for name, _ in VARIANTS}
for rnd in range(2):
    for name, fn in VARIANTS:
        rows[name].append(timed(fn, 400 if "shape" not in name else 150))
for name, _ in VARIANTS:
    N, K = (2304, Kx) if "QKV" in name else (6144, H) if "gate" in name else (H, H)
    fl = 2.0 * M * N * K
    ms = rows[name]
    print(f"{name:58s} {ms[0] * 1e3:7.1f} / {ms[1] * 1e3:7.1f} us   {fl / ms[0] / 1e9:6.0f} / {fl / ms[1] / 1e9:6.0f} TF/s", flush=True)
