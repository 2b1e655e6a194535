"""GPU-box check of tcavp_gemm (bf16 tcgen05 paths) against torch matmul + CUDA-event timings per shape.
    python tools/gemm_check.py [--time] [--big]
Run under `timeout` — a barrier mistake in a new kernel variant hangs instead of failing."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import tcavp_b200.lib as L  # noqa: E402

L.build()
from tcavp_b200 import ops  # noqa: E402

dev = torch.device("cuda:0")
torch.manual_seed(0)
SHAPES = [  # (M, N, K)  incl. ragged M / N / K tails
    (2048, 256, 64), (2048, 512, 768), (4096 + 77, 768, 768), (147456, 2304, 784), (147456, 768, 768), (147456, 6144, 768),
    (147456, 768, 3072), (2048 + 130, 320, 200), (36864, 12288, 4096), (36864, 4096, 4096), (36864, 22016, 4096), (36864, 4096, 11008),
    (36864 + 300, 11008 + 64, 4096),
]
if "--big" in sys.argv:      # the 7B-class shapes only (W larger than the 40 MB L2 panel budget)
    SHAPES = [s for s in SHAPES if s[2] >= 4096]
timing = "--time" in sys.argv
for (M, N, K) in SHAPES:
    a = (torch.randn(M, K, device=dev) * 0.5).bfloat16()
    w = (torch.randn(N, K, device=dev) * 0.05).bfloat16()
    bias = torch.randn(N, device=dev)
    res = torch.randn(M, N, device=dev).bfloat16()
    out = torch.empty(M, N, device=dev, dtype=torch.bfloat16)
    ops.gemm(a, w, out, bias=bias, residual=res)
    torch.cuda.synchronize()
    rows = torch.randint(0, M, (512,), device=dev)
    rows[:4] = torch.tensor([0, M - 1, min(M - 1, 128), min(M - 1, 255)], device=dev)
    want = a[rows].float() @ w.float().t() + bias + res[rows].float()
    err = float((out[rows].float() - want).abs().max())
    ok = err < 0.02 * float(want.abs().max()) + 0.05
    line = f"M{M} N{N} K{K}: max|err| {err:.4f} (ref max {float(want.abs().max()):.2f}) {'ok' if ok else 'FAIL'}"
    if timing:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(3):
            ops.gemm(a, w, out)
        e0.record()
        n = 10
        for _ in range(n):
            ops.gemm(a, w, out)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n
        line += f"  {ms * 1e3:.1f} us  {2.0 * M * N * K / ms / 1e9:.1f} TF/s"
    print(line, flush=True)
    if not ok:
        sys.exit(1)
print("gemm_check ok")
