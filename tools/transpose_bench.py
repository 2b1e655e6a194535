import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tcavp_b200 import ops
for (M, N, dt) in [(73728, 768, torch.bfloat16), (73728, 1536, torch.bfloat16), (73728, 768, torch.float32)]:
    x = torch.randn(M, N, device='cuda').to(dt)
    out = torch.empty(N, M, device='cuda', dtype=dt)
    for _ in range(3): ops.transpose(x, out, rows=M, cols=N)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(20): ops.transpose(x, out, rows=M, cols=N)
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 20
    print(M, N, dt, f"{ms*1e3:.1f} us  {2*M*N*x.element_size()/ms/1e6:.0f} GB/s", bool(torch.equal(out, x.t())))
