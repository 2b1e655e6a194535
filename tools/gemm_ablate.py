"""Times tcavp_gemm for ~1.5 s per shape with SM clock / power sampled through NVML, and reports per-clock tensor-pipe
utilisation (TF/s / (148 SM x 8192 FLOP/clk x clk))."""
import os, sys, time, threading, statistics, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import tcavp_b200.lib as L
L.build()
from tcavp_b200 import ops
import pynvml
pynvml.nvmlInit()
h = pynvml.nvmlDeviceGetHandleByIndex(0)
dev = torch.device("cuda:0")
shapes = [(147456, 768, 3072), (147456, 6144, 768), (147456, 2304, 784), (36864, 4096, 4096)]
if len(sys.argv) > 1:
    shapes = [tuple(int(v) for v in s.split("x")) for s in sys.argv[1:]]
for (M, N, K) in shapes:
    a = (torch.randn(M, K, device=dev) * 0.5).bfloat16(); w = (torch.randn(N, K, device=dev) * 0.05).bfloat16()
    out = torch.empty(M, N, device=dev, dtype=torch.bfloat16)
    for _ in range(3): ops.gemm(a, w, out)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ops.gemm(a, w, out); torch.cuda.synchronize()
    e0.record(); ops.gemm(a, w, out); e1.record(); torch.cuda.synchronize()
    ms_est = e0.elapsed_time(e1)
    n = max(20, int(1500.0 / ms_est))
    clk, pw, stop = [], [], False
    def sample():
        while not stop:
            clk.append(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)); pw.append(pynvml.nvmlDeviceGetPowerUsage(h) / 1e3)
            time.sleep(0.05)
    t = threading.Thread(target=sample); t.start()
    probe = torch.zeros(2, dtype=torch.int64, device=dev)
    side = torch.cuda.Stream()
    import ctypes
    if os.environ.get("CLOCK_PROBE"):   # perturbs the measurement (the probe warp shares one SM with a GEMM CTA)
        L.check(L.load().tcavp_clock_probe(ctypes.c_void_p(probe.data_ptr()), ctypes.c_ulonglong(int(0.6 * ms_est * n * 1e6)), ctypes.c_void_p(side.cuda_stream)))
    e0.record()
    for _ in range(n): ops.gemm(a, w, out)
    e1.record(); torch.cuda.synchronize()
    stop = True; t.join()
    ms = e0.elapsed_time(e1) / n
    tf = 2.0 * M * N * K / ms / 1e9
    c = statistics.median(clk[len(clk) // 2:]); p = statistics.median(pw[len(pw) // 2:])
    print(f"M{M} N{N} K{K}: {ms*1e3:.1f} us {tf:.0f} TF/s  clk {c:.0f} MHz  {p:.0f} W  util/clk {tf*1e12/(148*8192*c*1e6):.3f}  probe clk {float(probe[0])/max(float(probe[1]),1)*1e3:.0f} MHz -> util {tf*1e12/(148*8192*max(float(probe[0]),1)/max(float(probe[1]),1)*1e9):.3f}", flush=True)
