"""A/B timing of the LLM self-attention kernels on the bench shapes (run on the B200 box):
    python tools/attn_bench.py            # tcgen05 kernel (attention_tm.cu) and, in a child process, the mma.sync kernel
Prints microseconds per launch, achieved TFLOP/s (causal FLOPs) and the bytes-once bandwidth (q, k, v read + o written)."""
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
SHAPES = [("cfg2", 1024, 12, 12, 64), ("cfg3", 256, 32, 32, 128), ("gqa", 512, 32, 8, 64)]


def run():
    from tcavp_b200 import ops
    import tcavp_b200.lib as L_
    L_.build()
    L = 144
    for name, B, nh, nkv, dh in SHAPES:
        nq, nk = nh * dh, nkv * dh
        ld = nq + 2 * nk
        qkv = (torch.randn(B * L, ld, device="cuda") * 0.5).to(torch.bfloat16)
        out = torch.empty(B * L, nq, dtype=torch.bfloat16, device="cuda")
        km = torch.ones(B, L, dtype=torch.int32, device="cuda")

        def call():
            ops.attention(qkv, qkv[:, nq:], qkv[:, nq + nk:], out, B=B, H=nh, Hkv=nkv, Tq=L, Tk=L, dh=dh, q_strides=(L * ld, ld), k_strides=(L * ld, ld),
                          v_strides=(L * ld, ld), o_strides=(L * nq, nq), scale=dh ** -0.5, causal=True, key_mask=km)
        for _ in range(5):
            call()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
        ts = []
        for _ in range(20):
            flush.zero_()                          # L2 flush between timed launches
            e0.record()
            call()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e3)
        us = sorted(ts)[len(ts) // 2]
        fl = 4.0 * B * nh * L * L * dh * 0.5
        by = 2.0 * B * L * (2 * nq + 2 * nk)
        print(f"{os.environ.get('TCAVP_ATTN_TCGEN05', '1')} {name}: {us:8.1f} us  {fl / us / 1e6:7.1f} TFLOP/s  {by / us / 1e3:7.1f} GB/s", flush=True)


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "child":
        run()
    else:
        for flag in ("1", "0"):
            print(f"--- TCAVP_ATTN_TCGEN05={flag}", flush=True)
            subprocess.run([sys.executable, os.path.abspath(__file__), "child"], env=dict(os.environ, TCAVP_ATTN_TCGEN05=flag), check=False)
