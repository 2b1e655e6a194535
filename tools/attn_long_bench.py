"""Causal self-attention past 256 positions and the GQA backward (run on the B200 box, one process tree):
    python tools/attn_long_bench.py [--out FILE]
1. forward: the routed kernels (attn_tm_kernel at L <= 256, attn_tml_kernel above) against the TCAVP_ATTN_TCGEN05=0 routes
   (attn_flash_kernel at L <= 256, the SIMT attn_warp_kernel above), each in a child process;
2. backward: tcavp_attention_bwd_owned with the forward's logsumexp (key-blocked attn_bwd_kv_kernel + attn_bwd_q_kernel, or
   attn_bwd_tc_kernel for MHA at <= 256 positions) against ops.attention_bwd(o=None), the SIMT attn_bwd_kernel, at L <= 768;
3. whole steps: stage1_forward + backward of the 768-class model at L = 16 + 1024, and the trajectory fine-tune step (FineTuner) of
   the 768-class model at L = 528 and of the Llama-3.2-1B shape at L = 144 (its GQA backward): tokens / s and the attention share of
   the LaunchProfiler groups.
Every launch is timed with CUDA events, the L2 flushed (256 MB write) before each timed launch, median of 20; batches are sized so the
QKV activation alone exceeds the 126 MB L2.  The card name and power limit are printed first."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
SHAPES = [("768-class", 12, 12, 64), ("llama-3.2-1b", 32, 8, 64), ("7b", 32, 32, 128)]
LENGTHS = [144, 257, 528, 1040]


def _batch(L, ld):
    return max(2, -(-200_000_000 // (L * ld * 2)))


def _time(call, n=20):
    for _ in range(3):
        call()
    torch.cuda.synchronize()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ts = []
    for _ in range(n):
        flush.zero_()
        e0.record()
        call()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    return sorted(ts)[len(ts) // 2]


def _problem(name, nh, nkv, dh, L):
    nq, nk = nh * dh, nkv * dh
    ld = nq + 2 * nk
    B = _batch(L, ld)
    g = torch.Generator(device="cuda").manual_seed(L)
    qkv = torch.randn(B * L, ld, device="cuda", generator=g).to(torch.bfloat16)
    km = torch.ones(B, L, dtype=torch.int32, device="cuda")
    return B, nq, nk, ld, qkv, km


def forward_child():
    from tcavp_b200 import ops
    rows = []
    for name, nh, nkv, dh in SHAPES:
        for L in LENGTHS:
            B, nq, nk, ld, qkv, km = _problem(name, nh, nkv, dh, L)
            out = torch.empty(B * L, nq, dtype=torch.bfloat16, device="cuda")

            def call():
                ops.attention(qkv, qkv[:, nq:], qkv[:, nq + nk:], out, B=B, H=nh, Hkv=nkv, Tq=L, Tk=L, dh=dh, q_strides=(L * ld, ld),
                              k_strides=(L * ld, ld), v_strides=(L * ld, ld), o_strides=(L * nq, nq), scale=dh ** -0.5, causal=True, key_mask=km)
            us = _time(call)
            fl = 4.0 * B * nh * L * L * dh * 0.5
            by = 2.0 * B * L * (2 * nq + 2 * nk)
            rows.append(dict(pass_="fwd", shape=name, L=L, B=B, kernel=ops.last_kernel(), us=round(us, 1), tflops=round(fl / us / 1e6, 1),
                             gbs=round(by / us / 1e3, 1)))
            print(json.dumps(rows[-1]), flush=True)
            del qkv, out
    return rows


def backward():
    from tcavp_b200 import ops
    rows = []
    for name, nh, nkv, dh in SHAPES:
        for L in LENGTHS:
            B, nq, nk, ld, qkv, km = _problem(name, nh, nkv, dh, L)
            out = torch.empty(B * L, nq, dtype=torch.bfloat16, device="cuda")
            lse = torch.empty(B * nh * L, dtype=torch.float32, device="cuda")
            s = (L * ld, ld)
            ops.attention(qkv, qkv[:, nq:], qkv[:, nq + nk:], out, B=B, H=nh, Hkv=nkv, Tq=L, Tk=L, dh=dh, q_strides=s, k_strides=s, v_strides=s,
                          o_strides=(L * nq, nq), scale=dh ** -0.5, causal=True, key_mask=km, lse=lse)
            dout = torch.randn(B * L, nq, device="cuda").to(torch.bfloat16)
            d = torch.empty_like(qkv)
            fl = 10.0 * B * nh * L * L * dh * 0.5

            def new():
                ops.attention_bwd_owned(qkv, qkv[:, nq:], qkv[:, nq + nk:], dout, d, d[:, nq:], d[:, nq + nk:], B=B, H=nh, Hkv=nkv, Tq=L, Tk=L,
                                        dh=dh, q_strides=s, k_strides=s, v_strides=s, do_strides=(L * nq, nq), dq_strides=s, dk_strides=s,
                                        dv_strides=s, scale=dh ** -0.5, causal=True, key_mask=km, o=out, o_strides=(L * nq, nq), lse=lse)
            us = _time(new)
            row = dict(pass_="bwd", shape=name, L=L, B=B, kernel=ops.last_kernel(), us=round(us, 1), tflops=round(fl / us / 1e6, 1))
            if L <= 768:
                dk = torch.zeros(B * L, nk, dtype=torch.float32, device="cuda")
                dv = torch.zeros_like(dk)

                def simt():
                    ops.attention_bwd(qkv, qkv[:, nq:], qkv[:, nq + nk:], dout, d, dk, dv, B=B, H=nh, Hkv=nkv, Tq=L, Tk=L, dh=dh, q_strides=s,
                                      k_strides=s, v_strides=s, do_strides=(L * nq, nq), dq_strides=s, dk_strides=(L * nk, nk),
                                      dv_strides=(L * nk, nk), scale=dh ** -0.5, causal=True, key_mask=km)
                us0 = _time(simt, n=5)       # accumulates into dk / dv across calls: only the time is used
                row.update(simt_kernel=ops.last_kernel(), simt_us=round(us0, 1), simt_tflops=round(fl / us0 / 1e6, 1))
                del dk, dv
            rows.append(row)
            print(json.dumps(row), flush=True)
            del qkv, out, lse, dout, d
            torch.cuda.empty_cache()
    return rows


def stage1_step():
    import time
    import tcavp_b200 as T
    from tcavp_b200 import ops
    from oracle import restated
    mc = dict(T.MODEL_PRESETS["cfg1"])
    lc = T.resolve_llama(mc["base_model_name"])
    B, l_text = 8, 1024
    s = T.make_scenes(B, mc["seq_len"], mc["out_len"], l_text=l_text, vocab=lc["vocab_size"], seed=3)
    labels = restated.stage1_labels(s["input_ids"], s["attention_mask"], 600).cuda()
    m = T.MultiModalTrajectoryModel(**mc, compute_dtype="bf16")
    sd = m.state_dict()
    T.deterministic_fill_(sd, 13)
    m.load_state_dict(sd, strict=True)
    m = m.cuda().eval()
    args = (s["vision"].cuda(), s["input_ids"].cuda(), s["attention_mask"].cuda(), labels)

    def step():
        m.zero_grad(set_to_none=True)
        m.stage1_forward(*args).loss.backward()
    for _ in range(2):
        step()
    torch.cuda.synchronize()
    n = 5
    t0 = time.perf_counter()
    for _ in range(n):
        step()
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) / n * 1e3
    with ops.LaunchProfiler() as prof:
        step()
    groups = prof.summary()["groups"]
    attn = [g for g in groups if g["kernel"].startswith("attn_")]
    L = 16 + l_text
    row = dict(pass_="stage1_step", model="768-class (cfg1)", B=B, L=L, ms=round(ms, 2), tokens_per_s=round(B * L / ms * 1e3),
               attention_share=round(sum(g["share"] for g in attn), 4), attention_groups=attn)
    print(json.dumps(row), flush=True)
    return row


def finetune_step(label, preset, B, l_text, backbone=None):
    """The trajectory fine-tune step (FineTuner: forward, hand-written backward, AdamW; eager launches so that the LaunchProfiler sees
    every kernel) at L = 16 + l_text: tokens / s and the attention share of the profiled step."""
    import time
    import warnings
    import tcavp_b200 as T
    from tcavp_b200 import ops
    warnings.simplefilter("ignore")
    mc = dict(T.MODEL_PRESETS[preset])
    if backbone:
        mc["base_model_name"] = backbone
    lc = T.resolve_llama(mc["base_model_name"])
    s = T.make_scenes(B, mc["seq_len"], mc["out_len"], vision_dim=mc.get("vision_dim", 512), l_text=l_text, vocab=lc["vocab_size"], seed=3)
    m = T.MultiModalTrajectoryModel(**mc, compute_dtype="bf16")
    sd = m.state_dict()
    T.deterministic_fill_(sd, 13)
    m.load_state_dict(sd, strict=True)
    m = m.cuda().eval()
    ft = T.FineTuner(m, lr=1e-6, use_cuda_graph=False)
    args = (s["x"].cuda(), s["vision"].cuda(), ["ctx"] * B, s["polygon"].cuda(), s["poly_len"], s["y"].cuda(), s["norm_stat"],
            s["input_ids"].cuda(), s["attention_mask"].cuda())
    for _ in range(2):
        ft.step(*args)
    torch.cuda.synchronize()
    n = 5
    t0 = time.perf_counter()
    for _ in range(n):
        ft.step(*args)
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) / n * 1e3
    with ops.LaunchProfiler() as prof:
        ft.step(*args)
    groups = prof.summary()["groups"]
    attn = [g for g in groups if g["kernel"].startswith("attn_")]
    L = 16 + l_text
    row = dict(pass_="finetune_step", model=label, B=B, L=L, ms=round(ms, 2), tokens_per_s=round(B * L / ms * 1e3),
               attention_share=round(sum(g["share"] for g in attn), 4), attention_groups=attn[:6])
    print(json.dumps(row), flush=True)
    del ft, m
    torch.cuda.empty_cache()
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    a = ap.parse_args()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    print(f"card: {card}", flush=True)
    res = dict(card=card, forward={}, backward=None, stage1=None, finetune=None)
    for flag in ("1", "0"):
        print(f"--- forward, TCAVP_ATTN_TCGEN05={flag}", flush=True)
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child-forward"], env=dict(os.environ, TCAVP_ATTN_TCGEN05=flag),
                           capture_output=True, text=True)
        sys.stdout.write(r.stdout)
        sys.stderr.write(r.stderr[-2000:])
        res["forward"][flag] = [json.loads(x) for x in r.stdout.splitlines() if x.startswith("{")]
    import tcavp_b200.lib as L_
    L_.build()
    print("--- backward", flush=True)
    res["backward"] = backward()
    print("--- stage-1 step", flush=True)
    res["stage1"] = stage1_step()
    print("--- fine-tune steps", flush=True)
    res["finetune"] = [finetune_step("768-class (cfg1)", "cfg1", 64, 512),
                       finetune_step("Llama-3.2-1B shape (llama-1b-gqa: 32/8 heads of 64, 16 layers)", "cfg1", 64, 128, backbone="llama-1b-gqa")]
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "--child-forward":
        forward_child()
    else:
        main()
