"""Text generation on a B200: the eager KV-cache loop (generate_ids, torch RNG) against the seeded CUDA-graph device loop (seed=...), in
one process:

    python tools/generate_bench.py --out generate_bench.json

* Backbones: the 768-class Llama (cfg1), the Llama-3.2-1B shape (16 layers, H 2048, GQA 32 / 8, vocabulary 128 256; random weights) and
  GPT-2 (cfg1-gpt2).  B in {1, 16, 128}, prefix 144 positions (16 image tokens + 128 prompt ids), 128 new tokens, the reference's
  sampling parameters (temperature 0.9, top-k 40, top-p 0.9, repetition penalty 1.2, no-repeat-3-gram), no EOS, so both paths run
  all 128 steps.
* Each (shape, B) runs eager, device, eager, device after one warm-up call of each (the device loop's graph is captured there).  A
  call's time includes the prefill; ms per token = call time / 128.
* Floor: one read of the decoder weights plus lm_head per step at the 6.53 TB/s copy peak (DESIGN §5), computed from the shapes.
* Per-kernel breakdown: one decode iteration of the device loop run eagerly under ops.LaunchProfiler (the launches the graph replays).
* The card name and power limit are read in the same run."""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from fp8_bench import gpu_info  # noqa: E402

COPY_PEAK_TBS = 6.53
LLAMA32_1B = dict(vocab_size=128256, hidden_size=2048, intermediate_size=8192, num_hidden_layers=16, num_attention_heads=32,
                  num_key_value_heads=8, head_dim=64, rms_norm_eps=1e-5, rope_theta=500000.0, max_position_embeddings=131072,
                  tie_word_embeddings=True, rope_scaling=dict(rope_type="llama3", factor=32.0, low_freq_factor=1.0, high_freq_factor=4.0,
                                                              original_max_position_embeddings=8192))
SHAPES = {"llama-768": dict(preset="cfg1"), "llama3.2-1b": dict(preset="cfg1", base=LLAMA32_1B), "gpt2": dict(preset="cfg1-gpt2")}
Q_TOKENS, PROMPT, NEW = 16, 128, 128


def build(shape):
    import tcavp_b200 as T
    s = SHAPES[shape]
    cfg = dict(T.MODEL_PRESETS[s["preset"]])
    if "base" in s:
        cfg["base_model_name"] = s["base"]
    m = T.MultiModalTrajectoryModel(**cfg, compute_dtype="bf16", llm_param_dtype=torch.bfloat16, llm_device="cuda")
    g = torch.Generator(device="cuda").manual_seed(1)
    with torch.no_grad():
        for _, p in m.named_parameters():
            if p.is_cuda and p.dim() >= 2:
                p.copy_(torch.randn(p.shape, generator=g, device="cuda", dtype=torch.float32).mul_(p.shape[-1] ** -0.5))
    return m.to("cuda").eval(), cfg


def weight_bytes(lc):
    """Decoder weights + lm_head read once per decode step (bf16)."""
    H, I, nl, V = lc["hidden_size"], lc["intermediate_size"], lc["num_hidden_layers"], lc["vocab_size"]
    if lc.get("arch") == "gpt2":
        per = 3 * H * H + H * H + 2 * H * I
    else:
        nh, nkv, dh = lc["num_attention_heads"], lc["num_key_value_heads"], lc["head_dim"]
        per = (nh + 2 * nkv) * dh * H + nh * dh * H + 3 * I * H
    return 2.0 * (nl * per + V * H)


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    out = fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1), out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--shapes", default=",".join(SHAPES))
    ap.add_argument("--batches", default="1,16,128")
    args = ap.parse_args()
    import tcavp_b200 as T
    from tcavp_b200 import generate as G
    from tcavp_b200 import ops
    res = dict(info=gpu_info(), copy_peak_tb_s=COPY_PEAK_TBS, prefix=Q_TOKENS + PROMPT, new_tokens=NEW, runs=[], breakdown={})
    print(json.dumps(res["info"]), flush=True)
    kw = dict(max_new_tokens=NEW, temperature=0.9, top_k=40, top_p=0.9, repetition_penalty=1.2, no_repeat_ngram_size=3)
    for shape in args.shapes.split(","):
        m, cfg = build(shape)
        lc = T.resolve_llama(cfg["base_model_name"])
        vd, V = cfg.get("vision_dim", 512), lc["vocab_size"]
        floor_us = weight_bytes(lc) / (COPY_PEAK_TBS * 1e12) * 1e6
        for B in (int(b) for b in args.batches.split(",")):
            gen = torch.Generator(device="cuda").manual_seed(B)
            vision = torch.randn(B, 15, vd, device="cuda", generator=gen)           # 15 frames -> 16 Q-Former tokens
            ids = torch.randint(0, V, (B, PROMPT), device="cuda", generator=gen)
            legs = {"eager": lambda: G.generate_ids(m, vision, ids, **kw), "device": lambda: G.generate_ids(m, vision, ids, seed=1, **kw)}
            for f in legs.values():
                f()
            ms = {k: [] for k in legs}
            for _ in range(2):
                for k, f in legs.items():
                    t, out = timed(f)
                    assert out.shape == (B, PROMPT + NEW), out.shape
                    ms[k].append(t)
            row = dict(shape=shape, B=B, floor_us_per_step=round(floor_us, 1))
            for k, v in ms.items():
                best = min(v)
                row[k] = dict(ms_all=[round(x, 2) for x in v], ms_per_token=round(best / NEW, 4), tokens_per_s=round(B * NEW / (best * 1e-3), 1),
                              floor_share=round(floor_us * 1e-3 / (best / NEW), 4))
            res["runs"].append(row)
            print(json.dumps(row), flush=True)
            # one decode iteration of the device loop, eagerly, under the launch profiler
            loop = next(reversed(m.engine()._decode_loops.values()))
            torch.cuda.synchronize()
            loop.state.zero_()
            with ops.LaunchProfiler() as prof:
                loop.iteration()
            summ = prof.summary()
            res["breakdown"][f"{shape}/B{B}"] = summ["groups"]
        del m
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
