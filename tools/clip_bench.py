"""Cost of FineTuner's gradient clipping on a B200, in one process:

    python tools/clip_bench.py --out clip_bench.json

1. tcavp_clip_prologue (the norm pass: both launches) over flat fp32 buffers of the trainable sizes of the 768-shape (cfg2) and 7B (cfg3)
   fine-tune workloads of bench.TRAIN_WORKLOADS.  Two buffers of each size alternate (462 MB and 1.07 GB per cycle, against 126 MB
   of L2).  Reported as µs per call and TB/s of gradient read, against the 6.53 TB/s copy peak (DESIGN §5).
2. The cfg2-shape fine-tune step (train() mode, CUDA-graph replay, as bench.py --mode train runs it) without clipping and with
   max_grad_norm=1.0, each on its own model built from the same seed, alternated A-B-A-B, device events around each leg; then one
   profiled eager step of each for the per-launch times of the AdamW and norm kernels inside the step.
3. The card name and power limit, read in the same run."""
import argparse
import json
import os
import sys
import warnings

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import TRAIN_WORKLOADS, build_model, scenes_for  # noqa: E402
from fp8_bench import gpu_info  # noqa: E402

COPY_PEAK_TBS = 6.53


def trainable_numel(preset):
    """Length of FineTuner's flat buffer for a preset, from a model built on the meta device (no weights are materialised)."""
    import tcavp_b200 as T
    cfg = dict(T.MODEL_PRESETS[preset])
    big = cfg["base_model_name"] == "llama-7b"
    with torch.device("meta"):
        m = T.MultiModalTrajectoryModel(**cfg, compute_dtype="bf16", llm_param_dtype=torch.bfloat16 if big else None)
    return sum(p.numel() for _, p in m.trainable_named_parameters())


def time_prologue(n, calls):
    from tcavp_b200 import ops
    gen = torch.Generator(device="cuda").manual_seed(n)
    bufs = [torch.randn(n, device="cuda", generator=gen) * 1e-3 for _ in range(2)]
    rec, ws = ops.clip_record("cuda"), torch.empty(ops.CLIP_WORKSPACE_BYTES // 8, dtype=torch.float64, device="cuda")
    for b in bufs * 2:
        ops.clip_prologue(b, rec, ws, grad_scale=1.0, max_norm=1.0)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    rounds = []
    for _ in range(3):
        e0.record()
        for k in range(calls):
            ops.clip_prologue(bufs[k & 1], rec, ws, grad_scale=1.0, max_norm=1.0)
        e1.record()
        e1.synchronize()
        rounds.append(e0.elapsed_time(e1) * 1e3 / calls)
    us = min(rounds)
    tbs = n * 4 / (us * 1e-6) / 1e12
    return dict(n=n, bytes=n * 4, us_per_call=round(us, 2), us_all_rounds=[round(v, 2) for v in rounds], tb_per_s=round(tbs, 3),
                share_of_copy_peak=round(tbs / COPY_PEAK_TBS, 3), norm=float(rec[0]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--calls", type=int, default=50)
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    import tcavp_b200 as T
    from tcavp_b200 import ops
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    T.lib.build()
    warnings.simplefilter("ignore")
    res = dict(**gpu_info(), copy_peak_tb_per_s=COPY_PEAK_TBS)

    # 1. the norm pass alone
    res["prologue"] = {}
    for wl in ("cfg2", "cfg3"):
        preset = TRAIN_WORKLOADS[wl][0]
        res["prologue"][wl] = dict(preset=preset, **time_prologue(trainable_numel(preset), args.calls))
    torch.cuda.empty_cache()

    # 2. the cfg2-shape step without and with clipping
    preset, B, l_text = TRAIN_WORKLOADS["cfg2"]
    fts = {}
    for name, kw in (("off", {}), ("clip", dict(max_grad_norm=1.0))):
        model, cfg = build_model(preset, dev)
        model.train()
        fts[name] = T.FineTuner(model, lr=5e-4, weight_decay=1e-4, **kw)
    assert fts["clip"].flat_p.numel() == res["prologue"]["cfg2"]["n"]
    lc = T.resolve_llama(cfg["base_model_name"])
    s = scenes_for(cfg, B, l_text, 1234, lc["vocab_size"])
    d = {k: s[k].to(dev) for k in ("x", "y", "vision", "polygon", "input_ids", "attention_mask")}
    lens = torch.tensor(s["poly_len"], dtype=torch.int32, device=dev)
    ns = torch.tensor(s["norm_stat"], dtype=torch.float32, device=dev)

    def step(ft):
        return ft.step(d["x"], d["vision"], s["context_str"], d["polygon"], lens, d["y"], ns, d["input_ids"], d["attention_mask"])
    for ft in fts.values():                 # graph capture + warm-up
        for _ in range(3):
            step(ft)
    torch.cuda.synchronize()
    ms = {k: [] for k in fts}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(args.rounds):            # A-B-A-B: clock drift of the warming board hits both alike
        for k, ft in fts.items():
            step(ft)
            e0.record()
            for _ in range(args.steps):
                step(ft)
            e1.record()
            e1.synchronize()
            ms[k].append(e0.elapsed_time(e1) / args.steps)
    res["step_cfg2"] = dict(preset=preset, scenes_per_step=B, l_text=l_text, trainable_params=fts["clip"].flat_p.numel(),
                            method=f"{args.rounds} A-B-A-B rounds x {args.steps} steps per leg (CUDA-graph replay of forward + backward, "
                                   "then the optimiser launches), device events")
    for k in fts:
        res["step_cfg2"][k] = dict(ms_per_step=round(min(ms[k]), 3), ms_all_rounds=[round(v, 3) for v in ms[k]])
    off, on = res["step_cfg2"]["off"]["ms_per_step"], res["step_cfg2"]["clip"]["ms_per_step"]
    res["step_cfg2"]["clip_overhead_ms"] = round(on - off, 3)
    res["step_cfg2"]["clip_overhead_rel"] = round(on / off - 1, 4)
    res["step_cfg2"]["grad_norm_last_step"] = float(fts["clip"].grad_norm)
    # per-launch times inside one eager step of each (outside the timed legs)
    res["step_cfg2"]["in_step_launches"] = {}
    for k, ft in fts.items():
        ft.use_cuda_graph = False
        with ops.LaunchProfiler() as prof:
            step(ft)
        ft.use_cuda_graph = True
        res["step_cfg2"]["in_step_launches"][k] = [dict(kernel=g["kernel"], launches=g["launches"], time_ms=g["time_ms"],
                                                        tb_per_s=round(g["gbs"] / 1e3, 3)) for g in prof.summary()["groups"]
                                                   if g["kernel"] in ("adamw_kernel", "adamw_clipped_kernel", "clip_norm_kernel")]
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
