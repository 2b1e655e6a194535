#!/usr/bin/env python
"""bench.py — headline benchmark of the forward hot path (BASELINE.json: predicted scenes/sec with ADE/FDE).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path, one process per GPU
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle port) on host cores

A "step" is one forward pass (poly encoder + Q-Former + LoRA-Llama + LTSF fusion head + ADE/FDE reduction) over one
batch of synthetic highD-shaped scenes.  N=1 workload = BASELINE.json configs[1]: the GPT-2-small-class Llama
backbone (H=768, 12 layers, LoRA r=8), bf16, 1024 scenes per step.  With N>1 every rank runs its own 1024-scene
shard (scene-parallel, weak scaling) and the step ends with one all-reduce of (sum ADE, sum FDE, n).
Prints ONE JSON line on rank 0.  `--dump-outputs DIR` also writes what the last timed step returned, for an output-for-output
comparison of two builds.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# stdout carries exactly ONE JSON line: everything else a library writes to fd 1 (e.g. NCCL's version banner) goes to stderr.
_JSON_OUT = None


def _claim_stdout():
    """Called from the command-line entry only (importing this module has no side effects)."""
    global _JSON_OUT
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(obj):
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(obj) + "\n")
    out.flush()


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(path, arrays, scenes):
    """Writes the tensors the timed path returned in its last step as <path>/<name>.npy (float64 stays float64, every other dtype
    becomes float32), so that two builds can be compared output for output on the same seeded inputs.  Above 64 MB in all, the
    per-scene arrays (leading dimension `scenes`) keep one seeded sample of scenes, the same rows in each; the others stay whole."""
    import numpy as np
    arrs = {k: v.detach().to("cpu", torch.float64 if v.dtype == torch.float64 else torch.float32) for k, v in arrays.items()}
    total = sum(a.numel() * a.element_size() for a in arrs.values())
    budget = DUMP_LIMIT_BYTES - 4096 * len(arrs)        # room for the .npy headers
    per_scene = [k for k, a in arrs.items() if a.dim() and a.shape[0] == scenes]
    if total > budget and per_scene:
        fixed = total - sum(arrs[k].numel() * arrs[k].element_size() for k in per_scene)
        n = max(1, scenes * (budget - fixed) // (total - fixed))
        rows = torch.randperm(scenes, generator=torch.Generator().manual_seed(0))[:n].sort().values
        for k in per_scene:
            arrs[k] = arrs[k][rows]
    os.makedirs(path, exist_ok=True)
    for k, a in arrs.items():
        np.save(os.path.join(path, k + ".npy"), a.numpy())


METRIC = "predicted scenes/sec (forward + ADE/FDE)"
UNIT = "scenes/s"
WORKLOADS = {
    # name: (model preset, scenes per GPU per step, L_text)
    "cfg2": ("cfg1", 1024, 128),
    # the same workload on the GPT-2 architecture (gpt2-small: 768 / 12 layers / 12 heads / 3072, vocabulary 50257; not a default secondary)
    "cfg2-gpt2": ("cfg1-gpt2", 1024, 128),
    "cfg3": ("cfg3", 256, 128),
    # BASELINE.json configs[4]: encoder + fusion with a frozen backbone (final_hidden supplied, bf16), T_out 50, 4096 scenes
    "cfg5": ("cfg5", 4096, 128),
}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, src="fallback")


class ClockSampler:
    """SM clock / power / throttle reasons DURING the timed region.  NVML is read in-process every 20 ms (nvidia-smi takes
    ~0.3 s to start, longer than a short timed region); the nvidia-smi loop of the profiling recipe is the fallback."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        import threading
        self.sm, self.mx, self.pw, self.reasons = [], [], [], set()
        self.p = self.f = self.t = None
        self._stop = False
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and all(t.strip().isdigit() for t in vis.split(",")) else index
            h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            mx = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            bits = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}

            def loop():
                while not self._stop:
                    try:
                        self.sm.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                        self.mx.append(mx)
                        self.pw.append(pynvml.nvmlDeviceGetPowerUsage(h) / 1e3)
                        r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                        for n, b in bits.items():
                            if r & b:
                                self.reasons.add(n)
                    except Exception:
                        pass
                    time.sleep(0.02)
            self.t = threading.Thread(target=loop, daemon=True)
            self.t.start()
        except Exception:
            self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
            try:
                self.p = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                          stdout=self.f, stderr=subprocess.DEVNULL)
            except OSError:
                self.p = None

    def stop(self):
        if self.t is not None:
            self._stop = True
            self.t.join(timeout=2)
            sm, mx, reasons, src = self.sm, self.mx, self.reasons, "nvml, 20 ms period"
        else:
            if self.p is None:
                return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
            self.p.terminate()
            try:
                self.p.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.p.kill()
            self.f.flush()
            self.f.seek(0)
            sm, mx, reasons, src = [], [], set(), "nvidia-smi -lms 100"
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            for line in self.f.read().splitlines():
                c = [t.strip() for t in line.split(",")]
                if len(c) < 7:
                    continue
                try:
                    sm.append(float(c[0]))
                    mx.append(float(c[1]))
                except ValueError:
                    continue
                for n, v in zip(names, c[3:7]):
                    if v == "Active":
                        reasons.add(n)
            os.unlink(self.f.name)
        load = sm       # the sampler only lives inside the timed region: every sample is a sample under load
        out = {"sm_mhz": statistics.median(load) if load else None, "sm_max_mhz": max(mx) if mx else None,
               "reasons": sorted(reasons), "samples": len(sm), "source": src}
        if self.pw:
            out["power_w_max"] = round(max(self.pw), 1)
        return out


def build_model(preset, device, compute_dtype="bf16", over=None):
    import tcavp_b200 as T
    cfg = dict(T.MODEL_PRESETS[preset])
    cfg.update(over or {})
    big = cfg["base_model_name"] == "llama-7b"
    m = T.MultiModalTrajectoryModel(**cfg, compute_dtype=compute_dtype, llm_param_dtype=torch.bfloat16 if big else None,
                                    llm_device=device if big else None)
    if big:   # 7B: random-init on the device (a host-side seeded fill of 6.7 G values would take minutes)
        g = torch.Generator(device=device).manual_seed(1)
        with torch.no_grad():
            for n, p in m.named_parameters():
                if p.is_cuda and p.dim() >= 2:
                    p.copy_(torch.randn(p.shape, generator=g, device=device, dtype=torch.float32).mul_(p.shape[-1] ** -0.5))
        sd = {k: v for k, v in m.state_dict().items() if not v.is_cuda}
        T.deterministic_fill_(sd, 1)
    else:
        T.deterministic_fill_(m.state_dict(), 1)
    return m.to(device).eval(), cfg


def scenes_for(cfg, B, l_text, seed, vocab):
    import tcavp_b200 as T
    return T.make_scenes(B, cfg["seq_len"], cfg["out_len"], l_text=l_text, vocab=vocab, seed=seed, ragged_text=False)


def gemm_flops_per_scene(cfg, lc, L):
    """Algorithmic FLOPs of the dense contractions per scene (SURVEY.md §8d), LoRA included, lm_head excluded."""
    H, I, nl = lc["hidden_size"], lc["intermediate_size"], lc["num_hidden_layers"]
    nh = lc["num_attention_heads"]
    nkv, dh = lc.get("num_key_value_heads", nh), lc.get("head_dim", H // nh)
    if lc.get("arch") == "gpt2":         # c_attn (3H), c_proj, c_fc + mlp.c_proj (two H x I products, no gate), LoRA on c_attn
        r = cfg.get("lora_r", 8) if cfg.get("use_lora", True) else 0
        return L * nl * (2 * H * 3 * H + 2 * H * H + 2 * 2 * H * I + 2 * r * (H + 3 * H))
    per_tok = nl * (2 * H * (nh + 2 * nkv) * dh + 2 * nh * dh * H + 3 * 2 * H * I)
    r = cfg.get("lora_r", 8) if cfg.get("use_lora", True) else 0
    lora = nl * 2 * r * ((H + nh * dh) + (H + nkv * dh))
    return L * (per_tok + lora)


class _Ctx:
    """Process-wide state shared by the workloads of one bench run."""

    def __init__(self, args):
        import torch.distributed as dist
        self.dist = dist
        self.rank, self.world, self.local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        import tcavp_b200.lib as L_
        L_.build()
        L_.load()
        self.args = args

    def barrier(self):
        torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()

    def max_over_ranks(self, v):
        t = torch.tensor([v], dtype=torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def _roofline(prof, pk, ms_step, steps_profiled, extra=None, top=10):
    """Roofline block from a LaunchProfiler pass (CUDA events around every libtcavp launch, on the launching stream).  The pass is a
    SEPARATE repetition of the timed steps, after the timed region: the timed region itself carries no per-launch events."""
    summ = prof.summary()
    dom = summ["dominant"]
    groups = summ["groups"]
    r = {"bound": "tensor", "kernel": dom["kernel"], "achieved": round(dom["tflops"], 1), "peak": pk["tf_sustained"], "unit": "TFLOP/s",
         "frac": round(dom["tflops"] / pk["tf_sustained"], 4), "traffic": None,
         "peak_source": f"MEASURED_PEAKS.json bf16_tflops_sustained ({pk['src']})",
         "launches_timed": dom["launches"], "avg_launch_ms": round(dom["avg_ms"], 4),
         "share_of_step": round(dom["time_ms"] / steps_profiled / ms_step, 4),
         "measured": f"separate profiling pass of {steps_profiled} step(s) right after the timed region (same process, same clocks)",
         "by_group": groups[:top]}
    tensor = [g for g in groups if g["tflops"] > 0.0]
    t_t = sum(g["time_ms"] for g in tensor)
    if t_t > 0:
        r["all_tensor_kernels"] = {"achieved": round(sum(g["tflops"] * g["time_ms"] for g in tensor) / t_t, 1),
                                   "share_of_step": round(t_t / steps_profiled / ms_step, 4)}
    bw = [g for g in groups if g["tflops"] == 0.0 and g["gbs"] > 0.0]
    if bw:
        t_bw = sum(g["time_ms"] for g in bw)
        gb = sum(g["gbs"] * g["time_ms"] for g in bw) / t_bw
        r["hbm_kernels"] = {"bound": "hbm", "achieved": round(gb, 1), "peak": pk["hbm"], "unit": "GB/s", "frac": round(gb / pk["hbm"], 4),
                            "share_of_step": round(t_bw / steps_profiled / ms_step, 4),
                            "kernels": [{"kernel": g["kernel"], "gbs": g["gbs"], "share": g["share"]} for g in bw[:8]]}
    if extra:
        r.update(extra)
    return r, dom


def measure_infer(ctx, workload, steps, warmup, e2e=True, scenes=0, merge_lora=False, dump=None):
    """One inference workload: device-resident `value` leg (clean timed region), separate profiling pass, optional host-buffer e2e leg.
    `dump`: directory for what the last timed step returned (rank 0)."""
    import tcavp_b200 as T
    from tcavp_b200 import ops
    dist, rank, world, dev = ctx.dist, ctx.rank, ctx.world, ctx.dev
    preset, B, l_text = WORKLOADS[workload]
    if scenes:
        B = scenes
    model, cfg = build_model(preset, dev)
    if merge_lora:
        model.merge_lora_for_inference(True)
    lc = T.resolve_llama(cfg["base_model_name"])
    s = scenes_for(cfg, B, l_text, 1234 + rank, lc["vocab_size"])
    eng = model.engine()
    d = {k: s[k].to(dev) for k in ("x", "y", "vision", "polygon", "input_ids", "attention_mask")}
    d["lens"] = torch.tensor(s["poly_len"], dtype=torch.int32, device=dev)
    d["ns"] = torch.tensor(s["norm_stat"], dtype=torch.float32, device=dev)
    red = torch.zeros(3, dtype=torch.float32, device=dev)
    b_dev = torch.tensor(float(B), dtype=torch.float32, device=dev)
    max_poly = int(max(s["poly_len"]))     # dataset metadata (lane sizes are 14 / 22 / 32 / 33 points, reference graph.py): host-known
    frozen = workload == "cfg5"            # backbone output precomputed (ablation_study_without_lora.py path): encoder + fusion only
    fh_dev = fh_host = None
    if frozen:
        g = torch.Generator().manual_seed(77 + rank)
        fh_host = torch.randn(B, 16 + l_text, lc["hidden_size"], generator=g).to(torch.bfloat16)
        fh_dev = fh_host.to(dev)

    def step():
        o = eng.forward(d["x"], d["vision"], d["polygon"], d["lens"], d["input_ids"], d["attention_mask"], y=d["y"], norm_stat=d["ns"],
                        final_hidden=fh_dev, max_poly_len=max_poly, cuda_graph=graph)
        if world > 1:        # per-rank running sums; ONE all-reduce per evaluation pass (SURVEY §8e), inside the timed region
            red.add_(torch.stack((o["sum_ade"], o["sum_fde"], b_dev)))
        return o

    graph = bool(ctx.args.cuda_graph)          # one cudaGraphLaunch per step instead of ~200 kernel launches (fixed batch shape)
    for _ in range(max(warmup, 3)):
        o = step()
    if world > 1:
        dist.all_reduce(red)     # warm the communicator
        red.zero_()
    ctx.barrier()
    sampler = ClockSampler(ctx.local) if rank == 0 else None
    launches0 = ops.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        o = step()
    if world > 1:
        dist.all_reduce(red)         # (sum ADE, sum FDE, scenes) over all ranks and steps
    e1.record()
    ctx.barrier()
    launches = ops.launch_count() - launches0
    clocks = sampler.stop() if sampler else None
    ms = ctx.max_over_ranks(e0.elapsed_time(e1))
    if dump and rank == 0:          # before the passes below: with a CUDA graph, `o` holds the graph's static output buffers
        dump_outputs(dump, {k: v for k, v in o.items() if torch.is_tensor(v)}, B)
    value = world * B * steps / (ms / 1e3)
    ade, fde = float(o["sum_ade"]) / B, float(o["sum_fde"]) / B
    # ---- profiling pass (untimed): the same steps again with CUDA events around every launch ---------------
    n_prof = min(steps, 3)
    prof = ops.LaunchProfiler()
    graph = False                              # the profiling pass needs the individual launches
    lp0 = ops.launch_count()
    with prof:
        for _ in range(n_prof):
            step()
    graph = bool(ctx.args.cuda_graph)
    if graph:                                  # replayed launches are not seen by the library's counter: one eager step's count x steps
        launches = (ops.launch_count() - lp0) // n_prof * steps
    torch.cuda.synchronize()
    red.zero_()

    e2e_block = None
    if e2e:
        # ---- end-to-end leg: host (pinned) buffers through the public API, H2D + D2H inside the timed region ---
        h = {k: s[k].pin_memory() for k in ("x", "y", "vision", "polygon", "input_ids", "attention_mask")}
        h["lens"] = torch.tensor(s["poly_len"], dtype=torch.int32).pin_memory()
        h["ns"] = torch.tensor(s["norm_stat"], dtype=torch.float32).pin_memory()
        if frozen:
            h["fh"] = fh_host.pin_memory()
            for k in ("vision", "input_ids", "attention_mask"):     # not consumed on this path
                h.pop(k)
        h2d = sum(v.numel() * v.element_size() for v in h.values())
        # Two-deep software pipeline, as a serving loop would run it: step i+1 is enqueued (its bulk H2D travels on the engine's copy
        # stream under step i's kernels) before the host reads step i's result.  Every step still copies its own inputs from pinned host
        # memory and the host still reads every step's decoded trajectories + metrics, all inside the timed region.
        dec_host = [torch.empty(B, 2, cfg["out_len"], dtype=torch.float32).pin_memory() for _ in range(2)]
        met_host = [torch.empty(8, dtype=torch.float32).pin_memory() for _ in range(2)]
        done = [torch.cuda.Event() for _ in range(2)]
        d2h = dec_host[0].numel() * 4 + met_host[0].numel() * 4

        def e2e_enqueue(slot):
            if frozen:
                r = model.predict_with_metrics(h["x"], None, h["polygon"], h["lens"], h["y"], h["ns"], None, None, final_hidden=h["fh"],
                                               max_poly_len=max_poly, cuda_graph=graph)
            else:
                r = model.predict_with_metrics(h["x"], h["vision"], h["polygon"], h["lens"], h["y"], h["ns"], h["input_ids"], h["attention_mask"],
                                               max_poly_len=max_poly, cuda_graph=graph)
            dec_host[slot].copy_(r["decoded"], non_blocking=True)
            met_host[slot].copy_(r["metrics"], non_blocking=True)
            done[slot].record()

        def e2e_read(slot):
            done[slot].synchronize()                            # the caller reads the result here
            return float(met_host[slot][2]), float(met_host[slot][3]), float(dec_host[slot][-1, -1, -1])

        def e2e_run(n):
            for i in range(n):
                e2e_enqueue(i & 1)
                if i > 0:
                    e2e_read((i - 1) & 1)
            return e2e_read((n - 1) & 1)

        e2e_run(2)
        # host wall clock over K steps is exposed to a single scheduling hiccup of the host thread (one 40 ms stall = 10 % of a 10-step
        # region): the leg is repeated three times, every repeat is K full steps, and the MEDIAN repeat is reported (all three listed)
        e2e_repeats = []
        for _ in range(3):
            ctx.barrier()
            t0 = time.perf_counter()
            e2e_last = e2e_run(steps)
            torch.cuda.synchronize()
            e2e_s = time.perf_counter() - t0
            if abs(e2e_last[0] / B - ade) > 1e-3 * max(ade, 1.0):
                raise RuntimeError(f"end-to-end leg disagrees with the device-resident leg: ADE {e2e_last[0] / B} vs {ade}")
            e2e_repeats.append(world * B * steps / ctx.max_over_ranks(e2e_s))
        e2e_value = statistics.median(e2e_repeats)
        e2e_block = {"value": round(e2e_value, 2), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                     "api": "MultiModalTrajectoryModel.predict_with_metrics (pinned host tensors in, decoded + metrics out)",
                     "pipeline": "2-deep: step i+1 is enqueued before the host reads step i (bulk H2D on a copy stream)",
                     "timing": f"host wall clock over {steps} steps, max over ranks; median of 3 repeats",
                     "repeat_values": [round(v, 2) for v in e2e_repeats]}

    pk = peaks()
    Lseq = 16 + l_text
    roof, dom = _roofline(prof, pk, ms / steps, n_prof, {"algorithmic_flops_per_scene": gemm_flops_per_scene(cfg, lc, Lseq)})
    # DRAM bytes per launch of the dominant kernel, from the committed ncu capture of this same command (tools/profile.sh)
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tpath):
        t = json.load(open(tpath)).get(workload)
        if t and dom["kernel"].split("<")[0] in t.get("kernel", ""):
            roof["traffic"] = t["dram_bytes_per_launch"]
            roof["traffic_source"] = f"profiles/ncu_traffic.json ({t['source']}: mean of {t['launches']} launches of one step, dram__bytes_read+write)"
            roof["algorithmic_bytes_per_launch"] = round(dom["bytes"] / max(dom["launches"], 1))
    out = {
        "metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": max(warmup, 3),
        "ms_per_step": round(ms / steps, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": {"workload": (f"{workload}: encoder + lane-polygon encoder + cross-attention fusion + head only; frozen {cfg['base_model_name']} "
                                f"backbone output (B, {Lseq}, H) supplied in bf16, " if frozen else
                                f"{workload}: {cfg['base_model_name']} backbone, LoRA r={cfg.get('lora_r', 8)}, bf16 inference, ") +
                               f"{B} scenes/GPU/step, T_in {cfg['seq_len']} -> T_out {cfg['out_len']}, L = 16 image + {l_text} text tokens",
                   "scenes_per_gpu": B, "seq_len": Lseq, "parallelism": f"scene-parallel x{world}",
                   "launch": "one CUDA-graph replay per step (captured once per batch shape)" if graph else "eager kernel launches",
                   "timing": "value: CUDA events around the K steps, nothing else inside" + (" but one metric all-reduce after the last step" if world > 1 else "") +
                             "; roofline: separate profiling pass; e2e: host wall clock",
                   "l2": "per-step working set (>= 1 GB of activations) is far larger than the 126 MB L2; no explicit flush",
                   "lora": "merged into the base weights at pack time" if merge_lora else "unmerged (rank-r side path fused into the QKV GEMM)",
                   "weights": "seeded random init (no checkpoints offline)", "ade_px": round(ade, 3), "fde_px": round(fde, 3),
                   "gemm_route": ops._ROUTE["tuned"]},
        "gpu_launches": launches, "clocks": clocks, "roofline": roof,
    }
    if e2e_block:
        out["e2e"] = e2e_block
    keep = dict(model=model, cfg=cfg, lc=lc, l_text=l_text, frozen=frozen)
    return out, keep


TRAIN_WORKLOADS = {
    # name: (model preset, scenes per GPU per step, L_text)  — BASELINE.json configs[3]: LoRA fine-tune step, data parallel
    "cfg2": ("cfg1", 512, 128),
    "cfg3": ("cfg3", 128, 128),    # 103 GiB of the 180 GB at 128 scenes / GPU / step
    "cfg2-gpt2": ("cfg1-gpt2", 512, 128),    # the cfg2 shape on the GPT-2 architecture (HF GPT2LMHeadModel, c_attn LoRA)
}


def measure_train(ctx, workload, steps, warmup, scenes=0, dropout=None, dump=None):
    """One fine-tune step = forward + hand-written backward + ONE all-reduce of the trainable gradients + fused AdamW
    (tcavp_b200.FineTuner).  Metric: LoRA fine-tune tokens/sec (tokens = scenes x (16 image + L_text)).
    `dump`: directory for the (loss, decoded) of the last timed step (rank 0)."""
    import warnings

    import tcavp_b200 as T
    from tcavp_b200 import ops
    dist, rank, world, dev = ctx.dist, ctx.rank, ctx.world, ctx.dev
    preset, B, l_text = TRAIN_WORKLOADS[workload]
    if scenes:
        B = scenes
    over = {} if dropout is None else dict(lora_dropout=dropout, ltsf_dropout=dropout)
    model, cfg = build_model(preset, dev, over=over)
    model.train()        # the reference's fine-tune step runs in train() mode: lora / ltsf / nn.Transformer dropout 0.1 (SURVEY §8d(4))
    if dropout is not None:
        model.set_dropout(dropout)
    lc = T.resolve_llama(cfg["base_model_name"])
    s = scenes_for(cfg, B, l_text, 1234 + rank, lc["vocab_size"])
    d = {k: s[k].to(dev) for k in ("x", "y", "vision", "polygon", "input_ids", "attention_mask")}
    lens = torch.tensor(s["poly_len"], dtype=torch.int32, device=dev)
    ns = torch.tensor(s["norm_stat"], dtype=torch.float32, device=dev)
    warnings.simplefilter("ignore")
    ft = T.FineTuner(model, lr=5e-4, weight_decay=1e-4)

    def step():
        return ft.step(d["x"], d["vision"], s["context_str"], d["polygon"], lens, d["y"], ns, d["input_ids"], d["attention_mask"])

    losses = []
    for _ in range(max(warmup, 3)):
        losses.append(float(step()[0]))
    ctx.barrier()
    sampler = ClockSampler(ctx.local) if rank == 0 else None
    launches0 = ops.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss, decoded = step()
    e1.record()
    ctx.barrier()
    # forward + backward are replayed from a CUDA graph: the library's launch counter only sees the capture
    launches = (ops.launch_count() - launches0) + (ft.launches_per_step * steps if ft.use_cuda_graph else 0)
    clocks = sampler.stop() if sampler else None
    ms = ctx.max_over_ranks(e0.elapsed_time(e1))
    if dump and rank == 0:
        dump_outputs(dump, {"loss": loss, "decoded": decoded}, B)
    # the collective alone (same buffer, same communicator), outside the timed region
    ar_ms = ar_exposed_ms = None
    ar_ab = {"overlapped": [], "serial": []}
    if world > 1:
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ft.all_reduce_only()
        torch.cuda.synchronize()
        a0.record()
        for _ in range(5):
            ft.all_reduce_only()
        a1.record()
        torch.cuda.synchronize()
        ar_ms = ctx.max_over_ranks(a0.elapsed_time(a1) / 5)
        # what the exchange costs INSIDE the step: the same steps with the collective left out (measurement only), max over ranks
        n_x = max(2, min(steps, 5))
        ft.step(d["x"], d["vision"], s["context_str"], d["polygon"], lens, d["y"], ns, d["input_ids"], d["attention_mask"], skip_allreduce=True)
        ctx.barrier()
        a0.record()
        for _ in range(n_x):
            ft.step(d["x"], d["vision"], s["context_str"], d["polygon"], lens, d["y"], ns, d["input_ids"], d["attention_mask"], skip_allreduce=True)
        a1.record()
        torch.cuda.synchronize()
        ar_exposed_ms = ms / steps - ctx.max_over_ranks(a0.elapsed_time(a1)) / n_x
        # overlapped vs serial exchange, A-B-A-B in this process (same graphs, same GPUs, same clocks): ms per step, max over ranks
        keep_overlap = ft.overlap
        for rnd in range(2):
            for mode in (True, False):
                ft.overlap = mode
                ft.step(d["x"], d["vision"], s["context_str"], d["polygon"], lens, d["y"], ns, d["input_ids"], d["attention_mask"])
                ctx.barrier()
                a0.record()
                for _ in range(n_x):
                    ft.step(d["x"], d["vision"], s["context_str"], d["polygon"], lens, d["y"], ns, d["input_ids"], d["attention_mask"])
                a1.record()
                torch.cuda.synchronize()
                ar_ab["overlapped" if mode else "serial"].append(round(ctx.max_over_ranks(a0.elapsed_time(a1)) / n_x, 3))
        ft.overlap = keep_overlap
    # per-kernel breakdown: ONE extra eager (un-captured) step outside the timed region, CUDA events around every launch
    prof = ops.LaunchProfiler()
    ft.use_cuda_graph = False
    with prof:
        step()
    ft.use_cuda_graph = True
    torch.cuda.synchronize()
    Lseq = 16 + l_text
    value = world * B * Lseq * steps / (ms / 1e3)
    losses.append(float(loss))
    peak_gb = torch.cuda.max_memory_allocated() / 2 ** 30
    pk = peaks()
    roof, _ = _roofline(prof, pk, ms / steps, 1, {"breakdown": "one eager step after the timed region (the timed steps replay a CUDA graph)"})
    probs = model.train_engine()._dropout_probs()
    p_drop = {"lora": probs.get(("llm", "lora_q"), probs.get(("llm", "lora_c"), 0.0)), "gpt2_embd_attn_resid": probs.get(("llm", "attn")), "ltsf": probs.get(("ltsf", "ffn"), 0.0), "transformer_layers": probs.get(("qenc", "ffn"), 0.0),
              "applied": bool(ft.dropout_active), "masks": "counter-based (seed, step, site, element), regenerated in the backward pass"}
    out = {
        "metric": "LoRA fine-tune tokens/sec (forward + backward + grad all-reduce + AdamW)", "value": round(value, 1), "unit": "tokens/s",
        "n_gpus": world, "steps": steps, "warmup": max(warmup, 3), "ms_per_step": round(ms / steps, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"train-{workload}: {cfg['base_model_name']} backbone, LoRA r={cfg.get('lora_r', 8)}, bf16 compute / fp32 masters, "
                               f"{B} scenes/GPU/step, L = 16 image + {l_text} text tokens",
                   "dropout": p_drop,
                   "scenes_per_gpu": B, "seq_len": Lseq, "parallelism": f"data-parallel x{world}",
                   "allreduce_payload_bytes": ft.payload_bytes, "allreduce_alone_ms": None if ar_ms is None else round(ar_ms, 3),
                   "allreduce_exposed_ms": None if ar_exposed_ms is None else round(ar_exposed_ms, 3),
                   "allreduce_overlap_ab_ms_per_step": ar_ab if world > 1 else None,
                   "allreduce": ("two NCCL all-reduces per step over one flat fp32 buffer: the slice outside mllm.* (%d bytes, final before the "
                                 "decoder-stack backward) runs under the second CUDA graph, the mllm.* slice after it; exposed = step - step without the collective"
                                 % ((ft.flat_p.numel() - ft.n_late) * 4)) if ft.overlap else "one NCCL all-reduce of the flat trainable-gradient buffer per step",
                   "trainable_params": ft.flat_p.numel(), "gemm_route": ops._ROUTE["tuned"],
                   "loss_first_last": [round(losses[0], 3), round(losses[-1], 3)], "peak_mem_gib": round(peak_gb, 2)},
        "gpu_launches": launches, "clocks": clocks, "roofline": roof}
    return out


def measure_stage1(ctx, steps, warmup, scenes=0, dump=None):
    """Stage-1 (CausalLM) training step of the reference's scripts/check_generation.py loop at the 768-class shape: model.stage1_forward(...)
    -> outputs.loss.backward() -> AdamW on the mllm.* tensors.  Metric: tokens/sec through the model (scenes x (16 image + L_text));
    the labelled half of every sequence (64 answer tokens per scene) goes through lm_head (vocabulary 32000) in row chunks."""
    import warnings

    import tcavp_b200 as T
    from tcavp_b200 import ops
    rank, world, dev = ctx.rank, ctx.world, ctx.dev
    preset, B, l_text = TRAIN_WORKLOADS["cfg2"]
    if scenes:
        B = scenes
    model, cfg = build_model(preset, dev)
    model.eval()          # the stage-1 script trains in train() mode; dropout is measured by --mode train — this line isolates the objective
    lc = T.resolve_llama(cfg["base_model_name"])
    s = scenes_for(cfg, B, l_text, 4321 + rank, lc["vocab_size"])
    ids, am, vis = s["input_ids"].to(dev), s["attention_mask"].to(dev), s["vision"].to(dev)
    labels = ids.clone()
    labels[:, :l_text // 2] = -100
    labels[am == 0] = -100
    n_lab = int((labels != -100).sum())
    warnings.simplefilter("ignore")
    params = [p for n, p in model.named_parameters() if p.requires_grad and n.startswith("mllm.")]
    opt = torch.optim.AdamW(params, lr=1e-4, fused=True)

    def step():
        opt.zero_grad(set_to_none=True)
        out = model.stage1_forward(vis, ids, am, labels)
        out.loss.backward()
        if world > 1:
            for p in params:
                if p.grad is not None:
                    ctx.dist.all_reduce(p.grad)
        opt.step()
        return out.loss.detach()
    losses = [float(step()) for _ in range(max(warmup, 3))]
    ctx.barrier()
    sampler = ClockSampler(ctx.local) if rank == 0 else None
    n0 = ops.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss = step()
    e1.record()
    ctx.barrier()
    launches = ops.launch_count() - n0
    clocks = sampler.stop() if sampler else None
    ms = ctx.max_over_ranks(e0.elapsed_time(e1))
    if dump and rank == 0:
        dump_outputs(dump, {"loss": loss}, B)
    losses.append(float(loss))
    prof = ops.LaunchProfiler()
    with prof:
        step()
    torch.cuda.synchronize()
    Lseq = 16 + l_text
    roof, _ = _roofline(prof, peaks(), ms / steps, 1, {"breakdown": "one extra step after the timed region, CUDA events around every launch"})
    return {"metric": "stage-1 (CausalLM) training tokens/sec (forward + loss + backward + AdamW)", "value": round(world * B * Lseq * steps / (ms / 1e3), 1),
            "unit": "tokens/s", "n_gpus": world, "steps": steps, "warmup": max(warmup, 3), "ms_per_step": round(ms / steps, 3), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"stage1-cfg2: {cfg['base_model_name']} backbone, LoRA r={cfg.get('lora_r', 8)}, bf16 compute / fp32 masters, {B} scenes/GPU/step, "
                                   f"L = 16 image + {l_text} text tokens, {n_lab} labelled tokens/GPU/step through lm_head (vocabulary {lc['vocab_size']})",
                       "scenes_per_gpu": B, "seq_len": Lseq, "labelled_tokens_per_gpu": n_lab, "loss_first_last": [round(losses[0], 3), round(losses[-1], 3)],
                       "peak_mem_gib": round(torch.cuda.max_memory_allocated() / 2 ** 30, 2), "gemm_route": ops._ROUTE["tuned"]},
            "gpu_launches": launches, "clocks": clocks, "roofline": roof}


def _brief(d):
    """Secondary workloads ride inside the headline line: keep the judged fields, trim the per-kernel table."""
    r = dict(d["roofline"])
    r["by_group"] = r.get("by_group", [])[:6]
    keep = {k: d[k] for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "dtype", "gpu_launches", "clocks") if k in d}
    keep["config"] = d["config"]
    keep["roofline"] = r
    if "e2e" in d:
        keep["e2e"] = d["e2e"]
    return keep


def _free():
    import gc
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()


def run_ours(args):
    ctx = _Ctx(args)
    out, keep = measure_infer(ctx, args.workload, args.steps, args.warmup, e2e=True, scenes=args.scenes, merge_lora=args.merge_lora,
                              dump=args.dump_outputs)
    if ctx.world == 1 and ctx.rank == 0 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline(keep["model"], keep["cfg"], keep["lc"], keep["l_text"], sample=args.cpu_sample, repeats=2,
                                           frozen=keep["frozen"])
    del keep
    _free()
    # BASELINE.json names more configurations than the headline: measure them in the same process (same box, same clocks) so they are
    # part of the driver-run record — at N GPUs too (7B scene-sharded inference, 7B data-parallel fine-tune step with the gradient
    # all-reduce).  Only with the default headline workload; --no-secondary skips them.
    if args.workload == "cfg2" and not args.no_secondary and not args.scenes and not args.merge_lora:
        sec = {}
        k2 = max(args.secondary_steps, 5)
        extra = [("cfg2_gpt2", lambda: measure_infer(ctx, "cfg2-gpt2", k2, 3, e2e=True)[0])]      # the headline workload on the GPT-2 architecture
        if ctx.world == 1:
            extra.append(("stage1_cfg2", lambda: measure_stage1(ctx, k2, 3)))                    # CausalLM training step (single-GPU line)
            extra.append(("train_cfg2_gpt2", lambda: measure_train(ctx, "cfg2-gpt2", k2, 3)))    # fine-tune step on the GPT-2 architecture
        for name, fn in [("cfg3", lambda: measure_infer(ctx, "cfg3", k2, 3, e2e=True)[0]),
                         ("cfg5", lambda: measure_infer(ctx, "cfg5", max(k2, 10), 3, e2e=True)[0]),
                         ("train_cfg2", lambda: measure_train(ctx, "cfg2", k2, 3)),
                         ("train_cfg4", lambda: measure_train(ctx, "cfg3", k2, 3))] + extra:
            try:
                sec[name] = _brief(fn())
            except Exception as e:     # a secondary workload must never take the headline line down with it
                sec[name] = {"error": f"{type(e).__name__}: {str(e)[:300]}"}
            _free()
        out["secondary"] = sec
    if ctx.rank == 0:
        emit(out)
    ctx.close()


def run_train(args):
    """--mode train: the LoRA fine-tune step as the only workload of the run."""
    ctx = _Ctx(args)
    out = measure_train(ctx, args.workload, args.steps, args.warmup, scenes=args.scenes, dropout=args.dropout, dump=args.dump_outputs)
    if ctx.rank == 0:
        emit(out)
    ctx.close()


def _cpu_pair(step, repeats):
    """(median seconds without lm_head, median seconds as shipped = with the lm_head logits the reference computes and discards)."""
    def t(with_head):
        t0 = time.perf_counter()
        step(with_head)
        return time.perf_counter() - t0
    t(False)
    plain = statistics.median([t(False) for _ in range(repeats)])
    shipped = statistics.median([t(True) for _ in range(max(1, repeats - 1))])
    return plain, shipped


def cpu_baseline(model, cfg, lc, l_text, sample, repeats, frozen=False):
    """The reference's CPU path, restated (oracle/restated.py, validated against the reference in tests/), timed on the
    host cores on a bounded sample of the same workload (BASELINE.md §5: two figures, without and with the dead lm_head GEMM)."""
    from oracle import restated
    sd = {k: v.detach().float().cpu() for k, v in model.state_dict().items()}
    s = scenes_for(cfg, sample, l_text, 99, lc["vocab_size"])
    torch.set_num_threads(os.cpu_count())
    fh = torch.randn(sample, 16 + l_text, lc["hidden_size"]) if frozen else None

    def one(with_head):
        restated.forward(sd, cfg, lc, s["x"], s["vision"], s["polygon"], s["poly_len"], s["input_ids"], s["attention_mask"], s["y"], s["norm_stat"],
                         final_hidden=fh, with_lm_head=with_head and not frozen)
    plain, shipped = _cpu_pair(one, repeats)
    out = {"value": round(sample / plain, 2), "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
           "sample": f"{sample} scenes of the same workload per forward (BASELINE.json configs[0] size), fp32, median of {repeats} after 1 warm-up; "
                     "lm_head (dead compute in the reference) excluded"}
    if not frozen:
        out["as_shipped"] = {"value": round(sample / shipped, 2), "unit": UNIT,
                             "note": "with the vocabulary logits the shipped reference always computes and discards (HF lm_head, train.py:547-554)"}
    return out


def run_reference(args):
    """--impl reference: the reference's own algorithm on the host cores (oracle port; the Python reference itself cannot
    travel to the GPU box).  Rank 0 only.  `value` excludes the dead lm_head GEMM (the conservative figure: the CUDA arm does not
    compute it either); the as-shipped figure rides in cpu_baseline.as_shipped."""
    if int(os.environ.get("RANK", 0)) != 0:
        return
    import tcavp_b200 as T
    from oracle import restated
    preset, B, l_text = WORKLOADS[args.workload]
    cfg = dict(T.MODEL_PRESETS[preset])
    lc = T.resolve_llama(cfg["base_model_name"])
    sample = args.cpu_sample
    m = T.MultiModalTrajectoryModel(**cfg)
    sd = m.state_dict()
    T.deterministic_fill_(sd, 1)
    sd = {k: v.float() for k, v in sd.items()}
    s = scenes_for(cfg, sample, l_text, 1234, lc["vocab_size"])
    torch.set_num_threads(os.cpu_count())
    frozen = args.workload == "cfg5"
    fh = torch.randn(sample, 16 + l_text, lc["hidden_size"]) if frozen else None   # frozen-backbone path

    def step(with_head=False):
        return restated.forward(sd, cfg, lc, s["x"], s["vision"], s["polygon"], s["poly_len"], s["input_ids"], s["attention_mask"], s["y"], s["norm_stat"],
                                final_hidden=fh, with_lm_head=with_head and not frozen)
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    v = round(sample * args.steps / dt, 2)
    desc = f"{sample} scenes per step (BASELINE.json configs[0] size; bounded sample of the {B}-scene workload), fp32, all host threads, lm_head excluded"
    cb = {"value": v, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port", "sample": desc}
    if not frozen:
        t1 = time.perf_counter()
        n_sh = max(1, min(3, args.steps))
        for _ in range(n_sh):
            step(True)
        cb["as_shipped"] = {"value": round(sample * n_sh / (time.perf_counter() - t1), 2), "unit": UNIT,
                            "note": f"with the lm_head logits the shipped reference computes and discards; {n_sh} step(s) after the timed region"}
    emit(({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(dt / args.steps * 1e3, 2), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": {"workload": f"{args.workload}: same model/config as the CUDA arm; {desc}"},
        "cpu_baseline": cb,
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}))


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default="infer", choices=["infer", "train", "stage1"],
                    help="train: the LoRA fine-tune step (secondary metric); stage1: the CausalLM training step of scripts/check_generation.py")
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--scenes", type=int, default=0, help="override scenes per GPU per step")
    ap.add_argument("--cpu-sample", type=int, default=64, help="scenes per CPU forward (BASELINE.json configs[0]: 64)")
    ap.add_argument("--cuda-graph", type=int, default=1, help="1: replay the inference forward from a CUDA graph (one launch per step), 0: eager launches")
    ap.add_argument("--no-secondary", action="store_true", help="headline workload only (skip cfg3 / cfg5 / fine-tune secondaries)")
    ap.add_argument("--secondary-steps", type=int, default=5)
    ap.add_argument("--dropout", type=float, default=None, help="--mode train: override lora / ltsf / transformer dropout p (default: the reference's 0.1)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--merge-lora", action="store_true", help="serve-time option: fold LoRA into the base weights at pack time (not the default "
                    "benchmark configuration: the reference runs the unmerged peft form)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="CUDA path: write what the last timed step of the headline workload returned as DIR/<name>.npy (float32 / float64, at most 64 MB)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.impl == "reference" and a.dump_outputs:
        ap.error("--dump-outputs applies to the CUDA path only (not to --impl reference)")
    _claim_stdout()
    if a.impl == "reference":
        run_reference(a)
    elif a.mode == "train":
        run_train(a)
    elif a.mode == "stage1":
        _ctx = _Ctx(a)
        _out = measure_stage1(_ctx, a.steps, a.warmup, scenes=a.scenes, dump=a.dump_outputs)
        if _ctx.rank == 0:
            emit(_out)
        _ctx.close()
    else:
        run_ours(a)
