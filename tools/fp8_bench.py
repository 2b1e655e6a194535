"""fp8 serving mode against the bf16 engine, in one process on the same seeded inputs (run on a B200):

    python tools/fp8_bench.py --workload cfg2 --out fp8_cfg2.json [--proj wqkv wo wgu wdown]

Per workload: A-B-A-B rounds of CUDA-graph replays of the bf16 engine and the fp8 engine (device events around each leg), then one
profiled eager step of each (per-launch events: per-projection GEMM time, quantisation-pass time and bandwidth), then the output
difference fp8 vs bf16 (decoded, ADE / FDE, final_hidden).  `--proj` sets Engine.FP8_PROJ for the fp8 engine (default: the shipped
choice); the per-projection table compares every projection that ran in fp8 with its bf16 GEMM."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import WORKLOADS, build_model, scenes_for  # noqa: E402


def gpu_info():
    name = torch.cuda.get_device_name()
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True,
                            timeout=30).stdout.strip().splitlines()[torch.cuda.current_device()]
    except Exception as e:       # the number is reported without it rather than guessed
        pl = f"unavailable ({e})"
    return dict(gpu=name, power_limit_and_max_sm_clock=pl)


def proj_of(label, lc):
    """Decoder projection a GEMM launch label belongs to, from its [N, K] (None for every other GEMM)."""
    H, I, nh, nkv = lc["hidden_size"], lc["intermediate_size"], lc["num_attention_heads"], lc["num_key_value_heads"]
    dh = lc["head_dim"]
    if "[" not in label or not label.startswith("gemm_"):
        return None
    inner = label.split("[", 1)[1].rstrip("]")
    if inner.startswith("M"):          # small-M launches (the Q-Former's 16 query rows per scene) share [N, K] with decoder projections
        return None
    dims = {p[0]: int(p[1:]) for p in inner.split(",") if p[:1] in ("N", "K") and p[1:].isdigit()}
    N, K = dims.get("N"), dims.get("K")
    if N == (nh + 2 * nkv) * dh and H <= K < H + 64:     # bf16: K-extended by the LoRA side columns
        return "wqkv"
    return {(H, nh * dh): "wo", (2 * I, H): "wgu", (H, I): "wdown"}.get((N, K))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="cfg2", choices=["cfg2", "cfg3"])
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--proj", nargs="*", default=None)
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    import tcavp_b200 as T
    from tcavp_b200 import ops
    from tcavp_b200.engine import Engine
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    T.lib.build()
    preset, B, l_text = WORKLOADS[args.workload]
    model, cfg = build_model(preset, dev)
    lc = T.resolve_llama(cfg["base_model_name"])
    s = scenes_for(cfg, B, l_text, 1234, lc["vocab_size"])
    d = {k: s[k].to(dev) for k in ("x", "y", "vision", "polygon", "input_ids", "attention_mask")}
    lens = torch.tensor(s["poly_len"], dtype=torch.int32, device=dev)
    ns = torch.tensor(s["norm_stat"], dtype=torch.float32, device=dev)
    max_poly = int(max(s["poly_len"]))
    shipped = Engine.FP8_PROJ
    if args.proj is not None:
        Engine.FP8_PROJ = tuple(args.proj)
    with torch.no_grad():
        engines = {"bf16": Engine(model, "bf16"), "fp8": Engine(model, "bf16", fp8=True)}
    fp8_proj = Engine.FP8_PROJ
    Engine.FP8_PROJ = shipped

    def run(e, graph=True, keep=False):
        return e.forward(d["x"], d["vision"], d["polygon"], lens, d["input_ids"], d["attention_mask"], y=d["y"], norm_stat=ns,
                         max_poly_len=max_poly, cuda_graph=graph, keep_intermediates=keep)
    for e in engines.values():                  # graph capture + warm-up of every shape
        for _ in range(3):
            run(e)
    torch.cuda.synchronize()
    ms = {k: [] for k in engines}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(args.rounds):                # A-B-A-B: clock drift of the warming board hits both alike
        for k, e in engines.items():
            run(e)
            e0.record()
            for _ in range(args.steps):
                run(e)
            e1.record()
            e1.synchronize()
            ms[k].append(e0.elapsed_time(e1) / args.steps)
    res = dict(workload=args.workload, preset=preset, scenes_per_step=B, l_text=l_text, fp8_proj=list(fp8_proj), **gpu_info(),
               method=f"{args.rounds} A-B-A-B rounds x {args.steps} CUDA-graph replays per leg, device events; per-launch events in a separate eager step")
    for k in engines:
        best = min(ms[k])
        res[k] = dict(ms_per_step=round(best, 3), ms_all_rounds=[round(v, 3) for v in ms[k]], scenes_per_s=round(B / best * 1e3, 1))
    res["speedup_scenes_per_s"] = round(res["fp8"]["scenes_per_s"] / res["bf16"]["scenes_per_s"], 4)
    # per-launch profile of one eager step of each engine
    groups = {}
    for k, e in engines.items():
        run(e, graph=False)
        with ops.LaunchProfiler() as prof:
            run(e, graph=False)
        groups[k] = prof.summary()["groups"]
    table = {}
    for k, gs in groups.items():
        for g in gs:
            p = proj_of(g["kernel"], lc)
            if p is not None:
                table.setdefault(p, {})[k + "_gemm_ms"] = table.get(p, {}).get(k + "_gemm_ms", 0.0) + g["time_ms"]
                table[p].setdefault(k + "_kernels", []).append(g["kernel"])
    quant = [g for g in groups["fp8"] if g["kernel"].startswith("quant_e4m3_kernel")]
    res["quant_passes"] = [dict(kernel=g["kernel"], launches=g["launches"], time_ms=g["time_ms"], tb_per_s=round(g["gbs"] / 1e3, 3)) for g in quant]
    qms = {int(g["kernel"].split("[")[1].rstrip("]")): g["time_ms"] for g in quant}
    H, I = lc["hidden_size"], lc["intermediate_size"]
    nq = lc["num_attention_heads"] * lc["head_dim"]
    quant_cols = {"wqkv": H, "wo": nq, "wgu": H, "wdown": I}
    for p, row in table.items():
        if p in fp8_proj:
            # the quantisation passes of one width are shared out by launch count: QKV and gate/up both quantise the H-wide residual stream
            same = [q for q in fp8_proj if quant_cols[q] == quant_cols[p]]
            row["fp8_quant_ms"] = round(qms.get(quant_cols[p], 0.0) / len(same), 4)
            row["fp8_total_ms"] = round(row["fp8_gemm_ms"] + row["fp8_quant_ms"], 4)
            row["fp8_faster"] = row["fp8_total_ms"] < row.get("bf16_gemm_ms", float("inf"))
        for k in ("bf16_gemm_ms", "fp8_gemm_ms"):
            if k in row:
                row[k] = round(row[k], 4)
    res["per_projection_one_step"] = table
    res["profile_top"] = {k: gs[:12] for k, gs in groups.items()}
    # output difference fp8 vs bf16 on the same inputs
    with torch.no_grad():
        ob, o8 = run(engines["bf16"], graph=False, keep=True), run(engines["fp8"], graph=False, keep=True)
    torch.cuda.synchronize()
    fb, f8 = ob["final_hidden"].double(), o8["final_hidden"].double()
    ade_b, fde_b = float(ob["ade"].double().mean()), float(ob["fde"].double().mean())
    res["fp8_vs_bf16"] = dict(max_abs_d_decoded=float((o8["decoded"] - ob["decoded"]).abs().max()),
                              rel_d_ade=abs(float(o8["ade"].double().mean()) - ade_b) / ade_b, rel_d_fde=abs(float(o8["fde"].double().mean()) - fde_b) / fde_b,
                              rel_l2_final_hidden=float((f8 - fb).norm() / fb.norm()))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("workload", "gpu", "power_limit_and_max_sm_clock", "bf16", "fp8", "speedup_scenes_per_s", "fp8_vs_bf16")}))
    print(json.dumps(res["per_projection_one_step"]))
    print(json.dumps(res["quant_passes"]))


if __name__ == "__main__":
    main()
