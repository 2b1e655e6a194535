"""Calibration of the fp8 backbone bands of tests/test_fp8_gpu.py (run on a B200): for every Llama golden fixture, the fp8
engine's final_hidden relative L2 / row statistics / decoded / ADE / FDE against the reference golden, with and without multiplicative
noise injected into the weights of one decoder layer.    python tools/fp8_error_probe.py > fp8_probe.txt"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from conftest import build_filled_model, load_golden  # noqa: E402
from test_model_gpu import _rel_l2  # noqa: E402

FIXTURES = ["tiny_b6", "cfg1_b8", "cfg3l2_b16", "gqa_l2_b32", "llama32_1b_l2_b8"]


def run(fix, inject, fp8=True):
    m = build_filled_model(fix, "bf16", "cuda")
    m.fp8_backbone_for_inference(fp8)
    if inject:
        layer = m.mllm.llama_wrapper.causal_lm().model.layers[1]
        g = torch.Generator(device="cuda").manual_seed(5)
        with torch.no_grad():
            for p in layer.parameters():
                if p.dim() == 2:
                    p.mul_(1.0 + inject * torch.randn(p.shape, generator=g, device="cuda"))
    i = fix["inputs"]
    o = m.engine().forward(i["x"], i["vision"], i["polygon"], i["poly_len"], i["input_ids"], i["attention_mask"], y=i["y"],
                           norm_stat=i["norm_stat"], keep_intermediates=True)
    torch.cuda.synchronize()
    o = {k: (v.float().cpu() if torch.is_tensor(v) else v) for k, v in o.items()}
    g = fix["out"]
    n = g["final_hidden_head"].shape[0]
    am = g["final_hidden_absmean"]
    return dict(fh=_rel_l2(o["final_hidden"][:n], g["final_hidden_head"]),
                rowmean=float(((o["final_hidden"].mean(-1) - g["final_hidden_rowmean"]).abs() / am).max()),
                absmean=float(((o["final_hidden"].abs().mean(-1) - am).abs() / am).max()),
                maxabs=float((o["final_hidden"][:n] - g["final_hidden_head"]).abs().max() / g["final_hidden_head"].abs().max()),
                dec=float((o["decoded"] - g["decoded"]).abs().max()),
                ade=abs(float(o["ade"].mean()) - float(g["ade"].mean())) / float(g["ade"].mean()),
                fde=abs(float(o["fde"].mean()) - float(g["fde"].mean())) / float(g["fde"].mean()))


if __name__ == "__main__":
    print("GPU:", torch.cuda.get_device_name())
    for name in FIXTURES:
        fix = load_golden(name)
        for fp8, inject in ((False, 0.0), (True, 0.0), (True, 0.02), (True, 0.05), (True, 0.1)):
            r = run(fix, inject, fp8)
            print(name, "fp8" if fp8 else "bf16", f"inject={inject}", " ".join(f"{k}={v:.3e}" for k, v in r.items()), flush=True)
