"""Host-side checks of the fp8 serving mode (Engine(fp8=True) / fp8_backbone_for_inference): e4m3 weight packing and the option's
argument checks.  Packing runs on the host; nothing here needs a GPU."""
import pytest
import torch

import tcavp_b200 as T
from tcavp_b200.engine import Engine


def _filled_tiny(seed=3, **over):
    m = T.MultiModalTrajectoryModel(**dict(T.MODEL_PRESETS["tiny"], **over))
    sd = m.state_dict()
    T.deterministic_fill_(sd, seed)           # LoRA B non-zero too, so the merge is visible
    m.load_state_dict(sd, strict=True)
    return m.eval()


def _reference_w(m, e, li):
    """fp32 W' of layer li exactly as the bf16 pack defines it: LoRA merged, q / k rows RoPE-permuted, RMSNorm weights folded into the
    columns, gate / up interleaved."""
    wrap = m.mllm.llama_wrapper
    layer = wrap.causal_lm().model.layers[li]
    targets = tuple(wrap.llama_model.targets)
    sa, mlp = layer.self_attn, layer.mlp

    def w32(mod, name):
        if name in targets:
            return mod.base_layer.weight.double() + mod.scaling * (mod.lora_B["default"].weight.double() @ mod.lora_A["default"].weight.double())
        return mod.weight.double()
    ln1 = layer.input_layernorm.weight.double()
    ln2 = layer.post_attention_layernorm.weight.double()
    qkv = torch.cat([w32(sa.q_proj, "q_proj"), w32(sa.k_proj, "k_proj"), w32(sa.v_proj, "v_proj")])
    if e.llm["fuse_rope"]:
        qkv = qkv[e.llm["qk_perm"].cpu()]
    gu = torch.empty(2 * mlp.gate_proj.weight.shape[0], mlp.gate_proj.weight.shape[1], dtype=torch.float64)
    gu[0::2] = mlp.gate_proj.weight.double() * ln2
    gu[1::2] = mlp.up_proj.weight.double() * ln2
    return dict(wqkv=qkv * ln1, wo=sa.o_proj.weight.double(), wgu=gu, wdown=mlp.down_proj.weight.double())


def test_fp8_pack_dequantises_to_the_fp32_weight():
    m = _filled_tiny()
    with torch.no_grad():
        e = Engine(m, "bf16", fp8=True)
    assert e.llm["kx"] == 0 and e.llm["n_lora"] == 0                  # LoRA always merged
    assert e.FP8_PROJ and set(e.FP8_PROJ) <= {"wqkv", "wo", "wgu", "wdown"}
    for li, ly in enumerate(e.llm["layers"]):
        ref = _reference_w(m, e, li)
        for name in ("wqkv", "wo", "wgu", "wdown"):
            w = ly[name]
            if name not in e.FP8_PROJ:
                assert w.dtype == torch.bfloat16 and ("s_" + name) not in ly
                continue
            assert w.dtype == torch.float8_e4m3fn and w.shape == ref[name].shape          # no bf16 copy of an fp8 weight
            s = ly["s_" + name]
            assert s.dtype == torch.float32 and s.shape == (w.shape[0],)
            torch.testing.assert_close(s.double(), ref[name].abs().amax(1) / 448, rtol=1e-6, atol=0)
            deq = w.double() * s.double()[:, None]
            # e4m3: 3 mantissa bits (half-ulp 2^-4 relative), subnormal spacing 2^-9 of the row scale's 448
            bound = torch.maximum(ref[name].abs() * 2.0 ** -4, s.double()[:, None] * 2.0 ** -10) * (1 + 1e-6) + 1e-30
            assert bool(((deq - ref[name]).abs() <= bound).all()), name
            assert float(w.float().abs().amax()) == 448.0
    assert e.llm["embed"].dtype == torch.bfloat16 and e.llm["norm"].dtype == torch.float32


def test_fp8_pack_layout_is_the_bf16_merged_layout():
    """The reference W' above is the bf16 engine's merged pack (same permutation, fold and interleave) up to bf16 rounding."""
    m = _filled_tiny()
    with torch.no_grad():
        e8, eb = Engine(m, "bf16", fp8=True), Engine(m, "bf16", merge_lora=True)
    for li, ly in enumerate(eb.llm["layers"]):
        ref = _reference_w(m, e8, li)
        for name in ("wqkv", "wo", "wgu", "wdown"):
            torch.testing.assert_close(ly[name].double(), ref[name], rtol=2 ** -7, atol=1e-30)
    assert torch.equal(e8.llm["qk_perm"], eb.llm["qk_perm"])


def test_zero_weight_row_gets_zero_scale():
    m = _filled_tiny()
    with torch.no_grad():
        m.mllm.llama_wrapper.causal_lm().model.layers[0].mlp.down_proj.weight[5].zero_()
        e = Engine(m, "bf16", fp8=True)
    ly = e.llm["layers"][0]
    assert float(ly["s_wdown"][5]) == 0.0 and torch.count_nonzero(ly["wdown"][5].float()) == 0


def test_fp8_option_argument_checks_and_state_dict():
    m = _filled_tiny()
    sd0 = {k: v.clone() for k, v in m.state_dict().items()}
    assert m.fp8_backbone_for_inference(True) is m
    e = m.engine()
    assert e.fp8 and any(ly[n].dtype == torch.float8_e4m3fn for ly in e.llm["layers"] for n in e.FP8_PROJ)
    m.fp8_backbone_for_inference(False)
    assert m._engine is None and not m.engine().fp8
    sd1 = m.state_dict()
    assert list(sd1) == list(sd0) and all(torch.equal(sd1[k], sd0[k]) for k in sd0)
    with pytest.raises(ValueError):
        _filled_tiny(compute_dtype="fp32").fp8_backbone_for_inference()
    with pytest.raises(ValueError):
        Engine(m, "fp32", fp8=True)
    g = T.MultiModalTrajectoryModel(**dict(T.MODEL_PRESETS["tiny"], base_model_name="gpt2-tiny"))
    with pytest.raises(NotImplementedError):
        g.fp8_backbone_for_inference()
    with pytest.raises(NotImplementedError):
        Engine(g, "bf16", fp8=True)
    g.fp8_backbone_for_inference(False)           # turning it off is always allowed
