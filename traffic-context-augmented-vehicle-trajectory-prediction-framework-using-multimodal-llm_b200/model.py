"""Host-side mirror of the reference model contract (reference scripts/train.py:847-964).

`MultiModalTrajectoryModel` keeps the reference's constructor kwargs, forward() signature, sub-module
attribute names and state_dict key layout (SURVEY.md §8b), so it drops into the reference's
train/test drivers.  The nn.Module tree below is ONLY a parameter container with the reference's names —
its torch forward() methods are never called; all arithmetic runs in libtcavp.so through engine.py."""
import math

import torch
import torch.nn as nn

from . import ops
from .config import resolve_llama
from .engine import Engine
from .train_engine import TrainEngine


class _FineTuneStep(torch.autograd.Function):
    """One autograd node for the whole model: forward = TrainEngine.train_forward (libtcavp kernels, activations stashed),
    backward = TrainEngine.train_backward (hand-written backward kernels).  The trainable nn.Parameters are the node's
    inputs, so `loss.backward()` deposits their gradients exactly where torch.optim / DistributedDataParallel expect them
    (reference scripts/im_kim_train_GRN.py:1029-1040)."""

    @staticmethod
    def forward(ctx, eng, inputs, *params):
        out = eng.train_forward(**inputs)
        ctx.eng = eng
        ctx.stash = out.pop("_ctx")        # this call's activations (not the engine's single "last forward" slot)
        ctx.names = [n for n, _ in eng.params]
        ctx.mark_non_differentiable(out["decoded"])
        ctx.set_materialize_grads(False)
        return out["loss"].clone(), out["decoded"]

    @staticmethod
    def backward(ctx, gloss, _gdec):
        if gloss is None:
            return (None, None) + (None,) * len(ctx.names)
        stash, ctx.stash = ctx.stash, None
        if stash is None:
            raise RuntimeError("tcavp_b200: backward through the same fine-tune step twice (activations are freed after the first pass)")
        grads = ctx.eng.train_backward(gloss, ctx=stash)
        res = []
        for (name, p) in ctx.eng.params:
            g = grads.get(name)
            if g is not None:
                g = g.reshape(p.shape).to(p.dtype)
            res.append(g)
        return (None, None) + tuple(res)

class _Stage1Step(torch.autograd.Function):
    """Autograd node of the stage-1 (CausalLM) objective: forward = TrainEngine.lm_forward, backward = TrainEngine.lm_backward."""

    @staticmethod
    def forward(ctx, eng, inputs, *params):
        out = eng.lm_forward(**inputs)
        ctx.eng = eng
        ctx.stash = out.pop("_ctx")
        ctx.set_materialize_grads(False)
        return out["loss"].clone()

    @staticmethod
    def backward(ctx, gloss):
        n = len(ctx.eng.params)
        if gloss is None:
            return (None, None) + (None,) * n
        stash, ctx.stash = ctx.stash, None
        if stash is None:
            raise RuntimeError("tcavp_b200: backward through the same stage-1 step twice (activations are freed after the first pass)")
        grads = ctx.eng.lm_backward(gloss, stash)
        res = []
        for (name, p) in ctx.eng.params:
            g = grads.get(name)
            res.append(None if g is None else g.reshape(p.shape).to(p.dtype))
        return (None, None) + tuple(res)


class CausalLMOutput:
    """What the reference's stage-1 loop reads off the model call (scripts/check_generation.py: `outputs.loss`)."""
    __slots__ = ("loss", "n_tokens", "logits")

    def __init__(self, loss, n_tokens):
        self.loss, self.n_tokens, self.logits = loss, n_tokens, None


# --------------------------------------------------------------------------------------------------
# parameter containers (names = reference names)
# --------------------------------------------------------------------------------------------------


class LanePolygonEncoder(nn.Module):
    """reference scripts/train.py:352-383"""

    def __init__(self, d_model=64, nhead=4, num_layers=2, max_points=64):
        super().__init__()
        self.d_model, self.max_points, self.nhead = d_model, max_points, nhead
        self.input_proj = nn.Linear(2, d_model)
        enc_layer = nn.TransformerEncoderLayer(d_model=d_model, nhead=nhead, batch_first=True)
        self.encoder = nn.TransformerEncoder(enc_layer, num_layers=num_layers, enable_nested_tensor=False)
        self.pos_embedding = nn.Parameter(torch.zeros(1, max_points, d_model))


class BlipQFormer(nn.Module):
    """reference scripts/train.py:388-414"""

    def __init__(self, vision_dim=512, hidden_size=768, nhead=8, num_encoder_layers=4, num_decoder_layers=4,
                 num_query_tokens=16):
        super().__init__()
        self.num_query_tokens, self.hidden_size, self.nhead = num_query_tokens, hidden_size, nhead
        self.vision_proj = nn.Linear(vision_dim, hidden_size)
        enc_layer = nn.TransformerEncoderLayer(d_model=hidden_size, nhead=nhead, batch_first=True)
        self.encoder = nn.TransformerEncoder(enc_layer, num_layers=num_encoder_layers, enable_nested_tensor=False)
        self.query_tokens = nn.Parameter(torch.randn(num_query_tokens, hidden_size))
        dec_layer = nn.TransformerDecoderLayer(d_model=hidden_size, nhead=nhead, batch_first=True)
        self.decoder = nn.TransformerDecoder(dec_layer, num_layers=num_decoder_layers)


class _RMSNormW(nn.Module):
    def __init__(self, n, **kw):
        super().__init__()
        self.weight = nn.Parameter(torch.ones(n, **kw))


class _LlamaAttentionW(nn.Module):
    def __init__(self, c, **kw):
        super().__init__()
        H, nh, nkv, dh = c["hidden_size"], c["num_attention_heads"], c["num_key_value_heads"], c["head_dim"]
        self.q_proj = nn.Linear(H, nh * dh, bias=False, **kw)
        self.k_proj = nn.Linear(H, nkv * dh, bias=False, **kw)
        self.v_proj = nn.Linear(H, nkv * dh, bias=False, **kw)
        self.o_proj = nn.Linear(nh * dh, H, bias=False, **kw)


class _LlamaMLPW(nn.Module):
    def __init__(self, c, **kw):
        super().__init__()
        H, I = c["hidden_size"], c["intermediate_size"]
        self.gate_proj = nn.Linear(H, I, bias=False, **kw)
        self.up_proj = nn.Linear(H, I, bias=False, **kw)
        self.down_proj = nn.Linear(I, H, bias=False, **kw)


class _LlamaLayerW(nn.Module):
    def __init__(self, c, **kw):
        super().__init__()
        self.self_attn = _LlamaAttentionW(c, **kw)
        self.mlp = _LlamaMLPW(c, **kw)
        self.input_layernorm = _RMSNormW(c["hidden_size"], **kw)
        self.post_attention_layernorm = _RMSNormW(c["hidden_size"], **kw)


class _LlamaModelW(nn.Module):
    def __init__(self, c, **kw):
        super().__init__()
        self.embed_tokens = nn.Embedding(c["vocab_size"], c["hidden_size"], **kw)
        self.layers = nn.ModuleList([_LlamaLayerW(c, **kw) for _ in range(c["num_hidden_layers"])])
        self.norm = _RMSNormW(c["hidden_size"], **kw)


class LlamaForCausalLMW(nn.Module):
    """Key layout of HF LlamaForCausalLM (HF:430-500): model.* + lm_head.weight.  lm_head is kept for
    checkpoint interop (strict loads) but never computed: its logits are discarded by the reference
    (reference scripts/train.py:547-554)."""

    def __init__(self, c, **kw):
        super().__init__()
        self.config = dict(c)
        self.model = _LlamaModelW(c, **kw)
        self.lm_head = nn.Linear(c["hidden_size"], c["vocab_size"], bias=False, **kw)
        std = 0.02
        with torch.no_grad():
            for m in self.modules():
                if isinstance(m, (nn.Linear, nn.Embedding)):
                    m.weight.normal_(0.0, std)
        if c.get("tie_word_embeddings", False):
            # HF tie_weights(): lm_head.weight IS embed_tokens.weight (Llama-3.2-1B); state_dict() still lists both keys
            self.lm_head.weight = self.model.embed_tokens.weight

    def get_input_embeddings(self):
        return self.model.embed_tokens


class _Conv1DW(nn.Module):
    """transformers.pytorch_utils.Conv1D key layout: weight [in, out] (transposed w.r.t. nn.Linear), bias [out]."""

    def __init__(self, nx, nf, **kw):
        super().__init__()
        self.in_features, self.out_features = nx, nf
        self.weight = nn.Parameter(torch.empty(nx, nf, **kw).normal_(0.0, 0.02))
        self.bias = nn.Parameter(torch.zeros(nf, **kw))


class _GPT2AttnW(nn.Module):
    def __init__(self, H, **kw):
        super().__init__()
        self.c_attn = _Conv1DW(H, 3 * H, **kw)
        self.c_proj = _Conv1DW(H, H, **kw)


class _GPT2MLPW(nn.Module):
    def __init__(self, H, I, **kw):
        super().__init__()
        self.c_fc = _Conv1DW(H, I, **kw)
        self.c_proj = _Conv1DW(I, H, **kw)


class _GPT2BlockW(nn.Module):
    def __init__(self, c, **kw):
        super().__init__()
        H, eps = c["hidden_size"], c.get("layer_norm_epsilon", 1e-5)
        self.ln_1 = nn.LayerNorm(H, eps=eps, **kw)
        self.attn = _GPT2AttnW(H, **kw)
        self.ln_2 = nn.LayerNorm(H, eps=eps, **kw)
        self.mlp = _GPT2MLPW(H, c["intermediate_size"], **kw)


class _GPT2ModelW(nn.Module):
    def __init__(self, c, **kw):
        super().__init__()
        H = c["hidden_size"]
        self.wte = nn.Embedding(c["vocab_size"], H, **kw)
        self.wpe = nn.Embedding(c["n_positions"], H, **kw)
        self.h = nn.ModuleList([_GPT2BlockW(c, **kw) for _ in range(c["num_hidden_layers"])])
        self.ln_f = nn.LayerNorm(H, eps=c.get("layer_norm_epsilon", 1e-5), **kw)


class GPT2LMHeadModelW(nn.Module):
    """Key layout of HF GPT2LMHeadModel: transformer.{wte, wpe, h.N.{ln_1, attn.c_attn, attn.c_proj, ln_2, mlp.c_fc, mlp.c_proj}, ln_f} +
    lm_head.weight (tied to wte).  What `AutoModelForCausalLM.from_pretrained("gpt2")` gives the reference (scripts/train.py:427-431)."""

    def __init__(self, c, **kw):
        super().__init__()
        self.config = dict(c)
        self.transformer = _GPT2ModelW(c, **kw)
        self.lm_head = nn.Linear(c["hidden_size"], c["vocab_size"], bias=False, **kw)
        with torch.no_grad():
            self.transformer.wte.weight.normal_(0.0, 0.02)
            self.transformer.wpe.weight.normal_(0.0, 0.02)
        if c.get("tie_word_embeddings", True):
            self.lm_head.weight = self.transformer.wte.weight

    def get_input_embeddings(self):
        return self.transformer.wte


class LoraConv1DW(nn.Module):
    """peft lora.Linear around a Conv1D (fan_in_fan_out=True, what peft sets for GPT-2's c_attn): base_layer.{weight [in, out], bias},
    lora_A.default.weight [r, in], lora_B.default.weight [out, r];  y = x W + b + (x A^T) B^T alpha / r."""

    def __init__(self, base, r, alpha, dropout):
        super().__init__()
        kw = dict(device=base.weight.device, dtype=torch.float32)
        self.base_layer = base
        self.lora_A = nn.ModuleDict({"default": nn.Linear(base.in_features, r, bias=False, **kw)})
        self.lora_B = nn.ModuleDict({"default": nn.Linear(r, base.out_features, bias=False, **kw)})
        nn.init.kaiming_uniform_(self.lora_A["default"].weight, a=math.sqrt(5))
        nn.init.zeros_(self.lora_B["default"].weight)
        self.r, self.lora_alpha, self.scaling, self.lora_dropout_p = r, alpha, alpha / r, dropout


class LoraLinearW(nn.Module):
    """peft >= 0.7 lora.Linear key layout: base_layer.weight, lora_A.default.weight, lora_B.default.weight."""

    def __init__(self, base, r, alpha, dropout):
        super().__init__()
        kw = dict(device=base.weight.device, dtype=torch.float32)   # adapters are fp32 masters (peft: autocast_adapter_dtype)
        self.base_layer = base
        self.lora_A = nn.ModuleDict({"default": nn.Linear(base.in_features, r, bias=False, **kw)})
        self.lora_B = nn.ModuleDict({"default": nn.Linear(r, base.out_features, bias=False, **kw)})
        nn.init.kaiming_uniform_(self.lora_A["default"].weight, a=math.sqrt(5))
        nn.init.zeros_(self.lora_B["default"].weight)
        self.r, self.lora_alpha, self.scaling, self.lora_dropout_p = r, alpha, alpha / r, dropout


class _LoraModelW(nn.Module):
    def __init__(self, model):
        super().__init__()
        self.model = model


class PeftModelW(nn.Module):
    """peft.get_peft_model(LoraConfig(r, alpha, dropout, bias='none', CAUSAL_LM)) for a llama-type model:
    default targets q_proj, v_proj; base weights frozen (reference scripts/train.py:432-440)."""

    TARGETS = ("q_proj", "v_proj")

    def __init__(self, model, r, alpha, dropout, target_modules=None):
        super().__init__()
        gpt2 = isinstance(model, GPT2LMHeadModelW)
        self.targets = tuple(target_modules or (("c_attn",) if gpt2 else self.TARGETS))       # peft's default mapping per model_type
        ok = ("c_attn",) if gpt2 else ("q_proj", "k_proj", "v_proj")
        bad = [t for t in self.targets if t not in ok]
        if bad:
            raise NotImplementedError(f"LoRA targets {bad} are not supported ({'/'.join(ok)} only)")
        for p in model.parameters():
            p.requires_grad_(False)
        if gpt2:
            for blk in model.transformer.h:
                blk.attn.c_attn = LoraConv1DW(blk.attn.c_attn, r, alpha, dropout)
        for layer in ([] if gpt2 else model.model.layers):
            for t in self.targets:
                setattr(layer.self_attn, t, LoraLinearW(getattr(layer.self_attn, t), r, alpha, dropout))
        self.base_model = _LoraModelW(model)
        self.config = model.config

    def get_input_embeddings(self):
        return self.base_model.model.get_input_embeddings()


class LlamaWithCrossAttnPEFT(nn.Module):
    """reference scripts/train.py:419-453 (name is historical: there is no cross-attention inside the LLM)."""

    def __init__(self, base_model_name, use_lora=True, lora_r=8, lora_alpha=32, lora_dropout=0.1, **kw):
        super().__init__()
        cfg = resolve_llama(base_model_name)
        cfg.setdefault("num_key_value_heads", cfg["num_attention_heads"])
        cfg.setdefault("head_dim", cfg["hidden_size"] // cfg["num_attention_heads"])
        # AutoModelForCausalLM resolves the class from the checkpoint's model_type: Llama by default, GPT-2 for arch = "gpt2"
        self.llama_model = GPT2LMHeadModelW(cfg, **kw) if cfg.get("arch") == "gpt2" else LlamaForCausalLMW(cfg, **kw)
        self.use_lora = use_lora
        if use_lora:
            self.llama_model = PeftModelW(self.llama_model, lora_r, lora_alpha, lora_dropout)
        self.config = cfg
        self.hidden_size = cfg["hidden_size"]

    def causal_lm(self):
        return self.llama_model.base_model.model if self.use_lora else self.llama_model


class LlamaMultiModal(nn.Module):
    """reference scripts/train.py:459-575 ("TSUE")."""

    def __init__(self, base_model_name="meta-llama/Llama-2-7b-hf", use_lora=True, lora_r=8, lora_alpha=32, lora_dropout=0.1,
                 vision_dim=512, q_hidden_size=768, q_nhead=8, q_enc_layers=4, q_dec_layers=4, q_num_query_tokens=16, **kw):
        super().__init__()
        self.qformer = BlipQFormer(vision_dim, q_hidden_size, q_nhead, q_enc_layers, q_dec_layers, q_num_query_tokens)
        self.q_hidden_size = q_hidden_size
        self.llama_wrapper = LlamaWithCrossAttnPEFT(base_model_name, use_lora, lora_r, lora_alpha, lora_dropout, **kw)
        self.llama_hidden_size = self.llama_wrapper.hidden_size
        self.q_proj = nn.Linear(q_hidden_size, self.llama_hidden_size) if self.llama_hidden_size != q_hidden_size else nn.Identity()
        self.vision_modality_embedding = nn.Parameter(torch.randn(1, 1, self.llama_hidden_size))
        self.text_modality_embedding = nn.Parameter(torch.randn(1, 1, self.llama_hidden_size))
        self.tokenizer = None   # no hub access: callers pass input_ids / attention_mask (train.py:524 branch)

    def generate_batch(self, vision_embs, prompt_ids, tokenizer, max_new_tokens=128, temperature=0.9, top_k=40, top_p=0.9, device="cuda"):
        """reference scripts/train.py:577-654 (the per-epoch sample generation of train.py:1231-1241): sampled continuation of the
        prompt after the image-token prefix, decoded with `tokenizer`.  Runs on the owning model's engine — see generate.py."""
        owner = self._owner() if getattr(self, "_owner", None) is not None else None
        if owner is None:
            raise RuntimeError("generate_batch needs the MultiModalTrajectoryModel that owns this module (its engine runs the decoder)")
        from .generate import generate_batch
        return generate_batch(owner, vision_embs, prompt_ids, tokenizer, max_new_tokens=max_new_tokens, temperature=temperature, top_k=top_k,
                              top_p=top_p, device=device)


class SelfAttentionBlock(nn.Module):
    """reference scripts/train.py:659-686"""

    def __init__(self, embed_dim, nhead=1, dropout_rate=0.1):
        super().__init__()
        self.nhead = nhead
        self.norm1 = nn.LayerNorm(embed_dim)
        self.mha = nn.MultiheadAttention(embed_dim, num_heads=nhead, dropout=dropout_rate)
        self.dropout1 = nn.Dropout(dropout_rate)
        self.ffn = nn.Sequential(nn.Linear(embed_dim, embed_dim * 4), nn.ReLU(), nn.Dropout(dropout_rate),
                                 nn.Linear(embed_dim * 4, embed_dim))
        self.dropout2 = nn.Dropout(dropout_rate)
        self.norm2 = nn.LayerNorm(embed_dim)


class LTSF_NLinearEncoder(nn.Module):
    """reference scripts/train.py:688-716"""

    def __init__(self, window_size, individual, d_model):
        super().__init__()
        if not individual:
            raise NotImplementedError("individual=False is never used by the reference drivers (train.py:1103)")
        self.encoder_linears = nn.ModuleList([nn.Linear(window_size, window_size) for _ in range(d_model)])


class LTSF_NLinearDecoder(nn.Module):
    """reference scripts/train.py:718-806 ("MFP")"""

    def __init__(self, window_size, forecast_size, individual, d_model, polygon_embed_dim=64, use_post_mlp=True,
                 post_mlp_hidden_dim=64, dropout_rate=0.1, cross_dim=768, cross_nhead=2, output_feature_dim=2):
        super().__init__()
        if not individual:
            raise NotImplementedError("individual=False is never used by the reference drivers (train.py:1103)")
        self.decoder_linears = nn.ModuleList([nn.Linear(window_size, forecast_size) for _ in range(d_model)])
        self.lane_fc = nn.Linear(polygon_embed_dim, d_model * forecast_size)
        self.use_post_mlp = use_post_mlp
        if use_post_mlp:
            self.post_mlp = nn.Sequential(nn.Linear(d_model * forecast_size, post_mlp_hidden_dim), nn.ReLU(),
                                          nn.Dropout(dropout_rate), nn.Linear(post_mlp_hidden_dim, d_model * forecast_size))
        self.cross_nhead = cross_nhead
        self.cross_attn = nn.MultiheadAttention(embed_dim=cross_dim, num_heads=cross_nhead, dropout=dropout_rate, batch_first=False)
        self.dec_proj = nn.Linear(d_model, cross_dim)
        self.dec_unproj = nn.Linear(cross_dim, d_model)
        self.fusion_layer = nn.Sequential(nn.LayerNorm(d_model), nn.Linear(d_model, d_model), nn.ReLU(), nn.Linear(d_model, d_model))
        self.out_proj = nn.Linear(d_model, output_feature_dim)


class TransformerLTSF(nn.Module):
    """reference scripts/train.py:808-842"""

    def __init__(self, seq_len, out_len, individual, feature_size, d_model, polygon_embed_dim=64, use_post_mlp=True,
                 post_mlp_hidden_dim=64, nhead=1, dropout_rate=0.1, cross_dim=768, cross_nhead=2, output_feature_dim=2):
        super().__init__()
        self.token_proj = nn.Conv1d(feature_size, d_model, kernel_size=1)
        self.nlinear_encoder = LTSF_NLinearEncoder(seq_len, individual, d_model)
        self.pos_encoding = nn.Parameter(torch.zeros(1, d_model, seq_len))
        self.attn_block = SelfAttentionBlock(embed_dim=d_model, nhead=nhead, dropout_rate=dropout_rate)
        self.decoder = LTSF_NLinearDecoder(seq_len, out_len, individual, d_model, polygon_embed_dim, use_post_mlp,
                                           post_mlp_hidden_dim, dropout_rate, cross_dim, cross_nhead, output_feature_dim)


# --------------------------------------------------------------------------------------------------
# the model
# --------------------------------------------------------------------------------------------------


class MultiModalTrajectoryModel(nn.Module):
    """Drop-in for reference scripts/train.py:847-964.

    Extra (keyword-only, defaulted) arguments beyond the reference's:
      compute_dtype : "bf16" (tcgen05 tensor-core path) or "fp32" (exact-fp32 SIMT parity path)
      llm_param_dtype / llm_device : create the frozen backbone parameters directly in this dtype / on this
                      device (a 7B fp32 host copy is 27 GB; the reference always builds fp32 on CPU)
      llm_variant   : "wrapper" -> keys `mllm.llama_wrapper.llama_model.*` (train.py), "direct" ->
                      `mllm.llama_model.*` (im_kim_train_GRN.py:444-455) on save; both are accepted on load.
    """

    def __init__(self, seq_len, out_len, individual, feature_size=2, d_model=64, lane_polygon_d_model=64, lane_polygon_nhead=4,
                 lane_polygon_layers=2, max_polygon_points=64, use_post_mlp=True, post_mlp_hidden_dim=64,
                 base_model_name="meta-llama/Llama-7B", use_lora=True, lora_r=8, lora_alpha=32, lora_dropout=0.1, vision_dim=512,
                 q_hidden_size=768, q_nhead=8, q_enc_layers=4, q_dec_layers=4, q_num_query_tokens=16, ltsf_nhead=1,
                 ltsf_dropout=0.1, *, compute_dtype="bf16", llm_param_dtype=None, llm_device=None, llm_variant="wrapper"):
        super().__init__()
        if llm_variant not in ("wrapper", "direct"):
            raise ValueError("llm_variant must be 'wrapper' (train.py key layout) or 'direct' (im_kim_train_GRN.py key layout)")
        self.llm_variant = llm_variant
        if feature_size != 2:
            raise NotImplementedError("feature_size must be 2 ((x, y) trajectories)")
        kw = {}
        if llm_param_dtype is not None:
            kw["dtype"] = llm_param_dtype
        if llm_device is not None:
            kw["device"] = llm_device
        self.lane_polygon_encoder = LanePolygonEncoder(lane_polygon_d_model, lane_polygon_nhead, lane_polygon_layers, max_polygon_points)
        self.mllm = LlamaMultiModal(base_model_name, use_lora, lora_r, lora_alpha, lora_dropout, vision_dim, q_hidden_size, q_nhead,
                                    q_enc_layers, q_dec_layers, q_num_query_tokens, **kw)
        self.llama_hidden_size = self.mllm.llama_hidden_size
        import weakref
        object.__setattr__(self.mllm, "_owner", weakref.ref(self))          # generate_batch runs on this model's engine (not a submodule link)
        self.ltsf = TransformerLTSF(seq_len, out_len, individual, feature_size, d_model, lane_polygon_d_model, use_post_mlp,
                                    post_mlp_hidden_dim, ltsf_nhead, ltsf_dropout, self.llama_hidden_size, 2, feature_size)
        self.feature_size, self.out_len, self.seq_len, self.d_model = feature_size, out_len, seq_len, d_model
        self.hparams = dict(lora_r=lora_r, lora_alpha=lora_alpha, use_lora=use_lora, q_nhead=q_nhead, ltsf_nhead=ltsf_nhead,
                            lane_polygon_nhead=lane_polygon_nhead, use_post_mlp=use_post_mlp, q_num_query_tokens=q_num_query_tokens)
        self.compute_dtype = compute_dtype
        self._engine = None
        self._engine_sig = None
        self._train_engine = None
        self._train_sig = None
        self._register_load_state_dict_pre_hook(self._translate_keys)
        self.mllm._register_load_state_dict_pre_hook(self._translate_mllm_keys_hook)
        self._register_state_dict_hook(self._variant_keys)

    # ---- checkpoint interop (SURVEY.md §8b.3) -----------------------------------------------------
    def _translate_keys(self, state_dict, prefix, *args):
        """load_state_dict pre-hook of the whole model (keys `mllm.…`)."""
        self._translate_mllm_keys(state_dict, prefix + "mllm.")

    def _translate_mllm_keys_hook(self, state_dict, prefix, *args):
        """load_state_dict pre-hook of `model.mllm` — the reference restores stage-1 checkpoints with
        `model.mllm.load_state_dict(sd, strict=True)` (train.py:1137-1138), which never reaches the top-level hook."""
        self._translate_mllm_keys(state_dict, prefix)

    def _translate_mllm_keys(self, state_dict, root):
        """Accepts (a) the V2 layout `llama_model.` directly under mllm (im_kim_train_GRN.py:444-455) and (b) the peft<0.7 layout
        without `.base_layer` (implied by ablation_study_without_lora.py:1071-1079); (c) a LoRA checkpoint loaded into
        a use_lora=False model is stripped exactly like the reference's adjust_state_dict; (d) a checkpoint of a tied-embedding
        backbone that omits `lm_head.weight` (HF safetensors of Llama-3.2-1B) gets it aliased from `embed_tokens.weight`."""
        wrap = self.mllm.llama_wrapper
        want_lora = wrap.use_lora
        for k in list(state_dict.keys()):
            if not k.startswith(root):
                continue
            nk = k
            if nk.startswith(root + "llama_model."):
                nk = root + "llama_wrapper.llama_model." + nk[len(root + "llama_model."):]
            if not nk.startswith(root + "llama_wrapper."):
                continue
            if not want_lora:
                if "lora_A" in nk or "lora_B" in nk:
                    del state_dict[k]
                    continue
                nk = nk.replace("llama_model.base_model.model.", "llama_model.").replace(".base_layer.", ".")
            else:
                if "llama_model.base_model.model." not in nk:       # a plain (no-peft) backbone checkpoint into a LoRA model
                    nk = nk.replace("llama_wrapper.llama_model.", "llama_wrapper.llama_model.base_model.model.", 1)
                for t in wrap.llama_model.targets:
                    if nk.endswith(f".self_attn.{t}.weight"):
                        nk = nk[: -len("weight")] + "base_layer.weight"
            if nk != k:
                state_dict[nk] = state_dict.pop(k)
        if wrap.config.get("tie_word_embeddings", False):
            base = root + "llama_wrapper.llama_model." + ("base_model.model." if want_lora else "")
            if base + "lm_head.weight" not in state_dict and base + "model.embed_tokens.weight" in state_dict:
                state_dict[base + "lm_head.weight"] = state_dict[base + "model.embed_tokens.weight"]

    def _variant_keys(self, module, state_dict, prefix, local_metadata):
        """state_dict hook for llm_variant="direct": keys are written as `mllm.llama_model.*` (the V2 module tree of
        im_kim_train_GRN.py:444-455, which has no wrapper class between mllm and the HF / peft model)."""
        if self.llm_variant != "direct":
            return state_dict
        a, b = prefix + "mllm.llama_wrapper.llama_model.", prefix + "mllm.llama_model."
        for k in [k for k in state_dict if k.startswith(a)]:
            state_dict[b + k[len(a):]] = state_dict.pop(k)
        return state_dict

    # ---- trainable-only / LoRA-only checkpoints (SURVEY.md §8 f3) -----------------------------------------
    def trainable_state_dict(self):
        """Only what the fine-tune step changes: LoRA A / B, Q-Former, q_proj, modality embeddings, LTSF, lane-polygon encoder (the
        reference writes the full fp32 state dict every time it improves, 27 GB at the 7B shape: train.py:1219-1224)."""
        keep = {n for n, _ in self.trainable_named_parameters()}
        return {k: v for k, v in self.state_dict().items() if k in keep}

    def load_trainable_state_dict(self, state_dict, strict=True):
        """Inverse of trainable_state_dict(): every trainable tensor must be present (strict), frozen backbone weights stay as they are."""
        want = {n for n, _ in self.trainable_named_parameters()}
        if strict:
            missing, extra = sorted(want - set(state_dict)), sorted(set(state_dict) - set(self.state_dict()))
            if missing or extra:
                raise RuntimeError(f"load_trainable_state_dict: missing {missing[:5]} ({len(missing)}), unexpected {extra[:5]} ({len(extra)})")
        res = self.load_state_dict(state_dict, strict=False)
        self._engine = None
        return res

    def lora_state_dict(self, peft_format=True):
        """LoRA adapter tensors only.  peft_format: keys as `peft.get_peft_model_state_dict` writes them into adapter_model.safetensors —
        relative to the peft model (`base_model.model...`) and without the adapter name (`lora_A.weight`, not `lora_A.default.weight`)."""
        pre = "mllm.llama_wrapper.llama_model."
        out = {}
        for k, v in self.state_dict().items():
            if "lora_A" in k or "lora_B" in k:
                out[k[len(pre):].replace(".default.", ".") if peft_format else k] = v
        return out

    def load_lora_state_dict(self, state_dict, peft_format=True):
        pre = "mllm.llama_wrapper.llama_model."
        sd = {}
        for k, v in state_dict.items():
            if peft_format:
                k = pre + k.replace(".lora_A.weight", ".lora_A.default.weight").replace(".lora_B.weight", ".lora_B.default.weight")
            sd[k] = v
        want = {k for k in self.state_dict() if "lora_A" in k or "lora_B" in k}
        if set(sd) != want:
            raise RuntimeError(f"load_lora_state_dict: key mismatch (missing {sorted(want - set(sd))[:3]}, unexpected {sorted(set(sd) - want)[:3]})")
        res = self.load_state_dict(sd, strict=False)
        self._engine = None
        return res

    # ---- engine management -------------------------------------------------------------------------
    def set_compute_dtype(self, name):
        assert name in ("bf16", "fp32")
        self.compute_dtype = name
        self._engine = None
        return self

    def _signature(self):
        return (self.compute_dtype,) + tuple((p.data_ptr(), p._version) for p in self.parameters())

    def engine(self):
        sig = self._signature()
        if self._engine is None or sig != self._engine_sig:
            self._engine = Engine(self, self.compute_dtype, merge_lora=getattr(self, "_merge_lora", False), fp8=getattr(self, "_fp8", False))
            self._engine_sig = sig
        return self._engine

    @torch.no_grad()
    def best_of_k_metrics(self, candidates, y, norm_stat):
        """The reduction of the reference's best-of-K evaluation (scripts/test.py:1336-1368): `candidates` (B, K, 2, T_out) are K decoded
        trajectories per scene (e.g. from K stochastic forward passes), returns dict(min_ade[B], min_fde[B], min_rmse[B], sums[3]) on
        the device without a host sync.  (The candidate generation itself — MC-dropout passes — is not part of this package.)"""
        dev = next(self.ltsf.parameters()).device
        c = candidates.to(device=dev, dtype=torch.float32).contiguous()
        B, K, _, T = c.shape
        yy = y.to(device=dev, dtype=torch.float32).contiguous()
        ns = norm_stat if torch.is_tensor(norm_stat) else torch.tensor(norm_stat, dtype=torch.float32)
        ns = ns.to(device=dev, dtype=torch.float32).reshape(B, 4).contiguous()
        per = torch.empty(B, 3, dtype=torch.float32, device=dev)
        tot = torch.zeros(3, dtype=torch.float32, device=dev)
        ops.best_of_k(c, yy, ns, per, tot, B=B, K=K, T_out=T)
        return dict(min_ade=per[:, 0], min_fde=per[:, 1], min_rmse=per[:, 2], sums=tot)

    def merge_lora_for_inference(self, enabled=True):
        """Serve-time option: fold every LoRA pair into its base weight when the inference engine packs the backbone
        (W' = W + (alpha / r) B A, peft's merge semantics), so the decoder runs without the rank-r side path.  The module's own
        parameters (and state_dict()) are untouched; training always uses the unmerged form."""
        if bool(enabled) != getattr(self, "_merge_lora", False):
            self._merge_lora = bool(enabled)
            self._engine = None
        return self

    def fp8_backbone_for_inference(self, enabled=True):
        """Serve-time option: the inference engine runs the Llama decoder projections on e4m3 operands (tcgen05 kind::f8f6f4) — weights
        quantised once per output channel at pack time (LoRA merged), activations per row at run time, fp32 accumulation, the scales applied
        in the GEMM epilogue.  Everything that runs through engine() follows it (forward, predict_with_metrics, evaluate, CUDA-graph replay,
        generate_batch); train-mode passes, best_of_k, the fine-tune step and stage1_forward stay bf16.  The module's own parameters (and
        state_dict()) are untouched.  Needs compute_dtype "bf16" and a Llama-arch backbone."""
        if enabled and self.compute_dtype != "bf16":
            raise ValueError(f"the fp8 serving mode needs compute_dtype 'bf16' (model has {self.compute_dtype!r})")
        if enabled and self.mllm.llama_wrapper.config.get("arch") == "gpt2":
            raise NotImplementedError("the fp8 serving mode covers Llama-arch backbones only")
        if bool(enabled) != getattr(self, "_fp8", False):
            self._fp8 = bool(enabled)
            self._engine = None
        return self

    # ---- forward -----------------------------------------------------------------------------------
    def forward(self, x, vision_embs, context_str, lane_polygon_batch, lane_polygon_len, y=None, norm_stat=None, input_ids=None,
                attention_mask=None, labels=None):
        """Same contract as reference scripts/train.py:914-964.  `labels` is accepted and ignored: it only feeds HF's
        internal CE loss, which the reference discards (train.py:547-554).  `lane_polygon_len` / `norm_stat` may be
        Python lists (as the reference's collate produces) or device tensors."""
        if input_ids is None or attention_mask is None:
            # tokenizer branch (train.py:556-575; the V2 forward of im_kim_train_GRN.py:793-795 always takes it): context_str is tokenised
            # here exactly like the reference (padding=True, truncation=True).  There is no hub access to build the tokenizer from
            # base_model_name, so the caller attaches one: `model.mllm.tokenizer = AutoTokenizer.from_pretrained(...)`.
            tok = self.mllm.tokenizer
            if tok is None:
                raise NotImplementedError("tokenizer branch (train.py:556-575): attach a tokenizer (model.mllm.tokenizer = ...) or pass "
                                          "input_ids and attention_mask")
            if getattr(tok, "pad_token", None) is None and getattr(tok, "eos_token", None) is not None:
                tok.pad_token = tok.eos_token                                    # train.py:501-502
            enc = tok(list(context_str), return_tensors="pt", padding=True, truncation=True)
            input_ids, attention_mask = enc["input_ids"], enc["attention_mask"]
        if torch.is_grad_enabled() and y is not None and norm_stat is not None and any(p.requires_grad for p in self.parameters()):
            return self._train_step(x, vision_embs, lane_polygon_batch, lane_polygon_len, y, norm_stat, input_ids, attention_mask)
        if self.training and self.dropout_active():
            # train() mode without a gradient (the reference's best-of-K evaluation: `with torch.no_grad(): model.train()`, test.py:1308-1338):
            # one stochastic pass — every dropout site of the reference draws a fresh mask
            out = self.train_engine().train_forward(x=x, vision=vision_embs, polygon=lane_polygon_batch, poly_len=lane_polygon_len,
                                                    input_ids=input_ids, attention_mask=attention_mask, y=y, norm_stat=norm_stat, keep=False)
            if y is not None and norm_stat is not None:
                return out["loss"], out["decoded"]
            return out["decoded"]
        eng = self.engine()
        out = eng.forward(x, vision_embs, lane_polygon_batch, lane_polygon_len, input_ids, attention_mask, y=y, norm_stat=norm_stat)
        if y is not None and norm_stat is not None:
            return out["loss"], out["decoded"]
        return out["decoded"]

    # ---- fine-tune step (reference scripts/im_kim_train_GRN.py:1028-1041) ----------------------------
    def trainable_named_parameters(self):
        """(name, parameter) of every tensor the fine-tune step produces a gradient for: everything with requires_grad except
        non-LoRA backbone weights (peft freezes those, train.py:432-440; full backbone fine-tuning is out of scope)."""
        return [(n, p) for n, p in self.named_parameters() if p.requires_grad and ("llama_model" not in n or "lora_" in n)]

    def train_engine(self):
        """The engine of the differentiable path; rebuilt when the frozen backbone or the set of trainable tensors changes."""
        sig = (self.compute_dtype,) + tuple((p.data_ptr(), p.requires_grad) for p in self.parameters()) + \
            tuple(p._version for n, p in self.named_parameters() if "llama_model" in n and "lora_" not in n)
        if self._train_engine is None or sig != self._train_sig:
            self._train_engine = TrainEngine(self, self.compute_dtype)
            self._train_sig = sig
        return self._train_engine

    # ---- dropout (train mode) --------------------------------------------------------------------------
    def dropout_active(self):
        """True when a train-mode pass would drop anything (model.training and some site with p > 0)."""
        return self.training and any(p > 0.0 for p in self.train_engine()._dropout_probs().values())

    def set_dropout_seed(self, seed, step=0):
        """Masks are a pure function of (seed, step, site, element): the next train-mode pass uses (seed, step), the one after it
        step + 1, ...  Without a call the base seed is torch.initial_seed()."""
        self.train_engine().set_dropout_seed(seed, step)
        return self

    def set_dropout(self, p):
        """Sets every dropout probability of the model (lora_dropout, ltsf_dropout and the nn.Transformer layers' default 0.1) to `p`."""
        for m in self.modules():
            if isinstance(m, nn.Dropout):
                m.p = float(p)
            elif isinstance(m, nn.MultiheadAttention):
                m.dropout = float(p)
            elif isinstance(m, (LoraLinearW, LoraConv1DW)):
                m.lora_dropout_p = float(p)
        cfg = self.mllm.llama_wrapper.config
        if cfg.get("arch") == "gpt2":          # HF GPT2Config's own dropouts (embeddings, attention probabilities, the two c_proj outputs)
            cfg["attn_pdrop"] = cfg["resid_pdrop"] = cfg["embd_pdrop"] = float(p)
        return self

    @torch.no_grad()
    def best_of_k(self, x, vision_embs, lane_polygon_batch, lane_polygon_len, y, norm_stat, input_ids, attention_mask, num_candidates=10):
        """The reference's best-of-K evaluation of one batch (scripts/test.py:1308-1368): `num_candidates` stochastic passes in train()
        mode without gradients, then min-over-candidates ADE / FDE / RMSE per scene.  Returns best_of_k_metrics' dict plus the
        candidates (B, K, 2, T_out)."""
        was = self.training
        self.train()
        try:
            cands = [self(x, vision_embs, None, lane_polygon_batch, lane_polygon_len, input_ids=input_ids, attention_mask=attention_mask)
                     for _ in range(num_candidates)]
        finally:
            self.train(was)
        c = torch.stack(cands, dim=1)
        out = self.best_of_k_metrics(c, y, norm_stat)
        out["candidates"] = c
        return out

    def stage1_forward(self, vision_embs, input_ids, attention_mask, labels):
        """The stage-1 model call of the reference (scripts/check_generation.py:131-151: Q-Former image tokens + prompt / answer tokens
        through the LoRA-Llama CausalLM with `labels`): returns an object whose `.loss` is the token cross-entropy (HF:487-491 — shifted,
        -100 ignored, mean over labelled tokens).  In grad mode the loss carries the hand-written backward (LoRA A / B, Q-Former,
        q_proj, modality embeddings), so `outputs.loss.backward(); optimizer.step()` of that script works unchanged; under no_grad it is
        the evaluation loss.  The vocabulary logits are never materialised beyond one row chunk (`.logits` is None)."""
        eng = self.train_engine()
        inputs = dict(vision=vision_embs, input_ids=input_ids, attention_mask=attention_mask, labels=labels)
        if torch.is_grad_enabled() and any(p.requires_grad for _, p in eng.params):
            loss = _Stage1Step.apply(eng, inputs, *[p for _, p in eng.params])
            return CausalLMOutput(loss, None)
        out = eng.lm_forward(**inputs, keep=False)
        return CausalLMOutput(out["loss"], out["n_tokens"])

    def _train_step(self, x, vision_embs, lane_polygon_batch, lane_polygon_len, y, norm_stat, input_ids, attention_mask):
        eng = self.train_engine()
        inputs = dict(x=x, vision=vision_embs, polygon=lane_polygon_batch, poly_len=lane_polygon_len, input_ids=input_ids,
                      attention_mask=attention_mask, y=y, norm_stat=norm_stat)
        return _FineTuneStep.apply(eng, inputs, *[p for _, p in eng.params])

    @torch.no_grad()
    def predict_with_metrics(self, x, vision_embs, lane_polygon_batch, lane_polygon_len, y, norm_stat, input_ids, attention_mask,
                             final_hidden=None, max_poly_len=None, cuda_graph=False):
        """forward + the reference's test-loop reduction (train.py:1302-1322) in one pass.
        Returns dict(decoded, loss, sum_ade, sum_fde, ade[B], fde[B]) — all device tensors, no host sync.
        `max_poly_len`: host-known upper bound of lane_polygon_len when the lengths live on the device (padding rows are skipped).
        `final_hidden` (B, L, H): precomputed backbone output — the frozen-backbone path of
        scripts/ablation_study_without_lora.py (encoder + fusion only; vision / token inputs are then ignored).
        `cuda_graph`: replay the forward from a CUDA graph captured per batch shape (fixed-shape serving / evaluation loops); the
        returned tensors are then reused by the next call with the same shapes — copy what you keep."""
        return self.engine().forward(x, vision_embs, lane_polygon_batch, lane_polygon_len, input_ids, attention_mask, y=y,
                                     norm_stat=norm_stat, final_hidden=final_hidden, max_poly_len=max_poly_len, cuda_graph=cuda_graph)
