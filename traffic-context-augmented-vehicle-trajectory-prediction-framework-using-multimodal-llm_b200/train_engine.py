"""Fine-tune step: forward with activation stashing + hand-written backward over libtcavp.so
(reference scripts/im_kim_train_GRN.py:1028-1040: zero_grad / forward / loss.backward() / AdamW.step()).

The reference leaves the backward to torch autograd.  Here `TrainEngine.train_forward` runs the same kernels as the
inference engine (new buffers per block instead of in-place reuse, so every activation a gradient needs survives) and
`train_backward` walks the blocks in reverse calling the backward kernels of include/tcavp.h:
  * dX through every linear map = tcavp_gemm on a transposed weight copy (frozen LLM weights are transposed once);
  * dW of trainable weights     = tcavp_gemm(dY^T, X^T) after tcavp_transpose; biases / broadcast tables = tcavp_period_sum;
  * LoRA A / B gradients        = tcavp_skinny_dw (rank-r reductions over the token axis) — base weights get no gradient;
  * attention / LayerNorm / RMSNorm / SwiGLU / RoPE / NLinear / masked-mean / head backward kernels.
Gradients are produced in the reference's state_dict layout (fp32) and handed to torch through ONE autograd.Function
(model.py), so `loss.backward(); optimizer.step()` and DistributedDataParallel hooks work unchanged.
Dropout (train mode, every site of the reference: lora_dropout, ltsf_dropout, the nn.Transformer layers' 0.1) uses the counter-based
mask of tcavp_dropout — a pure function of (seed, site, element) that the backward pass re-creates, nothing is stored — see
`DropPlan`.  With `model.eval()` or every p = 0 the step is the deterministic one the p = 0 goldens pin."""
import math
import os

import torch

from . import ops
from .engine import Engine, _Lin, _f32


def _pad8(n):
    return (n + 7) // 8 * 8


# ---- dropout sites ------------------------------------------------------------------------------------------------------
# site id = module << 20 | layer << 8 | kind.  The oracle (oracle/dropout.py) derives the same ids from the ORDER in which the
# reference's forward calls F.dropout / scaled_dot_product_attention, so masks are bit-identical on both sides.
MOD = dict(poly=1, qenc=2, qdec=3, llm=4, ltsf=5, dec=6)
KIND = dict(sa_attn=0, drop1=1, ffn=2, drop2=3, ca_attn=4, drop3=5, post=6, cross_attn=7, lora_q=8, lora_k=9, lora_v=10, lora_c=11, embd=12, attn=13, resid1=14, resid2=15)


def site_id(mod, layer, kind):
    return (MOD[mod] << 20) | (layer << 8) | KIND[kind]


class DropPlan:
    """The dropout sites of ONE train-mode forward pass: `plan(mod, layer, kind)` -> ops.Drop or None (p = 0 / eval mode).
    All sites share one device seed tensor that is private to the pass, so the backward pass regenerates the same masks even if
    another forward ran in between."""

    def __init__(self, seed, probs):
        self.seed, self.probs = seed, probs
        self._cache = {}

    def __call__(self, mod, layer, kind):
        p = self.probs.get((mod, kind), 0.0) if self.seed is not None else 0.0
        if p <= 0.0:
            return None
        key = (mod, layer, kind)
        if key not in self._cache:
            self._cache[key] = ops.Drop(self.seed, site_id(mod, layer, kind), p)
        return self._cache[key]

    @property
    def active(self):
        return self.seed is not None and any(p > 0.0 for p in self.probs.values())


class TrainEngine(Engine):
    SPLIT_SMALL = False      # the fine-tune step keeps the fp32 layers in exact FFMA (their weights are re-packed every step)

    def __init__(self, model, compute_dtype="bf16"):
        super().__init__(model, compute_dtype)
        self.model = model
        self.G = {}
        self.grad_targets = None      # {reference parameter name: fp32 view to write its gradient into} (optional)
        self._flags()
        self._bwd_packed = False
        self._names()
        self._seed_state = None       # CUDA int32[2]: (base seed, step counter); bumped on the device after every train-mode forward
        self._seed_inc = None
        self.drop = DropPlan(None, {})

    # ---- bookkeeping --------------------------------------------------------------------------------
    def _flags(self):
        m = self.model
        rg = lambda mod: any(p.requires_grad for p in mod.parameters())   # noqa: E731
        self.tr_poly, self.tr_ltsf = rg(m.lane_polygon_encoder), rg(m.ltsf)
        self.tr_qf = rg(m.mllm.qformer) or rg(m.mllm.q_proj) or m.mllm.vision_modality_embedding.requires_grad
        self.tr_text = m.mllm.text_modality_embedding.requires_grad
        self.tr_lora = any(p.requires_grad for n, p in m.mllm.llama_wrapper.named_parameters() if "lora_" in n)
        self.need_llm_bwd = self.tr_qf or self.tr_text or self.tr_lora

    def _names(self):
        """(name, parameter) of every trainable tensor this engine produces a gradient for.  Non-LoRA LLM weights are treated
        as frozen even if requires_grad is set (full fine-tuning of the backbone is out of scope)."""
        self.params = self.model.trainable_named_parameters()
        wrap = self.model.mllm.llama_wrapper
        self.llm_prefix = ("mllm.llama_wrapper.llama_model." + ("base_model.model." if wrap.use_lora else "") +
                           ("transformer.h." if wrap.config.get("arch") == "gpt2" else "model.layers."))

    # ---- dropout plumbing -----------------------------------------------------------------------------
    def set_dropout_seed(self, base, step=0):
        """The next train-mode forward draws its masks from (base, step); every forward after it from step + 1, + 2, ..."""
        if self.dev.type != "cuda":
            raise ops._lib.TcavpError("dropout needs the model on a CUDA device")
        v = torch.tensor([int(base) & 0x7FFFFFFF, int(step) & 0x7FFFFFFF], dtype=torch.int32)
        if self._seed_state is None:
            self._seed_state = v.to(self.dev)
            self._seed_inc = torch.tensor([0, 1], dtype=torch.int32, device=self.dev)
        else:
            self._seed_state.copy_(v)

    def _dropout_probs(self):
        """p of every site, read from the container modules (the reference passes lora_dropout / ltsf_dropout to its constructors,
        train.py:432-440, 663-671, 745-754; nn.TransformerEncoderLayer / DecoderLayer keep torch's default 0.1, train.py:358, 402-405)."""
        m = self.model
        pr = {}

        def tl(mod, layers, dec=False):
            if len(layers) == 0:
                return
            l = layers[0]
            pr[(mod, "sa_attn")], pr[(mod, "drop1")] = float(l.self_attn.dropout), float(l.dropout1.p)
            pr[(mod, "ffn")], pr[(mod, "drop2")] = float(l.dropout.p), float(l.dropout2.p)
            if dec:
                pr[(mod, "ca_attn")], pr[(mod, "drop3")] = float(l.multihead_attn.dropout), float(l.dropout3.p)
        tl("poly", m.lane_polygon_encoder.encoder.layers)
        tl("qenc", m.mllm.qformer.encoder.layers)
        tl("qdec", m.mllm.qformer.decoder.layers, dec=True)
        ab = m.ltsf.attn_block
        pr[("ltsf", "sa_attn")] = float(ab.mha.dropout)
        pr[("ltsf", "drop1")], pr[("ltsf", "ffn")], pr[("ltsf", "drop2")] = float(ab.dropout1.p), float(ab.ffn[2].p), float(ab.dropout2.p)
        d = m.ltsf.decoder
        pr[("dec", "cross_attn")] = float(d.cross_attn.dropout)
        if d.use_post_mlp:
            pr[("dec", "post")] = float(d.post_mlp[2].p)
        wrap = m.mllm.llama_wrapper
        if wrap.config.get("arch") == "gpt2":
            # HF GPT2Config's own dropouts (modeling_gpt2.py: GPT2Model.drop on wte + wpe, attn_dropout on the probabilities, resid_dropout
            # after attn.c_proj, GPT2MLP.dropout after mlp.c_proj); a shape dict without the keys means 0
            c = wrap.config
            pr[("llm", "embd")], pr[("llm", "attn")] = float(c.get("embd_pdrop", 0.0)), float(c.get("attn_pdrop", 0.0))
            pr[("llm", "resid1")] = pr[("llm", "resid2")] = float(c.get("resid_pdrop", 0.0))
            if wrap.use_lora:
                pr[("llm", "lora_c")] = float(wrap.causal_lm().transformer.h[0].attn.c_attn.lora_dropout_p)
        elif wrap.use_lora:
            layer0 = wrap.causal_lm().model.layers[0].self_attn
            for t in wrap.llama_model.targets:
                pr[("llm", "lora_" + t[0])] = float(getattr(layer0, t).lora_dropout_p)
        return pr

    def _begin_pass(self):
        """Builds the DropPlan of this forward: active only in train mode with some p > 0; the pass gets a private copy of the seed."""
        probs = self._dropout_probs() if self.model.training else {}
        if not any(p > 0.0 for p in probs.values()):
            self.drop = DropPlan(None, {})
            return
        if self._seed_state is None:
            self.set_dropout_seed(torch.initial_seed() & 0x7FFFFFFF, 0)
        seed = self._seed_state.clone()
        self._seed_state.add_(self._seed_inc)         # device-side: a captured CUDA graph advances the step on every replay
        self.drop = DropPlan(seed, probs)

    def _drop_res(self, t, drop, residual):
        """residual + dropout(t), in place on t (the sub-layer output is not needed un-dropped)."""
        return ops.dropout(t, t, drop, rows=t.shape[0], cols=t.shape[1], ldi=t.stride(0), ldo=t.stride(0), residual=residual,
                           ldr=None if residual is None else residual.stride(0))

    def _drop_grad(self, dy, drop):
        """Gradient through a dropout site: the same mask and scale on a copy of dy (dy itself still feeds the residual branch)."""
        if drop is None:
            return dy
        return ops.dropout(dy, self._new(*dy.shape, dtype=dy.dtype), drop, rows=dy.shape[0], cols=dy.shape[1], ldi=dy.stride(0))

    @torch.no_grad()
    def sync_params(self):
        """Re-packs the trainable tensors from the nn.Parameters (they change every optimizer step); frozen LLM base weights
        stay packed."""
        m = self.model
        self._pack_poly(m.lane_polygon_encoder)
        self._pack_qformer(m.mllm)
        self._pack_ltsf(m.ltsf)
        self.lt["be_pos"] = self.lt["be"] + self.lt["pos"]
        if self.llm.get("arch") == "gpt2":
            if self.need_llm_bwd and not self._bwd_packed:
                for ly in self.llm["layers"]:
                    ly["wqkvT"] = ly["wqkv"].t().contiguous()           # [H + kx, 3H]: rows [0, H) -> d ln_1(x), rows [H, H + kx) -> d (x A^T)
                self._bwd_packed = True
            self._refresh_lora_gpt2()
            return
        if self.need_llm_bwd and not self._bwd_packed:
            for ly in self.llm["layers"]:
                ly["wdownT"] = ly["wdown"].t().contiguous()
                ly["wguT"] = ly["wgu"].t().contiguous()
                ly["woT"] = ly["wo"].t().contiguous()
                ly["wqkvT"] = ly["wqkv"].t().contiguous()
            self._bwd_packed = True
        self._refresh_lora()

    def _refresh_lora(self):
        L = self.llm
        if not L["kx"]:
            return
        wrap = self.model.mllm.llama_wrapper
        H, r, kx, nh, nkv, dh = L["H"], L["r"], L["kx"], L["nh"], L["nkv"], L["dh"]
        nq, nk = nh * dh, nkv * dh
        rows = {"q_proj": (0, nq), "k_proj": (nq, nq + nk), "v_proj": (nq + nk, nq + 2 * nk)}
        L["rows"] = rows
        for ly, layer in zip(L["layers"], wrap.causal_lm().model.layers):
            ext = torch.zeros(nq + 2 * nk, kx, dtype=torch.float32, device=self.dev)
            for ti, name in enumerate(L["targets"]):
                mod = getattr(layer.self_attn, name)
                r0, r1 = rows[name]
                ext[r0:r1, ti * r:(ti + 1) * r] = mod.lora_B["default"].weight.detach().float().to(self.dev) * mod.scaling
                ly["a_cat"][ti * r:(ti + 1) * r] = (mod.lora_A["default"].weight.detach().float().to(self.dev) * ly["ln1"][None, :]).to(self.act)
            if L["fuse_rope"]:
                ext = ext[L["qk_perm"]]
            ly["wqkv"][:, H:] = ext.to(self.act)
            if "wqkvT" in ly:
                ly["wqkvT"][H:, :] = ext.t().to(self.act)
            ly["a_catT"] = ly["a_cat"].t().contiguous()
            # lora_dropout (peft lora.Linear: lora_A(dropout(x)), train.py:432-440): every target sees its own mask of the normalised input,
            # so the side product is one masked copy + one skinny GEMM per target.  The masked copy is exact (x or 0); the 1 / (1 - p)
            # factor rides on the per-target weight ([A'_t ; 0] rows of the other targets zeroed, so the GEMMs accumulate).
            ly.pop("a_cat_t", None)
            ly.pop("a_cat_s", None)
            drops = self._lora_drops(0)
            if drops and self._lora_fused():
                # fused form (csrc/lora_drop.cu): the masks are regenerated on the operand fragments; one matrix with every target's
                # 1 / (1 - p) folded into its rows serves the forward product and the input gradient
                sc = torch.cat([torch.full((r,), d.scale, dtype=torch.float32, device=self.dev) for d in drops])
                ly["a_cat_s"] = (ly["a_cat"][:len(drops) * r].float() * sc[:, None]).to(self.act).contiguous()
                ly["lora_scales"] = sc
            elif drops:
                ly["a_cat_t"], ly["a_catT_t"] = [], []
                for ti, d in enumerate(drops):
                    w = torch.zeros_like(ly["a_cat"])
                    w[ti * r:(ti + 1) * r] = (ly["a_cat"][ti * r:(ti + 1) * r].float() * d.scale).to(self.act)
                    ly["a_cat_t"].append(w)
                    ly["a_catT_t"].append(w.t().contiguous())

    def _refresh_lora_gpt2(self):
        """c_attn's LoRA pair re-packed from the fp32 masters (they move every optimizer step): B alpha / r as the extra K columns of the
        fused QKV weight, A as the skinny operand; with lora_dropout live, A also with 1 / (1 - p) folded in (the masked copy is x or 0)."""
        L = self.llm
        if not L["kx"]:
            return
        H, r = L["H"], L["r"]
        d0 = self._lora_drops(0)
        for ly, blk in zip(L["layers"], self.model.mllm.llama_wrapper.causal_lm().transformer.h):
            ca = blk.attn.c_attn
            ext = (ca.lora_B["default"].weight.detach().float().to(self.dev) * ca.scaling).to(self.act)          # [3H, r]
            ly["wqkv"][:, H:H + r] = ext
            if "wqkvT" in ly:
                ly["wqkvT"][H:H + r, :] = ext.t()
            A = ca.lora_A["default"].weight.detach().float().to(self.dev)
            ly["a_cat"][:r] = A.to(self.act)
            ly["a_catT"] = ly["a_cat"].t().contiguous()
            ly.pop("a_cat_d", None)
            ly.pop("a_cat_s", None)
            if d0 and self._lora_fused():      # csrc/lora_drop.cu: the mask is regenerated on the operand fragments (no masked copy)
                ly["a_cat_s"] = (A * d0[0].scale).to(self.act).contiguous()
            elif d0:
                w = torch.zeros_like(ly["a_cat"])
                w[:r] = (A * d0[0].scale).to(self.act)
                ly["a_cat_d"], ly["a_catT_d"] = w, w.t().contiguous()

    def _lora_fused(self):
        """lora_dropout through the fused kernels (bf16 compute, rank 8 / 16, hidden size a multiple of 64); TCAVP_LORA_DROP_FUSED=0
        keeps the literal masked copy + skinny GEMM per target (A/B runs, and the fp32 parity mode)."""
        L = self.llm
        return (self.act == torch.bfloat16 and L["r"] in (8, 16) and L["H"] % 64 == 0 and 1 <= len(L["targets"]) <= 4
                and os.environ.get("TCAVP_LORA_DROP_FUSED", "1") != "0")

    def _lora_drops(self, li):
        """[ops.Drop per LoRA target] of decoder layer `li`, or None when lora_dropout is inactive."""
        L = self.llm
        if not L["kx"] or not self.drop.active:
            return None
        ds = [self.drop("llm", li, "lora_" + t[0]) for t in L["targets"]]
        if all(d is None for d in ds):
            return None
        return [d if d is not None else ops.Drop(self.drop.seed, site_id("llm", li, "lora_" + t[0]), 0.0) for d, t in zip(ds, L["targets"])]

    def _g(self, name, shape):
        """Zero-initialised fp32 gradient buffer for reference parameter `name`.  When the caller registered a target view for
        it (FineTuner: a slice of the flat all-reduce buffer, zeroed at the start of the step) the gradient is produced in
        place and never copied."""
        tgt = self.grad_targets.get(name) if self.grad_targets else None
        if tgt is not None and tgt.numel() == math.prod(shape):
            t = tgt.view(*shape)
        else:
            t = torch.zeros(*shape, dtype=torch.float32, device=self.dev)
        self.G[name] = t
        return t

    # ---- linear map: forward / backward ---------------------------------------------------------------
    def _lin(self, x, L, *, act=ops.ACT_NONE, residual=None, out_dtype=None):
        y = self._new(x.shape[0], L.N, dtype=out_dtype or x.dtype)
        return ops.gemm(x, L.w, y, bias=L.b, act=act, residual=residual)

    def _wT(self, L):
        if L.wT is None:
            if L.w.dtype == torch.bfloat16 and L.N % 8:
                raise ops._lib.TcavpError(f"backward of a bf16 linear needs out_features % 8 == 0 (got {L.N})")
            L.wT = ops.transpose(L.w, torch.empty(L.K, L.N, dtype=L.w.dtype, device=self.dev), rows=L.N, cols=L.K, ldi=L.w.stride(0))
        return L.wT

    def _dw_gemm(self, dy, x, out, *, N, K, lddy=None, ldx=None):
        """out[N, K] (fp32) = dy^T . x over the M rows; operands are transposed (and dtype-unified) explicitly."""
        M = dy.shape[0]
        if dy.dtype == torch.float32 or x.dtype == torch.float32 or 2.0 * M * N * K < 6e10:
            # no transposed copies: tensor-core kernel on the row-major bf16 operands (ldmatrix.trans), FFMA kernel for the fp32 layers;
            # only the very long contractions (K/V projection of the fusion cross-attention) go through transpose + tcgen05 GEMM
            return ops.dw(dy, x, out, M=M, N=N, K=K, lddy=dy.stride(0) if lddy is None else lddy, ldx=x.stride(0) if ldx is None else ldx)
        Mp = _pad8(M)
        td = x.dtype
        alloc = torch.zeros if Mp != M else torch.empty
        dyT = ops.transpose(dy, alloc(N, Mp, dtype=td, device=self.dev), rows=M, cols=N, ldi=dy.stride(0) if lddy is None else lddy, ldo=Mp)
        xT = ops.transpose(x, alloc(K, Mp, dtype=td, device=self.dev), rows=M, cols=K, ldi=x.stride(0) if ldx is None else ldx, ldo=Mp)
        return ops.gemm(dyT, xT, out, M=N, N=K, K=Mp)

    def _lin_bwd(self, dy, x, L, wname, bname, *, need_dx=True, dx_dtype=None, dx_residual=None, dw_out=None, db_out=None, train=True):
        """dy = gradient w.r.t. the pre-activation output.  Records dW / db under the reference parameter names."""
        M, N = dy.shape[0], L.N
        if train and bname is not None and L.b is not None:
            ops.period_sum(dy, db_out if db_out is not None else self._g(bname, (N,)), rows=M, cols=N, ldx=dy.stride(0))
        if train and wname is not None:
            self._dw_gemm(dy, x, dw_out if dw_out is not None else self._g(wname, (N, L.K)), N=N, K=L.K)
        if not need_dx:
            return None
        dx = self._new(M, L.K, dtype=dx_dtype or dy.dtype)
        dyc = dy if dy.dtype == L.w.dtype else ops.cast(dy, self._new(M, N, dtype=L.w.dtype), rows=M, cols=N, ldi=dy.stride(0))
        return ops.gemm(dyc, self._wT(L), dx, residual=dx_residual)

    def _relu_bwd(self, dy, y):
        return ops.relu_bwd(dy, y, self._new(*y.shape, dtype=y.dtype), rows=y.shape[0], cols=y.shape[1])

    def _ln_bwd(self, dy, x, ln, wname, bname, *, residual=None, dx_dtype=None, train=True):
        dx = self._new(*x.shape, dtype=dx_dtype or x.dtype)
        dw = self._g(wname, (x.shape[1],)) if train else None
        db = self._g(bname, (x.shape[1],)) if train else None
        return ops.layernorm_bwd(dy, x, ln[0], residual=residual, eps=ln[2], dx=dx, dw=dw, db=db)

    # ---- attention backward into packed gradient buffers ------------------------------------------------
    def _attn_lse(self, act, B, H, Hkv, L, dh, drop=None):
        """fp32 [B, H, L] logsumexp buffer for a causal self-attention forward whose backward recomputes the probabilities from it
        (ops.attention_lse_bwd_ok: past 256 positions or GQA); None otherwise."""
        if not ops.attention_lse_bwd_ok(act, H=H, Hkv=Hkv, Tq=L, Tk=L, dh=dh, drop=drop):
            return None
        return torch.empty(B * H * L, dtype=torch.float32, device=self.dev)

    def _attn_bwd(self, q, k, v, do, *, B, H, Hkv, Tq, Tk, dh, qs, ks, vs, dos, dq, dqs, dk_out, dv_out, ld_kv, scale, causal=False,
                  key_mask=None, o=None, drop=None, lse=None):
        """dq is written in place (strides dqs); dk / dv are accumulated in fp32 and cast into dk_out / dv_out (row stride ld_kv)."""
        if ops.attention_bwd_owned_ok(q, H=H, Hkv=Hkv, Tq=Tq, Tk=Tk, dh=dh, o=o, causal=causal, lse=lse, drop=drop, strides=(*qs, *ks, *vs, *dos)):
            # the CTAs that own a key block sum its gradient over every query (and GQA head): dk / dv land directly in the packed
            # gradient buffer (no fp32 staging, no casts)
            kvs = (Tk * ld_kv, ld_kv)
            ops.attention_bwd_owned(q, k, v, do, dq, dk_out, dv_out, B=B, H=H, Tq=Tq, Tk=Tk, dh=dh, q_strides=qs, k_strides=ks, v_strides=vs,
                                    do_strides=dos, dq_strides=dqs, dk_strides=kvs, dv_strides=kvs, scale=scale, causal=causal,
                                    key_mask=key_mask, o=o, o_strides=dos, drop=drop, Hkv=Hkv, lse=lse)
            return
        wk = Hkv * dh
        dk = torch.zeros(B * Tk, wk, dtype=torch.float32, device=self.dev)
        dv = torch.zeros(B * Tk, wk, dtype=torch.float32, device=self.dev)
        ops.attention_bwd(q, k, v, do, dq, dk, dv, B=B, H=H, Hkv=Hkv, Tq=Tq, Tk=Tk, dh=dh, q_strides=qs, k_strides=ks, v_strides=vs,
                          do_strides=dos, dq_strides=dqs, dk_strides=(Tk * wk, wk), dv_strides=(Tk * wk, wk), scale=scale, causal=causal,
                          key_mask=key_mask, o=o, o_strides=dos, drop=drop)
        ops.cast(dk, dk_out, rows=B * Tk, cols=wk, ldo=ld_kv)
        ops.cast(dv, dv_out, rows=B * Tk, cols=wk, ldo=ld_kv)

    def _self_attn_fwd(self, x, T, B, mha, key_mask=None, drop=None):
        E, heads = mha["E"], mha["heads"]
        qkv = ops.gemm(x, mha["qkv"].w, self._new(B * T, 3 * E, dtype=x.dtype), bias=mha["qkv"].b)
        a = self._new(B * T, E, dtype=x.dtype)
        dh = E // heads
        ops.attention(qkv, qkv[:, E:], qkv[:, 2 * E:], a, B=B, H=heads, Hkv=heads, Tq=T, Tk=T, dh=dh, q_strides=(T * 3 * E, 3 * E),
                      k_strides=(T * 3 * E, 3 * E), v_strides=(T * 3 * E, 3 * E), o_strides=(T * E, E), scale=dh ** -0.5, key_mask=key_mask,
                      drop=drop)
        return qkv, a

    def _self_attn_bwd(self, da, qkv, x, T, B, mha, pre, key_mask=None, dx_residual=None, train=True, o=None, drop=None):
        """-> dx (gradient w.r.t. the block input through the qkv projection, + dx_residual)."""
        E, heads = mha["E"], mha["heads"]
        dh = E // heads
        dqkv = self._new(B * T, 3 * E, dtype=qkv.dtype)
        s3 = (T * 3 * E, 3 * E)
        self._attn_bwd(qkv, qkv[:, E:], qkv[:, 2 * E:], da, B=B, H=heads, Hkv=heads, Tq=T, Tk=T, dh=dh, qs=s3, ks=s3, vs=s3, dos=(T * E, E),
                       dq=dqkv, dqs=s3, dk_out=dqkv[:, E:], dv_out=dqkv[:, 2 * E:], ld_kv=3 * E, scale=dh ** -0.5, key_mask=key_mask, o=o,
                       drop=drop)
        return self._lin_bwd(dqkv, x, mha["qkv"], pre + "in_proj_weight", pre + "in_proj_bias", dx_residual=dx_residual, train=train)

    def _cross_attn_fwd(self, xq, Tq, mem, Tk, B, mha, drop=None):
        E, heads = mha["E"], mha["heads"]
        dh = E // heads
        q = ops.gemm(xq, mha["q"].w, self._new(B * Tq, E), bias=mha["q"].b)
        kv = ops.gemm(mem, mha["kv"].w, self._new(B * Tk, 2 * E), bias=mha["kv"].b)
        a = self._new(B * Tq, E)
        ops.attention(q, kv, kv[:, E:], a, B=B, H=heads, Hkv=heads, Tq=Tq, Tk=Tk, dh=dh, q_strides=(Tq * E, E), k_strides=(Tk * 2 * E, 2 * E),
                      v_strides=(Tk * 2 * E, 2 * E), o_strides=(Tq * E, E), scale=dh ** -0.5, drop=drop)
        return q, kv, a

    def _cross_attn_bwd(self, da, q, kv, xq, Tq, mem, Tk, B, mha, pre, *, need_dmem=True, dmem_residual=None, dxq_residual=None, train=True,
                        o=None, drop=None):
        E, heads = mha["E"], mha["heads"]
        dh = E // heads
        dq = self._new(B * Tq, E, dtype=q.dtype)
        dkv = self._new(B * Tk, 2 * E, dtype=kv.dtype)
        s2 = (Tk * 2 * E, 2 * E)
        self._attn_bwd(q, kv, kv[:, E:], da, B=B, H=heads, Hkv=heads, Tq=Tq, Tk=Tk, dh=dh, qs=(Tq * E, E), ks=s2, vs=s2, dos=(Tq * E, E),
                       dq=dq, dqs=(Tq * E, E), dk_out=dkv, dv_out=dkv[:, E:], ld_kv=2 * E, scale=dh ** -0.5, o=o, drop=drop)
        dw = db = None
        if train:
            dw, db = self._g(pre + "in_proj_weight", (3 * E, E)), self._g(pre + "in_proj_bias", (3 * E,))
        dxq = self._lin_bwd(dq, xq, mha["q"], "", "", dx_residual=dxq_residual, dw_out=None if dw is None else dw[:E],
                            db_out=None if db is None else db[:E], train=train)
        dmem = self._lin_bwd(dkv, mem, mha["kv"], "", "", need_dx=need_dmem, dx_residual=dmem_residual, dw_out=None if dw is None else dw[E:],
                             db_out=None if db is None else db[E:], train=train)
        return dxq, dmem

    # ---- post-norm transformer layers (torch nn.TransformerEncoderLayer / DecoderLayer) ------------------
    # torch: x = norm1(x + dropout1(self_attn(x)));  x = norm2(x + dropout2(linear2(dropout(relu(linear1(x))))))   (+ the attention
    # module's own dropout on the probabilities).  `mod` / `li` name the dropout sites (DropPlan); with no active site the residual
    # add stays fused in the GEMM epilogue.
    def _sub_out(self, a, lin, residual, drop, out_dtype=None):
        """residual + dropout(a . W^T + b)"""
        if drop is None:
            return ops.gemm(a, lin.w, self._new(a.shape[0], lin.N, dtype=out_dtype or residual.dtype), bias=lin.b, residual=residual)
        t = ops.gemm(a, lin.w, self._new(a.shape[0], lin.N, dtype=out_dtype or residual.dtype), bias=lin.b)
        return self._drop_res(t, drop, residual)

    def _enc_fwd(self, x, T, B, L, key_mask=None, sa_f32=None, mod=None, li=0):
        D = (lambda kind: self.drop(mod, li, kind)) if mod else (lambda kind: None)
        sa = sa_f32 if sa_f32 is not None else L["sa"]
        qkv, a = self._self_attn_fwd(x, T, B, sa, key_mask, drop=D("sa_attn"))
        y1 = self._sub_out(a, sa["out"], x, D("drop1"))
        x1 = self._ln_res(y1, L["n1"], out=self._new(*x.shape))
        h = ops.gemm(x1, L["l1"].w, self._new(x.shape[0], L["l1"].N), bias=L["l1"].b, act=ops.ACT_RELU)
        if D("ffn") is not None:
            self._drop_res(h, D("ffn"), None)
        y2 = self._sub_out(h, L["l2"], x1, D("drop2"), out_dtype=self.act)
        x2 = self._ln_res(y2, L["n2"])
        return x2, (x, qkv, a, y1, x1, h, y2, sa)

    def _enc_bwd(self, dx2, ctx, T, B, L, pre, key_mask=None, need_dx=True, train=True, mod=None, li=0):
        D = (lambda kind: self.drop(mod, li, kind)) if mod else (lambda kind: None)
        x, qkv, a, y1, x1, h, y2, sa = ctx
        dy2 = self._ln_bwd(dx2, y2, L["n2"], pre + "norm2.weight", pre + "norm2.bias", train=train)
        dh = self._lin_bwd(self._drop_grad(dy2, D("drop2")), h, L["l2"], pre + "linear2.weight", pre + "linear2.bias", train=train)
        if D("ffn") is not None:          # h = dropout(relu(z)): h > 0 only where the unit was kept, so relu_bwd on the dropped h gates both
            self._drop_res(dh, D("ffn"), None)
        dpre = self._relu_bwd(dh, h)
        dx1 = self._lin_bwd(dpre, x1, L["l1"], pre + "linear1.weight", pre + "linear1.bias", dx_residual=dy2, train=train)
        dy1 = self._ln_bwd(dx1, y1, L["n1"], pre + "norm1.weight", pre + "norm1.bias", train=train)
        da = self._lin_bwd(self._drop_grad(dy1, D("drop1")), a, sa["out"], pre + "self_attn.out_proj.weight", pre + "self_attn.out_proj.bias",
                           train=train)
        if not need_dx and not train:
            return None
        return self._self_attn_bwd(da, qkv, x, T, B, sa, pre + "self_attn.", key_mask, dx_residual=dy1, train=train, o=a, drop=D("sa_attn"))

    def _dec_fwd(self, t, Q, mem, Tv, B, L, li=0):
        D = lambda kind: self.drop("qdec", li, kind)     # noqa: E731
        qkv, a = self._self_attn_fwd(t, Q, B, L["sa"], drop=D("sa_attn"))
        y1 = self._sub_out(a, L["sa"]["out"], t, D("drop1"))
        t1 = self._ln_res(y1, L["n1"])
        q, kv, c = self._cross_attn_fwd(t1, Q, mem, Tv, B, L["ca"], drop=D("ca_attn"))
        y2 = self._sub_out(c, L["ca"]["out"], t1, D("drop2"))
        t2 = self._ln_res(y2, L["n2"])
        h = ops.gemm(t2, L["l1"].w, self._new(t.shape[0], L["l1"].N), bias=L["l1"].b, act=ops.ACT_RELU)
        if D("ffn") is not None:
            self._drop_res(h, D("ffn"), None)
        y3 = self._sub_out(h, L["l2"], t2, D("drop3"))
        return y3, (t, qkv, a, y1, t1, q, kv, c, y2, t2, h)

    def _dec_bwd(self, dy3, ctx, Q, mem, Tv, B, L, pre, dmem, li=0):
        """dy3: gradient w.r.t. y3 (the input of norm3).  Returns (dt, dmem accumulated)."""
        D = lambda kind: self.drop("qdec", li, kind)     # noqa: E731
        t, qkv, a, y1, t1, q, kv, c, y2, t2, h = ctx
        dh = self._lin_bwd(self._drop_grad(dy3, D("drop3")), h, L["l2"], pre + "linear2.weight", pre + "linear2.bias")
        if D("ffn") is not None:
            self._drop_res(dh, D("ffn"), None)
        dpre = self._relu_bwd(dh, h)
        dt2 = self._lin_bwd(dpre, t2, L["l1"], pre + "linear1.weight", pre + "linear1.bias", dx_residual=dy3)
        dy2 = self._ln_bwd(dt2, y2, L["n2"], pre + "norm2.weight", pre + "norm2.bias")
        dc = self._lin_bwd(self._drop_grad(dy2, D("drop2")), c, L["ca"]["out"], pre + "multihead_attn.out_proj.weight",
                           pre + "multihead_attn.out_proj.bias")
        dt1, dmem = self._cross_attn_bwd(dc, q, kv, t1, Q, mem, Tv, B, L["ca"], pre + "multihead_attn.", dmem_residual=dmem, dxq_residual=dy2, o=c,
                                         drop=D("ca_attn"))
        dy1 = self._ln_bwd(dt1, y1, L["n1"], pre + "norm1.weight", pre + "norm1.bias")
        da = self._lin_bwd(self._drop_grad(dy1, D("drop1")), a, L["sa"]["out"], pre + "self_attn.out_proj.weight", pre + "self_attn.out_proj.bias")
        dt = self._self_attn_bwd(da, qkv, t, Q, B, L["sa"], pre + "self_attn.", dx_residual=dy1, o=a, drop=D("sa_attn"))
        return dt, dmem

    # ---- lane polygon encoder (reference scripts/train.py:362-383) ----------------------------------------
    def _poly_fwd(self, polygon, lens):
        p = self.poly
        B, P, D = polygon.shape[0], polygon.shape[1], p["D"]
        x0 = self._new(B * P, D, dtype=torch.float32)
        kmask = torch.empty(B, P, dtype=torch.int32, device=self.dev)
        ops.poly_embed(polygon, lens, p["w"], p["b"], p["pos"], x0, kmask, B=B, P=P, D=D)
        x, ctxs = x0, []
        for i, L in enumerate(p["layers"]):
            x, c = self._enc_fwd(x, P, B, L, kmask, sa_f32=p["sa0_f32"] if i == 0 else None, mod="poly", li=i)
            ctxs.append(c)
        if not p["layers"] and x.dtype != self.act:
            x = ops.cast(x, self._new(B * P, D), rows=B * P, cols=D)
        emb = ops.masked_mean(x, lens, self._new(B, D, dtype=self.small), B=B, P=P, D=D)
        return emb, (polygon, lens, kmask, ctxs, x.dtype, B, P, D)

    def _poly_bwd(self, demb, ctx):
        polygon, lens, kmask, ctxs, xdt, B, P, D = ctx
        p = self.poly
        pre = "lane_polygon_encoder."
        dx = ops.masked_mean_bwd(demb, lens, self._new(B * P, D, dtype=xdt), B=B, P=P, D=D)
        for i in reversed(range(len(ctxs))):
            dx = self._enc_bwd(dx, ctxs[i], P, B, p["layers"][i], f"{pre}encoder.layers.{i}.", kmask, mod="poly", li=i)
        # x0[b,p,:] = W . pt + bias + pos[p]   (train.py:364-365)
        M = B * P
        ops.period_sum(dx, self._g(pre + "input_proj.bias", (D,)), rows=M, cols=D)
        ops.period_sum(dx, self._g(pre + "pos_embedding", (1, P, D)), rows=M, cols=D, period=P)
        dxf = dx if dx.dtype == torch.float32 else ops.cast(dx, self._new(M, D, dtype=torch.float32), rows=M, cols=D)
        self._dw_gemm(dxf, polygon.view(M, 2), self._g(pre + "input_proj.weight", (D, 2)), N=D, K=2)

    # ---- Q-Former + fused-sequence assembly (reference scripts/train.py:408-414, 520-528) -------------------
    def _qformer_fwd(self, vision, fused, L_total):
        q = self.qf
        B, Tv, Dv = vision.shape
        Hq, Q = q["Hq"], q["Q"]
        v = vision.reshape(B * Tv, Dv)
        if v.dtype != self.act:
            v = ops.cast(v, self._new(B * Tv, Dv), rows=B * Tv, cols=Dv)
        x = ops.gemm(v, q["vproj"].w, self._new(B * Tv, Hq), bias=q["vproj"].b)
        enc = []
        for i, L in enumerate(q["enc"]):
            x, c = self._enc_fwd(x, Tv, B, L, mod="qenc", li=i)
            enc.append(c)
        t = ops.cast(q["query"], self._new(B * Q, Hq), rows=B * Q, cols=Hq, in_row_mod=Q)
        dec = []
        for i, L in enumerate(q["dec"]):
            y3, c = self._dec_fwd(t, Q, x, Tv, B, L, li=i)
            t = self._ln_res(y3, L["n3"])
            dec.append((c, y3))
        if q["qproj"] is not None:
            ops.gemm(t, q["qproj"].w, fused, bias=q["qproj"].b, remap=(Q, L_total, 0), ldo=fused.shape[-1])
        else:
            ops.add_rowvec(t, q["vis_mod"], fused, rows=B * Q, cols=Hq, remap=(Q, L_total, 0))
        return (v, x, enc, dec, t, B, Tv, Q, Hq)

    def _qformer_bwd(self, dfused, ctx, L_total):
        v, x, enc, dec, t, B, Tv, Q, Hq = ctx
        q = self.qf
        H = dfused.shape[-1]
        dimg = ops.copy_rows(dfused, self._new(B * Q, H), rows=B * Q, cols=H, in_remap=(Q, L_total, 0))
        ops.period_sum(dimg, self._g("mllm.vision_modality_embedding", (1, 1, H)), rows=B * Q, cols=H)
        if q["qproj"] is not None:
            dt = self._lin_bwd(dimg, t, q["qproj"], "mllm.q_proj.weight", "mllm.q_proj.bias")
        else:
            dt = dimg
        pre = "mllm.qformer."
        dmem = None
        for i in reversed(range(len(dec))):
            c, y3 = dec[i]
            L = q["dec"][i]
            dy3 = self._ln_bwd(dt, y3, L["n3"], f"{pre}decoder.layers.{i}.norm3.weight", f"{pre}decoder.layers.{i}.norm3.bias")
            dt, dmem = self._dec_bwd(dy3, c, Q, x, Tv, B, L, f"{pre}decoder.layers.{i}.", dmem, li=i)
        ops.period_sum(dt, self._g(pre + "query_tokens", (Q, Hq)), rows=B * Q, cols=Hq, period=Q)
        if dmem is None:    # no decoder layers: the encoder output is unused
            return
        dx = dmem
        for i in reversed(range(len(enc))):
            dx = self._enc_bwd(dx, enc[i], Tv, B, q["enc"][i], f"{pre}encoder.layers.{i}.", mod="qenc", li=i)
        self._lin_bwd(dx, v, q["vproj"], pre + "vision_proj.weight", pre + "vision_proj.bias", need_dx=False)

    # ---- LoRA-Llama stack (HF:375-427 + peft lora.Linear) -----------------------------------------------------
    def _new_xs(self, M):
        m = self.llm
        Kx = m["H"] + m["kx"]
        return torch.zeros(M, Kx, dtype=self.act, device=self.dev) if m["kx"] != m["n_lora"] else self._new(M, Kx)

    # ---- GPT-2-arch backbone (HF modeling_gpt2.py GPT2Model / GPT2Block, reached through scripts/train.py:445-453) ---------------
    def _gpt2_fwd(self, fused, mask, B, L):
        """Engine._gpt2_forward with every activation a gradient needs kept: per block (x_in, [ln_1(x) | LoRA side columns], qkv, attention
        output, x_mid, ln_2(x_mid), c_fc pre-activation).  gelu_new runs as a pass of its own so the pre-activation survives."""
        m = self.llm
        H, nh, dh, I, kx = m["H"], m["nh"], m["dh"], m["I"], m["kx"]
        M, Kx = B * L, H + kx
        if L > m["wpe"].shape[0]:
            raise ops._lib.TcavpError(f"sequence length {L} exceeds the backbone's n_positions {m['wpe'].shape[0]}")
        pos = ops.cast(m["wpe"], self._new(M, H), rows=M, cols=H, in_row_mod=L)
        x = ops.axpby(fused.view(M, H), self._new(M, H), rows=M, cols=H, b=pos)
        if self.drop("llm", 0, "embd") is not None:          # GPT2Model.drop(inputs_embeds + position_embeds)
            self._drop_res(x, self.drop("llm", 0, "embd"), None)
        sq = (L * 3 * H, 3 * H)
        ctxs, xm = [], None
        for li, ly in enumerate(m["layers"]):
            if kx:      # ln_1(x) lands directly in the leading columns of the K-extended operand [ln_1(x) | LoRA side columns]
                xs = torch.zeros(M, Kx, dtype=self.act, device=self.dev) if kx != m["n_lora"] else self._new(M, Kx)
                ops.layernorm_strided(x, ly["ln1"][0], ly["ln1"][1], xs, rows=M, cols=H, eps=ly["ln1"][2], ldo=Kx)
                drops = self._lora_drops(li)
                if drops and "a_cat_s" in ly:
                    ops.lora_a_drop(xs, ly["a_cat_s"], xs[:, H:], drops, M=M, H=H, r=m["r"], ldx=Kx, ldo=Kx)
                elif drops:      # peft: lora_A(dropout(ln_1(x))) — masked copy (exact: x or 0), 1 / (1 - p) rides on the weight
                    xm = self._new(M, H) if xm is None else xm
                    ops.dropout(xs, xm, drops[0], rows=M, cols=H, ldi=Kx, ldo=H, scale=1.0)
                    ops.gemm(xm, ly["a_cat_d"], xs[:, H:], M=M, N=m["n_lora"], K=H, ldo=Kx)
                else:
                    ops.gemm(xs, ly["a_cat"], xs[:, H:], M=M, N=m["n_lora"], K=H, lda=Kx, ldo=Kx)
                qkv = ops.gemm(xs, ly["wqkv"], self._new(M, 3 * H), M=M, N=3 * H, K=Kx, lda=Kx, bias=ly["bqkv"])
            else:
                xs = ops.layernorm(x, ly["ln1"][0], ly["ln1"][1], self._new(M, H), eps=ly["ln1"][2])
                qkv = ops.gemm(xs, ly["wqkv"], self._new(M, 3 * H), bias=ly["bqkv"])
            attn = self._new(M, H)
            lse = self._attn_lse(qkv, B, nh, nh, L, dh, self.drop("llm", li, "attn"))
            ops.attention(qkv, qkv[:, H:], qkv[:, 2 * H:], attn, B=B, H=nh, Hkv=nh, Tq=L, Tk=L, dh=dh, q_strides=sq, k_strides=sq, v_strides=sq,
                          o_strides=(L * H, H), scale=dh ** -0.5, causal=True, key_mask=mask, drop=self.drop("llm", li, "attn"), lse=lse)
            x_mid = self._sub_out(attn, ly["proj"], x, self.drop("llm", li, "resid1"))                  # x + resid_dropout(c_proj(a))
            h2 = ops.layernorm(x_mid, ly["ln2"][0], ly["ln2"][1], self._new(M, H), eps=ly["ln2"][2])
            pre = ops.gemm(h2, ly["fc"].w, self._new(M, I), bias=ly["fc"].b)
            mid = ops.gelu_tanh(pre, self._new(M, I), rows=M, cols=I)
            x_out = self._sub_out(mid, ly["mproj"], x_mid, self.drop("llm", li, "resid2"))              # x + dropout(mlp.c_proj(.))
            ctxs.append((x, xs, qkv, attn, x_mid, pre, lse))
            x = x_out
        fh = ops.layernorm(x, m["norm"][0], m["norm"][1], self._new(M, H), eps=m["norm"][2])
        return fh, (ctxs, x, mask, None, B, L)

    def _gpt2_bwd(self, dfh, ctx):
        """Backward of _gpt2_fwd.  The base weights, biases and LayerNorms of the backbone are frozen (peft), so only dX flows through
        them; c_attn's LoRA pair gets dB = (alpha / r) dqkv^T (dropout(h) A^T) and dA = (d(h A^T))^T dropout(h)."""
        ctxs, x_last, mask, _, B, L = ctx
        m = self.llm
        H, nh, dh, I, kx, r = m["H"], m["nh"], m["dh"], m["I"], m["kx"], m["r"]
        M, Kx = B * L, H + kx
        sq = (L * 3 * H, 3 * H)
        # frozen LayerNorm: dx only, the residual-branch gradient added in the same pass
        lnb = lambda dy, x, ln, add=None: ops.layernorm_bwd_dx(dy, x, ln[0], self._new(M, H), rows=M, cols=H, eps=ln[2], add=add)   # noqa: E731
        dx = lnb(dfh, x_last, m["norm"])
        xm = None
        for i in reversed(range(len(ctxs))):
            x_in, xs, qkv, attn, x_mid, pre, lse = ctxs[i]
            ly = m["layers"][i]
            dmid = self._lin_bwd(self._drop_grad(dx, self.drop("llm", i, "resid2")), None, ly["mproj"], None, None, train=False)
            dpre = ops.gelu_tanh_bwd(dmid, pre, dmid, rows=M, cols=I)
            dh2 = self._lin_bwd(dpre, None, ly["fc"], None, None, train=False)
            dx_mid = lnb(dh2, x_mid, ly["ln2"], dx)
            dattn = self._lin_bwd(self._drop_grad(dx_mid, self.drop("llm", i, "resid1")), None, ly["proj"], None, None, train=False)
            dqkv = self._new(M, 3 * H)
            self._attn_bwd(qkv, qkv[:, H:], qkv[:, 2 * H:], dattn, B=B, H=nh, Hkv=nh, Tq=L, Tk=L, dh=dh, qs=sq, ks=sq, vs=sq, dos=(L * H, H),
                           dq=dqkv, dqs=sq, dk_out=dqkv[:, H:], dv_out=dqkv[:, 2 * H:], ld_kv=3 * H, scale=dh ** -0.5, causal=True, key_mask=mask,
                           o=attn, drop=self.drop("llm", i, "attn"), lse=lse)
            dh1 = ops.gemm(dqkv, ly["wqkvT"][:H], self._new(M, H))
            if kx:
                du = ops.gemm(dqkv, ly["wqkvT"][H:], self._new(M, kx))               # gradient w.r.t. the LoRA side columns (dropout(h) A^T)
                drops = self._lora_drops(i)
                fused = bool(drops) and "a_cat_s" in ly
                if drops and not fused:
                    xm = self._new(M, H) if xm is None else xm
                if self.tr_lora:
                    dext = torch.zeros(3 * H, kx, dtype=torch.float32, device=self.dev)
                    ops.skinny_dw(dqkv, xs[:, H:], dext, M=M, N=3 * H, J=kx, ldy=3 * H, ldz=Kx)
                    dAp = torch.zeros(H, kx, dtype=torch.float32, device=self.dev)
                    if fused:
                        ops.lora_da_drop(xs, du, dAp, drops, M=M, H=H, r=r, ldx=Kx, lddt=kx)
                        dAp *= drops[0].scale
                    elif drops:
                        ops.dropout(xs, xm, drops[0], rows=M, cols=H, ldi=Kx, ldo=H, scale=1.0)
                        ops.skinny_dw(xm, du, dAp, M=M, N=H, J=kx, ldy=H, ldz=kx)
                        dAp *= drops[0].scale
                    else:
                        ops.skinny_dw(xs, du, dAp, M=M, N=H, J=kx, ldy=Kx, ldz=kx)
                    ca = self.model.mllm.llama_wrapper.causal_lm().transformer.h[i].attn.c_attn
                    pre_n = f"{self.llm_prefix}{i}.attn.c_attn."
                    self.G[pre_n + "lora_B.default.weight"] = (dext[:, :r] * ca.scaling).contiguous()
                    self.G[pre_n + "lora_A.default.weight"] = dAp[:, :r].t().contiguous()
                if fused:        # dh1 += mask o (du . A / (1 - p)), one pass
                    ops.lora_dx_drop(du, ly["a_cat_s"], dh1, drops, M=M, H=H, r=r, lddt=kx, lddx=H)
                elif drops:
                    tmp = ops.gemm(du, ly["a_catT_d"], xm, M=M, N=H, K=kx)
                    ops.dropout(tmp, dh1, drops[0], rows=M, cols=H, scale=1.0, accumulate=True)
                else:
                    ops.gemm(du, ly["a_catT"], dh1, M=M, N=H, K=kx, residual=dh1)
            dx = lnb(dh1, x_in, ly["ln1"], dx_mid)
        if self.drop("llm", 0, "embd") is not None:
            self._drop_res(dx, self.drop("llm", 0, "embd"), None)
        return dx      # gradient w.r.t. the fused input embeddings (wpe is frozen: the position term adds nothing)

    def _llm_fwd(self, fused, mask, B, L):
        m = self.llm
        if m.get("arch") == "gpt2":
            return self._gpt2_fwd(fused, mask, B, L)
        if not m["fuse_rope"]:
            raise ops._lib.TcavpError("the fine-tune step needs head_dim % 32 == 0 (fused RoPE layout)")
        H, nh, nkv, dh, I, kx = m["H"], m["nh"], m["nkv"], m["dh"], m["I"], m["kx"]
        M, Kx = B * L, H + kx
        key = (L, dh, 1)
        if key not in self._rope:
            self._rope[key] = ops.rope_table(L, dh, m["theta"], self.dev, layout=1)
        table = self._rope[key]
        rope = (table, L, dh, (nh + nkv) * dh)
        nq, nk = nh * dh, nkv * dh
        nqkv = nq + 2 * nk
        xs = self._new_xs(M)
        ops.cast(fused.view(M, H), xs, rows=M, cols=H, ldi=H, ldo=Kx)
        ctxs = []
        xm = None
        for li, ly in enumerate(m["layers"]):
            rstd1 = ops.row_rstd(xs, torch.empty(M, dtype=torch.float32, device=self.dev), rows=M, cols=H, ldx=Kx, eps=m["eps"])
            drops = self._lora_drops(li)
            if kx and drops and "a_cat_s" in ly:
                ops.lora_a_drop(xs, ly["a_cat_s"], xs[:, H:], drops, M=M, H=H, r=m["r"], ldx=Kx, ldo=Kx)
            elif kx and drops:
                if xm is None:
                    xm = self._new(M, H)
                for ti, d in enumerate(drops):
                    ops.dropout(xs, xm, d, rows=M, cols=H, ldi=Kx, ldo=H, scale=1.0)
                    ops.gemm(xm, ly["a_cat_t"][ti], xs[:, H:], M=M, N=m["n_lora"], K=H, ldo=Kx, residual=None if ti == 0 else xs[:, H:], ldr=Kx)
            elif kx:
                ops.gemm(xs, ly["a_cat"], xs[:, H:], M=M, N=m["n_lora"], K=H, lda=Kx, ldo=Kx)
            qkv = ops.gemm(xs, ly["wqkv"], self._new(M, nqkv), M=M, N=nqkv, K=Kx, lda=Kx, rope=rope, row_scale=rstd1)
            attn = self._new(M, nq)
            lse = self._attn_lse(qkv, B, nh, nkv, L, dh)
            ops.attention(qkv, qkv[:, nq:], qkv[:, nq + nk:], attn, B=B, H=nh, Hkv=nkv, Tq=L, Tk=L, dh=dh, q_strides=(L * nqkv, nqkv),
                          k_strides=(L * nqkv, nqkv), v_strides=(L * nqkv, nqkv), o_strides=(L * nq, nq), scale=dh ** -0.5, causal=True,
                          key_mask=mask, lse=lse)
            xs2 = self._new_xs(M)
            ops.gemm(attn, ly["wo"], xs2, ldo=Kx, residual=xs, ldr=Kx)
            rstd2 = ops.row_rstd(xs2, torch.empty(M, dtype=torch.float32, device=self.dev), rows=M, cols=H, ldx=Kx, eps=m["eps"])
            if self.act == torch.bfloat16 and (2 * I) % 32 == 0:
                # one pass: the SwiGLU epilogue emits mid and stashes the raw gate/up accumulators for swiglu_bwd
                gu = self._new(M, 2 * I)
                mid = ops.gemm(xs2, ly["wgu"], self._new(M, I), M=M, K=H, lda=Kx, act=ops.ACT_SWIGLU, row_scale=rstd2, aux_out=gu)
            else:
                gu = ops.gemm(xs2, ly["wgu"], self._new(M, 2 * I), M=M, K=H, lda=Kx, row_scale=rstd2)
                mid = ops.swiglu(gu, self._new(M, I), rows=M, I=I)
            xs3 = self._new_xs(M)
            ops.gemm(mid, ly["wdown"], xs3, ldo=Kx, residual=xs2, ldr=Kx)
            ctxs.append((xs, rstd1, qkv, attn, xs2, rstd2, gu, mid, lse))
            xs = xs3
        fh = ops.rmsnorm(xs, m["norm"], self._new(M, H), eps=m["eps"], rows=M, cols=H, ldi=Kx)
        return fh, (ctxs, xs, mask, table, B, L)

    def _llm_bwd(self, dfh, ctx):
        if self.llm.get("arch") == "gpt2":
            return self._gpt2_bwd(dfh, ctx)
        ctxs, xs_last, mask, table, B, L = ctx
        m = self.llm
        H, nh, nkv, dh, I, kx, r = m["H"], m["nh"], m["nkv"], m["dh"], m["I"], m["kx"], m["r"]
        M, Kx = B * L, H + kx
        nq, nk = nh * dh, nkv * dh
        nqkv = nq + 2 * nk
        sq = (L * nqkv, nqkv)
        dx = ops.rmsnorm_bwd(dfh, xs_last, self._new(M, H), rows=M, cols=H, eps=m["eps"], w=m["norm"], ldx=Kx)
        xm = None
        wrap = self.model.mllm.llama_wrapper
        if m["fuse_rope"] and "qk_inv_perm" not in m:
            m["qk_inv_perm"] = torch.argsort(m["qk_perm"])
        inv_perm = m["qk_inv_perm"] if m["fuse_rope"] else None
        for i in reversed(range(len(ctxs))):
            xs, rstd1, qkv, attn, xs2, rstd2, gu, mid, lse = ctxs[i]
            ly = m["layers"][i]
            if self.act == torch.bfloat16 and I % 32 == 0:
                # d(mid) never leaves the tile: the down_proj^T GEMM's epilogue reads the stashed (gate, up) pairs and writes (d gate, d up)
                dgu = ops.gemm(dx, ly["wdownT"], self._new(M, 2 * I), act=ops.ACT_SWIGLU_BWD, aux_out=gu)
            else:
                dmid = ops.gemm(dx, ly["wdownT"], self._new(M, I))
                dgu = ops.swiglu_bwd(dmid, gu, self._new(M, 2 * I), rows=M, I=I)
            dn2 = ops.gemm(dgu, ly["wguT"], self._new(M, H))
            dx2 = ops.rmsnorm_bwd(dn2, xs2, self._new(M, H), rows=M, cols=H, eps=m["eps"], add=dx, ldx=Kx)
            dattn = ops.gemm(dx2, ly["woT"], self._new(M, nq))
            dqkv = self._new(M, nqkv)
            self._attn_bwd(qkv, qkv[:, nq:], qkv[:, nq + nk:], dattn, B=B, H=nh, Hkv=nkv, Tq=L, Tk=L, dh=dh, qs=sq, ks=sq, vs=sq, dos=(L * nq, nq),
                           dq=dqkv, dqs=sq, dk_out=dqkv[:, nq:], dv_out=dqkv[:, nq + nk:], ld_kv=nqkv, scale=dh ** -0.5, causal=True, key_mask=mask,
                           o=attn, lse=lse)
            ops.rope_adjacent_(dqkv, rows=M, L=L, ld=nqkv, cols=nq + nk, dh=dh, table=table, inverse=True)
            dxs = ops.gemm(dqkv, ly["wqkvT"], self._new(M, Kx))            # [dn1 | dTn]
            drops = self._lora_drops(i)
            fused = bool(drops) and "a_cat_s" in ly
            if drops and not fused and xm is None:
                xm = self._new(M, H)
            if kx and self.tr_lora:
                dext = torch.zeros(nqkv, kx, dtype=torch.float32, device=self.dev)
                ops.skinny_dw(dqkv, xs[:, H:], dext, M=M, N=nqkv, J=kx, ldy=nqkv, ldz=Kx, row_scale=rstd1)
                dAp = torch.zeros(H, kx, dtype=torch.float32, device=self.dev)
                if fused:      # dA'_t = s_t * sum_m rstd[m] (mask_t o x)[m, :]^T dTn_t[m, :], masks regenerated on the fragments
                    ops.lora_da_drop(xs, dxs[:, H:], dAp, drops, M=M, H=H, r=r, ldx=Kx, lddt=Kx, row_scale=rstd1)
                    dAp[:, :len(drops) * r] *= ly["lora_scales"][None, :]
                elif drops:    # ... or literally: one masked copy + one reduction per target
                    for ti, d in enumerate(drops):
                        ops.dropout(xs, xm, d, rows=M, cols=H, ldi=Kx, ldo=H, scale=1.0)
                        dAt = torch.zeros(H, kx, dtype=torch.float32, device=self.dev)
                        ops.skinny_dw(xm, dxs[:, H:], dAt, M=M, N=H, J=kx, ldy=H, ldz=Kx, row_scale=rstd1)
                        dAp[:, ti * r:(ti + 1) * r] = dAt[:, ti * r:(ti + 1) * r] * d.scale
                else:
                    ops.skinny_dw(xs, dxs[:, H:], dAp, M=M, N=H, J=kx, ldy=Kx, ldz=Kx, row_scale=rstd1)
                if inv_perm is not None:
                    dext = dext[inv_perm]
                layer = wrap.causal_lm().model.layers[i].self_attn
                for ti, name in enumerate(m["targets"]):
                    r0, r1 = m["rows"][name]
                    mod = getattr(layer, name)
                    pre = f"{self.llm_prefix}{i}.self_attn.{name}."
                    self.G[pre + "lora_B.default.weight"] = (dext[r0:r1, ti * r:(ti + 1) * r] * mod.scaling).contiguous()
                    self.G[pre + "lora_A.default.weight"] = (dAp[:, ti * r:(ti + 1) * r] * ly["ln1"][:, None]).t().contiguous()
            if kx and fused:    # dn1 += sum_t mask_t o (dTn_t . s_t A'_t), one pass
                ops.lora_dx_drop(dxs[:, H:], ly["a_cat_s"], dxs, drops, M=M, H=H, r=r, lddt=Kx, lddx=Kx)
            elif kx and drops:  # ... or per target: rank-r GEMM into a scratch buffer + masked accumulate
                for ti, d in enumerate(drops):
                    tmp = ops.gemm(dxs[:, H:], ly["a_catT_t"][ti], xm, M=M, N=H, K=kx, lda=Kx, ldo=H)
                    ops.dropout(tmp, dxs, d, rows=M, cols=H, ldi=H, ldo=Kx, scale=1.0, accumulate=True)
            elif kx:
                ops.gemm(dxs[:, H:], ly["a_catT"], dxs, M=M, N=H, K=kx, lda=Kx, ldo=Kx, residual=dxs, ldr=Kx)    # dn1 += dTn . A'
            dx = ops.rmsnorm_bwd(dxs, xs, self._new(M, H), rows=M, cols=H, eps=m["eps"], add=dx2, lddy=Kx, ldx=Kx)
        return dx      # gradient w.r.t. the fused input embeddings (M, H)

    # ---- temporal encoder (reference scripts/train.py:837-840, 674-686) ------------------------------------------
    def _ltsf_enc_fwd(self, x, B):
        lt, C, T, sm = self.lt, self.C, self.T_in, self.small
        xT = ops.transpose(x, self._new(B * T, 2, dtype=sm), rows=2, cols=T, batch=B, in_bstride=2 * T, out_bstride=2 * T)
        xp = ops.gemm(xT, lt["wt"], self._new(B * T, C, dtype=sm), bias=lt["bt"])
        e0 = ops.nlinear_decode(xp, lt["we"], lt["be_pos"], None, self._new(B * T, C, dtype=sm), B=B, C=C, T_in=T, T_out=T)
        # reference SelfAttentionBlock (train.py:674-686): res1 = x_norm + dropout1(mha(x_norm)); out = norm2(res1) + dropout2(ffn(norm2(res1)))
        D = lambda kind: self.drop("ltsf", 0, kind)     # noqa: E731
        xn = self._ln_res(e0, lt["n1"])
        qkv, a = self._self_attn_fwd(xn, T, B, lt["mha"], drop=D("sa_attn"))
        y = self._sub_out(a, lt["mha"]["out"], xn, D("drop1"), out_dtype=sm)
        r = self._ln_res(y, lt["n2"])
        h = ops.gemm(r, lt["f0"].w, self._new(B * T, lt["f0"].N, dtype=sm), bias=lt["f0"].b, act=ops.ACT_RELU)
        if D("ffn") is not None:
            self._drop_res(h, D("ffn"), None)
        enc = self._sub_out(h, lt["f3"], r, D("drop2"), out_dtype=sm)
        return enc, (xT, xp, e0, xn, qkv, a, y, r, h, B)

    def _ltsf_enc_bwd(self, denc, ctx):
        xT, xp, e0, xn, qkv, a, y, r, h, B = ctx
        lt, C, T = self.lt, self.C, self.T_in
        pre = "ltsf.attn_block."
        D = lambda kind: self.drop("ltsf", 0, kind)     # noqa: E731
        dh = self._lin_bwd(self._drop_grad(denc, D("drop2")), h, lt["f3"], pre + "ffn.3.weight", pre + "ffn.3.bias")
        if D("ffn") is not None:
            self._drop_res(dh, D("ffn"), None)
        dpre = self._relu_bwd(dh, h)
        dr = self._lin_bwd(dpre, r, lt["f0"], pre + "ffn.0.weight", pre + "ffn.0.bias", dx_residual=denc)
        dy = self._ln_bwd(dr, y, lt["n2"], pre + "norm2.weight", pre + "norm2.bias")
        da = self._lin_bwd(self._drop_grad(dy, D("drop1")), a, lt["mha"]["out"], pre + "mha.out_proj.weight", pre + "mha.out_proj.bias")
        dxn = self._self_attn_bwd(da, qkv, xn, T, B, lt["mha"], pre + "mha.", dx_residual=dy, o=a, drop=D("sa_attn"))
        de0 = self._ln_bwd(dxn, e0, lt["n1"], pre + "norm1.weight", pre + "norm1.bias")
        # e0 = NLinear(xp; we, be) + pos   (bias and positional table share the [T, C] gradient)
        gb = torch.zeros(T, C, dtype=torch.float32, device=self.dev)
        ops.period_sum(de0, gb, rows=B * T, cols=C, period=T)
        self.G["_enc_bias_tc"] = gb
        dxp = self._new(B * T, C, dtype=self.small)
        ops.nlinear_bwd(de0, B=B, C=C, T_in=T, T_out=T, x_in=xp, w=lt["we"], din=dxp, dw=self._g("_enc_w_tsc", (T, T, C)))
        wt_lin = _Lin.__new__(_Lin)
        wt_lin.w, wt_lin.b, wt_lin.N, wt_lin.K, wt_lin.wT = lt["wt"], lt["bt"], C, 2, None
        self._lin_bwd(dxp, xT, wt_lin, "_token_w", "ltsf.token_proj.bias", need_dx=False)

    # ---- NLinear decoder + cross-attention fusion + head (reference scripts/train.py:767-806, 941-962) -----------------
    def _ltsf_dec_fwd(self, enc, poly_emb, fh, x, B, L, y, norm_stat):
        lt, C, T, To, sm = self.lt, self.C, self.T_in, self.T_out, self.small
        H = self.llm["H"]
        adj = ops.gemm(poly_emb, lt["lane_fc"].w, self._new(B, To * C, dtype=sm), bias=lt["lane_fc"].b)
        dec0 = ops.nlinear_decode(enc, lt["wd"], lt["bd"], adj, self._new(B, To * C, dtype=sm), B=B, C=C, T_in=T, T_out=To)
        hp = None
        dec = dec0
        if lt["post"] is not None:
            p0, p3 = lt["post"]
            hp = ops.gemm(dec0, p0.w, self._new(B, p0.N, dtype=sm), bias=p0.b, act=ops.ACT_RELU)
            if self.drop("dec", 0, "post") is not None:                                   # post_mlp: Linear, ReLU, Dropout, Linear (train.py:745-750)
                self._drop_res(hp, self.drop("dec", 0, "post"), None)
            dec = ops.gemm(hp, p3.w, self._new(B, To * C, dtype=sm), bias=p3.b)
        dec_t = dec.view(B * To, C)
        dq = dec_t if self.act == sm else ops.cast(dec_t, self._new(B * To, C), rows=B * To, cols=C)
        q0 = ops.gemm(dq, lt["dec_proj"].w, self._new(B * To, H), bias=lt["dec_proj"].b)
        q, kv, a = self._cross_attn_fwd(q0, To, fh, L, B, lt["cross"], drop=self.drop("dec", 0, "cross_attn"))
        co = ops.gemm(a, lt["cross"]["out"].w, self._new(B * To, H), bias=lt["cross"]["out"].b)
        fused = ops.gemm(co, lt["dec_unproj"].w, self._new(B * To, C, dtype=sm), bias=lt["dec_unproj"].b, residual=dec_t)
        f = self._ln_res(fused, lt["fl_ln"])
        l1 = self._mk_lin(lt["fl_w1"], lt["fl_b1"])
        l2 = self._mk_lin(lt["fl_w2"], lt["fl_b2"])
        lo = self._mk_lin(lt["wo"], lt["bo"])
        h1 = ops.gemm(f, l1.w, self._new(B * To, C, dtype=sm), bias=l1.b, act=ops.ACT_RELU)
        f2 = ops.gemm(h1, l2.w, self._new(B * To, C, dtype=sm), bias=l2.b)
        o = ops.gemm(f2, lo.w, self._new(B * To, 2, dtype=sm), bias=lo.b)
        decoded = ops.head_assemble(o, x, torch.empty(B, 2, To, dtype=torch.float32, device=self.dev), B=B, T_in=T, T_out=To)
        metrics = per_scene = None
        if y is not None:
            metrics = torch.zeros(8, dtype=torch.float32, device=self.dev)
            per_scene = torch.empty(B, 2, dtype=torch.float32, device=self.dev)
            ops.traj_metrics(decoded, y, norm_stat, metrics, per_scene, B=B, T_out=To)
        ctx = (enc, poly_emb, fh, adj, dec0, hp, dec_t, dq, q0, q, kv, a, co, fused, f, l1, l2, lo, h1, f2, decoded, y, norm_stat, B, L)
        return dict(decoded=decoded, metrics=metrics, per_scene=per_scene), ctx

    @staticmethod
    def _mk_lin(w, b):
        l = _Lin.__new__(_Lin)
        l.w, l.b, l.wT = w, b, None
        l.N, l.K = w.shape
        return l

    def _ltsf_dec_bwd(self, gloss, ctx, need_dfh):
        (enc, poly_emb, fh, adj, dec0, hp, dec_t, dq, q0, q, kv, a, co, fused, f, l1, l2, lo, h1, f2, decoded, y, norm_stat, B, L) = ctx
        lt, C, T, To, sm = self.lt, self.C, self.T_in, self.T_out, self.small
        pre = "ltsf.decoder."
        d_o = ops.traj_loss_bwd(decoded, y, norm_stat, self._new(B * To, 2, dtype=sm), B=B, T_out=To, gscale=gloss)
        df2 = self._lin_bwd(d_o, f2, lo, pre + "out_proj.weight", pre + "out_proj.bias")
        dh1 = self._lin_bwd(df2, h1, l2, pre + "fusion_layer.3.weight", pre + "fusion_layer.3.bias")
        dpre = self._relu_bwd(dh1, h1)
        df = self._lin_bwd(dpre, f, l1, pre + "fusion_layer.1.weight", pre + "fusion_layer.1.bias")
        dfused = self._ln_bwd(df, fused, lt["fl_ln"], pre + "fusion_layer.0.weight", pre + "fusion_layer.0.bias")
        # fused = dec_t + dec_unproj(co)
        dco = self._lin_bwd(dfused, co, lt["dec_unproj"], pre + "dec_unproj.weight", pre + "dec_unproj.bias", dx_dtype=self.act)
        da = self._lin_bwd(dco, a, lt["cross"]["out"], pre + "cross_attn.out_proj.weight", pre + "cross_attn.out_proj.bias")
        dq0, dfh = self._cross_attn_bwd(da, q, kv, q0, To, fh, L, B, lt["cross"], pre + "cross_attn.", need_dmem=need_dfh,
                                        drop=self.drop("dec", 0, "cross_attn"))
        ddec_t = self._lin_bwd(dq0, dq, lt["dec_proj"], pre + "dec_proj.weight", pre + "dec_proj.bias", dx_dtype=sm, dx_residual=dfused)
        ddec = ddec_t.view(B, To * C)
        if lt["post"] is not None:
            p0, p3 = lt["post"]
            dhp = self._lin_bwd(ddec, hp, p3, "_post3_w", "_post3_b")
            if self.drop("dec", 0, "post") is not None:
                self._drop_res(dhp, self.drop("dec", 0, "post"), None)
            dpre = self._relu_bwd(dhp, hp)
            ddec0 = self._lin_bwd(dpre, dec0, p0, "_post0_w", pre + "post_mlp.0.bias")
        else:
            ddec0 = ddec
        # dec0 = NLinear(enc; wd, bd) + adj
        ops.period_sum(ddec0.view(B * To, C), self._g("_dec_bias_tc", (To, C)), rows=B * To, cols=C, period=To)
        denc = self._new(B * T, C, dtype=sm)
        ops.nlinear_bwd(ddec0, B=B, C=C, T_in=T, T_out=To, x_in=enc, w=lt["wd"], din=denc, dw=self._g("_dec_w_tsc", (To, T, C)))
        dpoly = self._lin_bwd(ddec0, poly_emb, lt["lane_fc"], "_lane_w", "_lane_b")
        return denc, dpoly, dfh

    # ---- whole step -----------------------------------------------------------------------------------------------
    @torch.no_grad()
    def train_forward(self, x, vision, polygon, poly_len, input_ids, attention_mask, y=None, norm_stat=None, keep=True):
        """`keep=False`: a stochastic pass that will not be differentiated (best-of-K candidates) — the activation stash is dropped."""
        dev = self.dev
        if dev.type != "cuda":
            raise ops._lib.TcavpError("the model must be on a CUDA device (there is no CPU fallback): model.to('cuda')")
        self._begin_pass()
        self.sync_params()
        x = self._dev_f32(x)
        B = x.shape[0]
        polygon = self._dev_f32(polygon)
        lens = poly_len if torch.is_tensor(poly_len) else torch.tensor(list(poly_len), dtype=torch.int32)
        lens = lens.to(device=dev, dtype=torch.int32)
        if y is not None and norm_stat is not None:
            y = self._dev_f32(y)
            norm_stat = self._dev_f32(norm_stat).view(B, 4)
        else:
            y = norm_stat = None
        poly_emb, c_poly = self._poly_fwd(polygon, lens)
        vision = vision.to(dev)
        if vision.dtype not in (torch.float32, torch.bfloat16):
            vision = vision.float()
        ids = input_ids.to(device=dev, dtype=torch.int64).contiguous()
        am = attention_mask.to(device=dev, dtype=torch.int64).contiguous()
        Q, H = self.qf["Q"], self.llm["H"]
        L = Q + ids.shape[1]
        fused = self._new(B, L, H)
        mask = torch.empty(B, L, dtype=torch.int32, device=dev)
        c_qf = self._qformer_fwd(vision.contiguous(), fused, L)
        ops.embed_text(ids, am, self.llm["embed"], self.text_mod, fused, mask, B=B, L_text=ids.shape[1], n_img=Q, H=H)
        fh, c_llm = self._llm_fwd(fused, mask, B, L)
        enc, c_enc = self._ltsf_enc_fwd(x, B)
        out, c_dec = self._ltsf_dec_fwd(enc, poly_emb, fh, x, B, L, y, norm_stat)
        if y is not None:
            out["loss"] = out["metrics"][4]
        if not keep:
            self._ctx = None
            return out
        # the stash travels with the result (model.py keeps it on the autograd node), so two forwards may be in flight before either
        # backward runs (gradient accumulation over micro-batches, two losses summed); `_ctx` is only the default of train_backward
        out["_ctx"] = self._ctx = (c_poly, c_qf, c_llm, c_enc, c_dec, B, L, Q, H, ids.shape[1], self.drop)
        return out

    @torch.no_grad()
    def train_backward(self, gloss=None, ctx=None):
        """Runs the backward pass of a train_forward (`ctx` = its out["_ctx"]; default: the last one); returns
        {reference parameter name: fp32 gradient}."""
        return self.train_backward_late(self.train_backward_early(gloss, ctx))

    @torch.no_grad()
    def train_backward_early(self, gloss=None, ctx=None):
        """First part of the backward pass: regression head, cross-attention fusion, NLinear decoder, temporal encoder and lane-polygon
        encoder.  Every gradient outside `mllm.*` is FINAL when this returns (state["early"]: name -> gradient), which is what lets a
        data-parallel step start their all-reduce while the decoder-stack backward (the bulk of the step) still runs
        (finetune.py: FineTuner; the reference gets the same overlap from DistributedDataParallel's buckets, train.py:1127-1132).
        Returns the state `train_backward_late` continues from."""
        if ctx is None:
            ctx = self._ctx
        if ctx is None:
            raise ops._lib.TcavpError("train_backward: no forward pass to differentiate (or its activations were already consumed)")
        c_poly, c_qf, c_llm, c_enc, c_dec, B, L, Q, H, L_text, self.drop = ctx        # the masks of THAT forward pass
        if ctx is self._ctx:
            self._ctx = None
        self.G = {}
        if gloss is not None:
            gloss = gloss.detach().to(device=self.dev, dtype=torch.float32).reshape(1).contiguous()
        denc, dpoly, dfh = self._ltsf_dec_bwd(gloss, c_dec, self.need_llm_bwd)
        if self.tr_ltsf:
            self._ltsf_enc_bwd(denc, c_enc)
        if self.tr_poly:
            self._poly_bwd(dpoly, c_poly)
        early = self._unpack_grads()
        return dict(early=early, dfh=dfh, ctx=ctx, drop=self.drop)

    @torch.no_grad()
    def train_backward_late(self, state):
        """Second part: LoRA-Llama stack, text-modality embedding and Q-Former (`mllm.*` gradients); returns all gradients."""
        c_poly, c_qf, c_llm, c_enc, c_dec, B, L, Q, H, L_text, _ = state["ctx"]
        self.drop = state["drop"]
        out = state["early"]
        self.G = {}
        if self.need_llm_bwd:
            dfused = self._llm_bwd(state["dfh"], c_llm)
            if self.tr_text:
                dtxt = ops.copy_rows(dfused, self._new(B * L_text, H), rows=B * L_text, cols=H, in_remap=(L_text, L, Q))
                ops.period_sum(dtxt, self._g("mllm.text_modality_embedding", (1, 1, H)), rows=B * L_text, cols=H)
            if self.tr_qf:
                self._qformer_bwd(dfused, c_qf, L)
        out.update({k: v for k, v in self.G.items() if not k.startswith("_")})
        return out

    # ---- stage 1: CausalLM objective on the fused sequence (reference scripts/check_generation.py:131-151, train.py:533-547) ---------
    @torch.no_grad()
    def lm_forward(self, vision, input_ids, attention_mask, labels, keep=True):
        """Token cross-entropy of LlamaForCausalLM.forward(inputs_embeds=[image tokens | text], labels=[-100 ... | labels]) (HF:487-491):
        position t predicts token t + 1, image positions and -100 labels are ignored, mean over the labelled positions.  Only the
        labelled rows go through lm_head (row chunks, fp32 logits, tcavp_ce_loss does loss + d(logits) in one kernel); the hidden-state
        gradient is formed right away, so the [rows, vocab] logits never outlive a chunk.  Returns {"loss", "n_tokens", "_ctx"}."""
        dev = self.dev
        if dev.type != "cuda":
            raise ops._lib.TcavpError("the model must be on a CUDA device (there is no CPU fallback): model.to('cuda')")
        self._begin_pass()
        self.sync_params()
        vision = vision.to(dev)
        if vision.dtype not in (torch.float32, torch.bfloat16):
            vision = vision.float()
        ids = input_ids.to(device=dev, dtype=torch.int64).contiguous()
        am = attention_mask.to(device=dev, dtype=torch.int64).contiguous()
        lab = labels.to(device=dev, dtype=torch.int64)
        B, Lt = ids.shape
        Q, H = self.qf["Q"], self.llm["H"]
        L = Q + Lt
        fused = self._new(B, L, H)
        mask = torch.empty(B, L, dtype=torch.int32, device=dev)
        c_qf = self._qformer_fwd(vision.contiguous(), fused, L)
        ops.embed_text(ids, am, self.llm["embed"], self.text_mod, fused, mask, B=B, L_text=Lt, n_img=Q, H=H)
        fh, c_llm = self._llm_fwd(fused, mask, B, L)
        # target of fused position t = fused_labels[t + 1]; fused_labels = [-100] * Q ++ labels
        tgt = torch.full((B, L), -100, dtype=torch.int64, device=dev)
        tgt[:, Q - 1:L - 1] = lab
        idx = (tgt.view(-1) != -100).nonzero().squeeze(1)                  # labelled rows (one host sync: their number sizes the chunks)
        R = int(idx.numel())
        loss_sum = torch.zeros(1, dtype=torch.float32, device=dev)
        dh = None
        if R:
            hc = fh.view(B * L, H).index_select(0, idx)
            t = tgt.view(-1).index_select(0, idx)
            lm = self.lm_head()                                             # [V, H], tied to the embedding table when the checkpoint ties them
            V = lm.shape[0]
            V8 = (V + 7) // 8 * 8                                           # contraction length of the gradient GEMM (16-byte rows)
            if keep:
                if self.llm.get("lm_headT") is None:                        # [H, V8]: d(hidden) = d(logits) . W through the same GEMM
                    wt = torch.zeros(H, V8, dtype=lm.dtype, device=dev)
                    wt[:, :V] = lm.t()
                    self.llm["lm_headT"] = wt
                dh = self._new(R, H)
            chunk = max(1, min(R, (256 << 20) // (V * 4)))                  # <= 256 MB of fp32 logits at a time
            for r0 in range(0, R, chunk):
                rc = min(chunk, R - r0)
                logits = ops.gemm(hc[r0:r0 + rc], lm, self._new(rc, V, dtype=torch.float32))
                g = (self._new(rc, V8) if V8 == V else torch.zeros(rc, V8, dtype=self.act, device=dev)) if keep else None
                ops.ce_loss(logits, t[r0:r0 + rc], loss_sum, g, scale=1.0 / R)
                if keep:
                    ops.gemm(g, self.llm["lm_headT"], dh[r0:r0 + rc])
        out = {"loss": (loss_sum / max(R, 1)).squeeze(0), "n_tokens": R}
        if keep:
            out["_ctx"] = (c_qf, c_llm, dh, idx, B, L, Q, H, Lt, self.drop)
        return out

    @torch.no_grad()
    def lm_backward(self, gloss, ctx):
        """Backward of lm_forward: d(loss)/d(final hidden) scattered to its rows, then the decoder-stack / text-modality / Q-Former backward
        of the fine-tune step.  Returns {reference parameter name: fp32 gradient} (mllm.* only: nothing else is on this path)."""
        c_qf, c_llm, dh, idx, B, L, Q, H, Lt, self.drop = ctx
        self.G = {}
        if not self.need_llm_bwd:
            return {}
        dfh = torch.zeros(B * L, H, dtype=self.act, device=self.dev)
        if dh is not None:
            if gloss is not None:
                dh = dh * gloss.detach().to(device=self.dev, dtype=dh.dtype).reshape(1)
            dfh.index_copy_(0, idx, dh)
        dfused = self._llm_bwd(dfh, c_llm)
        if self.tr_text:
            dtxt = ops.copy_rows(dfused, self._new(B * Lt, H), rows=B * Lt, cols=H, in_remap=(Lt, L, Q))
            ops.period_sum(dtxt, self._g("mllm.text_modality_embedding", (1, 1, H)), rows=B * Lt, cols=H)
        if self.tr_qf:
            self._qformer_bwd(dfused, c_qf, L)
        return {k: v for k, v in self.G.items() if not k.startswith("_")}

    def _unpack_grads(self):
        """Packed-layout gradients -> reference state_dict layout (inverse of the pack-time permutations)."""
        G, C, T, To = self.G, self.C, self.T_in, self.T_out
        d = self.model.ltsf.decoder
        out = {k: v for k, v in G.items() if not k.startswith("_")}
        if "_enc_w_tsc" in G:
            w = G["_enc_w_tsc"].permute(2, 0, 1).contiguous()          # (C, t, s)
            b = G["_enc_bias_tc"].t().contiguous()                     # (C, t)
            for c in range(C):
                out[f"ltsf.nlinear_encoder.encoder_linears.{c}.weight"] = w[c]
                out[f"ltsf.nlinear_encoder.encoder_linears.{c}.bias"] = b[c]
            out["ltsf.pos_encoding"] = b.unsqueeze(0).clone()          # (1, C, T)
            out["ltsf.token_proj.weight"] = G["_token_w"].unsqueeze(-1)
        if "_dec_w_tsc" in G:
            w = G["_dec_w_tsc"].permute(2, 0, 1).contiguous()          # (C, To, s)
            b = G["_dec_bias_tc"].t().contiguous()
            for c in range(C):
                out[f"ltsf.decoder.decoder_linears.{c}.weight"] = w[c]
                out[f"ltsf.decoder.decoder_linears.{c}.bias"] = b[c]
            perm = (torch.arange(C, device=self.dev)[None, :] * To + torch.arange(To, device=self.dev)[:, None]).reshape(-1)
            lw = torch.empty_like(G["_lane_w"])
            lw[perm] = G["_lane_w"]
            lb = torch.empty_like(G["_lane_b"])
            lb[perm] = G["_lane_b"]
            out["ltsf.decoder.lane_fc.weight"], out["ltsf.decoder.lane_fc.bias"] = lw, lb
            if d.use_post_mlp:
                w0 = torch.empty_like(G["_post0_w"])
                w0[:, perm] = G["_post0_w"]
                w3 = torch.empty_like(G["_post3_w"])
                w3[perm] = G["_post3_w"]
                b3 = torch.empty_like(G["_post3_b"])
                b3[perm] = G["_post3_b"]
                out["ltsf.decoder.post_mlp.0.weight"], out["ltsf.decoder.post_mlp.3.weight"] = w0, w3
                out["ltsf.decoder.post_mlp.3.bias"] = b3
        return out
