"""Forward engine: packs the reference-layout parameters into device buffers laid out for the kernels
(fused QKV with the LoRA K-extension, interleaved gate/up, channel-contiguous NLinear weights, (t,c)-ordered
lane_fc / post_mlp) and drives libtcavp.so over one CUDA stream.  No torch arithmetic on the data path."""
import os

import torch

from . import ops
from .config import rope_inv_freq

_ACT = {"bf16": torch.bfloat16, "fp32": torch.float32}


def _f32(t, dev):
    return t.detach().to(device=dev, dtype=torch.float32).contiguous()


class _Lin:
    """Packed linear: weight in the activation dtype ([N, K] row-major), bias in fp32."""
    __slots__ = ("w", "b", "N", "K", "wT", "w3")

    def __init__(self, w, b, act, dev):
        self.w = w.detach().to(device=dev, dtype=act).contiguous()
        self.b = None if b is None else _f32(b, dev)
        self.N, self.K = self.w.shape
        self.wT = None   # [K, N] copy used by the backward pass (train_engine.py)
        self.w3 = None   # [N, 3K] bf16 [hi | lo | hi] split of an fp32 weight (Engine._split_small)


class Engine:
    # fp32 ("small") layers of the temporal path run on the tensor cores through a bf16 hi/lo split in bf16 compute mode
    SPLIT_SMALL = True
    # fp8 serving mode (fp8=True): the Llama decoder projections that run on e4m3 operands.  A projection is listed where its e4m3 GEMM
    # plus the quantisation pass in front of it measured faster than its bf16 GEMM at both the cfg2 and the cfg3 shape on B200 (DESIGN §5,
    # profiles/fp8_cfg*_r01_all4.json).  o_proj is not: at cfg2 its quantisation pass costs more than the e4m3 GEMM saves
    # (2.34 + 0.91 ms against 2.61 ms per step), so it keeps its bf16 weight.
    FP8_PROJ = ("wqkv", "wgu", "wdown")

    def __init__(self, model, compute_dtype="bf16", merge_lora=False, fp8=False):
        p0 = next(model.ltsf.parameters())
        if fp8 and compute_dtype != "bf16":
            raise ValueError(f"the fp8 serving mode runs on the bf16 engine (compute_dtype={compute_dtype!r})")
        self.fp8 = bool(fp8)
        self.merge_lora = merge_lora
        self.dev = dev = p0.device   # packing works anywhere (host-side tests); forward() requires CUDA
        self.act = act = _ACT[compute_dtype]
        # The temporal encoder block and the NLinear decoder / lane_fc / post_mlp are a few MFLOP per scene: they always
        # run in exact fp32 (SIMT), which keeps the regression path's residuals at full precision in bf16 mode.
        self.small = torch.float32
        self.model_hp = dict(model.hparams)
        self.T_in, self.T_out, self.C = model.seq_len, model.out_len, model.d_model
        with torch.no_grad():
            self._pack_poly(model.lane_polygon_encoder)
            self._pack_qformer(model.mllm)
            self._pack_llm(model.mllm)
            self._pack_ltsf(model.ltsf)
        self._rope = {}

    # ---- packing ----------------------------------------------------------------------------------
    def _mha(self, m, dtype=None):
        E, dt = m.embed_dim, dtype or self.act
        return dict(qkv=_Lin(m.in_proj_weight, m.in_proj_bias, dt, self.dev),
                    q=_Lin(m.in_proj_weight[:E], m.in_proj_bias[:E], dt, self.dev),
                    kv=_Lin(m.in_proj_weight[E:], m.in_proj_bias[E:], dt, self.dev),
                    out=_Lin(m.out_proj.weight, m.out_proj.bias, dt, self.dev), E=E, heads=m.num_heads)

    def _ln(self, m):
        return (_f32(m.weight, self.dev), _f32(m.bias, self.dev), m.eps)

    def _split_small(self, *lins):
        """Packs [w_hi | w_lo | w_hi] (bf16) next to an fp32 weight: x3 = [x_hi | x_hi | x_lo] (tcavp_split_bf16x3) against it in ONE
        bf16 tensor-core GEMM gives x_hi w_hi + x_hi w_lo + x_lo w_hi = the fp32 product to ~2^-16 relative, fp32 accumulation."""
        if not (self.SPLIT_SMALL and self.act == torch.bfloat16 and not os.environ.get("TCAVP_NO_SPLIT_SMALL")):
            return
        for L in lins:
            if L is not None and L.w.dtype == torch.float32 and L.K % 8 == 0:
                hi = L.w.to(torch.bfloat16)
                lo = (L.w - hi.float()).to(torch.bfloat16)
                L.w3 = torch.cat([hi, lo, hi], dim=1).contiguous()

    def _gemm_small(self, x, L, out, **kw):
        """Linear map of the fp32 temporal path: split-bf16 tensor-core GEMM when packed (bf16 compute mode), exact FFMA otherwise."""
        if L.w3 is not None and x.dtype == torch.float32 and x.is_contiguous():
            M = x.shape[0]
            x3 = ops.split3(x, self._new(M, 3 * L.K, dtype=torch.bfloat16), rows=M, cols=L.K)
            return ops.gemm(x3, L.w3, out, bias=L.b, **kw)
        return ops.gemm(x, L.w, out, bias=L.b, **kw)

    def _enc_layer(self, l):
        return dict(sa=self._mha(l.self_attn), l1=_Lin(l.linear1.weight, l.linear1.bias, self.act, self.dev),
                    l2=_Lin(l.linear2.weight, l.linear2.bias, self.act, self.dev), n1=self._ln(l.norm1), n2=self._ln(l.norm2))

    def _dec_layer(self, l):
        d = self._enc_layer(l)
        d["ca"] = self._mha(l.multihead_attn)
        d["n3"] = self._ln(l.norm3)
        return d

    def _pack_poly(self, m):
        self.poly = dict(D=m.d_model, P=m.max_points, heads=m.nhead, w=_f32(m.input_proj.weight, self.dev),
                         b=_f32(m.input_proj.bias, self.dev), pos=_f32(m.pos_embedding[0], self.dev),
                         layers=[self._enc_layer(l) for l in m.encoder.layers])
        # The first layer sees raw pixel coordinates (|x| ~ 1e3, train.py:364): its attention logits are ~1e6 and the
        # softmax is argmax-like, so bf16 operands would change which key wins.  That one attention sub-block therefore
        # always runs in exact fp32; everything after the first LayerNorm is O(1) and uses the activation dtype.
        if len(m.encoder.layers) > 0:
            self.poly["sa0_f32"] = self._mha(m.encoder.layers[0].self_attn, torch.float32)

    def _pack_qformer(self, mllm):
        q = mllm.qformer
        self.qf = dict(Hq=q.hidden_size, Q=q.num_query_tokens, heads=q.nhead, vproj=_Lin(q.vision_proj.weight, q.vision_proj.bias, self.act, self.dev),
                       enc=[self._enc_layer(l) for l in q.encoder.layers], dec=[self._dec_layer(l) for l in q.decoder.layers],
                       query=q.query_tokens.detach().to(self.dev, self.act).contiguous())
        vis = _f32(mllm.vision_modality_embedding.reshape(-1), self.dev)
        if isinstance(mllm.q_proj, torch.nn.Linear):
            self.qf["qproj"] = _Lin(mllm.q_proj.weight, mllm.q_proj.bias.detach().float().to(self.dev) + vis, self.act, self.dev)
        else:
            self.qf["qproj"] = None
        self.qf["vis_mod"] = vis
        self.text_mod = _f32(mllm.text_modality_embedding.reshape(-1), self.dev)

    def _pack_gpt2(self, mllm):
        """HF GPT2LMHeadModel (what AutoModelForCausalLM gives the reference for a GPT-2 checkpoint, scripts/train.py:427-431) with peft's
        default LoRA target c_attn.  Conv1D weights are [in, out]: packed transposed to the [N, K] operand layout of tcavp_gemm; the
        LoRA pair rides as extra K columns of the fused QKV weight ([ln_1(x) | ln_1(x) A^T] . [W^T | (alpha / r) B]^T), as in the Llama path."""
        wrap = mllm.llama_wrapper
        c = wrap.config
        lm = wrap.causal_lm()
        tr = lm.transformer
        self._lm_head_param, self._embed_param = lm.lm_head.weight, tr.wte.weight
        act, dev = self.act, self.dev
        H, nh, I = c["hidden_size"], c["num_attention_heads"], c["intermediate_size"]
        merge = bool(wrap.use_lora and getattr(self, "merge_lora", False))
        r = self.model_hp["lora_r"] if (wrap.use_lora and not merge) else 0
        kx = ((r + 7) // 8) * 8
        self.llm = dict(arch="gpt2", H=H, nh=nh, nkv=nh, dh=H // nh, I=I, eps=c.get("layer_norm_epsilon", 1e-5), kx=kx, n_lora=r, r=r,
                        vocab=c["vocab_size"], targets=("c_attn",) if r else (), layers=[], fuse_rope=False,
                        embed=tr.wte.weight.detach().to(dev, act).contiguous(), wpe=tr.wpe.weight.detach().to(dev, act).contiguous(),
                        norm=self._ln(tr.ln_f))
        for blk in tr.h:
            ca = blk.attn.c_attn
            wqkv = torch.zeros(3 * H, H + kx, dtype=act, device=dev)
            a_cat = None
            if wrap.use_lora:
                base_w, base_b = ca.base_layer.weight.detach().to(dev).float(), ca.base_layer.bias
                A, Bm = ca.lora_A["default"].weight.detach().to(dev).float(), ca.lora_B["default"].weight.detach().to(dev).float()
                if merge:
                    wqkv[:, :H] = (base_w.t() + ca.scaling * (Bm @ A)).to(act)
                else:
                    wqkv[:, :H] = base_w.t().to(act)
                    wqkv[:, H:H + r] = (Bm * ca.scaling).to(act)
                    a_cat = torch.zeros(kx, H, dtype=act, device=dev)
                    a_cat[:r] = A.to(act)
            else:
                base_b = ca.bias
                wqkv[:, :H] = ca.weight.detach().to(dev).t().to(act)
            lin = lambda cv: _Lin(cv.weight.detach().t(), cv.bias, act, dev)          # noqa: E731  Conv1D -> [N, K]
            self.llm["layers"].append(dict(wqkv=wqkv, bqkv=_f32(base_b, dev), a_cat=a_cat, ln1=self._ln(blk.ln_1), ln2=self._ln(blk.ln_2),
                                           proj=lin(blk.attn.c_proj), fc=lin(blk.mlp.c_fc), mproj=lin(blk.mlp.c_proj)))

    def _gpt2_forward(self, fused, mask, B, L, kv_out=None):
        """HF GPT2Model over inputs_embeds: + wpe[0 .. L), pre-norm blocks (LayerNorm -> fused c_attn (+ LoRA) -> causal attention with the
        key-padding mask -> c_proj + residual; LayerNorm -> c_fc + gelu_new -> c_proj + residual), ln_f.  Every projection is a
        tcavp_gemm with its bias / activation / residual in the epilogue; the attention is the tcgen05 kernel of the Llama path (no RoPE)."""
        m = self.llm
        H, nh, dh, I, kx = m["H"], m["nh"], m["dh"], m["I"], m["kx"]
        M, Kx = B * L, H + kx
        if L > m["wpe"].shape[0]:
            raise ops._lib.TcavpError(f"sequence length {L} exceeds the backbone's n_positions {m['wpe'].shape[0]}")
        pos = ops.cast(m["wpe"], self._new(M, H), rows=M, cols=H, in_row_mod=L)          # position ids 0 .. L-1 in every scene
        x = ops.axpby(fused.view(M, H), self._new(M, H), rows=M, cols=H, b=pos)
        xs = torch.zeros(M, Kx, dtype=self.act, device=self.dev) if kx != m["n_lora"] else self._new(M, Kx)
        h = self._new(M, H)
        qkv, attn, mid = self._new(M, 3 * H), self._new(M, H), self._new(M, I)
        for ly in m["layers"]:
            if kx:      # ln_1(x) lands directly in the leading columns of the K-extended operand
                ops.layernorm_strided(x, ly["ln1"][0], ly["ln1"][1], xs, rows=M, cols=H, eps=ly["ln1"][2], ldo=Kx)
                ops.gemm(xs, ly["a_cat"], xs[:, H:], M=M, N=m["n_lora"], K=H, lda=Kx, ldo=Kx)
                ops.gemm(xs, ly["wqkv"], qkv, M=M, N=3 * H, K=Kx, lda=Kx, bias=ly["bqkv"])
            else:
                ops.layernorm(x, ly["ln1"][0], ly["ln1"][1], h, eps=ly["ln1"][2])
                ops.gemm(h, ly["wqkv"], qkv, bias=ly["bqkv"])
            if kv_out is not None:       # prefill of a KV-cache decode: keys / values of every layer kept ([B, capacity, 2H])
                cache = torch.empty(B, kv_out[1], 2 * H, dtype=self.act, device=self.dev)
                cache[:, :L].copy_(qkv.view(B, L, 3 * H)[:, :, H:])
                kv_out[0].append(cache)
            ops.attention(qkv, qkv[:, H:], qkv[:, 2 * H:], attn, B=B, H=nh, Hkv=nh, Tq=L, Tk=L, dh=dh, q_strides=(L * 3 * H, 3 * H),
                          k_strides=(L * 3 * H, 3 * H), v_strides=(L * 3 * H, 3 * H), o_strides=(L * H, H), scale=dh ** -0.5, causal=True,
                          key_mask=mask)
            ops.gemm(attn, ly["proj"].w, x, bias=ly["proj"].b, residual=x)
            ops.layernorm(x, ly["ln2"][0], ly["ln2"][1], h, eps=ly["ln2"][2])
            ops.gemm(h, ly["fc"].w, mid, bias=ly["fc"].b, act=ops.ACT_GELU_TANH)
            ops.gemm(mid, ly["mproj"].w, x, bias=ly["mproj"].b, residual=x)
        return ops.layernorm(x, m["norm"][0], m["norm"][1], self._new(M, H), eps=m["norm"][2])

    def _gpt2_decode_step(self, x_new, caches, t):
        """llm_decode_step for a GPT-2-arch backbone: + wpe[t], the block sequence of _gpt2_forward on one row per sequence, the new key /
        value appended to the cache, one query over positions 0..t."""
        m = self.llm
        H, nh, dh, I, kx = m["H"], m["nh"], m["dh"], m["I"], m["kx"]
        B, Kx = x_new.shape[0], H + kx
        cap = caches[0].shape[1]
        if t >= cap or t >= m["wpe"].shape[0]:
            raise ops._lib.TcavpError(f"decode position {t} is past the cache capacity {cap} / n_positions {m['wpe'].shape[0]}")
        pos = ops.cast(m["wpe"][t:t + 1], self._new(B, H), rows=B, cols=H, in_row_mod=1)
        x = ops.axpby(x_new.reshape(B, H), self._new(B, H), rows=B, cols=H, b=pos)
        xs = torch.zeros(B, Kx, dtype=self.act, device=self.dev)
        h, qkv, attn, mid = self._new(B, H), self._new(B, 3 * H), self._new(B, H), self._new(B, I)
        for ly, cache in zip(m["layers"], caches):
            if kx:
                ops.layernorm_strided(x, ly["ln1"][0], ly["ln1"][1], xs, rows=B, cols=H, eps=ly["ln1"][2], ldo=Kx)
                ops.gemm(xs, ly["a_cat"], xs[:, H:], M=B, N=m["n_lora"], K=H, lda=Kx, ldo=Kx)
                ops.gemm(xs, ly["wqkv"], qkv, M=B, N=3 * H, K=Kx, lda=Kx, bias=ly["bqkv"])
            else:
                ops.layernorm(x, ly["ln1"][0], ly["ln1"][1], h, eps=ly["ln1"][2])
                ops.gemm(h, ly["wqkv"], qkv, bias=ly["bqkv"])
            cache[:, t].copy_(qkv[:, H:])
            ops.attention(qkv, cache, cache[:, :, H:], attn, B=B, H=nh, Hkv=nh, Tq=1, Tk=t + 1, dh=dh, q_strides=(3 * H, 3 * H),
                          k_strides=(cap * 2 * H, 2 * H), v_strides=(cap * 2 * H, 2 * H), o_strides=(H, H), scale=dh ** -0.5)
            ops.gemm(attn, ly["proj"].w, x, bias=ly["proj"].b, residual=x)
            ops.layernorm(x, ly["ln2"][0], ly["ln2"][1], h, eps=ly["ln2"][2])
            ops.gemm(h, ly["fc"].w, mid, bias=ly["fc"].b, act=ops.ACT_GELU_TANH)
            ops.gemm(mid, ly["mproj"].w, x, bias=ly["mproj"].b, residual=x)
        return ops.layernorm(x, m["norm"][0], m["norm"][1], self._new(B, H), eps=m["norm"][2])

    def _pack_llm(self, mllm):
        wrap = mllm.llama_wrapper
        c = wrap.config
        if c.get("arch") == "gpt2":
            if self.fp8:
                raise NotImplementedError("the fp8 serving mode covers Llama-arch backbones (GPT-2's LayerNorm mean and bias need another fold)")
            return self._pack_gpt2(mllm)
        lm = wrap.causal_lm()
        self._lm_head_param, self._embed_param = lm.lm_head.weight, lm.model.embed_tokens.weight
        act, dev = self.act, self.dev
        H, nh, nkv, dh, I = c["hidden_size"], c["num_attention_heads"], c["num_key_value_heads"], c["head_dim"], c["intermediate_size"]
        # serve-time option (SURVEY.md §8f.3): W' = W + (alpha/r) B A merged at pack time — no side path, K stays H (always so in fp8 mode)
        merge = bool(wrap.use_lora and (getattr(self, "merge_lora", False) or self.fp8))
        lora_targets = tuple(wrap.llama_model.targets) if wrap.use_lora else ()
        targets = () if merge else lora_targets
        r = self.model_hp["lora_r"] if (wrap.use_lora and not merge) else 0
        n_t = len(targets)
        kx = ((n_t * r + 7) // 8) * 8            # LoRA side columns appended to K (multiple of 8 for TMA strides)
        self.llm = dict(H=H, nh=nh, nkv=nkv, dh=dh, I=I, eps=c.get("rms_norm_eps", 1e-6), theta=rope_inv_freq(c),
                        kx=kx, n_lora=n_t * r, vocab=c["vocab_size"], layers=[],
                        embed=lm.model.embed_tokens.weight.detach().to(dev, act).contiguous(), norm=_f32(lm.model.norm.weight, dev))
        nq, nk = nh * dh, nkv * dh
        # RoPE fusion: within every q / k head, move rotation partners (i, i + dh/2) to adjacent rows (2i, 2i+1) so the
        # GEMM epilogue can rotate in registers; q.k is invariant under the shared permutation, v keeps its order.
        self.llm["fuse_rope"] = dh % 32 == 0 and not os.environ.get("TCAVP_NO_FUSE_ROPE")
        hp = torch.stack([torch.arange(dh // 2), torch.arange(dh // 2) + dh // 2], dim=1).reshape(-1)
        qk_perm = torch.cat([h * dh + hp for h in range(nh + nkv)] + [torch.arange(nq + nk, nq + 2 * nk)]).to(dev)
        self.llm["qk_perm"] = qk_perm
        self.llm["targets"], self.llm["r"] = tuple(targets), r
        for layer in lm.model.layers:
            sa = layer.self_attn
            rows = {"q_proj": (0, nq), "k_proj": (nq, nq + nk), "v_proj": (nq + nk, nq + 2 * nk)}
            wqkv = torch.zeros(nq + 2 * nk, H + kx, dtype=act, device=dev)
            a_cat = torch.zeros(max(kx, 1), H, dtype=act, device=dev) if kx else None
            for name, (r0, r1) in rows.items():
                mod = getattr(sa, name)
                if name in targets:
                    ti = targets.index(name)
                    wqkv[r0:r1, :H] = mod.base_layer.weight.detach().to(dev, act)
                    wqkv[r0:r1, H + ti * r: H + (ti + 1) * r] = (mod.lora_B["default"].weight.detach().float() * mod.scaling).to(dev, act)
                    a_cat[ti * r:(ti + 1) * r] = mod.lora_A["default"].weight.detach().to(dev, act)
                elif merge and name in lora_targets:
                    w = mod.base_layer.weight.detach().to(dev).float()
                    w = w + mod.scaling * (mod.lora_B["default"].weight.detach().to(dev).float() @ mod.lora_A["default"].weight.detach().to(dev).float())
                    wqkv[r0:r1, :H] = w.to(act)
                else:
                    wqkv[r0:r1, :H] = mod.weight.detach().to(dev, act)
            if self.llm["fuse_rope"]:
                wqkv = wqkv[qk_perm].contiguous()
            # RMSNorm fusion: w * (x * rstd) . W^T == rstd * (x . (W diag(w))^T): the norm weight is folded into the weight
            # columns (fp32 product, rounded once), rstd is applied to the accumulators in the GEMM epilogue.  The LoRA side
            # product then has to be T' = x . (A diag(w))^T WITHOUT rstd, so that rstd * ([x | T'] . [W' | sB]^T) is exact.
            ln1 = layer.input_layernorm.weight.detach().float().to(dev)
            ln2 = layer.post_attention_layernorm.weight.detach().float().to(dev)
            wqkv[:, :H] = (wqkv[:, :H].float() * ln1[None, :]).to(act)
            if a_cat is not None:
                a_cat = (a_cat.float() * ln1[None, :]).to(act)
            gu = torch.empty(2 * I, H, dtype=act, device=dev)
            gu[0::2] = (layer.mlp.gate_proj.weight.detach().to(dev).float() * ln2[None, :]).to(act)
            gu[1::2] = (layer.mlp.up_proj.weight.detach().to(dev).float() * ln2[None, :]).to(act)
            self.llm["layers"].append(dict(
                wqkv=wqkv, a_cat=a_cat, ln1=ln1, wo=sa.o_proj.weight.detach().to(dev, act).contiguous(), wgu=gu,
                wdown=layer.mlp.down_proj.weight.detach().to(dev, act).contiguous()))
            if self.fp8:
                self._pack_fp8(self.llm["layers"][-1], layer, lora_targets, qk_perm if self.llm["fuse_rope"] else None, ln1, ln2)

    def _pack_fp8(self, ly, layer, lora_targets, qk_perm, ln1, ln2):
        """Replaces the bf16 weights of the FP8_PROJ projections of one packed layer by e4m3 weights with per-output-channel scales:
        s_w[n] = amax(W'[n, :]) / 448, Wq = e4m3(W' / s_w) (zero rows: s_w = 0, Wq = 0).  W' is the fp32 weight the bf16 pack rounds
        once: LoRA merged, RMSNorm weight folded into the columns, q / k rows RoPE-permuted, gate / up interleaved — here rounded once,
        from fp32 straight to e4m3."""
        dev = self.dev
        sa, mlp = layer.self_attn, layer.mlp

        def w32(mod, name):
            if name in lora_targets:
                A, B = mod.lora_A["default"].weight.detach().to(dev).float(), mod.lora_B["default"].weight.detach().to(dev).float()
                return mod.base_layer.weight.detach().to(dev).float() + mod.scaling * (B @ A)
            return mod.weight.detach().to(dev).float()
        full = {}
        if "wqkv" in self.FP8_PROJ:
            w = torch.cat([w32(sa.q_proj, "q_proj"), w32(sa.k_proj, "k_proj"), w32(sa.v_proj, "v_proj")])
            full["wqkv"] = (w if qk_perm is None else w[qk_perm]) * ln1[None, :]
        if "wo" in self.FP8_PROJ:
            full["wo"] = w32(sa.o_proj, "o_proj")
        if "wgu" in self.FP8_PROJ:
            g, u = mlp.gate_proj.weight.detach().to(dev).float() * ln2[None, :], mlp.up_proj.weight.detach().to(dev).float() * ln2[None, :]
            full["wgu"] = torch.stack([g, u], dim=1).reshape(2 * g.shape[0], g.shape[1])
        if "wdown" in self.FP8_PROJ:
            full["wdown"] = mlp.down_proj.weight.detach().to(dev).float()
        for name, w in full.items():
            s = w.abs().amax(dim=1) / 448.0
            q = torch.where(s[:, None] > 0, w / torch.where(s > 0, s, 1.0)[:, None], 0.0)
            ly[name], ly["s_" + name] = q.to(torch.float8_e4m3fn).contiguous(), s.contiguous()

    def _proj(self, ly, name, a, out, *, rms=False, **kw):
        """One Llama decoder projection of the fp8 engine.  An e4m3 weight takes a per-row quantised copy of `a` (tcavp_quant_e4m3_rows,
        with LlamaRMSNorm's factor folded into the row factor when `rms`); a projection left in bf16 takes `a` itself with the RMSNorm
        factor from tcavp_row_rstd."""
        w, rows, cols, eps = ly[name], a.shape[0], a.shape[1], self.llm["eps"]
        if w.dtype == torch.float8_e4m3fn:
            aq, f = ops.quant_e4m3_rows(a, self._new(rows, cols, dtype=torch.float8_e4m3fn), self._new(rows, dtype=torch.float32),
                                        rms_eps=eps if rms else None)
            return ops.gemm(aq, w, out, row_scale=f, col_scale=ly["s_" + name], **kw)
        if rms:
            kw["row_scale"] = ops.row_rstd(a, self._new(rows, dtype=torch.float32), rows=rows, cols=cols, ldx=a.stride(0), eps=eps)
        return ops.gemm(a, w, out, **kw)

    def _pack_ltsf(self, lt):
        act, dev, small = self.act, self.dev, self.small
        C, T, To = self.C, self.T_in, self.T_out
        d = lt.decoder
        we = torch.stack([l.weight.detach() for l in lt.nlinear_encoder.encoder_linears]).float()   # (C, t, s)
        be = torch.stack([l.bias.detach() for l in lt.nlinear_encoder.encoder_linears]).float()     # (C, t)
        wd = torch.stack([l.weight.detach() for l in d.decoder_linears]).float()                    # (C, To, s)
        bd = torch.stack([l.bias.detach() for l in d.decoder_linears]).float()
        # (c,t)-flat -> (t,c)-flat permutation of the 64*T_out feature axis (lane_fc rows, post_mlp.0 cols, post_mlp.3 rows)
        pdev = d.lane_fc.weight.device
        if getattr(self, "_tc_perm", None) is None or self._tc_perm.device != pdev:     # built once: re-packing must stay capturable
            self._tc_perm = (torch.arange(C)[None, :] * To + torch.arange(To)[:, None]).reshape(-1).to(pdev)
        perm = self._tc_perm
        self.lt = dict(
            wt=_f32(lt.token_proj.weight[:, :, 0], dev), bt=_f32(lt.token_proj.bias, dev),
            we=we.permute(1, 2, 0).contiguous().to(dev), be=be.t().contiguous().to(dev),
            pos=_f32(lt.pos_encoding[0].t(), dev),
            n1=self._ln(lt.attn_block.norm1), n2=self._ln(lt.attn_block.norm2), mha=self._mha(lt.attn_block.mha, small),
            f0=_Lin(lt.attn_block.ffn[0].weight, lt.attn_block.ffn[0].bias, small, dev),
            f3=_Lin(lt.attn_block.ffn[3].weight, lt.attn_block.ffn[3].bias, small, dev),
            wd=wd.permute(1, 2, 0).contiguous().to(dev), bd=bd.t().contiguous().to(dev),
            lane_fc=_Lin(d.lane_fc.weight[perm], d.lane_fc.bias[perm], small, dev),
            dec_proj=_Lin(d.dec_proj.weight, d.dec_proj.bias, act, dev), dec_unproj=_Lin(d.dec_unproj.weight, d.dec_unproj.bias, act, dev),
            cross=self._mha(d.cross_attn),
            fl_ln=self._ln(d.fusion_layer[0]), fl_w1=_f32(d.fusion_layer[1].weight, dev), fl_b1=_f32(d.fusion_layer[1].bias, dev),
            fl_w2=_f32(d.fusion_layer[3].weight, dev), fl_b2=_f32(d.fusion_layer[3].bias, dev),
            wo=_f32(d.out_proj.weight, dev), bo=_f32(d.out_proj.bias, dev), post=None)
        if d.use_post_mlp:
            self.lt["post"] = (_Lin(d.post_mlp[0].weight[:, perm], d.post_mlp[0].bias, small, dev),
                               _Lin(d.post_mlp[3].weight[perm], d.post_mlp[3].bias[perm], small, dev))
        self._split_small(self.lt["mha"]["qkv"], self.lt["mha"]["out"], self.lt["f0"], self.lt["f3"], self.lt["lane_fc"],
                          *(self.lt["post"] or ()))
        self._absorb_cross(d.cross_attn)

    def _absorb_cross(self, mha):
        """Few queries (T_out) against many keys (L) in the fusion cross-attention (train.py:793-798): instead of projecting all L
        positions to K and V, the projections are absorbed into the query / output side —
            scores_h = Q_h K_h^T = (Q_h Wk_h) X^T            (the key bias is constant along the softmax axis and drops out)
            out_h    = P_h V_h   = (P_h X) Wv_h^T + bv_h      (rows of P sum to 1)
        so attention runs with keys = values = X (the backbone output, read in place, one shared 'KV head' of width H) and the two
        small projections fold into q_proj / out_proj:  Q' = q (Wk_h^T Wq_h)^T + bq_h Wk_h,  co = Z [Wo_h Wv_h]^T + (Wo bv + bo).
        Removes the [B L, 2H] K/V projection (the largest GEMM of the fusion block) and its round trip through HBM.  Exact algebra;
        used in bf16 compute mode (the fp32 parity mode keeps the reference's operation order)."""
        self.lt["absorb"] = None
        if not (self.SPLIT_SMALL and self.act == torch.bfloat16 and not os.environ.get("TCAVP_NO_ABSORB")):
            return
        E, heads = mha.embed_dim, mha.num_heads
        dh = E // heads
        if E % 64 or self.T_out > 64:
            return
        W = mha.in_proj_weight.detach().to(self.dev).float()
        bvec = mha.in_proj_bias.detach().to(self.dev).float()
        Wq, Wk, Wv = W[:E], W[E:2 * E], W[2 * E:]
        bq, bv = bvec[:E], bvec[2 * E:]
        Wo, bo = mha.out_proj.weight.detach().to(self.dev).float(), mha.out_proj.bias.detach().to(self.dev).float()
        mq, cq, mo = [], [], []
        for h in range(heads):
            sl = slice(h * dh, (h + 1) * dh)
            mq.append(Wk[sl].t() @ Wq[sl])            # [E, E]:  Q'_h = q . (Wk_h^T Wq_h)^T
            cq.append(bq[sl] @ Wk[sl])                # [E]
            mo.append(Wo[:, sl] @ Wv[sl])             # [E, E]:  co += Z_h . (Wo_h Wv_h)^T
        self.lt["absorb"] = dict(mq=torch.cat(mq, 0).to(self.act).contiguous(), cq=torch.cat(cq, 0).contiguous(),
                                 mo=torch.cat(mo, 1).to(self.act).contiguous(), co=(Wo @ bv + bo).contiguous(), E=E, heads=heads, dh=dh)

    # ---- building blocks --------------------------------------------------------------------------
    def _new(self, *shape, dtype=None):
        return torch.empty(*shape, dtype=dtype or self.act, device=self.dev)

    def _self_attention(self, x, rows_per_b, B, mha, key_mask=None):
        """x: (B*T, E) -> attention output (B*T, E) (before out_proj)."""
        E, heads = mha["E"], mha["heads"]
        T = rows_per_b
        qkv = self._gemm_small(x, mha["qkv"], self._new(B * T, 3 * E, dtype=x.dtype))
        out = self._new(B * T, E, dtype=x.dtype)
        dh = E // heads
        ops.attention(qkv, qkv[:, E:], qkv[:, 2 * E:], out, B=B, H=heads, Hkv=heads, Tq=T, Tk=T, dh=dh,
                      q_strides=(T * 3 * E, 3 * E), k_strides=(T * 3 * E, 3 * E), v_strides=(T * 3 * E, 3 * E),
                      o_strides=(T * E, E), scale=dh ** -0.5, key_mask=key_mask)
        return out

    def _cross_attention(self, xq, Tq, mem, Tk, B, mha):
        E, heads = mha["E"], mha["heads"]
        dh = E // heads
        q = ops.gemm(xq, mha["q"].w, self._new(B * Tq, E), bias=mha["q"].b)
        kv = ops.gemm(mem, mha["kv"].w, self._new(B * Tk, 2 * E), bias=mha["kv"].b)
        out = self._new(B * Tq, E)
        ops.attention(q, kv, kv[:, E:], out, B=B, H=heads, Hkv=heads, Tq=Tq, Tk=Tk, dh=dh, q_strides=(Tq * E, E),
                      k_strides=(Tk * 2 * E, 2 * E), v_strides=(Tk * 2 * E, 2 * E), o_strides=(Tq * E, E), scale=dh ** -0.5)
        return out

    def _ln_res(self, y, ln, out=None, **kw):
        return ops.layernorm(y, ln[0], ln[1], self._new(*y.shape, dtype=y.dtype) if out is None else out, eps=ln[2], **kw)

    def _encoder_layer(self, x, T, B, L, key_mask=None, sa_f32=None):
        """torch: nn.TransformerEncoderLayer (post-norm, ReLU).  `sa_f32`: run the attention sub-block on an fp32 input in
        exact fp32 and hand the LayerNorm output over in the activation dtype."""
        sa = sa_f32 if sa_f32 is not None else L["sa"]
        a = self._self_attention(x, T, B, sa, key_mask)
        y = ops.gemm(a, sa["out"].w, self._new(*x.shape, dtype=x.dtype), bias=sa["out"].b, residual=x)
        x = self._ln_res(y, L["n1"], out=self._new(*x.shape))
        if (x.dtype == torch.bfloat16 and x.shape[1] == 64 and L["l1"].N % 128 == 0 and L["l1"].N <= 8192 and L["l1"].b is not None
                and L["l2"].b is not None and not os.environ.get("TCAVP_NO_FFN_FUSED")):
            # d_model 64 (lane-polygon encoder): both linears, the residual and LayerNorm 2 in one tcgen05 kernel, hidden activation in TMEM
            return ops.ffn64_ln(x, L["l1"].w, L["l1"].b, L["l2"].w, L["l2"].b, L["n2"][0], L["n2"][1], self._new(*x.shape), eps=L["n2"][2])
        h = ops.gemm(x, L["l1"].w, self._new(x.shape[0], L["l1"].N), bias=L["l1"].b, act=ops.ACT_RELU)
        y = ops.gemm(h, L["l2"].w, self._new(*x.shape), bias=L["l2"].b, residual=x)
        return self._ln_res(y, L["n2"])

    # ---- sub-models ---------------------------------------------------------------------------------
    def poly_forward(self, polygon, lens, max_len=None):
        """reference scripts/train.py:362-383 -> (B, D) fp32.  `max_len` (host-known upper bound of lane_polygon_len): rows past the
        longest polygon are pure padding — masked as keys, skipped by the masked mean — so the encoder runs on the first
        round_up(max_len, 16) points only."""
        p = self.poly
        if max_len is not None:
            Pp = max(16, (int(max_len) + 15) // 16 * 16)
            if Pp < polygon.shape[1]:
                polygon = polygon[:, :Pp].contiguous()
        B, P, D = polygon.shape[0], polygon.shape[1], p["D"]
        x = self._new(B * P, D, dtype=torch.float32)
        kmask = torch.empty(B, P, dtype=torch.int32, device=self.dev)
        ops.poly_embed(polygon, lens, p["w"], p["b"], p["pos"], x, kmask, B=B, P=P, D=D)
        for i, L in enumerate(p["layers"]):
            x = self._encoder_layer(x, P, B, L, kmask, sa_f32=p["sa0_f32"] if i == 0 else None)
        if not p["layers"] and x.dtype != self.act:
            x = ops.cast(x, self._new(B * P, D), rows=B * P, cols=D)
        return ops.masked_mean(x, lens, self._new(B, D, dtype=self.small), B=B, P=P, D=D)

    def qformer_into(self, vision, fused, L_total):
        """reference scripts/train.py:408-414, 520-522: writes image tokens (+vision modality) into fused[:, :Q]."""
        q = self.qf
        B, Tv, Dv = vision.shape
        Hq, Q = q["Hq"], q["Q"]
        v = vision.reshape(B * Tv, Dv)
        if v.dtype != self.act:
            v = ops.cast(v, self._new(B * Tv, Dv), rows=B * Tv, cols=Dv)
        x = ops.gemm(v, q["vproj"].w, self._new(B * Tv, Hq), bias=q["vproj"].b)
        for L in q["enc"]:
            x = self._encoder_layer(x, Tv, B, L)
        t = ops.cast(q["query"], self._new(B * Q, Hq), rows=B * Q, cols=Hq, in_row_mod=Q)
        n = len(q["dec"])
        for i, L in enumerate(q["dec"]):
            a = self._self_attention(t, Q, B, L["sa"])
            y = ops.gemm(a, L["sa"]["out"].w, self._new(B * Q, Hq), bias=L["sa"]["out"].b, residual=t)
            t = self._ln_res(y, L["n1"])
            a = self._cross_attention(t, Q, x, Tv, B, L["ca"])
            y = ops.gemm(a, L["ca"]["out"].w, self._new(B * Q, Hq), bias=L["ca"]["out"].b, residual=t)
            t = self._ln_res(y, L["n2"])
            h = ops.gemm(t, L["l1"].w, self._new(B * Q, L["l1"].N), bias=L["l1"].b, act=ops.ACT_RELU)
            y = ops.gemm(h, L["l2"].w, self._new(B * Q, Hq), bias=L["l2"].b, residual=t)
            if i == n - 1 and q["qproj"] is None:
                # Identity q_proj (H == 768): the last LayerNorm scatters straight into the fused buffer
                self._ln_res(y, L["n3"], out=fused, remap=(Q, L_total, 0), rowvec=q["vis_mod"])
                return
            t = self._ln_res(y, L["n3"])
        if q["qproj"] is not None:
            ops.gemm(t, q["qproj"].w, fused, bias=q["qproj"].b, remap=(Q, L_total, 0), ldo=fused.shape[-1])
        else:   # zero decoder layers
            ops.add_rowvec(t, q["vis_mod"], fused, rows=B * Q, cols=Hq, remap=(Q, L_total, 0))

    def llm_forward(self, fused, mask, B, L, kv_out=None):
        """HF:375-427 LlamaModel over inputs_embeds with LoRA on q/k/v (in place on `fused`); returns the
        post-final-norm hidden states (= hidden_states[-1], reference scripts/train.py:553).
        `kv_out` = (list, capacity): the prefill of a KV-cache decode — every layer's rotated keys and values are also stored in a
        [B, capacity, 2 * n_kv * head_dim] cache appended to the list (generate.py; `llm_decode_step` continues from them)."""
        m = self.llm
        if m.get("arch") == "gpt2":
            return self._gpt2_forward(fused, mask, B, L, kv_out)
        H, nh, nkv, dh, I, kx = m["H"], m["nh"], m["nkv"], m["dh"], m["I"], m["kx"]
        M = B * L
        key = (L, dh, 1 if m["fuse_rope"] else 0)
        if key not in self._rope:
            self._rope[key] = ops.rope_table(L, dh, m["theta"], self.dev, layout=key[2])
        table = self._rope[key]
        Kx = H + kx
        # residual stream in K-extended rows: columns [0,H) hold x, columns [H,H+kx) receive the LoRA side product
        xs = torch.zeros(M, Kx, dtype=self.act, device=self.dev) if kx != m["n_lora"] else self._new(M, Kx)
        ops.cast(fused.view(M, H), xs, rows=M, cols=H, ldi=H, ldo=Kx)
        x = xs[:, :H]
        rstd = torch.empty(M, dtype=torch.float32, device=self.dev)
        nqkv = (nh + 2 * nkv) * dh
        qkv = self._new(M, nqkv)
        attn = self._new(M, nh * dh)
        mid = self._new(M, I)
        rope = (table, L, dh, (nh + nkv) * dh) if m["fuse_rope"] else None
        # RMSNorm statistics ride on the GEMMs that write the residual stream: o_proj / down_proj add each row's sum of squares
        # into a zeroed [2 * layers, M] fixed-point table (integer atomics: order-independent, bit-reproducible) and the next projection
        # turns it into rstd in its epilogue, so the only separate
        # pass over the residual stream is the one before the first layer (bf16 tensor-core path; fp32 keeps tcavp_row_rstd).
        nl = len(m["layers"])
        fuse_ss = self.act == torch.bfloat16 and not self.fp8 and not os.environ.get("TCAVP_NO_FUSE_RSTD")
        ss = torch.zeros(2 * nl, M, dtype=torch.int64, device=self.dev) if fuse_ss else None
        for li, ly in enumerate(m["layers"]):
            if self.fp8:            # LoRA merged: kx == 0, x == xs
                self._proj(ly, "wqkv", x, qkv, rms=True, rope=rope)
            else:
                if fuse_ss and li > 0:
                    norm1 = dict(row_sumsq=(ss[2 * li - 1], H, m["eps"]))
                else:
                    ops.row_rstd(xs, rstd, rows=M, cols=H, ldx=Kx, eps=m["eps"])
                    norm1 = dict(row_scale=rstd)
                if kx:
                    ops.gemm(xs, ly["a_cat"], xs[:, H:], M=M, N=m["n_lora"], K=H, lda=Kx, ldo=Kx)
                ops.gemm(xs, ly["wqkv"], qkv, M=M, N=nqkv, K=Kx, lda=Kx, rope=rope, **norm1)
            if rope is None:
                ops.rope_(qkv, rows=M, L=L, ld=nqkv, n_q_heads=nh, n_k_heads=nkv, dh=dh, table=table)
            if kv_out is not None:
                cache = torch.empty(B, kv_out[1], 2 * nkv * dh, dtype=self.act, device=self.dev)
                cache[:, :L].copy_(qkv.view(B, L, nqkv)[:, :, nh * dh:])
                kv_out[0].append(cache)
            ops.attention(qkv, qkv[:, nh * dh:], qkv[:, (nh + nkv) * dh:], attn, B=B, H=nh, Hkv=nkv, Tq=L, Tk=L, dh=dh,
                          q_strides=(L * nqkv, nqkv), k_strides=(L * nqkv, nqkv), v_strides=(L * nqkv, nqkv),
                          o_strides=(L * nh * dh, nh * dh), scale=dh ** -0.5, causal=True, key_mask=mask)
            if self.fp8:
                self._proj(ly, "wo", attn, x, residual=x)
                self._proj(ly, "wgu", x, mid, rms=True, act=ops.ACT_SWIGLU)
                self._proj(ly, "wdown", mid, x, residual=x)
            elif fuse_ss:
                ops.gemm(attn, ly["wo"], x, ldo=Kx, residual=x, ldr=Kx, sumsq_out=ss[2 * li])
                ops.gemm(xs, ly["wgu"], mid, M=M, K=H, lda=Kx, act=ops.ACT_SWIGLU, row_sumsq=(ss[2 * li], H, m["eps"]))
                ops.gemm(mid, ly["wdown"], x, ldo=Kx, residual=x, ldr=Kx, sumsq_out=ss[2 * li + 1] if li + 1 < nl else None)
            else:
                ops.gemm(attn, ly["wo"], x, ldo=Kx, residual=x, ldr=Kx)
                ops.row_rstd(xs, rstd, rows=M, cols=H, ldx=Kx, eps=m["eps"])
                ops.gemm(xs, ly["wgu"], mid, M=M, K=H, lda=Kx, act=ops.ACT_SWIGLU, row_scale=rstd)
                ops.gemm(mid, ly["wdown"], x, ldo=Kx, residual=x, ldr=Kx)
        return ops.rmsnorm(xs, m["norm"], self._new(M, H), eps=m["eps"], rows=M, cols=H, ldi=Kx)

    def llm_decode_step(self, x_new, caches, t):
        """One decode step of the KV-cache path (SURVEY.md §8 f4; HF generate with past_key_values): `x_new` (B, H) = the embedding of
        the token at position `t` of every sequence, `caches` = the per-layer [B, capacity, 2 n_kv dh] key / value caches filled up to
        position t - 1 by `llm_forward(kv_out=...)` / earlier steps.  The new row's rotated key and value are appended, its query attends
        over positions 0..t (one query, no mask needed), and the post-final-norm hidden state (B, H) is returned.  Same kernels as the
        full forward: tcavp_gemm with the RMSNorm row factor / LoRA K-extension / RoPE / SwiGLU epilogues, tcavp_attention."""
        m = self.llm
        if m.get("arch") == "gpt2":
            return self._gpt2_decode_step(x_new, caches, t)
        H, nh, nkv, dh, I, kx = m["H"], m["nh"], m["nkv"], m["dh"], m["I"], m["kx"]
        B = x_new.shape[0]
        cap = caches[0].shape[1]
        if t >= cap:
            raise ops._lib.TcavpError(f"llm_decode_step: position {t} is past the cache capacity {cap}")
        lay = 1 if m["fuse_rope"] else 0
        key = (cap, dh, lay)
        if key not in self._rope:
            self._rope[key] = ops.rope_table(cap, dh, m["theta"], self.dev, layout=lay)
        full = self._rope[key]
        table = (full[:, t:t + 1] if lay == 1 else full[t:t + 1]).contiguous()       # the one position this step needs (rope_L = 1)
        Kx, nq, nk = H + kx, nh * dh, nkv * dh
        nqkv = nq + 2 * nk
        xs = torch.zeros(B, Kx, dtype=self.act, device=self.dev)
        ops.cast(x_new.reshape(B, H), xs, rows=B, cols=H, ldi=H, ldo=Kx)
        x = xs[:, :H]
        rstd = torch.empty(B, dtype=torch.float32, device=self.dev)
        qkv, attn, mid = self._new(B, nqkv), self._new(B, nq), self._new(B, I)
        rope = (table, 1, dh, nq + nk) if m["fuse_rope"] else None
        for ly, cache in zip(m["layers"], caches):
            if self.fp8:            # LoRA merged: kx == 0, x == xs
                self._proj(ly, "wqkv", x, qkv, rms=True, rope=rope)
            else:
                ops.row_rstd(xs, rstd, rows=B, cols=H, ldx=Kx, eps=m["eps"])
                if kx:
                    ops.gemm(xs, ly["a_cat"], xs[:, H:], M=B, N=m["n_lora"], K=H, lda=Kx, ldo=Kx)
                ops.gemm(xs, ly["wqkv"], qkv, M=B, N=nqkv, K=Kx, lda=Kx, rope=rope, row_scale=rstd)
            if rope is None:
                ops.rope_(qkv, rows=B, L=1, ld=nqkv, n_q_heads=nh, n_k_heads=nkv, dh=dh, table=table)
            cache[:, t].copy_(qkv[:, nq:])
            ops.attention(qkv, cache, cache[:, :, nk:], attn, B=B, H=nh, Hkv=nkv, Tq=1, Tk=t + 1, dh=dh, q_strides=(nqkv, nqkv),
                          k_strides=(cap * 2 * nk, 2 * nk), v_strides=(cap * 2 * nk, 2 * nk), o_strides=(nq, nq), scale=dh ** -0.5)
            if self.fp8:
                self._proj(ly, "wo", attn, x, residual=x)
                self._proj(ly, "wgu", x, mid, rms=True, act=ops.ACT_SWIGLU)
                self._proj(ly, "wdown", mid, x, residual=x)
                continue
            ops.gemm(attn, ly["wo"], x, ldo=Kx, residual=x, ldr=Kx)
            ops.row_rstd(xs, rstd, rows=B, cols=H, ldx=Kx, eps=m["eps"])
            ops.gemm(xs, ly["wgu"], mid, M=B, K=H, lda=Kx, act=ops.ACT_SWIGLU, row_scale=rstd)
            ops.gemm(mid, ly["wdown"], x, ldo=Kx, residual=x, ldr=Kx)
        return ops.rmsnorm(xs, m["norm"], self._new(B, H), eps=m["eps"], rows=B, cols=H, ldi=Kx)

    def ltsf_encode(self, x, B):
        """reference scripts/train.py:837-840 -> enc (B*T_in, C)."""
        lt, C, T, sm = self.lt, self.C, self.T_in, self.small
        e0 = ops.ltsf_encode(x, lt["wt"], lt["bt"], lt["we"], lt["be"], lt["pos"], self._new(B * T, C, dtype=sm), B=B, F=2, C=C, T_in=T)
        xn = self._ln_res(e0, lt["n1"])
        a = self._self_attention(xn, T, B, lt["mha"])
        y = self._gemm_small(a, lt["mha"]["out"], self._new(B * T, C, dtype=sm), residual=xn)
        r = self._ln_res(y, lt["n2"])
        h = self._gemm_small(r, lt["f0"], self._new(B * T, lt["f0"].N, dtype=sm), act=ops.ACT_RELU)
        return self._gemm_small(h, lt["f3"], self._new(B * T, C, dtype=sm), residual=r)

    def ltsf_decode(self, enc, poly_emb, fh, x, B, L, y=None, norm_stat=None):
        """reference scripts/train.py:767-806 + 941-943 (+ 945-962 / 1302-1322 when y is given)."""
        lt, C, T, To, sm = self.lt, self.C, self.T_in, self.T_out, self.small
        H = self.llm["H"]
        adj = self._gemm_small(poly_emb, lt["lane_fc"], self._new(B, To * C, dtype=sm))
        dec = ops.nlinear_decode(enc, lt["wd"], lt["bd"], adj, self._new(B, To * C, dtype=sm), B=B, C=C, T_in=T, T_out=To)
        if lt["post"] is not None:
            p0, p3 = lt["post"]
            h = self._gemm_small(dec, p0, self._new(B, p0.N, dtype=sm), act=ops.ACT_RELU)
            dec = self._gemm_small(h, p3, self._new(B, To * C, dtype=sm))
        dec_t = dec.view(B * To, C)                  # fp32 residual path of the regression head
        dq = dec_t if self.act == sm else ops.cast(dec_t, self._new(B * To, C), rows=B * To, cols=C)
        q = ops.gemm(dq, lt["dec_proj"].w, self._new(B * To, H), bias=lt["dec_proj"].b)
        ab = lt.get("absorb")
        if ab is not None and fh.dtype == self.act and To <= 64 and L <= 256:
            E, heads = ab["E"], ab["heads"]
            qp = ops.gemm(q, ab["mq"], self._new(B * To, heads * E), bias=ab["cq"])
            z = self._new(B * To, heads * E)
            ops.attention(qp, fh, fh, z, B=B, H=heads, Hkv=1, Tq=To, Tk=L, dh=E, q_strides=(To * heads * E, heads * E), k_strides=(L * E, E),
                          v_strides=(L * E, E), o_strides=(To * heads * E, heads * E), scale=ab["dh"] ** -0.5)
            co = ops.gemm(z, ab["mo"], self._new(B * To, H), bias=ab["co"])
        else:
            a = self._cross_attention(q, To, fh, L, B, lt["cross"])
            co = ops.gemm(a, lt["cross"]["out"].w, self._new(B * To, H), bias=lt["cross"]["out"].b)
        fused = ops.gemm(co, lt["dec_unproj"].w, self._new(B * To, C, dtype=sm), bias=lt["dec_unproj"].b, residual=dec_t)
        decoded = torch.empty(B, 2, To, dtype=torch.float32, device=self.dev)
        out = {"decoded": decoded}
        metrics = per_scene = None
        if y is not None:
            metrics = torch.zeros(8, dtype=torch.float32, device=self.dev)
            per_scene = torch.empty(B, 2, dtype=torch.float32, device=self.dev)
        ops.fusion_head(fused, lt["fl_ln"][0], lt["fl_ln"][1], lt["fl_w1"], lt["fl_b1"], lt["fl_w2"], lt["fl_b2"], lt["wo"], lt["bo"], x,
                        decoded, y=y, norm_stat=norm_stat, metrics=metrics, per_scene=per_scene, B=B, C=C, T_in=T, T_out=To,
                        tensor_cores=(self.act == torch.bfloat16 and self.SPLIT_SMALL and not os.environ.get("TCAVP_NO_SPLIT_SMALL")
                                      and not os.environ.get("TCAVP_NO_HEAD_TC")))
        if y is not None:
            out.update(metrics=metrics, per_scene=per_scene)
        return out

    # ---- text-generation side path (generate.py) -------------------------------------------------------
    def lm_head(self):
        """[V, H] vocabulary projection in the activation dtype (HF:487-491); never used by forward() — its logits are discarded there."""
        if self.llm.get("lm_head") is None:
            w = self._lm_head_param
            tied = w.data_ptr() == self._embed_param.data_ptr()
            self.llm["lm_head"] = self.llm["embed"] if tied else w.detach().to(self.dev, self.act).contiguous()
        return self.llm["lm_head"]

    @torch.no_grad()
    def token_embeds(self, ids, text_modality=False):
        """ids (B, T) int64 -> (B, T, H) embedding rows, optionally + text_modality_embedding."""
        B, T = ids.shape
        H = self.llm["H"]
        out = self._new(B, T, H)
        if not hasattr(self, "_zero_mod"):
            self._zero_mod = torch.zeros(H, dtype=torch.float32, device=self.dev)
        ops.embed_text(ids.to(device=self.dev, dtype=torch.int64).contiguous(), None, self.llm["embed"], self.text_mod if text_modality else self._zero_mod,
                       out, None, B=B, L_text=T, n_img=0, H=H)
        return out

    @torch.no_grad()
    def prefix_embeds(self, vision, prompt_ids):
        """Image tokens (+ vision modality) followed by the prompt embeddings (+ text modality): reference train.py:585-598."""
        vision = vision.to(self.dev)
        if vision.dtype not in (torch.float32, torch.bfloat16):
            vision = vision.float()
        ids = prompt_ids.to(device=self.dev, dtype=torch.int64).contiguous()
        B, Lp = ids.shape
        Q, H = self.qf["Q"], self.llm["H"]
        L = Q + Lp
        fused = self._new(B, L, H)
        mask = torch.empty(B, L, dtype=torch.int32, device=self.dev)
        self.qformer_into(vision.contiguous(), fused, L)
        ops.embed_text(ids, None, self.llm["embed"], self.text_mod, fused, mask, B=B, L_text=Lp, n_img=Q, H=H)
        return fused

    # ---- full forward -------------------------------------------------------------------------------
    def _dev_f32(self, t):
        if not torch.is_tensor(t):
            t = torch.tensor(t, dtype=torch.float32)
        return t.to(device=self.dev, dtype=torch.float32, non_blocking=True).contiguous()

    @torch.no_grad()
    def forward(self, x, vision, polygon, poly_len, input_ids, attention_mask, y=None, norm_stat=None, final_hidden=None,
                keep_intermediates=False, max_poly_len=None, cuda_graph=False):
        """`cuda_graph`: replay the ~200 launches of one forward from a CUDA graph captured per input-shape signature (serving loops
        with a fixed batch shape).  The returned tensors are then the graph's static outputs: consume (or copy) them before the next
        call with the same shapes."""
        dev = self.dev
        if dev.type != "cuda":
            raise ops._lib.TcavpError("the model must be on a CUDA device (there is no CPU fallback): model.to('cuda')")
        x = self._dev_f32(x)
        B = x.shape[0]
        polygon = self._dev_f32(polygon)
        lens = poly_len if torch.is_tensor(poly_len) else torch.tensor(list(poly_len), dtype=torch.int32)
        if max_poly_len is None and not lens.is_cuda and lens.numel() > 0:
            max_poly_len = int(lens.max())          # host-resident lengths (the reference passes a Python list): no device sync needed
        lens = lens.to(device=dev, dtype=torch.int32, non_blocking=True)
        if y is not None and norm_stat is not None:
            y = self._dev_f32(y)
            norm_stat = self._dev_f32(norm_stat).view(B, 4)
        else:
            y = norm_stat = None
        # Host-resident (pinned) bulk inputs travel on a side stream while the polygon / temporal encoders — which only need the
        # small tensors already queued above — run on the compute stream; the compute stream joins right before the first consumer.
        bulk = [t for t in ((vision, input_ids, attention_mask) if final_hidden is None else (final_hidden,)) if torch.is_tensor(t) and not t.is_cuda]
        copied = None
        if bulk and all(t.is_pinned() for t in bulk):
            if getattr(self, "_copy_stream", None) is None:
                self._copy_stream = torch.cuda.Stream(device=dev)
            main = torch.cuda.current_stream()
            # no wait on `main`: the sources are host buffers and the destinations are fresh allocations of the copy stream, so the copy
            # of call i+1 may run under the kernels of call i (a caller that enqueues the next batch before reading the last result)
            with torch.cuda.stream(self._copy_stream):
                moved = {id(t): t.to(dev, non_blocking=True) for t in bulk}
                copied = torch.cuda.Event()
                copied.record()
            for t in moved.values():
                t.record_stream(main)
            pick = lambda t: moved.get(id(t), t) if torch.is_tensor(t) else t      # noqa: E731
            if final_hidden is None:
                vision, input_ids, attention_mask = pick(vision), pick(input_ids), pick(attention_mask)
            else:
                final_hidden = pick(final_hidden)
        if final_hidden is None:
            vision = vision.to(dev, non_blocking=True)
            if vision.dtype not in (torch.float32, torch.bfloat16):
                vision = vision.float()
            vision = vision.contiguous()
            input_ids = input_ids.to(device=dev, dtype=torch.int64, non_blocking=True).contiguous()
            attention_mask = attention_mask.to(device=dev, dtype=torch.int64, non_blocking=True).contiguous()
        else:
            final_hidden = final_hidden.to(device=dev, dtype=self.act, non_blocking=True).contiguous()
        dev_in = dict(x=x, vision=vision, polygon=polygon, lens=lens, input_ids=input_ids, attention_mask=attention_mask, y=y, norm_stat=norm_stat,
                      final_hidden=final_hidden)
        if cuda_graph and not keep_intermediates:
            return self._forward_graphed(dev_in, max_poly_len, copied)
        return self._forward_device(dev_in, max_poly_len, copied, keep_intermediates)

    def _forward_graphed(self, dev_in, max_poly_len, copied):
        """One CUDA graph per (shapes, dtypes, max_poly_len) signature; inputs are copied into the graph's static buffers (device to
        device, a few tens of MB) and the ~200 kernel launches of the forward become one cudaGraphLaunch."""
        sig = tuple((k, None if v is None else (tuple(v.shape), v.dtype)) for k, v in dev_in.items()) + (max_poly_len,)
        cache = self.__dict__.setdefault("_graphs", {})
        ent = cache.pop(sig, None)
        if copied is not None:
            torch.cuda.current_stream().wait_event(copied)
        if ent is None:
            static = {k: (None if v is None else v.clone()) for k, v in dev_in.items()}
            side = torch.cuda.Stream(device=self.dev)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2):                 # lazy packing, rope tables, cudaFuncSetAttribute, allocator warm-up
                    self._forward_device(static, max_poly_len, None, False)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                out = self._forward_device(static, max_poly_len, None, False)
            ent = (g, static, out)
            while len(cache) >= 4:
                cache.pop(next(iter(cache)))
        cache[sig] = ent
        g, static, out = ent
        for k, v in dev_in.items():
            if v is not None:
                static[k].copy_(v, non_blocking=True)
        g.replay()
        return out

    def _forward_device(self, d, max_poly_len, copied, keep_intermediates):
        """The device part of forward(): every input already lives on the device (capturable in a CUDA graph)."""
        dev = self.dev
        x, vision, polygon, lens, y, norm_stat, final_hidden = d["x"], d["vision"], d["polygon"], d["lens"], d["y"], d["norm_stat"], d["final_hidden"]
        B = x.shape[0]
        out = {}
        poly_emb = self.poly_forward(polygon, lens, max_poly_len)
        enc = self.ltsf_encode(x, B)
        if copied is not None:
            torch.cuda.current_stream().wait_event(copied)
        if final_hidden is None:
            ids, am = d["input_ids"], d["attention_mask"]
            Q, H = self.qf["Q"], self.llm["H"]
            L = Q + ids.shape[1]
            fused = self._new(B, L, H)
            mask = torch.empty(B, L, dtype=torch.int32, device=dev)
            self.qformer_into(vision, fused, L)
            ops.embed_text(ids, am, self.llm["embed"], self.text_mod, fused, mask, B=B, L_text=ids.shape[1], n_img=Q, H=H)
            if keep_intermediates:
                out["image_tokens_plus_mod"] = fused[:, :Q].float()
            fh = self.llm_forward(fused, mask, B, L)
        else:
            fh = final_hidden
            L = fh.shape[1]
            fh = fh.view(B * L, -1)
        out.update(self.ltsf_decode(enc, poly_emb, fh, x, B, L, y, norm_stat))
        if y is not None:
            m = out["metrics"]
            out["loss"] = m[4]                                  # MSE_x + MSE_y, reference scripts/train.py:959-961
            out["sum_ade"], out["sum_fde"] = m[2], m[3]
            out["ade"], out["fde"] = out["per_scene"][:, 0], out["per_scene"][:, 1]
        if keep_intermediates:
            out["poly_emb"] = poly_emb.float()
            out["final_hidden"] = fh.view(B, L, -1).float()
            out["enc"] = enc.view(B, self.T_in, self.C).permute(0, 2, 1).float()
        return out
