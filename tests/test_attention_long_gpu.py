"""Causal self-attention past 256 positions and GQA backward on tensor cores: the key-blocked tcgen05 forward (attn_tml_kernel), the
optional logsumexp output of tcavp_attention, and the key-blocked backward (attn_bwd_kv_kernel + attn_bwd_q_kernel) that rebuilds the
probabilities from it.  Checked against fp32 torch / autograd, and at model level the stage-1 objective at 1040 positions against the
CPU oracle."""
import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = "cuda"


@pytest.fixture(scope="module")
def ops(lib_built):
    import tcavp_b200.ops as O
    return O


def _problem(B, L, H, Hkv, dh, seed):
    """Packed [B * L, (H + 2 Hkv) dh] bf16 QKV activation (the layout of the decoder's fused QKV GEMM) and ragged key masks:
    scene 0 unmasked, scene 1 only keys 0-2 (rows past 2 see 3 keys), scene 2 the first 5 keys masked (rows 0-4 see none),
    later scenes random right padding."""
    g = torch.Generator().manual_seed(seed)
    nqkv = (H + 2 * Hkv) * dh
    qkv = (torch.randn(B * L, nqkv, generator=g) * 1.5).to(torch.bfloat16).to(DEV)
    mask = torch.ones(B, L, dtype=torch.int32)
    if B > 1:
        mask[1, 3:] = 0
    if B > 2:
        mask[2, :5] = 0
    for b in range(3, B):
        mask[b, int(torch.randint(L // 2, L + 1, (1,), generator=g)):] = 0
    return qkv, mask.to(DEV)


def _views(qkv, B, L, H, Hkv, dh):
    x = qkv.float().view(B, L, H + 2 * Hkv, dh)
    return x[:, :, :H], x[:, :, H:H + Hkv], x[:, :, H + Hkv:]


def _reference(q, k, v, mask, scale):
    """fp32 causal + key-padding attention; q [B, L, H, dh], k / v [B, L, Hkv, dh] -> out [B, L, H, dh], lse [B, H, L]."""
    B, L, H, dh = q.shape
    rep = H // k.shape[2]
    kk, vv = k.repeat_interleave(rep, dim=2), v.repeat_interleave(rep, dim=2)
    s = torch.einsum("bihd,bjhd->bhij", q, kk) * scale
    ok = torch.ones(L, L, dtype=torch.bool, device=q.device).tril()[None, None] & (mask[:, None, None, :] != 0)
    s = s.masked_fill(~ok, float("-inf"))
    lse = torch.logsumexp(s, dim=-1)
    p = torch.where(ok, torch.exp(s - lse[..., None].clamp_min(-1e30)), torch.zeros_like(s))
    return torch.einsum("bhij,bjhd->bihd", p, vv), lse


def _forward(ops, qkv, mask, B, L, H, Hkv, dh, lse=True):
    nqkv = (H + 2 * Hkv) * dh
    out = torch.empty(B * L, H * dh, dtype=torch.bfloat16, device=DEV)
    ls = torch.empty(B * H * L, dtype=torch.float32, device=DEV) if lse else None
    s = (L * nqkv, nqkv)
    ops.attention(qkv, qkv[:, H * dh:], qkv[:, (H + Hkv) * dh:], out, B=B, H=H, Hkv=Hkv, Tq=L, Tk=L, dh=dh, q_strides=s, k_strides=s,
                  v_strides=s, o_strides=(L * H * dh, H * dh), scale=dh ** -0.5, causal=True, key_mask=mask, lse=ls)
    return out, ls


SHAPES = [(64, 32, 8), (128, 8, 2), (64, 12, 12)]      # (head_dim, H, Hkv): the Llama-3.2-1B group shape, a 128-wide GQA head, MHA


@pytest.mark.parametrize("L", [257, 300, 528, 1040, 2048])
@pytest.mark.parametrize("dh,H,Hkv", SHAPES)
def test_long_forward_matches_torch(ops, L, dh, H, Hkv):
    B = 3
    if L == 2048 and H == 32:
        H, Hkv = 8, 2                                   # keeps the fp32 reference's [B, H, L, L] scores small
    qkv, mask = _problem(B, L, H, Hkv, dh, seed=L + dh + H)
    out, lse = _forward(ops, qkv, mask, B, L, H, Hkv, dh)
    torch.cuda.synchronize()
    assert ops.last_kernel() == "attn_tml_kernel"
    q, k, v = _views(qkv, B, L, H, Hkv, dh)
    want, wlse = _reference(q, k, v, mask, dh ** -0.5)
    torch.testing.assert_close(out.float().view(B, L, H, dh), want, rtol=2e-2, atol=2e-2)
    lse = lse.view(B, H, L)
    assert torch.isneginf(lse[2, :, :5]).all() and torch.isneginf(wlse[2, :, :5]).all()
    assert (out.view(B, L, H, dh)[2, :5] == 0).all()              # rows with no visible key: output 0
    fin = torch.isfinite(wlse)
    assert torch.equal(fin, torch.isfinite(lse))
    torch.testing.assert_close(lse[fin], wlse[fin], rtol=1e-4, atol=1e-4)
    # scene b alone gives the same bits as scene b inside the batch
    b = 1
    nqkv = (H + 2 * Hkv) * dh
    alone, _ = _forward(ops, qkv[b * L:(b + 1) * L].contiguous(), mask[b:b + 1].contiguous(), 1, L, H, Hkv, dh)
    assert torch.equal(alone, out[b * L:(b + 1) * L]), nqkv


@pytest.mark.parametrize("L", [144, 200])
def test_lse_on_the_tile_kernel(ops, L):
    """attn_tm_kernel (128 <= L <= 256) writes the logsumexp when asked, and the output bits do not depend on whether it was asked."""
    B, H, Hkv, dh = 5, 8, 2, 64
    qkv, mask = _problem(B, L, H, Hkv, dh, seed=L)
    out, lse = _forward(ops, qkv, mask, B, L, H, Hkv, dh)
    assert ops.last_kernel() == "attn_tm_kernel"
    out0, _ = _forward(ops, qkv, mask, B, L, H, Hkv, dh, lse=False)
    assert torch.equal(out, out0)
    q, k, v = _views(qkv, B, L, H, Hkv, dh)
    _, wlse = _reference(q, k, v, mask, dh ** -0.5)
    lse = lse.view(B, H, L)
    fin = torch.isfinite(wlse)
    assert torch.equal(fin, torch.isfinite(lse)) and torch.isneginf(lse[~fin]).all()
    torch.testing.assert_close(lse[fin], wlse[fin], rtol=1e-4, atol=1e-4)


def _grad_close(got, want, name):
    err = float((got.float() - want).norm() / (want.norm() + 1e-30))
    mx = float((got.float() - want).abs().max())
    assert err < 2e-2 and mx < 2e-2 * float(want.abs().max()) + 1e-3, (name, err, mx, float(want.abs().max()))


@pytest.mark.parametrize("L,dh,H,Hkv", [(144, 64, 32, 8), (300, 64, 12, 12), (768, 128, 8, 2), (1040, 64, 4, 2), (1040, 128, 4, 4)])
def test_long_gqa_backward_matches_autograd(ops, L, dh, H, Hkv):
    B = 3
    qkv, mask = _problem(B, L, H, Hkv, dh, seed=7 * L + H)
    out, lse = _forward(ops, qkv, mask, B, L, H, Hkv, dh)
    g = torch.Generator().manual_seed(L)
    dout = torch.randn(B * L, H * dh, generator=g).to(torch.bfloat16).to(DEV)
    nqkv = (H + 2 * Hkv) * dh
    s = (L * nqkv, nqkv)

    def backward():
        d = torch.full_like(qkv, float("nan"))
        ops.attention_bwd_owned(qkv, qkv[:, H * dh:], qkv[:, (H + Hkv) * dh:], dout, d, d[:, H * dh:], d[:, (H + Hkv) * dh:], B=B, H=H, Hkv=Hkv,
                                Tq=L, Tk=L, dh=dh, q_strides=s, k_strides=s, v_strides=s, do_strides=(L * H * dh, H * dh), dq_strides=s,
                                dk_strides=s, dv_strides=s, scale=dh ** -0.5, causal=True, key_mask=mask, o=out,
                                o_strides=(L * H * dh, H * dh), lse=lse)
        return d

    assert ops.attention_bwd_owned_ok(qkv, H=H, Hkv=Hkv, Tq=L, Tk=L, dh=dh, o=out, causal=True, lse=lse)
    d1 = backward()
    assert ops.last_kernel() == "attn_bwd_q_kernel"
    d2 = backward()
    torch.cuda.synchronize()
    assert torch.equal(d1, d2)                                       # deterministic: no floating-point atomics
    q, k, v = (t.clone().requires_grad_(True) for t in _views(qkv, B, L, H, Hkv, dh))
    want, _ = _reference(q, k, v, mask, dh ** -0.5)
    want.backward(dout.float().view(B, L, H, dh))
    dq, dk, dv = _views(d1, B, L, H, Hkv, dh)
    assert torch.isfinite(d1.float()).all()
    _grad_close(dq, q.grad, "dq")
    _grad_close(dk, k.grad, "dk")
    _grad_close(dv, v.grad, "dv")


def _assert_long_routes(prof, L, n_layers=2):
    """Every decoder layer ran its self-attention forward on attn_tml_kernel and its backward on the key-blocked pair."""
    labels = [r[0] for r in prof.rec]
    assert labels.count(f"attn_tml_kernel[dh64,L{L}]") == n_layers, sorted(set(labels))
    assert labels.count(f"attn_bwd_kv_q_kernels[dh64,q{L},k{L}]") == n_layers, sorted(set(labels))


STAGE1_LLAMA = dict(vocab_size=97, hidden_size=256, intermediate_size=512, num_hidden_layers=2, num_attention_heads=4, num_key_value_heads=2,
                    head_dim=64, rms_norm_eps=1e-6, rope_theta=10000.0)


def test_bf16_stage1_at_1040_positions_tracks_oracle(lib_built):
    """stage1_forward at L = 16 image + 1024 text tokens on a 2-layer GQA backbone (head_dim 64): forward on attn_tml_kernel, backward on
    the key-blocked kernels (the SIMT backward stops at 768 keys).  Bands of test_bf16_stage1_tracks_reference."""
    import tcavp_b200 as T
    from oracle import restated
    mc = dict(T.MODEL_PRESETS["tiny"], base_model_name=dict(STAGE1_LLAMA))
    s = T.make_scenes(2, mc["seq_len"], mc["out_len"], vision_dim=mc["vision_dim"], l_text=1024, vocab=97, seed=31)
    labels = restated.stage1_labels(s["input_ids"], s["attention_mask"], 600)
    ref = T.MultiModalTrajectoryModel(**mc)
    sd = ref.state_dict()
    T.deterministic_fill_(sd, 13)
    want_loss, want = restated.stage1_loss_and_grads({k: v.clone() for k, v in sd.items()}, mc, T.resolve_llama(mc["base_model_name"]),
                                                     s["vision"], s["input_ids"], s["attention_mask"], labels)
    m = T.MultiModalTrajectoryModel(**mc, compute_dtype="bf16")
    m.load_state_dict(sd, strict=True)
    m = m.to(DEV).eval()
    with T.ops.LaunchProfiler() as prof:
        out = m.stage1_forward(s["vision"].cuda(), s["input_ids"].cuda(), s["attention_mask"].cuda(), labels.cuda())
        out.loss.backward()
    torch.cuda.synchronize()
    _assert_long_routes(prof, 1040)
    assert abs(float(out.loss) - float(want_loss)) / float(want_loss) < 2e-2, (float(out.loss), float(want_loss))
    gmax = max(float(g.norm()) for g in want.values())
    low, bad, checked = [], [], 0
    for n, p in m.named_parameters():
        if n not in want or p.grad is None:
            continue
        g, w = p.grad.float().cpu().flatten(), want[n].flatten()
        if float(w.norm()) < 1e-4 * gmax:
            continue
        checked += 1
        cos = float(torch.dot(g, w) / (g.norm() * w.norm() + 1e-30))
        ratio = float(g.norm() / (w.norm() + 1e-30))
        if cos < 0.98 or not 0.9 < ratio < 1.1:
            low.append((n, round(cos, 4), round(ratio, 4)))
        if cos < 0.95 or not 0.8 < ratio < 1.25:
            bad.append((n, round(cos, 4), round(ratio, 4)))
    assert checked > 10 and not bad, (checked, bad[:10])
    assert len(low) <= max(1, checked // 50), (checked, low[:10])


# ---------------------------------------------------------------------------------------------------------------------------------
# The trajectory fine-tune step at 16 image + 512 text tokens = 528 positions, on 2-layer backbones with head_dim 64: Llama MHA (the
# 768-class train path), Llama GQA, and the GPT-2 architecture.  The fusion cross-attention then runs against 528 keys as well.
FT_BACKBONES = {
    "llama_mha": dict(STAGE1_LLAMA, num_key_value_heads=4),
    "llama_gqa": dict(STAGE1_LLAMA),
    "gpt2": dict(arch="gpt2", vocab_size=97, hidden_size=256, intermediate_size=1024, num_hidden_layers=2, num_attention_heads=4,
                 n_positions=1024, layer_norm_epsilon=1e-5, tie_word_embeddings=True, attn_pdrop=0.1, resid_pdrop=0.1, embd_pdrop=0.1),
}
ILL = ("lane_polygon_encoder.pos_embedding", "lane_polygon_encoder.input_proj", "lane_polygon_encoder.encoder.layers.0.self_attn.in_proj")


def _ft_setup(backbone, B=2, l_text=512):
    import tcavp_b200 as T
    mc = dict(T.MODEL_PRESETS["tiny"], base_model_name=dict(FT_BACKBONES[backbone]))
    s = T.make_scenes(B, mc["seq_len"], mc["out_len"], vision_dim=mc["vision_dim"], l_text=l_text, vocab=97, seed=77)
    g = torch.Generator().manual_seed(78)           # polygons as in the gradient goldens: no empty polygon, pixel-scale points
    s["poly_len"] = [33, 14][:B]
    pts = torch.rand(B, 64, 2, generator=g) * torch.tensor([3839.0, 750.0]) + torch.tensor([0.0, 700.0])
    keep = torch.arange(64)[None, :] < torch.tensor(s["poly_len"])[:, None]
    s["polygon"] = torch.where(keep[..., None], pts, torch.zeros_like(pts))
    sd = T.MultiModalTrajectoryModel(**mc).state_dict()
    T.deterministic_fill_(sd, 13)
    return T, mc, s, sd


def _bf16_model(T, mc, sd):
    m = T.MultiModalTrajectoryModel(**mc, compute_dtype="bf16")
    m.load_state_dict(sd, strict=True)
    return m.to(DEV).eval()


def _ft_args(s):
    return (s["x"].cuda(), s["vision"].cuda(), ["ctx"] * s["x"].shape[0], s["polygon"].cuda(), s["poly_len"], s["y"].cuda(), s["norm_stat"],
            s["input_ids"].cuda(), s["attention_mask"].cuda())


def _bands(got, want, skip=ILL):
    """cosine >= 0.98 and norm within 10 % per tensor above the noise floor (at most 1 % outside), cosine >= 0.95 / 20 % for all."""
    gmax = max(float(w.norm()) for w in want.values())
    low, bad, checked = [], [], 0
    for n, g in got.items():
        w = want[n]
        if n.startswith(skip) or float(w.norm()) < 1e-4 * gmax:
            continue
        g, w = g.float().cpu().flatten(), w.float().cpu().flatten()
        checked += 1
        cos = float(torch.dot(g, w) / (g.norm() * w.norm() + 1e-30))
        ratio = float(g.norm() / (w.norm() + 1e-30))
        if cos < 0.98 or not 0.9 < ratio < 1.1:
            low.append((n, round(cos, 4), round(ratio, 4)))
        if cos < 0.95 or not 0.8 < ratio < 1.25:
            bad.append((n, round(cos, 4), round(ratio, 4)))
    assert checked > 20 and not bad, (checked, bad[:10])
    assert len(low) <= max(0, checked // 100), (checked, low[:10])


@pytest.mark.parametrize("backbone", sorted(FT_BACKBONES))
def test_bf16_finetune_step_at_528_positions_tracks_oracle(lib_built, backbone):
    """The bf16 trajectory fine-tune step (forward + hand-written backward) at L = 528 against restated.loss_and_grads on the CPU, with
    the bands of tests/test_train_gpu.py::test_bf16_gradients_track_reference; the decoder self-attention ran on the long kernels."""
    from oracle import restated
    T, mc, s, sd = _ft_setup(backbone)
    want_loss, _, want = restated.loss_and_grads({k: v.clone() for k, v in sd.items()}, mc, T.resolve_llama(mc["base_model_name"]), s["x"],
                                                 s["vision"], s["polygon"], s["poly_len"], s["input_ids"], s["attention_mask"], s["y"],
                                                 s["norm_stat"])
    m = _bf16_model(T, mc, sd)
    x, vis, ctx, poly, plen, y, ns, ids, am = _ft_args(s)
    import warnings
    with warnings.catch_warnings(), T.ops.LaunchProfiler() as prof:
        warnings.simplefilter("ignore")
        loss, _ = m(x, vis, ctx, poly, plen, y=y, norm_stat=ns, input_ids=ids, attention_mask=am)
        loss.backward()
    torch.cuda.synchronize()
    _assert_long_routes(prof, 528)
    assert abs(float(loss) - float(want_loss)) / float(want_loss) < 2e-2, (float(loss), float(want_loss))
    _bands({n: p.grad for n, p in m.named_parameters() if p.requires_grad}, want)


@pytest.mark.parametrize("backbone", ["llama_gqa", "gpt2"])
def test_graph_captured_finetuner_at_528_positions_matches_eager(lib_built, backbone):
    """FineTuner replaying its CUDA graphs (the per-layer logsumexp buffers are allocated inside the captured forward and read by the
    captured backward) against the eager FineTuner from the same weights, over two optimizer steps: losses within 2 %, the flat-bucket
    gradients of every step within the gradient bands."""
    import warnings
    T, mc, s, sd = _ft_setup(backbone)
    args = _ft_args(s)
    warnings.simplefilter("ignore")
    fts = [T.FineTuner(_bf16_model(T, mc, sd), lr=5e-4, weight_decay=1e-4, use_cuda_graph=g) for g in (False, True)]
    for step in range(2):
        (le, _), (lg, _) = (ft.step(*args) for ft in fts)
        torch.cuda.synchronize()
        assert torch.isfinite(lg) and abs(float(lg) - float(le)) <= 2e-2 * abs(float(le)), (step, float(lg), float(le))
        eager = dict(zip(fts[0].names, fts[0].bucket.views))
        _bands(dict(zip(fts[1].names, fts[1].bucket.views)), {n: v.clone() for n, v in eager.items()})


def test_bf16_prefill_past_256_positions_then_decode_matches_fp32(lib_built):
    """Engine.llm_forward(kv_out=...) over a 16 + 300 = 316-position prefix (attn_tml_kernel), then three KV-cache decode steps reading
    keys past 256: the bf16 hidden states against the fp32 engine within the bf16 backbone band (relative L2 1e-2 at 2 layers)."""
    import tcavp_b200 as T
    from test_model_gpu import bf16_rel_l2_band
    mc = dict(T.MODEL_PRESETS["tiny"], base_model_name=dict(STAGE1_LLAMA))
    sd = T.MultiModalTrajectoryModel(**mc).state_dict()
    T.deterministic_fill_(sd, 13)
    s = T.make_scenes(2, mc["seq_len"], mc["out_len"], vision_dim=mc["vision_dim"], l_text=303, vocab=97, seed=5)
    vision, ids, extra_ids = s["vision"], s["input_ids"][:, :300], s["input_ids"][:, 300:303]
    hs = {}
    for dt in ("fp32", "bf16"):
        m = T.MultiModalTrajectoryModel(**mc, compute_dtype=dt)
        m.load_state_dict(sd, strict=True)
        eng = m.to(DEV).eval().engine()
        pre = eng.prefix_embeds(vision, ids)
        P, H = pre.shape[1], pre.shape[2]
        assert P == 316
        extra = eng.token_embeds(extra_ids.to(DEV))
        ones = torch.ones(2, P, dtype=torch.int32, device=DEV)
        caches = []
        with T.ops.LaunchProfiler() as prof:
            h0 = eng.llm_forward(pre.clone(), ones, 2, P, kv_out=(caches, P + 3)).view(2, P, H).float()
        if dt == "bf16":
            assert [r[0] for r in prof.rec].count("attn_tml_kernel[dh64,L316]") == 2, sorted({r[0] for r in prof.rec})
        steps = [eng.llm_decode_step(extra[:, j].contiguous(), caches, P + j).float() for j in range(3)]
        hs[dt] = (h0, torch.stack(steps, dim=1))
    band = bf16_rel_l2_band(2)
    for got, want in zip(hs["bf16"], hs["fp32"]):
        rel = float((got - want).norm() / want.norm())
        assert rel < band, (rel, band)


@pytest.mark.parametrize("case", ["bf16_gqa_L100", "fp32_L300", "fp32_dh32_L100"])
def test_lse_of_the_flash_and_simt_kernels(ops, case):
    """The logsumexp written by attn_flash_kernel (bf16 below 128 positions, here with GQA and then fed to the key-blocked backward),
    attn_warp_kernel and attn_row_kernel (fp32), against torch."""
    dtype, L, dh, H, Hkv, kern = {"bf16_gqa_L100": (torch.bfloat16, 100, 64, 8, 2, "attn_flash_kernel"),
                                  "fp32_L300": (torch.float32, 300, 64, 4, 2, "attn_warp_kernel"),
                                  "fp32_dh32_L100": (torch.float32, 100, 32, 4, 4, "attn_row_kernel")}[case]
    B = 3
    qkv, mask = _problem(B, L, H, Hkv, dh, seed=L + dh)
    qkv = qkv.to(dtype)
    nqkv = (H + 2 * Hkv) * dh
    s = (L * nqkv, nqkv)
    out = torch.empty(B * L, H * dh, dtype=dtype, device=DEV)
    lse = torch.empty(B * H * L, dtype=torch.float32, device=DEV)
    ops.attention(qkv, qkv[:, H * dh:], qkv[:, (H + Hkv) * dh:], out, B=B, H=H, Hkv=Hkv, Tq=L, Tk=L, dh=dh, q_strides=s, k_strides=s,
                  v_strides=s, o_strides=(L * H * dh, H * dh), scale=dh ** -0.5, causal=True, key_mask=mask, lse=lse)
    torch.cuda.synchronize()
    assert ops.last_kernel() == kern
    q, k, v = _views(qkv, B, L, H, Hkv, dh)
    want, wlse = _reference(q, k, v, mask, dh ** -0.5)
    lse = lse.view(B, H, L)
    fin = torch.isfinite(wlse)
    assert torch.equal(fin, torch.isfinite(lse)) and torch.isneginf(lse[~fin]).all()
    torch.testing.assert_close(lse[fin], wlse[fin], rtol=1e-4, atol=1e-4)
    if dtype != torch.bfloat16:
        return
    g = torch.Generator().manual_seed(L)
    dout = torch.randn(B * L, H * dh, generator=g).to(torch.bfloat16).to(DEV)
    d = torch.full_like(qkv, float("nan"))
    ops.attention_bwd_owned(qkv, qkv[:, H * dh:], qkv[:, (H + Hkv) * dh:], dout, d, d[:, H * dh:], d[:, (H + Hkv) * dh:], B=B, H=H, Hkv=Hkv,
                            Tq=L, Tk=L, dh=dh, q_strides=s, k_strides=s, v_strides=s, do_strides=(L * H * dh, H * dh), dq_strides=s,
                            dk_strides=s, dv_strides=s, scale=dh ** -0.5, causal=True, key_mask=mask, o=out, o_strides=(L * H * dh, H * dh),
                            lse=lse.view(-1))
    assert ops.last_kernel() == "attn_bwd_q_kernel"
    q, k, v = (t.clone().requires_grad_(True) for t in _views(qkv, B, L, H, Hkv, dh))
    want, _ = _reference(q, k, v, mask, dh ** -0.5)
    want.backward(dout.float().view(B, L, H, dh))
    dq, dk, dv = _views(d, B, L, H, Hkv, dh)
    _grad_close(dq, q.grad, "dq")
    _grad_close(dk, k.grad, "dk")
    _grad_close(dv, v.grad, "dv")
