"""fp8 (e4m3) serving mode on the GPU: tcavp_quant_e4m3_rows bit-exact against torch's float8_e4m3fn cast, the e4m3 forms of tcavp_gemm
against the fp32 product of the dequantised operands, the argument checks, and the fp8 engine against the Llama goldens."""
import ctypes

import pytest
import torch

pytestmark = pytest.mark.gpu

import tcavp_b200 as T  # noqa: E402
from conftest import build_filled_model, load_golden  # noqa: E402
from tcavp_b200 import ops  # noqa: E402

F8 = torch.float8_e4m3fn


@pytest.fixture(autouse=True)
def _no_tf32():
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32 = old


def _ref_quant(x):
    """The definition: s = 448 / amax (fp32, correctly rounded), q = e4m3(x * s), f = amax / 448; zero rows give q = 0, f = 0.
    (torch evaluates `448 / t` as 448 * reciprocal(t) and `t / 448` as t * (1 / 448); fp64 quotients rounded once to fp32 are the
    correctly rounded fp32 quotients.)"""
    xf = x.float()
    amax = xf.abs().amax(1)
    s = torch.where(amax > 0, (448.0 / amax.double()).float(), torch.zeros_like(amax))
    return (xf * s[:, None]).to(F8), (amax.double() / 448.0).float()


def _rows(rows, cols, ld, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(rows, ld, generator=g, device="cuda").mul_(torch.rand(rows, 1, generator=g, device="cuda") * 4).bfloat16()
    x[:, cols:] = 1e30           # padding past cols must be ignored
    if rows > 3:
        x[1, :cols] = 0          # all-zero row
        x[2, 7] = float(x[2, :cols].abs().amax()) * 1e4     # one outlier
    return x


@pytest.mark.parametrize("cols", [128, 256, 768, 2048, 3072, 4096, 8192, 11008])
@pytest.mark.parametrize("rows,pad", [(37, 0), (1031, 32)])
def test_quant_rows_is_bit_exact(lib_built, cols, rows, pad):
    x = _rows(rows, cols, cols + pad, cols + rows)
    q = torch.full((rows, cols + 16), 0x55, dtype=torch.uint8, device="cuda").view(F8)
    f = torch.empty(rows, dtype=torch.float32, device="cuda")
    ops.quant_e4m3_rows(x, q, f, cols=cols)
    qr, fr = _ref_quant(x[:, :cols])
    assert torch.equal(q[:, :cols].view(torch.uint8), qr.view(torch.uint8))
    assert torch.equal(q[:, cols:].view(torch.uint8), torch.full_like(q[:, cols:].view(torch.uint8), 0x55))     # ldo > cols: untouched
    assert torch.equal(f, fr)
    if rows > 3:
        assert float(f[1]) == 0 and torch.count_nonzero(q[1, :cols].view(torch.uint8)) == 0
    f2 = torch.empty_like(f)
    ops.quant_e4m3_rows(x, q, f2, cols=cols, rms_eps=1e-6)
    assert torch.equal(q[:, :cols].view(torch.uint8), qr.view(torch.uint8))
    xd = x[:, :cols].double()
    want = torch.rsqrt(xd.pow(2).mean(1) + 1e-6) * fr.double()
    torch.testing.assert_close(f2.double(), want, rtol=1e-6, atol=0)
    assert ops.last_kernel() == "quant_e4m3_kernel"


def _quant_w(w):
    s = w.abs().amax(1) / 448
    return torch.where(s[:, None] > 0, w / torch.where(s > 0, s, 1.0)[:, None], 0.0).to(F8), s


def _operands(M, N, K, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    a = torch.randn(M, K, generator=g, device="cuda").bfloat16()
    w = torch.randn(N, K, generator=g, device="cuda") * 0.05
    aq = torch.empty(M, K, dtype=F8, device="cuda")
    fa = torch.empty(M, dtype=torch.float32, device="cuda")
    ops.quant_e4m3_rows(a, aq, fa)
    wq, sw = _quant_w(w)
    # fp32 product of the dequantised operands (fp64 on the device, no TF32)
    acc = (aq.double() * fa.double()[:, None]) @ (wq.double() * sw.double()[:, None]).t()
    return aq, fa, wq.contiguous(), sw.contiguous(), acc


def _close(got, want, what):
    # fp32 accumulation of exact e4m3 products + one bf16 rounding of the output
    err = (got.double() - want).abs()
    bound = 2.0 ** -8 * want.abs() + 2e-3 * float(want.abs().max())
    assert bool((err <= bound).all()), (what, float(err.max()), float(want.abs().max()))


ROUTES = [(300, 32, "gemm_tc_kernel<32,e4m3>"), (300, 64, "gemm_tc_kernel<64,e4m3>"), (300, 100, "gemm_tc_kernel<128,e4m3>"),
          (300, 200, "gemm_tc_kernel<256,e4m3>"), (4100, 520, "gemm_tc_pair_kernel<256,e4m3>")]


@pytest.mark.parametrize("M,N,kern", ROUTES)
@pytest.mark.parametrize("K", [16, 144, 768, 3072])
def test_e4m3_gemm_every_route(lib_built, M, N, kern, K):
    aq, fa, wq, sw, acc = _operands(M, N, K, M + N + K)
    out = torch.empty(M, N, dtype=torch.bfloat16, device="cuda")
    ops.gemm(aq, wq, out, row_scale=fa, col_scale=sw)
    torch.cuda.synchronize()
    assert ops.last_kernel() == kern
    _close(out, acc, kern)
    out32 = torch.empty(M, N, dtype=torch.float32, device="cuda")       # fp32 output: accumulation precision alone
    ops.gemm(aq, wq, out32, row_scale=fa, col_scale=sw)
    err = float((out32.double() - acc).abs().max() / acc.abs().max())
    # measured on B200: 6e-8 (K = 16) .. 4.8e-7 (K = 3072) — fp32 accumulation in TMEM, every route
    assert err < 2e-6, (kern, K, err)


@pytest.mark.parametrize("M,N,kern", [ROUTES[3], ROUTES[4]])
def test_e4m3_gemm_epilogues(lib_built, M, N, kern):
    K = 768
    aq, fa, wq, sw, acc = _operands(M, N, K, 11)
    # + bf16 residual aliasing the output, ldo > N
    buf = torch.randn(M, N + 32, device="cuda").bfloat16()
    res0 = buf[:, :N].double().clone()
    ops.gemm(aq, wq, buf, ldo=N + 32, residual=buf, ldr=N + 32, row_scale=fa, col_scale=sw)
    assert ops.last_kernel() == kern
    _close(buf[:, :N], acc + res0, "residual")
    # SwiGLU on interleaved (gate, up) rows with their own column scales
    mid = torch.empty(M, N // 2, dtype=torch.bfloat16, device="cuda")
    ops.gemm(aq, wq, mid, act=ops.ACT_SWIGLU, row_scale=fa, col_scale=sw)
    gt, up = acc[:, 0::2], acc[:, 1::2]
    _close(mid, gt * torch.sigmoid(gt) * up, "swiglu")
    # fused RoPE on adjacent permuted columns (heads of 64, position m % L)
    L, dh, cols = 48, 64, (N // 64) * 64
    t1 = ops.rope_table(L, dh, 10000.0, "cuda", layout=1)
    t0 = ops.rope_table(L, dh, 10000.0, "cuda", layout=0).double()
    out = torch.empty(M, N, dtype=torch.bfloat16, device="cuda")
    ops.gemm(aq, wq, out, rope=(t1, L, dh, cols), row_scale=fa, col_scale=sw)
    want = acc.clone()
    pos = torch.arange(M, device="cuda") % L
    cs = t0[pos]                                  # [M, dh/2, 2]
    for h in range(cols // dh):
        a0, a1 = acc[:, h * dh:(h + 1) * dh:2], acc[:, h * dh + 1:(h + 1) * dh:2]
        want[:, h * dh:(h + 1) * dh:2] = a0 * cs[..., 0] - a1 * cs[..., 1]
        want[:, h * dh + 1:(h + 1) * dh:2] = a1 * cs[..., 0] + a0 * cs[..., 1]
    _close(out, want, "rope")


def test_e4m3_gemm_argument_checks(lib_built):
    M, N, K = 64, 64, 128
    aq, fa, wq, sw, _ = _operands(M, N, K, 3)
    out = torch.empty(M, N, dtype=torch.bfloat16, device="cuda")
    lib = T.lib.load()

    def call(**kw):
        g = ops.GemmArgs()
        g.M, g.N, g.K = M, N, kw.pop("K", K)
        g.A, g.lda, g.W, g.ldw, g.in_dtype = aq.data_ptr(), K, wq.data_ptr(), K, ops.E4M3
        g.out, g.ldo, g.out_dtype, g.act = out.data_ptr(), N, ops.BF16, kw.pop("act", ops.ACT_NONE)
        g.row_scale, g.col_scale = fa.data_ptr(), sw.data_ptr()
        for k, v in kw.items():
            setattr(g, k, v)
        return lib.tcavp_gemm(ctypes.byref(g), ops._stream())
    assert call() == 0
    assert call(col_scale=None) == -1                                  # TCAVP_ERR_ARG
    assert call(K=120) == -1                                           # K % 16 != 0
    ss = torch.zeros(M, dtype=torch.int64, device="cuda")
    aux = torch.empty(M, N, dtype=torch.bfloat16, device="cuda")
    assert call(sumsq_out=ss.data_ptr()) == -1
    assert call(row_sumsq=ss.data_ptr(), row_scale=None, sumsq_inv_cols=1.0 / K) == -1
    assert call(act=ops.ACT_SWIGLU, aux_out=aux.data_ptr(), ld_aux=N) == -1
    assert call(act=ops.ACT_SWIGLU_BWD, aux_out=aux.data_ptr(), ld_aux=2 * N) == -1
    g = ops.GemmArgs()                                                 # bf16 operands with a column scale
    a16, w16 = torch.zeros(M, K, dtype=torch.bfloat16, device="cuda"), torch.zeros(N, K, dtype=torch.bfloat16, device="cuda")
    g.M, g.N, g.K, g.A, g.lda, g.W, g.ldw, g.in_dtype = M, N, K, a16.data_ptr(), K, w16.data_ptr(), K, ops.BF16
    g.out, g.ldo, g.out_dtype, g.col_scale = out.data_ptr(), N, ops.BF16, sw.data_ptr()
    assert lib.tcavp_gemm(ctypes.byref(g), ops._stream()) == -1
    with pytest.raises(TypeError):
        ops.gemm(aq, w16, out, col_scale=sw)                           # mixed operand dtypes


# ---- the fp8 engine against the reference goldens -----------------------------------------------------------------------------
LLAMA_FIXTURES = ["tiny_b6", "cfg1_b8", "cfg3l2_b16", "gqa_l2_b32", "llama32_1b_l2_b8"]
# fp8 bands, calibrated on B200 (tools/fp8_error_probe.py, profiles/fp8_probe_r01.txt; with o_proj in e4m3 too:
# profiles/fp8_probe_r01_all4.txt).  e4m3 operands (3 mantissa bits) put final_hidden at 4.0-4.4e-2 relative L2 after two decoder layers
# and 6.5e-2 after twelve (bf16: 0.6-1.0e-2), row statistics within 1.0e-2.  The fp8 mode does NOT meet the bf16 north-star criteria
# (decoded within 2e-2, ADE / FDE within 0.5 %): measured decoded max |err| 4.5e-2 .. 1.21e-1, ADE 0.5 .. 2.7 %, FDE 0.4 .. 6.8 % across
# these fixtures; the head does not absorb e4m3 backbone noise.  The decoded / ADE / FDE bands below are the measured fp8 ones with
# margin, stated as such.  10 % multiplicative noise on ONE layer's weights gives 9.2e-2 .. 1.34e-1 relative L2, which the
# injected-error test must catch.
def fp8_rel_l2_band(n_layers):
    return 6.0e-2 + 3.0e-3 * n_layers        # 6.6e-2 at 2 layers, 9.6e-2 at 12


FP8_ROW_STAT = 2.0e-2
FP8_DECODED_ATOL = 0.25
FP8_ADE_FDE_REL = 8e-2
INJECT = 0.1


def _fp8_forward(fix, inject=0.0):
    m = build_filled_model(fix, "bf16", "cuda").fp8_backbone_for_inference()
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
    return m, {k: (v.float().cpu() if torch.is_tensor(v) else v) for k, v in o.items()}


def _check_fp8(m, o, g):
    assert float((o["decoded"] - g["decoded"]).abs().max()) < FP8_DECODED_ATOL
    for k in ("ade", "fde"):
        got, want = float(o[k].mean()), float(g[k].mean())
        assert abs(got - want) / want < FP8_ADE_FDE_REL, (k, got, want)
    n = g["final_hidden_head"].shape[0]
    fh = o["final_hidden"]
    r = float((fh[:n].double() - g["final_hidden_head"].double()).norm() / g["final_hidden_head"].double().norm())
    n_layers = len(m.mllm.llama_wrapper.causal_lm().model.layers)
    assert r < fp8_rel_l2_band(n_layers), ("final_hidden relative L2", r, n_layers)
    am = g["final_hidden_absmean"]
    assert float(((fh.mean(-1) - g["final_hidden_rowmean"]).abs() / am).max()) < FP8_ROW_STAT
    assert float(((fh.abs().mean(-1) - am).abs() / am).max()) < FP8_ROW_STAT


@pytest.mark.parametrize("name", LLAMA_FIXTURES)
def test_fp8_forward_matches_reference(lib_built, name):
    fix = load_golden(name)
    m, o = _fp8_forward(fix)
    assert m.engine().fp8 and any(ly[k].dtype == F8 for ly in m.engine().llm["layers"] for k in m.engine().FP8_PROJ)
    _check_fp8(m, o, fix["out"])


@pytest.mark.parametrize("name", ["cfg1_b8", "gqa_l2_b32"])
def test_fp8_check_catches_an_injected_backbone_error(lib_built, name):
    fix = load_golden(name)
    m, o = _fp8_forward(fix, INJECT)
    with pytest.raises(AssertionError):
        _check_fp8(m, o, fix["out"])


def test_fp8_sub_batch_graph_replay_and_switching_off(lib_built):
    fix = load_golden("tiny_b6")
    m = build_filled_model(fix, "bf16", "cuda")
    i = fix["inputs"]
    fresh = m.engine().forward(i["x"], i["vision"], i["polygon"], i["poly_len"], i["input_ids"], i["attention_mask"])["decoded"].clone()
    m.fp8_backbone_for_inference()
    e = m.engine()
    full = e.forward(i["x"], i["vision"], i["polygon"], i["poly_len"], i["input_ids"], i["attention_mask"], keep_intermediates=True)
    sub = e.forward(i["x"][2:5], i["vision"][2:5], i["polygon"][2:5], i["poly_len"][2:5], i["input_ids"][2:5], i["attention_mask"][2:5],
                    keep_intermediates=True)
    assert torch.equal(full["decoded"][2:5], sub["decoded"]) and torch.equal(full["final_hidden"][2:5], sub["final_hidden"])
    assert not torch.equal(full["decoded"], fresh)               # the option is live
    lens = torch.tensor(i["poly_len"], dtype=torch.int32)
    args = [t.cuda() for t in (i["x"], i["vision"], i["polygon"], lens, i["y"], torch.tensor(i["norm_stat"]), i["input_ids"], i["attention_mask"])]
    eager = m.predict_with_metrics(*args, max_poly_len=64)["decoded"].clone()
    for _ in range(2):
        got = m.predict_with_metrics(*args, max_poly_len=64, cuda_graph=True)["decoded"]
        torch.cuda.synchronize()
        assert torch.equal(got, eager)
    m.fp8_backbone_for_inference(False)
    off = m.engine().forward(i["x"], i["vision"], i["polygon"], i["poly_len"], i["input_ids"], i["attention_mask"])["decoded"]
    assert torch.equal(off, fresh)


def test_train_step_ignores_the_fp8_option(lib_built):
    """A train-mode step runs on the bf16 fine-tune engine whatever the serving option says.  (Two identical steps are not bit-identical
    to each other — the backward's fp32 atomics reorder — so the gradients are compared within that run-to-run noise.)"""
    fix = load_golden("tiny_b6")
    i = fix["inputs"]

    def grads(fp8):
        m = build_filled_model(fix, "bf16", "cuda").fp8_backbone_for_inference(fp8)
        m.set_dropout(0.0)
        m.train()
        loss, _ = m(i["x"].cuda(), i["vision"].cuda(), None, i["polygon"].cuda(), i["poly_len"], y=i["y"].cuda(), norm_stat=i["norm_stat"],
                    input_ids=i["input_ids"].cuda(), attention_mask=i["attention_mask"].cuda())
        loss.backward()
        torch.cuda.synchronize()
        assert not m.train_engine().fp8 and m._engine is None         # no inference engine was built, the train engine is bf16
        return {n: p.grad.clone() for n, p in m.named_parameters() if p.grad is not None}
    a, b, a2 = grads(False), grads(True), grads(False)
    assert a.keys() == b.keys() and len(a) > 0
    for k in a:
        noise = float((a2[k] - a[k]).abs().max())
        assert float((b[k] - a[k]).abs().max()) <= 4 * noise + 1e-6 * float(a[k].abs().max()), k


def test_fp8_decode_steps_match_the_full_forward(lib_built):
    fix = load_golden("tiny_b6")
    m = build_filled_model(fix, "bf16", "cuda").fp8_backbone_for_inference()
    eng = m.engine()
    i = fix["inputs"]
    H = eng.llm["H"]
    pre = eng.prefix_embeds(i["vision"][:2], i["input_ids"][:2, :9])
    extra = eng.token_embeds(i["input_ids"][:2, 9:12])
    full = torch.cat([pre, extra], 1).contiguous()
    P, Lf = pre.shape[1], full.shape[1]
    ones = torch.ones(2, Lf, dtype=torch.int32, device="cuda")
    want = eng.llm_forward(full.clone(), ones, 2, Lf).view(2, Lf, H).float().cpu()
    caches = []
    got0 = eng.llm_forward(pre.clone(), ones[:, :P].contiguous(), 2, P, kv_out=(caches, Lf)).view(2, P, H).float().cpu()
    # a decode step quantises one row at a time (same per-row scales and e4m3 operands); attention over a different key count and the
    # one-row GEMM routes reorder fp32 sums, hence the bf16 tolerance pattern of test_generate_gpu.py
    ht = dict(rtol=4e-2, atol=4e-2 * float(want.abs().max()))
    torch.testing.assert_close(got0, want[:, :P], **ht)
    for j in range(3):
        h = eng.llm_decode_step(extra[:, j].contiguous(), caches, P + j).float().cpu()
        torch.testing.assert_close(h, want[:, P + j], **ht)
