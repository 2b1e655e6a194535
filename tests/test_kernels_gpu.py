"""Per-kernel parity: every C-ABI entry point against the CPU oracle (oracle/restated.py) on seeded inputs.
fp32 paths: rtol 1e-4 (the north-star fp32 tolerance); bf16 paths: compared with the oracle run on the
bf16-rounded inputs, so only accumulation order / output rounding differ."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import restated as R  # noqa: E402


@pytest.fixture(scope="module")
def ops(lib_built):
    from tcavp_b200 import ops as o
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    sm, major, _ = o.device_info()
    assert major == 10, f"libtcavp is built for sm_100a only (device is cc {major}.x)"
    return o


def _rand(*shape, seed=0, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(*shape, generator=g) * scale


DEV = "cuda"

GEMM_SHAPES = [(1, 16, 64), (100, 24, 72), (128, 64, 64), (300, 100, 136), (257, 256, 768), (1000, 600, 200),
               (130, 2304, 784), (64, 1600, 64), (515, 64, 1600), (384, 6144, 768), (200, 768, 3072)]


@pytest.mark.parametrize("M,N,K", GEMM_SHAPES)
@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_gemm_plain(ops, M, N, K, dtype):
    td = torch.float32 if dtype == "fp32" else torch.bfloat16
    a, w = _rand(M, K, seed=1).to(td), _rand(N, K, seed=2, scale=K ** -0.5).to(td)
    want = a.float() @ w.float().t()
    out = torch.empty(M, N, dtype=torch.float32, device=DEV)
    ops.gemm(a.to(DEV), w.to(DEV), out)
    torch.testing.assert_close(out.cpu(), want, rtol=1e-4, atol=1e-4)


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("act", ["none", "relu", "swiglu", "gelu_tanh"])
def test_gemm_epilogue(ops, dtype, act):
    td = torch.float32 if dtype == "fp32" else torch.bfloat16
    M, N, K = 333, 200, 136
    a, w = _rand(M, K, seed=3).to(td), _rand(N, K, seed=4, scale=K ** -0.5).to(td)
    No = N // 2 if act == "swiglu" else N
    bias = _rand(No, seed=5)
    res = _rand(M, No, seed=6).to(td)
    acc = a.float() @ w.float().t()
    if act == "swiglu":
        want = torch.nn.functional.silu(acc[:, 0::2]) * acc[:, 1::2] + bias
    else:
        want = acc + bias
        if act == "relu":
            want = torch.relu(want)
        elif act == "gelu_tanh":            # HF ACT2FN["gelu_new"] (GPT-2 mlp.c_fc)
            want = torch.nn.functional.gelu(want, approximate="tanh")
    want = want + res.float()
    for out_dtype in (torch.float32, td):
        out = torch.empty(M, No, dtype=out_dtype, device=DEV)
        ops.gemm(a.to(DEV), w.to(DEV), out, bias=bias.to(DEV), residual=res.to(DEV),
                 act={"none": ops.ACT_NONE, "relu": ops.ACT_RELU, "swiglu": ops.ACT_SWIGLU, "gelu_tanh": ops.ACT_GELU_TANH}[act])
        tol = dict(rtol=1e-4, atol=1e-4) if out_dtype == torch.float32 else dict(rtol=1e-2, atol=1e-2)
        if act == "gelu_tanh" and dtype == "bf16" and out_dtype == torch.float32:
            tol = dict(rtol=2e-3, atol=2e-3)      # bf16 operands use the hardware tanh (relative error ~2^-11) whatever the output dtype
        torch.testing.assert_close(out.float().cpu(), want, **tol)


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_gemm_inplace_residual_strided_and_remap(ops, dtype):
    td = torch.float32 if dtype == "fp32" else torch.bfloat16
    # in-place residual (o_proj / down_proj pattern)
    M, N, K = 260, 128, 64
    a, w, x = _rand(M, K, seed=7).to(td), _rand(N, K, seed=8, scale=0.1).to(td), _rand(M, N, seed=9).to(td)
    xd = x.to(DEV)
    ops.gemm(a.to(DEV), w.to(DEV), xd, residual=xd)
    torch.testing.assert_close(xd.float().cpu(), (a.float() @ w.float().t() + x.float()).to(td).float(), rtol=1e-2, atol=1e-2)
    # K-extension pattern: A has a wider row than K, output lands in the trailing columns of the same buffer
    H, kx = 128, 16
    buf = torch.zeros(M, H + kx, dtype=td)
    buf[:, :H] = _rand(M, H, seed=10).to(td)
    acat = _rand(kx, H, seed=11, scale=H ** -0.5).to(td)
    bd = buf.to(DEV)
    ops.gemm(bd, acat.to(DEV), bd[:, H:], M=M, N=kx, K=H, lda=H + kx, ldo=H + kx)
    want = buf[:, :H].float() @ acat.float().t()
    torch.testing.assert_close(bd[:, H:].float().cpu(), want.to(td).float(), rtol=1e-2, atol=1e-2)
    torch.testing.assert_close(bd[:, :H].cpu(), buf[:, :H])
    # row remap: 16 rows per scene scattered into rows [0,16) of a (B, L, H) buffer
    B, Q, L = 5, 16, 40
    t, wq = _rand(B * Q, 64, seed=12).to(td), _rand(H, 64, seed=13, scale=0.125).to(td)
    fused = torch.full((B, L, H), 7.0, dtype=td, device=DEV)
    ops.gemm(t.to(DEV), wq.to(DEV), fused, remap=(Q, L, 0), ldo=H)
    want = (t.float() @ wq.float().t()).view(B, Q, H)
    torch.testing.assert_close(fused[:, :Q].float().cpu(), want.to(td).float(), rtol=1e-2, atol=1e-2)
    assert (fused[:, Q:] == 7.0).all()


def test_gemm_rejects_bad_arguments(ops):
    from tcavp_b200.lib import TcavpError
    a = torch.zeros(4, 12, dtype=torch.bfloat16, device=DEV)
    with pytest.raises(TcavpError, match="multiples of 8"):
        ops.gemm(a, torch.zeros(8, 12, dtype=torch.bfloat16, device=DEV), torch.zeros(4, 8, device=DEV))
    with pytest.raises(TcavpError, match="CUDA tensors"):
        ops.gemm(torch.zeros(4, 8), torch.zeros(8, 8), torch.zeros(4, 8))
    out = torch.zeros(0, 8, device=DEV)
    ops.gemm(torch.zeros(0, 8, device=DEV), torch.zeros(8, 8, device=DEV), out, M=0)   # empty batch is a no-op


def _attn_ref(q, k, v, scale, causal, key_mask):
    # q (B,Tq,H,dh) k/v (B,Tk,Hkv,dh)
    B, Tq, H, dh = q.shape
    Hkv = k.shape[2]
    k = k.repeat_interleave(H // Hkv, dim=2)
    v = v.repeat_interleave(H // Hkv, dim=2)
    s = torch.einsum("bihd,bjhd->bhij", q, k) * scale
    if causal:
        s = s.masked_fill(~torch.tril(torch.ones(Tq, k.shape[1], dtype=torch.bool)), float("-inf"))
    if key_mask is not None:
        s = s.masked_fill(~key_mask.bool()[:, None, None, :], float("-inf"))
    p = torch.nan_to_num(torch.softmax(s, dim=-1), nan=0.0)
    return torch.einsum("bhij,bjhd->bihd", p, v)


ATTN_CASES = [
    # B, H, Hkv, Tq, Tk, dh, causal, masked
    (3, 4, 4, 64, 64, 16, False, True),     # lane polygon encoder
    (2, 8, 8, 15, 15, 96, False, False),    # Q-Former encoder
    (2, 8, 8, 16, 15, 96, False, False),    # Q-Former decoder cross
    (3, 2, 2, 15, 15, 32, False, False),    # LTSF attn block
    (2, 2, 2, 25, 144, 384, False, False),  # LTSF cross-attn, H=768
    (1, 2, 2, 25, 40, 2048, False, False),  # LTSF cross-attn, H=4096
    (3, 2, 2, 50, 144, 384, False, True),   # LTSF cross-attn, 50-step horizon (cfg5), with a key mask incl. an empty row
    (2, 2, 2, 64, 250, 384, False, False),  # widest supported few-query shape
    (2, 2, 2, 12, 30, 384, False, False),   # fewer queries than one padded m-tile pair
    (2, 12, 12, 144, 144, 64, True, True),  # LLM 768-class
    (2, 4, 2, 40, 40, 32, True, True),      # tiny GQA
    (1, 8, 2, 70, 70, 128, True, True),     # 7B-style head_dim with GQA
    # tcgen05 / TMEM kernel (attention_tm.cu): causal, head_dim 64 / 128, 128 <= L <= 256
    (3, 12, 12, 144, 144, 64, True, True),  # L = 144: tile A = rows 16..143, tile B = rows 0..15; ragged key masks
    (2, 8, 2, 144, 144, 128, True, True),   # 7B head_dim, GQA, two 64-column boxes per operand
    (2, 4, 4, 128, 128, 64, True, False),   # exactly one tile
    (2, 4, 2, 160, 160, 64, True, True),    # 32-row tile B
    (1, 4, 4, 256, 256, 64, True, True),    # both tiles full
    (2, 2, 2, 136, 136, 64, True, True),    # L not a multiple of 16: padded key columns / query rows come from the next scene
    (2, 2, 1, 176, 176, 128, True, False),  # head_dim 128 with a 48-row tile B
]


@pytest.mark.parametrize("B,H,Hkv,Tq,Tk,dh,causal,masked", ATTN_CASES)
@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_attention(ops, B, H, Hkv, Tq, Tk, dh, causal, masked, dtype):
    td = torch.float32 if dtype == "fp32" else torch.bfloat16
    q, k, v = _rand(B, Tq, H, dh, seed=1).to(td), _rand(B, Tk, Hkv, dh, seed=2).to(td), _rand(B, Tk, Hkv, dh, seed=3).to(td)
    km = None
    if masked:
        lens = torch.tensor([Tk, max(1, Tk // 2), 0][:B]) if not causal else torch.tensor([Tk, max(1, Tk // 2), 3][:B])
        km = (torch.arange(Tk)[None, :] < lens[:, None]).int()
    want = _attn_ref(q.float(), k.float(), v.float(), dh ** -0.5, causal, km)
    out = torch.empty(B, Tq, H, dh, dtype=td, device=DEV)
    ops.attention(q.to(DEV), k.to(DEV), v.to(DEV), out, B=B, H=H, Hkv=Hkv, Tq=Tq, Tk=Tk, dh=dh, q_strides=(Tq * H * dh, H * dh),
                  k_strides=(Tk * Hkv * dh, Hkv * dh), v_strides=(Tk * Hkv * dh, Hkv * dh), o_strides=(Tq * H * dh, H * dh),
                  scale=dh ** -0.5, causal=causal, key_mask=None if km is None else km.to(DEV))
    tol = dict(rtol=1e-4, atol=1e-5) if dtype == "fp32" else dict(rtol=2e-2, atol=2e-2)
    torch.testing.assert_close(out.float().cpu(), want, **tol)


@pytest.mark.parametrize("B,Tq,Tk,dh", [
    (5, 25, 144, 768),      # cfg2: 25-step horizon against the 144-token fused sequence, 768-class hidden size
    (300, 50, 144, 768),    # cfg5: 50-step horizon, more scenes than SMs (two items per CTA: accumulator-buffer parities, ring wrap-around)
    (3, 64, 256, 256),      # full query tile, widest key tile (TMEM columns 0..511 all used), two output chunks
    (150, 12, 40, 128),     # one output chunk per scene (the running chunk counter alternates buffers across scenes), Tk not a multiple of 16
    (2, 25, 144, 4096),     # 7B-class hidden size: 64 phase-1 stages and 32 output chunks per scene
])
def test_cross_attention_tcgen05_two_heads_on_a_shared_kv_head(ops, B, Tq, Tk, dh):
    """The absorbed fusion cross-attention (engine.py: Engine._absorb_cross; reference train.py:793-798): two query heads of width dh
    against keys = values = the backbone output, attention_xt.cu (tcgen05 / TMEM / TMA)."""
    q = (_rand(B, Tq, 2, dh, seed=11) * 0.5).bfloat16()
    x = _rand(B, Tk, 1, dh, seed=12).bfloat16()
    scale = (dh // 2) ** -0.5 / 8
    want = _attn_ref(q.float(), x.float(), x.float(), scale, False, None)
    xd = x.to(DEV)
    out = torch.full((B, Tq, 2, dh), float("nan"), dtype=torch.bfloat16, device=DEV)
    n0 = ops.launch_count()
    ops.attention(q.to(DEV), xd, xd, out, B=B, H=2, Hkv=1, Tq=Tq, Tk=Tk, dh=dh, q_strides=(Tq * 2 * dh, 2 * dh), k_strides=(Tk * dh, dh),
                  v_strides=(Tk * dh, dh), o_strides=(Tq * 2 * dh, 2 * dh), scale=scale)
    assert ops.launch_count() == n0 + 1 and ops.last_kernel() == "attn_xt_kernel"      # not the mma.sync fallback
    torch.testing.assert_close(out.float().cpu(), want, rtol=2e-2, atol=2e-2)
    # the rows of the padded 64-row query tiles are never stored: a guard band behind the output stays untouched
    guard = torch.full((B * Tq + 8, 2 * dh), 7.0, dtype=torch.bfloat16, device=DEV)
    ops.attention(q.to(DEV), xd, xd, guard, B=B, H=2, Hkv=1, Tq=Tq, Tk=Tk, dh=dh, q_strides=(Tq * 2 * dh, 2 * dh), k_strides=(Tk * dh, dh),
                  v_strides=(Tk * dh, dh), o_strides=(Tq * 2 * dh, 2 * dh), scale=scale)
    assert bool((guard[B * Tq:] == 7.0).all())
    torch.testing.assert_close(guard[:B * Tq].view(B, Tq, 2, dh).float().cpu(), want, rtol=2e-2, atol=2e-2)


@pytest.mark.parametrize("nh,nkv,dh,B", [(12, 12, 64, 160), (32, 8, 128, 20)])
def test_llm_attention_tcgen05_on_the_packed_qkv_layout(ops, nh, nkv, dh, B, tmp_path):
    """The engine's call: q / k / v are column slices of one packed [B L, (nh + 2 nkv) dh] activation, more (scene, head) items than
    SMs (persistent loop, both stages of the TMA ring), ragged key masks — against the reference and against the mma.sync kernel."""
    import os
    import subprocess
    L = 144
    nq, nk = nh * dh, nkv * dh
    g = torch.Generator().manual_seed(nh)
    qkv = (torch.randn(B * L, nq + 2 * nk, generator=g) * 0.7).to(torch.bfloat16)
    lens = torch.randint(100, L + 1, (B,), generator=g)
    km = (torch.arange(L)[None, :] < lens[:, None]).int()
    n_ref = 3                                             # the reference on a few scenes only (host)
    q, k, v = (t.float().view(B, L, -1, dh) for t in (qkv[:, :nq], qkv[:, nq:nq + nk], qkv[:, nq + nk:]))
    want = _attn_ref(q[:n_ref], k[:n_ref], v[:n_ref], dh ** -0.5, True, km[:n_ref])
    d = qkv.to(DEV)
    out = torch.empty(B * L, nq, dtype=torch.bfloat16, device=DEV)
    n0 = ops.launch_count()
    ops.attention(d, d[:, nq:], d[:, nq + nk:], out, B=B, H=nh, Hkv=nkv, Tq=L, Tk=L, dh=dh, q_strides=(L * (nq + 2 * nk), nq + 2 * nk),
                  k_strides=(L * (nq + 2 * nk), nq + 2 * nk), v_strides=(L * (nq + 2 * nk), nq + 2 * nk), o_strides=(L * nq, nq), scale=dh ** -0.5,
                  causal=True, key_mask=km.to(DEV))
    assert ops.launch_count() - n0 == 1
    got = out.float().cpu().view(B, L, nh, dh)
    torch.testing.assert_close(got[:n_ref], want, rtol=2e-2, atol=2e-2)
    # every scene against the mma.sync kernel (TCAVP_ATTN_TCGEN05=0 is read once per process: ask a child process)
    path = str(tmp_path)
    torch.save(dict(qkv=qkv, km=km, nh=nh, nkv=nkv, dh=dh, B=B, L=L), os.path.join(path, "attn_ab_in.pt"))
    code = ("import sys, torch; sys.path.insert(0, %r); import tcavp_b200 as T; from tcavp_b200 import ops\n"
            "z = torch.load(%r); d = z['qkv'].cuda(); nh, nkv, dh, B, L = z['nh'], z['nkv'], z['dh'], z['B'], z['L']; nq, nk = nh * dh, nkv * dh\n"
            "out = torch.empty(B * L, nq, dtype=torch.bfloat16, device='cuda'); s = (L * (nq + 2 * nk), nq + 2 * nk)\n"
            "ops.attention(d, d[:, nq:], d[:, nq + nk:], out, B=B, H=nh, Hkv=nkv, Tq=L, Tk=L, dh=dh, q_strides=s, k_strides=s, v_strides=s, "
            "o_strides=(L * nq, nq), scale=dh ** -0.5, causal=True, key_mask=z['km'].cuda())\n"
            "torch.save(out.cpu(), %r)\n") % (os.path.dirname(os.path.dirname(os.path.abspath(__file__))), os.path.join(path, "attn_ab_in.pt"),
                                              os.path.join(path, "attn_ab_out.pt"))
    import sys
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, TCAVP_ATTN_TCGEN05="0"), capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    old = torch.load(os.path.join(path, "attn_ab_out.pt")).float().view(B, L, nh, dh)
    torch.testing.assert_close(got, old, rtol=2e-2, atol=2e-2)


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("rows,cols", [(37, 64), (20, 768), (5, 4096), (9, 100)])
def test_norms(ops, dtype, rows, cols):
    td = torch.float32 if dtype == "fp32" else torch.bfloat16
    x, r = _rand(rows, cols, seed=1).to(td), _rand(rows, cols, seed=2).to(td)
    w, b = 1 + 0.1 * _rand(cols, seed=3), 0.1 * _rand(cols, seed=4)
    tol = dict(rtol=1e-4, atol=1e-5) if dtype == "fp32" else dict(rtol=1e-2, atol=1e-2)
    out = ops.layernorm(x.to(DEV), w.to(DEV), b.to(DEV), torch.empty(rows, cols, dtype=td, device=DEV), residual=r.to(DEV))
    torch.testing.assert_close(out.float().cpu(), R.layer_norm(x.float() + r.float(), w, b), **tol)
    out = ops.layernorm(x.to(DEV), w.to(DEV), b.to(DEV), torch.empty(rows, cols, dtype=torch.float32, device=DEV))
    torch.testing.assert_close(out.cpu(), R.layer_norm(x.float(), w, b), rtol=1e-4, atol=1e-5)
    wide = torch.zeros(rows, cols + 16, dtype=td, device=DEV)
    ops.rmsnorm(x.to(DEV), w.to(DEV), wide, eps=1e-6, rows=rows, cols=cols, ldo=cols + 16)
    torch.testing.assert_close(wide[:, :cols].float().cpu(), R.rms_norm(x.float(), w, 1e-6), **tol)
    assert (wide[:, cols:] == 0).all()


def test_layernorm_remap_rowvec(ops):
    B, Q, L, H = 3, 16, 24, 64
    x, w, b, vec = _rand(B * Q, H, seed=1), 1 + 0.1 * _rand(H, seed=2), 0.1 * _rand(H, seed=3), _rand(H, seed=4)
    fused = torch.zeros(B, L, H, device=DEV)
    ops.layernorm(x.to(DEV), w.to(DEV), b.to(DEV), fused, remap=(Q, L, 0), rowvec=vec.to(DEV))
    torch.testing.assert_close(fused[:, :Q].cpu(), (R.layer_norm(x, w, b) + vec).view(B, Q, H), rtol=1e-4, atol=1e-5)
    assert (fused[:, Q:] == 0).all()


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("rows,cols,ldo", [(1000, 768, 776), (37, 128, 136), (300, 512, 512), (9, 40, 44), (5000, 1024, 1040)])
def test_layernorm_strided(ops, dtype, rows, cols, ldo):
    """LayerNorm written into the leading columns of a wider operand (GPT-2 path: ln_1(x) -> [ln_1(x) | LoRA side columns]): the bulk-copy
    kernel (bf16, 256..1024 columns) and the element-wise one; the columns past `cols` are left alone."""
    td = torch.float32 if dtype == "fp32" else torch.bfloat16
    x = (_rand(rows, cols, seed=21) * 1.5 + 0.2).to(td)
    w, b = 1 + 0.1 * _rand(cols, seed=22), 0.1 * _rand(cols, seed=23)
    out = torch.full((rows, ldo), 5.0, dtype=td, device=DEV)
    ops.layernorm_strided(x.to(DEV), w.to(DEV), b.to(DEV), out, rows=rows, cols=cols, eps=1e-5, ldo=ldo)
    tol = dict(rtol=1e-4, atol=1e-4) if dtype == "fp32" else dict(rtol=2e-2, atol=2e-2)
    torch.testing.assert_close(out[:, :cols].float().cpu(), R.layer_norm(x.float(), w, b), **tol)
    assert bool((out[:, cols:] == 5.0).all())


@pytest.mark.parametrize("rows,cols,out_dtype,remap", [(65536 + 37, 768, "bf16", False), (70001, 512, "fp32", False), (65536, 1024, "bf16", False),
                                                       (66000, 256, "bf16", True)])
def test_layernorm_many_bf16_rows_through_the_bulk_copy_ring(ops, rows, cols, out_dtype, remap):
    """>= 65536 bf16 rows take layernorm_pipe_kernel (rows staged through shared memory by cp.async.bulk, four rows in flight per warp):
    row counts that leave the last ring slots of some warps empty, every column class, both output dtypes, row remap + row vector."""
    g = torch.Generator().manual_seed(5)
    x = (torch.randn(rows, cols, generator=g) * 2 + 0.3 * torch.randn(rows, 1, generator=g)).bfloat16()
    w, b = 1 + 0.1 * _rand(cols, seed=6), 0.1 * _rand(cols, seed=7)
    od = torch.bfloat16 if out_dtype == "bf16" else torch.float32
    want = R.layer_norm(x.float(), w, b)
    tol = dict(rtol=2e-2, atol=2e-2) if out_dtype == "bf16" else dict(rtol=1e-4, atol=1e-4)
    if remap:
        gi, go = 16, 24                                   # rows of 16-row groups land in 24-row groups (the Q-Former -> fused-sequence scatter)
        vec = _rand(cols, seed=8)
        n_groups = rows // gi
        rows = n_groups * gi
        out = torch.zeros(n_groups * go, cols, dtype=od, device=DEV)
        ops.layernorm(x[:rows].to(DEV), w.to(DEV), b.to(DEV), out, remap=(gi, go, 0), rowvec=vec.to(DEV), rows=rows, cols=cols)
        got = out.view(n_groups, go, cols)
        torch.testing.assert_close(got[:, :gi].float().cpu(), (want[:rows] + vec).view(n_groups, gi, cols), **tol)
        assert bool((got[:, gi:] == 0).all())
        return
    out = torch.empty(rows, cols, dtype=od, device=DEV)
    ops.layernorm(x.to(DEV), w.to(DEV), b.to(DEV), out)
    torch.testing.assert_close(out.float().cpu(), want, **tol)


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("nh,nkv,dh,theta", [(12, 12, 64, 10000.0), (4, 2, 32, 10000.0), (8, 2, 128, 500000.0)])
def test_rope(ops, dtype, nh, nkv, dh, theta):
    td = torch.float32 if dtype == "fp32" else torch.bfloat16
    B, L = 2, 144
    ld = (nh + 2 * nkv) * dh
    qkv = _rand(B * L, ld, seed=1).to(td)
    cos, sin = R.rope_cos_sin(L, dh, theta)
    table = ops.rope_table(L, dh, theta, DEV)
    torch.testing.assert_close(table[..., 0].cpu(), cos[:, : dh // 2], rtol=0, atol=2e-6)
    torch.testing.assert_close(table[..., 1].cpu(), sin[:, : dh // 2], rtol=0, atol=2e-6)
    q = qkv[:, : nh * dh].float().view(B, L, nh, dh)
    k = qkv[:, nh * dh:(nh + nkv) * dh].float().view(B, L, nkv, dh)
    c, s = cos[None, :, None, :], sin[None, :, None, :]
    wq, wk = q * c + R.rotate_half(q) * s, k * c + R.rotate_half(k) * s
    d = qkv.to(DEV)
    ops.rope_(d, rows=B * L, L=L, ld=ld, n_q_heads=nh, n_k_heads=nkv, dh=dh, table=table)
    tol = dict(rtol=1e-4, atol=1e-5) if dtype == "fp32" else dict(rtol=1e-2, atol=2e-2)
    torch.testing.assert_close(d[:, : nh * dh].float().cpu().view(B, L, nh, dh), wq, **tol)
    torch.testing.assert_close(d[:, nh * dh:(nh + nkv) * dh].float().cpu().view(B, L, nkv, dh), wk, **tol)
    torch.testing.assert_close(d[:, (nh + nkv) * dh:].cpu(), qkv[:, (nh + nkv) * dh:])   # v untouched


def test_embed_text_cast_rowvec(ops):
    B, Lt, Q, H, V = 3, 10, 16, 64, 50
    ids = torch.randint(0, V, (B, Lt), generator=torch.Generator().manual_seed(1))
    am = (torch.arange(Lt)[None, :] < torch.tensor([10, 4, 1])[:, None]).long()
    emb, tm = _rand(V, H, seed=2), _rand(H, seed=3)
    fused = torch.zeros(B, Q + Lt, H, device=DEV)
    mask = torch.zeros(B, Q + Lt, dtype=torch.int32, device=DEV)
    ops.embed_text(ids.to(DEV), am.to(DEV), emb.to(DEV), tm.to(DEV), fused, mask, B=B, L_text=Lt, n_img=Q, H=H)
    torch.testing.assert_close(fused[:, Q:].cpu(), emb[ids] + tm)
    assert (fused[:, :Q] == 0).all()
    assert torch.equal(mask.cpu(), torch.cat([torch.ones(B, Q, dtype=torch.int32), am.int()], 1))
    q = _rand(Q, H, seed=4)
    out = ops.cast(q.to(DEV), torch.empty(B * Q, H, dtype=torch.bfloat16, device=DEV), rows=B * Q, cols=H, in_row_mod=Q)
    torch.testing.assert_close(out.float().cpu(), q.bfloat16().float().repeat(B, 1))
    x = _rand(B * Q, H, seed=5)
    o2 = torch.zeros(B, Q + Lt, H, device=DEV)
    ops.add_rowvec(x.to(DEV), tm.to(DEV), o2, rows=B * Q, cols=H, remap=(Q, Q + Lt, 0))
    torch.testing.assert_close(o2[:, :Q].cpu(), (x + tm).view(B, Q, H))


@pytest.mark.parametrize("B,P,D", [(4, 64, 64), (4, 48, 64), (4, 64, 6)])      # 16-byte path (D % 4 == 0, fp32 out) and the element-wise one
def test_poly_embed_and_masked_mean(ops, B, P, D):
    poly = torch.rand(B, P, 2, generator=torch.Generator().manual_seed(1)) * 1000
    lens = torch.tensor([0, P, 1, 33], dtype=torch.int32)
    w, b, pos = _rand(D, 2, seed=2, scale=0.01), _rand(D, seed=3), _rand(P, D, seed=4)
    out = torch.empty(B * P, D, device=DEV)
    km = torch.empty(B, P, dtype=torch.int32, device=DEV)
    ops.poly_embed(poly.to(DEV), lens.to(DEV), w.to(DEV), b.to(DEV), pos.to(DEV), out, km, B=B, P=P, D=D)
    want = poly @ w.t() + b + pos
    torch.testing.assert_close(out.cpu().view(B, P, D), want, rtol=1e-5, atol=1e-4)
    assert torch.equal(km.cpu(), (torch.arange(P)[None, :] < lens[:, None]).int())
    mm = ops.masked_mean(out, lens.to(DEV), torch.empty(B, D, device=DEV), B=B, P=P, D=D).cpu()
    for i, n in enumerate(lens.tolist()):
        ref = want[i, :n].mean(0) if n > 0 else torch.zeros(D)
        torch.testing.assert_close(mm[i], ref, rtol=1e-4, atol=1e-3)


def _ltsf_sd(C, T, To, seed=0):
    sd = {"ltsf.token_proj.weight": _rand(C, 2, 1, seed=seed + 1), "ltsf.token_proj.bias": _rand(C, seed=seed + 2),
          "ltsf.pos_encoding": _rand(1, C, T, seed=seed + 3, scale=0.1)}
    for i in range(C):
        sd[f"ltsf.nlinear_encoder.encoder_linears.{i}.weight"] = _rand(T, T, seed=seed + 10 + i, scale=T ** -0.5)
        sd[f"ltsf.nlinear_encoder.encoder_linears.{i}.bias"] = _rand(T, seed=seed + 100 + i, scale=0.1)
        sd[f"ltsf.decoder.decoder_linears.{i}.weight"] = _rand(To, T, seed=seed + 200 + i, scale=T ** -0.5)
        sd[f"ltsf.decoder.decoder_linears.{i}.bias"] = _rand(To, seed=seed + 300 + i, scale=0.1)
    return sd


@pytest.mark.parametrize("T,To", [(15, 25), (6, 12), (30, 30), (18, 30), (10, 20), (20, 50), (15, 50)])
def test_ltsf_encode_and_nlinear_decode(ops, T, To):
    B, C = 7, 64
    sd = _ltsf_sd(C, T, To)
    x = torch.rand(B, 2, T, generator=torch.Generator().manual_seed(5))
    want = R.ltsf_encoder(sd, x)                                    # (B, C, T)
    we, be = R.stack_individual(sd, "ltsf.nlinear_encoder.encoder_linears.", C)
    enc = torch.empty(B, T, C, device=DEV)
    ops.ltsf_encode(x.to(DEV), sd["ltsf.token_proj.weight"][:, :, 0].contiguous().to(DEV), sd["ltsf.token_proj.bias"].to(DEV),
                    we.permute(1, 2, 0).contiguous().to(DEV), be.t().contiguous().to(DEV),
                    sd["ltsf.pos_encoding"][0].t().contiguous().to(DEV), enc, B=B, F=2, C=C, T_in=T)
    torch.testing.assert_close(enc.cpu().permute(0, 2, 1), want, rtol=1e-4, atol=1e-5)
    wd, bd = R.stack_individual(sd, "ltsf.decoder.decoder_linears.", C)
    adj = _rand(B, To, C, seed=9)
    last = want[:, :, -1:]
    wdec = torch.einsum("cot,bct->bco", wd, want - last) + bd[None] + last + adj.permute(0, 2, 1)
    dec = torch.empty(B, To, C, device=DEV)
    ops.nlinear_decode(enc, wd.permute(1, 2, 0).contiguous().to(DEV), bd.t().contiguous().to(DEV), adj.to(DEV), dec, B=B, C=C, T_in=T, T_out=To)
    torch.testing.assert_close(dec.cpu().permute(0, 2, 1), wdec, rtol=1e-4, atol=1e-5)


@pytest.mark.parametrize("tc", [False, True])
@pytest.mark.parametrize("B,To", [(5, 25), (300, 50), (1, 1), (1300, 50), (9, 7)])
def test_fusion_head_and_metrics(ops, B, To, tc):
    """`tc`: the split-bf16 tensor-core kernel of the bf16 compute mode (fusion_head_tc_kernel) — held to the same fp32-class tolerance
    as the exact FFMA kernel; 1300 scenes = more 8-scene groups than resident CTAs (the grid-stride loop), (9, 7) = a ragged last group."""
    C, T = 64, 15
    fused = _rand(B * To, C, seed=1)
    p = "ltsf.decoder."
    sd = {p + "fusion_layer.0.weight": 1 + 0.1 * _rand(C, seed=2), p + "fusion_layer.0.bias": 0.1 * _rand(C, seed=3),
          p + "fusion_layer.1.weight": _rand(C, C, seed=4, scale=0.125), p + "fusion_layer.1.bias": 0.1 * _rand(C, seed=5),
          p + "fusion_layer.3.weight": _rand(C, C, seed=6, scale=0.125), p + "fusion_layer.3.bias": 0.1 * _rand(C, seed=7),
          p + "out_proj.weight": _rand(2, C, seed=8, scale=0.125), p + "out_proj.bias": 0.1 * _rand(2, seed=9)}
    x = torch.rand(B, 2, T, generator=torch.Generator().manual_seed(10))
    y = torch.rand(B, 2, To, generator=torch.Generator().manual_seed(11))
    g = torch.Generator().manual_seed(12)
    mn = torch.rand(B, 2, generator=g) * 2000
    ns = torch.stack([mn[:, 0], mn[:, 0] + 100 + 1400 * torch.rand(B, generator=g), mn[:, 1], mn[:, 1] + 5 + 75 * torch.rand(B, generator=g)], 1)
    f = R.layer_norm(fused, sd[p + "fusion_layer.0.weight"], sd[p + "fusion_layer.0.bias"])
    f = R.linear(torch.relu(R.linear(f, sd[p + "fusion_layer.1.weight"], sd[p + "fusion_layer.1.bias"])), sd[p + "fusion_layer.3.weight"], sd[p + "fusion_layer.3.bias"])
    want = R.linear(f, sd[p + "out_proj.weight"], sd[p + "out_proj.bias"]).view(B, To, 2).permute(0, 2, 1) + x[:, :, -1:]
    dv = {k: v.to(DEV) for k, v in sd.items()}
    decoded = torch.empty(B, 2, To, device=DEV)
    metrics = torch.zeros(8, device=DEV)
    per = torch.empty(B, 2, device=DEV)
    ops.fusion_head(fused.to(DEV), dv[p + "fusion_layer.0.weight"], dv[p + "fusion_layer.0.bias"], dv[p + "fusion_layer.1.weight"],
                    dv[p + "fusion_layer.1.bias"], dv[p + "fusion_layer.3.weight"], dv[p + "fusion_layer.3.bias"], dv[p + "out_proj.weight"],
                    dv[p + "out_proj.bias"], x.to(DEV), decoded, y=y.to(DEV), norm_stat=ns.to(DEV), metrics=metrics, per_scene=per,
                    B=B, C=C, T_in=T, T_out=To, tensor_cores=tc)
    assert ops.last_kernel() == ("fusion_head_tc_kernel" if tc else "fusion_head_kernel")
    torch.testing.assert_close(decoded.cpu(), want, rtol=1e-4, atol=2e-5 if tc else 1e-5)
    ade, fde = R.ade_fde(want, y, ns)
    loss = R.mse_loss(want, y, ns)
    # de-normalised pixel errors: a 1e-5 coordinate error of the split-bf16 form is 0.015 px on a 1500 px range
    tol = dict(rtol=1e-3, atol=5e-2) if tc else dict(rtol=1e-4, atol=1e-3)
    torch.testing.assert_close(per[:, 0].cpu(), ade, **tol)
    torch.testing.assert_close(per[:, 1].cpu(), fde, **tol)
    m = metrics.cpu()
    torch.testing.assert_close(m[2], ade.sum(), rtol=1e-4, atol=1e-3 * B if tc else 1e-3)
    torch.testing.assert_close(m[3], fde.sum(), rtol=1e-4, atol=1e-3 * B if tc else 1e-3)
    torch.testing.assert_close(m[4], loss, rtol=1e-4, atol=1e-3)
    # standalone metrics kernel on the same prediction
    m2, per2 = torch.zeros(8, device=DEV), torch.empty(B, 2, device=DEV)
    ops.traj_metrics(decoded, y.to(DEV), ns.to(DEV), m2, per2, B=B, T_out=To)
    torch.testing.assert_close(per2.cpu(), per.cpu(), rtol=1e-5, atol=1e-4)
    torch.testing.assert_close(m2[:5].cpu(), m[:5], rtol=1e-4, atol=1e-3)


@pytest.mark.parametrize("M,F", [
    (4096, 2048),        # the lane-polygon encoder: 64 points x 64 scenes, nn.TransformerEncoderLayer's default dim_feedforward
    (256 * 150 + 77, 2048),   # more 256-row steps than SMs (x double buffer, accumulator re-arm across steps) + a ragged last step
    (300, 128),          # a single hidden chunk per step
    (1000, 640),         # five chunks: odd chunk counts flip the barrier parities from step to step
])
def test_ffn64_layernorm_fused(ops, M, F):
    """out = LayerNorm(x + linear2(relu(linear1(x)))) of a d_model = 64 post-norm encoder layer (reference train.py:358) in one tcgen05
    kernel (ffn_tm.cu) against the two-GEMM + LayerNorm form in fp32 on the same bf16 operands."""
    g = torch.Generator().manual_seed(M + F)
    x = torch.randn(M, 64, generator=g).bfloat16()
    w1 = (torch.randn(F, 64, generator=g) * 0.125).bfloat16()
    w2 = (torch.randn(64, F, generator=g) * F ** -0.5).bfloat16()
    b1, b2 = torch.randn(F, generator=g) * 0.1, torch.randn(64, generator=g) * 0.1
    lw, lb = 1 + 0.1 * torch.randn(64, generator=g), 0.1 * torch.randn(64, generator=g)
    h = torch.relu(x.float() @ w1.float().t() + b1).bfloat16().float()          # the kernel feeds the second product bf16 activations
    want = torch.nn.functional.layer_norm((x.float() + h @ w2.float().t() + b2).bfloat16().float(), (64,), lw, lb, 1e-5)
    out = torch.full((M + 4, 64), 9.0, dtype=torch.bfloat16, device=DEV)
    ops.ffn64_ln(x.to(DEV), w1.to(DEV), b1.to(DEV), w2.to(DEV), b2.to(DEV), lw.to(DEV), lb.to(DEV), out[:M], eps=1e-5)
    assert ops.last_kernel() == "ffn64_ln_kernel"
    torch.testing.assert_close(out[:M].float().cpu(), want, rtol=2e-2, atol=2e-2)
    assert bool((out[M:] == 9.0).all())          # rows of the padded last tile are never stored


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("nh,nkv,dh", [(12, 12, 64), (4, 2, 32), (4, 2, 128)])
def test_gemm_fused_rope(ops, dtype, nh, nkv, dh):
    """QKV projection with HF's rotary embedding fused into the epilogue (rotation partners made adjacent by a row
    permutation of W) == plain projection followed by the oracle's apply_rotary_pos_emb, up to that permutation."""
    td = torch.float32 if dtype == "fp32" else torch.bfloat16
    B, L, K = 3, 40, 136
    N = (nh + 2 * nkv) * dh
    x, w = _rand(B * L, K, seed=1).to(td), _rand(N, K, seed=2, scale=K ** -0.5).to(td)
    hp = torch.stack([torch.arange(dh // 2), torch.arange(dh // 2) + dh // 2], dim=1).reshape(-1)
    perm = torch.cat([h * dh + hp for h in range(nh + nkv)] + [torch.arange((nh + nkv) * dh, N)])
    table = ops.rope_table(L, dh, 10000.0, DEV, layout=1)
    out = torch.empty(B * L, N, dtype=torch.float32, device=DEV)
    ops.gemm(x.to(DEV), w[perm].contiguous().to(DEV), out, rope=(table, L, dh, (nh + nkv) * dh))
    y = (x.float() @ w.float().t()).view(B, L, N)
    cos, sin = R.rope_cos_sin(L, dh, 10000.0)
    qk = y[..., : (nh + nkv) * dh].reshape(B, L, nh + nkv, dh)
    qk = qk * cos[None, :, None, :] + R.rotate_half(qk) * sin[None, :, None, :]
    want = torch.cat([qk.reshape(B, L, -1), y[..., (nh + nkv) * dh:]], dim=-1).view(B * L, N)[:, perm]
    torch.testing.assert_close(out.cpu(), want, rtol=1e-4, atol=1e-4)


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_fused_rmsnorm_gemm(ops, dtype):
    """RMSNorm folded into the consuming projection: rstd from tcavp_row_rstd applied as the GEMM's row scale on
    weights pre-multiplied by the norm weight == oracle rms_norm followed by the projection (incl. SwiGLU)."""
    td = torch.float32 if dtype == "fp32" else torch.bfloat16
    M, H, N, kx = 300, 128, 192, 16
    xs = torch.zeros(M, H + kx, dtype=td)
    xs[:, :H] = _rand(M, H, seed=1, scale=3.0).to(td)
    g, w = 1 + 0.1 * _rand(H, seed=2), _rand(N, H, seed=3, scale=H ** -0.5)
    wf = (w * g[None, :]).to(td)
    want = R.rms_norm(xs[:, :H].float(), g, 1e-6) @ w.t()
    d = xs.to(DEV)
    rstd = ops.row_rstd(d, torch.empty(M, device=DEV), rows=M, cols=H, ldx=H + kx, eps=1e-6)
    ref = torch.rsqrt((xs[:, :H].float() ** 2).mean(-1) + 1e-6)
    torch.testing.assert_close(rstd.cpu(), ref, rtol=1e-5, atol=1e-6)
    out = ops.gemm(d, wf.to(DEV), torch.empty(M, N, device=DEV), M=M, K=H, lda=H + kx, row_scale=rstd)
    tol = dict(rtol=1e-4, atol=1e-4) if dtype == "fp32" else dict(rtol=2e-2, atol=2e-2)
    torch.testing.assert_close(out.cpu(), want, **tol)
    out = ops.gemm(d, wf.to(DEV), torch.empty(M, N // 2, device=DEV), M=M, K=H, lda=H + kx, row_scale=rstd, act=ops.ACT_SWIGLU)
    torch.testing.assert_close(out.cpu(), torch.nn.functional.silu(want[:, 0::2]) * want[:, 1::2], **tol)
    o2 = ops.rmsnorm(d, g.to(DEV), torch.empty(M, H, device=DEV), eps=1e-6, rows=M, cols=H, ldi=H + kx)
    torch.testing.assert_close(o2.cpu(), R.rms_norm(xs[:, :H].float(), g, 1e-6), **tol)


# ---- large problems: the CTA-pair (cta_group::2) kernel (M >= 2048, N > 128) and the wide 512 x 256 kernel (K >= 2048, M >= 8192) ----
LARGE = [(4173, 768, 768), (2048, 384, 200), (9000, 512, 2048 + 64), (8192 + 77, 300 + 4, 4096), (16384, 256, 2048)]


@pytest.mark.parametrize("M,N,K", LARGE)
def test_gemm_large_bias_residual(ops, M, N, K):
    a, w = _rand(M, K, seed=1, scale=0.5).bfloat16(), _rand(N, K, seed=2, scale=K ** -0.5).bfloat16()
    bias, res = _rand(N, seed=3), _rand(M, N, seed=4).bfloat16()
    want = a.float() @ w.float().t() + bias + res.float()
    for td in (torch.bfloat16, torch.float32):
        out = torch.full((M, N + 16), float("nan"), dtype=td, device=DEV)
        ops.gemm(a.to(DEV), w.to(DEV), out, bias=bias.to(DEV), residual=res.to(DEV), N=N, ldo=N + 16)
        torch.testing.assert_close(out[:, :N].float().cpu(), want, rtol=2e-2 if td == torch.bfloat16 else 1e-3, atol=2e-2)
        assert torch.isnan(out[:, N:].float()).all()          # nothing written past the logical width
    relu = ops.gemm(a.to(DEV), w.to(DEV), torch.empty(M, N, dtype=torch.bfloat16, device=DEV), bias=bias.to(DEV), act=ops.ACT_RELU)
    torch.testing.assert_close(relu.float().cpu(), torch.relu(a.float() @ w.float().t() + bias), rtol=2e-2, atol=2e-2)


@pytest.mark.parametrize("M,H,I", [(4200, 256, 384), (8300, 2048, 128)])
def test_gemm_large_norm_chain(ops, M, H, I):
    """Decoder sub-block plumbing at kernel-variant sizes: a producer GEMM (+residual) accumulates each output row's sum of squares
    (sumsq_out); the consumer applies rsqrt(sumsq / H + eps) as its row factor (row_sumsq) with the SwiGLU epilogue and stashes the raw
    gate/up accumulators (aux_out) — against oracle rms_norm + projections in fp32."""
    kx = 16
    x0 = _rand(M, H, seed=1).bfloat16()
    w0 = _rand(H, H, seed=2, scale=H ** -0.5).bfloat16()
    g, wgu = 1 + 0.1 * _rand(H, seed=3), _rand(2 * I, H, seed=4, scale=H ** -0.5)
    wf = (wgu * g[None, :]).bfloat16()
    xs = torch.zeros(M, H + kx, dtype=torch.bfloat16, device=DEV)
    xs[:, :H] = x0.to(DEV)
    a = _rand(M, H, seed=5).bfloat16()
    ss = torch.zeros(M, dtype=torch.int64, device=DEV)
    ops.gemm(a.to(DEV), w0.to(DEV), xs[:, :H], ldo=H + kx, residual=xs[:, :H], ldr=H + kx, sumsq_out=ss)       # x1 = x0 + a W0^T (in place)
    x1 = (x0.float() + a.float() @ w0.float().t())
    torch.testing.assert_close(xs[:, :H].float().cpu(), x1, rtol=2e-2, atol=2e-2)
    torch.testing.assert_close(ss.cpu().double().mul(2.0 ** -20).float(), (x1 ** 2).sum(-1), rtol=2e-3, atol=1e-2)
    x1b = xs[:, :H].float().cpu()                                            # the rounded values the consumer actually reads
    aux = torch.empty(M, 2 * I, dtype=torch.bfloat16, device=DEV)
    mid = ops.gemm(xs, wf.to(DEV), torch.empty(M, I, dtype=torch.bfloat16, device=DEV), M=M, K=H, lda=H + kx, act=ops.ACT_SWIGLU,
                   row_sumsq=(ss, H, 1e-6), aux_out=aux)
    rstd = torch.rsqrt((x1 ** 2).mean(-1) + 1e-6)
    gu = (x1b @ wf.float().t()) * rstd[:, None]
    torch.testing.assert_close(aux.float().cpu(), gu, rtol=2e-2, atol=2e-2)
    torch.testing.assert_close(mid.float().cpu(), torch.nn.functional.silu(gu[:, 0::2]) * gu[:, 1::2], rtol=3e-2, atol=2e-2)


def test_gemm_large_fused_rope_and_lora_extension(ops):
    """QKV projection shape of the 768-class backbone at full row count: K-extended rows [x | x A^T] against [W | s B] with RoPE in the
    epilogue of the pair kernel."""
    nh, dh, L, B, H, r = 12, 64, 144, 16, 768, 16
    M, N, Kx = B * L, 3 * nh * dh, H + r
    x = torch.zeros(M, Kx, dtype=torch.bfloat16)
    x[:, :H] = _rand(M, H, seed=1).bfloat16()
    A = _rand(r, H, seed=2, scale=H ** -0.5).bfloat16()
    x[:, H:] = (x[:, :H].float() @ A.float().t()).bfloat16()
    w = torch.cat([_rand(N, H, seed=3, scale=H ** -0.5), _rand(N, r, seed=4, scale=0.1)], dim=1).bfloat16()
    hp = torch.stack([torch.arange(dh // 2), torch.arange(dh // 2) + dh // 2], dim=1).reshape(-1)
    perm = torch.cat([h * dh + hp for h in range(2 * nh)] + [torch.arange(2 * nh * dh, N)])
    table = ops.rope_table(L, dh, 10000.0, DEV, layout=1)
    out = torch.empty(M, N, dtype=torch.bfloat16, device=DEV)
    ops.gemm(x.to(DEV), w[perm].contiguous().to(DEV), out, rope=(table, L, dh, 2 * nh * dh))
    y = (x.float() @ w.float().t()).view(B, L, N)
    cos, sin = R.rope_cos_sin(L, dh, 10000.0)
    qk = y[..., : 2 * nh * dh].reshape(B, L, 2 * nh, dh)
    qk = qk * cos[None, :, None, :] + R.rotate_half(qk) * sin[None, :, None, :]
    want = torch.cat([qk.reshape(B, L, -1), y[..., 2 * nh * dh:]], dim=-1).view(M, N)[:, perm]
    torch.testing.assert_close(out.float().cpu(), want, rtol=2e-2, atol=2e-2)


@pytest.mark.parametrize("wide_k,kernel", [(2048, "gemm_tc_wide_kernel"), (0, "gemm_tc_pair_kernel<256>")], ids=["wide", "pair"])
def test_gemm_wide_kernel_sampled_rows(ops, wide_k, kernel):
    """The 512 x 256 pair tile (K >= 2048 and >= 4 waves of tiles) at a 7B-like shape; the CPU check samples rows (incl. the first / last
    row of several 128-row halves) instead of forming the whole product.  Which kernel serves long contractions is tuned per board
    (ops.autotune_gemm_route), so both are pinned here in turn (`pair`: the 256 x 256 pair tile on the same problem)."""
    import tcavp_b200.lib as L
    ops.autotune_gemm_route()                         # whatever the process decided is restored below
    old = L.load().tcavp_gemm_wide_min_k(wide_k)
    try:
        _wide_kernel_case(ops, kernel)
    finally:
        L.load().tcavp_gemm_wide_min_k(old)


def test_gemm_route_autotune_reports_a_decision(ops):
    t = ops.autotune_gemm_route()
    assert t["source"] in ("autotune", "TCAVP_GEMM_WIDE_K") and ops._ROUTE["wide_k"] in (0, 2048) or t["source"] == "TCAVP_GEMM_WIDE_K"
    if t["source"] == "autotune":
        assert t["wide_ms"] > 0 and t["pair_ms"] > 0 and t["long_k_kernel"] in ("gemm_tc_wide_kernel", "gemm_tc_pair_kernel")


def _wide_kernel_case(ops, kernel):
    M, N, K = 40960 + 37, 1024, 2048 + 64
    g = torch.Generator(device=DEV).manual_seed(5)
    a = (torch.randn(M, K, device=DEV, generator=g) * 0.5).bfloat16()
    w = (torch.randn(N, K, device=DEV, generator=g) * K ** -0.5).bfloat16()
    bias = torch.randn(N, device=DEV, generator=g)
    res = torch.randn(M, N, device=DEV, generator=g).bfloat16()
    ss = torch.zeros(M, dtype=torch.int64, device=DEV)
    out = torch.empty(M, N, dtype=torch.bfloat16, device=DEV)
    ops.gemm(a, w, out, bias=bias, residual=res, sumsq_out=ss)
    assert ops.last_kernel() == kernel
    rows = torch.randint(0, M, (384,), generator=torch.Generator().manual_seed(6))
    rows[:10] = torch.tensor([0, 127, 128, 255, 256, 511, 512, 40959, 40960, M - 1])
    rows = rows.to(DEV)
    want = a[rows].float() @ w.float().t() + bias + res[rows].float()
    torch.testing.assert_close(out[rows].float(), want, rtol=2e-2, atol=2e-2)
    torch.testing.assert_close(ss[rows].double().mul(2.0 ** -20).float(), (want ** 2).sum(-1), rtol=3e-3, atol=1e-1)
    sw = ops.gemm(a, w, torch.empty(M, N // 2, dtype=torch.bfloat16, device=DEV), act=ops.ACT_SWIGLU)
    y = a[rows].float() @ w.float().t()
    torch.testing.assert_close(sw[rows].float(), torch.nn.functional.silu(y[:, 0::2]) * y[:, 1::2], rtol=3e-2, atol=2e-2)


def test_profiler_labels_name_the_launched_kernel(ops):
    """LaunchProfiler labels of ops.gemm / ops.attention: the kernel tcavp_gemm / tcavp_attention launched (tcavp_last_kernel) plus
    the problem shape, for one shape per route; the long-K route is pinned both ways.  An empty GEMM launches nothing and is not recorded."""
    import tcavp_b200.lib as L

    def gemm(M, N, K, dtype=torch.bfloat16):
        a, w = torch.randn(M, K, device=DEV), torch.randn(N, K, device=DEV) * K ** -0.5
        out = torch.empty(M, N, device=DEV, dtype=torch.float32 if dtype == torch.float32 else torch.bfloat16)
        if dtype == torch.float8_e4m3fn:
            ops.gemm(a.to(dtype), w.to(dtype), out, col_scale=torch.ones(N, device=DEV))
        else:
            ops.gemm(a.to(dtype), w.to(dtype), out)

    def attention(B, H, Hkv, Tq, Tk, dh, causal=False, dtype=torch.bfloat16, shared_kv=False):
        q = torch.randn(B, Tq, H, dh, device=DEV).to(dtype)
        k = torch.randn(B, Tk, Hkv, dh, device=DEV).to(dtype)
        v = k if shared_kv else torch.randn(B, Tk, Hkv, dh, device=DEV).to(dtype)
        ops.attention(q, k, v, torch.empty_like(q), B=B, H=H, Hkv=Hkv, Tq=Tq, Tk=Tk, dh=dh, q_strides=(Tq * H * dh, H * dh),
                      k_strides=(Tk * Hkv * dh, Hkv * dh), v_strides=(Tk * Hkv * dh, Hkv * dh), o_strides=(Tq * H * dh, H * dh),
                      scale=dh ** -0.5, causal=causal)

    ops.autotune_gemm_route()                         # before the pins below; whatever the process decided is restored at the end
    old = L.load().tcavp_gemm_wide_min_k(-1)
    try:
        with ops.LaunchProfiler() as prof:
            gemm(300, 32, 64)
            gemm(300, 64, 64)
            gemm(300, 100, 64)
            gemm(300, 200, 64)
            gemm(4100, 520, 64)
            gemm(32768, 256, 64)
            gemm(0, 256, 64)
            gemm(100, 24, 72, torch.float32)
            gemm(300, 200, 128, torch.float8_e4m3fn)
            gemm(4100, 520, 128, torch.float8_e4m3fn)
            L.load().tcavp_gemm_wide_min_k(2048)
            gemm(16384, 2560, 2048)
            L.load().tcavp_gemm_wide_min_k(0)
            gemm(16384, 2560, 2048)
            attention(2, 4, 4, 144, 144, 64, causal=True)
            attention(2, 2, 1, 25, 144, 256, shared_kv=True)
            attention(2, 2, 2, 25, 144, 384)
            attention(2, 8, 8, 15, 15, 96)
            attention(3, 2, 2, 15, 15, 32, dtype=torch.float32)
            attention(2, 8, 8, 15, 15, 96, dtype=torch.float32)
    finally:
        L.load().tcavp_gemm_wide_min_k(old)
    assert [r[0] for r in prof.rec] == [
        "gemm_tc_kernel<32>[N32,K64]", "gemm_tc_kernel<64>[N64,K64]", "gemm_tc_kernel<128>[N100,K64]", "gemm_tc_kernel<256>[N200,K64]",
        "gemm_tc_pair_kernel<256>[M4100,N520,K64]", "gemm_tc_pair_kernel<256>[N256,K64]", "gemm_simt_kernel",
        "gemm_tc_kernel<256,e4m3>[N200,K128]", "gemm_tc_pair_kernel<256,e4m3>[M4100,N520,K128]",
        "gemm_tc_wide_kernel[N2560,K2048]", "gemm_tc_pair_kernel<256>[M16384,N2560,K2048]",
        "attn_tm_kernel[dh64,L144]", "attn_xt_kernel[dh256,q25,k144]", "attn_x_kernel", "attn_flash_kernel[dh96,q15,k15]",
        "attn_row_kernel[dh32,q15,k15]", "attn_warp_kernel[dh96,q15,k15]"]
    # algorithmic bytes: the shared K = V head of attn_xt_kernel is read once, the K and V heads of attn_x_kernel once each
    assert prof.rec[12][2] == 2 * 2 * 256 * (2 * 2 * 25 + 1 * 144) and prof.rec[13][2] == 2 * 2 * 384 * (2 * 2 * 25 + 2 * 2 * 144)


@pytest.mark.parametrize("pw", [1, 3, 5])
def test_gemm_panel_tile_order(ops, pw):
    """Panel-major tile order of the persistent tcgen05 kernels (W larger than L2): forced panel widths, every kernel variant, ragged
    edges, whole output compared.  The width is read once per process, so the check runs as a script (tools/panel_order_check.py)."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, TCAVP_GEMM_PANEL_FORCE=str(pw))
    r = subprocess.run([sys.executable, os.path.join(root, "tools", "panel_order_check.py")], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "panel_order_check ok" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


@pytest.mark.parametrize("B,K,T", [(7, 10, 25), (300, 3, 50), (1, 1, 1), (5, 20, 40)])
def test_best_of_k_reduction(ops, B, K, T):
    """tcavp_best_of_k against the restated candidate reduction of the reference's best-of-K evaluation (scripts/test.py:1336-1368)."""
    cand, y = torch.rand(B, K, 2, T, generator=torch.Generator().manual_seed(1)), torch.rand(B, 2, T, generator=torch.Generator().manual_seed(2))
    ns = [(100.0 + i, 900.0 + 3 * i, 700.0 + i, 760.0 + 2 * i) for i in range(B)]
    want = R.best_of_k(cand, y, ns)
    per = torch.empty(B, 3, device=DEV)
    tot = torch.zeros(3, device=DEV)
    ops.best_of_k(cand.to(DEV), y.to(DEV), torch.tensor(ns, device=DEV), per, tot, B=B, K=K, T_out=T)
    for i in range(3):
        torch.testing.assert_close(per[:, i].cpu(), want[i], rtol=1e-4, atol=1e-3)
        torch.testing.assert_close(tot[i].cpu(), want[i].sum(), rtol=1e-4, atol=1e-2)


def test_model_best_of_k_metrics_entry_point(lib_built):
    """MultiModalTrajectoryModel.best_of_k_metrics (the public entry of the reference's best-of-K reduction, scripts/test.py:1336-1368)
    with host tensors and a list-typed norm_stat, against the restated reduction."""
    import tcavp_b200 as T
    m = T.MultiModalTrajectoryModel(**T.MODEL_PRESETS["tiny"]).to(DEV)
    B, K, To = 9, 6, 12
    cand, y = torch.rand(B, K, 2, To, generator=torch.Generator().manual_seed(3)), torch.rand(B, 2, To, generator=torch.Generator().manual_seed(4))
    ns = [(50.0 + i, 700.0 + 5 * i, 710.0 + i, 790.0 + 3 * i) for i in range(B)]
    got = m.best_of_k_metrics(cand, y, ns)
    want = R.best_of_k(cand, y, ns)
    for key, w in zip(("min_ade", "min_fde", "min_rmse"), want):
        torch.testing.assert_close(got[key].cpu(), w, rtol=1e-4, atol=1e-3)
    torch.testing.assert_close(got["sums"].cpu(), torch.stack([w.sum() for w in want]), rtol=1e-4, atol=1e-2)
