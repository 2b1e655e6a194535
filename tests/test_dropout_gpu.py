"""Train-mode dropout (SURVEY.md §8 rows a11 / f2): the counter-based masks of include/tcavp.h on the CUDA path against the oracle's
host evaluation of the same function — bit-exact masks at kernel level, gradient parity of the whole fine-tune step against goldens
minted from the UNMODIFIED reference in train() mode (oracle/make_golden.py DROP_FIXTURES), the CUDA-graph loop drawing fresh masks
on every replay, and the best-of-K evaluation of scripts/test.py:1308-1368."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import tcavp_b200 as T  # noqa: E402
from conftest import load_golden  # noqa: E402
from oracle import dropout as OD  # noqa: E402
from oracle import restated  # noqa: E402
from test_oracle_cpu import _check_against_compressed  # noqa: E402
from test_train_gpu import ILL, _model, _step  # noqa: E402

DEV = "cuda"


def _seed(base, step):
    return torch.tensor([base, step], dtype=torch.int32, device=DEV)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("rows,cols,ld", [(37, 64, 64), (5, 13, 20), (1000, 776, 776), (3, 8, 8)])
def test_dropout_kernel_mask_is_the_oracle_mask(lib_built, dtype, rows, cols, ld):
    from tcavp_b200 import ops
    g = torch.Generator().manual_seed(rows * cols)
    x = (torch.rand(rows, ld, generator=g) + 0.5).to(dtype).to(DEV)          # strictly positive: kept elements are non-zero
    res = torch.randn(rows, cols, generator=g).to(DEV)
    site, p = OD.site_id("qenc", 2, "drop1"), 0.1
    d = ops.Drop(_seed(123, 9), site, p)
    keep = torch.from_numpy(OD.keep_mask(123, 9, site, p, rows * cols)).view(rows, cols).to(DEV)
    out = torch.empty(rows, cols, dtype=dtype, device=DEV)
    ops.dropout(x, out, d, rows=rows, cols=cols, ldi=ld)
    assert torch.equal(out != 0, keep)
    want = torch.where(keep, x[:, :cols].float() / (1 - p), torch.zeros((), device=DEV)).to(dtype)
    torch.testing.assert_close(out, want, rtol=1e-6 if dtype == torch.float32 else 8e-3, atol=0)
    # residual + accumulate forms; in-place
    acc = torch.ones(rows, cols, dtype=torch.float32, device=DEV)
    ops.dropout(x, acc, d, rows=rows, cols=cols, ldi=ld, residual=res, accumulate=True, scale=1.0)
    torch.testing.assert_close(acc, 1.0 + res + torch.where(keep, x[:, :cols].float(), torch.zeros((), device=DEV)), rtol=1e-6, atol=1e-6)
    y = x.clone()
    ops.dropout(y, y, d, rows=rows, cols=cols, ldi=ld, ldo=ld)
    assert torch.equal(y[:, :cols] != 0, keep) and torch.equal(y[:, cols:], x[:, cols:])
    # p = 0 keeps everything; another step gives another mask
    ops.dropout(x, out, ops.Drop(_seed(123, 9), site, 0.0), rows=rows, cols=cols, ldi=ld)
    assert torch.equal(out, x[:, :cols])
    if rows * cols > 1000:
        ops.dropout(x, out, ops.Drop(_seed(123, 10), site, p), rows=rows, cols=cols, ldi=ld)
        assert not torch.equal(out != 0, keep)


@pytest.mark.parametrize("M,H,r,probs,ld_extra", [
    (300, 768, 8, (0.1, 0.1), 16),            # 768-class: q_proj + v_proj (peft default targets), K-extended rows [H + 16]
    (77, 128, 16, (0.1, 0.0, 0.3), 48),       # rank 16, three targets, one of them without dropout, ragged row tile
    (1000, 4096, 16, (0.1, 0.1), 32),         # 7B geometry
    (130, 64, 8, (0.5, 0.1, 0.1, 0.2), 32),   # four targets, a single 64-column stage
])
def test_fused_lora_dropout_kernels(lib_built, M, H, r, probs, ld_extra):
    """peft lora.Linear in train mode (train.py:432-440): lora_A(dropout(x)) with one mask per target.  The fused kernels (csrc/lora_drop.cu,
    masked fragments in dw_tc.cu) against the literal form built from the oracle's masks — forward product, input gradient, lora_A gradient."""
    from tcavp_b200 import ops
    n = len(probs)
    NL, Kx = n * r, H + ld_extra
    g = torch.Generator().manual_seed(M + H)
    xs = torch.randn(M, Kx, generator=g).bfloat16().to(DEV)                 # K-extended residual rows [x | side columns]
    A = (torch.randn(NL, H, generator=g) * 0.05).bfloat16().to(DEV)
    dT = torch.randn(M, Kx, generator=g).bfloat16().to(DEV)                 # [dn1 | dT] as the QKV^T GEMM leaves it
    rstd = (torch.rand(M, generator=g) + 0.5).to(DEV)
    seed = _seed(4242, 3)
    sites = [OD.site_id("llm", 5 + t // 3, "lora_" + "qkv"[t % 3]) for t in range(n)]
    drops = [ops.Drop(seed, s_, p) for s_, p in zip(sites, probs)]
    keep = [torch.from_numpy(OD.keep_mask(4242, 3, s_, p, M * H)).view(M, H).to(DEV).float() if p > 0 else torch.ones(M, H, device=DEV)
            for s_, p in zip(sites, probs)]
    x = xs[:, :H].float()
    # forward: T[:, t r : (t + 1) r] = (mask_t o x) A_t^T; the columns behind NL keep their contents
    out = xs.clone()
    ops.lora_a_drop(out, A, out[:, H:], drops, M=M, H=H, r=r, ldx=Kx, ldo=Kx)
    want = torch.cat([(keep[t] * x) @ A[t * r:(t + 1) * r].float().t() for t in range(n)], 1)
    torch.testing.assert_close(out[:, H:H + NL].float(), want, rtol=2e-2, atol=2e-2 * float(want.abs().max()))
    assert torch.equal(out[:, :H], xs[:, :H]) and torch.equal(out[:, H + NL:], xs[:, H + NL:])
    # input gradient: dx += sum_t mask_t o (dT_t A_t), in place on the first H columns
    dx = dT.clone()
    ops.lora_dx_drop(dx[:, H:], A, dx, drops, M=M, H=H, r=r, lddt=Kx, lddx=Kx)
    want = dT[:, :H].float() + sum(keep[t] * (dT[:, H + t * r:H + (t + 1) * r].float() @ A[t * r:(t + 1) * r].float()) for t in range(n))
    torch.testing.assert_close(dx[:, :H].float(), want, rtol=2e-2, atol=2e-2 * float(want.abs().max()))
    assert torch.equal(dx[:, H:], dT[:, H:])
    # lora_A gradient: dA[h, j] = sum_m rstd[m] mask_t(m, h) x[m, h] dT[m, j]
    dA = torch.zeros(H, NL, dtype=torch.float32, device=DEV)
    ops.lora_da_drop(xs, dT[:, H:], dA, drops, M=M, H=H, r=r, ldx=Kx, lddt=Kx, row_scale=rstd)
    dTs = (dT[:, H:H + NL].float() * rstd[:, None]).bfloat16().float()      # the kernel applies the row factor to the narrow operand in bf16
    want = torch.cat([(keep[t] * x).t() @ dTs[:, t * r:(t + 1) * r] for t in range(n)], 1)
    torch.testing.assert_close(dA, want, rtol=2e-2, atol=1e-2 * float(want.abs().max()))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("B,H,Tq,Tk,dh,masked,causal", [(3, 4, 33, 33, 16, True, False), (2, 2, 15, 15, 32, False, False), (2, 8, 16, 15, 96, False, False),
                                                        (2, 2, 12, 40, 64, False, False), (2, 2, 25, 144, 384, False, False),
                                                        (3, 4, 40, 40, 32, True, True), (2, 12, 144, 144, 64, True, True)])
def test_attention_dropout_forward_and_backward(lib_built, dtype, B, H, Tq, Tk, dh, masked, causal):
    """Dropout on the attention probabilities (forward and backward kernels) against autograd through the same math with the oracle mask.
    The causal cases are the GPT-2-arch backbone in train mode (HF attn_pdrop: causal + key-padding mask + dropout on the probabilities)."""
    from tcavp_b200 import ops
    g = torch.Generator().manual_seed(B * Tq + dh)
    E = H * dh
    q, k, v = (torch.randn(B, T_, E, generator=g).to(dtype) for T_ in (Tq, Tk, Tk))
    do = torch.randn(B, Tq, E, generator=g).to(dtype)
    km = None
    if masked:
        km = (torch.arange(Tk)[None, :] < torch.tensor([Tk, 7, 20][:B])[:, None]).to(torch.int32)
        if causal:      # right padding never masks a row completely under the causal mask
            km = (torch.arange(Tk)[None, :] < torch.tensor([Tk, Tk - 9, Tk - 17][:B])[:, None]).to(torch.int32)
    site, p, scale = OD.site_id("poly", 1, "sa_attn"), 0.1, dh ** -0.5
    f = torch.from_numpy(OD.keep_mask(77, 2, site, p, B * H * Tq * Tk).astype(np.float32) / (1 - p)).view(B, H, Tq, Tk)
    qf, kf, vf = (t.float().clone().requires_grad_(True) for t in (q, k, v))
    s = (qf.view(B, Tq, H, dh).transpose(1, 2) @ kf.view(B, Tk, H, dh).transpose(1, 2).transpose(-1, -2)) * scale
    if km is not None:
        s = s.masked_fill(km[:, None, None, :] == 0, float("-inf"))
    if causal:
        s = s.masked_fill(~torch.ones(Tq, Tk, dtype=torch.bool).tril(), float("-inf"))
    o_ref = ((torch.softmax(s, -1) * f) @ vf.view(B, Tk, H, dh).transpose(1, 2)).transpose(1, 2).reshape(B, Tq, E)
    gq, gk, gv = torch.autograd.grad(o_ref, (qf, kf, vf), do.float())
    d = ops.Drop(_seed(77, 2), site, p)
    qd, kd, vd, dod = (t.to(DEV).contiguous() for t in (q, k, v, do))
    kmd = None if km is None else km.to(DEV)
    out = torch.empty(B, Tq, E, dtype=dtype, device=DEV)
    st = lambda T_: (T_ * E, E)    # noqa: E731
    ops.attention(qd, kd, vd, out, B=B, H=H, Hkv=H, Tq=Tq, Tk=Tk, dh=dh, q_strides=st(Tq), k_strides=st(Tk), v_strides=st(Tk), o_strides=st(Tq),
                  scale=scale, key_mask=kmd, drop=d, causal=causal)
    tol = dict(rtol=2e-4, atol=2e-4) if dtype == torch.float32 else dict(rtol=3e-2, atol=3e-2)
    torch.testing.assert_close(out.float().cpu(), o_ref.detach(), **tol)
    dq = torch.empty(B, Tq, E, dtype=dtype, device=DEV)
    dk, dv = torch.zeros(B, Tk, E, device=DEV), torch.zeros(B, Tk, E, device=DEV)
    ops.attention_bwd(qd, kd, vd, dod, dq, dk, dv, B=B, H=H, Hkv=H, Tq=Tq, Tk=Tk, dh=dh, q_strides=st(Tq), k_strides=st(Tk), v_strides=st(Tk),
                      do_strides=st(Tq), dq_strides=st(Tq), dk_strides=st(Tk), dv_strides=st(Tk), scale=scale, key_mask=kmd, o=out, o_strides=st(Tq),
                      drop=d, causal=causal)
    btol = dict(rtol=1e-3, atol=1e-3) if dtype == torch.float32 else dict(rtol=5e-2, atol=5e-2 * float(gq.abs().max()))
    torch.testing.assert_close(dq.float().cpu(), gq, **btol)
    torch.testing.assert_close(dk.cpu(), gk, **btol)
    torch.testing.assert_close(dv.cpu(), gv, **btol)
    if ops.attention_bwd_owned_ok(qd, H=H, Hkv=H, Tq=Tq, Tk=Tk, dh=dh, o=out, causal=causal):
        # the "owned" form the fine-tune step uses (one CTA owns every key row: dk / dv stored directly in bf16)
        dq2 = torch.empty(B, Tq, E, dtype=dtype, device=DEV)
        dk2, dv2 = torch.empty(B, Tk, E, dtype=dtype, device=DEV), torch.empty(B, Tk, E, dtype=dtype, device=DEV)
        ops.attention_bwd_owned(qd, kd, vd, dod, dq2, dk2, dv2, B=B, H=H, Tq=Tq, Tk=Tk, dh=dh, q_strides=st(Tq), k_strides=st(Tk), v_strides=st(Tk),
                                do_strides=st(Tq), dq_strides=st(Tq), dk_strides=st(Tk), dv_strides=st(Tk), scale=scale, key_mask=kmd, o=out,
                                o_strides=st(Tq), drop=d, causal=causal)
        torch.testing.assert_close(dq2.float().cpu(), gq, **btol)
        torch.testing.assert_close(dk2.float().cpu(), gk, rtol=5e-2, atol=5e-2 * float(gk.abs().max()))
        torch.testing.assert_close(dv2.float().cpu(), gv, rtol=5e-2, atol=5e-2 * float(gv.abs().max()))


def _drop_oracle(fix):
    return OD.DropOracle(fix["dropout"]["seed"], fix["dropout"]["step"], OD.default_probs(fix["model_cfg"], llama_cfg=fix["llama_cfg"]))


@pytest.mark.parametrize("name", ["tiny_b5_grads_drop", "cfg1_b3_grads_drop", "gpt2_tiny_b5_grads_drop", "gpt2_l2_b3_grads_drop"])
def test_fp32_train_mode_gradients_match_reference(lib_built, name):
    """The whole fine-tune step in train() mode (p = 0.1 at every site of the reference) against the golden of the unmodified reference
    run with the same masks: loss, decoded, and the gradient of every trainable tensor."""
    fix = load_golden(name)
    m = _model(fix, "fp32")
    assert m.training and m.dropout_active()
    m.set_dropout_seed(fix["dropout"]["seed"], fix["dropout"]["step"])
    loss, dec = _step(m, fix["inputs"])
    loss.backward()
    torch.cuda.synchronize()
    torch.testing.assert_close(loss.detach().cpu(), fix["loss"], rtol=1e-4, atol=0)
    torch.testing.assert_close(dec.cpu(), fix["decoded"], rtol=1e-4, atol=5e-4)
    got = {n: p.grad for n, p in m.named_parameters() if p.requires_grad}
    assert set(got) == set(fix["grads"])
    worst, failures = {}, []
    for k, want in fix["grads"].items():
        ref = want["full"] if "full" in want else want["head"]
        scale = float(ref.abs().max()) + 1e-8
        ill = k.startswith(ILL)
        try:
            _check_against_compressed(got[k], want, rtol=0.3 if ill else 5e-3, atol=(0.3 if ill else 1e-3) * scale + 1e-6, key=k)
        except AssertionError as e:
            failures.append((k, str(e)[:200]))
    assert not failures, failures[:5]
    # the next pass draws from step + 1: a different loss on the same batch; re-seeding reproduces the first one
    l2, _ = _step(m, fix["inputs"])
    assert abs(float(l2) - float(loss)) > 1e-6 * abs(float(loss))
    m.set_dropout_seed(fix["dropout"]["seed"], fix["dropout"]["step"])
    l3, _ = _step(m, fix["inputs"])
    torch.testing.assert_close(l3.detach(), loss.detach(), rtol=1e-6, atol=0)
    # eval() switches every site off: the p = 0 golden
    m.eval()
    l4, _ = _step(m, fix["inputs"])
    torch.testing.assert_close(l4.detach().cpu(), load_golden(name.replace("_drop", ""))["loss"], rtol=1e-4, atol=0)


@pytest.mark.parametrize("name", ["tiny_b5_grads_drop", "gpt2_l2_b3_grads_drop", "gpt2_tiny_b5_grads_drop"])
def test_bf16_train_mode_gradients_track_the_oracle(lib_built, name):
    """bf16 train mode (gpt2_l2: LoRA r 8 on a 768-wide c_attn, so lora_dropout runs through the fused mask-regenerating kernels)."""
    fix = load_golden(name)
    m = _model(fix, "bf16")
    m.set_dropout_seed(fix["dropout"]["seed"], fix["dropout"]["step"])
    loss, _ = _step(m, fix["inputs"])
    loss.backward()
    torch.cuda.synchronize()
    assert abs(float(loss) - float(fix["loss"])) / float(fix["loss"]) < 2e-2
    mm = T.MultiModalTrajectoryModel(**fix["model_cfg"])
    sd = mm.state_dict()
    T.deterministic_fill_(sd, fix["weight_seed"])
    i = fix["inputs"]
    with restated.dropout(_drop_oracle(fix)):
        _, _, o_grads = restated.loss_and_grads(sd, fix["model_cfg"], fix["llama_cfg"], i["x"], i["vision"], i["polygon"], i["poly_len"], i["input_ids"],
                                                i["attention_mask"], i["y"], i["norm_stat"])
    gmax = max(float(g.norm()) for g in o_grads.values())
    low, checked = [], 0
    for n, p in m.named_parameters():
        if not p.requires_grad:
            continue
        g, w = p.grad.float().cpu().flatten(), o_grads[n].flatten()
        if float(w.norm()) < 1e-4 * gmax or n.startswith(ILL):
            continue
        checked += 1
        cos = float(torch.dot(g, w) / (g.norm() * w.norm() + 1e-30))
        ratio = float(g.norm() / (w.norm() + 1e-30))
        if cos < 0.95 or not 0.8 < ratio < 1.25:
            low.append((n, round(cos, 4), round(ratio, 4)))
    assert checked > 300 and not low, low[:10]


@pytest.mark.parametrize("graph", [False, True])
def test_finetuner_draws_fresh_masks_every_step(lib_built, graph):
    """FineTuner in train mode: replaying the captured CUDA graph advances the step counter on the device, so the same batch gives a
    different loss on every step with lr = 0 (only the masks change), and a re-seeded tuner reproduces the sequence."""
    fix = load_golden("tiny_b5_grads_drop")
    i = fix["inputs"]

    def run():
        m = _model(fix, "fp32")
        ft = T.FineTuner(m, lr=0.0, weight_decay=0.0, use_cuda_graph=graph)
        m.set_dropout_seed(4242, 0)
        ctx = ["c"] * i["x"].shape[0]
        out = []
        for _ in range(4):
            loss, _ = ft.step(i["x"].cuda(), i["vision"].cuda(), ctx, i["polygon"].cuda(), i["poly_len"], i["y"].cuda(), i["norm_stat"],
                              i["input_ids"].cuda(), i["attention_mask"].cuda())
            out.append(float(loss))
        return out
    a, b = run(), run()
    assert len(set(round(v, 3) for v in a)) == 4, a
    if not graph:
        assert a == pytest.approx(b, rel=1e-6)


def test_best_of_k_matches_k_oracle_passes(lib_built):
    """model.best_of_k (reference scripts/test.py:1308-1368): K stochastic passes in train() mode under no_grad + the min-over-candidates
    reduction, against K passes of the restatement with the same (seed, step + k) masks."""
    fix = load_golden("tiny_b5_grads_drop")
    m = _model(fix, "fp32")
    i = fix["inputs"]
    K = 4
    m.eval()
    m.set_dropout_seed(99, 5)
    r = m.best_of_k(i["x"].cuda(), i["vision"].cuda(), i["polygon"].cuda(), i["poly_len"], i["y"].cuda(), i["norm_stat"], i["input_ids"].cuda(),
                    i["attention_mask"].cuda(), num_candidates=K)
    assert not m.training and r["candidates"].shape == (i["x"].shape[0], K, 2, fix["model_cfg"]["out_len"])
    mm = T.MultiModalTrajectoryModel(**fix["model_cfg"])
    sd = mm.state_dict()
    T.deterministic_fill_(sd, fix["weight_seed"])
    cands = []
    for k in range(K):
        with restated.dropout(OD.DropOracle(99, 5 + k, OD.default_probs(fix["model_cfg"]))):
            cands.append(restated.forward(sd, fix["model_cfg"], fix["llama_cfg"], i["x"], i["vision"], i["polygon"], i["poly_len"], i["input_ids"],
                                          i["attention_mask"])["decoded"])
    want = torch.stack(cands, dim=1)
    torch.testing.assert_close(r["candidates"].cpu(), want, rtol=1e-4, atol=5e-4)
    assert float((want[:, 0] - want[:, 1]).abs().max()) > 1e-3          # the candidates really differ
    w_ade, w_fde, w_rmse = restated.best_of_k(want, i["y"], i["norm_stat"])
    torch.testing.assert_close(r["min_ade"].cpu(), w_ade, rtol=1e-4, atol=1e-2)
    torch.testing.assert_close(r["min_fde"].cpu(), w_fde, rtol=1e-4, atol=1e-2)
    torch.testing.assert_close(r["min_rmse"].cpu(), w_rmse, rtol=1e-4, atol=1e-2)
