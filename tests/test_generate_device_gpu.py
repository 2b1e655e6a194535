"""The seeded device decode loop of generate.py and its kernels (include/tcavp.h, "text generation on the device"):
tcavp_sample_next against process_logits and a host restatement of its draw, tcavp_decode_attention against torch, and the CUDA-graph
loop against the eager KV-cache path.

Documented differences from process_logits (the only ones the comparisons allow):
  * top-p near the boundary: a token whose ascending cumulative mass lies within 1e-6 of 1 - top_p may land on either side (the kernel
    sums integer weights, torch sums fp32 probabilities in sorted order);
  * tie groups: tokens equal to the k-th value are all kept by both; a tie group at the top-p boundary is kept whole by the kernel,
    while torch's sort keeps the part that sorts last."""
import math

import pytest
import torch

gpu = pytest.mark.gpu

from conftest import build_filled_model, load_golden  # noqa: E402
from tcavp_b200 import generate as G  # noqa: E402
from tcavp_b200 import ops  # noqa: E402

M32 = 0xFFFFFFFF


def _mix(x):
    x &= M32
    x ^= x >> 16
    x = (x * 0x7FEB352D) & M32
    x ^= x >> 15
    x = (x * 0x846CA68B) & M32
    x ^= x >> 16
    return x


def _uniform32(seed_lo, seed_hi, row, step):
    key = _mix(seed_lo ^ _mix(seed_hi + 0x9E3779B9))
    return _mix(_mix(key ^ step) ^ ((row * 0x85EBCA6B + 0x632BE5AB) & M32))


def _restated_draw(work, seed_lo, seed_hi, step):
    """Host restatement of the draw: integer weights floor(exp(x - max) * 2^40) in token order, r = floor(u * W / 2^32), first cumsum > r."""
    toks = []
    for row in range(work.shape[0]):
        x = work[row]
        e = torch.exp(x - x.max())                                   # same fp32 exp on the device
        w = torch.floor(e.double() * 2.0 ** 40).to(torch.int64).cpu()
        cum = torch.cumsum(w, 0)
        W = int(cum[-1])
        r = (_uniform32(seed_lo, seed_hi, row, step) * W) >> 32
        toks.append(int(torch.searchsorted(cum, torch.tensor([r]), right=True)[0]))
    return toks


class _Sampler:
    def __init__(self, B, V, hist_len, extra=4):
        dev = "cuda"
        self.work = torch.empty(B, V, dtype=torch.float32, device=dev)
        self.hist = torch.zeros(B, hist_len + extra, dtype=torch.int64, device=dev)
        self.state = torch.zeros(3, dtype=torch.int32, device=dev)
        self.done = torch.zeros(B, dtype=torch.int32, device=dev)
        self.tokens = torch.zeros(B, dtype=torch.int64, device=dev)
        self.seed = torch.tensor([0x1234567, -5], dtype=torch.int32, device=dev)
        self.hist_len = hist_len

    def __call__(self, logits, seq=None, step=0, **kw):
        if seq is not None:
            self.hist[:, :seq.shape[1]] = seq
        self.state.zero_()
        self.state[0] = step
        self.done.zero_()
        ops.sample_next(logits, self.work, self.hist, self.state, self.done, self.tokens, hist_offset=self.hist_len - step, seed=self.seed, **kw)
        return self.tokens.clone()


def _history(B, V, n, gen):
    """Token histories with repeats and a live 3-gram ban: the last two tokens repeat an earlier bigram."""
    seq = torch.randint(0, min(V, 23), (B, n), generator=gen)
    seq[:, -2:] = seq[:, 3:5]
    return seq


def _logits(B, V, gen):
    x = torch.randn(B, V, generator=gen) * 3.0
    x[:, 5] = -math.inf                                     # -inf inputs
    x[0, 7] = x[0, 8] = x[0].max() + 1.0                    # a tie at the top
    x[1, 11:14] = x[1].max() + 0.25                         # a three-way tie at the top
    return x


def _boundary_exempt(ref, pre, top_p):
    """Tokens whose ascending cumulative mass lies within 1e-6 of 1 - top_p, and tie groups (equal values before top-p, `pre`) that top-p
    cut apart (see the module docstring)."""
    ex = torch.zeros_like(ref, dtype=torch.bool)
    if top_p is None or not 0.0 < top_p < 1.0:
        return ex
    srt, idx = torch.sort(ref.double(), dim=-1)
    cum = srt.softmax(-1).cumsum(-1)
    near = (cum - (1.0 - top_p)).abs() < 1e-6
    ex = ex.scatter(1, idx, near)
    for b in range(ref.shape[0]):
        vals, counts = torch.unique(pre[b][torch.isfinite(pre[b])], return_counts=True)
        for v in vals[counts > 1]:
            group = pre[b] == v
            kept = torch.isfinite(ref[b][group])
            if kept.any() and not kept.all():
                ex[b] |= group
    return ex


@gpu
@pytest.mark.parametrize("V", [37, 32000, 128256])
@pytest.mark.parametrize("temperature,top_k,top_p", [(0.9, 40, 0.9), (1.0, 0, 0.5), (0.7, 10 ** 6, 0.95), (1.3, 7, 1.0), (1.0, 0, None),
                                                     (0.8, 3, 0.3)])
def test_sampler_processors_match_process_logits(lib_built, V, temperature, top_k, top_p):
    gen = torch.Generator().manual_seed(V + top_k)
    B, n = 6, 40
    x, seq = _logits(B, V, gen), _history(B, V, n, gen)
    s = _Sampler(B, V, n)
    s(x.cuda(), seq.cuda(), temperature=temperature, top_k=top_k, top_p=top_p, repetition_penalty=1.2, no_repeat_ngram_size=3)
    got = s.work.cpu()
    ref = G.process_logits(x.clone(), seq, temperature, top_k, top_p, 1.2, 3)
    pre = G.process_logits(x.clone(), seq, temperature, top_k, None, 1.2, 3)
    assert torch.isinf(ref[:, 5]).all() and (torch.isinf(ref) & (ref < 0)).any(dim=1).all()
    ok_got, ok_ref = torch.isfinite(got), torch.isfinite(ref)
    differ = ok_got != ok_ref
    assert not (differ & ~_boundary_exempt(ref, pre, top_p)).any(), differ.nonzero()
    for b in range(B):
        if not differ[b].any():
            torch.testing.assert_close(got[b].softmax(-1), ref[b].softmax(-1), rtol=0, atol=1e-6)
    # greedy: argmax of the processed logits, lowest index on ties (row 0 / 1 have tied maxima unless a processor moved them)
    tok = s(x.cuda(), seq.cuda(), do_sample=False, repetition_penalty=1.2, no_repeat_ngram_size=3)
    want = G.process_logits(x.clone(), seq, 1.0, 0, None, 1.2, 3).argmax(-1)
    assert torch.equal(tok.cpu(), want)


@gpu
@pytest.mark.parametrize("V,top_k,top_p", [(37, 0, None), (32000, 40, 0.9), (128256, 0, 0.95)])
def test_sampler_draw_matches_the_host_restatement_bit_for_bit(lib_built, V, top_k, top_p):
    gen = torch.Generator().manual_seed(3)
    B, n = 64, 12
    s = _Sampler(B, V, n)
    lo, hi = [int(v) & M32 for v in s.seed.cpu()]
    seq = _history(B, V, n, gen).cuda()
    for step in range(6):
        x = _logits(B, V, gen).cuda()
        tok = s(x, seq, step=step, temperature=0.9, top_k=top_k, top_p=top_p, repetition_penalty=1.2, no_repeat_ngram_size=3)
        assert tok.tolist() == _restated_draw(s.work, lo, hi, step), step
        assert torch.isfinite(s.work[torch.arange(B), tok]).all()


@gpu
def test_sampler_draws_follow_the_processed_distribution(lib_built):
    """2e5 draws of one logits row (the hash decorrelates rows and steps): chi-square against softmax(process_logits); the seed is fixed,
    so the statistic is deterministic."""
    from scipy.stats import chisquare
    gen = torch.Generator().manual_seed(11)
    V, B, steps = 37, 2000, 100
    x = torch.randn(1, V, generator=gen) * 1.5
    s = _Sampler(B, V, steps, extra=1)             # history unused: no penalty, no n-gram ban
    xs = x.expand(B, V).contiguous().cuda()
    counts = torch.zeros(V, dtype=torch.int64, device="cuda")
    for step in range(steps):
        tok = s(xs, step=step, temperature=0.8, top_k=20, top_p=0.9)
        counts += torch.bincount(tok, minlength=V)
    p = G.process_logits(x.clone(), torch.zeros(1, 0, dtype=torch.long), 0.8, 20, 0.9, 1.0, 0).softmax(-1)[0].double()
    kept = p > 0
    assert int(counts[~kept.cuda()].sum()) == 0
    obs, exp = counts.cpu()[kept].double(), p[kept] * (B * steps)
    assert float(exp.min()) > 5
    assert chisquare(obs.numpy(), exp.numpy()).pvalue > 1e-3


@gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("dh,ratio", [(64, 1), (64, 4), (128, 1), (128, 4), (32, 2)])
@pytest.mark.parametrize("tk", [1, 129, 300, 1040])
def test_decode_attention_matches_torch_and_appends_the_new_row(lib_built, dtype, dh, ratio, tk):
    gen = torch.Generator().manual_seed(dh + ratio + tk)
    B, Hkv, cap, offset = 3, 2, 1100, 7
    H = Hkv * ratio
    nq, nk = H * dh, Hkv * dh
    p = tk - 1
    qkv = torch.randn(B, nq + 2 * nk, generator=gen).to(dtype).cuda()
    cache = torch.randn(B, cap, 2 * nk, generator=gen).to(dtype).cuda()
    old = cache.clone()
    out = torch.empty(B, nq, dtype=dtype, device="cuda")
    counter = torch.tensor([p - offset], dtype=torch.int32, device="cuda")
    ws = ops.decode_attention_workspace(B, H, dh, cap, "cuda")
    scale = dh ** -0.5
    ops.decode_attention(qkv, qkv[:, nq:], qkv[:, nq + nk:], cache, cache[:, :, nk:], out, ws, counter, offset=offset, B=B, H=H, Hkv=Hkv, dh=dh,
                         capacity=cap, q_sb=nq + 2 * nk, new_sb=nq + 2 * nk, cache_sb=cap * 2 * nk, cache_st=2 * nk, o_sb=nq, scale=scale)
    torch.testing.assert_close(cache[:, p], qkv[:, nq:], rtol=0, atol=0)
    assert torch.equal(cache[:, :p], old[:, :p]) and torch.equal(cache[:, p + 1:], old[:, p + 1:])
    kv = cache[:, :p + 1].double().cpu()
    q = qkv[:, :nq].double().cpu().view(B, H, dh)
    K = kv[:, :, :nk].view(B, p + 1, Hkv, dh).repeat_interleave(ratio, dim=2)
    Vv = kv[:, :, nk:].view(B, p + 1, Hkv, dh).repeat_interleave(ratio, dim=2)
    att = torch.softmax(torch.einsum("bhd,bthd->bht", q, K) * scale, dim=-1)
    want = torch.einsum("bht,bthd->bhd", att, Vv).reshape(B, nq)
    tol = dict(rtol=1e-5, atol=1e-5) if dtype == torch.float32 else dict(rtol=2e-2, atol=2e-2)
    torch.testing.assert_close(out.double().cpu(), want, **tol)


def _prompt(fix, B, Lp):
    i = fix["inputs"]
    return i["vision"][:B].cuda(), i["input_ids"][:B, :Lp].cuda()


@gpu
@pytest.mark.parametrize("fixture", ["tiny_b6", "gpt2_tiny_b6", "llama32_1b_l2_b8"])
def test_greedy_device_loop_matches_the_eager_kv_cache_loop_fp32(lib_built, fixture):
    fix = load_golden(fixture)
    m = build_filled_model(fix, "fp32", "cuda")
    vision, ids = _prompt(fix, 2, 9)
    kw = dict(max_new_tokens=12, do_sample=False, repetition_penalty=1.2, no_repeat_ngram_size=3)
    want = G.generate_ids(m, vision, ids, **kw)
    got = G.generate_ids(m, vision, ids, seed=0, **kw)
    assert got.shape == want.shape == (2, 9 + 12)
    assert torch.equal(got, want)


def _step_logits_device_vs_eager(m, vision, ids, steps=3):
    """Per-step logits of llm_decode_step_device and llm_decode_step fed the same tokens after the same prefill."""
    eng = m.engine()
    pre = eng.prefix_embeds(vision, ids)
    B, P, H = pre.shape
    cap = P + steps + 1
    ones = torch.ones(B, P, dtype=torch.int32, device="cuda")
    ce, cd = [], []
    eng.llm_forward(pre.clone(), ones, B, P, kv_out=(ce, cap))
    eng.llm_forward(pre.clone(), ones, B, P, kv_out=(cd, cap))
    head, ws = eng.lm_head(), eng.decode_workspace(B, cap)
    counter = torch.zeros(1, dtype=torch.int32, device="cuda")
    toks = ids[:, :steps].contiguous()
    out = []
    for j in range(steps):
        t = toks[:, j].contiguous()
        he = eng.llm_decode_step(eng.token_embeds(t[:, None]).view(B, H), ce, P + j)
        counter.fill_(j)
        hd = eng.llm_decode_step_device(t, cd, counter, P, ws)
        le = ops.gemm(he, head, torch.empty(B, head.shape[0], device="cuda"))
        ld = ops.gemm(hd, head, torch.empty(B, head.shape[0], device="cuda"))
        out.append((ld.cpu(), le.cpu()))
    return out


@gpu
@pytest.mark.parametrize("fixture,fp8", [("tiny_b6", False), ("gpt2_tiny_b6", False), ("llama32_1b_l2_b8", False), ("llama32_1b_l2_b8", True)])
def test_device_decode_step_logits_match_the_eager_step_bf16(lib_built, fixture, fp8):
    fix = load_golden(fixture)
    m = build_filled_model(fix, "bf16", "cuda")
    if fp8:
        m.fp8_backbone_for_inference()
    vision, ids = _prompt(fix, 2, 9)
    for ld, le in _step_logits_device_vs_eager(m, vision, ids):
        torch.testing.assert_close(ld, le, rtol=4e-2, atol=4e-2 * float(le.abs().max()))
    # and the whole loop runs on this engine
    seq = G.generate_ids(m, vision, ids, max_new_tokens=6, seed=1)
    assert seq.shape == (2, 15) and torch.equal(seq[:, :9], ids)


@gpu
def test_seeds_reproduce_and_eos_rows_are_padded(lib_built):
    fix = load_golden("tiny_b6")
    m = build_filled_model(fix, "bf16", "cuda")
    vision, ids = _prompt(fix, 4, 9)
    kw = dict(max_new_tokens=16, temperature=1.5, top_k=0, top_p=None, repetition_penalty=1.0, no_repeat_ngram_size=0)
    torch.manual_seed(0)
    a = G.generate_ids(m, vision, ids, seed=123, **kw)
    torch.manual_seed(99)
    b = G.generate_ids(m, vision, ids, seed=123, **kw)
    c = G.generate_ids(m, vision, ids, seed=124, **kw)
    assert torch.equal(a, b) and not torch.equal(a, c)
    assert a.shape == (4, 9 + 16)
    # EOS: the same draws up to each row's first EOS, pad after it; the output ends at the first step after which every row is done
    new = a[:, 9:].cpu()
    eos = int(new[0, 2])
    pad = 0 if eos != 0 else 1
    e = G.generate_ids(m, vision, ids, seed=123, eos_token_id=eos, pad_token_id=pad, **kw).cpu()
    first = [int((r == eos).nonzero()[0]) if (r == eos).any() else None for r in new]
    n = max(f for f in first) + 1 if all(f is not None for f in first) else 16
    assert e.shape == (4, 9 + n)
    for r, f in enumerate(first):
        stop = n if f is None else f + 1
        assert torch.equal(e[r, 9:9 + stop], new[r, :stop])
        assert (e[r, 9 + stop:] == pad).all()
    # every row done: eos = pad tokens everywhere after the first all-done step
    a1 = G.generate_ids(m, vision, ids[:1], seed=123, **kw)
    g = G.generate_ids(m, vision, ids[:1], seed=123, eos_token_id=int(a1[0, 9]), pad_token_id=pad, **kw)
    assert g.shape == (1, 10)


@gpu
def test_the_decode_loop_does_not_synchronise_and_replays_its_graph(lib_built, monkeypatch):
    fix = load_golden("gpt2_tiny_b6")
    m = build_filled_model(fix, "bf16", "cuda")
    vision, ids = _prompt(fix, 2, 9)
    loop = G._device_loop

    def strict(*a, **k):
        torch.cuda.set_sync_debug_mode("error")
        try:
            return loop(*a, **k)
        finally:
            torch.cuda.set_sync_debug_mode(0)
    monkeypatch.setattr(G, "_device_loop", strict)
    kw = dict(max_new_tokens=10, eos_token_id=96, pad_token_id=0)
    n0 = G.CAPTURES
    x = G.generate_ids(m, vision, ids, seed=5, **kw)
    assert G.CAPTURES == n0 + 1
    y = G.generate_ids(m, vision, ids, seed=5, **kw)
    assert G.CAPTURES == n0 + 1 and torch.equal(x, y)
    G.generate_ids(m, vision, ids, seed=5, max_new_tokens=11, eos_token_id=96, pad_token_id=0)
    assert G.CAPTURES == n0 + 2


@gpu
def test_generate_batch_with_a_seed_through_the_mllm(lib_built):
    fix = load_golden("tiny_b6")
    m = build_filled_model(fix, "bf16", "cuda")
    vision, ids = _prompt(fix, 2, 12)
    ref = G.generate_ids(m, vision, ids, max_new_tokens=16, temperature=0.9, top_k=40, top_p=0.9, eos_token_id=96, pad_token_id=0, seed=7).cpu()
    marker_tok = int(ref[0, 14])
    marker = "No right-following vehicle."

    class Tok:
        eos_token_id, pad_token_id = 96, 0

        def decode(self, row, skip_special_tokens=True):
            return " ".join(marker if int(t) == marker_tok else f"t{int(t)}" for t in row if not (skip_special_tokens and int(t) in (0, 96)))
    m.mllm.tokenizer = Tok()
    texts = m.mllm.generate_batch(vision_embs=vision, prompt_ids=ids, tokenizer=m.mllm.tokenizer, max_new_tokens=16, temperature=0.9, top_k=40,
                                  top_p=0.9, device="cuda", seed=7)
    want = []
    for row in ref:
        t = Tok().decode(row)
        want.append(t[: t.index(marker) + len(marker)] if marker in t else t)
    assert texts == want and marker in texts[0] and texts[0].endswith(marker)
