"""Fine-tune step parity (SURVEY.md §8 row a11): gradients of every trainable tensor from the hand-written CUDA backward
against (a) the golden gradients minted from the unmodified reference and (b) autograd through the CPU oracle on the same
inputs.  These fixtures run in eval mode (every dropout off, reference scripts/im_kim_train_GRN.py:1029-1040 semantics otherwise);
train mode with the reference's dropout at every site is tests/test_dropout_gpu.py."""
import pytest
import torch

pytestmark = pytest.mark.gpu

import tcavp_b200 as T  # noqa: E402
from conftest import load_golden  # noqa: E402
from oracle import restated  # noqa: E402
from test_oracle_cpu import _check_against_compressed  # noqa: E402

# The first lane-polygon attention sees raw pixel coordinates (logits ~1e6): its fp32 gradients are ill-conditioned (the
# reference's own fp32 backward is 20-30 % off its fp64 result there, oracle/make_golden.py).  Those tensors get a wider band.
ILL = ("lane_polygon_encoder.pos_embedding", "lane_polygon_encoder.input_proj", "lane_polygon_encoder.encoder.layers.0.self_attn.in_proj")


def _model(fix, dtype, frozen_mllm=False):
    m = T.MultiModalTrajectoryModel(**fix["model_cfg"], compute_dtype=dtype)
    sd = m.state_dict()
    T.deterministic_fill_(sd, fix["weight_seed"])
    m.load_state_dict(sd, strict=True)
    if frozen_mllm:                                     # reference scripts/train.py:1141-1142
        for p in m.mllm.parameters():
            p.requires_grad_(False)
    # p = 0 goldens were minted in eval mode (every dropout off, autograd on); `*_drop` goldens in train() mode
    m = m.to("cuda")
    return m.train() if fix.get("dropout") else m.eval()


def _step(m, i):
    dev = {k: (v.cuda() if torch.is_tensor(v) else v) for k, v in i.items()}
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        loss, dec = m(dev["x"], dev["vision"], ["ctx"] * dev["x"].shape[0], dev["polygon"], i["poly_len"], y=dev["y"], norm_stat=i["norm_stat"],
                      input_ids=dev["input_ids"], attention_mask=dev["attention_mask"])
    return loss, dec


def _oracle(fix):
    m = T.MultiModalTrajectoryModel(**fix["model_cfg"])
    sd = m.state_dict()
    T.deterministic_fill_(sd, fix["weight_seed"])
    i = fix["inputs"]
    return restated.loss_and_grads(sd, fix["model_cfg"], fix["llama_cfg"], i["x"], i["vision"], i["polygon"], i["poly_len"], i["input_ids"],
                                   i["attention_mask"], i["y"], i["norm_stat"])


@pytest.mark.parametrize("name", ["tiny_b5_grads", "cfg1_b3_grads", "cfg3l2_b4_grads", "gpt2_tiny_b5_grads", "gpt2_l2_b3_grads"])
def test_fp32_gradients_match_reference(lib_built, name):
    fix = load_golden(name)
    m = _model(fix, "fp32")
    loss, dec = _step(m, fix["inputs"])
    assert loss.requires_grad and not dec.requires_grad
    loss.backward()
    torch.cuda.synchronize()
    torch.testing.assert_close(loss.detach().cpu(), fix["loss"], rtol=1e-4, atol=0)
    torch.testing.assert_close(dec.cpu(), fix["decoded"], rtol=1e-4, atol=5e-4)
    got = {n: p.grad for n, p in m.named_parameters() if p.requires_grad}
    assert set(got) == set(fix["grads"])
    o_loss, _, o_grads = _oracle(fix)
    # Band relative to each tensor's largest gradient entry.  At the 7B-class geometry (contractions of 4096 / 11008 / 22016 terms summed
    # in plain fp32 order, then carried back through both decoder layers and the whole Q-Former) the fp32 noise floor of the deepest
    # tensors (Q-Former encoder, vision_proj) sits at ~2e-3 of their largest entry on < 1 % of the elements; the 768-class chain stays
    # under 1e-3.  The fp64 golden is the reference in both cases.
    band = 4e-3 if name == "cfg3l2_b4_grads" else 1e-3
    worst, failures = {}, []
    for k, want in fix["grads"].items():
        assert got[k] is not None, f"no gradient for {k}"
        ref = want["full"] if "full" in want else want["head"]
        scale = float(ref.abs().max()) + 1e-8
        ill = k.startswith(ILL)
        full = o_grads[k]
        err = float((got[k].float().cpu() - full).abs().max()) / (float(full.abs().max()) + 1e-8)
        worst[k] = err
        try:
            _check_against_compressed(got[k], want, rtol=0.3 if ill else 5e-3, atol=(0.3 if ill else band) * scale + 1e-6, key=k)
            assert err < (0.3 if ill else 2 * band), (k, err)
        except AssertionError as e:
            # where does the error sit?  (a ReLU unit whose pre-activation is ~0 for one token flips between fp32 evaluation orders and
            # moves exactly one row of linear1.weight / one entry of linear1.bias)
            d = (got[k].float().cpu() - full).abs().reshape(full.shape[0], -1) / (float(full.abs().max()) + 1e-8)
            rows = d.max(dim=1).values
            top = torch.topk(rows, min(4, rows.numel()))
            failures.append((k, err, str(e)[:200], {"rows_over_band": int((rows > band).sum()), "n_rows": int(rows.numel()),
                                                    "top_rows": [(int(i), float(v)) for v, i in zip(top.values, top.indices)],
                                                    "frac_elems_over_band": float((d > band).float().mean())}))
    top = sorted(worst.items(), key=lambda kv: -kv[1])[:8]
    print("worst relative-to-max gradient errors:", top)
    # A ReLU unit whose pre-activation is within fp32 rounding of zero for one token is not differentiable there: its gate can differ
    # between two correct fp32 evaluation orders (and the fp64 golden), which moves exactly ONE row of that layer's linear1.weight /
    # one entry of linear1.bias by that token's whole contribution, and — through the unit — every gradient upstream of it by a small
    # amount that shows up in the row / column sums.  Such a flip is accepted when it is confined to <= 2 units of a layer and every
    # other element of every tensor stays inside the element-wise band.
    flips = [f for f in failures if f[0].endswith(("linear1.weight", "linear1.bias", "ffn.0.weight", "ffn.0.bias")) and 0 < f[3]["rows_over_band"] <= 2
             and f[3]["top_rows"][min(2, len(f[3]["top_rows"]) - 1)][1] < band]
    if flips:
        rest = [f for f in failures if f not in flips and not f[1] < 2 * band]
        print("ReLU-boundary flips:", [(f[0], f[3]["top_rows"][:2]) for f in flips])
        assert not rest, rest[:5]
    else:
        assert not failures, failures[:5]


@pytest.mark.parametrize("name", ["tiny_b5_grads", "cfg1_b3_grads", "cfg3l2_b4_grads", "gpt2_tiny_b5_grads", "gpt2_l2_b3_grads"])
def test_bf16_gradients_track_reference(lib_built, name):
    """bf16 storage: per-tensor direction and size of the gradient (cosine >= 0.98, norm within 10 %) for every tensor whose
    gradient is not itself at the noise floor."""
    fix = load_golden(name)
    m = _model(fix, "bf16")
    loss, _ = _step(m, fix["inputs"])
    loss.backward()
    torch.cuda.synchronize()
    assert abs(float(loss) - float(fix["loss"])) / float(fix["loss"]) < 2e-2
    _, _, o_grads = _oracle(fix)
    gmax = max(float(g.norm()) for g in o_grads.values())
    low, bad, checked = [], [], 0
    for n, p in m.named_parameters():
        if not p.requires_grad:
            continue
        g, w = p.grad.float().cpu().flatten(), o_grads[n].flatten()
        if float(w.norm()) < 1e-4 * gmax or n.startswith(ILL):
            continue
        checked += 1
        cos = float(torch.dot(g, w) / (g.norm() * w.norm() + 1e-30))
        ratio = float(g.norm() / (w.norm() + 1e-30))
        if cos < 0.98 or not 0.9 < ratio < 1.1:
            low.append((n, round(cos, 4), round(ratio, 4)))
        if cos < 0.95 or not 0.8 < ratio < 1.25:
            bad.append((n, round(cos, 4), round(ratio, 4)))
    # every tensor inside the wide band; at most 1 % of them (single channels of the 64 per-channel NLinear maps at the real geometry)
    # outside the tight one
    assert not bad, bad[:10]
    assert len(low) <= max(0, checked // 100), (checked, low[:10])


def test_frozen_mllm_mode_skips_llm_backward(lib_built):
    """reference scripts/train.py:1141-1145: the whole MLLM is frozen, only the polygon encoder and LTSF train."""
    fix = load_golden("tiny_b5_grads")
    m = _model(fix, "fp32", frozen_mllm=True)
    from tcavp_b200 import ops
    loss, _ = _step(m, fix["inputs"])
    n0 = ops.launch_count()
    loss.backward()
    n_frozen = ops.launch_count() - n0
    for n, p in m.named_parameters():
        assert (p.grad is not None) == (p.requires_grad), n
    _, _, o_grads = _oracle(fix)
    for n, p in m.named_parameters():
        if p.requires_grad and not n.startswith(ILL):
            err = float((p.grad.cpu() - o_grads[n]).abs().max()) / (float(o_grads[n].abs().max()) + 1e-8)
            assert err < 2e-3, (n, err)
    m2 = _model(fix, "fp32")
    loss2, _ = _step(m2, fix["inputs"])
    n0 = ops.launch_count()
    loss2.backward()
    assert ops.launch_count() - n0 > n_frozen      # the full mode also walks the LLM and the Q-Former


def test_adamw_steps_reduce_the_loss_and_match_torch_optimizer(lib_built):
    fix = load_golden("tiny_b5_grads")
    from tcavp_b200 import ops
    from tcavp_b200.distributed import FlatGradBucket
    m = _model(fix, "fp32")
    m_ref = _model(fix, "fp32")
    opt = torch.optim.AdamW([p for p in m_ref.parameters() if p.requires_grad], lr=5e-4, weight_decay=1e-4)
    bucket = FlatGradBucket(m.parameters())
    flat_p = torch.cat([p.detach().reshape(-1) for p in bucket.params])
    exp_avg, exp_avg_sq = torch.zeros_like(flat_p), torch.zeros_like(flat_p)
    losses = []
    for step in range(1, 4):
        # native loop: flat gradient bucket (one all-reduce in a multi-GPU job) + fused AdamW over the flat buffers
        bucket.zero_()
        loss, _ = _step(m, fix["inputs"])
        loss.backward()
        ops.adamw_(flat_p, bucket.flat, exp_avg, exp_avg_sq, lr=5e-4, weight_decay=1e-4, step=step)
        off = 0
        with torch.no_grad():
            for p in bucket.params:
                p.copy_(flat_p[off:off + p.numel()].view_as(p))
                off += p.numel()
        losses.append(float(loss))
        # reference loop (im_kim_train_GRN.py:1028-1040) with torch.optim.AdamW on the same gradients
        opt.zero_grad()
        l2, _ = _step(m_ref, fix["inputs"])
        l2.backward()
        opt.step()
        assert abs(float(l2) - float(loss)) <= 1e-4 * abs(float(loss))
    assert losses[-1] < losses[0], losses
    for (n, a), (_, b) in zip(m.named_parameters(), m_ref.named_parameters()):
        # the key third of every in_proj_bias has an identically zero true gradient (softmax is invariant to a key bias): what
        # reaches AdamW there is rounding noise whose sign decides the update
        if a.requires_grad and not n.startswith(ILL) and not n.endswith("in_proj_bias"):
            # AdamW's update is ~lr * sign(g) early on: an element whose gradient sits at the atomics' rounding noise can flip,
            # so the check is on the fraction of elements that moved differently, not on every element
            bad = ((a - b).abs() > 1e-5 + 1e-3 * b.abs()).float().mean()
            assert float(bad) < 2e-3, (n, float(bad))


@pytest.mark.parametrize("graph", [False, True])
def test_finetuner_matches_the_reference_loop(lib_built, graph):
    """tcavp_b200.FineTuner (gradients written straight into the flat bucket, optional CUDA-graph replay of forward+backward,
    fused AdamW) against the reference's loop — forward, loss.backward(), torch.optim.AdamW.step() (im_kim_train_GRN.py:1028-1040)."""
    fix = load_golden("tiny_b5_grads")
    i = fix["inputs"]
    m, m_ref = _model(fix, "fp32"), _model(fix, "fp32")
    opt = torch.optim.AdamW([p for p in m_ref.parameters() if p.requires_grad], lr=5e-4, weight_decay=1e-4)
    import warnings
    warnings.simplefilter("ignore")
    ft = T.FineTuner(m, lr=5e-4, weight_decay=1e-4, use_cuda_graph=graph)
    ctx = ["ctx"] * i["x"].shape[0]
    for step in range(3):
        loss, dec = ft.step(i["x"].cuda(), i["vision"].cuda(), ctx, i["polygon"].cuda(), i["poly_len"], i["y"].cuda(), i["norm_stat"],
                            i["input_ids"].cuda(), i["attention_mask"].cuda())
        opt.zero_grad()
        l2, d2 = _step(m_ref, i)
        l2.backward()
        if step == 0:      # same weights on both sides: the flat-bucket gradients are the autograd gradients
            torch.cuda.synchronize()
            assert sorted(ft.names) == sorted(n for n, _ in m.trainable_named_parameters())
            n_late = sum(v.numel() for n, v in zip(ft.names, ft.bucket.views) if n.startswith("mllm."))
            assert n_late == ft.n_late and all(n.startswith("mllm.") == (k < sum(x.startswith("mllm.") for x in ft.names)) for k, n in enumerate(ft.names))
            for n, v in zip(ft.names, ft.bucket.views):      # flat layout: mllm.* first (final late), the early-final slice behind it
                g = dict(m_ref.named_parameters())[n].grad
                if not n.startswith(ILL):
                    torch.testing.assert_close(v, g, rtol=2e-3, atol=1e-6 + 1e-4 * float(g.abs().max()), msg=lambda s, n=n: f"{n}: {s}")
        opt.step()
        assert abs(float(l2) - float(loss)) <= 2e-4 * abs(float(loss)), (step, float(l2), float(loss))
        torch.testing.assert_close(dec, d2, rtol=1e-3, atol=1e-3)
    assert ft.launches_per_step > 100
