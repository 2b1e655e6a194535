"""Gradient-norm clipping and non-finite step skipping of the native fine-tune loop (reference modify_scripts/modify_train.py:1190-1196,
scripts/modify_im_kim_train.py: clip_grad_norm_ before optimizer.step(), a NaN loss skips the step): the norm prologue against an fp64
norm, the clipped AdamW against tcavp_adamw, FineTuner(max_grad_norm / skip_nonfinite) against the reference loop with
torch.nn.utils.clip_grad_norm_ and torch.optim.AdamW, and the skip decision across two ranks."""
import math
import socket

import pytest
import torch
import torch.distributed as dist

pytestmark = pytest.mark.gpu

import tcavp_b200 as T  # noqa: E402
from conftest import load_golden  # noqa: E402
from tcavp_b200 import ops  # noqa: E402
from test_train_gpu import ILL, _model, _step  # noqa: E402

DEV = "cuda"


def _workspace():
    return torch.empty(ops.CLIP_WORKSPACE_BYTES // 8, dtype=torch.float64, device=DEV)


def _prologue(g, grad_scale=1.0, max_norm=None, loss=None, skip_nonfinite=False):
    rec = ops.clip_record(DEV)
    ops.clip_prologue(g, rec, _workspace(), grad_scale=grad_scale, max_norm=max_norm, loss=loss, skip_nonfinite=skip_nonfinite)
    torch.cuda.synchronize()
    return rec


def _skip(rec):
    return int(rec.view(torch.int32)[2])


def _ordered(x):
    """fp32 bit patterns as integers that are monotonic in the value: a difference of k = k ulps apart."""
    i = x.contiguous().view(torch.int32).long()
    return torch.where(i < 0, -(i & 0x7FFFFFFF), i)


def _ulps(a, b):
    return int((_ordered(a) - _ordered(b)).abs().max())


# ---- tcavp_clip_prologue ---------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("n,offset", [(1, 0), (255, 0), (255, 1), (2 ** 20 + 3, 0), (2 ** 20 + 3, 1), (60_000_000, 0)])
def test_prologue_norm_matches_fp64(lib_built, n, offset):
    """offset 1 puts the buffer off its 16-byte alignment (the scalar path)."""
    gen = torch.Generator(device=DEV).manual_seed(n + offset)
    buf = torch.randn(n + offset, device=DEV, generator=gen) * torch.exp(2.0 * torch.randn(n + offset, device=DEV, generator=gen))
    g = buf[offset:]
    rec = _prologue(g, grad_scale=0.5, max_norm=1.0)
    want = float(torch.linalg.vector_norm(0.5 * g.double()))
    assert abs(float(rec[0]) - want) <= 1e-6 * want, (float(rec[0]), want)
    assert _skip(rec) == 0 and int(rec.view(torch.int32)[3]) == 0


def test_prologue_is_bitwise_reproducible_in_calls_and_graph_replays(lib_built):
    gen = torch.Generator(device=DEV).manual_seed(7)
    g = torch.randn(2 ** 24 + 5, device=DEV, generator=gen)
    rec, ws = ops.clip_record(DEV), _workspace()
    runs = []
    for _ in range(2):
        ops.clip_prologue(g, rec, ws, grad_scale=0.25, max_norm=3.0)
        runs.append(rec.clone())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        ops.clip_prologue(g, rec, ws, grad_scale=0.25, max_norm=3.0)
    for _ in range(2):
        rec.zero_()
        graph.replay()
        runs.append(rec.clone())
    torch.cuda.synchronize()
    for r in runs[1:]:
        assert torch.equal(r.view(torch.int32), runs[0].view(torch.int32))
    assert 0 < float(runs[0][1]) < 1


def test_prologue_nonfinite_gradient_and_loss(lib_built):
    g = torch.randn(100_003, device=DEV)
    g[777] = math.inf
    rec = _prologue(g, max_norm=1.0)
    assert float(rec[0]) == math.inf and _skip(rec) == 0          # no skip unless asked
    assert _skip(_prologue(g, max_norm=1.0, skip_nonfinite=True)) == 1
    g[777] = math.nan
    rec = _prologue(g, max_norm=1.0, skip_nonfinite=True)
    assert math.isnan(float(rec[0])) and math.isnan(float(rec[1])) and _skip(rec) == 1
    g[777] = 0.5
    for loss, skip in ((1.25, 0), (math.nan, 1), (math.inf, 1), (-math.inf, 1)):
        rec = _prologue(g, max_norm=1.0, loss=torch.tensor(loss, device=DEV), skip_nonfinite=True)
        assert _skip(rec) == skip, loss
        assert math.isfinite(float(rec[0]))


def test_prologue_clip_coef_is_torchs(lib_built):
    gen = torch.Generator(device=DEV).manual_seed(11)
    g = torch.randn(3_000_017, device=DEV, generator=gen) * 0.01
    for max_norm in (1e-3, 0.37, 1.0, 17.0, 1e4):
        rec = _prologue(g, grad_scale=0.5, max_norm=max_norm)
        norm = rec[0:1].clone()
        want = torch.clamp(max_norm / (norm + 1e-6), max=1.0)         # torch.nn.utils.clip_grad_norm_ on the same fp32 norm
        assert _ulps(rec[1:2], want) <= 1, (max_norm, float(rec[1]), float(want))
    assert float(_prologue(g, max_norm=None)[1]) == 1.0


# ---- tcavp_adamw_clipped ---------------------------------------------------------------------------------------------------------

def _state(n, seed):
    gen = torch.Generator(device=DEV).manual_seed(seed)
    return [torch.randn(n, device=DEV, generator=gen) for _ in range(2)] + [torch.zeros(n, device=DEV) for _ in range(2)]


def test_adamw_clipped_with_unit_coefficient_matches_adamw(lib_built):
    n = 1_000_003
    p, _, m, v = _state(n, 3)
    p2, m2, v2 = p.clone(), m.clone(), v.clone()
    rec = ops.clip_record(DEV)
    rec[1] = 1.0
    step, skipped = torch.zeros((), dtype=torch.int32, device=DEV), torch.zeros((), dtype=torch.int32, device=DEV)
    gen = torch.Generator(device=DEV).manual_seed(4)
    for t in range(1, 4):
        g = torch.randn(n, device=DEV, generator=gen)
        ops.adamw_(p, g, m, v, lr=5e-4, weight_decay=1e-4, step=t, grad_scale=0.5)
        ops.adamw_clipped_(p2, g, m2, v2, record=rec, step=step, skipped=skipped, lr=5e-4, weight_decay=1e-4, grad_scale=0.5)
    torch.cuda.synchronize()
    assert int(step) == 3 and int(skipped) == 0
    assert torch.equal(m, m2) and torch.equal(v, v2)
    assert _ulps(p, p2) <= 1                # bias corrections: the host's powf there, the device's here


def test_adamw_clipped_scales_the_gradient_by_the_coefficient(lib_built):
    n = 65_537
    p, g, m, v = _state(n, 5)
    p2, m2, v2 = p.clone(), m.clone(), v.clone()
    rec = ops.clip_record(DEV)
    rec[1] = 0.25
    step = torch.zeros((), dtype=torch.int32, device=DEV)
    ops.adamw_(p, g, m, v, lr=5e-4, weight_decay=1e-4, step=1, grad_scale=0.125)
    ops.adamw_clipped_(p2, g, m2, v2, record=rec, step=step, lr=5e-4, weight_decay=1e-4, grad_scale=0.5)
    torch.cuda.synchronize()
    assert torch.equal(m, m2) and torch.equal(v, v2) and _ulps(p, p2) <= 1


def test_adamw_clipped_skip_touches_nothing(lib_built):
    n = 300_007
    p, g, m, v = _state(n, 6)
    m.normal_()
    v.uniform_()
    rec = ops.clip_record(DEV)
    rec[1] = 0.5
    rec.view(torch.int32)[2] = 1
    step = torch.full((), 5, dtype=torch.int32, device=DEV)
    skipped = torch.full((), 2, dtype=torch.int32, device=DEV)
    before = [t.clone() for t in (p, g, m, v, step)]
    ops.adamw_clipped_(p, g, m, v, record=rec, step=step, skipped=skipped, lr=5e-4, weight_decay=1e-4)
    torch.cuda.synchronize()
    for a, b in zip(before, (p, g, m, v, step)):
        assert torch.equal(a.view(torch.int32), b.view(torch.int32))
    assert int(skipped) == 3


# ---- FineTuner ---------------------------------------------------------------------------------------------------------------------

def _ft_args(i, y=None):
    return (i["x"].cuda(), i["vision"].cuda(), ["ctx"] * i["x"].shape[0], i["polygon"].cuda(), i["poly_len"],
            (i["y"] if y is None else y).cuda(), i["norm_stat"], i["input_ids"].cuda(), i["attention_mask"].cuda())


def _flat_views(ft, flat):
    off = 0
    for n, p in zip(ft.names, ft.params):
        yield n, flat[off:off + p.numel()].view_as(p)
        off += p.numel()


@pytest.mark.parametrize("frozen_mllm", [False, True])
@pytest.mark.parametrize("graph", [False, True])
def test_finetuner_clipping_matches_the_reference_loop(lib_built, graph, frozen_mllm):
    """FineTuner(max_grad_norm=1.0) against forward, loss.backward(), clip_grad_norm_(params, 1.0), torch.optim.AdamW.step()
    (scripts/modify_im_kim_train.py).  frozen_mllm: only the encoders and the head train, so the late (mllm.*) slice is empty."""
    fix = load_golden("tiny_b5_grads")
    i = fix["inputs"]
    m, m_ref = _model(fix, "fp32", frozen_mllm), _model(fix, "fp32", frozen_mllm)
    params_ref = [p for p in m_ref.parameters() if p.requires_grad]
    opt = torch.optim.AdamW(params_ref, lr=5e-4, weight_decay=1e-4)
    import warnings
    warnings.simplefilter("ignore")
    c = 1.0
    ft = T.FineTuner(m, lr=5e-4, weight_decay=1e-4, use_cuda_graph=graph, max_grad_norm=c)
    assert (ft.n_late == 0) == frozen_mllm
    named_ref = dict(m_ref.named_parameters())
    for step in range(3):
        loss, dec = ft.step(*_ft_args(i))
        opt.zero_grad()
        l2, d2 = _step(m_ref, i)
        l2.backward()
        ref_norm = float(torch.nn.utils.clip_grad_norm_(params_ref, c))
        opt.step()
        torch.cuda.synchronize()
        norm = float(ft.grad_norm)
        assert norm > c and float(ft._clip_rec[1]) < 1, (step, norm)           # clipping engaged
        assert abs(norm - ref_norm) <= 1e-4 * ref_norm, (step, norm, ref_norm)
        assert abs(float(l2) - float(loss)) <= 2e-4 * abs(float(loss)), (step, float(l2), float(loss))
        torch.testing.assert_close(dec, d2, rtol=1e-3, atol=1e-3)
        if step == 0:
            # same weights on both sides: the first moment is (1 - beta1) x the CLIPPED gradient on both, compared with the band
            # test_finetuner_matches_the_reference_loop puts on the gradients, scaled by the same factor
            scale = 0.1 * float(ft._clip_rec[1])
            for n, ea in _flat_views(ft, ft.exp_avg):
                if n.startswith(ILL):
                    continue
                want = opt.state[named_ref[n]]["exp_avg"]
                torch.testing.assert_close(ea, want, rtol=2e-3, atol=1e-6 * scale + 1e-4 * float(want.abs().max()),
                                           msg=lambda s, n=n: f"{n}: {s}")
    assert int(ft.step_counter) == 3 and int(ft.skipped_steps) == 0 and ft.steps == 3


@pytest.mark.parametrize("graph", [False, True])
def test_finetuner_skips_a_nonfinite_loss_like_the_reference(lib_built, graph):
    """A NaN in y makes the loss NaN: the step leaves parameters, moments and the device step untouched, and the following steps
    match a reference loop that did `if not torch.isfinite(loss): continue` (modify_scripts/modify_train.py:1190-1196)."""
    fix = load_golden("tiny_b5_grads")
    i = fix["inputs"]
    y_nan = i["y"].clone()
    y_nan.view(-1)[3] = math.nan
    m, m_ref = _model(fix, "fp32"), _model(fix, "fp32")
    opt = torch.optim.AdamW([p for p in m_ref.parameters() if p.requires_grad], lr=5e-4, weight_decay=1e-4)
    import warnings
    warnings.simplefilter("ignore")
    ft = T.FineTuner(m, lr=5e-4, weight_decay=1e-4, use_cuda_graph=graph, skip_nonfinite=True)
    for k, y in enumerate([None, y_nan, None, None]):
        if k == 1:
            torch.cuda.synchronize()
            before = [t.clone() for t in (ft.flat_p, ft.exp_avg, ft.exp_avg_sq, ft.step_counter)]
        loss, dec = ft.step(*_ft_args(i, y))
        opt.zero_grad()
        l2, d2 = _step(m_ref, dict(i, y=i["y"] if y is None else y))
        if k == 1:
            torch.cuda.synchronize()
            assert not math.isfinite(float(loss)) and not torch.isfinite(l2)
            for a, b in zip(before, (ft.flat_p, ft.exp_avg, ft.exp_avg_sq, ft.step_counter)):
                assert torch.equal(a.view(torch.int32), b.view(torch.int32))
            assert int(ft.skipped_steps) == 1 and int(ft.step_counter) == 1
            continue
        l2.backward()
        opt.step()
        assert abs(float(l2) - float(loss)) <= 2e-4 * abs(float(loss)), (k, float(l2), float(loss))
        torch.testing.assert_close(dec, d2, rtol=1e-3, atol=1e-3)
    assert int(ft.step_counter) == 3 and int(ft.skipped_steps) == 1


def _labels(fn):
    prof = ops.LaunchProfiler()
    with prof:
        fn()
    torch.cuda.synchronize()
    return {rec[0].split("[")[0] for rec in prof.rec}


def test_launch_sequence_has_the_clip_kernels_only_when_asked(lib_built):
    fix = load_golden("tiny_b5_grads")
    i = fix["inputs"]
    import warnings
    warnings.simplefilter("ignore")
    off = T.FineTuner(_model(fix, "fp32"), use_cuda_graph=False)
    got = _labels(lambda: off.step(*_ft_args(i)))
    assert "adamw_kernel" in got and not {"clip_norm_kernel", "adamw_clipped_kernel", "mark_nonfinite_kernel"} & got
    assert off.grad_norm is None and off.step_counter is None and off.skipped_steps is None
    on = T.FineTuner(_model(fix, "fp32"), use_cuda_graph=False, max_grad_norm=1.0)
    got = _labels(lambda: on.step(*_ft_args(i)))
    assert {"clip_norm_kernel", "adamw_clipped_kernel"} <= got and "adamw_kernel" not in got


# ---- two ranks ---------------------------------------------------------------------------------------------------------------------

def _two_rank_worker(rank, backend, port):
    import warnings
    warnings.simplefilter("ignore")
    torch.cuda.set_device(rank if backend == "nccl" else 0)
    dist.init_process_group(backend, init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=2)
    try:
        fix = load_golden("tiny_b5_grads")
        i = fix["inputs"]
        sel = slice(2 * rank, 2 * rank + 2)
        part = {k: v[sel] for k, v in i.items()}
        y_nan = part["y"].clone()
        y_nan.view(-1)[0] = math.nan
        for overlap, frozen in ((False, False), (True, False), (True, True)):
            ft = T.FineTuner(_model(fix, "fp32", frozen), lr=5e-4, weight_decay=1e-4, overlap_allreduce=overlap, max_grad_norm=1.0,
                             skip_nonfinite=True)
            p0 = ft.flat_p.clone()
            ft.step(*_ft_args(part, y_nan if rank == 1 else None))          # only rank 1 sees the NaN: both ranks skip
            torch.cuda.synchronize()
            assert torch.equal(ft.flat_p, p0), (rank, overlap, frozen)
            assert int(ft.skipped_steps) == 1 and int(ft.step_counter) == 0, (rank, overlap, frozen)
            for _ in range(2):
                ft.step(*_ft_args(part))
            torch.cuda.synchronize()
            assert int(ft.step_counter) == 2 and float(ft._clip_rec[1]) < 1
            mine = torch.cat([ft.flat_p, ft.grad_norm.reshape(1)])
            mine = mine if backend == "nccl" else mine.cpu()
            both = [torch.empty_like(mine) for _ in range(2)]
            dist.all_gather(both, mine)
            assert torch.equal(both[0], both[1]), (rank, overlap, frozen)       # same parameters and norm, bit for bit
            assert not torch.equal(ft.flat_p, p0)
    finally:
        dist.destroy_process_group()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.parametrize("backend", ["nccl", "gloo"])
def test_two_ranks_skip_together_and_stay_identical(lib_built, backend):
    """nccl: one rank per GPU.  gloo: both ranks on one GPU, so the rank-consistency path also runs on a one-GPU machine."""
    if backend == "nccl" and torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    mp.spawn(_two_rank_worker, args=(backend, _free_port()), nprocs=2, join=True)
