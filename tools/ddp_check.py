"""2-GPU check of the reference's own training loop on this model: DistributedDataParallel + torch.optim.AdamW + loss.backward()
(reference scripts/train.py:1127-1132, im_kim_train_GRN.py:1028-1040), and of tcavp_b200.FineTuner with its flat-gradient NCCL all-reduce.
Both must reproduce a single-process run on the concatenated batch (gradient averaging == mean of the per-rank MSE losses).  A third leg
runs FineTuner(max_grad_norm=1.0, skip_nonfinite=True): a NaN loss on rank 1 alone must make every rank skip, and two clipped steps must
reproduce the single-process run with clip_grad_norm_(params, 1.0) before AdamW.
    torchrun --nproc-per-node 2 tools/ddp_check.py"""
import os, sys, warnings
import torch
import torch.distributed as dist
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import tcavp_b200 as T
from conftest import load_golden

warnings.simplefilter("ignore")
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
dist.init_process_group("nccl")
fix = load_golden("tiny_b5_grads")
i = fix["inputs"]
B = 4                                                   # 2 scenes per rank
sel = slice(rank * 2, rank * 2 + 2)


def model():
    m = T.MultiModalTrajectoryModel(**fix["model_cfg"], compute_dtype="fp32")
    sd = m.state_dict(); T.deterministic_fill_(sd, fix["weight_seed"]); m.load_state_dict(sd, strict=True)
    return m.cuda().eval()      # deterministic comparison: every dropout off (train mode draws rank-dependent masks)


def batch(s):
    return (i["x"][s].cuda(), i["vision"][s].cuda(), ["c"] * 2, i["polygon"][s].cuda(), i["poly_len"][s]), dict(
        y=i["y"][s].cuda(), norm_stat=i["norm_stat"][s], input_ids=i["input_ids"][s].cuda(), attention_mask=i["attention_mask"][s].cuda())


# ---- (a) reference loop under DDP vs one process on the 4-scene batch ----
m = model()
ddp = torch.nn.parallel.DistributedDataParallel(m, device_ids=[torch.cuda.current_device()])
opt = torch.optim.AdamW([p for p in ddp.parameters() if p.requires_grad], lr=5e-4, weight_decay=1e-4)
a, kw = batch(sel)
for _ in range(2):
    opt.zero_grad()
    loss, _ = ddp(*a, **kw)
    loss.backward()
    opt.step()
ref = model()
opt2 = torch.optim.AdamW([p for p in ref.parameters() if p.requires_grad], lr=5e-4, weight_decay=1e-4)
af = (i["x"][:B].cuda(), i["vision"][:B].cuda(), ["c"] * B, i["polygon"][:B].cuda(), i["poly_len"][:B])
kwf = dict(y=i["y"][:B].cuda(), norm_stat=i["norm_stat"][:B], input_ids=i["input_ids"][:B].cuda(), attention_mask=i["attention_mask"][:B].cuda())
for _ in range(2):
    opt2.zero_grad()
    l2, _ = ref(*af, **kwf)
    l2.backward()
    opt2.step()
# ---- (b) FineTuner (flat gradient bucket, one NCCL all-reduce, fused AdamW) ----
m3 = model()
ft = T.FineTuner(m3, lr=5e-4, weight_decay=1e-4, use_cuda_graph=True)
for _ in range(2):
    ft.step(a[0], a[1], a[2], a[3], a[4], kw["y"], kw["norm_stat"], kw["input_ids"], kw["attention_mask"])
torch.cuda.synchronize()
# ---- (c) FineTuner with clipping and non-finite skipping vs the single-process loop with clip_grad_norm_ ----
m4 = model()
ft4 = T.FineTuner(m4, lr=5e-4, weight_decay=1e-4, use_cuda_graph=True, max_grad_norm=1.0, skip_nonfinite=True)
p0 = ft4.flat_p.clone()
y_nan = kw["y"].clone()
y_nan.view(-1)[0] = float("nan")
ft4.step(a[0], a[1], a[2], a[3], a[4], y_nan if rank == 1 else kw["y"], kw["norm_stat"], kw["input_ids"], kw["attention_mask"])
torch.cuda.synchronize()
bad_skip = int(not torch.equal(ft4.flat_p, p0) or int(ft4.skipped_steps) != 1 or int(ft4.step_counter) != 0)
for _ in range(2):
    ft4.step(a[0], a[1], a[2], a[3], a[4], kw["y"], kw["norm_stat"], kw["input_ids"], kw["attention_mask"])
ref_c = model()
params_c = [p for p in ref_c.parameters() if p.requires_grad]
opt_c = torch.optim.AdamW(params_c, lr=5e-4, weight_decay=1e-4)
for _ in range(2):
    opt_c.zero_grad()
    l3, _ = ref_c(*af, **kwf)
    l3.backward()
    torch.nn.utils.clip_grad_norm_(params_c, 1.0)
    opt_c.step()
torch.cuda.synchronize()
ILL = ("lane_polygon_encoder.pos_embedding", "lane_polygon_encoder.input_proj", "lane_polygon_encoder.encoder.layers.0.self_attn.in_proj")
bad_ddp = bad_ft = bad_clip = n = 0
for (k, p), (_, q), (_, r), (_, qc), (_, rc) in zip(m.named_parameters(), ref.named_parameters(), m3.named_parameters(),
                                                    ref_c.named_parameters(), m4.named_parameters()):
    if not p.requires_grad or k.startswith(ILL) or k.endswith("in_proj_bias"):
        continue
    n += 1
    tol = 1e-5 + 2e-3 * q.abs()
    bad_ddp += float(((p - q).abs() > tol).float().mean()) > 5e-3
    bad_ft += float(((r - q).abs() > tol).float().mean()) > 5e-3
    bad_clip += float(((rc - qc).abs() > 1e-5 + 2e-3 * qc.abs()).float().mean()) > 5e-3
t = torch.tensor([bad_ddp, bad_ft, bad_clip, bad_skip], device="cuda", dtype=torch.float32)
dist.all_reduce(t)
if rank == 0:
    print(f"ddp_check: {n} tensors; DDP-vs-single mismatching tensors {int(t[0])}, FineTuner-vs-single {int(t[1])}, "
          f"clipped FineTuner-vs-single {int(t[2])}; ranks that did not skip the NaN step {int(t[3])}")
    print("ddp_check ok" if float(t.sum()) == 0 else "ddp_check FAILED")
dist.destroy_process_group()
