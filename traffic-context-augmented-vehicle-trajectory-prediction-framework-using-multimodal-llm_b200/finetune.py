"""Native fine-tune loop (reference scripts/im_kim_train_GRN.py:1019-1041: zero_grad -> forward -> loss.backward() ->
AdamW.step(), wrapped in DistributedDataParallel, train.py:1127-1132).

`FineTuner` keeps every trainable tensor in ONE flat fp32 parameter buffer (the nn.Parameters are re-pointed to views of
it), their gradients in one flat buffer (`distributed.FlatGradBucket`) and the AdamW moments in two more, so a step is:
forward + hand-written backward (train_engine.py, gradients written straight into their slices of the flat buffer) -> the
all-reduce of the trainable gradients over NCCL (LoRA / Q-Former / encoder / fusion only; frozen base weights never move)
-> ONE fused AdamW launch (tcavp_adamw).  Forward + backward of a fixed batch shape are captured once in TWO CUDA graphs and
replayed (two host calls instead of ~900 kernel launches per step).  The cut sits where the backward pass enters the decoder
stack: everything outside `mllm.*` (regression head, cross-attention fusion — 4 H^2 parameters, half of the payload at the 7B
shape —, temporal and lane-polygon encoders) has its final gradient by then, so that slice of the flat buffer is all-reduced on
NCCL's stream WHILE the second graph (LoRA-Llama + Q-Former backward, the bulk of the step) runs; only the `mllm.*` slice is
exchanged after it.  DistributedDataParallel gets the same overlap from its gradient buckets (train.py:1127-1132).  The reference's own loop (torch.optim.AdamW + DDP
+ loss.backward()) also works unchanged on the same model — this class is the faster equivalent.

`max_grad_norm` / `skip_nonfinite` add the reference's two training safeguards (modify_scripts/modify_train.py:1190-1196: skip a step
whose loss is NaN, clip_grad_norm_; scripts/modify_im_kim_train.py: clip_grad_norm_(…, 1.0)).  Both are decided on the device, after the
all-reduce, so the step still needs no host synchronisation: tcavp_clip_prologue reads the reduced gradient once and writes the norm, the
clip coefficient and the skip flag, and tcavp_adamw_clipped applies them with the optimiser step count kept on the device."""
import math
import os

import torch
import torch.distributed as dist

from . import ops
from .distributed import FlatGradBucket


class FineTuner:
    def __init__(self, model, lr=5e-4, weight_decay=1e-4, betas=(0.9, 0.999), eps=1e-8, group=None, use_cuda_graph=True, max_graphs=8,
                 overlap_allreduce=None, max_grad_norm=None, skip_nonfinite=False):
        """max_grad_norm: clip the global L2 norm of the averaged gradient to this value before AdamW, as
        torch.nn.utils.clip_grad_norm_(params, max_grad_norm) after DDP's averaging does.  skip_nonfinite: leave the parameters, the
        moments and the step count untouched when the loss of any rank or the gradient norm is not finite (the reference's
        `if not torch.isfinite(loss): continue`).  A skipped step has still drawn its dropout masks: the mask counter advances inside
        the captured forward, as the reference's RNG advances in its forward."""
        if max_grad_norm is not None:
            max_grad_norm = float(max_grad_norm)
            if not (math.isfinite(max_grad_norm) and max_grad_norm > 0):
                raise ValueError(f"max_grad_norm must be finite and > 0, got {max_grad_norm}")
        self.max_grad_norm, self.skip_nonfinite = max_grad_norm, bool(skip_nonfinite)
        self.model, self.group = model, group
        self.lr, self.wd, self.betas, self.eps = lr, weight_decay, betas, eps
        named = model.trainable_named_parameters()
        # flat layout: `mllm.*` first (gradients final at the END of the backward pass), everything else behind it (final EARLY)
        named = [(n, p) for n, p in named if n.startswith("mllm.")] + [(n, p) for n, p in named if not n.startswith("mllm.")]
        self.n_late = sum(p.numel() for n, p in named if n.startswith("mllm."))
        # Overlapping pays when the early-final slice is a real share of the payload (7B shape: 275 of 537 MB — the 4 H^2 cross-attention
        # fusion weights); at the 768 shape it is 14 of 231 MB and the NCCL kernel only gets in the way of the persistent GEMM kernels
        # it shares the SMs with (measured on 2 B200: 88.8 vs 82.9 ms per step), so small slices ride in the one all-reduce at the end.
        # TCAVP_FT_OVERLAP=0 / 1 forces either form (A/B runs).
        n_early = sum(p.numel() for n, p in named if not n.startswith("mllm."))
        env = os.environ.get("TCAVP_FT_OVERLAP")
        if overlap_allreduce is not None:
            self.overlap = bool(overlap_allreduce)
        elif env is not None:
            self.overlap = env != "0"
        else:
            self.overlap = n_early * 4 >= (32 << 20)
        self.names = [n for n, _ in named]
        self.params = [p for _, p in named]
        if not self.params:
            raise ValueError("no trainable parameters")
        if any(p.dtype != torch.float32 for p in self.params):
            raise TypeError("trainable parameters must be fp32 (master weights)")
        dev = self.params[0].device
        n = sum(p.numel() for p in self.params)
        self.flat_p = torch.empty(n, dtype=torch.float32, device=dev)
        off = 0
        with torch.no_grad():
            for p in self.params:
                v = self.flat_p[off:off + p.numel()].view_as(p)
                v.copy_(p)
                p.data = v
                off += p.numel()
        self.bucket = FlatGradBucket(self.params)
        self.targets = dict(zip(self.names, self.bucket.views))
        self.exp_avg = torch.zeros_like(self.flat_p)
        self.exp_avg_sq = torch.zeros_like(self.flat_p)
        self.steps = 0                # step() calls
        # clip / skip state: the tcavp_clip_record of the last step, the prologue's workspace, the optimiser step count and the number of
        # skipped steps (device int32 each: a skip decided on the device cannot tell the host which step number comes next)
        self._clip_rec = self._clip_ws = self.step_counter = self.skipped_steps = None
        if self.max_grad_norm is not None or self.skip_nonfinite:
            self._clip_rec = ops.clip_record(dev)
            self._clip_ws = torch.empty(ops.CLIP_WORKSPACE_BYTES // 8, dtype=torch.float64, device=dev)
            self.step_counter = torch.zeros((), dtype=torch.int32, device=dev)
            self.skipped_steps = torch.zeros((), dtype=torch.int32, device=dev)
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.use_cuda_graph = use_cuda_graph
        # one captured graph (+ its static input buffers and output tensors) per input-shape signature: the reference collate pads the
        # prompt to the longest sequence of each batch (train.py:323-325), so L_text moves from step to step and a single-slot cache would
        # re-capture almost every step.  Least-recently-used entries are dropped beyond `max_graphs` (each holds one step's activations).
        self._graphs = {}
        self.max_graphs = max_graphs
        self.captures = 0
        self.launches_per_step = 0    # libtcavp launches of one forward + backward (captured launches are replayed, not re-counted)
        # train() mode applies the reference's dropout at every site (counter-based masks; the step counter lives on the device and is
        # advanced inside the captured graph).  Ranks draw different masks, as DDP ranks with different RNG offsets do.
        self.dropout_active = model.dropout_active()
        if self.dropout_active:
            rank = dist.get_rank(group) if dist.is_initialized() else 0
            model.set_dropout_seed((torch.initial_seed() + 7919 * rank) & 0x7FFFFFFF, 0)

    @property
    def grad_norm(self):
        """Device fp32 scalar: the global gradient norm of the last step before clipping (what clip_grad_norm_ returns); None when
        neither option is set.  The next step overwrites it."""
        return None if self._clip_rec is None else self._clip_rec[0]

    @property
    def payload_bytes(self):
        """Bytes exchanged by the one all-reduce of a step."""
        return self.bucket.flat.numel() * self.bucket.flat.element_size()

    # ---- forward + backward into the flat gradient buffer (no autograd graph, no per-tensor accumulation) --------------
    def _copy_grads(self, grads):
        for name, g in grads.items():
            view = self.targets.get(name)
            if view is not None and g is not None and g.data_ptr() != view.data_ptr():
                view.copy_(g.reshape(view.shape))

    @torch.no_grad()
    def _fwd_early(self, inp):
        """Forward + the part of the backward pass that finishes every gradient outside `mllm.*`."""
        eng = self.model.train_engine()
        eng.grad_targets = self.targets
        self.bucket.flat.zero_()
        try:
            out = eng.train_forward(**inp)
            st = eng.train_backward_early(None)
            self._copy_grads(st["early"])
        except BaseException:
            eng.grad_targets = None
            raise
        return (out["loss"], out["decoded"]), st

    @torch.no_grad()
    def _late(self, st):
        eng = self.model.train_engine()
        try:
            grads = eng.train_backward_late(st)
            self._copy_grads({k: v for k, v in grads.items() if k.startswith("mllm.")})
        finally:
            eng.grad_targets = None

    def _fwd_bwd(self, inp):
        out, st = self._fwd_early(inp)
        self._late(st)
        return out

    def _device_inputs(self, x, vision_embs, lane_polygon_batch, lane_polygon_len, y, norm_stat, input_ids, attention_mask):
        dev = self.flat_p.device
        lens = lane_polygon_len if torch.is_tensor(lane_polygon_len) else torch.tensor(list(lane_polygon_len), dtype=torch.int32)
        ns = norm_stat if torch.is_tensor(norm_stat) else torch.tensor(norm_stat, dtype=torch.float32)
        f32 = lambda t: t.to(device=dev, dtype=torch.float32, non_blocking=True).contiguous()      # noqa: E731
        vis = vision_embs.to(dev, non_blocking=True)
        if vis.dtype not in (torch.float32, torch.bfloat16):
            vis = vis.float()
        return dict(x=f32(x), vision=vis.contiguous(), polygon=f32(lane_polygon_batch), poly_len=lens.to(device=dev, dtype=torch.int32),
                    input_ids=input_ids.to(device=dev, dtype=torch.int64).contiguous(),
                    attention_mask=attention_mask.to(device=dev, dtype=torch.int64).contiguous(), y=f32(y), norm_stat=f32(ns).view(-1, 4))

    def _stages(self, inp):
        """The step's device work as two callables: first() -> (loss, decoded) runs forward + early backward, second() the rest."""
        if not self.use_cuda_graph:
            box = {}

            def first():
                box["n0"] = ops.launch_count()
                out, box["st"] = self._fwd_early(inp)
                return out

            def second():
                self._late(box.pop("st"))
                self.launches_per_step = ops.launch_count() - box["n0"]
            return first, second
        sig = tuple((k, tuple(v.shape), v.dtype) for k, v in inp.items())
        ent = self._graphs.pop(sig, None)
        if ent is None:
            # static input buffers + two eager steps on a side stream (lazy packing, cudaFuncSetAttribute, allocator warm-up), then capture
            static = {k: v.clone() for k, v in inp.items()}
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                for _ in range(2):
                    self._fwd_bwd(static)
            torch.cuda.current_stream().wait_stream(s)
            torch.cuda.synchronize()
            g1, g2 = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
            n0 = ops.launch_count()
            with torch.cuda.graph(g1):
                out, st = self._fwd_early(static)
            with torch.cuda.graph(g2, pool=g1.pool()):        # same private pool: the activation stash of g1 stays allocated for g2
                self._late(st)
            del st
            ent = (g1, g2, static, out, ops.launch_count() - n0)
            self.captures += 1
            while len(self._graphs) >= max(1, self.max_graphs):
                self._graphs.pop(next(iter(self._graphs)))        # dicts keep insertion order: the first key is the least recently used
        self._graphs[sig] = ent                                   # (re-)inserted last = most recently used
        g1, g2, static, out, self.launches_per_step = ent

        def first():
            for k, v in inp.items():
                static[k].copy_(v, non_blocking=True)
            g1.replay()
            # the graph's output tensors are overwritten by the next replay: hand out copies
            return out[0].clone(), out[1].clone()
        return first, g2.replay

    def _run(self, inp):
        first, second = self._stages(inp)
        r = first()
        second()
        return r

    def all_reduce_only(self):
        """The step's collective on its own (bench.py times it outside the step to report what the exchange costs)."""
        if self.world > 1:
            dist.all_reduce(self.bucket.flat, op=dist.ReduceOp.SUM, group=self.group)

    def step(self, x, vision_embs, context_str, lane_polygon_batch, lane_polygon_len, y, norm_stat, input_ids, attention_mask, *,
             skip_allreduce=False):
        """One optimisation step on this rank's shard of the batch; returns (loss, decoded) like the reference forward.
        `skip_allreduce` (measurement only): leaves the collective out, so step time minus this = the exposed cost of the exchange."""
        inp = self._device_inputs(x, vision_embs, lane_polygon_batch, lane_polygon_len, y, norm_stat, input_ids, attention_mask)
        first, second = self._stages(inp)
        loss, decoded = first()
        flat = self.bucket.flat
        works = []
        reduce = self.world > 1 and not skip_allreduce
        # a non-finite loss on this rank turns one gradient element NaN before that element's all-reduce: the reduced norm is then
        # NaN on every rank, and every rank skips
        mark = reduce and self.skip_nonfinite
        if reduce and self.overlap and self.n_late < flat.numel():
            # gradients behind n_late are final: their exchange runs on NCCL's stream under the decoder-stack backward
            if mark:
                ops.mark_nonfinite_(loss, flat[self.n_late:])
            works.append(dist.all_reduce(flat[self.n_late:], op=dist.ReduceOp.SUM, group=self.group, async_op=True))
            second()
            if self.n_late:
                works.append(dist.all_reduce(flat[:self.n_late], op=dist.ReduceOp.SUM, group=self.group, async_op=True))
        else:
            second()
            if mark:
                ops.mark_nonfinite_(loss, flat)
            if reduce:
                works.append(dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=self.group, async_op=True))
        for w in works:
            w.wait()                     # the current stream waits for the collective (no host block with NCCL)
        self.steps += 1
        if self._clip_rec is None:
            ops.adamw_(self.flat_p, flat, self.exp_avg, self.exp_avg_sq, lr=self.lr, betas=self.betas, eps=self.eps,
                       weight_decay=self.wd, step=self.steps, grad_scale=1.0 / self.world)
        else:
            ops.clip_prologue(flat, self._clip_rec, self._clip_ws, grad_scale=1.0 / self.world, max_norm=self.max_grad_norm, loss=loss,
                              skip_nonfinite=self.skip_nonfinite)
            ops.adamw_clipped_(self.flat_p, flat, self.exp_avg, self.exp_avg_sq, record=self._clip_rec, step=self.step_counter,
                               skipped=self.skipped_steps, lr=self.lr, betas=self.betas, eps=self.eps, weight_decay=self.wd,
                               grad_scale=1.0 / self.world)
        self.model._engine = None        # parameters changed behind torch's version counters: drop the inference packing
        return loss.detach(), decoded
