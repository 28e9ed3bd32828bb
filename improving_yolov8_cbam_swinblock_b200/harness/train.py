"""Synthetic-batch data-parallel training step for the custom YOLOv8-CBAM-Swin graph (SURVEY section 8(d)/(e)).

Mirrors the reference's hot loop (engine/trainer.py:367-399,614-622): H2D copy + ``img.float()/255`` (detect/train.py:
90-115), autocast forward, v8 detection loss, ``loss.sum() * world_size`` (trainer.py:386-388; DDP averages grads),
backward, ONE all-reduce of the flat gradient buffer (NCCL over NVLink; gradients only -- the path's one exchange step),
``clip_grad_norm_(10)``,
SGD(momentum 0.937, nesterov) with the trainer's three parameter groups (trainer.py:788-830) and the EMA update
(torch_utils.py:657-672).  One process per GPU; nothing but gradients crosses GPUs.
"""
from __future__ import annotations

import math

import torch
import torch.nn as nn

from . import graph, loss as hloss


def param_groups(model: nn.Module, weight_decay: float = 5e-4):
    """trainer.py:818-827: biases -> g2 (no decay), norm weights -> g1 (no decay), other weights -> g0 (decay)."""
    bn = tuple(v for k, v in nn.__dict__.items() if "Norm" in k)
    g0, g1, g2 = [], [], []
    for mod_name, mod in model.named_modules():
        for pn, p in mod.named_parameters(recurse=False):
            if not p.requires_grad:
                continue
            full = f"{mod_name}.{pn}" if mod_name else pn
            if "bias" in full:
                g2.append(p)
            elif isinstance(mod, bn):
                g1.append(p)
            else:
                g0.append(p)
    return [{"params": g0, "weight_decay": weight_decay}, {"params": g1, "weight_decay": 0.0},
            {"params": g2, "weight_decay": 0.0}]


class EMA:
    """ModelEMA (torch_utils.py:620-672) with foreach updates instead of the per-tensor Python loop."""

    def __init__(self, model, decay=0.9999, tau=2000):
        self.shadow = [p.detach().clone().float() for p in model.state_dict().values() if p.dtype.is_floating_point]
        self.decay, self.tau, self.updates = decay, tau, 0

    @torch.no_grad()
    def update(self, model):
        self.updates += 1
        d = self.decay * (1 - math.exp(-self.updates / self.tau))
        cur = [p.detach() for p in model.state_dict().values() if p.dtype.is_floating_point]
        # v = d*v + (1-d)*p in ONE multi-tensor pass (the two-op form read and wrote every shadow tensor twice per step)
        torch._foreach_lerp_(self.shadow, cur, 1 - d)


class Trainer:
    """One process per GPU.  world_size > 1: every rank holds a replica; the local backward accumulates into ONE flat
    fp32 gradient buffer (each ``p.grad`` is a view of it, laid out like the parameter) and the path's single exchange
    step is one NCCL/gloo all-reduce(SUM) of that buffer -- gradients only.  Summing per-rank gradients of the local
    ``loss.sum()`` equals the reference's ``loss * world_size`` followed by DDP's mean (trainer.py:278,386-388).  Doing
    the all-reduce explicitly (instead of through DDP's autograd hooks) keeps forward+backward CUDA-graph capturable."""

    def __init__(self, blocks: dict, scale="n", nc=80, device="cuda", amp_dtype=torch.bfloat16, world_size=1,
                 local_rank=0, channels_last=True, lr=0.01, momentum=0.937, seed=0, ema=True):
        self.device = torch.device(device)
        self.world_size = world_size
        self.amp_dtype = amp_dtype
        self.channels_last = channels_last and self.device.type == "cuda"
        torch.manual_seed(seed)  # identical init on every rank
        model = graph.DetectionGraph(blocks, scale, nc)
        for n_, p in model.named_parameters():
            if ".dfl" in n_:
                p.requires_grad_(False)  # trainer.py:243-262 always freezes the DFL conv
        model = model.to(self.device).train()
        if self.channels_last:
            model = model.to(memory_format=torch.channels_last)
        self.raw = self.model = model
        self.criterion = hloss.DetectionLoss(nc, model.stride)
        # SURVEY 8(f)-4: fused classification term (the kernel moves 16-byte vectors of class logits: nc a multiple of 8)
        if blocks.get("cls_loss") is not None and self.device.type == "cuda" and nc % 8 == 0:
            self.criterion.cls_loss = blocks["cls_loss"]
            model.model[-1].split_outputs = True
            if blocks.get("det_loss") is not None:   # assigner + box / DFL terms as kernels too (SURVEY 8(f)-4)
                self.criterion.det_kernels = blocks["det_loss"]
        fused = self.device.type == "cuda"
        self.opt = torch.optim.SGD(param_groups(model), lr=lr, momentum=momentum, nesterov=True, fused=fused)
        self.ema = EMA(model) if ema else None
        self.max_boxes = None
        self._input_prep = blocks.get("input_prep")   # SURVEY 8(f)-2: the uint8 -> float NHWC input seam (None = stock ops)
        self._params = [p for p in model.parameters() if p.requires_grad]
        self._flat = None
        if world_size > 1:
            self._flat = torch.zeros(sum(p.numel() for p in self._params), dtype=torch.float32, device=self.device)
            off = 0
            self._views = []
            for p in self._params:
                p.grad = self._flat[off:off + p.numel()].as_strided(p.shape, p.stride())  # same memory order as the parameter
                self._views.append(p.grad)
                off += p.numel()
            # Autograd ACCUMULATES into an existing .grad (one add kernel per parameter and step, ~160 launches, plus the zero fill).
            # Instead the backward produces fresh gradients and ONE multi-tensor copy moves them into the flat buffer.
        # SURVEY 8(f)-3: under autocast every stock convolution casts its f32 weight to the compute dtype in the forward and its
        # 16-bit weight gradient back to f32 in the backward -- two tiny kernels per layer and step (~100 launches).  Instead: one
        # 16-bit leaf per layer, all refreshed by ONE multi-tensor copy at the start of the step and all gradients copied back by
        # ONE multi-tensor copy after the backward.  Same values as autocast's casts (bit-identical step).
        self._w16 = []   # (Conv module, f32 parameter, 16-bit leaf, f32 gradient buffer)
        if self.device.type == "cuda" and amp_dtype in (torch.bfloat16, torch.float16):
            for m_ in model.modules():
                if isinstance(m_, graph.Conv) and m_.conv_fn is None and m_.conv.bias is None and m_.conv.weight.requires_grad \
                        and m_.conv.padding_mode == "zeros":
                    p = m_.conv.weight
                    leaf = p.detach().to(amp_dtype).requires_grad_(True)   # keeps the parameter's (channels_last) strides
                    g32 = p.grad if p.grad is not None else torch.zeros_like(p)
                    m_.w16 = leaf
                    self._w16.append((m_, p, leaf, g32))
        self._graph, self._graph_b, self._graph_error, self._static, self._static_items = None, None, None, None, None
        self._graph_mode = None
        self._prefetched, self._copy_stream = None, None

    def to_device(self, host_batch):
        return {k: v.to(self.device, non_blocking=True) for k, v in host_batch.items()}

    # ---- the step, in two halves so that the gradient exchange sits between them ---------------------------------
    def _forward_loss(self, dev_batch):
        use_amp = self.amp_dtype is not None and self.amp_dtype != torch.float32
        raw = dev_batch["img"]
        if self._input_prep is not None and raw.is_cuda and raw.dtype == torch.uint8 and self.channels_last and raw.is_contiguous() \
                and raw.shape[1] <= 4 and (raw.shape[2] * raw.shape[3]) % 4 == 0:
            # one kernel: uint8 NCHW -> f32 division -> compute dtype, NHWC (what autocast hands the first conv anyway)
            img = self._input_prep(raw, self.amp_dtype if use_amp else torch.float32, 255.0)
        else:
            img = raw.float() / 255  # detect/train.py:100
            if self.channels_last:
                img = img.contiguous(memory_format=torch.channels_last)
        with torch.autocast(self.device.type, dtype=self.amp_dtype or torch.bfloat16, enabled=use_amp):
            feats = self.model(img)
            return self.criterion(feats, dev_batch, max_boxes=self.max_boxes)   # the loss casts to f32 after gathering

    def _fwd_bwd(self, dev_batch):
        if self._flat is not None:
            for p in self._params:
                p.grad = None               # fresh gradients from the backward, gathered into the flat buffer below
        if self._w16:
            with torch.no_grad():
                torch._foreach_copy_([t[2] for t in self._w16], [t[1] for t in self._w16])   # f32 weights -> 16-bit leaves
            for t in self._w16:
                t[2].grad = None
        loss, items = self._forward_loss(dev_batch)
        loss.sum().backward()
        if self._w16:
            live = [t for t in self._w16 if t[2].grad is not None]
            with torch.no_grad():
                torch._foreach_copy_([t[3] for t in live], [t[2].grad for t in live])       # 16-bit gradients -> f32 .grad
            for _, p, _, g32 in live:
                p.grad = g32
        if self._flat is not None:
            src, dst, missing = [], [], []
            for p, v in zip(self._params, self._views):
                if p.grad is None:
                    missing.append(v)       # a parameter the loss did not reach: its slot must read zero
                elif p.grad is not v:
                    src.append(p.grad)
                    dst.append(v)
            with torch.no_grad():
                if dst:
                    torch._foreach_copy_(dst, src)
                if missing:
                    torch._foreach_zero_(missing)
            for p, v in zip(self._params, self._views):
                p.grad = v
        return items

    def _exchange(self):
        if self._flat is not None:
            import torch.distributed as dist

            dist.all_reduce(self._flat)     # SUM over ranks; gradients only -- the one exchange step of the path

    def _update(self):
        torch.nn.utils.clip_grad_norm_(self._params, max_norm=10.0, foreach=True)
        self.opt.step()
        if self._flat is None:
            self.opt.zero_grad(set_to_none=True)

    # ---- CUDA-graph replay of the step (SURVEY 8(f)-3: host-side step overhead) ------------------------------
    def enable_graph(self, dev_batch, warmup: int = 3) -> bool:
        """Capture the step into CUDA graphs (shapes are static for the synthetic batches): one graph at world_size 1
        (forward + loss + backward + clip + SGD); at world_size > 1 graph A = forward + loss + backward, the all-reduce
        launched eagerly between, graph B = clip + SGD.  Falls back to eager launches (returns False) if capture fails."""
        if self.device.type != "cuda" or self._graph is not None:
            return self._graph is not None
        try:
            self._static = {k: v.clone() for k, v in dev_batch.items()}
            cur = torch.cuda.current_stream(self.device)
            side = torch.cuda.Stream(self.device)
            side.wait_stream(cur)
            with torch.cuda.stream(side):
                for _ in range(max(warmup, 3)):
                    self._fwd_bwd(self._static)
                    self._exchange()
                    self._update()
            cur.wait_stream(side)
            torch.cuda.synchronize(self.device)
            ga = torch.cuda.CUDAGraph()
            if self._flat is None:
                with torch.cuda.graph(ga):
                    self._static_items = self._fwd_bwd(self._static)
                    self._update()
            else:
                # thread_local: the NCCL watchdog thread may make CUDA calls while this thread captures.  The all-reduce stays
                # outside the graphs: capturing it too measured no faster at N=2 (20.7-21.3 vs 20.4 ms/step)
                gb = torch.cuda.CUDAGraph()
                with torch.cuda.graph(ga, capture_error_mode="thread_local"):
                    self._static_items = self._fwd_bwd(self._static)
                self._exchange()
                with torch.cuda.graph(gb, pool=ga.pool(), capture_error_mode="thread_local"):
                    self._update()
                self._graph_b = gb
                self._graph_mode = "two graphs around an eager all-reduce"
            self._graph = ga
        except Exception as e:  # noqa: BLE001  capture is an optimisation; eager launches remain correct
            self._graph, self._graph_b, self._graph_error = None, None, f"{type(e).__name__}: {e}"
            torch.cuda.synchronize(self.device)
        return self._graph is not None

    def release_graphs(self):
        """Destroy the captured graphs and fall back to eager launches.  The graphs hold no NCCL kernels (the all-reduce runs
        eagerly between them), so the communicator does not depend on them."""
        self._graph, self._graph_b, self._static_items = None, None, None
        if self.device.type == "cuda":
            import gc

            gc.collect()
            torch.cuda.synchronize(self.device)

    def step(self, dev_batch):
        """One optimizer step on a device-resident batch; returns the detached loss items [box, cls, dfl]."""
        if self._graph is not None:
            for k, v in dev_batch.items():
                self._static[k].copy_(v, non_blocking=True)
            self._graph.replay()
            if self._graph_b is not None:
                self._exchange()
                self._graph_b.replay()
            items = self._static_items.clone()
        else:
            items = self._fwd_bwd(dev_batch)
            self._exchange()
            self._update()
        if self.ema is not None:
            self.ema.update(self.raw)
        return items

    def step_from_host(self, host_batch, next_host_batch=None):
        """The user-facing call: pinned host batch in, host loss items out (H2D + D2H inside).  ``next_host_batch``
        (optional) is what a data loader would hand over next: its H2D copy is issued on a copy stream before this call
        blocks on the loss, so it overlaps this step's compute (every step still copies its own inputs exactly once)."""
        if self.device.type != "cuda":
            return self.step(self.to_device(host_batch)).cpu()
        cur = torch.cuda.current_stream(self.device)
        if self._prefetched is not None and self._prefetched[0] is host_batch:
            dev_batch, ev = self._prefetched[1], self._prefetched[2]
            cur.wait_event(ev)
        else:
            dev_batch = self.to_device(host_batch)
        self._prefetched = None
        items = self.step(dev_batch)
        if next_host_batch is not None:
            if self._copy_stream is None:
                self._copy_stream = torch.cuda.Stream(self.device)
            with torch.cuda.stream(self._copy_stream):
                nxt = self.to_device(next_host_batch)
                ev = torch.cuda.Event()
                ev.record(self._copy_stream)
            for v in dev_batch.values():
                v.record_stream(cur)
            self._prefetched = (next_host_batch, nxt, ev)
        return items.cpu()
