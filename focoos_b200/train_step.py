"""Optimiser / data-parallel side of the fine-tune step (SURVEY §8 a21), mirroring the reference:

  get_optimizer_params / build_optimizer   focoos/trainer/solver/build.py:40-138   (one param group per tensor, backbone lr x0.1, norm wd 0)
  TrainerLoop.run_step / clip_grads        focoos/trainer/trainer.py:723-794       (GradScaler(init 2^10), clip 0.1 twice, AdamW)
  create_ddp_model                         focoos/utils/distributed/dist.py:138-157 (DistributedDataParallel -> bucketed gradient all-reduce)

B200 design: every trainable tensor lives in ONE flat fp32 buffer (parameters, gradients, both Adam moments: 4 x 174 MB
for fai-detr-l), so the whole optimiser step is three launches (ops.grad_stats -> ops.optim_finalize -> ops.adamw_step)
with the loss scale, the clip coefficient and the skip-on-inf decision kept in a device-side control block (no host
sync), and the data-parallel exchange is an NCCL all-reduce of contiguous slices of the flat gradient buffer, issued
bucket by bucket (reverse parameter order, as the backward pass produces them) from autograd's post-accumulate hooks.
"""
from __future__ import annotations

from typing import Dict, Iterable, List, Optional, Sequence

import torch
import torch.distributed as dist
import torch.nn as nn

from . import ops

CTRL_SCALE, CTRL_GROWTH_TRACKER, CTRL_FOUND_INF, CTRL_GRAD_NORM, CTRL_GMUL, CTRL_STEP, CTRL_BC1, CTRL_BC2_SQRT, CTRL_CLIP_COEF = range(9)
CTRL_WORDS = 16

_NORM_TYPES = (nn.BatchNorm1d, nn.BatchNorm2d, nn.BatchNorm3d, nn.SyncBatchNorm, nn.GroupNorm, nn.InstanceNorm1d, nn.InstanceNorm2d, nn.InstanceNorm3d,
               nn.LayerNorm, nn.LocalResponseNorm)


def freeze_backbone_norm(model: nn.Module) -> None:
    """With backbone_config.freeze_norm the reference swaps every backbone BatchNorm2d for FrozenBatchNorm2d
    (nn/backbone/resnet.py:226-250): weight/bias become buffers - in the state_dict, not in model.parameters() - and the layer
    normalises with its RUNNING statistics in training too.  Here: requires_grad=False, which the training graph
    (fai_detr_train.DetrTrainGraph.bn) reads as "frozen": running statistics, no buffer update, no weight / bias gradient.
    (The registry's fai-detr configs set freeze_norm=false: all 501 tensors train.)"""
    for name, mod in model.named_modules():
        if "backbone" in name and isinstance(mod, nn.BatchNorm2d):
            mod.frozen_stats = True
            for p in mod.parameters(recurse=False):
                p.requires_grad_(False)


def freeze_backbone_at(model: nn.Module, freeze_at: int, num_stages: int = 4) -> None:
    """ResnetConfig.freeze_at >= 0 (nn/backbone/resnet.py:221-224): the stem and the first `freeze_at` stages get no gradient (their BatchNorms stay
    ordinary train-mode layers unless freeze_norm is also set)."""
    if freeze_at < 0:
        return
    bb = model.pixel_decoder.backbone
    mods = [bb.conv1] + [bb.res_layers[i] for i in range(min(freeze_at, num_stages))]
    for m in mods:
        for p in m.parameters():
            p.requires_grad_(False)


def get_optimizer_params(model: nn.Module, base_lr: float, weight_decay: float, weight_decay_norm: float = 0.0, weight_decay_embed: float = 0.0,
                         backbone_multiplier: float = 1.0, decoder_multiplier: float = 1.0, head_multiplier: float = 1.0) -> List[Dict]:
    """build.py:40-101: one group per trainable tensor; adds "name" for checkpoints/tests."""
    groups, memo = [], set()
    for module_name, module in model.named_modules():
        for pname, value in module.named_parameters(recurse=False):
            if not value.requires_grad or id(value) in memo:
                continue
            memo.add(id(value))
            lr, wd = base_lr, weight_decay
            if "backbone" in module_name:
                lr *= backbone_multiplier
                if backbone_multiplier == 0:
                    wd = 0.0
            if "pixel_decoder" in module_name:
                lr *= decoder_multiplier
                if backbone_multiplier == 0:  # sic (build.py:83)
                    wd = 0.0
            if "head" in module_name and "classifier" not in module_name:
                lr *= head_multiplier
                if head_multiplier == 0:
                    wd = 0.0
            if isinstance(module, _NORM_TYPES):
                wd = weight_decay_norm
            if isinstance(module, nn.Embedding) or "pos_embed" in pname:
                wd = weight_decay_embed
            if "relative_position_bias_table" in pname:
                wd = 0.0
            groups.append({"params": [value], "lr": lr, "weight_decay": wd, "name": f"{module_name}.{pname}" if module_name else pname})
    return groups


class FlatAdamW:
    """AdamW + full-model gradient clipping + GradScaler over one flat buffer.  `param_groups` as returned by get_optimizer_params."""

    def __init__(self, param_groups: Sequence[Dict], betas=(0.9, 0.999), eps: float = 1e-8, clip_gradients: float = 0.1, clip_passes: int = 2, amp: bool = True,
                 init_scale: float = 2.0 ** 10, growth_factor: float = 2.0, backoff_factor: float = 0.5, growth_interval: int = 2000, world_size: int = 1,
                 chunk_elems: int = 1 << 16):
        params = [g["params"][0] for g in param_groups]
        assert params and all(len(g["params"]) == 1 for g in param_groups), "one tensor per group (build.py:101)"
        dev = params[0].device
        if dev.type != "cuda" and ops._backend is None:
            raise RuntimeError("focoos_b200: the optimiser step runs on a CUDA device only (no CPU fallback)")
        assert all(p.dtype == torch.float32 and p.device == dev for p in params), "fp32 master parameters on one device"
        self.param_groups, self.names = list(param_groups), [g.get("name", str(i)) for i, g in enumerate(param_groups)]
        self.betas, self.eps, self.clip, self.clip_passes, self.amp = betas, eps, float(clip_gradients), int(clip_passes), bool(amp)
        self.growth, self.backoff, self.growth_interval, self.world_size = growth_factor, backoff_factor, growth_interval, world_size
        offs, total = [], 0
        for p in params:
            offs.append(total)
            total += (p.numel() + 3) // 4 * 4
        self.offsets, self.total = offs, total
        self.flat_params = torch.zeros(total, dtype=torch.float32, device=dev)
        self.flat_grads = torch.zeros(total, dtype=torch.float32, device=dev)
        self.exp_avg = torch.zeros(total, dtype=torch.float32, device=dev)
        self.exp_avg_sq = torch.zeros(total, dtype=torch.float32, device=dev)
        with torch.no_grad():
            for p, o in zip(params, offs):
                view = self.flat_params[o:o + p.numel()].view_as(p)
                view.copy_(p)
                p.data = view
                p.grad = self.flat_grads[o:o + p.numel()].view_as(p)
        self.params = params
        cs, cl, cg = [], [], []
        for i, (p, o) in enumerate(zip(params, offs)):
            n = (p.numel() + 3) // 4 * 4
            for s in range(0, n, chunk_elems):
                cs.append(o + s)
                cl.append(min(chunk_elems, n - s))
                cg.append(i)
        self.chunk_start = torch.tensor(cs, dtype=torch.int64, device=dev)
        self.chunk_len = torch.tensor(cl, dtype=torch.int32, device=dev)
        self.chunk_seg = torch.tensor(cg, dtype=torch.int32, device=dev)
        self.seg_lr = torch.tensor([g["lr"] for g in param_groups], dtype=torch.float32, device=dev)
        self.seg_wd = torch.tensor([g["weight_decay"] for g in param_groups], dtype=torch.float32, device=dev)
        self.ctrl = torch.zeros(CTRL_WORDS, dtype=torch.float32, device=dev)
        self.ctrl[CTRL_SCALE] = init_scale if amp else 1.0
        self.ws = ops._be().optim_workspace(dev)
        self._fired: Optional[List[bool]] = None  # set by track_unused_parameters()
        self._hooks = []

    # -- GradScaler-shaped helpers (device scalars: no host sync on the step path)
    @property
    def loss_scale(self) -> torch.Tensor:
        return self.ctrl[CTRL_SCALE]

    def scale_loss(self, loss: torch.Tensor) -> torch.Tensor:
        return loss * self.ctrl[CTRL_SCALE].to(loss.dtype) if self.amp else loss

    def track_unused_parameters(self) -> None:
        """torch.optim skips a tensor whose .grad is None (no update, no weight decay) and clip_grad_norm_ ignores it - e.g. the dead
        `mask_features` conv of fai-detr (SURVEY a6).  Here gradients are views of a zeroed flat buffer and never None, so backward marks
        the tensors it reached through post-accumulate hooks and step() skips the others."""
        if self._fired is None:
            self._fired = [False] * len(self.params)
            for i, p in enumerate(self.params):
                self._hooks.append(p.register_post_accumulate_grad_hook(lambda _p, i=i: self._fired.__setitem__(i, True)))

    def zero_grad(self) -> None:
        self.flat_grads.zero_()
        if self._fired is not None:
            self._fired = [False] * len(self.params)
        for p, o in zip(self.params, self.offsets):  # autograd may have replaced .grad (set_to_none callers)
            if p.grad is None or p.grad.data_ptr() != self.flat_grads.data_ptr() + 4 * o:
                p.grad = self.flat_grads[o:o + p.numel()].view_as(p)

    def step(self, lr_factor: float = 1.0) -> None:
        """unscale + inf check + clip (x clip_passes) + AdamW + loss-scale update; gradients are expected to hold the SUM over ranks."""
        be = ops._be()
        be.grad_stats(self.flat_grads, self.ws)
        be.optim_finalize(self.ws, self.ctrl, self.clip, self.clip_passes, 1.0 / self.world_size, self.amp, self.growth, self.backoff, self.growth_interval,
                          self.betas[0], self.betas[1])
        active = None if self._fired is None else torch.tensor(self._fired, dtype=torch.int32).to(self.flat_params.device, non_blocking=True)
        be.adamw_step(self.flat_params, self.flat_grads, self.exp_avg, self.exp_avg_sq, self.chunk_start, self.chunk_len, self.chunk_seg, self.seg_lr, self.seg_wd,
                      active, float(lr_factor), self.betas[0], self.betas[1], self.eps, self.ctrl)

    def stats(self) -> Dict[str, float]:
        """host read-back (syncs): for logging / tests only."""
        c = self.ctrl.cpu()
        ci = c.view(torch.int32)
        return {"scale": float(c[CTRL_SCALE]), "growth_tracker": int(ci[CTRL_GROWTH_TRACKER]), "found_inf": int(ci[CTRL_FOUND_INF]), "grad_norm": float(c[CTRL_GRAD_NORM]),
                "step": int(ci[CTRL_STEP]), "clip_coef": float(c[CTRL_CLIP_COEF])}

    def state_dict(self) -> Dict:
        return {"names": list(self.names), "offsets": list(self.offsets), "exp_avg": self.exp_avg.clone(), "exp_avg_sq": self.exp_avg_sq.clone(), "ctrl": self.ctrl.clone()}

    def load_state_dict(self, sd: Dict) -> None:
        assert sd["names"] == self.names and sd["offsets"] == self.offsets, "optimizer state does not match this model"
        self.exp_avg.copy_(sd["exp_avg"])
        self.exp_avg_sq.copy_(sd["exp_avg_sq"])
        self.ctrl.copy_(sd["ctrl"])


class GradBucketReducer:
    """Data-parallel gradient exchange (what DistributedDataParallel does for the reference, dist.py:152): SUM all-reduce of
    contiguous slices of the flat gradient buffer.  Buckets follow reverse parameter order (the order backward fills them) and
    never split a tensor; the 1/world averaging is folded into FlatAdamW's gradient multiplier, not a separate pass."""

    def __init__(self, opt: FlatAdamW, bucket_bytes: int = 25 << 20, group=None, model: Optional[nn.Module] = None, broadcast: bool = True):
        self.opt, self.group = opt, group
        self.enabled = dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1
        if self.enabled and broadcast:
            # DistributedDataParallel's constructor broadcasts rank 0's parameters and buffers (dist.py:152): replicas start identical even if the
            # caller seeded them differently, and BatchNorm running statistics do not diverge from step 0
            dist.broadcast(opt.flat_params, src=0, group=group)
            if model is not None:
                for b in model.buffers():
                    if b.is_floating_point() or b.dtype in (torch.int64, torch.int32):
                        dist.broadcast(b, src=0, group=group)
        ends = opt.offsets[1:] + [opt.total]
        self.buckets: List[List[int]] = []  # [start, end, first_seg, last_seg]
        cur_end, cur_start, last = opt.total, opt.total, len(opt.offsets) - 1
        for i in range(len(opt.offsets) - 1, -1, -1):
            cur_start = opt.offsets[i]
            if (cur_end - cur_start) * 4 >= bucket_bytes or i == 0:
                self.buckets.append([cur_start, cur_end, i, last])
                cur_end, last = cur_start, i - 1
        self.seg_bucket = [0] * len(opt.offsets)
        for b, (_, _, lo, hi) in enumerate(self.buckets):
            for s in range(lo, hi + 1):
                self.seg_bucket[s] = b
        self._pending = [0] * len(self.buckets)
        self._handles = []
        self._hooks = []
        self._static_unused = None  # learnt at the first finish(): tensors backward never reaches (e.g. fai-detr's dead mask_features conv, SURVEY a6)
        self.reset()

    def reset(self):
        self._pending = [hi - lo + 1 for _, _, lo, hi in self.buckets]
        self._launched = [False] * len(self.buckets)
        self._seen = [False] * len(self.opt.offsets)
        self._next = 0  # buckets go out STRICTLY in index order on every rank: collectives must be issued in the same order everywhere
        self._handles = []
        for seg in (self._static_unused or ()):  # structurally unused tensors count as ready from the start, or they would hold every later bucket back
            self._seen[seg] = True
            self._pending[self.seg_bucket[seg]] -= 1

    def _launch(self, b: int):
        if self._launched[b]:
            return
        self._launched[b] = True
        if self.enabled:
            s, e = self.buckets[b][:2]
            self._handles.append(dist.all_reduce(self.opt.flat_grads[s:e], op=dist.ReduceOp.SUM, group=self.group, async_op=True))

    def mark_ready(self, seg: int):
        b = self.seg_bucket[seg]
        if self._seen[seg]:
            if self._launched[b]:  # (also: a tensor learnt as unused that now received a gradient after its bucket left)  # a second backward before finish(): its gradient would be added onto an already-summed slice
                raise RuntimeError("GradBucketReducer: gradient accumulated into a bucket that was already exchanged - call finish() after every backward")
            return
        self._seen[seg] = True
        self._pending[b] -= 1
        # a bucket may only go out once every earlier bucket has: a parameter that is unused on ONE rank must not reorder that rank's collectives
        while self._next < len(self.buckets) and self._pending[self._next] == 0:
            self._launch(self._next)
            self._next += 1

    def attach_hooks(self):
        """overlap with backward: each parameter's post-accumulate hook marks its slice ready; full buckets go out immediately."""
        for i, p in enumerate(self.opt.params):
            self._hooks.append(p.register_post_accumulate_grad_hook(lambda _p, i=i: self.mark_ready(i)))

    def detach_hooks(self):
        for h in self._hooks:
            h.remove()
        self._hooks = []
        for h in self.opt._hooks:
            h.remove()
        self.opt._hooks = []
        self.opt._fired = None

    def finish(self):
        """launch whatever backward did not touch (unused parameters keep zero gradients) and wait for every bucket."""
        if self._static_unused is None and self._hooks:
            self._static_unused = {i for i, seen in enumerate(self._seen) if not seen}
        for b in range(len(self.buckets)):
            self._launch(b)
        for h in self._handles:
            h.wait()
        self.reset()


class TrainStep:
    """TrainerLoop.run_step (trainer.py:723-773) for one already-preprocessed batch."""

    def __init__(self, model: nn.Module, opt: FlatAdamW, reducer: Optional[GradBucketReducer] = None):
        self.model, self.opt, self.reducer = model, opt, reducer

    def __call__(self, images, targets, lr_factor: float = 1.0) -> Dict[str, torch.Tensor]:
        self.opt.zero_grad()
        crit = getattr(self.model, "criterion", None)
        if callable(crit) and targets and hasattr(targets[0], "labels"):
            # the rank-averaged box count needs a host read-back when several ranks train: do it before anything of this step is enqueued
            from .criterion import global_num_boxes
            c = crit()
            if hasattr(c, "num_boxes_hint"):
                c.num_boxes_hint = global_num_boxes(targets, images.device)
        loss_dict = self.model(images, targets).loss
        if isinstance(loss_dict, torch.Tensor):
            losses, loss_dict = loss_dict, {"total_loss": loss_dict}
        else:
            losses = sum(loss_dict.values())
        self.opt.scale_loss(losses).backward()
        if self.reducer is not None:
            self.reducer.finish()
        self.opt.step(lr_factor)
        return loss_dict
