"""DETR training criterion on the B200 (SURVEY §8 a20), mirroring the reference classes:

  BoxHungarianMatcher   focoos/models/fai_detr/modelling.py:643-758  (cost on the GPU, assignment on the GPU instead of scipy on the CPU)
  SetCriterion          focoos/models/fai_detr/modelling.py:408-612  (losses "vfl" + "boxes", deep supervision over the aux outputs)
  DETRTargets           focoos/models/fai_detr/ports.py:16-19

All supervised layers (final + aux decoder layers + encoder proposals) go through ONE cost launch, ONE assignment
launch and ONE loss launch; the loss kernel also produces d(loss)/d(logits) and d(loss)/d(boxes), which a
torch.autograd.Function hands back to whatever produced the predictions.  No CPU path: tensors must be CUDA tensors.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict, List, Sequence, Tuple

import torch

from . import ops


@dataclass
class DETRTargets:
    labels: torch.Tensor  # [n] int64 class ids
    boxes: torch.Tensor   # [n,4] cxcywh normalised to [0,1]


def _pack_targets(targets: Sequence[DETRTargets], device):
    counts = [int(t.labels.shape[0]) for t in targets]
    off = torch.tensor([0] + list(torch.tensor(counts).cumsum(0).tolist()) if counts else [0], dtype=torch.int32)
    if sum(counts) == 0:
        return None, None, off.to(device), counts
    tl = torch.cat([t.labels.reshape(-1) for t in targets]).to(device=device, dtype=torch.int32).contiguous()
    tb = torch.cat([t.boxes.reshape(-1, 4) for t in targets]).to(device=device, dtype=torch.float32).contiguous()
    return tl, tb, off.to(device), counts


def match(logits, boxes, targets: Sequence[DETRTargets], cost_class=2.0, cost_bbox=5.0, cost_giou=2.0, alpha=0.25, gamma=2.0, return_cost=False):
    """logits [L,B,Q,C] f32 raw, boxes [L,B,Q,4] cxcywh -> match_q [L,T] int32 (query assigned to each concatenated target)."""
    L, B, Q, C = logits.shape
    tl, tb, toff, counts = _pack_targets(targets, logits.device)
    if tl is None:
        return torch.empty((L, 0), dtype=torch.int32, device=logits.device)
    if max(counts) > Q:
        raise RuntimeError(f"focoos_b200: an image has {max(counts)} targets but the model has {Q} queries")
    T = tl.shape[0]
    cost = torch.empty((L, T, Q), dtype=torch.float32, device=logits.device)
    be = ops._be()
    be.detr_match_cost(logits.contiguous(), boxes.contiguous(), tl, tb, toff, (cost_class, cost_bbox, cost_giou), alpha, gamma, cost)
    match_q = torch.empty((L, T), dtype=torch.int32, device=logits.device)
    be.hungarian(cost, toff, B, max(counts), match_q)
    return (match_q, cost) if return_cost else match_q


class _DetrLossFn(torch.autograd.Function):
    """losses [L,3] = weighted (vfl, bbox, giou) per supervised layer; gradients come out of the same kernel launch."""

    @staticmethod
    def forward(ctx, logits, boxes, tl, tb, toff, match_q, num_boxes, wts, alpha, gamma):
        L, B, Q, C = logits.shape
        dev = logits.device
        losses = torch.empty((L, 3), dtype=torch.float32, device=dev)
        g_logits = torch.empty((L, B, Q, C), dtype=torch.float32, device=dev)
        g_l1 = torch.empty((L, B, Q, 4), dtype=torch.float32, device=dev)
        g_giou = torch.empty((L, B, Q, 4), dtype=torch.float32, device=dev)
        ops._be().detr_loss(logits.contiguous(), boxes.contiguous(), tl, tb, toff, match_q, num_boxes, wts, alpha, gamma, losses, g_logits, g_l1, g_giou)
        ctx.save_for_backward(g_logits, g_l1, g_giou)
        return losses

    @staticmethod
    def backward(ctx, g):
        g_logits, g_l1, g_giou = ctx.saved_tensors
        g = g.to(torch.float32)
        gl = g_logits * g[:, 0].reshape(-1, 1, 1, 1)
        gb = g_l1 * g[:, 1].reshape(-1, 1, 1, 1) + g_giou * g[:, 2].reshape(-1, 1, 1, 1)
        return gl, gb, None, None, None, None, None, None, None, None


class BoxHungarianMatcher(torch.nn.Module):
    """modelling.py:643-758; only the focal-cost variant the fai-detr configs use (use_focal_loss=True)."""

    def __init__(self, cost_class: float = 1, cost_bbox: float = 1, cost_giou: float = 1, use_focal_loss=True, alpha=0.25, gamma=2.0):
        super().__init__()
        assert cost_class != 0 or cost_bbox != 0 or cost_giou != 0, "all costs cant be 0"
        if not use_focal_loss:
            raise NotImplementedError("focoos_b200: only the focal matching cost (matcher_use_focal_loss=True, fai_detr/config.py:59) is built")
        self.cost_class, self.cost_bbox, self.cost_giou, self.alpha, self.gamma = float(cost_class), float(cost_bbox), float(cost_giou), float(alpha), float(gamma)

    def match_layers(self, logits, boxes, targets):
        return match(logits, boxes, targets, self.cost_class, self.cost_bbox, self.cost_giou, self.alpha, self.gamma)

    @torch.no_grad()
    def forward(self, outputs: Dict[str, torch.Tensor], targets: List[DETRTargets]) -> List[Tuple[torch.Tensor, torch.Tensor]]:
        """Same return contract as the reference: per image (query indices ascending, matching target indices), int64 on the CPU."""
        mq = self.match_layers(outputs["pred_logits"][None], outputs["pred_boxes"][None], targets)[0].cpu().to(torch.int64)
        out, o = [], 0
        for t in targets:
            n = int(t.labels.shape[0])
            q = mq[o:o + n]
            order = torch.argsort(q)
            out.append((q[order], order))
            o += n
        return out


def global_num_boxes(targets, dev) -> float:
    """number of target boxes averaged over the data-parallel ranks, clamped at 1 (modelling.py:566-571).  One process: host arithmetic only.  Several ranks: a scalar
    all-reduce and a read-back - a host synchronisation, which is why TrainStep calls this BEFORE the forward pass is enqueued (SetCriterion.num_boxes_hint) instead
    of stalling the launch queue between the forward and the backward pass."""
    n = float(sum(int(t.labels.shape[0]) for t in targets))
    if torch.distributed.is_available() and torch.distributed.is_initialized() and torch.distributed.get_world_size() > 1:
        nb = torch.tensor([n], dtype=torch.float32, device=dev)
        torch.distributed.all_reduce(nb)
        n = float(nb.item()) / torch.distributed.get_world_size()
    return max(n, 1.0)


class SetCriterion(torch.nn.Module):
    """modelling.py:408-612 with losses ["vfl", "boxes"] (fai_detr/config.py:47) and deep supervision."""

    def __init__(self, num_classes: int, matcher: BoxHungarianMatcher, weight_dict: dict, losses=("vfl", "boxes"), eos_coef: float = 0.1,
                 num_points: int = 0, deep_supervision: bool = True, focal_alpha: float = 0.75, focal_gamma: float = 2.0, **_unused):
        super().__init__()
        if sorted(losses) != ["boxes", "vfl"]:
            raise NotImplementedError(f"focoos_b200: criterion losses {list(losses)} not built (only ['vfl', 'boxes'])")
        self.num_classes, self.matcher, self.weight_dict, self.losses = num_classes, matcher, dict(weight_dict), list(losses)
        self.deep_supervision, self.focal_alpha, self.focal_gamma, self.eos_coef = deep_supervision, float(focal_alpha), float(focal_gamma), eos_coef
        self.num_boxes_hint = None  # optional float: global_num_boxes(targets) computed by the caller ahead of the forward pass (consumed by the next forward)
        self.forced_match = None  # optional [L,T] int tensor: use these assignments instead of running the matcher (teacher forcing in parity tests)
        self.last_match = None    # the assignments used by the most recent forward, [L,T] int32 on the device

    def forward(self, outputs: dict, targets: List[DETRTargets]) -> Dict[str, torch.Tensor]:
        layers = [outputs] + (list(outputs.get("aux_outputs", [])) if self.deep_supervision else [])
        logits = torch.stack([o["pred_logits"] for o in layers]).to(torch.float32)
        boxes = torch.stack([o["pred_boxes"] for o in layers]).to(torch.float32)
        if not logits.is_cuda and ops._backend is None:
            raise RuntimeError("focoos_b200: the criterion runs on a CUDA device only (no CPU fallback)")
        dev = logits.device
        # number of target boxes averaged over the ranks (modelling.py:566-571)
        num_boxes = self.num_boxes_hint if self.num_boxes_hint is not None else global_num_boxes(targets, dev)
        self.num_boxes_hint = None
        tl, tb, toff, counts = _pack_targets(targets, dev)
        with torch.no_grad():
            if self.forced_match is not None:
                mq = self.forced_match.to(device=dev, dtype=torch.int32).contiguous()
                assert tuple(mq.shape) == (logits.shape[0], 0 if tl is None else tl.shape[0])
            else:
                mq = self.matcher.match_layers(logits.detach(), boxes.detach(), targets) if tl is not None else None
            self.last_match = mq
        w = (float(self.weight_dict.get("loss_vfl", 1.0)), float(self.weight_dict.get("loss_bbox", 1.0)), float(self.weight_dict.get("loss_giou", 1.0)))
        table = _DetrLossFn.apply(logits, boxes, tl, tb, toff, mq, num_boxes, w, self.focal_alpha, self.focal_gamma)
        if mq is not None and self.forced_match is None:
            # the device Hungarian writes -1 for an image whose cost matrix holds NaN / inf (scipy's linear_sum_assignment raises "matrix contains invalid numeric
            # entries" in the reference, matcher :744): poison the losses instead of silently training on dropped targets - the loss scaler's found_inf then
            # skips the step (amp), and without a scaler the NaN is visible in the very next log line.  Device-side select: no host synchronisation.
            table = torch.where((mq < 0).any(), torch.full_like(table, float("nan")), table)
        out = {}
        for l in range(table.shape[0]):
            sfx = "" if l == 0 else f"_{l - 1}"
            out["loss_vfl" + sfx], out["loss_bbox" + sfx], out["loss_giou" + sfx] = table[l, 0], table[l, 1], table[l, 2]
        return out
