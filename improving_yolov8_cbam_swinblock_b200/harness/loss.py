"""Detection loss used by the throughput harness: BCE + CIoU + DFL with task-aligned assignment.

Caller-side code (SURVEY section 2.1 marks ``utils/loss.py:152-255`` / ``utils/tal.py:14-327`` as "reused as-is by
the training harness"; the reference package cannot travel to the GPU box, so this is a dense restatement).
It computes the same function as ``v8DetectionLoss.__call__`` + ``TaskAlignedAssigner.forward`` but with
mask-multiplies instead of boolean indexing and no ``.item()``-style host syncs, so one training step can
be enqueued without the host waiting on the device.  tests/test_det_loss_oracle.py checks the assigner and the three loss
components on CPU against oracle/det_loss.py, a line-by-line restatement of the reference that shares no code with this one.
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F

from .graph import make_anchors


def _ciou(b1, b2, eps=1e-7):
    """CIoU of xyxy boxes, broadcast over leading dims (utils/metrics.py bbox_iou, xywh=False, CIoU=True)."""
    b1_x1, b1_y1, b1_x2, b1_y2 = b1.unbind(-1)
    b2_x1, b2_y1, b2_x2, b2_y2 = b2.unbind(-1)
    w1, h1 = b1_x2 - b1_x1, b1_y2 - b1_y1 + eps
    w2, h2 = b2_x2 - b2_x1, b2_y2 - b2_y1 + eps
    inter = (torch.minimum(b1_x2, b2_x2) - torch.maximum(b1_x1, b2_x1)).clamp(0) * (
        torch.minimum(b1_y2, b2_y2) - torch.maximum(b1_y1, b2_y1)).clamp(0)
    union = w1 * h1 + w2 * h2 - inter + eps
    iou = inter / union
    cw = torch.maximum(b1_x2, b2_x2) - torch.minimum(b1_x1, b2_x1)
    ch = torch.maximum(b1_y2, b2_y2) - torch.minimum(b1_y1, b2_y1)
    c2 = cw.pow(2) + ch.pow(2) + eps
    rho2 = ((b2_x1 + b2_x2 - b1_x1 - b1_x2).pow(2) + (b2_y1 + b2_y2 - b1_y1 - b1_y2).pow(2)) / 4
    v = (4 / math.pi ** 2) * ((w2 / h2).atan() - (w1 / h1).atan()).pow(2)
    with torch.no_grad():
        alpha = v / (v - iou + (1 + eps))
    return iou - (rho2 / c2 + v * alpha)


@torch.no_grad()
def task_aligned_assign(pd_scores, pd_bboxes, anc_points, gt_labels, gt_bboxes, mask_gt,
                        topk=10, alpha=0.5, beta=6.0, eps=1e-9, bbox_scores=None, nc=None, sparse=False):
    """Dense TaskAlignedAssigner (utils/tal.py:52-130): returns target_bboxes, target_scores, fg_mask.
    ``bbox_scores`` [bs, nmax, na] (optional): the predicted score of every anchor for each GT's own class, gathered by the
    caller (then ``pd_scores`` may be None).  ``sparse``: return the targets as (label [bs,na], value [bs,na]) instead of the
    dense one-hot ``target_scores`` -- target_scores[b,a,c] = value[b,a] * (c == label[b,a])."""
    if pd_scores is not None:
        bs, na, nc = pd_scores.shape
    else:
        bs, _, na = bbox_scores.shape
    nmax = gt_bboxes.shape[1]
    lt, rb = gt_bboxes.view(bs, nmax, 1, 4).chunk(2, -1)
    deltas = torch.cat((anc_points.view(1, 1, na, 2) - lt, rb - anc_points.view(1, 1, na, 2)), -1)
    mask_in_gts = deltas.amin(-1).gt(eps).to(pd_bboxes.dtype)  # [bs, nmax, na]
    m = mask_in_gts * mask_gt  # mask_gt: [bs, nmax, 1]
    if bbox_scores is None:
        lbl = gt_labels.long().clamp(0, nc - 1).view(bs, nmax, 1).expand(bs, nmax, na)
        bbox_scores = pd_scores.transpose(1, 2).gather(1, lbl)  # pd_scores[b, a, label[b, j]]
    bbox_scores = bbox_scores * m
    overlaps = _ciou(gt_bboxes.view(bs, nmax, 1, 4), pd_bboxes.view(bs, 1, na, 4)).clamp(0) * m
    align = bbox_scores.pow(alpha) * overlaps.pow(beta)
    _, topk_idx = torch.topk(align, topk, dim=-1)
    mask_topk = torch.zeros_like(align).scatter_(-1, topk_idx, 1.0) * mask_gt
    mask_pos = mask_topk * m
    fg = mask_pos.sum(-2)
    multi = (fg.unsqueeze(1) > 1).expand(-1, nmax, -1)
    is_max = torch.zeros_like(mask_pos).scatter_(1, overlaps.argmax(1, keepdim=True), 1.0)
    mask_pos = torch.where(multi, is_max, mask_pos)
    fg = mask_pos.sum(-2)
    tgt_idx = mask_pos.argmax(-2)  # [bs, na]
    flat_idx = tgt_idx + torch.arange(bs, device=tgt_idx.device).view(-1, 1) * nmax
    target_labels = gt_labels.long().flatten()[flat_idx].clamp(0)
    target_bboxes = gt_bboxes.reshape(-1, 4)[flat_idx]
    align = align * mask_pos
    pos_align = align.amax(-1, keepdim=True)
    pos_ovl = (overlaps * mask_pos).amax(-1, keepdim=True)
    norm = (align * pos_ovl / (pos_align + eps)).amax(-2).unsqueeze(-1)
    if sparse:   # (label, value) per anchor: background anchors get label -1 / value 0
        fgm = fg > 0
        return target_bboxes, (torch.where(fgm, target_labels, -1), norm.squeeze(-1) * fgm), fgm
    target_scores = F.one_hot(target_labels, nc).to(pd_bboxes.dtype) * (fg > 0).unsqueeze(-1)
    return target_bboxes, target_scores * norm, fg > 0


class DetectionLoss:
    """box/cls/dfl gains 7.5 / 0.5 / 1.5 (cfg/default.yaml:98-100); returns (loss.sum()*batch, items)."""

    def __init__(self, nc, strides, reg_max=16, box=7.5, cls=0.5, dfl=1.5, topk=10):
        self.nc, self.reg_max, self.no = nc, reg_max, nc + 4 * reg_max
        self.strides = [float(s) for s in strides]
        self.gains = (box, cls, dfl)
        self.topk = topk

    def targets_dense(self, batch, batch_size, max_boxes, wh, device):
        """[n,1+1+4] rows -> [B, max_boxes, 5] (cls, xyxy pixels), zero rows = padding (loss.py:175-190)."""
        bi = batch["batch_idx"].to(device).long().view(-1)
        n = bi.numel()
        out = torch.zeros(batch_size, max_boxes, 5, device=device)
        if n == 0:
            return out
        counts = torch.zeros(batch_size, dtype=torch.long, device=device).scatter_add_(0, bi, torch.ones_like(bi))  # no host sync
        start = torch.cumsum(counts, 0) - counts
        order = torch.argsort(bi, stable=True)
        rank = torch.empty_like(bi)
        rank[order] = torch.arange(n, device=device) - start[bi[order]]
        rows = torch.cat((batch["cls"].to(device).view(-1, 1).float(), batch["bboxes"].to(device).float()), 1)
        out[bi, rank] = rows
        xy, half = out[..., 1:3] * wh, out[..., 3:5] * wh / 2
        out[..., 1:5] = torch.cat((xy - half, xy + half), -1)
        return out

    cls_loss = None   # optional fused classification term: callable(cls_maps, label [B,A], value [B,A]) -> BCE sum (SURVEY 8(f)-4)

    det_kernels = None   # optional fused decode / assigner / box+DFL kernels (functional.DetLossKernels): SURVEY 8(f)-4

    def _call_fused(self, pairs, batch, max_boxes):
        """The whole loss on kernels: decode -> task-aligned assignment -> (box, DFL) sums and the classification sum, all read
        from the Detect head's maps in place (utils/loss.py:207-255 computes the same three numbers)."""
        K = self.det_kernels
        boxes, clss = [p[0] for p in pairs], [p[1] for p in pairs]
        device, bs = boxes[0].device, boxes[0].shape[0]
        h, w = boxes[0].shape[2:]
        wh = torch.stack((torch.full((), w * self.strides[0], device=device), torch.full((), h * self.strides[0], device=device)))
        gt = self.targets_dense(batch, bs, max_boxes, wh, device)        # [B, nmax, 5]: class, xyxy (pixels)
        with torch.no_grad():
            pred, scores = K.decode(boxes, clss, self.strides, gt)
            tlabel, tval, tbox = K.assign(pred, scores, gt, [f.shape[2:] for f in boxes], self.strides, topk=self.topk)
        tss = tval.sum().clamp(min=1.0)
        lcls = self.cls_loss(clss, tlabel, tval) / tss
        sums = K.box_dfl(boxes, tbox, tval) / tss
        loss = torch.stack((sums[0] * self.gains[0], lcls.float() * self.gains[1], sums[1] * self.gains[2]))
        return loss * bs, loss.detach()

    def _call_split(self, pairs, batch, max_boxes):
        """The same loss on the Detect head's un-concatenated (box, cls) maps: the class logits are never gathered into a
        [B, 8400, nc] tensor -- the assigner gathers the nmax scores it needs per anchor, the BCE term is one fused kernel
        over the class maps (utils/loss.py:207-255 computes the same three numbers)."""
        boxes, clss = [p[0] for p in pairs], [p[1] for p in pairs]
        device, bs = boxes[0].device, boxes[0].shape[0]
        pred_distri = torch.cat([f.permute(0, 2, 3, 1).reshape(bs, -1, self.reg_max * 4) for f in boxes], 1).float()
        dtype = pred_distri.dtype
        h, w = boxes[0].shape[2:]
        wh = torch.stack((torch.full((), w * self.strides[0], device=device), torch.full((), h * self.strides[0], device=device)))
        anchor_points, stride_tensor = make_anchors(boxes, self.strides, 0.5)
        t = self.targets_dense(batch, bs, max_boxes, wh, device)
        gt_labels, gt_bboxes = t[..., :1], t[..., 1:5]
        mask_gt = gt_bboxes.sum(2, keepdim=True).gt(0.0).to(torch.float32)
        b, a, c = pred_distri.shape
        proj = torch.arange(self.reg_max, dtype=dtype, device=device)
        dist = pred_distri.view(b, a, 4, c // 4).softmax(3).matmul(proj)
        pred_bboxes = torch.cat((anchor_points - dist[..., :2], anchor_points + dist[..., 2:]), -1)
        nmax = gt_bboxes.shape[1]
        with torch.no_grad():   # sigmoid(logit[b, a, label[b, j]]) for every GT j: the only class scores the assigner reads
            lbl = gt_labels.long().clamp(0, self.nc - 1).view(bs, 1, nmax)
            raw = torch.cat([f.permute(0, 2, 3, 1).reshape(bs, -1, self.nc).gather(2, lbl.expand(bs, f.shape[2] * f.shape[3], nmax))
                             for f in clss], 1)
            bbox_scores = raw.float().sigmoid().transpose(1, 2)
        target_bboxes, (tlabel, tval), fg = task_aligned_assign(
            None, (pred_bboxes.detach() * stride_tensor).float(), (anchor_points * stride_tensor).float(), gt_labels, gt_bboxes, mask_gt,
            topk=self.topk, bbox_scores=bbox_scores, nc=self.nc, sparse=True)
        tss = tval.sum().clamp(min=1.0)
        lcls = self.cls_loss(clss, tlabel, tval) / tss
        target_bboxes = target_bboxes / stride_tensor
        weight = tval * fg
        iou = _ciou(pred_bboxes.float(), target_bboxes)
        lbox = ((1.0 - iou) * weight).sum() / tss
        ltrb = torch.cat((anchor_points - target_bboxes[..., :2], target_bboxes[..., 2:] - anchor_points), -1)
        ltrb = ltrb.clamp(0, self.reg_max - 1 - 0.01)
        tl = ltrb.long()
        wl = (tl + 1) - ltrb
        logp = F.log_softmax(pred_distri.view(b, a, 4, self.reg_max).float(), -1)
        ce_l = -logp.gather(-1, tl.unsqueeze(-1)).squeeze(-1)
        ce_r = -logp.gather(-1, (tl + 1).unsqueeze(-1)).squeeze(-1)
        ldfl = (((ce_l * wl + ce_r * (1 - wl)).mean(-1)) * weight).sum() / tss
        loss = torch.stack((lbox * self.gains[0], lcls.float() * self.gains[1], ldfl * self.gains[2]))
        return loss * bs, loss.detach()

    def __call__(self, feats, batch, max_boxes=None):
        if isinstance(feats[0], (tuple, list)):
            if self.cls_loss is not None and max_boxes:
                if self.det_kernels is not None and self.det_kernels.supported([p[0] for p in feats], self.reg_max):
                    return self._call_fused(feats, batch, max_boxes)
                return self._call_split(feats, batch, max_boxes)
            feats = [torch.cat(p, 1) for p in feats]
        device = feats[0].device
        bs = feats[0].shape[0]
        # loss.py:207-213 builds [B, no, A] and permutes to [B, A, ·]; the same values are gathered anchor-major directly:
        # for channels_last maps `permute(0,2,3,1).reshape(B, HW, no)` is a free view, so the three per-level reshape copies
        # and the two permute+contiguous passes collapse into this one cat (in the activation dtype) + one cast to f32
        xa = torch.cat([f.permute(0, 2, 3, 1).reshape(bs, -1, self.no) for f in feats], 1).float()
        pred_distri, pred_scores = xa.split((self.reg_max * 4, self.nc), 2)
        pred_scores = pred_scores.contiguous()
        pred_distri = pred_distri.contiguous()
        dtype = pred_scores.dtype
        h, w = feats[0].shape[2:]
        wh = torch.stack((torch.full((), w * self.strides[0], device=device),      # fill kernels, no host->device copy:
                          torch.full((), h * self.strides[0], device=device)))     # the step stays CUDA-graph capturable
        anchor_points, stride_tensor = make_anchors(feats, self.strides, 0.5)
        if max_boxes is None:
            bi = batch["batch_idx"].long().view(-1)
            max_boxes = int(torch.bincount(bi, minlength=bs).max()) if bi.numel() else 0
        if max_boxes == 0:
            zero = pred_scores.sum() * 0
            lcls = F.binary_cross_entropy_with_logits(pred_scores, torch.zeros_like(pred_scores), reduction="sum")
            loss = torch.stack((zero, lcls * self.gains[1], zero)).float()
            return loss * bs, loss.detach()
        t = self.targets_dense(batch, bs, max_boxes, wh, device)
        gt_labels, gt_bboxes = t[..., :1], t[..., 1:5]
        mask_gt = gt_bboxes.sum(2, keepdim=True).gt(0.0).to(torch.float32)

        b, a, c = pred_distri.shape
        proj = torch.arange(self.reg_max, dtype=dtype, device=device)
        dist = pred_distri.view(b, a, 4, c // 4).softmax(3).matmul(proj)
        pred_bboxes = torch.cat((anchor_points - dist[..., :2], anchor_points + dist[..., 2:]), -1)

        target_bboxes, target_scores, fg = task_aligned_assign(
            pred_scores.detach().sigmoid().float(), (pred_bboxes.detach() * stride_tensor).float(),
            (anchor_points * stride_tensor).float(), gt_labels, gt_bboxes, mask_gt, topk=self.topk)
        tss = target_scores.sum().clamp(min=1.0)
        lcls = F.binary_cross_entropy_with_logits(pred_scores, target_scores.to(dtype), reduction="sum") / tss

        target_bboxes = target_bboxes / stride_tensor
        weight = target_scores.sum(-1) * fg
        iou = _ciou(pred_bboxes.float(), target_bboxes)
        lbox = ((1.0 - iou) * weight).sum() / tss
        ltrb = torch.cat((anchor_points - target_bboxes[..., :2], target_bboxes[..., 2:] - anchor_points), -1)
        ltrb = ltrb.clamp(0, self.reg_max - 1 - 0.01)
        tl = ltrb.long()
        wl = (tl + 1) - ltrb
        logp = F.log_softmax(pred_distri.view(b, a, 4, self.reg_max).float(), -1)
        ce_l = -logp.gather(-1, tl.unsqueeze(-1)).squeeze(-1)
        ce_r = -logp.gather(-1, (tl + 1).unsqueeze(-1)).squeeze(-1)
        ldfl = (((ce_l * wl + ce_r * (1 - wl)).mean(-1)) * weight).sum() / tss
        loss = torch.stack((lbox * self.gains[0], lcls.float() * self.gains[1], ldfl * self.gains[2]))
        return loss * bs, loss.detach()
