"""Seeded detection-loss scenes shared by tests/test_det_loss_oracle.py (CPU) and tests/test_gpu_det_edges.py (GPU).

Each scene is a small batch -- Detect head maps (float64 logits, NCHW) and a label list in the trainer's format -- built to
exercise one edge of the task-aligned assigner or of the box / DFL / classification terms.  ``Scene.check`` asserts, through the
restated reference (``oracle/det_loss.py``), that the scene really contains its case, so an edit that removes the case fails
instead of silently testing less.  Coordinates are dyadic: every box corner is exact in float32 and float64.
"""
from __future__ import annotations

from dataclasses import dataclass, field

import torch

from oracle import det_loss as od

REG = 16


@dataclass
class Scene:
    name: str
    nc: int
    sizes: list                    # [(h, w)] per level
    strides: list
    box: list                      # [B, 64, h, w] float64 DFL logits per level
    cls: list                      # [B, nc, h, w] float64 class logits per level
    labels: list                   # [(image, class, x1, y1, x2, y2)] in pixels
    topks: tuple = (10,)
    case: str = ""
    check: object = None           # callable(Scene, OracleRun) asserting the case
    extra: dict = field(default_factory=dict)

    @property
    def bs(self):
        return self.box[0].shape[0]

    @property
    def imgsz(self):                # (h, w) in pixels
        return self.sizes[0][0] * self.strides[0], self.sizes[0][1] * self.strides[0]

    @property
    def A(self):
        return sum(h * w for h, w in self.sizes)

    def batch(self, dtype=torch.float64, device="cpu"):
        """The trainer's label format: batch_idx, cls, normalised xywh."""
        h, w = self.imgsz
        t = torch.tensor([list(r) for r in self.labels], dtype=torch.float64).view(-1, 6)
        xy = (t[:, 2:4] + t[:, 4:6]) / 2
        wh = t[:, 4:6] - t[:, 2:4]
        scale = torch.tensor([w, h], dtype=torch.float64)
        return {"batch_idx": t[:, 0].to(dtype).to(device), "cls": t[:, 1:2].to(dtype).to(device),
                "bboxes": torch.cat((xy / scale, wh / scale), 1).to(dtype).to(device)}

    def max_boxes(self):
        counts = [sum(1 for r in self.labels if r[0] == b) for b in range(self.bs)]
        return max(counts + [1])

    def gt(self, dtype=torch.float64, device="cpu"):
        """Dense [B, nmax >= 1, 5] GT tensor (class, xyxy pixels) as v8DetectionLoss.preprocess builds it, padded to one row."""
        crit = od.v8DetectionLoss(self.nc, self.strides, device=device)
        g = crit.targets(self.batch(dtype, device), self.bs, torch.tensor(self.imgsz, dtype=dtype, device=device))
        if g.shape[1] == 0:
            g = torch.zeros(self.bs, 1, 5, dtype=dtype, device=device)
        return g

    def feats(self, dtype=torch.float64, device="cpu"):
        return [torch.cat((b, c), 1).to(device=device, dtype=dtype).contiguous() for b, c in zip(self.box, self.cls)]

    def maps(self, dtype, device):
        cl = lambda t: t.to(device=device, dtype=dtype).contiguous(memory_format=torch.channels_last)  # noqa: E731
        return [cl(b) for b in self.box], [cl(c) for c in self.cls]


@dataclass
class OracleRun:
    """Targets of the oracle's TaskAlignedAssigner in the kernel's sparse form, plus the assigner's intermediates."""
    tlabel: torch.Tensor   # [B, A] int64, -1 = background
    tval: torch.Tensor     # [B, A]
    tbox: torch.Tensor     # [B, A, 4] pixels (zeros on background)
    fg: torch.Tensor       # [B, A] bool
    last: dict
    gt: torch.Tensor
    anc: torch.Tensor      # [A, 2] pixels
    pred: torch.Tensor     # [B, A, 4] the decoded boxes (grid units) the assigner was given
    scores: torch.Tensor   # [B, A, nc] the class scores the assigner was given


def decode(scene, dtype=torch.float64, device="cpu"):
    """Oracle bbox_decode of the scene's box logits: predicted boxes [B, A, 4] in grid units."""
    crit = od.v8DetectionLoss(scene.nc, scene.strides, device=device)
    bs = scene.bs
    pd = torch.cat([b.to(device=device, dtype=dtype).reshape(bs, 4 * REG, -1) for b in scene.box], 2).permute(0, 2, 1).contiguous()
    anc, _ = od.make_anchors(scene.box, scene.strides)
    return crit.bbox_decode(anc.to(device=device, dtype=dtype), pd)


def class_scores(scene, dtype=torch.float64, device="cpu"):
    bs = scene.bs
    x = torch.cat([c.to(device=device, dtype=dtype).reshape(bs, scene.nc, -1) for c in scene.cls], 2).permute(0, 2, 1)
    return x.sigmoid().contiguous()


def run_oracle(scene, topk=10, stable=True, dtype=torch.float64, device="cpu", pred=None, scores=None, gt=None):
    """The oracle assigner on ``pred`` (grid units, [B, A, 4]) and ``scores`` ([B, A, nc]); by default the scene's own decoded
    boxes and sigmoid class scores in ``dtype``."""
    pred = decode(scene, dtype, device) if pred is None else pred.to(device=device, dtype=dtype)
    scores = class_scores(scene, dtype, device) if scores is None else scores.to(device=device, dtype=dtype)
    gt = scene.gt(dtype, device) if gt is None else gt.to(device=device, dtype=dtype)
    anc, st = od.make_anchors([b.to(device=device, dtype=dtype) for b in scene.box], scene.strides)
    asg = od.TaskAlignedAssigner(topk=topk, num_classes=scene.nc, alpha=0.5, beta=6.0, stable_topk=stable)
    mask_gt = gt[..., 1:5].sum(2, keepdim=True).gt_(0.0)
    labels, tbox, tscores, fg, _ = asg(scores, pred * st, anc * st, gt[..., :1], gt[..., 1:5], mask_gt)
    tlabel = torch.where(fg, labels, torch.full_like(labels, -1))
    return OracleRun(tlabel, tscores.sum(-1), tbox * fg.unsqueeze(-1), fg, asg.last, gt, anc * st, pred, scores)


def scores_from_gathered(gathered, gt, nc):
    """[B, nmax, A] scores of every GT's own class (what det_decode returns) -> [B, A, nc] for the reference's assigner.
    GTs of the same class carry the same scores; the other classes are never read."""
    B, nmax, A = gathered.shape
    out = torch.zeros(B, A, nc, dtype=gathered.dtype, device=gathered.device)
    lbl = gt[..., 0].long().clamp(0, nc - 1)
    for b in range(B):
        for j in range(nmax):
            out[b, :, lbl[b, j]] = gathered[b, j]
    return out


def topk_gaps(run, topk):
    """Relative gap between the k-th and (k+1)-th alignment metric of every valid GT (1 where fewer than k are positive)."""
    m = run.last["align_metric"]
    srt = m.sort(-1, descending=True).values
    kth, nxt = srt[..., topk - 1], srt[..., topk] if srt.shape[-1] > topk else torch.zeros_like(srt[..., 0])
    gap = torch.where(kth > 0, (kth - nxt) / kth.clamp(min=1e-300), torch.ones_like(kth))
    valid = run.gt[..., 1:5].sum(-1) > 0
    return gap[valid]


def claim_gaps(run):
    """For anchors claimed by several GTs: relative gap between the largest and second-largest overlap (1 if unique)."""
    multi = run.last["mask_pos_pre"].sum(-2) > 1
    if not bool(multi.any()):
        return torch.ones(0, dtype=run.tval.dtype)
    o = run.last["overlaps"].sort(-2, descending=True).values   # [B, nmax, A]
    if o.shape[1] < 2:
        return torch.ones(0, dtype=run.tval.dtype)
    top, second = o[:, 0], o[:, 1]
    gap = torch.where(top > second, (top - second) / top.clamp(min=1e-300), torch.zeros_like(top))
    return gap[multi & (top > second)]


def oracle_loss(s, topk, dtype=torch.float64, device="cpu", box=None, cls=None):
    """v8DetectionLoss (stable top-k) in ``dtype`` on the scene's maps (or on ``box`` / ``cls``): items and the gradient of
    every box and class map."""
    box = [b.detach().to(device=device, dtype=dtype).contiguous().requires_grad_(True) for b in (box or s.box)]
    cls = [c.detach().to(device=device, dtype=dtype).contiguous().requires_grad_(True) for c in (cls or s.cls)]
    crit = od.v8DetectionLoss(s.nc, s.strides, tal_topk=topk, stable_topk=True, device=device)
    loss, items = crit([torch.cat((b, c), 1) for b, c in zip(box, cls)], s.batch(dtype, device))
    loss.backward()
    return items, [t.grad for t in box + cls]


def assert_selection_margins(s, topk, device="cpu", pred=None, scores=None):
    """Every GT's top-k boundary and every multi-claim overlap maximum is separated by > 1e-4 relative, so last-bit
    differences of the decode cannot change which anchors are selected."""
    r = run_oracle(s, topk=topk, device=device, pred=pred, scores=scores)
    gaps, claims = topk_gaps(r, topk), claim_gaps(r)
    assert bool((gaps > 1e-4).all()), f"top-k boundary gaps {gaps[gaps <= 1e-4].tolist()}"
    assert bool((claims > 1e-4).all()), f"multi-claim overlap gaps {claims[claims <= 1e-4].tolist()}"


# ---- construction helpers ---------------------------------------------------------------------------------------
def _gen(seed):
    return torch.Generator().manual_seed(seed)


def _rand_maps(bs, nc, sizes, seed, spread=1.0, cls_scale=2.0, cls_shift=-1.0):
    g = _gen(seed)
    box = [spread * torch.randn(bs, 4 * REG, h, w, generator=g, dtype=torch.float64) for h, w in sizes]
    cls = [cls_scale * torch.randn(bs, nc, h, w, generator=g, dtype=torch.float64) + cls_shift for h, w in sizes]
    return box, cls


def pair_peaked(bins):
    """DFL logits with +100 on bins c and c+1 of each side (0 elsewhere): softmax (0.5, 0.5) exactly, so the decoded distance
    is exactly c + 0.5 in every precision and the predicted edge x + 0.5 -/+ (c + 0.5) is an integer, while the softmax still
    has a gradient.  ``bins``: [B, 4, h, w] integers in 0..14 -> [B, 64, h, w]."""
    B, _, h, w = bins.shape
    x = torch.zeros(B, 4, REG, h, w, dtype=torch.float64)
    x.scatter_(2, bins.long().unsqueeze(2), 100.0)
    x.scatter_(2, bins.long().unsqueeze(2) + 1, 100.0)
    return x.view(B, 4 * REG, h, w)


def _rand_labels(bs, n, imgsz, nc, seed, lo=0.05, hi=0.35, grid=1.0):
    g = _gen(seed)
    H, W = imgsz
    out = []
    for b in range(bs):
        for _ in range(n):
            cx, cy = (0.15 + 0.7 * torch.rand(2, generator=g)).tolist()
            bw, bh = (lo + (hi - lo) * torch.rand(2, generator=g)).tolist()
            x1, x2 = max(0.0, (cx - bw / 2) * W), min(float(W), (cx + bw / 2) * W)
            y1, y2 = max(0.0, (cy - bh / 2) * H), min(float(H), (cy + bh / 2) * H)
            q = lambda v: round(v / grid) * grid  # noqa: E731  (dyadic corners)
            out.append((b, int(torch.randint(0, nc, (1,), generator=g)), q(x1), q(y1), q(x2), q(y2)))
    return out


SIZES3 = [(16, 16), (8, 8), (4, 4)]
STRIDES3 = [8.0, 16.0, 32.0]


# ---- the scenes ---------------------------------------------------------------------------------------------------
def _check_duplicate(s, r):
    pre, ov, idx = r.last["mask_pos_pre"], r.last["overlaps"], r.last["target_gt_idx"]
    both = (pre[0, 0] > 0) & (pre[0, 1] > 0)
    assert torch.equal(ov[0, 0], ov[0, 1]), "duplicate GTs must have identical overlaps"
    assert bool(both.any()), "no anchor is claimed by both duplicate GTs"
    assert bool((idx[0][both] == 0).all()) and bool(r.fg[0][both].all()), "a tie across GTs must go to the lower GT index"
    assert int(r.tlabel[0][both][0]) == int(r.gt[0, 0, 0])


def duplicate():
    box, cls = _rand_maps(2, 8, SIZES3, 11)
    lab = [(0, 1, 32, 32, 80, 72), (0, 2, 32, 32, 80, 72), (0, 3, 72, 16, 120, 56), (1, 5, 16, 40, 64, 100)]
    return Scene("duplicate", 8, SIZES3, STRIDES3, box, cls, lab, case="identical boxes, different classes", check=_check_duplicate)


def _check_nested(s, r):
    pre, idx = r.last["mask_pos_pre"], r.last["target_gt_idx"]
    multi = pre.sum(-2) > 1                                           # [B, A]
    sel_by_winner = pre.gather(1, idx.unsqueeze(1)).squeeze(1) > 0
    hit = multi & ~sel_by_winner & r.fg
    assert bool(hit.any()), "no multi-claimed anchor goes to a GT that did not select it"


def nested():
    box, cls = _rand_maps(2, 8, SIZES3, 21)
    lab = [(0, 0, 16, 16, 112, 112), (0, 1, 40, 40, 72, 72), (0, 2, 48, 40, 80, 72), (1, 3, 8, 8, 120, 120), (1, 4, 56, 56, 88, 80)]
    return Scene("nested", 8, SIZES3, STRIDES3, box, cls, lab, case="multi-claim to a non-selecting GT", check=_check_nested)


def _check_subcell(s, r):
    j = s.extra["sub"]
    assert bool(r.gt[0, j, 1:5].sum() > 0), "the sub-cell GT must be valid"
    assert int(r.last["mask_in_gts"][0, j].sum()) == 0, "an anchor centre lies inside the sub-cell GT"
    assert not bool((r.last["mask_pos"][0, j] > 0).any())
    g2 = r.gt.clone()
    g2[0, j] = 0
    r2 = run_oracle(s, gt=g2, dtype=r.tval.dtype, device=r.tval.device, pred=r.pred, scores=r.scores)
    assert torch.equal(r2.fg, r.fg) and torch.equal(r2.tlabel, r.tlabel) and torch.equal(r2.tval, r.tval), "the sub-cell GT changed others"


def subcell():
    box, cls = _rand_maps(1, 8, SIZES3, 31)
    lab = [(0, 2, 24, 24, 72, 64), (0, 3, 61, 61, 66, 66), (0, 4, 64, 72, 112, 120)]
    return Scene("subcell", 8, SIZES3, STRIDES3, box, cls, lab, case="valid GT with no anchor centre inside",
                 check=_check_subcell, extra={"sub": 1})


def _check_sparse(s, r):
    m, inb, pre = r.last["align_metric"][0, 0], r.last["mask_in_gts"][0, 0] > 0, r.last["mask_pos_pre"][0, 0] > 0
    npos = int((m > 0).sum())
    assert 0 < npos < 10, f"{npos} positive candidates: the top-k must run out early"
    assert bool((inb & (r.last["overlaps"][0, 0] == 0)).any()), "no in-box anchor with CIoU <= 0"
    zero_fg = pre & (m == 0)
    assert bool(zero_fg.any()), "the reference's top-k must pick a zero-metric in-box anchor"
    # stable top-k: the zero picks are the lowest anchor indices
    picks = r.last["topk_idxs"][0, 0]
    zero_picks = picks[m[picks] == 0]
    want = torch.nonzero(m == 0).flatten()[: zero_picks.numel()]
    assert torch.equal(zero_picks.sort().values, want.to(zero_picks.device)), "zero picks are not the lowest anchor indices"
    assert bool((r.tval[0][zero_fg] == 0).all())


def sparse():
    box, cls = _rand_maps(2, 8, SIZES3, 41)
    # anchors 0 and 1 (pixel centres (4,4) and (12,4)) inside the corner GT get (almost) zero-width predictions: a single peak on
    # bin 0 for the left and right sides, so CIoU < 0 there and their metric is 0
    zero_width = pair_peaked(torch.tensor([0, 3, 0, 3]).view(1, 4, 1, 1))[0, :, 0, 0]
    zero_width[0:REG] = torch.tensor([100.0] + [0.0] * 15)
    zero_width[2 * REG:3 * REG] = torch.tensor([100.0] + [0.0] * 15)
    box[0][0, :, 0, 0] = zero_width
    box[0][0, :, 0, 1] = zero_width
    lab = [(0, 0, 0, 0, 20, 20), (0, 6, 64, 56, 112, 104), (1, 1, 40, 24, 88, 72)]
    return Scene("sparse", 8, SIZES3, STRIDES3, box, cls, lab, case="fewer positives than topk, zero-metric in-box picks",
                 check=_check_sparse)


def _check_boundary(s, r):
    anc, gt = r.anc, r.gt[0]
    d = torch.cat((anc[None] - gt[:, None, 1:3], gt[:, None, 3:5] - anc[None]), -1).amin(-1)   # [nmax, A]
    on_edge = d == 0
    assert bool(on_edge.any()), "no anchor centre on a GT edge"
    assert not bool((r.last["mask_in_gts"][0][on_edge] > 0).any()), "an anchor on the edge counted as inside"
    H, W = s.imgsz
    assert bool((gt[:, 1] == 0).any() and (gt[:, 2] == 0).any() and (gt[:, 3] == W).any() and (gt[:, 4] == H).any())
    # the edge anchors would be picked if they were inside: the small GT has fewer positives than topk
    assert int((r.last["align_metric"][0, 0] > 0).sum()) < 10


def boundary():
    box, cls = _rand_maps(1, 8, SIZES3, 51)
    lab = [(0, 1, 4, 4, 20, 20), (0, 2, 0, 88, 40, 128), (0, 3, 96, 0, 128, 36), (0, 4, 44, 36, 76, 68)]
    return Scene("boundary", 8, SIZES3, STRIDES3, box, cls, lab, case="edges on anchor centres, boxes on the image border",
                 check=_check_boundary)


def _check_padding(s, r):
    g = r.gt
    assert float(g[0, 1, 1:5].abs().sum()) == 0 and float(g[0, 2, 1:5].sum()) > 0, "padding row must sit before a valid row"
    assert float(g[1].abs().sum()) == 0 and not bool(r.fg[1].any()), "image 1 must be empty"
    assert bool(r.fg[0].any()) and bool(r.fg[2].any())


def padding():
    box, cls = _rand_maps(3, 8, SIZES3, 61)
    lab = [(0, 1, 16, 16, 56, 64), (0, 0, 0, 0, 0, 0), (0, 7, 64, 48, 120, 100), (2, 3, 24, 64, 80, 120)]
    return Scene("padding", 8, SIZES3, STRIDES3, box, cls, lab, case="padding row before a valid row; empty image",
                 check=_check_padding)


def _check_empty(s, r):
    assert float(r.gt.abs().sum()) == 0 and not bool(r.fg.any())


def empty():
    box, cls = _rand_maps(2, 8, SIZES3, 71)
    return Scene("empty", 8, SIZES3, STRIDES3, box, cls, [], case="no GT in the batch", check=_check_empty)


def _check_crowd(s, r):
    assert int((r.gt[0, :, 1:5].sum(-1) > 0).sum()) >= 100


def crowd():
    sizes, strides = [(32, 32), (16, 16), (8, 8)], STRIDES3
    box, cls = _rand_maps(1, 16, sizes, 83)
    lab = _rand_labels(1, 110, (256, 256), 16, 82, lo=0.02, hi=0.2)
    return Scene("crowd", 16, sizes, strides, box, cls, lab, topks=(1, 10, 13, 64), case=">= 100 boxes in one image",
                 check=_check_crowd)


def _check_tie(s, r):
    m = r.last["align_metric"][0, 0]
    srt = m.sort(descending=True).values
    for k in s.topks:
        assert srt[k - 1] > 0 and srt[k - 1] == srt[k], f"topk={k}: the k-th and (k+1)-th metric are not an exact tie"


def tie():
    bs, nc = 1, 8
    box = [torch.zeros(bs, 4 * REG, h, w, dtype=torch.float64) for h, w in SIZES3]     # uniform: every distance 7.5
    cls = [torch.zeros(bs, nc, h, w, dtype=torch.float64) for h, w in SIZES3]          # every score 0.5
    lab = [(0, 3, 40, 44, 88, 84)]                                                     # symmetric about (64, 64)
    return Scene("tie", nc, SIZES3, STRIDES3, box, cls, lab, topks=(10,), case="exact metric tie at the k-th place",
                 check=_check_tie)


def _check_saturated(s, r):
    x = torch.cat([c.flatten() for c in s.cls])
    assert bool((x.abs() == 30).all()) and bool((x > 0).any()) and bool((x < 0).any())
    assert bool(r.fg.any())


def saturated():
    box, cls = _rand_maps(2, 8, SIZES3, 91)
    g = _gen(92)
    cls = [torch.where(torch.rand(c.shape, generator=g, dtype=torch.float64) < 0.5, 30.0, -30.0) for c in cls]
    lab = _rand_labels(2, 4, (128, 128), 8, 93)
    return Scene("saturated", 8, SIZES3, STRIDES3, box, cls, lab, case="class logits of +-30", check=_check_saturated)


def _check_fg(s, r):
    assert bool(r.fg.any())


def geometry(kind):
    if kind == "one_level":
        sizes, strides = [(20, 24)], [8.0]
    elif kind == "four_levels":
        sizes, strides = [(32, 32), (16, 16), (8, 8), (4, 4)], [4.0, 8.0, 16.0, 32.0]
    elif kind == "nonsquare":
        sizes, strides = [(12, 20), (6, 10), (3, 5)], STRIDES3
    elif kind == "big1024":
        sizes, strides = [(128, 128), (64, 64), (32, 32)], STRIDES3
    else:
        raise ValueError(kind)
    bs = 1 if kind == "big1024" else 2
    box, cls = _rand_maps(bs, 8, sizes, 101 + len(sizes))
    H, W = sizes[0][0] * strides[0], sizes[0][1] * strides[0]
    lab = _rand_labels(bs, 6, (H, W), 8, 111 + len(sizes))
    return Scene(kind, 8, sizes, strides, box, cls, lab, case=kind, check=_check_fg)


def _check_edges(s, r):
    for dt in (torch.float32, torch.float64):
        d = decode(s, dt)
        assert torch.equal(d, d.round()), f"{dt}: decoded edges are not exact integers"
    assert bool(r.fg.any())


def edges():
    """Pair-peaked DFL logits everywhere (integer predicted edges, exact in every precision); GTs for the whole loss.  The
    box / DFL tests add explicit targets per anchor (``edge_targets``)."""
    bs, nc = 2, 8
    g = _gen(121)
    box = [pair_peaked(torch.randint(1, 12, (bs, 4, h, w), generator=g)) for h, w in SIZES3]
    cls = [2 * torch.randn(bs, nc, h, w, generator=g, dtype=torch.float64) - 1 for h, w in SIZES3]
    lab = [(0, 1, 16, 24, 72, 88), (0, 5, 80, 8, 120, 48), (1, 2, 8, 56, 120, 120), (1, 6, 40, 8, 88, 40)]
    return Scene("edges", nc, SIZES3, STRIDES3, box, cls, lab, case="integer predicted edges", check=_check_edges)


def edge_targets(scene):
    """Explicit (target box [B, A, 4] grid units, weight [B, A], fg [B, A]) over the edge scene's predicted boxes, cycling per
    anchor through: target = prediction (min / max ties on all four edges); one tied edge with target distances on integers and
    above 14.99; boxes that touch (intersection width exactly 0); disjoint boxes; fg with weight 0; background."""
    pred = decode(scene)                                              # [B, A, 4] grid units, integers
    anc, _ = od.make_anchors(scene.box, scene.strides)
    B, A = pred.shape[:2]
    g = _gen(131)
    tb = torch.zeros(B, A, 4, dtype=torch.float64)
    w = (0.1 + 0.9 * torch.rand(B, A, generator=g, dtype=torch.float64))
    fg = torch.ones(B, A, dtype=torch.bool)
    kind = torch.arange(A).remainder(7).expand(B, A)
    ax, ay = anc[:, 0].expand(B, A), anc[:, 1].expand(B, A)
    px1, py1, px2, py2 = pred.unbind(-1)
    cases = {
        0: (px1, py1, px2, py2),                                      # identical: every min / max ties
        1: (px1, ay - 3.0, ax + 15.0, ay + 17.0),                     # x1 tied; distances 3 (integer), 15 and 17 (> 14.99)
        2: (px2, py1, px2 + 4.0, py2),                                # touching: intersection width exactly 0
        3: (px2 + 2.0, py2 + 1.0, px2 + 6.0, py2 + 5.0),              # disjoint
        4: (ax - 20.0, ay - 15.0, ax + 7.0, py2),                     # y2 tied; 20, 15 clamp to 14.99
        5: (px1 - 1.0, py1, px2 + 1.0, py2 + 2.0),                    # fg with weight 0
        6: (px1, py1, px2, py2),                                      # background
    }
    for k, (x1, y1, x2, y2) in cases.items():
        sel = kind == k
        tb[sel] = torch.stack((x1, y1, x2, y2), -1)[sel]
    w[kind == 5] = 0.0
    w[kind == 6] = 0.0
    fg[kind == 6] = False
    return tb, w, fg, kind


SCENES = {
    "duplicate": duplicate, "nested": nested, "subcell": subcell, "sparse": sparse, "boundary": boundary, "padding": padding,
    "empty": empty, "crowd": crowd, "tie": tie, "saturated": saturated, "edges": edges,
    "one_level": lambda: geometry("one_level"), "four_levels": lambda: geometry("four_levels"),
    "nonsquare": lambda: geometry("nonsquare"), "big1024": lambda: geometry("big1024"),
}


def make(name):
    return SCENES[name]()


def cases(names=None):
    """(scene name, topk) pairs: every scene at each of its topk values."""
    out = []
    for n in (names or SCENES):
        s = make(n)
        out += [(n, k) for k in s.topks]
    return out
