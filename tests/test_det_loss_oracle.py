"""CPU: the harness restatement of the detection loss (harness/loss.py) against the line-by-line restatement of the reference
(oracle/det_loss.py: Ultralytics 8.3.108 v8DetectionLoss + TaskAlignedAssigner + BboxLoss), on the edge scenes of
tests/det_scenes.py.  This is what pins the harness loss -- and through it the kernels, which tests/test_gpu_det_edges.py
compares with the same oracle -- to the reference's function."""
import pytest
import torch

import det_scenes as ds
from oracle import det_loss as od
from test_loss_split import _dense_bce
from util import rel_err

ALL = ds.cases()
LOSS = [c for c in ALL if c[0] != "tie"]   # the exact-tie scene has no well-defined selection under rounding


@pytest.mark.parametrize("name,topk", ALL)
def test_scene_contains_its_case(name, topk):
    s = ds.make(name)
    s.check(s, ds.run_oracle(s, topk=topk))


@pytest.mark.parametrize("name,topk", ALL)
def test_harness_assigner_matches_oracle_fp64(name, topk):
    """harness.loss.task_aligned_assign, dense and sparse=True, against the reference's assigner as written (torch.topk)."""
    from improving_yolov8_cbam_swinblock_b200.harness import loss as hl

    s = ds.make(name)
    pred, scores = ds.decode(s), ds.class_scores(s)
    r = ds.run_oracle(s, topk=topk, stable=False, pred=pred, scores=scores)
    gt = r.gt
    anc, st = od.make_anchors(s.box, s.strides)
    mask_gt = gt[..., 1:5].sum(2, keepdim=True).gt(0).double()
    args = (scores, pred * st, anc * st, gt[..., :1], gt[..., 1:5], mask_gt)
    tb, tsc, fg = hl.task_aligned_assign(*args, topk=topk)
    assert torch.equal(fg, r.fg), f"fg sets differ at {int((fg != r.fg).sum())} anchors"
    want_sc = torch.nn.functional.one_hot(r.tlabel.clamp(min=0), s.nc).double() * r.tval.unsqueeze(-1)
    torch.testing.assert_close(tsc, want_sc, rtol=1e-12, atol=0)
    assert torch.equal(tb[fg], r.tbox[r.fg])
    lbl = gt[..., 0].long().clamp(0, s.nc - 1).unsqueeze(1).expand(-1, s.A, -1)
    gathered = scores.gather(2, lbl).transpose(1, 2)   # [B, nmax, A]: what the split form hands the assigner
    tb2, (lab, val), fg2 = hl.task_aligned_assign(None, *args[1:], topk=topk, bbox_scores=gathered, nc=s.nc, sparse=True)
    assert torch.equal(fg2, r.fg) and torch.equal(lab.long(), r.tlabel)
    torch.testing.assert_close(val, r.tval, rtol=1e-12, atol=0)
    assert torch.equal(tb2[fg2], r.tbox[r.fg])


def _harness_loss(s, topk, split):
    from improving_yolov8_cbam_swinblock_b200.harness import loss as hl

    crit = hl.DetectionLoss(s.nc, s.strides, topk=topk)
    box = [b.clone().requires_grad_(True) for b in s.box]
    cls = [c.clone().requires_grad_(True) for c in s.cls]
    if split:
        crit.cls_loss = _dense_bce
        loss, items = crit(list(zip(box, cls)), s.batch(torch.float32), max_boxes=s.max_boxes())
    else:
        loss, items = crit([torch.cat((b, c), 1) for b, c in zip(box, cls)], s.batch(torch.float32), max_boxes=s.max_boxes())
    loss.sum().backward()
    return items, [t.grad for t in box + cls]


@pytest.mark.parametrize("split", [False, True], ids=["dense", "split"])
@pytest.mark.parametrize("name,topk", LOSS)
def test_harness_loss_matches_oracle(name, topk, split):
    """DetectionLoss (f32 inside) against the reference's v8DetectionLoss in fp64: three items, gradients of all head maps."""
    s = ds.make(name)
    ds.assert_selection_margins(s, topk)
    items, grads = _harness_loss(s, topk, split)
    witems, wgrads = ds.oracle_loss(s, topk)
    torch.testing.assert_close(items.double(), witems, rtol=2e-5, atol=1e-6)
    for g, w in zip(grads, wgrads):
        assert rel_err(g, w) < 2e-5, rel_err(g, w)
