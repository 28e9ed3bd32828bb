"""CPU: the harness loss on the Detect head's un-concatenated (box, cls) maps with (label, value) targets -- the form the fused
classification-loss kernel consumes (SURVEY 8(f)-4) -- equals the dense form.  Both forms are pinned to the reference's v8DetectionLoss by
tests/test_det_loss_oracle.py, against the line-by-line restatement oracle/det_loss.py."""
import torch
import torch.nn.functional as F


def _dense_bce(maps, label, value):
    bs = maps[0].shape[0]
    nc = maps[0].shape[1]
    x = torch.cat([m.permute(0, 2, 3, 1).reshape(bs, -1, nc) for m in maps], 1).float()
    t = F.one_hot(label.clamp(min=0).long(), nc).float() * (value * (label >= 0)).unsqueeze(-1)
    return F.binary_cross_entropy_with_logits(x, t, reduction="sum")


def test_split_form_equals_dense_form_values_and_gradients():
    from improving_yolov8_cbam_swinblock_b200.harness import loss as hl, synthetic

    torch.manual_seed(0)
    nc, bs = 80, 3
    strides = [8.0, 16.0, 32.0]
    sizes = [(16, 16), (8, 8), (4, 4)]
    batch = synthetic.make_batch(bs, 128, nc, seed=4)
    box = [torch.randn(bs, 64, h, w, requires_grad=True) for h, w in sizes]
    cls = [(torch.randn(bs, nc, h, w) - 2).requires_grad_(True) for h, w in sizes]
    crit = hl.DetectionLoss(nc, strides)
    dense_feats = [torch.cat((b, c), 1) for b, c in zip(box, cls)]
    l0, i0 = crit(dense_feats, batch, max_boxes=8)
    l0.sum().backward()
    g0 = [t.grad.clone() for t in box + cls]
    for t in box + cls:
        t.grad = None
    crit.cls_loss = _dense_bce
    l1, i1 = crit(list(zip(box, cls)), batch, max_boxes=8)
    l1.sum().backward()
    torch.testing.assert_close(i1, i0, rtol=1e-5, atol=1e-6)
    for a, b in zip([t.grad for t in box + cls], g0):
        torch.testing.assert_close(a, b, rtol=1e-4, atol=1e-7)
    # pairs without a fused kernel fall back to the dense form
    crit.cls_loss = None
    l2, i2 = crit(list(zip(box, cls)), batch, max_boxes=8)
    torch.testing.assert_close(i2, i0, rtol=1e-6, atol=1e-7)
