"""-m gpu: the fused classification-loss kernels (csrc/det_loss.cu) against torch's BCEWithLogits on the dense one-hot target
(utils/loss.py:235 with the target of tal.py:98-107): value and the gradient of every class map."""
import pytest
import torch
import torch.nn.functional as F

from util import rel_err

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16, torch.float32])
@pytest.mark.parametrize("bs,nc,sizes", [(2, 80, [(8, 8), (4, 4), (2, 2)]), (64, 80, [(80, 80), (40, 40), (20, 20)]), (3, 16, [(5, 7)])])
def test_cls_bce_sum_matches_torch(dtype, bs, nc, sizes):
    from improving_yolov8_cbam_swinblock_b200 import functional as Fb

    torch.manual_seed(bs + nc)
    maps = [(2 * torch.randn(bs, nc, h, w, device="cuda") - 1).to(dtype).contiguous(memory_format=torch.channels_last).requires_grad_(True)
            for h, w in sizes]
    A = sum(h * w for h, w in sizes)
    label = torch.randint(-1, nc, (bs, A), device="cuda")
    label[torch.rand(bs, A, device="cuda") < 0.9] = -1
    value = torch.rand(bs, A, device="cuda") * (label >= 0)
    got = Fb.cls_bce_sum(maps, label, value)
    (got * 0.37).backward()
    x = torch.cat([m.detach().permute(0, 2, 3, 1).reshape(bs, -1, nc) for m in maps], 1).double().requires_grad_(True)
    t = F.one_hot(label.clamp(min=0), nc).double() * value.double().unsqueeze(-1)
    want = F.binary_cross_entropy_with_logits(x, t, reduction="sum")
    (want * 0.37).backward()
    assert rel_err(got, want) < 1e-5, (float(got), float(want))
    off = 0
    for m, (h, w) in zip(maps, sizes):
        g = m.grad.permute(0, 2, 3, 1).reshape(bs, h * w, nc)
        assert m.grad.is_contiguous(memory_format=torch.channels_last)
        assert rel_err(g, x.grad[:, off:off + h * w]) < (1e-6 if dtype == torch.float32 else 4e-3)
        off += h * w
    # deterministic
    assert torch.equal(got, Fb.cls_bce_sum([m.detach() for m in maps], label, value))


# ---- assigner + box / DFL kernels (csrc/det_assign.cu) -----------------------------------------------------------
def _maps(bs, nc, sizes, dtype, seed, spread=1.0):
    torch.manual_seed(seed)
    cl = lambda t: t.to(dtype).contiguous(memory_format=torch.channels_last)  # noqa: E731
    box = [cl(spread * torch.randn(bs, 64, h, w, device="cuda")) for h, w in sizes]
    cls = [cl(2 * torch.randn(bs, nc, h, w, device="cuda") - 1) for h, w in sizes]
    return box, cls


def _gt(bs, nmax, imgsz, nc, seed, empty_image=True):
    g = torch.Generator().manual_seed(seed)
    n = torch.randint(1, nmax + 1, (bs,), generator=g)
    if empty_image:
        n[-1] = 0
    out = torch.zeros(bs, nmax, 5)
    for b in range(bs):
        k = int(n[b])
        c = torch.rand(k, 2, generator=g) * 0.6 + 0.2
        wh = torch.rand(k, 2, generator=g) * 0.3 + 0.05
        out[b, :k, 0] = torch.randint(0, nc, (k,), generator=g).float()
        out[b, :k, 1:3] = (c - wh / 2) * imgsz
        out[b, :k, 3:5] = (c + wh / 2) * imgsz
    return out.cuda()


CASES = [(3, 80, [(16, 16), (8, 8), (4, 4)], 128, 5), (4, 80, [(80, 80), (40, 40), (20, 20)], 640, 8), (2, 16, [(12, 20)], 160, 3),
         (2, 16, [(32, 32), (16, 16), (8, 8), (4, 4)], 128, 4), (2, 8, [(12, 20), (6, 10), (3, 5)], 96, 4)]


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16, torch.float32])
@pytest.mark.parametrize("bs,nc,sizes,imgsz,nmax", CASES)
def test_det_decode_matches_torch(dtype, bs, nc, sizes, imgsz, nmax):
    """utils/loss.py:199 bbox_decode (softmax over the 16 bins x arange) and the class scores the assigner gathers."""
    from improving_yolov8_cbam_swinblock_b200 import functional as Fb
    from improving_yolov8_cbam_swinblock_b200.harness.graph import make_anchors

    strides = [imgsz / s[0] for s in sizes]
    box, cls = _maps(bs, nc, sizes, dtype, 1)
    gt = _gt(bs, nmax, imgsz, nc, 2)
    pred, scores = Fb.det_decode(box, cls, strides, gt)
    pd = torch.cat([f.permute(0, 2, 3, 1).reshape(bs, -1, 64) for f in box], 1).double()
    anc, _ = make_anchors([f.float() for f in box], strides, 0.5)
    dist = pd.view(bs, -1, 4, 16).softmax(3) @ torch.arange(16, dtype=torch.float64, device="cuda")
    want = torch.cat((anc.double() - dist[..., :2], anc.double() + dist[..., 2:]), -1)
    torch.testing.assert_close(pred.double(), want, rtol=1e-5, atol=1e-5)
    lbl = gt[..., 0].long().clamp(0, nc - 1).view(bs, 1, nmax)
    raw = torch.cat([f.permute(0, 2, 3, 1).reshape(bs, -1, nc).gather(2, lbl.expand(bs, f.shape[2] * f.shape[3], nmax)) for f in cls], 1)
    torch.testing.assert_close(scores, raw.float().sigmoid().transpose(1, 2), rtol=1e-6, atol=1e-7)


@pytest.mark.parametrize("bs,nc,sizes,imgsz,nmax", CASES)
@pytest.mark.parametrize("spread", [1.0, 3.0])
def test_tal_assign_matches_the_torch_restatement(bs, nc, sizes, imgsz, nmax, spread):
    """tal.py:41-327 as restated in harness/loss.py:task_aligned_assign (pinned against the restated reference, oracle/det_loss.py,
    by tests/test_det_loss_oracle.py), on the same decoded boxes / scores: identical targets wherever either target is non-zero.
    The kernel copies the restatement's f32 arithmetic, so only an exact metric tie at a GT's k-th place (torch.topk orders
    ties arbitrarily, the kernel takes the lower anchor index) could separate them; these random inputs have none."""
    from improving_yolov8_cbam_swinblock_b200 import functional as Fb
    from improving_yolov8_cbam_swinblock_b200.harness import loss as hl
    from improving_yolov8_cbam_swinblock_b200.harness.graph import make_anchors

    strides = [imgsz / s[0] for s in sizes]
    box, cls = _maps(bs, nc, sizes, torch.float32, 3, spread)
    gt = _gt(bs, nmax, imgsz, nc, 4)
    pred, scores = Fb.det_decode(box, cls, strides, gt)
    tlabel, tval, tbox = Fb.tal_assign(pred, scores, gt, [f.shape[2:] for f in box], strides)
    anc, st = make_anchors(box, strides, 0.5)
    mask_gt = gt[..., 1:5].sum(2, keepdim=True).gt(0).float()
    wb, (wl, wv), wfg = hl.task_aligned_assign(None, pred * st, anc * st, gt[..., :1], gt[..., 1:5], mask_gt, bbox_scores=scores, nc=nc,
                                               sparse=True)
    pos = (wv > 0) | (tval > 0)
    assert int(pos.sum()) > 5 * bs
    mism = (tval - wv).abs() > 1e-6 * wv.abs().clamp(min=1e-3)
    assert int(mism.sum()) == 0, f"{int(mism.sum())} of {int(pos.sum())} positives differ"
    assert torch.equal(tlabel[pos].long(), wl[pos])
    assert torch.equal(tbox[pos], (wb / st)[pos])
    # run-to-run identical
    t2 = Fb.tal_assign(pred, scores, gt, [f.shape[2:] for f in box], strides)
    assert torch.equal(t2[0], tlabel) and torch.equal(t2[1], tval) and torch.equal(t2[2], tbox)


@pytest.mark.parametrize("dtype,tol", [(torch.bfloat16, 1e-2), (torch.float16, 2e-3), (torch.float32, 2e-5)])
@pytest.mark.parametrize("bs,nc,sizes,imgsz,nmax", CASES)
def test_box_dfl_sums_and_gradient_match_torch(dtype, tol, bs, nc, sizes, imgsz, nmax):
    """loss.py:84-107 BboxLoss (CIoU + DFL) in fp64 on the same (rounded) logits and the same targets."""
    from improving_yolov8_cbam_swinblock_b200 import functional as Fb
    from improving_yolov8_cbam_swinblock_b200.harness import loss as hl
    from improving_yolov8_cbam_swinblock_b200.harness.graph import make_anchors

    strides = [imgsz / s[0] for s in sizes]
    box, cls = _maps(bs, nc, sizes, dtype, 5)
    gt = _gt(bs, nmax, imgsz, nc, 6)
    pred, scores = Fb.det_decode(box, cls, strides, gt)
    tlabel, tval, tbox = Fb.tal_assign(pred, scores, gt, [f.shape[2:] for f in box], strides)
    maps = [b.clone().requires_grad_(True) for b in box]
    sums = Fb.box_dfl_sums(maps, tbox, tval)
    up = 4096.0 if dtype == torch.float16 else 1.0   # fp16 gradients need the loss scale the trainer's GradScaler applies
    (sums[0] * (0.7 * up) + sums[1] * (1.3 * up)).backward()
    # fp64 restatement
    anc, _ = make_anchors([f.float() for f in box], strides, 0.5)
    anc = anc.double()
    x = torch.cat([f.permute(0, 2, 3, 1).reshape(bs, -1, 64) for f in box], 1).double().requires_grad_(True)
    dist = x.view(bs, -1, 4, 16).softmax(3) @ torch.arange(16, dtype=torch.float64, device="cuda")
    pb = torch.cat((anc - dist[..., :2], anc + dist[..., 2:]), -1)
    w = tval.double()
    lbox = ((1.0 - hl._ciou(pb, tbox.double())) * w).sum()
    ltrb = torch.cat((anc - tbox.double()[..., :2], tbox.double()[..., 2:] - anc), -1).clamp(0, 16 - 1 - 0.01)
    tl = ltrb.long()
    wl = (tl + 1) - ltrb
    logp = F.log_softmax(x.view(bs, -1, 4, 16), -1)
    ce = -logp.gather(-1, tl.unsqueeze(-1)).squeeze(-1) * wl - logp.gather(-1, (tl + 1).unsqueeze(-1)).squeeze(-1) * (1 - wl)
    ldfl = (ce.mean(-1) * w).sum()
    (lbox * (0.7 * up) + ldfl * (1.3 * up)).backward()
    assert rel_err(sums[0], lbox) < 1e-5 and rel_err(sums[1], ldfl) < 1e-5, (sums.tolist(), float(lbox), float(ldfl))
    off = 0
    for m, (h, wd) in zip(maps, sizes):
        g = m.grad.permute(0, 2, 3, 1).reshape(bs, h * wd, 64)
        assert m.grad.is_contiguous(memory_format=torch.channels_last)
        assert rel_err(g, x.grad[:, off:off + h * wd]) < tol, rel_err(g, x.grad[:, off:off + h * wd])
        off += h * wd
    assert torch.equal(sums, Fb.box_dfl_sums([b for b in box], tbox, tval))


@pytest.mark.parametrize("dtype,tol", [(torch.bfloat16, 1e-2), (torch.float32, 1e-4)])
def test_whole_loss_on_kernels_equals_the_split_form(dtype, tol):
    """DetectionLoss with det_kernels (decode / assigner / box+DFL kernels) against the same loss with only the fused
    classification term (the path round 2 measured so far): three loss items and the gradient of every head map."""
    from improving_yolov8_cbam_swinblock_b200 import functional as Fb
    from improving_yolov8_cbam_swinblock_b200.harness import loss as hl, synthetic

    bs, nc, sizes, strides = 4, 80, [(80, 80), (40, 40), (20, 20)], [8.0, 16.0, 32.0]
    box, cls = _maps(bs, nc, sizes, dtype, 7)
    batch = {k: (v.cuda() if torch.is_tensor(v) else v) for k, v in synthetic.make_batch(bs, 640, nc, seed=3).items()}
    res = []
    for fused in (False, True):
        crit = hl.DetectionLoss(nc, strides)
        crit.cls_loss = Fb.cls_bce_sum
        crit.det_kernels = Fb.DetLossKernels if fused else None
        b = [t.clone().requires_grad_(True) for t in box]
        c = [t.clone().requires_grad_(True) for t in cls]
        loss, items = crit(list(zip(b, c)), batch, max_boxes=8)
        loss.sum().backward()
        res.append((items, [t.grad for t in b + c]))
    torch.testing.assert_close(res[1][0], res[0][0], rtol=2e-4, atol=1e-5)
    for g1, g0 in zip(res[1][1], res[0][1]):
        assert rel_err(g1, g0) < tol, rel_err(g1, g0)
