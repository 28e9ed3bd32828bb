"""-m gpu: the detection-loss kernels (csrc/det_assign.cu, csrc/det_loss.cu) against the restated reference (oracle/det_loss.py)
on the edge scenes of tests/det_scenes.py: the assigner bit for bit, decode, box / DFL sums and gradients, the whole loss, and
the classification term at saturated logits."""
import dataclasses

import pytest
import torch
import torch.nn.functional as F

import det_scenes as ds
from oracle import det_loss as od
from util import rel_err

pytestmark = pytest.mark.gpu

ALL = ds.cases()
LOSS = [c for c in ALL if c[0] != "tie"]
DEV = "cuda"


def _kernel_assign(s, topk):
    from improving_yolov8_cbam_swinblock_b200 import functional as Fb

    box, cls = s.maps(torch.float32, DEV)
    gt = s.gt(torch.float32, DEV)
    pred, scores = Fb.det_decode(box, cls, s.strides, gt)
    tlabel, tval, tbox = Fb.tal_assign(pred, scores, gt, s.sizes, s.strides, topk=topk)
    return gt, pred, scores, tlabel, tval, tbox


def _strides(s, dtype):
    _, st = od.make_anchors(s.box, s.strides)
    return st.to(device=DEV, dtype=dtype)


@pytest.mark.parametrize("name,topk", ALL)
def test_tal_assign_is_the_reference_assigner_bit_for_bit(name, topk):
    """Same decoded boxes and scores on both sides; the oracle in f32 with the stable top-k (ties: lower anchor index).
    The one accepted difference: the reference's top-k may pick zero-metric anchors inside a GT (fg with target value 0);
    the kernel leaves them as background."""
    s = ds.make(name)
    gt, pred, scores, tlabel, tval, tbox = _kernel_assign(s, topk)
    r = ds.run_oracle(s, topk=topk, stable=True, dtype=torch.float32, device=DEV, pred=pred,
                      scores=ds.scores_from_gathered(scores, gt, s.nc), gt=gt)
    s.check(s, r)   # the case is there on the kernel's own inputs too
    zero_fg = r.fg & (r.tval == 0)
    assert bool((tlabel[zero_fg] == -1).all()) and bool((tval[zero_fg] == 0).all())
    if name == "sparse":
        assert bool(zero_fg.any())
    keep = ~zero_fg
    assert torch.equal(tlabel.long()[keep], r.tlabel[keep]), f"{int((tlabel.long() != r.tlabel)[keep].sum())} labels differ"
    want_box = r.tbox / _strides(s, torch.float32)
    assert torch.equal(tbox[keep], want_box[keep])
    ulp = torch.nextafter(r.tval.abs(), torch.full_like(r.tval, float("inf"))) - r.tval.abs()
    assert bool(((tval - r.tval).abs() <= ulp)[keep].all()), float((tval - r.tval).abs()[keep].max())
    # run-to-run identical
    t2 = _kernel_assign(s, topk)
    assert torch.equal(t2[3], tlabel) and torch.equal(t2[4], tval) and torch.equal(t2[5], tbox)


@pytest.mark.parametrize("name,topk", ALL)
def test_tal_assign_against_the_reference_numerics(name, topk):
    """The reference as written (torch.topk) in fp64 on the kernel's decoded boxes / scores: every disagreement must be an
    fp64 near-tie (relative gap < 1e-5 at the k-th place of a GT containing the anchor)."""
    s = ds.make(name)
    gt, pred, scores, tlabel, tval, tbox = _kernel_assign(s, topk)
    r = ds.run_oracle(s, topk=topk, stable=False, dtype=torch.float64, device=DEV, pred=pred,
                      scores=ds.scores_from_gathered(scores.double(), gt, s.nc), gt=gt)
    want = torch.where(r.fg & (r.tval == 0), torch.full_like(r.tlabel, -1), r.tlabel)
    mism = tlabel.long() != want
    m = r.last["align_metric"]
    srt = m.sort(-1, descending=True).values
    kth, nxt = srt[..., topk - 1], srt[..., topk]
    near = (kth > 0) & ((kth - nxt) <= 1e-5 * kth)                       # [B, nmax]
    inside = r.last["mask_in_gts"] > 0                                    # [B, nmax, A]
    explained = (inside & near.unsqueeze(-1)).any(1)                      # [B, A]
    bad = mism & ~explained
    print(f"{name} topk={topk}: {int(mism.sum())} disagreements with the fp64 reference, all near-ties")
    assert not bool(bad.any()), f"{int(bad.sum())} disagreements are not fp64 near-ties"


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("name", ["edges", "tie", "saturated"])
def test_det_decode_edges(dtype, name):
    """Pair-peaked (integer edges) and uniform (7.5 bins) DFL logits decode exactly; saturated (+-30) class logits."""
    from improving_yolov8_cbam_swinblock_b200 import functional as Fb

    s = ds.make(name)
    box, cls = s.maps(dtype, DEV)
    gt = s.gt(torch.float32, DEV)
    pred, scores = Fb.det_decode(box, cls, s.strides, gt)
    r = dataclasses.replace(s, box=[b.double().cpu() for b in box], cls=[c.double().cpu() for c in cls])
    want = ds.decode(r, torch.float64, DEV)
    if name == "saturated":
        torch.testing.assert_close(pred.double(), want, rtol=1e-5, atol=1e-5)
    else:
        assert torch.equal(pred.double(), want), float((pred.double() - want).abs().max())
    lbl = gt[..., 0].long().clamp(0, s.nc - 1)
    x = torch.cat([c.double().reshape(s.bs, s.nc, -1) for c in cls], 2)          # [B, nc, A]
    want_sc = x.gather(1, lbl.unsqueeze(-1).expand(-1, -1, s.A)).sigmoid()     # [B, nmax, A]
    torch.testing.assert_close(scores.double(), want_sc, rtol=1e-6, atol=1e-7)


@pytest.mark.parametrize("dtype,tol", [(torch.bfloat16, 1e-2), (torch.float16, 2e-3), (torch.float32, 1e-5)])
def test_box_dfl_edges_match_reference_autograd(dtype, tol):
    """box_dfl_sums and its gradient against fp64 autograd through the oracle's BboxLoss + DFLoss on explicit targets: min / max
    ties (ATen's half split), target distances on integers and above 14.99, touching and disjoint boxes, fg with weight 0."""
    from improving_yolov8_cbam_swinblock_b200 import functional as Fb

    s = ds.make("edges")
    tb, w, fg, kind = ds.edge_targets(s)
    box, _ = s.maps(dtype, DEV)
    maps = [b.clone().requires_grad_(True) for b in box]
    sums = Fb.box_dfl_sums(maps, tb.float().to(DEV), w.float().to(DEV))
    up = 4096.0 if dtype == torch.float16 else 1.0
    (sums[0] * (0.7 * up) + sums[1] * (1.3 * up)).backward()
    # fp64 reference on the same (rounded) logits
    x = torch.cat([b.detach().double().reshape(s.bs, 64, -1) for b in box], 2).permute(0, 2, 1).contiguous().requires_grad_(True)
    crit = od.v8DetectionLoss(s.nc, s.strides, device=DEV)
    anc, _ = od.make_anchors([b.double() for b in box], s.strides)
    pb = crit.bbox_decode(anc, x)
    assert torch.equal(pb, pb.round())
    li, ld = od.BboxLoss(16)(x, pb, anc, tb.to(DEV), w.to(DEV).unsqueeze(-1), 1, fg.to(DEV))
    (li * (0.7 * up) + ld * (1.3 * up)).backward()
    assert rel_err(sums[0], li) < 1e-5 and rel_err(sums[1], ld) < 1e-5, (sums.tolist(), float(li), float(ld))
    got = torch.cat([m.grad.permute(0, 2, 3, 1).reshape(s.bs, -1, 64) for m in maps], 1).double()
    assert rel_err(got, x.grad) < tol, rel_err(got, x.grad)
    # identical boxes: ATen's half split on min / max ties makes the CIoU gradient vanish there (a full split would leave
    # h / union per edge); compared on the scale of the whole gradient, since the exact value is 0 up to rounding
    tie = (kind == 0).to(DEV)
    scale = float(x.grad.abs().max())
    assert float((got[tie] - x.grad[tie]).abs().max()) <= tol * scale, float((got[tie] - x.grad[tie]).abs().max())
    assert torch.equal(got[~fg.to(DEV)], torch.zeros_like(got[~fg.to(DEV)]))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("name,topk", LOSS)
def test_whole_loss_on_kernels_matches_reference(dtype, name, topk):
    """DetectionLoss on the decode / assigner / box+DFL / BCE kernels against the oracle's v8DetectionLoss in fp64 on the same
    (rounded) maps: three items and the gradients of all head maps.  The selection margins are asserted first, so the
    comparison is exact by construction."""
    from improving_yolov8_cbam_swinblock_b200 import functional as Fb
    from improving_yolov8_cbam_swinblock_b200.harness import loss as hl

    s = ds.make(name)
    box, cls = s.maps(dtype, DEV)
    r = dataclasses.replace(s, box=[b.double().cpu() for b in box], cls=[c.double().cpu() for c in cls])
    ds.assert_selection_margins(r, topk, device=DEV)
    crit = hl.DetectionLoss(s.nc, s.strides, topk=topk)
    crit.cls_loss = Fb.cls_bce_sum
    crit.det_kernels = Fb.DetLossKernels
    b = [t.clone().requires_grad_(True) for t in box]
    c = [t.clone().requires_grad_(True) for t in cls]
    loss, items = crit(list(zip(b, c)), s.batch(torch.float32, DEV), max_boxes=s.max_boxes())
    loss.sum().backward()
    witems, wgrads = ds.oracle_loss(r, topk, device=DEV)
    torch.testing.assert_close(items.double(), witems, rtol=1e-4, atol=1e-6)
    tol = 1e-4 if dtype == torch.float32 else 1e-2
    for t, wg in zip(b + c, wgrads):
        assert rel_err(t.grad, wg) < tol, rel_err(t.grad, wg)
    if name == "empty":
        assert float(items[0]) == 0 and float(items[2]) == 0


@pytest.mark.parametrize("nc", [8, 16, 80])
def test_bce_edges(nc):
    """Classification term in f32 at saturated logits (+-30, +-80), positive labels on lanes 0, 7, 8 and nc-1 of the 16-byte
    vectors, positive values 0 and 1."""
    from improving_yolov8_cbam_swinblock_b200 import functional as Fb

    bs, sizes = 2, [(4, 4), (2, 2)]
    g = torch.Generator().manual_seed(nc)
    A = sum(h * w for h, w in sizes)
    mags = torch.tensor([30.0, 80.0])
    maps = []
    for h, w in sizes:
        v = mags[torch.randint(0, 2, (bs, nc, h, w), generator=g)] * (torch.randint(0, 2, (bs, nc, h, w), generator=g) * 2 - 1)
        maps.append(v.to(DEV).contiguous(memory_format=torch.channels_last).requires_grad_(True))
    lanes = torch.tensor([q for q in (0, 7, 8, nc - 1) if q < nc])
    label = lanes[torch.arange(bs * A) % lanes.numel()].view(bs, A)
    label[:, ::5] = -1
    value = torch.rand(bs, A, generator=g)
    value[:, 1::4] = 0.0
    value[:, 2::4] = 1.0
    value = value * (label >= 0)
    got = Fb.cls_bce_sum(maps, label.to(DEV), value.to(DEV))
    (got * 0.37).backward()
    x = torch.cat([m.detach().permute(0, 2, 3, 1).reshape(bs, -1, nc) for m in maps], 1).double().requires_grad_(True)
    t = F.one_hot(label.clamp(min=0), nc).double().to(DEV) * value.double().to(DEV).unsqueeze(-1)
    want = F.binary_cross_entropy_with_logits(x, t, reduction="sum")
    (want * 0.37).backward()
    assert rel_err(got, want) < 1e-5, (float(got), float(want))
    gk = torch.cat([m.grad.permute(0, 2, 3, 1).reshape(bs, -1, nc) for m in maps], 1)
    torch.testing.assert_close(gk.double(), x.grad, rtol=1e-5, atol=1e-7)


def test_tal_assign_rejects_anchors_beyond_shared_memory():
    """1024^2 (21 504 anchors) runs (scene big1024 above); 1280^2 (33 600 anchors) is refused on the host with
    B200_ERR_UNSUPPORTED before any launch."""
    from improving_yolov8_cbam_swinblock_b200 import functional as Fb

    sizes, strides = [(160, 160), (80, 80), (40, 40)], [8.0, 16.0, 32.0]
    A = sum(h * w for h, w in sizes)
    assert A == 33600
    gt = torch.tensor([[[1.0, 100.0, 100.0, 300.0, 300.0]]], device=DEV)
    pred = torch.zeros(1, A, 4, device=DEV)
    scores = torch.zeros(1, 1, A, device=DEV)
    with pytest.raises(RuntimeError, match=r"code 6\).*33600 anchors do not fit in shared memory"):
        Fb.tal_assign(pred, scores, gt, sizes, strides)
    torch.cuda.synchronize()
