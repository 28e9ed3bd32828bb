"""-m gpu: the whole custom YOLOv8-CBAM-Swin graph with the B200 blocks vs the same graph with the oracle blocks
(identical weights, identical synthetic batch): logits, the three loss components and every parameter gradient."""
import copy

import pytest
import torch

from util import rel_err

pytestmark = pytest.mark.gpu


def _build(blocks, scale, nc, seed):
    from improving_yolov8_cbam_swinblock_b200.harness import graph

    torch.manual_seed(seed)
    return graph.DetectionGraph(blocks, scale, nc)


@pytest.mark.parametrize("scale", ["n", "s"])
def test_whole_model_fp32_vs_oracle_blocks(scale):
    import improving_yolov8_cbam_swinblock_b200 as P
    from improving_yolov8_cbam_swinblock_b200.harness import graph, loss as hl, synthetic
    from oracle import modules as om

    torch.backends.cudnn.allow_tf32 = False  # stock convs would otherwise run TF32 and drown the comparison
    torch.backends.cuda.matmul.allow_tf32 = False
    ob = {"CBAM": om.CBAM, "SwinBlock": om.SwinBlock, "SPPF": om.make_sppf(graph.Conv)}
    ref = _build(ob, scale, 80, 1)
    mine = _build(P.BLOCKS, scale, 80, 2)
    assert list(ref.state_dict().keys()) == list(mine.state_dict().keys())
    mine.load_state_dict(ref.state_dict())
    ref, mine = ref.cuda().train(), mine.cuda().train()
    batch = synthetic.make_batch(4, 320, 80, seed=7)
    dev_batch = {k: v.cuda() for k, v in batch.items()}
    img = dev_batch["img"].float() / 255
    crit = hl.DetectionLoss(80, ref.stride)
    fr, fm = ref(img), mine(img.contiguous(memory_format=torch.channels_last))
    for a, b in zip(fm, fr):
        assert rel_err(a, b) < 1e-4
    lr, ir = crit(fr, dev_batch, max_boxes=8)
    lm, im = crit(fm, dev_batch, max_boxes=8)
    torch.testing.assert_close(im, ir, rtol=1e-4, atol=1e-5)
    lr.sum().backward()
    lm.sum().backward()
    gr, gm = dict(ref.named_parameters()), dict(mine.named_parameters())
    gmax = max(float(p.grad.abs().max()) for p in gr.values() if p.grad is not None)
    for k, p in gr.items():
        if p.grad is None:
            assert gm[k].grad is None
            continue
        err = float((gm[k].grad - p.grad).abs().max())
        assert err <= 2e-4 * gmax, f"{k}: {err:.3e} (gmax {gmax:.3e})"


def test_module_protocols_on_gpu():
    """deepcopy / pickle / half / DDP-wrap behaviours the trainer relies on (SURVEY section 8b)."""
    import io

    import improving_yolov8_cbam_swinblock_b200 as P
    from improving_yolov8_cbam_swinblock_b200.harness import graph

    m = _build(P.BLOCKS, "n", 3, 0).cuda().eval()
    x = torch.rand(1, 3, 64, 64, device="cuda")
    y = m(x)[0]
    m2 = copy.deepcopy(m)
    buf = io.BytesIO()
    torch.save(m, buf)
    buf.seek(0)
    m3 = torch.load(buf, weights_only=False)
    assert torch.equal(m2(x)[0], y) and torch.equal(m3(x)[0], y)
    yh = m2.half()(x.half())[0]
    assert yh.dtype == torch.float16 and rel_err(yh, y) < 5e-2


@pytest.mark.parametrize("scale", ["s", "m"])
def test_scaled_variants_train_step_bf16(scale):
    """BASELINE configs[3]: the s / m width-depth variants (SwinBlock [256] / [384]; m has head dim 192, served by the
    SIMT attention kernels) take a finite bf16 training step with the B200 blocks and the fused Conv epilogue."""
    import improving_yolov8_cbam_swinblock_b200 as P
    from improving_yolov8_cbam_swinblock_b200.harness import synthetic, train

    tr = train.Trainer(P.BLOCKS, scale, 80, device="cuda:0", amp_dtype=torch.bfloat16)
    tr.max_boxes = synthetic.BOXES_PER_IMAGE
    batch = tr.to_device(synthetic.make_batch(2, 320, 80, seed=5))
    before = [p.detach().clone() for p in tr.raw.parameters()]
    items = tr.step(batch)
    assert torch.isfinite(items).all()
    moved = sum(int(not torch.equal(a, b)) for a, b in zip(before, tr.raw.parameters()))
    assert moved > 0.9 * len(before)


@pytest.mark.parametrize("from_host", [False, True])
def test_graph_replayed_step_equals_eager_step(from_host):
    """The headline number comes from ``Trainer.enable_graph`` (CUDA-graph replay of fwd+loss+bwd+clip+SGD) and, for e2e,
    ``step_from_host`` with the next batch prefetched on a copy stream: both must produce the eager step's numbers.
    Two trainers from identical init see the same 5 batches; ``enable_graph`` itself takes 3 real warm-up steps on its
    capture batch, so the eager trainer takes the same 3 first."""
    import improving_yolov8_cbam_swinblock_b200 as P
    from improving_yolov8_cbam_swinblock_b200.harness import synthetic, train

    torch.backends.cudnn.deterministic = True
    try:
        trs = [train.Trainer(P.BLOCKS, "n", 80, device="cuda:0", amp_dtype=torch.bfloat16, seed=3) for _ in range(2)]
        for t in trs:
            t.max_boxes = synthetic.BOXES_PER_IMAGE
        graphed, eager = trs
        for a, b in zip(graphed.raw.state_dict().values(), eager.raw.state_dict().values()):
            assert torch.equal(a, b)
        host = [synthetic.make_batch(4, 256, 80, seed=20 + i, pin=True) for i in range(5)]
        cap = graphed.to_device(host[0])
        assert graphed.enable_graph(cap), graphed._graph_error
        for _ in range(3):   # what enable_graph's warm-up did to the other trainer
            eager._fwd_bwd(cap)
            eager._exchange()
            eager._update()
        for i in range(5):
            if from_host:
                lg = graphed.step_from_host(host[i], host[(i + 1) % 5])
                le = eager.step_from_host(host[i])
            else:
                lg = graphed.step(graphed.to_device(host[i])).cpu()
                le = eager.step(eager.to_device(host[i])).cpu()
            torch.testing.assert_close(lg, le, rtol=2e-3, atol=1e-4, msg=f"step {i}: loss items {lg} vs {le}")
        worst = 0.0
        for (k, a), b in zip(graphed.raw.state_dict().items(), eager.raw.state_dict().values()):
            if a.dtype.is_floating_point:
                worst = max(worst, rel_err(a, b) if float(b.abs().max()) > 0 else float(a.abs().max()))
        assert worst < 2e-3, f"parameters after 5 replayed steps differ from the eager ones: {worst:.2e}"
        for a, b in zip(graphed.ema.shadow, eager.ema.shadow):
            assert rel_err(a, b) < 2e-3 or float(b.abs().max()) == 0
    finally:
        torch.backends.cudnn.deterministic = False


def test_whole_model_bf16_vs_oracle_blocks():
    """bf16 autocast (the benchmarked configuration): the graph with the B200 blocks against the same graph with the
    oracle blocks evaluated in fp32 -- logits and loss items within the bf16 bar.  Whole-network bf16 back-propagation
    through 27 randomly initialised layers amplifies rounding noise whatever implements the blocks, so the parameter
    gradients are held to the yardstick the reference itself would meet: the error of the oracle-block graph under the
    SAME bf16 autocast (stock PyTorch kernels) against its own fp32 run."""
    import improving_yolov8_cbam_swinblock_b200 as P
    from improving_yolov8_cbam_swinblock_b200.harness import graph, loss as hl, synthetic
    from oracle import modules as om

    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    ob = {"CBAM": om.CBAM, "SwinBlock": om.SwinBlock, "SPPF": om.make_sppf(graph.Conv)}
    ref = _build(ob, "n", 80, 1)
    mine = _build(P.BLOCKS, "n", 80, 2)
    mine.load_state_dict(ref.state_dict())
    ref, mine = ref.cuda().train(), mine.cuda().train().to(memory_format=torch.channels_last)
    ref16 = copy.deepcopy(ref)
    batch = synthetic.make_batch(8, 320, 80, seed=9)
    dev_batch = {k: v.cuda() for k, v in batch.items()}
    img = dev_batch["img"].float() / 255
    crit = hl.DetectionLoss(80, ref.stride)
    fr = ref(img)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        fm = mine(img.contiguous(memory_format=torch.channels_last))
        f16 = ref16(img)
    for a, b, c in zip(fm, fr, f16):
        assert rel_err(a, b) < max(3e-2, 1.5 * rel_err(c, b)), (rel_err(a, b), rel_err(c, b))
    lr, ir = crit(fr, dev_batch, max_boxes=8)
    lm, im = crit(fm, dev_batch, max_boxes=8)
    l16, _ = crit(f16, dev_batch, max_boxes=8)
    torch.testing.assert_close(im, ir, rtol=3e-2, atol=1e-3)
    lr.sum().backward()
    lm.sum().backward()
    l16.sum().backward()
    gr, gm, g16 = dict(ref.named_parameters()), dict(mine.named_parameters()), dict(ref16.named_parameters())
    bad, num, num16, den = [], 0.0, 0.0, 0.0
    for k, p in gr.items():
        if p.grad is None:
            continue
        e, e16 = rel_err(gm[k].grad, p.grad), rel_err(g16[k].grad, p.grad)
        num += float((gm[k].grad.double() - p.grad.double()).pow(2).sum())
        num16 += float((g16[k].grad.double() - p.grad.double()).pow(2).sum())
        den += float(p.grad.double().pow(2).sum())
        if e > 3.0 * e16 + 2e-2:   # single parameters (e.g. the 98-element CBAM conv: a cancelling sum over B*H*W) are noisy in both
            bad.append((k, round(e, 4), round(e16, 4)))
    assert not bad, bad
    # all gradients together: the B200-block graph is as close to the fp32 truth as the stock bf16 graph is
    assert (num / den) ** 0.5 <= 1.25 * (num16 / den) ** 0.5 + 1e-2, ((num / den) ** 0.5, (num16 / den) ** 0.5)


def test_weight_leaves_step_is_bit_identical_to_leafless_trainer():
    """The Trainer hands every stock convolution a 16-bit leaf copy of its weight (one multi-tensor refresh per step, one
    multi-tensor copy of the gradients back) instead of autocast's per-layer cast kernels: same values, so three steps must
    leave bit-identical parameters and loss items (cuDNN deterministic, same algorithms for the same shapes).  The
    reference trainer has its leaves taken away, so its convolutions go through autocast's casts."""
    import improving_yolov8_cbam_swinblock_b200 as P
    from improving_yolov8_cbam_swinblock_b200.harness import synthetic, train

    torch.backends.cudnn.deterministic = True
    try:
        a = train.Trainer(P.BLOCKS, "n", 80, device="cuda:0", amp_dtype=torch.bfloat16, seed=5)
        b = train.Trainer(P.BLOCKS, "n", 80, device="cuda:0", amp_dtype=torch.bfloat16, seed=5)
        for m, *_ in b._w16:
            m.w16 = None
        b._w16 = []
        assert len(a._w16) > 30 and not b._w16
        for t in (a, b):
            t.max_boxes = synthetic.BOXES_PER_IMAGE
        for i in range(3):
            batch = synthetic.make_batch(4, 256, 80, seed=40 + i)
            la = a.step(a.to_device(batch))
            lb = b.step(b.to_device(batch))
            assert torch.equal(la, lb), f"step {i}: {la} vs {lb}"
        for (k, va), vb in zip(a.raw.state_dict().items(), b.raw.state_dict().values()):
            assert torch.equal(va, vb), k
    finally:
        torch.backends.cudnn.deterministic = False
