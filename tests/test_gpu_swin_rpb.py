"""-m gpu: SwinBlockRPB (Swin's learned relative-position bias) on the tcgen05 and SIMT attention kernels, against the fp64
oracle (tests/swin_rpb_oracle.py: oracle/blocks.swin_forward plus the bias, whose index is built the way Swin's code builds it),
against each other, and
inside the whole training step.  Bars as tests/test_gpu_swin.py: f32 1e-5, bf16 2e-2, f16 4e-3 relative error."""
import pytest
import torch

from swin_rpb_oracle import swin_rpb_forward
from util import rel_err, to_cl

pytestmark = pytest.mark.gpu

TOL = {torch.float32: 1e-5, torch.bfloat16: 2e-2, torch.float16: 4e-3}


def _block(C, heads, ws, shift, seed, table_scale=3.0, sign=False):
    import improving_yolov8_cbam_swinblock_b200.modules as M

    torch.manual_seed(seed)
    blk = M.SwinBlockRPB(C, heads, ws, shift)
    with torch.no_grad():
        for k, p in blk.named_parameters():
            if "norm" in k or k.endswith("bias"):
                p.add_(0.2 * torch.randn_like(p))
        blk.attn.out_proj.weight.mul_(4.0)   # a larger attention share of y, so that the bias visibly moves the output
        t = torch.randn_like(blk.relative_position_bias_table)
        blk.relative_position_bias_table.copy_(table_scale * (torch.sign(t) if sign else t))
    return blk


def _check_vs_oracle(shape, heads, ws, shift, dtype, seed, table_scale=3.0, sign=False):
    from oracle import blocks as ob

    tol = TOL[dtype]
    blk = _block(shape[1], heads, ws, shift, seed, table_scale, sign)
    x = torch.randn(shape).to(dtype)
    gy = torch.randn(shape).to(dtype)
    po = {k: v.detach().double().requires_grad_(True) for k, v in blk.named_parameters()}
    table = po.pop("relative_position_bias_table")
    xo = x.double().requires_grad_(True)
    yo = swin_rpb_forward(xo, po, heads, ws, shift, table)
    yo.backward(gy.double())
    with torch.no_grad():   # the bias is large enough for the comparison to see it
        y_nob = ob.swin_forward(x.double(), po, heads, ws, shift)
    assert rel_err(y_nob, yo) >= 10 * tol, rel_err(y_nob, yo)
    blk = blk.cuda()
    xc = to_cl(x.cuda()).requires_grad_(True)
    with torch.autocast("cuda", dtype=dtype, enabled=dtype != torch.float32):
        y = blk(xc)
    y.backward(to_cl(gy.cuda()))
    assert torch.isfinite(y).all() and torch.isfinite(xc.grad).all()
    assert rel_err(y.float(), yo) <= tol, f"y {rel_err(y.float(), yo):.2e}"
    assert rel_err(xc.grad.float(), xo.grad) <= tol, f"gx {rel_err(xc.grad.float(), xo.grad):.2e}"
    for k, p in blk.named_parameters():
        want = table.grad if k == "relative_position_bias_table" else po[k].grad
        e = rel_err(p.grad.float(), want)
        assert e <= max(tol, 1e-4), f"grad {k}: {e:.2e}"


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16, torch.float32])
@pytest.mark.parametrize("cfg", [((2, 128, 40, 40), 2, 7, 0), ((1, 256, 20, 20), 2, 7, 0), ((2, 64, 16, 24), 2, 8, 0),
                                 ((1, 384, 14, 14), 2, 7, 0), ((2, 128, 23, 9), 4, 7, 0),     # test_vs_oracle's five
                                 ((1, 128, 17, 12), 2, 7, 0),                                   # padded map
                                 ((2, 128, 5, 4), 2, 7, 0),                                     # smaller than one window
                                 ((2, 128, 21, 21), 2, 7, 3), ((1, 64, 24, 16), 1, 8, 4)])      # shifted windows
def test_vs_oracle(dtype, cfg):
    shape, heads, ws, shift = cfg
    _check_vs_oracle(shape, heads, ws, shift, dtype, seed=sum(shape) + ws + shift)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("shift", [0, 3])
def test_large_table_entries_stay_finite_and_match(dtype, shift):
    """+-30 entries: near one-hot softmax rows; the max subtraction keeps exp finite on both paths."""
    _check_vs_oracle((1, 128, 14, 14), 2, 7, shift, dtype, seed=7 + shift, table_scale=30.0, sign=True)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("nwin,nWh,ws,C,nh,shift", [(72, 8, 7, 128, 2, 3), (36, 1, 7, 256, 2, 0), (12, 1, 7, 384, 2, 0),
                                                    (48, 6, 8, 128, 2, 4), (301, 1, 7, 128, 2, 0)])
def test_tc_matches_simt_with_bias(dtype, nwin, nWh, ws, C, nh, shift):
    """tcgen05 attention with bias vs the fp32 SIMT kernel with bias on the same (rounded) qkv: o, lse, gqkv, gtable."""
    from improving_yolov8_cbam_swinblock_b200 import functional as Fb

    torch.manual_seed(nwin + ws + C)
    L = ws * ws
    grid = (nWh, nwin // nWh, ws, shift)
    T = nwin * L
    qkv = torch.randn(T, 3 * C, device="cuda").to(dtype)
    go = torch.randn(T, C, device="cuda").to(dtype)
    table = torch.randn((2 * ws - 1) ** 2, nh, device="cuda")
    bias = Fb.rpb_expand(table, ws)
    try:
        Fb.USE_TC_ATTENTION = False
        o_ref, lse_ref = Fb.attn_forward(qkv.float(), T, L, C, nh, grid, bias)
        g_ref, gt_ref = Fb.attn_backward(qkv.float(), o_ref, lse_ref, go.float(), T, L, C, nh, grid, bias)
    finally:
        Fb.USE_TC_ATTENTION = True
    assert lib_tc(T, L, C, nh, dtype)
    o, lse = Fb.attn_forward(qkv, T, L, C, nh, grid, bias)
    g, gt = Fb.attn_backward(qkv, o, lse, go, T, L, C, nh, grid, bias)
    bf = dtype == torch.bfloat16
    assert rel_err(o, o_ref) < (1e-2 if bf else 2e-3), rel_err(o, o_ref)
    torch.testing.assert_close(lse, lse_ref, rtol=1e-3, atol=2e-3)
    assert rel_err(g, g_ref) < (1.5e-2 if bf else 3e-3), rel_err(g, g_ref)
    assert rel_err(gt, gt_ref) < (1.5e-2 if bf else 3e-3), rel_err(gt, gt_ref)


def lib_tc(T, L, C, nh, dtype):
    from improving_yolov8_cbam_swinblock_b200 import _lib

    return bool(_lib.lib().b200_swin_attn_tc_supported(T, L, C, nh, _lib.dtype_code(dtype)))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("shift", [0, 3])
def test_zero_table_equals_swinblock_bit_for_bit(dtype, shift, monkeypatch):
    """A zero table adds +0 to every score: the block is SwinBlock's stage-by-stage path, forward and every shared gradient."""
    import improving_yolov8_cbam_swinblock_b200.modules as M
    from improving_yolov8_cbam_swinblock_b200 import functional as Fb

    monkeypatch.setattr(Fb, "USE_FUSED_ATTN", False)
    torch.manual_seed(11)
    rpb = M.SwinBlockRPB(128, 2, 7, shift).cuda()
    with torch.no_grad():
        rpb.relative_position_bias_table.zero_()
    ref = M.SwinBlock(128, 2, 7, shift).cuda()
    ref.load_state_dict(rpb.state_dict(), strict=False)
    x = torch.randn(2, 128, 20, 19, device="cuda").to(dtype)
    g = torch.randn(2, 128, 20, 19, device="cuda").to(dtype)
    out = []
    for m in (rpb, ref):
        xi = to_cl(x).requires_grad_(True)
        with torch.autocast("cuda", dtype=dtype, enabled=dtype != torch.float32):
            y = m(xi)
        y.backward(to_cl(g))
        out.append((y.detach(), xi.grad, {k: p.grad for k, p in m.named_parameters()}))
    (y0, gx0, gp0), (y1, gx1, gp1) = out
    assert torch.equal(y0, y1) and torch.equal(gx0, gx1)
    for k in gp1:
        assert torch.equal(gp0[k], gp1[k]), k
    assert gp0["relative_position_bias_table"].abs().sum() > 0


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_backward_is_deterministic(dtype):
    blk = _block(128, 2, 7, 3, seed=5).cuda()
    x = to_cl(torch.randn(4, 128, 28, 28, device="cuda").to(dtype))
    g = to_cl(torch.randn(4, 128, 28, 28, device="cuda").to(dtype))
    runs = []
    for _ in range(2):
        blk.zero_grad(set_to_none=True)
        xi = x.clone().requires_grad_(True)
        with torch.autocast("cuda", dtype=dtype, enabled=dtype != torch.float32):
            y = blk(xi)
        y.backward(g)
        runs.append((xi.grad.clone(), {k: p.grad.clone() for k, p in blk.named_parameters()}))
    assert torch.equal(runs[0][0], runs[1][0])
    for k in runs[0][1]:
        assert torch.equal(runs[0][1][k], runs[1][1][k]), k


def test_full_size_bf16_vs_oracle_on_gpu():
    """[64,128,40,40], ws 7, bf16 against the oracle evaluated in fp32 on the same GPU: output, input and every gradient."""
    torch.backends.cuda.matmul.allow_tf32 = False
    blk = _block(128, 2, 7, 0, seed=0).cuda()
    x = torch.randn(64, 128, 40, 40, device="cuda").to(torch.bfloat16)
    g = torch.randn(64, 128, 40, 40, device="cuda").to(torch.bfloat16)
    po = {k: v.detach().float().requires_grad_(True) for k, v in blk.named_parameters()}
    table = po.pop("relative_position_bias_table")
    xo = x.float().requires_grad_(True)
    yo = swin_rpb_forward(xo, po, 2, 7, 0, table)
    yo.backward(g.float())
    xi = to_cl(x).requires_grad_(True)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        y = blk(xi)
    y.backward(to_cl(g))
    assert rel_err(y, yo) < 2e-2 and rel_err(xi.grad, xo.grad) < 2e-2, (rel_err(y, yo), rel_err(xi.grad, xo.grad))
    for k, p in blk.named_parameters():
        want = table.grad if k == "relative_position_bias_table" else po[k].grad
        assert rel_err(p.grad, want) < 2e-2, (k, rel_err(p.grad, want))


def test_bias_bypasses_the_fused_attention_half(monkeypatch):
    """With a table the attention half runs stage by stage; the fused MLP half is still used."""
    from improving_yolov8_cbam_swinblock_b200 import functional as Fb

    names = []
    real_call, real_block = Fb.call, Fb.swin_attn_block_forward_raw

    def spy_call(name, *a, **k):
        names.append(name)
        return real_call(name, *a, **k)

    def spy_block(*a, **k):
        names.append("swin_attn_block_forward_raw")
        return real_block(*a, **k)

    monkeypatch.setattr(Fb, "call", spy_call)
    monkeypatch.setattr(Fb, "swin_attn_block_forward_raw", spy_block)
    blk = _block(128, 2, 7, 0, seed=3).cuda()
    x = to_cl(torch.randn(2, 128, 40, 40, device="cuda")).requires_grad_(True)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        y = blk(x)
    y.float().sum().backward()
    assert "swin_attn_block_forward_raw" not in names and "b200_swin_attn_block_fwd" not in names
    assert "b200_swin_mlp_fwd" in names and "b200_swin_mlp_bwd" in names
    assert "b200_swin_attn_fwd_tc_rpb" in names and "b200_swin_attn_bwd_tc_rpb" in names
    assert "b200_swin_rpb_expand" in names
    # the same module without a table takes the fused attention half (the switch this test relies on is live)
    import improving_yolov8_cbam_swinblock_b200.modules as M

    names.clear()
    ref = M.SwinBlock(128, 2, 7).cuda()
    with torch.autocast("cuda", dtype=torch.bfloat16):
        ref(x)
    assert "swin_attn_block_forward_raw" in names


def test_whole_model_graph_replay_with_bias():
    """Trainer on the fork's model with SwinBlockRPB (bf16): the CUDA graph captures, the replayed step equals the eager step
    over 5 steps (protocol and tolerances of test_graph_replayed_step_equals_eager_step), both tables learn."""
    import improving_yolov8_cbam_swinblock_b200 as P
    from improving_yolov8_cbam_swinblock_b200.harness import synthetic, train

    blocks = {**P.BLOCKS, "SwinBlock": P.SwinBlockRPB}
    torch.backends.cudnn.deterministic = True
    try:
        trs = [train.Trainer(blocks, "n", 80, device="cuda:0", amp_dtype=torch.bfloat16, seed=3) for _ in range(2)]
        for t in trs:
            t.max_boxes = synthetic.BOXES_PER_IMAGE
        graphed, eager = trs
        for a, b in zip(graphed.raw.state_dict().values(), eager.raw.state_dict().values()):
            assert torch.equal(a, b)
        tables = [m.relative_position_bias_table for m in eager.raw.modules() if isinstance(m, P.SwinBlockRPB)]
        assert len(tables) == 2
        before = [t.detach().clone() for t in tables]
        host = [synthetic.make_batch(4, 256, 80, seed=20 + i, pin=True) for i in range(5)]
        cap = graphed.to_device(host[0])
        assert graphed.enable_graph(cap), graphed._graph_error
        assert graphed._graph_error is None
        for k in range(3):   # what enable_graph's warm-up did to the other trainer
            eager._fwd_bwd(cap)
            if k == 0:
                for t in tables:
                    assert t.grad is not None and float(t.grad.abs().sum()) > 0
            eager._exchange()
            eager._update()
        for t, b in zip(tables, before):
            assert not torch.equal(t.detach(), b)
        for i in range(5):
            lg = graphed.step(graphed.to_device(host[i])).cpu()
            le = eager.step(eager.to_device(host[i])).cpu()
            torch.testing.assert_close(lg, le, rtol=2e-3, atol=1e-4, msg=f"step {i}: loss items {lg} vs {le}")
        worst = 0.0
        for (k, a), b in zip(graphed.raw.state_dict().items(), eager.raw.state_dict().values()):
            if a.dtype.is_floating_point:
                worst = max(worst, rel_err(a, b) if float(b.abs().max()) > 0 else float(a.abs().max()))
        assert worst < 2e-3, f"parameters after 5 replayed steps differ from the eager ones: {worst:.2e}"
    finally:
        torch.backends.cudnn.deterministic = False
