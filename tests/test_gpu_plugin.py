"""-m gpu: the drop-in claim on a GPU.  ``ultralytics_plugin.install()`` rebinds CBAM / SwinBlock / SPPF (and, optionally,
Conv's epilogue and the C2f / Concat seams) in the UNMODIFIED reference package (``oracle/_ref``: the verbatim copy made by
``oracle/build_ref.py`` -- ``/root/reference`` does not exist on the GPU box), ``parse_model`` (``nn/tasks.py:1438,1503-1506``)
builds the real ``DetectionModel`` from the yaml dict, and its own ``_predict_once`` / ``v8DetectionLoss`` run on CUDA through
the B200 kernels."""
import io
import pickle

import pytest
import torch

from oracle import ref_loader, ref_step
from util import rel_err

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not ref_loader.available(),
                                                  reason="drives the reference Ultralytics package, which the repository does not ship")]


@pytest.fixture()
def plugin():
    import improving_yolov8_cbam_swinblock_b200.ultralytics_plugin as plugin

    ref_loader.import_ultralytics()
    yield plugin
    plugin.uninstall()


def test_real_detection_model_trains_one_step_through_the_plugin(plugin):
    """fp32 (tight bars): the plugged real model == the harness graph with the same blocks and weights -- logits, the three
    loss items from the reference's own v8DetectionLoss vs the harness loss, and every parameter gradient."""
    import improving_yolov8_cbam_swinblock_b200 as P
    from improving_yolov8_cbam_swinblock_b200.harness import graph, loss as hl, synthetic

    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    table = plugin.install(conv_epilogue=True, seams=True)
    torch.manual_seed(0)
    ref = ref_step.build_model("n", 80)
    assert type(ref.model[7]) is table["SwinBlock"] and type(ref.model[10]) is table["CBAM"] and type(ref.model[11]) is table["SPPF"]
    assert type(ref.model[0]) is plugin.Conv
    mine = graph.DetectionGraph(P.BLOCKS, "n", 80)
    assert list(ref.state_dict()) == list(mine.state_dict())
    mine.load_state_dict(ref.state_dict())
    ref = ref.cuda().train().to(memory_format=torch.channels_last)
    mine = mine.cuda().train().to(memory_format=torch.channels_last)
    batch = {k: v.cuda() for k, v in synthetic.make_batch(4, 320, 80, seed=7).items()}
    img = (batch["img"].float() / 255).contiguous(memory_format=torch.channels_last)
    from improving_yolov8_cbam_swinblock_b200 import _lib

    n0 = _lib.launch_count()
    loss_r, items_r = ref(dict(batch, img=img))              # BaseModel.forward(dict) -> _predict_once -> v8DetectionLoss
    assert _lib.launch_count() - n0 >= 60, "the real model's forward did not go through libb200yolo.so"
    fm = mine(img)
    loss_m, items_m = hl.DetectionLoss(80, mine.stride)(fm, batch, max_boxes=8)
    torch.testing.assert_close(items_m, items_r, rtol=1e-4, atol=1e-5)
    loss_r.sum().backward()
    loss_m.sum().backward()
    gr, gm = dict(ref.named_parameters()), dict(mine.named_parameters())
    gmax = max(float(p.grad.abs().max()) for p in gr.values() if p.grad is not None)
    for k, p in gr.items():
        if p.grad is None:
            assert gm[k].grad is None, k
            continue
        err = float((gm[k].grad - p.grad).abs().max())
        assert err <= 2e-4 * gmax, f"{k}: {err:.3e} (gmax {gmax:.3e})"


def test_real_trainer_step_bf16_autocast_through_the_plugin(plugin):
    """The reference's trainer-style step (oracle/ref_step.py) with the plugin installed: bf16 autocast, finite loss,
    parameters move, EMA updates -- 'drops into the existing trainer unchanged'."""
    from improving_yolov8_cbam_swinblock_b200.harness import synthetic

    plugin.install(conv_epilogue=True, seams=True)
    tr = ref_step.RefTrainer("n", 80, "cuda:0", amp="bf16", channels_last=True)
    before = [p.detach().clone() for p in tr.model.parameters()]
    batch = tr.to_device(synthetic.make_batch(4, 320, 80, seed=3))
    items = [tr.step(batch) for _ in range(2)][-1]
    assert torch.isfinite(items).all()
    moved = sum(int(not torch.equal(a, b)) for a, b in zip(before, tr.model.parameters()))
    assert moved > 0.9 * len(before)


def test_reference_pickles_load_under_the_plugin_and_run_on_cuda(plugin):
    """Whole-module checkpoints pickled by the REFERENCE classes (trainer.py:537-554, loaded at tasks.py:1222) unpickle as
    the B200 classes once the plugin is installed -- without their __init__ having run, so forward may only rely on state the
    reference also stores (window_size, attn.num_heads, m.kernel_size)."""
    from ultralytics.nn.modules.block import SPPF as RSPPF
    from ultralytics.nn.modules.swin_block import SwinBlock as RSwin

    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.manual_seed(0)
    rs, rp = RSwin(64, 2, 7).eval(), RSPPF(64, 64, 7).eval()
    x = torch.randn(2, 64, 20, 20)
    with torch.no_grad():
        want_s, want_p = rs(x), rp(x)
    blobs = [pickle.dumps(rs), pickle.dumps(rp)]
    buf = io.BytesIO()
    torch.save(rs, buf)
    table = plugin.install()
    ms, mp_ = (pickle.loads(b) for b in blobs)
    assert type(ms) is table["SwinBlock"] and type(mp_) is table["SPPF"]
    assert not hasattr(ms, "num_heads") and not hasattr(mp_, "k")       # the reference never stored them
    with torch.no_grad():
        got_s, got_p = ms.cuda()(x.cuda()), mp_.cuda()(x.cuda())
    assert rel_err(got_s.cpu(), want_s) < 1e-5 and rel_err(got_p.cpu(), want_p) < 1e-5
    buf.seek(0)
    m3 = torch.load(buf, weights_only=False)
    assert type(m3) is table["SwinBlock"]
