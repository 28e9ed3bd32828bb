"""CPU: the harness' caller-side graph and loss compute the same function as the reference's DetectionModel +
v8DetectionLoss on identical weights, against the stored fixture ``tests/golden/model/detection_n_256.npz``
(``python -m oracle.make_golden model``).  The committed fixture has ``source = "harness"``: the harness produced it where the
reference was absent, so for the loss it shows only that the harness still computes what it computed then.  What pins the loss
to the reference's function is tests/test_det_loss_oracle.py (oracle/det_loss.py).  The plugin tests below drive the reference package itself and run only where it
is importable (``oracle/_ref``, made by ``oracle/build_ref.py``); the repository does not ship it."""
import os

import numpy as np
import pytest
import torch

from oracle import make_golden as mg
from oracle import ref_loader
from util import GOLDEN

needs_reference = pytest.mark.skipif(not ref_loader.available(),
                                     reason="imports classes of the reference Ultralytics package, which the repository does not ship")


def test_graph_and_loss_match_reference():
    g = np.load(os.path.join(GOLDEN, "model", "detection_n_256.npz"))
    mine, loss_fn = mg._harness_model()
    mg.fill_seeded(mine)
    preds, items, grads = mg.model_step(mine, loss_fn)
    for i, p in enumerate(preds):
        assert list(p.shape) == g[f"map{i}_shape"].tolist()
        got = p.reshape(-1)[torch.from_numpy(g[f"map{i}_idx"]).long()]
        torch.testing.assert_close(got, torch.from_numpy(g[f"map{i}_val"]), rtol=1e-4, atol=1e-4)
        torch.testing.assert_close(p.mean((0, 2, 3)), torch.from_numpy(g[f"map{i}_chmean"]), rtol=1e-4, atol=1e-4)
    torch.testing.assert_close(items, torch.from_numpy(g["items"]), rtol=1e-4, atol=1e-5)
    assert list(grads) == g["gnames"].tolist()
    tol = 1e-4 * float(g["gmax"])
    flat = torch.cat([v.reshape(-1) for v in grads.values()])
    err = (flat[torch.from_numpy(g["g_idx"]).long()] - torch.from_numpy(g["g_val"])).abs()
    assert float(err.max()) < tol, f"sampled gradients: {float(err.max()):.3e} >= {tol:.3e}"
    for (k, v), n in zip(grads.items(), g["g_norm"]):
        assert abs(float(v.norm()) - float(n)) <= tol * v.numel() ** 0.5, k


@needs_reference
def test_plugin_rebinds_reference_namespaces():
    import improving_yolov8_cbam_swinblock_b200.ultralytics_plugin as plugin

    ref_loader.import_ultralytics()
    from ultralytics.nn import tasks
    from ultralytics.nn.tasks import DetectionModel, yaml_model_load

    table = plugin.install()
    try:
        assert tasks.CBAM is table["CBAM"] and tasks.SwinBlock is table["SwinBlock"] and tasks.SPPF is table["SPPF"]
        d = yaml_model_load(ref_loader.REF_ROOT + "/ultralytics/cfg/models/v8/yolov8s.yaml")  # the yaml as shipped
        m = DetectionModel(d, ch=3, nc=1, verbose=False)  # CPU stride pass runs through our shape probes
        assert type(m.model[7]) is table["SwinBlock"] and type(m.model[10]) is table["CBAM"]
        assert type(m.model[11]) is table["SPPF"] and m.model[12].k == 7
        assert sum(p.numel() for p in m.parameters()) == 13405269  # SURVEY D4 probe
        m.fuse()  # SPPF.cv1/cv2 are the reference's Conv: BN folded
        assert not hasattr(m.model[11].cv1, "bn")
    finally:
        plugin.uninstall()
    assert tasks.CBAM is not table["CBAM"]


@needs_reference
def test_plugin_seams_patch_is_value_neutral_and_reversible():
    import torch

    import improving_yolov8_cbam_swinblock_b200.ultralytics_plugin as plugin

    ref_loader.import_ultralytics()
    from ultralytics.nn.modules.block import C2f
    from ultralytics.nn.modules.conv import Concat

    torch.manual_seed(0)
    blk = C2f(16, 16, n=2, shortcut=True).eval()
    x = torch.randn(2, 16, 8, 8)
    ref = blk(x)
    ref_cat = Concat(1)([x, x * 2])
    orig = C2f.forward
    plugin.install(seams=True)
    try:
        assert C2f.forward is not orig
        assert torch.equal(blk(x), ref)                      # CPU tensors: the stock ops behind the same call sites
        assert torch.equal(Concat(1)([x, x * 2]), ref_cat)
        assert torch.equal(Concat(2)([x, x]), torch.cat([x, x], 2))
    finally:
        plugin.uninstall()
    assert C2f.forward is orig


@needs_reference
def test_reference_pickles_unpickle_as_plugin_classes_with_reference_state_only():
    """ADVICE r1: SPPF.forward / SwinBlock.forward must not read attributes the reference classes never store (k,
    num_heads): a module pickled by the reference and loaded after install() has run no __init__ of ours."""
    import pickle

    import improving_yolov8_cbam_swinblock_b200.ultralytics_plugin as plugin

    ref_loader.import_ultralytics()
    from ultralytics.nn.modules.block import SPPF as RSPPF
    from ultralytics.nn.modules.swin_block import SwinBlock as RSwin

    blobs = [pickle.dumps(RSwin(32, 2, 7)), pickle.dumps(RSPPF(32, 32, 7))]
    table = plugin.install()
    try:
        ms, mp_ = (pickle.loads(b) for b in blobs)
        assert type(ms) is table["SwinBlock"] and type(mp_) is table["SPPF"]
        assert ms.attn.num_heads == 2 and ms.window_size == 7 and mp_.m.kernel_size == 7
        x = torch.zeros(1, 32, 9, 9)   # shape probe path
        assert ms(x).shape == x.shape and mp_(x).shape == x.shape
    finally:
        plugin.uninstall()
