"""TEST INFRASTRUCTURE ONLY -- generate tests/golden/*.npz from the REAL reference modules.

Run in the dev container (where /root/reference exists):  ``python -m oracle.make_golden``.
The reference's own tests hold no vectors for CBAM / SwinBlock / SPPF (SURVEY D9), so these fixtures --
outputs and autograd gradients of the unmodified reference classes on seeded inputs -- are the parity pin
for ``oracle/blocks.py`` and, on the GPU box (where the reference is absent), for the CUDA kernels.
Each file is a flat npz: ``x``, ``gy`` (upstream grad), ``y``, ``gx``, ``w.<state_dict key>``, ``gw.<key>``.

``python -m oracle.make_golden model`` writes the model-level fixture ``tests/golden/model/detection_n_256.npz`` instead:
one fp32 training forward + loss + backward of YOLOv8n-CBAM-Swin (``SwinBlock [128]``) at batch 2, 256^2, nc=80 on the
seeded synthetic batch, with weights set by ``fill_seeded`` (a per-tensor rule keyed by the state_dict name, so any model
with the same state_dict keys gets the same weights).  It stores the three loss items, a fixed sample and the per-channel
means of the three prediction maps, a fixed sample of the flattened parameter gradients and every gradient's norm.  The
values come from the reference's ``DetectionModel`` + ``v8DetectionLoss`` when the reference is importable and from the
harness graph with the oracle blocks + the harness loss otherwise; ``source`` in the file says which.
"""
import math
import os
import sys
import zlib

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import ref_loader  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
MODEL_FIXTURE = os.path.join(OUT, "model", "detection_n_256.npz")
MODEL_BATCH, MODEL_IMGSZ, MODEL_NC, MODEL_DATA_SEED = 2, 256, 80, 5


@torch.no_grad()
def fill_seeded(model):
    """Every floating state_dict entry from its own generator seeded by crc32(name): running means N(0, 0.1^2), running
    variances U[0.5, 1.5], 1-D weights (norm affines) 1 + N(0, 0.1^2), biases N(0, 0.1^2), other weights U(+-1/sqrt(fan_in)).
    The Detect head's output biases are set as the reference's ``Detect.bias_init`` sets them (box 1.0, class
    log(5 / nc / (640 / stride)^2)), so the loss sits where training starts; the DFL projection (fixed arange, not trained)
    keeps its value."""
    detect = len(model.model) - 1
    for name, t in model.state_dict().items():
        if not t.dtype.is_floating_point or ".dfl." in name:
            continue
        g = torch.Generator().manual_seed(zlib.crc32(name.encode()))
        parts = name.split(".")
        if parts[:2] == ["model", str(detect)] and parts[2] in ("cv2", "cv3") and parts[4:] == ["2", "bias"]:
            v = torch.full(t.shape, 1.0 if parts[2] == "cv2" else math.log(5 / t.numel() / (640 / (8 * 2 ** int(parts[3]))) ** 2))
        elif name.endswith("running_mean") or name.endswith("bias"):
            v = 0.1 * torch.randn(t.shape, generator=g)
        elif name.endswith("running_var"):
            v = 0.5 + torch.rand(t.shape, generator=g)
        elif t.dim() == 1:
            v = 1 + 0.1 * torch.randn(t.shape, generator=g)
        else:
            v = (2 * torch.rand(t.shape, generator=g) - 1) / (t[0].numel() ** 0.5)
        t.copy_(v)


def model_step(model, loss_fn):
    """fp32 train-mode forward + loss + backward on the fixture's batch -> (prediction maps, loss items, {name: grad})."""
    from improving_yolov8_cbam_swinblock_b200.harness import synthetic

    batch = synthetic.make_batch(MODEL_BATCH, MODEL_IMGSZ, MODEL_NC, seed=MODEL_DATA_SEED)
    model.train()
    preds = model(batch["img"].float() / 255)
    loss, items = loss_fn(preds, batch)
    loss.sum().backward()
    grads = {k: p.grad.detach().clone() for k, p in model.named_parameters() if p.grad is not None}
    return [p.detach() for p in preds], items.detach(), grads


def _harness_model():
    from improving_yolov8_cbam_swinblock_b200.harness import graph, loss as hl
    from oracle import modules as om

    m = graph.DetectionGraph({"CBAM": om.CBAM, "SwinBlock": om.SwinBlock, "SPPF": om.make_sppf(graph.Conv)}, "n", MODEL_NC)
    return m, lambda preds, batch: hl.DetectionLoss(MODEL_NC, m.stride)(preds, batch, max_boxes=8)


def _reference_model():
    ref_loader.import_ultralytics()
    from ultralytics.cfg import get_cfg
    from ultralytics.nn.tasks import DetectionModel, yaml_model_load
    from ultralytics.utils.loss import v8DetectionLoss

    d = yaml_model_load(ref_loader.REF_ROOT + "/ultralytics/cfg/models/v8/yolov8n.yaml")
    d["backbone"][7][3] = [128]
    d["head"][3][3] = [128]
    m = DetectionModel(d, ch=3, nc=MODEL_NC, verbose=False)
    m.args = get_cfg()
    return m, lambda preds, batch: v8DetectionLoss(m)(preds, batch)


def model_fixture(samples=4096, grad_samples=16384):
    source = "reference" if ref_loader.available() else "harness"
    model, loss_fn = _reference_model() if source == "reference" else _harness_model()
    fill_seeded(model)
    preds, items, grads = model_step(model, loss_fn)
    g = torch.Generator().manual_seed(0)
    d = {"source": np.array(source), "items": items.numpy()}
    for i, p in enumerate(preds):
        idx = torch.randperm(p.numel(), generator=g)[:samples].sort().values
        d[f"map{i}_shape"] = np.array(p.shape)
        d[f"map{i}_idx"], d[f"map{i}_val"] = idx.numpy().astype(np.int32), p.reshape(-1)[idx].numpy()
        d[f"map{i}_chmean"] = p.mean((0, 2, 3)).numpy()
    flat = torch.cat([v.reshape(-1) for v in grads.values()])
    idx = torch.randperm(flat.numel(), generator=g)[:grad_samples].sort().values
    d["gnames"] = np.array(list(grads))
    d["g_idx"], d["g_val"] = idx.numpy().astype(np.int32), flat[idx].numpy()
    d["g_norm"] = np.array([float(v.norm()) for v in grads.values()], np.float32)
    d["gmax"] = np.array(float(flat.abs().max()), np.float32)
    os.makedirs(os.path.dirname(MODEL_FIXTURE), exist_ok=True)
    np.savez_compressed(MODEL_FIXTURE, **d)
    print(f"wrote {MODEL_FIXTURE} (source: {source}, {os.path.getsize(MODEL_FIXTURE) // 1024} KiB)")


def _run(mod, x, seed):
    g = torch.Generator().manual_seed(seed)
    x = x.clone().requires_grad_(True)
    y = mod(x)
    gy = torch.randn(y.shape, generator=g)
    y.backward(gy)
    d = {"x": x.detach().numpy(), "gy": gy.numpy(), "y": y.detach().numpy(), "gx": x.grad.numpy()}
    for k, v in mod.state_dict().items():
        d["w." + k] = v.numpy()
    for k, p in mod.named_parameters():
        if p.grad is not None:
            d["gw." + k] = p.grad.numpy()
    return d


def main():
    os.makedirs(OUT, exist_ok=True)
    ref_loader.import_ultralytics()
    from ultralytics.nn.modules.block import SPPF
    from ultralytics.nn.modules.cbam import CBAM, ChannelAttention, SpatialAttention
    from ultralytics.nn.modules.swin_block import SwinBlock

    # ---- CBAM: lazy (channels=None -> ratio 16), explicit small (ratio 8), odd spatial sizes
    for name, ctor, shape, seed in [
        ("cbam_lazy_c32", lambda: CBAM(), (2, 32, 9, 10), 11),
        ("cbam_c64_r8", lambda: CBAM(64), (2, 64, 5, 7), 12),
        ("cbam_lazy_c256_p5", lambda: CBAM(), (1, 256, 20, 20), 13),
    ]:
        torch.manual_seed(seed)
        m = ctor()
        x = torch.randn(shape)
        with torch.no_grad():
            m(x)  # lazy MLP creation happens inside forward (cbam.py:31-33)
        np.savez_compressed(os.path.join(OUT, name + ".npz"), **_run(m, x, seed + 100))
    # sub-modules return the maps only (cbam.py:38,53)
    torch.manual_seed(21)
    ca, sa = ChannelAttention(32, 16), SpatialAttention(3)
    x = torch.randn(2, 32, 6, 5)
    np.savez_compressed(os.path.join(OUT, "cbam_ca_c32.npz"), **_run(ca, x, 121))
    np.savez_compressed(os.path.join(OUT, "cbam_sa_k3.npz"), **_run(sa, x, 122))

    # ---- SwinBlock: padded (9x10 -> 14x14), exact multiple (14x7), ws=8/heads=4, single window smaller than ws
    for name, args, shape, seed in [
        ("swin_c16_pad", (16, 2, 7), (2, 16, 9, 10), 31),
        ("swin_c32_exact", (32, 2, 7), (1, 32, 14, 7), 32),
        ("swin_c32_ws8_h4", (32, 4, 8), (2, 32, 10, 17), 33),
        ("swin_c16_tiny", (16, 2, 7), (1, 16, 3, 4), 34),
        ("swin_c128_p4", (128, 2, 7), (1, 128, 20, 20), 35),
    ]:
        torch.manual_seed(seed)
        m = SwinBlock(*args)
        # non-trivial LN affine + biases so the padded-token (= norm1.bias) path is exercised (SURVEY D3)
        with torch.no_grad():
            for k, p in m.named_parameters():
                if "norm" in k or "bias" in k:
                    p.add_(0.3 * torch.randn_like(p))
        d = _run(m, torch.randn(shape), seed + 100)
        d["args"] = np.array(args)
        np.savez_compressed(os.path.join(OUT, name + ".npz"), **d)

    # ---- SPPF pool cascade with torch's indices (values + argmax are the bit-exact contract)
    for name, k, shape, mode, seed in [
        ("sppf_k5_rand", 5, (2, 8, 9, 11), "rand", 41),
        ("sppf_k7_rand", 7, (1, 8, 20, 20), "rand", 42),
        ("sppf_k5_ties", 5, (2, 4, 12, 7), "ties", 43),
        ("sppf_k7_const_nan", 7, (1, 4, 8, 8), "const_nan", 44),
        ("sppf_k5_small", 5, (1, 3, 2, 3), "rand", 45),
    ]:
        torch.manual_seed(seed)
        m = SPPF(shape[1] * 2, shape[1] * 2, k)
        y0 = torch.randn(shape)
        if mode == "ties":
            y0 = torch.relu(y0).bfloat16().float().round()  # heavy plateaus -> tie rule decides routing
        elif mode == "const_nan":
            y0 = torch.full(shape, 1.5)
            y0[0, 1, 3, 4] = float("nan")
            y0[0, 2] = float("-inf")
            y0[0, 3, 2, 2] = float("inf")
        ys, idx = [y0], []
        for _ in range(3):
            v, i = torch.nn.functional.max_pool2d(ys[-1], m.m.kernel_size, m.m.stride, m.m.padding,
                                                  return_indices=True)
            ys.append(v)
            idx.append(i)
        cat = torch.cat(ys, 1)
        d = {"y0": y0.numpy(), "cat": cat.numpy(), "idx": torch.stack(idx).numpy().astype(np.int32), "k": np.array(k)}
        if mode in ("rand", "ties"):
            g = torch.Generator().manual_seed(seed + 100)
            y0g = y0.clone().requires_grad_(True)
            yy = [y0g]
            yy.extend(m.m(yy[-1]) for _ in range(3))  # block.py:224-225
            gcat = torch.randn(cat.shape, generator=g)
            torch.cat(yy, 1).backward(gcat)
            d["gcat"], d["gy0"] = gcat.numpy(), y0g.grad.numpy()
        np.savez_compressed(os.path.join(OUT, name + ".npz"), **d)

    # ---- full SPPF module (cv1 -> pool cascade -> cv2), train-mode BN, k=5
    torch.manual_seed(51)
    m = SPPF(16, 16, 5).train()
    d = _run(m, torch.randn(2, 16, 6, 6), 151)
    np.savez_compressed(os.path.join(OUT, "sppf_module_k5.npz"), **d)
    # ---- the reference Conv block (conv -> BatchNorm2d -> SiLU, conv.py:37-79), train mode: pins the fused epilogue
    from ultralytics.nn.modules.conv import Conv

    for name, args, shape, seed in [("conv_k1_c16", (8, 16, 1, 1), (3, 8, 6, 5), 61), ("conv_k3_c32", (16, 32, 3, 2), (2, 16, 9, 9), 62)]:
        torch.manual_seed(seed)
        m = Conv(*args).train()
        with torch.no_grad():
            m.bn.weight.add_(0.3 * torch.randn_like(m.bn.weight))
            m.bn.bias.add_(0.3 * torch.randn_like(m.bn.bias))
        before = {k: v.clone() for k, v in m.state_dict().items()}
        x = torch.randn(shape)
        d = _run(m, x, seed + 100)
        for k, v in before.items():
            d["w0." + k] = v.numpy()       # state BEFORE the forward (running stats are updated by it)
        with torch.no_grad():
            d["conv_out"] = m.conv(x).numpy()
        d["bn_eps"], d["bn_momentum"] = np.array(m.bn.eps), np.array(m.bn.momentum)
        np.savez_compressed(os.path.join(OUT, name + ".npz"), **d)
    tot = sum(os.path.getsize(os.path.join(OUT, f)) for f in os.listdir(OUT))
    print("wrote", len(os.listdir(OUT)), "fixtures,", tot // 1024, "KiB")


if __name__ == "__main__":
    model_fixture() if sys.argv[1:] == ["model"] else main()
