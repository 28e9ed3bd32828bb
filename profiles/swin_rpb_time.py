"""Cost of the learned relative-position bias (SwinBlockRPB) on the B200, in one process:

  1. tcgen05 window attention alone, forward and backward, with and without the bias, on the same qkv, at the model's P4
     SwinBlock [64,128,40,40] (2 heads, bf16) for ws 7 and ws 8;
  2. the expand kernel and, from a torch.profiler pass over the backward with bias, the split of that call into the
     workspace clear, the attention kernel and the two fold kernels;
  3. the whole block forward and backward, SwinBlock against SwinBlockRPB (autocast bf16);
  4. the whole-model training step (harness Trainer, CUDA-graph replay, batch 64 at 640), SwinBlock against SwinBlockRPB.

Kernel-level legs (1-3): every timed call is preceded by a 256 MB L2 flush and a ~1 ms spin kernel on the same stream, so the
start event is recorded while the GPU is busy and neither a warm L2 nor the host's launch latency is inside the event pair.
The two arms of each comparison alternate call by call; the median of ITERS calls is reported.  The card's name and power
limit are recorded with the numbers.

usage: python profiles/swin_rpb_time.py [--out swin_rpb.json] [--steps 30]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import improving_yolov8_cbam_swinblock_b200 as P  # noqa: E402
from improving_yolov8_cbam_swinblock_b200 import functional as Fb  # noqa: E402

dev = torch.device("cuda:0")
dt = torch.bfloat16
ITERS = 21
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)


def _one(fn, do_flush=True):
    if do_flush:
        flush.zero_()
    torch.cuda._sleep(2_000_000)
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    fn()
    e.record()
    e.synchronize()
    return s.elapsed_time(e) * 1e3   # us


def ab(fa, fb, iters=ITERS):
    """alternating A/B timing -> (median A us, median B us)."""
    for _ in range(3):
        fa(), fb()
    ta, tb = [], []
    for _ in range(iters):
        ta.append(_one(fa))
        tb.append(_one(fb))
    return sorted(ta)[iters // 2], sorted(tb)[iters // 2]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name(0)


def attn_legs(res):
    for ws in (7, 8):
        Hp = -(-40 // ws) * ws
        nW = Hp // ws
        L, C, nh = ws * ws, 128, 2
        T = 64 * nW * nW * L
        grid = (nW, nW, ws, 0)
        torch.manual_seed(ws)
        qkv = torch.randn(T, 3 * C, device=dev).to(dt)
        go = torch.randn(T, C, device=dev).to(dt)
        table = 0.02 * torch.randn((2 * ws - 1) ** 2, nh, device=dev)
        bias = Fb.rpb_expand(table, ws)
        o, lse = Fb.attn_forward(qkv, T, L, C, nh, grid)
        ob_, lseb = Fb.attn_forward(qkv, T, L, C, nh, grid, bias)
        f0, f1 = ab(lambda: Fb.attn_forward(qkv, T, L, C, nh, grid), lambda: Fb.attn_forward(qkv, T, L, C, nh, grid, bias))
        b0, b1 = ab(lambda: Fb.attn_backward(qkv, o, lse, go, T, L, C, nh, grid),
                    lambda: Fb.attn_backward(qkv, ob_, lseb, go, T, L, C, nh, grid, bias))
        ex = sorted(_one(lambda: Fb.rpb_expand(table, ws)) for _ in range(ITERS))[ITERS // 2]
        # split of the backward-with-bias call by kernel (separate, profiled pass; the profiler's own overhead is outside kernels)
        from torch.profiler import ProfilerActivity, profile

        for _ in range(2):
            Fb.attn_backward(qkv, ob_, lseb, go, T, L, C, nh, grid, bias)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(10):
                Fb.attn_backward(qkv, ob_, lseb, go, T, L, C, nh, grid, bias)
            torch.cuda.synchronize()
        split = {}
        for ev in prof.key_averages():
            if ev.device_type.name == "CUDA" or getattr(ev, "self_device_time_total", 0):
                name = ev.key
                for short in ("swin_attn_bwd_tc_kernel", "rpb_fold_slots_kernel", "rpb_fold_scatter_kernel", "Memset"):
                    if short in name:
                        us = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)
                        split[short] = round(us / max(ev.count, 1), 2)
        r = {"ws": ws, "tokens": T, "attn_fwd_us": round(f0, 2), "attn_fwd_rpb_us": round(f1, 2), "fwd_ratio": round(f1 / f0, 3),
             "attn_bwd_us": round(b0, 2), "attn_bwd_rpb_us": round(b1, 2), "bwd_ratio": round(b1 / b0, 3),
             "expand_us": round(ex, 2), "bwd_rpb_split_us": split}
        print(json.dumps(r), flush=True)
        res["attention"].append(r)


def block_legs(res):
    for ws in (7, 8):
        torch.manual_seed(0)
        a = P.SwinBlock(128, 2, ws).to(dev)
        b = P.SwinBlockRPB(128, 2, ws).to(dev)
        b.load_state_dict(a.state_dict(), strict=False)
        x = torch.randn(64, 128, 40, 40, device=dev).to(dt).contiguous(memory_format=torch.channels_last)
        g = torch.randn_like(x)

        def fwd(m):
            with torch.no_grad(), torch.autocast("cuda", dtype=dt):
                m(x)

        xs = {}

        def fwd_train(m):
            xi = x.detach().requires_grad_(True)
            with torch.autocast("cuda", dtype=dt):
                xs[id(m)] = (xi, m(xi))

        def bwd(m):
            xi, y = xs[id(m)]
            torch.autograd.grad(y, [xi] + list(m.parameters()), g, retain_graph=True)

        f0, f1 = ab(lambda: fwd(a), lambda: fwd(b))
        fwd_train(a), fwd_train(b)
        b0, b1 = ab(lambda: bwd(a), lambda: bwd(b))
        r = {"ws": ws, "shape": [64, 128, 40, 40], "block_fwd_us": round(f0, 2), "block_fwd_rpb_us": round(f1, 2),
             "block_bwd_us": round(b0, 2), "block_bwd_rpb_us": round(b1, 2)}
        print(json.dumps(r), flush=True)
        res["block"].append(r)
        del xs


def step_legs(res, steps):
    from improving_yolov8_cbam_swinblock_b200.harness import synthetic, train

    batch, imgsz = 64, 640
    arms = {"SwinBlock": P.BLOCKS, "SwinBlockRPB": {**P.BLOCKS, "SwinBlock": P.SwinBlockRPB}}
    trs = {}
    host = [synthetic.make_batch(batch, imgsz, 80, seed=1234 + 100 * i, pin=True) for i in range(2)]
    for name, blocks in arms.items():
        tr = train.Trainer(blocks, "n", 80, device="cuda:0", amp_dtype=dt, seed=0)
        tr.max_boxes = synthetic.BOXES_PER_IMAGE
        d = [tr.to_device(h) for h in host]
        for i in range(3):
            tr.step(d[i % 2])
        graphed = tr.enable_graph(d[0])
        for i in range(3):
            tr.step(d[i % 2])
        trs[name] = (tr, d, graphed)
    times = {k: [] for k in arms}
    for rep in range(5):   # alternating arms, `steps` graph-replayed steps each
        for name, (tr, d, _) in trs.items():
            torch.cuda.synchronize()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for i in range(steps):
                tr.step(d[i % 2])
            e.record()
            e.synchronize()
            times[name].append(s.elapsed_time(e) / steps)
    for name, (tr, d, graphed) in trs.items():
        ms = sorted(times[name])[2]
        r = {"arm": name, "graphed": bool(graphed), "batch": batch, "imgsz": imgsz, "step_ms": round(ms, 3),
             "img_per_s": round(batch / ms * 1e3, 1), "step_ms_all": [round(t, 3) for t in times[name]]}
        print(json.dumps(r), flush=True)
        res["train_step"].append(r)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="swin_rpb.json")
    ap.add_argument("--steps", type=int, default=30)
    args = ap.parse_args()
    res = {"card": card(), "method": "CUDA events, L2 flushed (256 MB) + 1 ms spin before each timed call, arms alternated, "
           f"median of {ITERS}; train step: median of 5 alternating windows of {args.steps} graph-replayed steps",
           "attention": [], "block": [], "train_step": []}
    print(res["card"], flush=True)
    attn_legs(res)
    block_legs(res)
    step_legs(res, args.steps)
    os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
    json.dump(res, open(args.out, "w"), indent=1)
    print("wrote", args.out)
