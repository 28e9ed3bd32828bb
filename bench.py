#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric: training images/s of the custom YOLOv8n-CBAM-Swin model at 640^2,
batch 64 per GPU, data-parallel (DDP / NCCL gradient all-reduce) on synthetic COCO-shaped batches, bf16 autocast,
plus the per-module roofline numbers of the hand-written kernels.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

Prints ONE JSON line on rank 0.  Keys beyond the base contract: ``e2e`` (same metric through the user-facing
``Trainer.step_from_host``: pinned host batch in, host loss out), ``roofline`` (dominant hand-written kernel, timed
with CUDA events on the launching stream inside the timed region), ``modules`` (per-kernel % of roofline, standalone,
L2 flushed between launches), ``cpu_baseline`` (the oracle port of the reference blocks inside the same graph on the
host cores, bounded sample), ``clocks``, ``gpu_launches``.

``--impl reference`` times the reference's own CPU implementation of the path: the UNMODIFIED ``DetectionModel`` +
``v8DetectionLoss`` from ``oracle/_ref`` (a verbatim copy of the reference package made by ``oracle/build_ref.py``; it is
pure Python, so this is what "compiling the reference" means here) for exactly K timed + W warm-up steps, fp32, all host
threads, at the largest per-step batch that fits the time budget -- and prints the batch / steps / dtype it really ran.
``gpu_eager_baseline`` (own arm, N=1) = the same unmodified reference run eagerly on the GPU: the bar to beat.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", ""):
    os.environ["NCCL_DEBUG"] = "WARN"  # keep NCCL's version banner off stdout: rank 0 prints exactly one JSON line

SCALE, NC, IMGSZ, PER_GPU_BATCH = "n", 80, 640, 64


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"], "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.proc, self.idx = None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def _cpu_info():
    model = "unknown"
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                model = ln.split(":", 1)[1].strip()
                break
    except OSError:
        pass
    return {"nproc": os.cpu_count() or 1, "cpu_model": model}


def _median_ms(fn, warm, reps):
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(1e3 * (time.perf_counter() - t0))
    return statistics.median(ts)


DUMP_MAX_ELEMS = 1 << 22   # per dumped array: 16 MB of float32 at any --scale


def dump_outputs(out_dir, loss_items, state_dict):
    """--dump-outputs: what the timed training step hands its caller after its last step, as float32 .npy files --
    ``loss_items`` [box, cls, dfl] and ``model_state``, every floating state_dict entry of the trained model flattened in
    logical (NCHW) order and concatenated in state_dict order; above DUMP_MAX_ELEMS a fixed seeded sample of it.  Two
    builds run with the same arguments see the same inputs, so their dumps compare output for output."""
    import numpy as np
    import torch

    flat = torch.cat([v.detach().float().reshape(-1).cpu() for v in state_dict.values() if v.dtype.is_floating_point])
    if flat.numel() > DUMP_MAX_ELEMS:
        flat = flat[torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_MAX_ELEMS].sort().values]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "loss_items.npy"), loss_items.detach().float().cpu().numpy())
    np.save(os.path.join(out_dir, "model_state.npy"), flat.numpy())


def _ref_kind():
    """'reference' when the unmodified reference package is importable (oracle/_ref, made by oracle/build_ref.py, or
    /root/reference in the dev container); 'port' (oracle/modules.py in the harness graph) otherwise."""
    from oracle import ref_step

    return "reference" if ref_step.available() else "port"


def _make_cpu_trainer(kind):
    import torch

    if kind == "reference":
        from oracle import ref_step

        tr = ref_step.RefTrainer(SCALE, NC, "cpu", amp=None, ema=True)
        return tr, tr.step, tr.model
    from improving_yolov8_cbam_swinblock_b200.harness import graph, synthetic, train
    from oracle import modules as om

    blocks = {"CBAM": om.CBAM, "SwinBlock": om.SwinBlock, "SPPF": om.make_sppf(graph.Conv)}
    tr = train.Trainer(blocks, SCALE, NC, device="cpu", amp_dtype=None, ema=True)
    tr.max_boxes = synthetic.BOXES_PER_IMAGE
    return tr, tr.step, tr.raw


def cpu_reference_run(steps, warmup, batch=None, budget_s=150.0, dump_dir=None):
    """The reference's own CPU implementation of the measured path -- the UNMODIFIED ``DetectionModel`` +
    ``v8DetectionLoss`` + trainer-style SGD/EMA step (oracle/ref_step.py over oracle/_ref), fp32, all host threads --
    for exactly ``warmup`` + ``steps`` steps.  ``batch=None``: the largest per-step batch in {64,32,16,8,4,2} whose
    (warmup+steps) steps fit ``budget_s`` according to one probe step at batch 4.  ``dump_dir``: see dump_outputs()."""
    import torch

    from improving_yolov8_cbam_swinblock_b200.harness import synthetic

    kind = _ref_kind()
    cores = os.cpu_count() or 1
    try:   # all host cores, whatever mask the launcher left on this process
        os.sched_setaffinity(0, range(cores))
    except (AttributeError, OSError):
        pass
    torch.set_num_threads(cores)
    tr, step, model = _make_cpu_trainer(kind)
    if batch is None:
        probe = synthetic.make_batch(4, IMGSZ, NC, seed=99)
        step(probe)
        t0 = time.perf_counter()
        step(probe)
        per_img = (time.perf_counter() - t0) / 4
        batch = 2
        for b in (64, 32, 16, 8, 4):
            if per_img * b * (steps + warmup) <= budget_s:
                batch = b
                break
    host = synthetic.make_batch(batch, IMGSZ, NC, seed=1234)
    for _ in range(warmup):
        step(host)
    t0 = time.perf_counter()
    for _ in range(steps):
        items = step(host)
    dt = time.perf_counter() - t0
    if dump_dir:
        dump_outputs(dump_dir, items, model.state_dict())
    what = ("unmodified reference DetectionModel + v8DetectionLoss (oracle/_ref = verbatim copy of the reference package), trainer-style "
            "step (oracle/ref_step.py)") if kind == "reference" else "oracle/modules.py blocks in the harness graph (reference package not available)"
    return {"value": batch * steps / dt, "unit": "img/s", "cores": cores, "kind": kind, "batch": batch, "steps": steps, "warmup": warmup,
            "ms_per_step": 1e3 * dt / steps, **_cpu_info(),
            "sample": f"{steps} timed (+{warmup} warm-up) fp32 training steps (fwd + v8 loss + bwd + clip + SGD + EMA) of YOLOv8{SCALE}-CBAM-Swin "
                      f"at {IMGSZ}^2, batch {batch}, {cores} torch threads: {what}"}


def cpu_baseline_leg(train_steps=3, train_batch=8, sweep_reps=10, sweep_batch=8):
    """BASELINE.md section 4 items 1-3 on the box's host cores (bounded: ~30-40 s):
    (1) configs[0]: fp32 inference, batch 1, eval + inference_mode, 3 warm-up + 10 timed, median -- at all cores and at the
        reference's default of ONE thread (ultralytics/__init__.py:8-9 sets OMP_NUM_THREADS=1);
    (2) training step at batch ``train_batch`` (all cores; one step at 1 thread);
    (3) module sweep: reference CBAM / SPPF / SwinBlock modules, fwd and fwd+bwd, ``sweep_reps`` reps, median."""
    import torch

    from improving_yolov8_cbam_swinblock_b200.harness import synthetic

    kind = _ref_kind()
    cores = os.cpu_count() or 1
    try:   # a launcher / communicator may have narrowed this process's CPU mask: the leg is defined on ALL host cores
        os.sched_setaffinity(0, range(cores))
    except (AttributeError, OSError):
        pass
    torch.set_num_threads(cores)
    tr, step, model = _make_cpu_trainer(kind)
    host = synthetic.make_batch(train_batch, IMGSZ, NC, seed=1234)
    step(host)
    t0 = time.perf_counter()
    for _ in range(train_steps):
        step(host)
    dt = time.perf_counter() - t0
    out = {"value": train_batch * train_steps / dt, "unit": "img/s", "cores": cores, "kind": kind, **_cpu_info(),
           "sample": f"{train_steps} fp32 training steps (fwd + v8 loss + bwd + clip + SGD + EMA) of YOLOv8{SCALE}-CBAM-Swin at {IMGSZ}^2, "
                     f"batch {train_batch}, {cores} threads, " + ("unmodified reference (oracle/_ref)" if kind == "reference" else "oracle port")}
    torch.set_num_threads(1)
    small = synthetic.make_batch(2, IMGSZ, NC, seed=1)
    t0 = time.perf_counter()
    step(small)
    out["train_1thread_img_s"] = round(2 / (time.perf_counter() - t0), 3)
    # (1) configs[0]
    model.eval()
    img1 = host["img"][:1].float() / 255
    with torch.inference_mode():
        out["inference_b1_fp32_ms_1thread"] = round(_median_ms(lambda: model(img1), 1, 3), 2)
        torch.set_num_threads(cores)
        out["inference_b1_fp32_ms"] = round(_median_ms(lambda: model(img1), 3, 10), 2)
    model.train()
    out["inference_note"] = ("configs[0]: batch 1, 640^2, fp32, eval + inference_mode, median; all cores: 3 warm-up + 10 timed; "
                             "1 thread (the reference's OMP_NUM_THREADS default): 1 warm-up + 3 timed")
    # (3) module sweep on the reference's own module classes
    sweep = []
    try:
        if kind == "reference":
            from oracle import ref_loader

            ref_loader.import_ultralytics()
            from ultralytics.nn.modules.block import SPPF as RSPPF
            from ultralytics.nn.modules.cbam import CBAM as RCBAM
            from ultralytics.nn.modules.swin_block import SwinBlock as RSwin
        else:
            from improving_yolov8_cbam_swinblock_b200.harness import graph
            from oracle import modules as om

            RCBAM, RSwin, RSPPF = om.CBAM, om.SwinBlock, om.make_sppf(graph.Conv)
        from improving_yolov8_cbam_swinblock_b200.harness.sweep import CHANNELS

        c3, c4, c5 = CHANNELS[SCALE]
        B = sweep_batch
        cases = [("CBAM", lambda: RCBAM(), (B, c5, 20, 20)), ("CBAM", lambda: RCBAM(), (B, c4, 40, 40)),
                 ("CBAM", lambda: RCBAM(), (B, c3, 80, 80)),
                 ("SPPF_k5", lambda: RSPPF(c5, c5, 5), (B, c5, 20, 20)), ("SPPF_k7", lambda: RSPPF(c5, c5, 7), (B, c5, 20, 20)),
                 ("SwinBlock_ws7", lambda: RSwin(c4, 2, 7), (B, c4, 40, 40)), ("SwinBlock_ws8", lambda: RSwin(c4, 2, 8), (B, c4, 40, 40))]
        for name, mk, shape in cases:
            torch.manual_seed(0)
            mod = mk().train()
            x = torch.randn(shape)
            with torch.no_grad():
                mod(x)   # lazy CBAM MLP
                fwd = _median_ms(lambda: mod(x), 2, sweep_reps)
            xg = x.clone().requires_grad_(True)

            def fb():
                y = mod(xg)
                y.backward(torch.ones_like(y))

            sweep.append({"module": name, "shape": list(shape), "fwd_ms": round(fwd, 3), "fwd_bwd_ms": round(_median_ms(fb, 2, sweep_reps), 3)})
    except Exception as e:  # noqa: BLE001  the sweep is a reported extra: never lose the bench line over it
        sweep.append({"error": f"{type(e).__name__}: {e}"})
    out["module_sweep"] = {"threads": cores, "reps": sweep_reps, "dtype": "f32", "rows": sweep,
                           "note": f"reference module classes on the host cores, batch {sweep_batch} (bounded sample), median of {sweep_reps}"}
    return out


def cpu_baseline_bounded(timeout_s=150):
    """cpu_baseline_leg() in a FRESH interpreter with a hard time limit: what rank 0 runs at world_size > 1.  Under torchrun the
    parent carries OMP_NUM_THREADS=1, a live NCCL communicator and its helper threads; the 2-GPU run of round 2 showed the
    in-process leg taking > 5 min there (40 s stand-alone), and the bench line is only printed after it.  The child sees no GPU,
    none of the launcher's thread / rendezvous variables, and is killed at the limit -- the record then says so."""
    drop = ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "RANK", "LOCAL_RANK", "WORLD_SIZE", "LOCAL_WORLD_SIZE", "GROUP_RANK", "ROLE_RANK",
            "MASTER_ADDR", "MASTER_PORT", "TORCHELASTIC_RUN_ID", "TORCHELASTIC_RESTART_COUNT", "TORCHELASTIC_MAX_RESTARTS")
    env = {k: v for k, v in os.environ.items() if k not in drop}
    env["CUDA_VISIBLE_DEVICES"] = ""
    root = os.path.dirname(os.path.abspath(__file__))
    code = (f"import json, sys; sys.path.insert(0, {root!r}); import bench; bench.SCALE = {SCALE!r}; "
            "print('CPU_BASELINE_JSON ' + json.dumps(bench.cpu_baseline_leg()))")
    try:
        r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=timeout_s, env=env, cwd=root)
    except subprocess.TimeoutExpired:
        return {"skipped": f"the host-core leg exceeded its {timeout_s} s limit in a child process on this box (measured at N=1: see that line)"}
    for ln in r.stdout.splitlines():
        if ln.startswith("CPU_BASELINE_JSON "):
            out = json.loads(ln[len("CPU_BASELINE_JSON "):])
            out["ran_in"] = "child process (no GPU, launcher thread variables cleared)"
            return out
    return {"skipped": f"child process failed (rc {r.returncode}): {(r.stderr or r.stdout)[-300:]}"}


def gpu_eager_baseline_leg(steps, warmup, batch, device):
    """The honest bar (BASELINE.md section 4 item 4): the reference ships no CUDA, so "the reference on a B200" is its
    unmodified modules through cuDNN / cuBLAS / ATen eager.  Same synthetic batches, same step (oracle/ref_step.py), bf16
    autocast and the trainer's native fp16 + GradScaler (trainer.py:274-276,383)."""
    import torch

    from improving_yolov8_cbam_swinblock_b200.harness import synthetic
    from oracle import ref_step

    if not ref_step.available():
        return {"unavailable": "oracle/_ref (copy of the reference package, oracle/build_ref.py) not present"}
    out = {"unit": "img/s", "batch": batch, "steps": steps, "warmup": warmup,
           "what": "unmodified reference DetectionModel + v8DetectionLoss + SGD + ModelEMA, PyTorch eager on the same GPU, device-resident uint8 batches"}
    host = [synthetic.make_batch(batch, IMGSZ, NC, seed=1234 + 100 * i) for i in range(2)]
    for amp in ("bf16", "fp16"):
        try:
            tr = ref_step.RefTrainer(SCALE, NC, device, amp=amp, ema=True)
            dev = [tr.to_device(h) for h in host]
            for i in range(warmup):
                tr.step(dev[i % 2])
            torch.cuda.synchronize()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for i in range(steps):
                tr.step(dev[i % 2])
            e.record()
            torch.cuda.synchronize()
            ms = s.elapsed_time(e) / steps
            out[amp] = {"value": batch / (ms * 1e-3), "ms_per_step": ms}
            del tr, dev
            torch.cuda.empty_cache()
        except Exception as ex:  # noqa: BLE001
            out[amp] = {"error": f"{type(ex).__name__}: {ex}"}
            torch.cuda.empty_cache()
    return out


_record_out = None


def _claim_stdout():
    """stdout carries exactly ONE line (the JSON record): libraries that write to fd 1 (NCCL prints its version banner there
    when the first communicator is created) are sent to stderr; the record goes to a private copy of the real stdout."""
    global _record_out
    sys.stdout.flush()
    _record_out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def print_record(line):
    _record_out.write(json.dumps(line) + "\n")
    _record_out.flush()


def _at_least_one(s):
    n = int(s)
    if n < 1:
        raise argparse.ArgumentTypeError(f"{n}: at least one timed step")
    return n


def main():
    _claim_stdout()
    if os.environ.get("B200_BENCH_WATCHDOG"):  # debugging aid: dump every thread's stack and exit if the run stalls
        import faulthandler

        faulthandler.dump_traceback_later(int(os.environ["B200_BENCH_WATCHDOG"]), exit=True)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=_at_least_one, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=PER_GPU_BATCH, help="per-GPU batch (default = BASELINE config)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-eager", action="store_true", help="skip the reference-eager-on-this-GPU leg")
    ap.add_argument("--ref-batch", type=int, default=None, help="--impl reference: per-step batch (default: largest that fits the time budget)")
    ap.add_argument("--no-sweep", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch every step eagerly (no CUDA-graph replay)")
    ap.add_argument("--cudnn-benchmark", type=int, default=0, help="torch.backends.cudnn.benchmark for the stock convolutions (A/B switch)")
    ap.add_argument("--scale", default=SCALE, choices=["n", "s", "m"],
                    help="width/depth variant (BASELINE configs[3]: s/m with SwinBlock [256]/[384]); default n = the headline config")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last timed step's loss items and the trained model state as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference" and args.ref_batch is None:
        ap.error("--dump-outputs with --impl reference needs --ref-batch: the default batch is picked from a timed probe step")
    globals()["SCALE"] = args.scale
    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    swin_dim = {"n": 128, "s": 256, "m": 384}[SCALE]
    config = {"workload": f"configs[{2 if SCALE == 'n' else 3}]: YOLOv8{SCALE}-CBAM-Swin (yolov8.yaml:734-776, SwinBlock [{swin_dim}]) training fwd+bwd+SGD+EMA, "
                          f"synthetic COCO-shaped batches {IMGSZ}x{IMGSZ}, nc={NC}, 8 boxes/img",
              "per_gpu_batch": args.batch, "global_batch": args.batch * world, "parallelism": f"dp{world}",
              "amp": "bf16 autocast", "memory_format": "channels_last",
              "l2": "each step touches >1 GB of activations (> 126 MB L2); module sweep flushes L2 between launches"}

    if args.impl == "reference":
        if rank != 0:
            return
        cb = cpu_reference_run(args.steps, args.warmup, batch=args.ref_batch, dump_dir=args.dump_outputs)
        rconfig = dict(config)   # what this arm actually ran: CPU, fp32, its own per-step batch
        rconfig.update(per_gpu_batch=cb["batch"], global_batch=cb["batch"], parallelism="cpu", amp="none (fp32)", memory_format="contiguous (NCHW)",
                       l2="n/a (host cores)", device=f"host CPU, {cb['cores']} threads", sample_of_workload=cb["batch"] != args.batch,
                       steps_run=cb["steps"], warmup_run=cb["warmup"])
        line = {"impl": "reference", "metric": "train_images_per_sec", "value": cb["value"], "unit": "img/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": cb["ms_per_step"], "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": rconfig,
                "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "nproc", "cpu_model", "batch")},
                "e2e": {"value": cb["value"], "unit": "img/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print_record(line)
        return

    import torch
    import torch.distributed as dist

    import improving_yolov8_cbam_swinblock_b200 as P
    from improving_yolov8_cbam_swinblock_b200 import _lib
    from improving_yolov8_cbam_swinblock_b200.harness import sweep, synthetic, train

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the B200 kernels have no CPU path)")
    torch.cuda.set_device(local_rank)
    torch.backends.cudnn.benchmark = bool(args.cudnn_benchmark)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    _lib.lib()  # fail loudly here if libb200yolo.so is missing
    tr = train.Trainer(P.BLOCKS, SCALE, NC, device=f"cuda:{local_rank}", amp_dtype=torch.bfloat16, world_size=world,
                       local_rank=local_rank, channels_last=True)
    tr.max_boxes = synthetic.BOXES_PER_IMAGE
    host = [synthetic.make_batch(args.batch, IMGSZ, NC, seed=1234 + rank + 100 * i, pin=True) for i in range(2)]
    dev = [tr.to_device(h) for h in host]
    h2d = synthetic.batch_nbytes(host[0])

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local_rank])
        torch.cuda.synchronize()

    def timed(fn, steps, collective=True):
        """collective=False: rank-local leg (run by rank 0 alone after the other ranks left): no barrier / all-reduce."""
        barrier() if collective else torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for i in range(steps):
            fn(i)
        e.record()
        barrier() if collective else torch.cuda.synchronize()
        ms = torch.tensor([s.elapsed_time(e)], device=f"cuda:{local_rank}")
        if world > 1 and collective:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)  # max over ranks
        return float(ms.item())

    for i in range(args.warmup):
        tr.step(dev[i % 2])
    # per-kernel roofline leg: the same K steps launched eagerly with CUDA events around every C-ABI call (events cannot
    # be recorded inside a replayed graph); the headline legs below replay the step as a CUDA graph when capture works
    _lib.enable_timing(True)
    ms_eager = timed(lambda i: tr.step(dev[i % 2]), args.steps)
    ktimes = _lib.timing_summary()
    _lib.enable_timing(False)
    graphed = (not args.no_graph) and tr.enable_graph(dev[0])
    for i in range(args.warmup):
        tr.step(dev[i % 2])
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = _lib.launch_count()
    last = {}

    def dev_step(i):
        last["items"] = tr.step(dev[i % 2])

    ms_dev = timed(dev_step, args.steps)
    launches = _lib.launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:   # before the e2e leg below trains the model further
        dump_outputs(args.dump_outputs, last["items"], tr.raw.state_dict())
    for i in range(2):
        tr.step_from_host(host[i % 2], host[(i + 1) % 2])

    def e2e_step(i):
        # the next pinned batch is handed over like a data loader would: its H2D copy overlaps this step's compute
        last["loss"] = tr.step_from_host(host[i % 2], host[(i + 1) % 2])

    ms_e2e = timed(e2e_step, args.steps)
    imgs = args.batch * world * args.steps
    kernels_per_step = sum(n for n, _ in ktimes.values()) / max(args.steps, 1) if ktimes else 0   # C-ABI calls per step
    config["launch_mode"] = (("CUDA-graph replay of fwd+loss+bwd+clip+SGD" if world == 1 else
                              "CUDA-graph replay: graph A fwd+loss+bwd into one flat gradient buffer, one eager NCCL all-reduce, graph B clip+SGD") +
                             " (captured once; gpu_launches = C-ABI kernel calls replayed inside the graph)") if graphed else f"eager launches ({tr._graph_error or 'graph capture disabled'})"
    if graphed and world > 1:
        config["launch_mode"] += f"; multi-GPU capture: {tr._graph_mode}" + (f" ({tr._graph_error})" if tr._graph_error else "")
    config["eager_ms_per_step"] = ms_eager / args.steps
    def shutdown():
        """Tear the process group down without ever hanging the run: graphs that captured NCCL kernels go first, and a timer
        force-exits (status 0: the record is already printed) if communicator destruction blocks."""
        if world > 1:
            import threading

            t = threading.Timer(45.0, lambda: os._exit(0))
            t.daemon = True
            t.start()
            try:
                dist.destroy_process_group()
            finally:
                t.cancel()

    if rank != 0:
        tr.release_graphs()
        shutdown()
        return

    peaks = _peaks()
    # dominant hand-written kernel inside the timed region -> roofline (algorithmic work from SURVEY section 8(d))
    work = sweep.algorithmic_work(SCALE, args.batch)
    roof = None
    if ktimes:
        tot = {k: n * ms for k, (n, ms) in ktimes.items()}
        # `roofline` = the hand-written kernel with the largest share of the step among ALL of them (hot-path blocks, Conv
        # epilogue, seams alike); every kernel's own fraction is under all_kernels, the per-block rows under blocks
        hot = tot
        top = max(hot, key=hot.get)
        n, ms = ktimes[top]
        w = work.get(top) or sweep.gemm_work(top, peaks) or sweep.fused_work(top) or sweep.bn_work(top) or sweep.seam_work(top)
        if not w:
            roof = {"kernel": top, "avg_ms": ms, "calls": n, "note": "no algorithmic-work entry",
                    "kernels_ms_per_step": {k: v / args.steps for k, v in sorted(tot.items(), key=lambda kv: -kv[1])}}
        else:
            achieved = w["amount"] / (ms * 1e-3) / (1e9 if w["bound"] == "hbm" else 1e12)
            peak = peaks["hbm_gbs"] if w["bound"] == "hbm" else peaks["bf16_tflops_sustained"]
            traffic = None  # dram__bytes_read+write per launch from the committed ncu --set full capture of this kernel
            for tname in ("traffic_r02.json", "traffic_r01.json"):
                tpath = os.path.join(ROOT, "profiles", tname)
                if traffic is None and os.path.isfile(tpath):
                    traffic = json.load(open(tpath)).get(sweep.ncu_kernel_name(top) or "")
            roof = {"kernel": top, "bound": w["bound"], "achieved": achieved, "peak": peak, "unit": "GB/s" if w["bound"] == "hbm" else "TFLOP/s",
                    "frac": achieved / peak, "traffic": traffic, "avg_ms": ms, "calls": n, "peak_source": peaks["source"] + " (sustained)",
                    "algorithmic": w["note"],
                    "share_of_step": tot[top] / ms_eager, "kernels_ms_per_step": {k: v / args.steps for k, v in sorted(tot.items(), key=lambda kv: -kv[1])}}
    if roof is not None:  # every hand-written kernel of the step: mean ms per launch + fraction of its roofline
        allk = {}
        for k, (n_, ms_) in ktimes.items():
            w_ = work.get(k) or sweep.gemm_work(k, peaks) or sweep.fused_work(k) or sweep.bn_work(k) or sweep.seam_work(k)
            ent = {"calls_per_step": n_ / args.steps, "avg_ms": round(ms_, 5)}
            if w_:
                pk = peaks["hbm_gbs"] if w_["bound"] == "hbm" else peaks["bf16_tflops_sustained"]
                ent.update(bound=w_["bound"], frac=round(w_["amount"] / (ms_ * 1e-3) / (1e9 if w_["bound"] == "hbm" else 1e12) / pk, 4))
            allk[k] = ent
        roof["all_kernels"] = allk
    line = {"metric": "train_images_per_sec", "value": imgs / (ms_dev * 1e-3), "unit": "img/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic", "config": config, "clocks": clocks,
            "gpu_launches": int(launches) if not graphed else int(kernels_per_step * args.steps),
            "e2e": {"value": imgs / (ms_e2e * 1e-3), "unit": "img/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 12,
                    "ms_per_step": ms_e2e / args.steps, "loss_items": [float(v) for v in last["loss"]]},
            "roofline": roof}
    # BASELINE config 1: bf16 inference, batch 64, forward only (eval mode, device-resident batch)
    tr.raw.eval()
    with torch.inference_mode(), torch.autocast("cuda", dtype=torch.bfloat16):
        imgf = (dev[0]["img"].float() / 255).contiguous(memory_format=torch.channels_last)
        for _ in range(3):
            tr.raw(imgf)
        inf_fn, inf_mode, g_inf = (lambda i: tr.raw(imgf)), "eager launches", None
        if graphed:   # the eager forward is host-bound (~400 launches in < 8 ms): replay it as a CUDA graph like the training step
            try:
                torch.cuda.synchronize()
                g_inf = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g_inf):
                    inf_out = tr.raw(imgf)  # noqa: F841  (kept alive: the graph's output buffers)
                inf_fn, inf_mode = (lambda i: g_inf.replay()), "CUDA-graph replay"
            except Exception as e:  # noqa: BLE001  capture is an optimisation; the eager forward stays correct
                sys.stderr.write(f"[bench] inference graph capture failed: {type(e).__name__}: {e}\n")
                torch.cuda.synchronize()
                inf_fn, g_inf = (lambda i: tr.raw(imgf)), None
        ms_inf = timed(inf_fn, args.steps, collective=False)
        del g_inf
    tr.raw.train()
    line["inference"] = {"value": args.batch * args.steps / (ms_inf * 1e-3), "unit": "img/s", "ms_per_batch": ms_inf / args.steps,
                         "config": f"configs[1]: bf16 autocast, batch 64, forward only, eval mode, 1 GPU, {inf_mode}"}
    if not args.no_sweep:
        line["modules"] = sweep.run(SCALE, args.batch, peaks, iters=10)
        if roof is not None:   # per-block rows with SURVEY 8(d)'s bounds: CBAM / SPPF vs HBM, whole SwinBlock vs tensor peak
            keep = ("cbam_fwd", "cbam_bwd", "sppf_pool_fwd_k5", "sppf_pool_bwd_k5", "sppf_pool_fwd_k7", "sppf_pool_bwd_k7",
                    "swin_block_fwd_ws7", "swin_block_bwd_ws7")
            roof["blocks"] = [{k: r[k] for k in ("kernel", "shape", "ms", "bound", "achieved", "peak", "unit", "frac")}
                              for r in line["modules"] if r["kernel"] in keep and (not r["kernel"].startswith("cbam") or r["note"] == "P5")]
    if world == 1 and not args.no_gpu_eager:
        del tr, dev
        torch.cuda.empty_cache()
        line["gpu_eager_baseline"] = gpu_eager_baseline_leg(args.steps, args.warmup, args.batch, f"cuda:{local_rank}")
        bf = line["gpu_eager_baseline"].get("bf16", {})
        if "value" in bf:
            line["vs_eager"] = {"value": line["value"] / bf["value"], "e2e": line["e2e"]["value"] / bf["value"],
                                "note": "this arm / the unmodified reference run eagerly on the same GPU (bf16 autocast); >1 = faster"}
    if not args.no_cpu_baseline:
        # N=1: in process (the driver's headline line).  N>1: bounded child process -- see cpu_baseline_bounded()
        line["cpu_baseline"] = cpu_baseline_leg() if world == 1 else cpu_baseline_bounded()
    print_record(line)
    if "tr" in locals():
        tr.release_graphs()
    shutdown()


if __name__ == "__main__":
    main()
