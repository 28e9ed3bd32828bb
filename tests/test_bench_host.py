"""Host-side pieces of bench.py that need no GPU: the bounded child-process form of the host-core baseline leg (what rank 0 runs at
world_size > 1), the roofline entries of the shape-tagged launches added in round 2 and ``--dump-outputs``."""
import json
import os
import subprocess
import sys
import time

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_bounded_cpu_baseline_gives_up_at_its_limit_instead_of_stalling_the_record():
    import bench

    t0 = time.time()
    out = bench.cpu_baseline_bounded(timeout_s=2)
    assert time.time() - t0 < 30
    assert set(out) == {"skipped"} and "2 s limit" in out["skipped"]


def test_roofline_entries_of_the_round_2_launch_tags():
    from improving_yolov8_cbam_swinblock_b200.harness import sweep

    n = 64 * 320 * 320 * 16 + 64 * 160 * 160 * 32
    for tag in ("b200_conv3x3_dgrad_s2[64x320x320x16<-32]", "b200_conv3x3_fwd_s2[64x320x320x16->32]",
                "b200_conv3x3_wgrad[64x320x320x16->32,s2]"):
        w = sweep.seam_work(tag)
        assert w["bound"] == "hbm" and w["amount"] == 2.0 * n, tag
    w = sweep.seam_work("b200_nhwc_add[409600x64x2]")
    assert w["amount"] == 3.0 * 409600 * 64 * 2          # two gradient maps read, their sum written, 2 bytes per element
    w = sweep.seam_work("b200_stem_conv_fwd[64x640x640x3->16]")
    assert w["amount"] == (64 * 640 * 640 * 3 + 64 * 320 * 320 * 16) * 2.0
    assert sweep.seam_work("b200_nhwc_concat[409600x64]")["amount"] == 2.0 * 409600 * 64 * 2
    assert sweep.seam_work("b200_unknown[1x2]") is None


def test_dump_outputs_writes_float32_arrays_and_samples_large_states_the_same_way_every_time(tmp_path, monkeypatch):
    import bench

    monkeypatch.setattr(bench, "DUMP_MAX_ELEMS", 50)
    items = torch.tensor([1.5, 2.5, 3.5])
    w = torch.randn(6, 10, 1, 1, dtype=torch.float64).contiguous(memory_format=torch.channels_last)
    sd = {"w": w, "n": torch.tensor(3), "b": torch.ones(4, dtype=torch.bfloat16)}
    bench.dump_outputs(str(tmp_path / "small"), items, {"w": w[:2], "n": sd["n"]})
    small = np.load(tmp_path / "small" / "model_state.npy")
    assert small.dtype == np.float32 and np.array_equal(small, w[:2].float().numpy().reshape(-1))   # logical order, not memory order
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), items, sd)
    assert sorted(os.listdir(tmp_path / "a")) == ["loss_items.npy", "model_state.npy"]
    got = np.load(tmp_path / "a" / "loss_items.npy")
    assert got.dtype == np.float32 and got.tolist() == [1.5, 2.5, 3.5]
    full = np.concatenate([w.float().numpy().reshape(-1), np.ones(4, np.float32)])
    a, b = np.load(tmp_path / "a" / "model_state.npy"), np.load(tmp_path / "b" / "model_state.npy")
    assert a.dtype == np.float32 and a.shape == (50,) and np.array_equal(a, b)
    assert np.isin(a, full).all()


def test_dump_outputs_from_the_command_line_repeats_exactly(tmp_path):
    """Two runs with the same arguments see the same inputs and write the same outputs.  The host-core arm (--impl
    reference) at batch 1 keeps this cheap enough to run without a GPU."""
    for d in ("a", "b"):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "0",
                            "--ref-batch", "1", "--dump-outputs", str(tmp_path / d)], capture_output=True, text=True, timeout=600, cwd=tmp_path)
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout)["steps"] == 2
    for name in ("loss_items", "model_state"):
        a, b = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert a.dtype == np.float32 and np.isfinite(a).all() and np.array_equal(a, b), name
    assert np.load(tmp_path / "a" / "loss_items.npy").shape == (3,)


def test_reference_arm_runs_exactly_the_requested_steps_and_dumps_the_last_one(tmp_path, monkeypatch):
    import bench

    model = torch.nn.Linear(2, 2)
    calls = []

    def step(batch):
        calls.append(batch["img"].shape[0])
        return torch.tensor([float(len(calls)), 0.0, 0.0])

    monkeypatch.setattr(bench, "_make_cpu_trainer", lambda kind: (None, step, model))
    out = bench.cpu_reference_run(3, 2, batch=1, dump_dir=str(tmp_path))
    assert calls == [1] * 5 and out["steps"] == 3 and out["warmup"] == 2
    assert np.load(tmp_path / "loss_items.npy").tolist() == [5.0, 0.0, 0.0]


@pytest.mark.parametrize("args,msg", [(["--steps", "0"], "at least one timed step"),
                                      (["--impl", "reference", "--dump-outputs", "x"], "needs --ref-batch")])
def test_bench_rejects_arguments_it_cannot_honour(args, msg, tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=120, cwd=tmp_path)
    assert r.returncode == 2 and msg in r.stderr and r.stdout == ""
    assert not os.listdir(tmp_path)
