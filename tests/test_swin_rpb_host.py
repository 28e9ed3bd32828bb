"""CPU: SwinBlockRPB (Swin's learned relative-position bias on the SwinBlock) -- the oracle's bias, the module's boundary,
the C-ABI's argument checks (they run before any CUDA call) and the plugin's yaml name."""
import copy
import ctypes as C
import inspect
import io
import pickle
import sys
import types

import pytest
import torch

import improving_yolov8_cbam_swinblock_b200 as P
from improving_yolov8_cbam_swinblock_b200.harness import graph, train
from oracle import blocks as ob
from swin_rpb_oracle import relative_position_index, swin_rpb_forward


def _params(C_, seed=0):
    torch.manual_seed(seed)
    m = P.SwinBlock(C_, 2, 3)
    with torch.no_grad():
        for k, p in m.named_parameters():
            if "norm" in k or "bias" in k:
                p.add_(0.3 * torch.randn_like(p))
    return {k: v.detach().double() for k, v in m.named_parameters()}


# ---------------------------------------------------------------- oracle
@pytest.mark.parametrize("shift", [0, 1])
def test_zero_table_oracle_equals_oracle_without_bias(shift):
    p = _params(8)
    x = torch.randn(2, 8, 7, 5, dtype=torch.float64)
    want = ob.swin_forward(x, p, 2, 3, shift)
    got = swin_rpb_forward(x, p, 2, 3, shift, torch.zeros(25, 2, dtype=torch.float64))
    assert torch.equal(got, want)


@pytest.mark.parametrize("ws", range(1, 9))
def test_swin_built_index_equals_closed_form(ws):
    idx = relative_position_index(ws)
    L = ws * ws
    i = torch.arange(L)[:, None]
    j = torch.arange(L)[None, :]
    closed = (i // ws - j // ws + ws - 1) * (2 * ws - 1) + (i % ws - j % ws + ws - 1)
    assert idx.shape == (L, L) and torch.equal(idx, closed)
    assert int(idx.min()) == 0 and int(idx.max()) == (2 * ws - 1) ** 2 - 1


def test_table_gradcheck_shifted_and_padded():
    p = _params(4, seed=1)
    torch.manual_seed(2)
    x = torch.randn(1, 4, 5, 4, dtype=torch.float64)   # 5x4 map, ws 3: padded to 6x6; shift 1
    t = (0.5 * torch.randn(25, 2, dtype=torch.float64)).requires_grad_(True)
    assert torch.autograd.gradcheck(lambda tb: swin_rpb_forward(x, p, 2, 3, 1, tb), (t,))


def test_bias_changes_the_oracle():
    p = _params(8)
    x = torch.randn(1, 8, 6, 6, dtype=torch.float64)
    t = torch.randn(25, 2, dtype=torch.float64)
    assert not torch.allclose(swin_rpb_forward(x, p, 2, 3, 0, t), ob.swin_forward(x, p, 2, 3))


# ---------------------------------------------------------------- module
def test_signature_and_subclass():
    sig = inspect.signature(P.SwinBlockRPB.__init__)
    assert [(n, q.default) for n, q in list(sig.parameters.items())[1:]] == [
        ("dim", inspect.Parameter.empty), ("num_heads", 2), ("window_size", 7), ("shift_size", 0)]
    m = P.SwinBlockRPB(32)
    assert isinstance(m, P.SwinBlock)
    with pytest.raises(ValueError):
        P.SwinBlockRPB(32, 2, 9)


def test_state_dict_is_swinblock_plus_table():
    m, ref = P.SwinBlockRPB(64, 4, 8), P.SwinBlock(64, 4, 8)
    sd, rsd = m.state_dict(), ref.state_dict()
    assert sorted(sd) == sorted(list(rsd) + ["relative_position_bias_table"])
    for k in rsd:
        assert sd[k].shape == rsd[k].shape
    t = sd["relative_position_bias_table"]
    assert t.shape == (15 * 15, 4) and t.dtype == torch.float32
    assert 0.015 < float(t.std()) < 0.025   # trunc_normal_(std=0.02) as Swin calls it (its cut-off is at +-2, absolute)


def test_swinblock_state_dict_loads_with_only_the_table_missing():
    m = P.SwinBlockRPB(32, 2, 7)
    r = m.load_state_dict(P.SwinBlock(32, 2, 7).state_dict(), strict=False)
    assert r.missing_keys == ["relative_position_bias_table"] and r.unexpected_keys == []


def test_deepcopy_and_pickle_round_trip():
    m = P.SwinBlockRPB(32, 2, 7, 3)
    for m2 in (copy.deepcopy(m), pickle.loads(pickle.dumps(m))):
        assert type(m2) is P.SwinBlockRPB and m2.shift_size == 3
        assert all(torch.equal(a, b) for a, b in zip(m.state_dict().values(), m2.state_dict().values()))
    buf = io.BytesIO()
    torch.save(m, buf)
    buf.seek(0)
    assert torch.equal(torch.load(buf, weights_only=False).relative_position_bias_table, m.relative_position_bias_table)


def test_cpu_zero_shape_probe():
    m = P.SwinBlockRPB(16, 2, 7)
    y = m(torch.zeros(1, 16, 9, 9))
    assert y.shape == (1, 16, 9, 9) and not y.any()
    with pytest.raises(RuntimeError, match="no CPU path"):
        m(torch.randn(1, 16, 9, 9))


def test_table_is_in_the_no_decay_group():
    m = P.SwinBlockRPB(32, 2, 7)
    g0, g1, g2 = (g["params"] for g in train.param_groups(m))
    t = m.relative_position_bias_table
    assert any(p is t for p in g2) and not any(p is t for p in g0 + g1)
    assert len(g2) == 7


def test_detection_graph_with_the_bias_holds_two_tables():
    m = graph.DetectionGraph({**P.BLOCKS, "SwinBlock": P.SwinBlockRPB}, "n", 80)
    tabs = [k for k in m.state_dict() if k.endswith("relative_position_bias_table")]
    assert len(tabs) == 2
    assert isinstance(m.model[7], P.SwinBlockRPB) and isinstance(m.model[16], P.SwinBlockRPB)
    assert m.stride.tolist() == [8.0, 16.0, 32.0]
    assert sum(p.numel() for p in m.parameters()) == 3726642 + 2 * 169 * 2


# ---------------------------------------------------------------- C-ABI argument checks (no GPU needed)
def test_rpb_entry_points_reject_bad_arguments():
    from improving_yolov8_cbam_swinblock_b200 import _lib
    import improving_yolov8_cbam_swinblock_b200.functional  # noqa: F401  registers the swin entry points

    L = _lib.lib()
    one = C.c_void_p(16)
    # expand: window too large, table rows not matching ws, null pointers
    assert L.b200_swin_rpb_expand(one, 17 * 17, one, 9, 2, None) == 6
    assert L.b200_swin_rpb_expand(one, 169, one, 8, 2, None) == 1 and b"rows" in L.b200_last_error()
    assert L.b200_swin_rpb_expand(None, 169, one, 7, 2, None) == 1 and b"null" in L.b200_last_error()
    assert L.b200_swin_rpb_expand(one, 169, None, 7, 2, None) == 1
    for fwd in ("b200_swin_attn_fwd_rpb", "b200_swin_attn_fwd_tc_rpb"):
        f = getattr(L, fwd)
        dt = 1
        assert f(one, one, one, one, 81 * 4, 81, 128, 2, 0, 0, 9, 0, dt, None) == 6, fwd          # 9x9 window
        assert f(one, one, one, one, 49 * 4, 49, 128, 2, 0, 0, 8, 0, dt, None) == 1, fwd          # ws does not match L
        assert f(one, None, one, one, 49 * 4, 49, 128, 2, 0, 0, 7, 0, dt, None) == 1, fwd         # no bias
        assert b"null" in L.b200_last_error()
    T, Lw, Cc, nh = 49 * 4, 49, 128, 2
    for tc in (0, 1):
        need = L.b200_swin_rpb_workspace_bytes(T, Lw, nh, tc)
        assert need >= 4 * nh * 4096 * 4
        # (... bias, gqkv, gtable, table_rows, workspace, workspace_bytes, tokens, L, C, nh, nWh, nWw, ws, shift, dtype, stream)
        args = [one] * (4 if tc else 5) + [one, one, 169, one, need, T, Lw, Cc, nh, 0, 0, 7, 0, 1, None]
        f = L.b200_swin_attn_bwd_tc_rpb if tc else L.b200_swin_attn_bwd_rpb
        bad = list(args)
        bad[-11] = need - 4                                       # workspace too small
        assert f(*bad) == 5 and b"workspace" in L.b200_last_error()
        bad = list(args)
        bad[-13] = 121                                            # table of ws 6 with ws 7
        assert f(*bad) == 1 and b"rows" in L.b200_last_error()
        bad = list(args)
        bad[-14] = None                                           # no gtable
        assert f(*bad) == 1 and b"null" in L.b200_last_error()
        bad = list(args)
        bad[-4] = 9                                               # ws 9 > 8
        assert f(*bad) == 6
    assert L.b200_swin_rpb_workspace_bytes(T, Lw, nh, 0) == (4 + 1) * nh * 4096 * 4
    assert L.b200_swin_rpb_workspace_bytes(64 * 36 * 49, 49, 2, 1) == (4 * 160 + 1) * 2 * 4096 * 4
    assert L.b200_swin_rpb_workspace_bytes(100, 49, 2, 1) == 0


# ---------------------------------------------------------------- plugin
def test_plugin_adds_and_removes_the_yaml_name(monkeypatch):
    from improving_yolov8_cbam_swinblock_b200 import modules, ultralytics_plugin as plugin

    class StockConv(torch.nn.Module):
        def __init__(self, *a, **k):
            super().__init__()

    class StockSwin(torch.nn.Module):
        pass

    stubs = {}
    for name in ("ultralytics", "ultralytics.nn", "ultralytics.nn.tasks", "ultralytics.nn.modules", "ultralytics.nn.modules.cbam",
                 "ultralytics.nn.modules.swin_block", "ultralytics.nn.modules.block", "ultralytics.nn.modules.conv",
                 "ultralytics.nn.modules.head"):
        stubs[name] = types.ModuleType(name)
        monkeypatch.setitem(sys.modules, name, stubs[name])
    stubs["ultralytics.nn.modules.conv"].Conv = StockConv
    for name in ("ultralytics.nn.tasks", "ultralytics.nn.modules", "ultralytics.nn.modules.swin_block"):
        stubs[name].SwinBlock = StockSwin
    stubs["ultralytics.nn.modules.cbam"].ChannelAttention = object
    stubs["ultralytics.nn.modules.cbam"].SpatialAttention = object
    monkeypatch.setattr(plugin, "Conv", None)
    monkeypatch.setattr(plugin, "SPPF", None)
    try:
        table = plugin.install()
        assert table["SwinBlockRPB"] is modules.SwinBlockRPB
        for name in ("ultralytics.nn.tasks", "ultralytics.nn.modules"):
            assert stubs[name].SwinBlockRPB is modules.SwinBlockRPB
            assert stubs[name].SwinBlock is modules.SwinBlock
        assert not hasattr(stubs["ultralytics.nn.modules.swin_block"], "SwinBlockRPB")
        plugin.install()   # idempotent
    finally:
        plugin.uninstall()
    for name in ("ultralytics.nn.tasks", "ultralytics.nn.modules"):
        assert not hasattr(stubs[name], "SwinBlockRPB")
        assert stubs[name].SwinBlock is StockSwin
