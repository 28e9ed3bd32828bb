"""Bind the B200 blocks into an (unmodified) Ultralytics checkout of the reference fork.

``parse_model`` resolves yaml strings with ``globals()[m]`` in ``ultralytics.nn.tasks`` (tasks.py:1438) and builds
its ``base_modules`` set from the same globals at call time (tasks.py:1375-1412), so rebinding three names there
(and in ``ultralytics.nn.modules`` for ``from ... import`` users / pickles) IS the integration:

    import improving_yolov8_cbam_swinblock_b200.ultralytics_plugin as plugin
    plugin.install()            # before building DetectionModel / YOLO(...)
    ...
    plugin.uninstall()

Classes are created once at import (bound to the reference's own ``Conv`` so ``fuse()`` still sees Conv
instances) and live at module level here, so whole-model pickles (trainer.py:531-562) resolve them by path.
"""
from __future__ import annotations

import importlib

from . import modules as _m

_TARGETS = ("ultralytics.nn.tasks", "ultralytics.nn.modules", "ultralytics.nn.modules.cbam",
            "ultralytics.nn.modules.swin_block", "ultralytics.nn.modules.block")
_saved: dict = {}
_added: list = []   # (module, name) that install() created rather than rebound
_NEW_TARGETS = ("ultralytics.nn.tasks", "ultralytics.nn.modules")
_saved_methods: dict = {}

CBAM = _m.CBAM
ChannelAttentionMap = _m.ChannelAttention
SpatialAttentionMap = _m.SpatialAttention
SwinBlock = _m.SwinBlock
SwinBlockRPB = _m.SwinBlockRPB   # extension: no such name in the reference, so install() adds it where parse_model looks
SPPF = None  # created by install() against ultralytics' Conv
Conv = None  # ultralytics' Conv with the fused BN+SiLU epilogue (SURVEY 8(f)-1), created by install()
_CONV_TARGETS = ("ultralytics.nn.tasks", "ultralytics.nn.modules", "ultralytics.nn.modules.conv",
                 "ultralytics.nn.modules.block", "ultralytics.nn.modules.head")


def _c2f_forward(self, x):
    """block.py C2f.forward with the NHWC seam kernels (SURVEY 8(f)-2); CPU tensors take the stock ops inside."""
    from . import functional as Fb

    y = list(Fb.nhwc_chunk(self.cv1(x), 2))
    inp = Fb.nhwc_concat([y[-1]])   # dense second half for the bottlenecks' 3x3 convs and shortcut adds
    for m in self.m:
        inp = m(inp)
        y.append(inp)
    return self.cv2(Fb.nhwc_concat(y))


def _concat_forward(self, x):
    """conv.py Concat.forward: channel concat through b200_nhwc_concat, any other dimension through torch.cat."""
    import torch

    from . import functional as Fb

    return Fb.nhwc_concat(x) if self.d == 1 else torch.cat(x, self.d)


_SEAM_PATCHES = (("ultralytics.nn.modules.block", "C2f", "forward", _c2f_forward),
                 ("ultralytics.nn.modules.conv", "Concat", "forward", _concat_forward))


def install(conv_epilogue: bool = False, seams: bool = False):
    """Rebind CBAM / SwinBlock / SPPF in the reference's namespaces and add SwinBlockRPB to ``ultralytics.nn.tasks`` /
    ``ultralytics.nn.modules`` (so a yaml row ``[-1, 1, SwinBlockRPB, [128]]`` parses like SwinBlock).  Returns the
    {name: class} table.

    SPPF's own cv1/cv2 always use the fused BN+SiLU epilogue; ``conv_epilogue=True`` additionally rebinds ``Conv``
    itself (a subclass of the reference's, same state_dict / ``fuse()`` behaviour) so every Conv caller gets it.
    ``seams=True`` replaces ``C2f.forward`` and ``Concat.forward`` (same classes, same parameters) by versions that
    move data with the NHWC concat kernel; both are undone by ``uninstall()``."""
    global SPPF, Conv
    conv_mod = importlib.import_module("ultralytics.nn.modules.conv")
    if Conv is None:
        Conv = _m.make_conv(_saved.get(("ultralytics.nn.modules.conv", "Conv"), conv_mod.Conv), module=__name__)
    if SPPF is None:
        SPPF = _m.make_sppf(Conv, module=__name__)
    table = {"CBAM": CBAM, "SwinBlock": SwinBlock, "SPPF": SPPF, "SwinBlockRPB": SwinBlockRPB}
    if conv_epilogue:
        for modname in _CONV_TARGETS:
            mod = importlib.import_module(modname)
            if hasattr(mod, "Conv"):
                _saved.setdefault((modname, "Conv"), getattr(mod, "Conv"))
                setattr(mod, "Conv", Conv)
    if seams:
        for modname, clsname, attr, fn in _SEAM_PATCHES:
            cls_ = getattr(importlib.import_module(modname), clsname)
            _saved_methods.setdefault((modname, clsname, attr), cls_.__dict__[attr])
            setattr(cls_, attr, fn)
    for modname in _TARGETS:
        mod = importlib.import_module(modname)
        for name, cls in table.items():
            if hasattr(mod, name) and (modname, name) not in _added:
                _saved.setdefault((modname, name), getattr(mod, name))
                setattr(mod, name, cls)
            elif modname in _NEW_TARGETS and name == "SwinBlockRPB":
                if (modname, name) not in _added:
                    _added.append((modname, name))
                setattr(mod, name, cls)
    # cbam.py's own ChannelAttention / SpatialAttention (maps only).  NOTE: ultralytics.nn.modules exports the
    # *stock* conv.py classes under these names (modules/__init__.py:66,78; SURVEY D5) -- those are left alone.
    cb = importlib.import_module("ultralytics.nn.modules.cbam")
    for name, cls in (("ChannelAttention", ChannelAttentionMap), ("SpatialAttention", SpatialAttentionMap)):
        _saved.setdefault((cb.__name__, name), getattr(cb, name))
        setattr(cb, name, cls)
    return table


def uninstall():
    for (modname, name), cls in list(_saved.items()):
        setattr(importlib.import_module(modname), name, cls)
    _saved.clear()
    for modname, name in _added:
        mod = importlib.import_module(modname)
        if hasattr(mod, name):
            delattr(mod, name)
    _added.clear()
    for (modname, clsname, attr), fn in list(_saved_methods.items()):
        setattr(getattr(importlib.import_module(modname), clsname), attr, fn)
    _saved_methods.clear()
