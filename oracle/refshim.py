"""TEST INFRASTRUCTURE — never imported by the product path.

Makes the UNMODIFIED reference (facebookresearch/SlowFast, copied into oracle/_ref by build() through
oracle/install_ref.py) importable offline by providing tiny stand-ins for its un-vendored Python dependencies (fvcore, iopath,
pytorchvideo, detectron2, simplejson, matplotlib, av) and the ``vision.fair.slowfast`` namespace its tools import
(SURVEY.md §8b/§8c).  Used only to (a) pin ``oracle/torch_oracle.py`` against the reference's own modules and
(b) generate the golden fixtures under ``tests/golden``, (c) run the reference itself as the CPU / ATen-GPU baseline of
``bench.py`` and in the driver tests (tools/train_net.py, test_net.py).  oracle/_ref is git-ignored and travels with the
built tree; ``baseline/_ref`` (installed by ``baseline/install_ref.sh``, byte-identical python files) is also searched.

The stand-ins restate published behaviour of those packages:
  fvcore.nn.weight_init.c2_msra_fill  = kaiming_normal_(mode="fan_out", nonlinearity="relu"), bias 0
  fvcore.nn.weight_init.c2_xavier_fill = kaiming_uniform_(a=1), bias 0
  pytorchvideo.layers.swish.Swish      = x * sigmoid(x)
  pytorchvideo SoftTargetCrossEntropyLoss = mean over batch of sum(-t * log_softmax(x))
"""
from __future__ import annotations

import ast
import copy
import importlib
import os
import sys
import time
import types

_REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _find_reference_root() -> str:
    """The unmodified reference: $SLOWFAST_REFERENCE_ROOT, else the copy build() makes in oracle/_ref
    (oracle/install_ref.py), else the offline install made by baseline/install_ref.sh (both git-ignored)."""
    cands = [os.environ.get("SLOWFAST_REFERENCE_ROOT"), os.path.join(_REPO, "oracle", "_ref"),
             os.path.join(_REPO, "baseline", "_ref")]
    for c in cands:
        if c and os.path.isdir(os.path.join(c, "slowfast")) and os.path.isdir(os.path.join(c, "configs")):
            return c
    return cands[1]


REFERENCE_ROOT = _find_reference_root()


def reference_available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "slowfast"))


def _mod(name: str, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    m.__path__ = []  # behave as a package so that submodules can hang off it
    sys.modules[name] = m
    parent, _, child = name.rpartition(".")
    if parent and parent in sys.modules:
        setattr(sys.modules[parent], child, m)
    return m


def _install_fvcore():
    import torch.nn as nn
    import yaml

    class Registry:
        def __init__(self, name):
            self._name = name
            self._obj_map = {}

        def _do_register(self, name, obj):
            assert name not in self._obj_map, f"'{name}' already registered in '{self._name}'"
            self._obj_map[name] = obj

        def register(self, obj=None):
            if obj is None:
                def deco(fn):
                    self._do_register(fn.__name__, fn)
                    return fn
                return deco
            self._do_register(obj.__name__, obj)
            return obj

        def get(self, name):
            if name not in self._obj_map:
                raise KeyError(f"No object named '{name}' found in '{self._name}' registry!")
            return self._obj_map[name]

        def __contains__(self, name):
            return name in self._obj_map

    class CfgNode(dict):
        """yacs-style config node: attribute access, yaml merge, KEY VALUE list merge, clone, dump."""

        def __init__(self, init_dict=None, key_list=None, new_allowed=False):
            super().__init__()
            for k, v in (init_dict or {}).items():
                self[k] = CfgNode(v) if isinstance(v, dict) and not isinstance(v, CfgNode) else v

        def __getattr__(self, name):
            if name in self:
                return self[name]
            raise AttributeError(name)

        def __setattr__(self, name, value):
            self[name] = value

        def clone(self):
            return copy.deepcopy(self)

        def __deepcopy__(self, memo):
            out = CfgNode()
            for k, v in self.items():
                out[k] = copy.deepcopy(v, memo)
            return out

        def _merge(self, other):
            for k, v in other.items():
                if isinstance(v, dict) and k in self and isinstance(self[k], CfgNode):
                    self[k]._merge(v)
                else:
                    if isinstance(v, str):
                        try:  # yacs decodes string values with literal_eval: "(2, 4, 4)" -> tuple, "1e-4" -> float
                            v = ast.literal_eval(v)
                        except (ValueError, SyntaxError):
                            pass
                    if k in self and isinstance(self[k], float) and isinstance(v, int) and not isinstance(v, bool):
                        v = float(v)
                    if isinstance(v, tuple) and k in self and isinstance(self[k], list):
                        v = list(v)
                    self[k] = CfgNode(v) if isinstance(v, dict) else v

        def merge_from_file(self, path):
            with open(path) as f:
                self._merge(yaml.safe_load(f) or {})

        def merge_from_other_cfg(self, other):
            self._merge(other)

        def merge_from_list(self, lst):
            assert len(lst) % 2 == 0
            for k, v in zip(lst[0::2], lst[1::2]):
                node = self
                parts = k.split(".")
                for p in parts[:-1]:
                    node = node[p]
                if isinstance(v, str):
                    try:
                        v = ast.literal_eval(v)
                    except (ValueError, SyntaxError):
                        pass
                node[parts[-1]] = v

        def dump(self, **kw):
            def plain(n):
                return {k: plain(v) if isinstance(v, CfgNode) else v for k, v in n.items()}
            return yaml.safe_dump(plain(self), **kw)

        def freeze(self):
            pass

        def defrost(self):
            pass

    class Timer:
        def __init__(self):
            self.reset()

        def reset(self):
            self._start = time.perf_counter()
            self._paused = None
            self._total_paused = 0.0
            self._count_start = 1

        def pause(self):
            if self._paused is None:
                self._paused = time.perf_counter()

        def is_paused(self):
            return self._paused is not None

        def resume(self):
            if self._paused is not None:
                self._total_paused += time.perf_counter() - self._paused
                self._paused = None
                self._count_start += 1

        def seconds(self):
            end = self._paused if self._paused is not None else time.perf_counter()
            return end - self._start - self._total_paused

        def avg_seconds(self):
            return self.seconds() / self._count_start

    def c2_msra_fill(module):
        nn.init.kaiming_normal_(module.weight, mode="fan_out", nonlinearity="relu")
        if module.bias is not None:
            nn.init.constant_(module.bias, 0)

    def c2_xavier_fill(module):
        nn.init.kaiming_uniform_(module.weight, a=1)
        if module.bias is not None:
            nn.init.constant_(module.bias, 0)

    def _unavailable(*a, **k):
        raise RuntimeError("fvcore stand-in: flop/activation counting is not provided offline")

    # fvcore.nn.precise_bn (published algorithm): BN layers in training mode get momentum 1.0, `num_iters` forward passes run
    # under no_grad, and the per-batch statistics each pass leaves in running_mean / running_var are averaged
    BN_TYPES = (nn.BatchNorm1d, nn.BatchNorm2d, nn.BatchNorm3d, nn.SyncBatchNorm)

    def get_bn_modules(model):
        return [m for m in model.modules() if m.training and isinstance(m, BN_TYPES)]

    def update_bn_stats(model, data_loader, num_iters=200):
        import itertools

        import torch
        bn_layers = get_bn_modules(model)
        if len(bn_layers) == 0:
            return
        momentum_actual = [bn.momentum for bn in bn_layers]
        for bn in bn_layers:
            bn.momentum = 1.0
        running_mean = [torch.zeros_like(bn.running_mean) for bn in bn_layers]
        running_var = [torch.zeros_like(bn.running_var) for bn in bn_layers]
        ind = -1
        for ind, inputs in enumerate(itertools.islice(data_loader, num_iters)):
            with torch.no_grad():
                model(inputs)
            for i, bn in enumerate(bn_layers):
                running_mean[i] += (bn.running_mean - running_mean[i]) / (ind + 1)
                running_var[i] += (bn.running_var - running_var[i]) / (ind + 1)
        assert ind == num_iters - 1, f"update_bn_stats: the loader ran out after {ind + 1} of {num_iters} iterations"
        for i, bn in enumerate(bn_layers):
            bn.running_mean = running_mean[i]
            bn.running_var = running_var[i]
            bn.momentum = momentum_actual[i]

    _mod("fvcore")
    _mod("fvcore.common")
    _mod("fvcore.common.registry", Registry=Registry)
    _mod("fvcore.common.config", CfgNode=CfgNode)
    _mod("fvcore.common.timer", Timer=Timer)
    _mod("fvcore.nn")
    _mod("fvcore.nn.weight_init", c2_msra_fill=c2_msra_fill, c2_xavier_fill=c2_xavier_fill)
    _mod("fvcore.nn.flop_count", flop_count=_unavailable)
    _mod("fvcore.nn.activation_count", activation_count=_unavailable)
    _mod("fvcore.nn.precise_bn", get_bn_modules=get_bn_modules, update_bn_stats=update_bn_stats)


def _install_misc():
    import json

    import torch
    import torch.nn as nn

    class _PathManager:
        def open(self, path, mode="r", **kw):
            return open(path, mode)

        def exists(self, p):
            return os.path.exists(p)

        def isfile(self, p):
            return os.path.isfile(p)

        def isdir(self, p):
            return os.path.isdir(p)

        def ls(self, p):
            return os.listdir(p)

        def mkdirs(self, p):
            os.makedirs(p, exist_ok=True)

        def get_local_path(self, p, **kw):
            return p

        def rm(self, p):
            os.remove(p)

    class PathManagerFactory:
        @staticmethod
        def get(*a, **k):
            return _PathManager()

    _mod("iopath")
    _mod("iopath.common")
    _mod("iopath.common.file_io", PathManagerFactory=PathManagerFactory, g_pathmgr=_PathManager())

    class Swish(nn.Module):
        def forward(self, x):
            return x * torch.sigmoid(x)

    class SoftTargetCrossEntropyLoss(nn.Module):
        def __init__(self, ignore_index=-100, reduction="mean", normalize_targets=True):
            super().__init__()
            self.reduction = reduction
            self.normalize_targets = normalize_targets

        def forward(self, x, y):
            if self.normalize_targets:
                y = y / y.sum(dim=-1, keepdim=True).clamp_min(1e-8)
            loss = torch.sum(-y * torch.nn.functional.log_softmax(x.float(), dim=-1), dim=-1)
            return loss.mean() if self.reduction == "mean" else loss

    class _NoSyncBN1d(nn.BatchNorm1d):
        def __init__(self, num_sync_devices=1, global_sync=False, **kw):
            super().__init__(**kw)

    class _NoSyncBN3d(nn.BatchNorm3d):
        def __init__(self, num_sync_devices=1, global_sync=False, **kw):
            super().__init__(**kw)

    def _cat_all_gather(t, local=False):
        return t

    _mod("pytorchvideo")
    _mod("pytorchvideo.layers")
    _mod("pytorchvideo.layers.swish", Swish=Swish)
    _mod("pytorchvideo.layers.batch_norm", NaiveSyncBatchNorm1d=_NoSyncBN1d, NaiveSyncBatchNorm3d=_NoSyncBN3d)
    _mod("pytorchvideo.layers.distributed", cat_all_gather=_cat_all_gather, get_local_process_group=lambda: None,
         get_local_rank=lambda: 0, get_local_size=lambda: 1, get_world_size=lambda: 1,
         init_distributed_training=lambda *a, **k: None)
    _mod("pytorchvideo.losses")
    _mod("pytorchvideo.losses.soft_target_cross_entropy", SoftTargetCrossEntropyLoss=SoftTargetCrossEntropyLoss)

    class ROIAlign(nn.Module):
        def __init__(self, output_size, spatial_scale, sampling_ratio, aligned=True):
            super().__init__()
            self.args = (output_size, spatial_scale, sampling_ratio, aligned)

        def forward(self, x, rois):
            from torchvision.ops import roi_align
            o, s, r, a = self.args
            return roi_align(x, rois, o, s, r, a)

    _mod("detectron2")
    _mod("detectron2.layers", ROIAlign=ROIAlign)
    def _sj_dumps(obj, **kw):  # simplejson.dumps(use_decimal=True) serialises decimal.Decimal as a number
        import decimal
        kw.pop("use_decimal", None)
        return json.dumps(obj, default=lambda o: float(o) if isinstance(o, decimal.Decimal) else str(o), **kw)

    _mod("simplejson", dumps=_sj_dumps, loads=json.loads)
    if "matplotlib" not in sys.modules:
        try:
            importlib.import_module("matplotlib.pyplot")
        except Exception:  # noqa: BLE001
            _mod("matplotlib")
            _mod("matplotlib.pyplot")
    try:
        importlib.import_module("av")
    except Exception:  # noqa: BLE001
        _mod("av")


_installed = False


def install() -> None:
    """Install the stand-ins and put the reference on sys.path (idempotent)."""
    global _installed
    if _installed:
        return
    if not reference_available():
        raise RuntimeError(f"reference tree not found at {REFERENCE_ROOT} (build() installs it when a checkout is readable)")
    _install_fvcore()
    _install_misc()
    for name in ("vision", "vision.fair", "vision.fair.slowfast"):
        m = types.ModuleType(name)
        m.__path__ = [REFERENCE_ROOT] if name == "vision.fair.slowfast" else []
        sys.modules[name] = m
    sys.modules["vision"].fair = sys.modules["vision.fair"]
    sys.modules["vision.fair"].slowfast = sys.modules["vision.fair.slowfast"]
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    _installed = True


def load_cfg(yaml_relpath: str, overrides=()):
    """Reference config for ``configs/<yaml_relpath>`` with KEY VALUE overrides, NUM_GPUS 0 (CPU)."""
    install()
    from slowfast.config.defaults import assert_and_infer_cfg, get_cfg

    cfg = get_cfg()
    cfg.merge_from_file(os.path.join(REFERENCE_ROOT, "configs", yaml_relpath))
    cfg.merge_from_list(["NUM_GPUS", 0] + list(overrides))
    return assert_and_infer_cfg(cfg)


def build_reference_model(cfg):
    install()
    import torch
    from slowfast.models import build_model

    torch.manual_seed(cfg.RNG_SEED)
    model = build_model(cfg)
    inner = getattr(model, "module", model)
    assert type(inner).__module__.startswith("slowfast."), (
        f"build_model returned {type(inner).__module__}.{type(inner).__name__}: the reference's MODEL_REGISTRY is still "
        "pointed at the engine classes (integration.register(replace=True)); restore the stock entries first")
    return model
