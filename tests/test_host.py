"""CPU: host-side logic — C-ABI exports, state_dict / init parity of the engine modules, config presets."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


def test_library_exports_every_declared_symbol():
    from slowfast_b200 import lib as L
    from slowfast_b200.build import build_native
    build_native()
    header = open(os.path.join(ROOT, "include", "slowfast_b200.h")).read()
    declared = set(re.findall(r"\b(sfb_[a-z0-9_]+)\s*\(", header))
    assert declared, "no declarations found"
    dll = ctypes.CDLL(str(L.lib_path()))
    for name in sorted(declared):
        assert hasattr(dll, name), f"{name} declared in include/slowfast_b200.h but not exported"
    assert set(L.exported_symbols()) == declared, (set(L.exported_symbols()) ^ declared)
    lib = L.load()
    assert lib.sfb_abi_version() == 1
    assert lib.sfb_build_arch() == b"sm_100a"


def test_no_cpu_fallback():
    """Without a CUDA device the product path raises instead of computing on the CPU."""
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    from slowfast_b200.config import get_cfg
    from slowfast_b200.lib import NativeLibraryError
    from slowfast_b200.nets.resnet import B200SlowFast
    cfg = get_cfg("SLOWFAST_8x8_R50", DATA={"NUM_FRAMES": 8, "TRAIN_CROP_SIZE": 32})
    m = B200SlowFast(cfg)
    with pytest.raises(NativeLibraryError):
        m([torch.zeros(1, 3, 2, 32, 32), torch.zeros(1, 3, 8, 32, 32)])


def test_slowfast_state_dict_matches_reference_keys():
    from slowfast_b200.config import get_cfg
    from slowfast_b200.nets.resnet import B200SlowFast
    gold = torch.load(os.path.join(GOLDEN, "slowfast_r50_224.pt"))
    m = B200SlowFast(get_cfg("SLOWFAST_8x8_R50"))
    keys = [(k, tuple(v.shape)) for k, v in m.state_dict().items()]
    assert keys == [(k, tuple(shape)) for k, shape in gold["keys"]]
    assert sum(p.numel() for p in m.parameters()) == 34566488  # 34.57 M (projects/pytorchvideo/README.md:34)
    # BN modules stay torch _NormBase instances (optimizer.py:41-56 groups parameters by that)
    n_bn = sum(isinstance(x, torch.nn.modules.batchnorm._NormBase) for x in m.modules())
    assert n_bn == 110


def _reference_init(yaml, overrides=()):
    """The reference's resolved config and the digests of its freshly initialised state (oracle/make_golden_reference.py)."""
    from oracle.make_golden_reference import init_key
    return torch.load(os.path.join(GOLDEN, "reference_init.pt"))[init_key(yaml, list(overrides))]


def _reference_cfg(yaml, ref, overrides=()):
    """The reference's own CfgNode when the reference is installed (oracle/_ref), else its stored resolved values."""
    from oracle import refshim
    from slowfast_b200.config import Cfg
    if refshim.reference_available():
        return refshim.load_cfg(yaml, list(overrides))
    return Cfg(ref["cfg"])


def _assert_same_init(state, ref):
    from oracle.make_golden_reference import layout_digest, tensor_digest
    assert layout_digest(state) == ref["layout"], "state_dict names / shapes / order differ from the reference's"
    bad = [k for i, (k, v) in enumerate(state.items()) if tensor_digest(v) != ref["values"][8 * i:8 * i + 8]]
    assert not bad, bad[:5]


def test_slowfast_init_is_bit_identical_to_reference_when_available():
    """Same seed, same initial weights as the reference's build_model, compared through the digests of its state."""
    from slowfast_b200.config import get_cfg
    from slowfast_b200.nets.resnet import B200SlowFast
    ref = _reference_init("Kinetics/SLOWFAST_8x8_R50.yaml")
    torch.manual_seed(ref["cfg"]["RNG_SEED"])
    _assert_same_init(B200SlowFast(get_cfg("SLOWFAST_8x8_R50")).state_dict(), ref)
    # and the engine classes accept the reference's own resolved config
    torch.manual_seed(ref["cfg"]["RNG_SEED"])
    _assert_same_init(B200SlowFast(_reference_cfg("Kinetics/SLOWFAST_8x8_R50.yaml", ref)).state_dict(), ref)


def test_integration_registers_into_reference_registry():
    """slowfast.models.build_model (the unmodified reference) hands out the engine class after register()."""
    from oracle import refshim
    if not refshim.reference_available():
        pytest.skip("no reference tree (build() copies it into oracle/_ref when a checkout is readable)")
    refshim.install()
    import slowfast_b200.integration as integ
    from slowfast.models import build_model
    from slowfast.models.build import MODEL_REGISTRY
    from slowfast_b200.nets.resnet import B200SlowFast
    saved = dict(MODEL_REGISTRY._obj_map)
    try:
        served = integ.register(replace=True)
        assert "B200SlowFast" in served and "SlowFast" in served
        assert {"B200ResNet", "B200MViT", "B200X3D", "X3D", "B200MaskMViT", "MaskMViT"} <= set(served)
        cfg = refshim.load_cfg("Kinetics/SLOWFAST_8x8_R50.yaml")
        model = build_model(cfg)                       # reference code path: registry lookup -> cls(cfg)
        assert isinstance(model, B200SlowFast)
        cfg2 = refshim.load_cfg("Kinetics/SLOWFAST_8x8_R50.yaml", ["MODEL.MODEL_NAME", "B200SlowFast"])
        assert isinstance(build_model(cfg2), B200SlowFast)
        # the reference's optimizer builder accepts the module tree (BN / non-BN / zero-WD grouping, optimizer.py:41-91)
        import slowfast.models.optimizer as optim
        opt = optim.construct_optimizer(model, cfg)
        assert sum(len(g["params"]) for g in opt.param_groups) == len(list(model.parameters()))
    finally:
        MODEL_REGISTRY._obj_map.clear()
        MODEL_REGISTRY._obj_map.update(saved)


MODELS = {
    # golden file -> (preset, yaml, engine class path, parameter count)
    "c2d_r50_small": ("C2D_8x8_R50", "Kinetics/C2D_8x8_R50.yaml", "slowfast_b200.nets.resnet_single:B200ResNet"),
    "mvitv2_s_224": ("MVITv2_S_16x4", "Kinetics/MVITv2_S_16x4.yaml", "slowfast_b200.nets.mvit:B200MViT"),
    "x3d_m_224": ("X3D_M", "Kinetics/X3D_M.yaml", "slowfast_b200.nets.x3d:B200X3D"),
    "maskfeat_s_224": ("MVITv2_S_16x4_MaskFeat_PT", "masked_ssl/k400_MVITv2_S_16x4_MaskFeat_PT.yaml",
                       "slowfast_b200.nets.maskfeat:B200MaskMViT"),
    # the shipped MaskFeat yaml as is: MViTv1-style blocks (DIM_MUL_IN_ATT False: channel expansion in the MLP)
    "maskfeat_s_shipped_small": ("MVITv2_S_16x4_MaskFeat_PT", "masked_ssl/k400_MVITv2_S_16x4_MaskFeat_PT.yaml",
                                 "slowfast_b200.nets.maskfeat:B200MaskMViT"),
}
EXTRA_OVERRIDES = {"maskfeat_s_224": ["MVIT.DIM_MUL_IN_ATT", True],
                   "maskfeat_s_shipped_small": ["MVIT.DIM_MUL_IN_ATT", False, "DATA.NUM_FRAMES", 8,
                                                "DATA.TRAIN_CROP_SIZE", 64, "DATA.TEST_CROP_SIZE", 64]}


def _engine_class(spec):
    import importlib
    mod, cls = spec.split(":")
    return getattr(importlib.import_module(mod), cls)


@pytest.mark.parametrize("gold_name", sorted(MODELS))
def test_state_dict_matches_reference_keys(gold_name):
    """Every engine model exposes exactly the reference's state_dict (names, order, shapes) - the checkpoint and
    optimizer-grouping contract of SURVEY.md section 8b."""
    from slowfast_b200.config import get_cfg
    preset, _, spec = MODELS[gold_name]
    gold = torch.load(os.path.join(GOLDEN, gold_name + ".pt"))
    cfg = get_cfg(preset)
    ov = EXTRA_OVERRIDES.get(gold_name, [])
    for k, v in zip(ov[0::2], ov[1::2]):
        sec, key = k.split(".")
        cfg[sec][key] = v
    m = _engine_class(spec)(cfg)
    keys = [(k, tuple(v.shape)) for k, v in m.state_dict().items()]
    assert keys == [(k, tuple(shape)) for k, shape in gold["keys"]]


@pytest.mark.parametrize("gold_name", sorted(MODELS))
def test_init_is_bit_identical_to_reference_when_available(gold_name):
    from slowfast_b200.config import get_cfg
    preset, yaml, spec = MODELS[gold_name]
    ov = EXTRA_OVERRIDES.get(gold_name, [])
    ref = _reference_init(yaml, ov)
    torch.manual_seed(ref["cfg"]["RNG_SEED"])
    cfg = get_cfg(preset)
    for k, v in zip(ov[0::2], ov[1::2]):
        sec, key = k.split(".")
        cfg[sec][key] = v
    _assert_same_init(_engine_class(spec)(cfg).state_dict(), ref)
    torch.manual_seed(ref["cfg"]["RNG_SEED"])
    _assert_same_init(_engine_class(spec)(_reference_cfg(yaml, ref, ov)).state_dict(), ref)  # the reference's config as-is


def test_x3d_widths_and_parameter_count():
    from slowfast_b200.config import get_cfg
    from slowfast_b200.nets.x3d import B200X3D, se_width
    m = B200X3D(get_cfg("X3D_M"))
    assert [getattr(m, f"s{i}").num_blocks for i in range(2, 6)] == [3, 5, 11, 7]
    assert [getattr(m, f"s{i}").pathway0_res0._dim_inner for i in range(2, 6)] == [54, 108, 216, 432]
    assert [se_width(c, 0.0625) for c in (54, 108, 216, 432)] == [8, 8, 16, 32]
    assert sum(p.numel() for p in m.parameters()) == 3794322  # 3.79 M (X3D-M, Kinetics-400 head)


MORE_YAMLS = ["Kinetics/SLOW_8x8_R50.yaml", "Kinetics/SLOW_4x16_R50.yaml", "Kinetics/I3D_8x8_R50.yaml",
              "Kinetics/I3D_8x8_R101.yaml", "Kinetics/SLOWFAST_4x16_R50.yaml", "Kinetics/X3D_S.yaml",
              "Kinetics/X3D_XS.yaml", "Kinetics/X3D_L.yaml", "Kinetics/MVITv2_B_32x3.yaml",
              "masked_ssl/k400_MVITv2_L_16x4_MaskFeat_PT.yaml"]


@pytest.mark.parametrize("yaml", MORE_YAMLS)
def test_engine_accepts_other_reference_yamls(yaml):
    """The engine classes are built straight from the reference's resolved config for the other shipped recipes of the
    same model families (Slow / I3D / R101, SlowFast 4x16, X3D-XS/S/L, MViTv2-B, MaskFeat MViTv2-L): identical
    state_dict (names, order, shapes) and bit-identical initialisation under the same seed."""
    from slowfast_b200.integration import ENGINE_CLASSES, _resolve
    ref = _reference_init(yaml)
    rcfg = _reference_cfg(yaml, ref)
    cls = _resolve(ENGINE_CLASSES[rcfg.MODEL.MODEL_NAME])
    torch.manual_seed(rcfg.RNG_SEED)
    _assert_same_init(cls(rcfg).state_dict(), ref)


def test_kernel_selection_predicates_without_a_gpu():
    """Shape predicates of the specialised kernels are pure host logic in the C library: the Toeplitz stem takes the fast
    pathway's geometry (3 -> 8, [kt,7,7], stride (1,2,2), pad 3) and nothing else; the fused attention takes head_dim 96 with the
    8x7x7 key grid only."""
    from slowfast_b200 import lib as L, ops
    lib = L.load()
    ok = ops.stem8_supported
    assert ok(3, 8, (5, 7, 7), (1, 2, 2), (2, 3, 3), 32, 224, 224)          # SlowFast fast pathway
    assert ok(3, 8, (5, 7, 7), (1, 2, 2), (2, 3, 3), 8, 64, 64)             # test fixtures
    assert ok(3, 8, (1, 7, 7), (1, 2, 2), (0, 3, 3), 4, 48, 32)
    assert not ok(3, 64, (1, 7, 7), (1, 2, 2), (0, 3, 3), 8, 224, 224)      # slow pathway / C2D: 64 output channels
    assert not ok(3, 8, (5, 7, 7), (1, 2, 2), (2, 3, 3), 32, 256, 256)      # test crop 256: 128 output columns > 120
    assert not ok(3, 8, (5, 7, 7), (1, 2, 2), (2, 3, 3), 32, 224, 232)      # width not a multiple of 16
    assert not ok(3, 8, (5, 3, 3), (1, 2, 2), (2, 1, 1), 32, 224, 224)      # X3D-like 3x3
    assert ops.stem8_plane_dims(8, 32, 224, 224) == (8, 64, 112, 120, 8)
    assert lib.sfb_attn_fwd_supported(393, 96, 8, 7, 7) in (0, 1)          # (0 when SFB_ATTN_FUSED=0)
    assert not lib.sfb_attn_fwd_supported(1569, 96, 8, 14, 14)
    assert not lib.sfb_attn_fwd_supported(393, 64, 8, 7, 7)
    assert int(lib.sfb_attn_fwd_selector_bytes()) == 400 * 64 * 2
