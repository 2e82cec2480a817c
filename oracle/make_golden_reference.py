"""TEST INFRASTRUCTURE.  Needs the unmodified reference (see oracle/refshim.py); CPU only:

    python oracle/make_golden_reference.py

Stores what the CPU tests compare against the reference itself, so that they run without it:
  tests/golden/reference_init.pt    for each recipe (yaml + overrides): the sections of the reference's resolved config
                                    that the model builders read (plain nested dict), a digest of its state_dict layout
                                    (names, shapes, order) and, in that order, an 8-byte SHA-256 prefix of every freshly
                                    initialised entry (tests/test_host.py: bit-identical initialisation);
  tests/golden/reference_logits.pt  the reference modules' logits on seeded fixtures (tests/test_oracle.py: the oracle
                                    restatement in train and eval mode, and the fully convolutional test-crop head); the
                                    state layout is the one stored in the named golden case.
"""
from __future__ import annotations

import hashlib
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import refshim, torch_oracle as TO  # noqa: E402

# (yaml, overrides) of every recipe whose initialisation tests/test_host.py checks
INIT_CASES = [
    ("Kinetics/SLOWFAST_8x8_R50.yaml", []),
    ("Kinetics/C2D_8x8_R50.yaml", []),
    ("Kinetics/MVITv2_S_16x4.yaml", []),
    ("Kinetics/X3D_M.yaml", []),
    ("masked_ssl/k400_MVITv2_S_16x4_MaskFeat_PT.yaml", ["MVIT.DIM_MUL_IN_ATT", True]),
    ("masked_ssl/k400_MVITv2_S_16x4_MaskFeat_PT.yaml", ["MVIT.DIM_MUL_IN_ATT", False, "DATA.NUM_FRAMES", 8,
                                                        "DATA.TRAIN_CROP_SIZE", 64, "DATA.TEST_CROP_SIZE", 64]),
    ("Kinetics/SLOW_8x8_R50.yaml", []), ("Kinetics/SLOW_4x16_R50.yaml", []), ("Kinetics/I3D_8x8_R50.yaml", []),
    ("Kinetics/I3D_8x8_R101.yaml", []), ("Kinetics/SLOWFAST_4x16_R50.yaml", []), ("Kinetics/X3D_S.yaml", []),
    ("Kinetics/X3D_XS.yaml", []), ("Kinetics/X3D_L.yaml", []), ("Kinetics/MVITv2_B_32x3.yaml", []),
    ("masked_ssl/k400_MVITv2_L_16x4_MaskFeat_PT.yaml", []),
]
SMALL = ["DATA.NUM_FRAMES", 8, "DATA.TRAIN_CROP_SIZE", 64, "MODEL.DROPOUT_RATE", 0.0]
# config sections read by slowfast_b200's model builders
CFG_SECTIONS = ("MODEL", "DATA", "RESNET", "SLOWFAST", "X3D", "MVIT", "MASK", "NONLOCAL", "DETECTION", "BN", "MULTIGRID",
                "SOLVER", "RNG_SEED", "NUM_GPUS")


def init_key(yaml: str, overrides) -> str:
    return yaml + "|" + " ".join(map(str, overrides))


def tensor_digest(t: torch.Tensor) -> bytes:
    return hashlib.sha256(t.detach().contiguous().cpu().numpy().tobytes()).digest()[:8]


def layout_digest(state) -> str:
    return hashlib.sha256(";".join(f"{k}:{tuple(v.shape)}" for k, v in state.items()).encode()).hexdigest()


def plain(node):
    if isinstance(node, dict):
        return {k: plain(v) for k, v in node.items()}
    if isinstance(node, (list, tuple)):
        return type(node)(plain(v) for v in node)
    return node


def init_case(yaml, overrides):
    rcfg = refshim.load_cfg(yaml, overrides)
    sd = refshim.build_reference_model(rcfg).state_dict()
    return dict(cfg={k: plain(rcfg[k]) for k in CFG_SECTIONS if k in rcfg}, layout=layout_digest(sd),
                values=b"".join(tensor_digest(v) for v in sd.values()))


def layout_of(state, golden_case: str) -> str:
    """``golden_case``, after checking that its stored state layout is ``state``'s."""
    gold = torch.load(os.path.join(ROOT, "tests", "golden", golden_case + ".pt"))
    assert [(k, tuple(v.shape)) for k, v in state.items()] == [(k, tuple(s)) for k, s in gold["keys"]], golden_case
    return golden_case


def live_logits():
    out = {}
    cfg = refshim.load_cfg("Kinetics/SLOWFAST_8x8_R50.yaml", SMALL)
    model = refshim.build_reference_model(cfg)
    state = TO.fixture_state(model.state_dict(), 99)
    model.load_state_dict(state)
    model.train()
    inputs = TO.synthetic_inputs(cfg, 1, 5)
    train = model([t.clone() for t in inputs]).detach()
    model.eval()
    out["slowfast_train_eval"] = dict(yaml="Kinetics/SLOWFAST_8x8_R50.yaml", overrides=SMALL, state_seed=99, batch=1,
                                      in_seed=5, layout=layout_of(state, "slowfast_r50_small"),
                                      train=train, eval=model([t.clone() for t in inputs]).detach())
    for yaml, layout in (("Kinetics/SLOWFAST_8x8_R50.yaml", "slowfast_r50_small"),
                         ("Kinetics/C2D_8x8_R50.yaml", "c2d_r50_small")):
        over = SMALL + ["DATA.TEST_CROP_SIZE", 96]
        cfg = refshim.load_cfg(yaml, over)
        model = refshim.build_reference_model(cfg)
        state = TO.fixture_state(model.state_dict(), 17)
        model.load_state_dict(state)
        model.eval()
        inputs = TO.synthetic_inputs(cfg, 2, 6, crop=96)
        with torch.no_grad():
            ref = model([t.clone() for t in inputs])
        out["eval_head|" + yaml] = dict(yaml=yaml, overrides=over, state_seed=17, batch=2, in_seed=6, crop=96,
                                        layout=layout_of(state, layout), eval=ref)
    return out


def main():
    torch.set_num_threads(os.cpu_count())
    gdir = os.path.join(ROOT, "tests", "golden")
    init = {init_key(y, o): init_case(y, o) for y, o in INIT_CASES}
    logits = live_logits()
    for name, obj in (("reference_init.pt", init), ("reference_logits.pt", logits)):
        path = os.path.join(gdir, name)
        torch.save(obj, path)
        print(f"wrote {path} ({os.path.getsize(path) / 1024:.1f} KiB)")


if __name__ == "__main__":
    main()
