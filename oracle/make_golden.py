"""TEST INFRASTRUCTURE.  Run in the BUILD CONTAINER (needs /root/reference):

    python oracle/make_golden.py

For each golden case it (1) builds the UNMODIFIED reference model through ``oracle/refshim.py``, loads the seeded
fixture state, runs forward + backward on seeded synthetic clips (CPU, fp32); (2) checks that the restatement in
``oracle/torch_oracle.py`` reproduces the reference's logits, parameter gradients and updated BN running statistics;
(3) writes a small golden file (logits, per-parameter gradient digests, running-stat digests) to ``tests/golden``.
Nothing here runs on the GPU box; the committed golden files are what travels.
"""
from __future__ import annotations

import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import refshim, torch_oracle as TO  # noqa: E402

CASES = {
    # name: (yaml, overrides, batch, input seed, state seed)
    "slowfast_r50_small": ("Kinetics/SLOWFAST_8x8_R50.yaml",
                           ["DATA.NUM_FRAMES", 16, "DATA.TRAIN_CROP_SIZE", 64, "MODEL.DROPOUT_RATE", 0.0], 2, 11, 5),
    "slowfast_r50_224": ("Kinetics/SLOWFAST_8x8_R50.yaml", ["MODEL.DROPOUT_RATE", 0.0], 2, 12, 6),
    "mvitv2_s_small": ("Kinetics/MVITv2_S_16x4.yaml",
                       ["DATA.NUM_FRAMES", 8, "DATA.TRAIN_CROP_SIZE", 64, "DATA.TEST_CROP_SIZE", 64, "MODEL.DROPOUT_RATE", 0.0,
                        "MVIT.DROPPATH_RATE", 0.0], 2, 31, 32),
    "mvitv2_s_224": ("Kinetics/MVITv2_S_16x4.yaml", ["MODEL.DROPOUT_RATE", 0.0, "MVIT.DROPPATH_RATE", 0.0], 1, 33, 34),
    # MaskFeat on the MViTv2-S encoder (DIM_MUL_IN_ATT True: the engine's MViT block; the shipped yaml leaves the
    # MViTv1-style default False, which only moves the channel expansion from the attention to the MLP)
    "maskfeat_s_small": ("masked_ssl/k400_MVITv2_S_16x4_MaskFeat_PT.yaml",
                         ["MVIT.DIM_MUL_IN_ATT", True, "DATA.NUM_FRAMES", 8, "DATA.TRAIN_CROP_SIZE", 64,
                          "DATA.TEST_CROP_SIZE", 64], 2, 51, 52),
    # the shipped yaml as is (MViTv1-style blocks: channel expansion in the MLP)
    "maskfeat_s_shipped_small": ("masked_ssl/k400_MVITv2_S_16x4_MaskFeat_PT.yaml",
                                 ["DATA.NUM_FRAMES", 8, "DATA.TRAIN_CROP_SIZE", 64, "DATA.TEST_CROP_SIZE", 64], 2, 55, 56),
    "maskfeat_s_224": ("masked_ssl/k400_MVITv2_S_16x4_MaskFeat_PT.yaml", ["MVIT.DIM_MUL_IN_ATT", True], 1, 53, 54),
    "x3d_m_small": ("Kinetics/X3D_M.yaml",
                    ["DATA.NUM_FRAMES", 4, "DATA.TRAIN_CROP_SIZE", 64, "MODEL.DROPOUT_RATE", 0.0], 2, 41, 42),
    "x3d_m_224": ("Kinetics/X3D_M.yaml", ["MODEL.DROPOUT_RATE", 0.0], 1, 43, 44),
    "slow_r50_small": ("Kinetics/SLOW_8x8_R50.yaml",
                       ["DATA.NUM_FRAMES", 8, "DATA.TRAIN_CROP_SIZE", 64, "MODEL.DROPOUT_RATE", 0.0], 2, 23, 24),
    "i3d_r50_small": ("Kinetics/I3D_8x8_R50.yaml",
                      ["DATA.NUM_FRAMES", 8, "DATA.TRAIN_CROP_SIZE", 64, "MODEL.DROPOUT_RATE", 0.0], 2, 25, 26),
    "c2d_r50_small": ("Kinetics/C2D_8x8_R50.yaml",
                      ["DATA.NUM_FRAMES", 8, "DATA.TRAIN_CROP_SIZE", 64, "MODEL.DROPOUT_RATE", 0.0], 2, 21, 22),
    # MViTv2-B (24 blocks, 32 frames): BASELINE config 5's encoder
    "mvitv2_b_small": ("Kinetics/MVITv2_B_32x3.yaml",
                       ["DATA.NUM_FRAMES", 8, "DATA.TRAIN_CROP_SIZE", 64, "DATA.TEST_CROP_SIZE", 64, "MODEL.DROPOUT_RATE", 0.0,
                        "MVIT.DROPPATH_RATE", 0.0], 2, 61, 62),
    "mvitv2_b_224": ("Kinetics/MVITv2_B_32x3.yaml", ["MODEL.DROPOUT_RATE", 0.0, "MVIT.DROPPATH_RATE", 0.0], 1, 63, 64),
    # BASELINE config 5 (MViTv2-B MaskFeat 32x224x224): composed per SURVEY.md section 3.5 - see MASKFEAT_B below
    "maskfeat_b_small": ("masked_ssl/k400_MVITv2_S_16x4_MaskFeat_PT.yaml", "MASKFEAT_B_SMALL", 2, 65, 66),
    "maskfeat_b_224": ("masked_ssl/k400_MVITv2_S_16x4_MaskFeat_PT.yaml", "MASKFEAT_B", 1, 67, 68),
}

# the MVIT block of configs/Kinetics/MVITv2_B_32x3.yaml on top of the S MaskFeat yaml (MASK / AUG / SOLVER blocks), last Q
# stride [21,1,2,2] -> [21,1,1,1], PRETRAIN_DEPTH [23], mask cube window 16x7x7 (= slowfast_b200.config MVITv2_B_32x3_MaskFeat_PT)
MASKFEAT_B = ["DATA.NUM_FRAMES", 32, "MVIT.DEPTH", 24, "MVIT.DIM_MUL", [[2, 2.0], [5, 2.0], [21, 2.0]],
              "MVIT.HEAD_MUL", [[2, 2.0], [5, 2.0], [21, 2.0]],
              "MVIT.POOL_Q_STRIDE", [[i, 1, 2, 2] if i in (2, 5) else [i, 1, 1, 1] for i in range(24)],
              "MVIT.DIM_MUL_IN_ATT", True, "MVIT.MLP_RATIO", 4.0, "MASK.PRETRAIN_DEPTH", [23],
              "AUG.MASK_WINDOW_SIZE", [16, 7, 7]]
NAMED_OVERRIDES = {
    "MASKFEAT_B": MASKFEAT_B,
    "MASKFEAT_B_SMALL": MASKFEAT_B + ["DATA.NUM_FRAMES", 8, "DATA.TRAIN_CROP_SIZE", 64, "DATA.TEST_CROP_SIZE", 64],
}
# cases that additionally store SAMPLED parameter gradients (256 evenly spaced elements per parameter) and the
# reference's own fp32-vs-fp64 error on those samples (the envelope a parity-mode engine is held to a multiple of)
SAMPLED = {"slowfast_r50_224", "x3d_m_224", "slowfast_r50_small", "x3d_m_small"}


def sample_idx(numel: int, k: int = 256) -> torch.Tensor:
    return torch.linspace(0, numel - 1, min(numel, k)).round().long()


def digest(t: torch.Tensor):
    f = t.detach().double().flatten()
    return dict(norm=f.norm().item(), sum=f.sum().item(), head=f[:4].tolist(), numel=f.numel())


LABELS_WHOLE = 100000   # HOG targets up to this many values are stored whole; larger ones as a seeded sample of rows
LABELS_SAMPLED = 50000  # (so that a golden file stays under 1 MB)


def store_labels(gold, labels: torch.Tensor) -> None:
    """``labels``, or for large targets a fixed seeded sample of its rows (``label_rows``), plus the digest of all."""
    labels = labels.detach()
    gold["labels_digest"] = digest(labels)
    if labels.numel() <= LABELS_WHOLE:
        gold["labels"] = labels.clone()
        return
    k = max(1, LABELS_SAMPLED // labels[0].numel())
    rows = torch.randperm(labels.shape[0], generator=torch.Generator().manual_seed(0))[:k].sort().values
    gold["label_rows"] = rows
    gold["labels"] = labels[rows].clone()


def run_case(name, yaml, overrides, batch, in_seed, st_seed):
    if isinstance(overrides, str):
        overrides = NAMED_OVERRIDES[overrides]
    cfg = refshim.load_cfg(yaml, overrides)
    model = refshim.build_reference_model(cfg)
    state = TO.fixture_state(model.state_dict(), st_seed)
    model.load_state_dict(state, strict=True)
    model.train()
    ref_labels = None
    if cfg.MASK.ENABLE:  # MaskFeat: x = [frames, meta, mask] -> (preds, labels)
        inputs = TO.maskfeat_inputs(cfg, batch, in_seed)
        preds, labels = model([inputs[0].clone(), torch.Tensor(), inputs[1].clone()])
        assert len(preds) == 1 and labels[0][1] == 1.0 and labels[0][2] == "mse"
        logits, ref_labels = preds[0], labels[0][0]
        o_labels = TO.maskfeat_labels(cfg, inputs[0], inputs[1])
        err_lab = (o_labels - ref_labels).abs().max().item()
        print(f"[{name}] oracle HOG labels vs reference: max abs {err_lab:.2e} over {tuple(ref_labels.shape)}")
        assert err_lab < 1e-6
    else:
        inputs = TO.synthetic_inputs(cfg, batch, in_seed)
        logits = model([t.clone() for t in inputs])
    dlogits = torch.randn(logits.shape, generator=torch.Generator().manual_seed(in_seed + 1000))
    logits.backward(dlogits)
    ref_grads = {k: p.grad for k, p in model.named_parameters()}
    ref_state = model.state_dict()

    # ---- pin the restatement against the reference itself
    o_logits, o_grads = TO.forward_backward(cfg, state, inputs, dlogits)
    work = {k: v.clone() for k, v in state.items()}
    TO.forward(cfg, work, inputs, True)
    err_logits = (o_logits - logits.detach()).abs().max().item() / logits.detach().abs().max().item()
    # gradients that are zero in exact arithmetic (e.g. MViT norm_k.bias: a constant key shift cancels in the softmax)
    # are pure rounding noise in ANY implementation: compare against a floor of 1e-2 x the median gradient norm
    norms = sorted(g.norm().item() for g in ref_grads.values())
    floor = 1e-2 * norms[len(norms) // 2]
    err_grad = max(((o_grads[k] - ref_grads[k]).norm() / ref_grads[k].norm().clamp_min(floor)).item()
                   for k in ref_grads)
    err_rs = max([((work[k] - ref_state[k]).abs().max() / ref_state[k].abs().max().clamp_min(1e-20)).item()
                  for k in ref_state if "running_" in k] + [0.0])
    print(f"[{name}] oracle vs reference: logits rel {err_logits:.2e}  worst param-grad rel-L2 {err_grad:.2e}  "
          f"running stats rel {err_rs:.2e}")
    assert err_logits < 1e-5 and err_grad < 1e-4 and err_rs < 1e-5, "oracle restatement disagrees with the reference"

    gold = dict(
        case=name, yaml=yaml, overrides=overrides, batch=batch, in_seed=in_seed, st_seed=st_seed,
        logits=logits.detach().clone(),
        grads={k: digest(g) for k, g in ref_grads.items()},
        grad_norm_floor=floor,
        running={k: digest(v) for k, v in ref_state.items() if "running_" in k},
        keys=[(k, tuple(v.shape)) for k, v in ref_state.items()],
        oracle_check=dict(logits=err_logits, grads=err_grad, running=err_rs),
        torch=str(torch.__version__),
    )
    if name in SAMPLED:
        # the reference's OWN fp32 rounding error: same modules, same state, run in fp64
        model64 = refshim.build_reference_model(cfg).double()
        model64.load_state_dict({k: (v.double() if v.is_floating_point() else v) for k, v in state.items()})
        model64.train()
        l64 = model64([t.double() for t in inputs])
        l64.backward(dlogits.double())
        g64 = {k: p.grad for k, p in model64.named_parameters()}
        gold["grad_samples"] = {k: g.flatten()[sample_idx(g.numel())].clone() for k, g in ref_grads.items()}
        env = {}
        for k, g in ref_grads.items():
            i = sample_idx(g.numel())
            a, b = g.flatten()[i].double(), g64[k].flatten()[i]
            env[k] = ((a - b).norm() / b.norm().clamp_min(1e-30)).item()
        gold["grad_env"] = env
        gold["logits_env"] = ((logits.detach().double() - l64.detach()).abs().max() / l64.detach().abs().max()).item()
        e = sorted(env.values())
        print(f"[{name}] reference fp32 vs fp64: logits {gold['logits_env']:.2e}; sampled-gradient rel-L2 median "
              f"{e[len(e) // 2]:.2e} max {e[-1]:.2e}")
    if ref_labels is not None:
        store_labels(gold, ref_labels)
    out = os.path.join(ROOT, "tests", "golden", name + ".pt")
    torch.save(gold, out)
    print(f"[{name}] wrote {out} ({os.path.getsize(out) / 1024:.1f} KiB)")


def main():
    torch.set_num_threads(os.cpu_count())
    only = sys.argv[1:] or list(CASES)
    for name in only:
        run_case(name, *CASES[name])


if __name__ == "__main__":
    main()
