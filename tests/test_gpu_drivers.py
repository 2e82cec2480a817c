"""The north star's drop-in claim, executed: the reference's UNMODIFIED ``tools/train_net.py::train`` and
``tools/test_net.py::test`` run on the GPU with the engine models served by ``slowfast.models.build_model``
(MODEL_REGISTRY swap, INTEGRATION.md section 2), and produce the losses / test scores the STOCK models produce in the same
drivers on the same synthetic clips.

What runs unmodified: build_model (+ .cuda(), + the DDP wrap for NUM_GPUS 2), construct_optimizer (BN / zero-WD parameter
grouping by module type), the loaders, train_epoch (autocast context, GradScaler, grad-norm clipping, LR policy, meters),
save_checkpoint / load_test_checkpoint (state_dict key parity), eval_epoch, perform_test (multi-view ensembling).
Reference tree: oracle/_ref (copied by build(), oracle/install_ref.py) through oracle/refshim.py; tests skip when it is
absent.
"""
import os
import tempfile

import pytest
import torch

pytestmark = pytest.mark.gpu

CASES = {
    "slowfast": ("Kinetics/SLOWFAST_8x8_R50.yaml", 16, ["MODEL.DROPOUT_RATE", 0.0, "SOLVER.BASE_LR", 0.002]),
    "c2d": ("Kinetics/C2D_8x8_R50.yaml", 8, ["MODEL.DROPOUT_RATE", 0.0, "SOLVER.BASE_LR", 0.002]),
    "x3d": ("Kinetics/X3D_M.yaml", 4, ["MODEL.DROPOUT_RATE", 0.0, "SOLVER.BASE_LR", 0.002]),
    "mvit": ("Kinetics/MVITv2_S_16x4.yaml", 8,
             ["MODEL.DROPOUT_RATE", 0.0, "MVIT.DROPPATH_RATE", 0.0, "MIXUP.ENABLE", False, "AUG.ENABLE", False,
              "AUG.NUM_SAMPLE", 1, "MODEL.LOSS_FUNC", "cross_entropy", "SOLVER.BASE_LR", 1e-4]),
}


@pytest.fixture(autouse=True)
def _restore_stock_registry():
    """The driver tests swap the reference's MODEL_REGISTRY entries for the engine classes; later test modules (same process)
    build REFERENCE models through build_model and must get the stock classes back."""
    yield
    import driver_harness as H
    if H.setup_reference() is not None:
        H.use_engine(False)


def _harness():
    import driver_harness as H
    if H.setup_reference() is None:
        pytest.skip("no reference tree (build() copies it into oracle/_ref when a checkout is readable)")
    return H


def _run(H, family, engine, extra=(), num_gpus=1):
    yaml, frames, over = CASES[family]
    H.use_engine(engine)
    cfg = H.driver_cfg(yaml, num_gpus, list(over) + list(extra), frames=frames, batch=4)
    torch.backends.cudnn.allow_tf32 = False          # the stock arm must be the reference's fp32 arithmetic
    torch.backends.cuda.matmul.allow_tf32 = False
    rec_train, _ = H.run_train(cfg)
    rec_test, result = (None, None)
    if not cfg.MASK.ENABLE:
        rec_test, result = H.run_test(cfg)           # loads the checkpoint train() just wrote into OUTPUT_DIR
    return cfg, rec_train, rec_test, result


@pytest.mark.parametrize("family", list(CASES))
def test_unmodified_train_and_test_drivers_match_stock_models(family, cuda_device):
    H = _harness()
    _, st_train, st_test, _ = _run(H, family, engine=False)
    cfg, en_train, en_test, result = _run(H, family, engine=True)
    from slowfast.models import build_model
    m = build_model(cfg)
    assert type(m).__name__.startswith("B200"), type(m)
    assert len(en_train["train"]) == len(st_train["train"]) == 3
    for i, (a, b) in enumerate(zip(en_train["train"], st_train["train"])):
        rel = abs(a["loss"] - b["loss"]) / abs(b["loss"])
        gn = abs(a["grad_norm"] - b["grad_norm"]) / abs(b["grad_norm"])
        print(f"{family}: iter {i} loss engine {a['loss']:.6f} stock {b['loss']:.6f} (rel {rel:.1e}); grad-norm rel {gn:.1e}")
        assert rel < (1e-3 if i == 0 else 1e-2), (i, a, b)
        assert gn < 0.1, (i, a["grad_norm"], b["grad_norm"])
        assert a["lr"] == b["lr"] and a["mb"] == b["mb"]
    assert len(en_train["val"]) == len(st_train["val"]) > 0          # eval_epoch ran on the engine (eval-mode program)
    # test(): softmax scores of every view from the checkpoint each run saved (weights differ by 3 SGD steps of drift)
    assert len(en_test["test"]) == len(st_test["test"]) > 0
    for a, b in zip(en_test["test"], st_test["test"]):
        assert torch.equal(a["ids"], b["ids"]) and torch.equal(a["labels"], b["labels"])
        assert a["preds"].shape == b["preds"].shape
        assert torch.allclose(a["preds"].sum(1), torch.ones(a["preds"].shape[0]), atol=1e-4)
        assert ((a["preds"] - b["preds"]).abs().max() / b["preds"].abs().max()).item() < 5e-2
    assert "Top5 Acc" in result


def test_mixed_precision_flag_through_the_unmodified_driver(cuda_device):
    """TRAIN.MIXED_PRECISION True: train_epoch wraps the step in torch.cuda.amp.autocast and scales the loss with a
    GradScaler (train_net.py:113,152-172).  The engine's autograd node keeps its own precision (parity mode), so the
    first-iteration loss must equal the non-AMP run's; scaled gradients must come back unscaled (finite grad norm)."""
    H = _harness()
    _, base, _, _ = _run(H, "slowfast", engine=True)
    _, amp, _, _ = _run(H, "slowfast", engine=True, extra=["TRAIN.MIXED_PRECISION", True])
    a, b = amp["train"][0], base["train"][0]
    assert abs(a["loss"] - b["loss"]) / abs(b["loss"]) < 1e-3, (a, b)
    assert abs(a["grad_norm"] - b["grad_norm"]) / abs(b["grad_norm"]) < 2e-2, (a, b)
    assert all(torch.isfinite(torch.tensor(r["loss"])) for r in amp["train"])


def test_maskfeat_pretraining_through_the_unmodified_driver(cuda_device):
    """MASK.ENABLE: train_epoch unpacks (preds, labels) from the model and feeds MultipleMSELoss (train_net.py:130-131)."""
    H = _harness()
    H.use_engine(True)
    over = ["SOLVER.BASE_LR", 1e-4, "MVIT.DIM_MUL_IN_ATT", True]
    cfg_e = H.driver_cfg("masked_ssl/k400_MVITv2_S_16x4_MaskFeat_PT.yaml", 1, over, frames=8, batch=4)
    en, _ = H.run_train(cfg_e)
    H.use_engine(False)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    cfg_s = H.driver_cfg("masked_ssl/k400_MVITv2_S_16x4_MaskFeat_PT.yaml", 1, over, frames=8, batch=4)
    st, _ = H.run_train(cfg_s)
    for i, (a, b) in enumerate(zip(en["train"], st["train"])):
        rel = abs(a["loss"] - b["loss"]) / abs(b["loss"])
        print(f"maskfeat: iter {i} loss engine {a['loss']:.6f} stock {b['loss']:.6f} (rel {rel:.1e})")
        assert rel < (1e-3 if i == 0 else 1e-2)


@pytest.mark.parametrize("engine", [True])
def test_two_gpu_ddp_through_build_model(engine, cuda_device):
    """NUM_GPUS 2: build_model wraps the module in DistributedDataParallel (build.py:66-76); the engine's single autograd
    node hands every parameter gradient to DDP's reducer.  Compared with the stock model under the same DDP driver."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    H = _harness()
    import torch.multiprocessing as mp
    recs = {}
    for eng in (False, True):
        yaml, frames, over = CASES["slowfast"]
        out_dir = tempfile.mkdtemp(prefix="sfb_ddp_")
        cfg_args = dict(yaml=yaml, num_gpus=2, overrides=list(over), out_dir=out_dir, batch=4, frames=frames)
        ret = os.path.join(out_dir, "rec.pt")
        port = 29610 + (1 if eng else 0)
        mp.spawn(H._worker, nprocs=2, args=(2, "train", f"tcp://127.0.0.1:{port}", cfg_args, eng, ret))
        recs[eng] = torch.load(ret, weights_only=False)
    for i, (a, b) in enumerate(zip(recs[True]["train"], recs[False]["train"])):
        rel = abs(a["loss"] - b["loss"]) / abs(b["loss"])
        print(f"ddp2: iter {i} loss engine {a['loss']:.6f} stock {b['loss']:.6f} (rel {rel:.1e})")
        assert rel < (1e-3 if i == 0 else 1e-2)
        assert abs(a["grad_norm"] - b["grad_norm"]) / abs(b["grad_norm"]) < 0.1


def test_precise_bn_through_the_unmodified_driver(cuda_device):
    """tools/train_net.py calculate_and_update_precise_bn (:425-446) -> fvcore update_bn_stats (stand-in restating the
    published algorithm in oracle/refshim.py): BN momentum is set to 1.0, forward passes run in train mode under no_grad,
    the per-batch statistics left in the (real nn.BatchNorm3d) buffers are averaged and ASSIGNED back as new tensors.
    Engine vs stock model from the same state; afterwards a train step must still work (the engine re-captures its
    programs when buffer pointers change)."""
    H = _harness()
    from slowfast.models import build_model
    from tools.train_net import calculate_and_update_precise_bn
    from slowfast.datasets import loader
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yaml, frames, over = CASES["slowfast"]
    stats = {}
    for eng in (False, True):
        H.use_engine(eng)
        cfg = H.driver_cfg(yaml, 1, list(over), frames=frames, batch=4)
        torch.manual_seed(0)
        model = build_model(cfg)
        if eng:
            assert type(model).__name__ == "B200SlowFast"
            # two ordinary train-mode forwards first, so that precise-BN meets already-captured programs
            x = [t.cuda() for t in next(iter(loader.construct_loader(cfg, "train")))[0]]
            for _ in range(3):
                model.train()
                model(x).sum().backward()
        else:
            ref_state = {k: v.clone() for k, v in model.state_dict().items()}
        if eng:
            model.load_state_dict(ref_state)
        pl = loader.construct_loader(cfg, "train", is_precise_bn=True)
        model.train()
        torch.manual_seed(1234)   # the loader shuffles (RandomSampler): both arms must see the same three batches
        calculate_and_update_precise_bn(pl, model, num_iters=3, use_gpu=True)
        stats[eng] = {k: v.detach().cpu().clone() for k, v in model.state_dict().items() if "running_" in k}
        if eng:
            model.train()
            for _ in range(3):
                out = model(x)
                out.sum().backward()
            assert torch.isfinite(out).all()
    for k in stats[False]:
        a, b = stats[True][k], stats[False][k]
        assert (a - b).abs().max().item() < 2e-3 * b.abs().max().item(), (k, (a - b).abs().max().item())
