"""TEST INFRASTRUCTURE: run the reference's UNMODIFIED drivers (tools/train_net.py ``train(cfg)``, tools/test_net.py
``test(cfg)``) on a synthetic dataset, with either the stock models or the engine's drop-ins behind
``slowfast.models.build_model``.

The reference tree comes from ``oracle/refshim.py`` (the byte-identical copy build() makes in oracle/_ref, or the
offline install under baseline/_ref).  Nothing in the reference is edited; the harness only
  * registers a ``Synthetic`` dataset class in the reference's DATASET_REGISTRY (its designated extension point,
    slowfast/datasets/build.py:8-13) and selects it with TRAIN.DATASET / TEST.DATASET,
  * calls ``slowfast_b200.integration.register(replace=True)`` (INTEGRATION.md section 2),
  * records what ``TrainMeter.update_stats`` / ``TestMeter.update_stats`` are handed (a wrapper around the reference's
    own methods), which is how the tests read the losses the driver computed.
"""
from __future__ import annotations

import contextlib
import os
import sys
import tempfile

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def setup_reference():
    from oracle import refshim
    if not refshim.reference_available():
        return None
    refshim.install()
    _register_synthetic()
    return refshim


def _register_synthetic():
    from slowfast.datasets import utils as dsutils
    from slowfast.datasets.build import DATASET_REGISTRY

    if "Synthetic" in DATASET_REGISTRY._obj_map:
        return

    class Synthetic(torch.utils.data.Dataset):
        """Seeded Kinetics-shaped clips: item i is randn(3, T, crop, crop) (SURVEY.md 8d) packed per pathway by the
        reference's own ``pack_pathway_output`` (datasets/utils.py:78); label i % classes; MaskFeat adds the cube mask
        the Kinetics loader generates (kinetics.py:450-452)."""

        def __init__(self, cfg, mode, num_retries=0):
            self.cfg, self.mode = cfg, mode
            self.views = cfg.TEST.NUM_ENSEMBLE_VIEWS * cfg.TEST.NUM_SPATIAL_CROPS if mode == "test" else 1
            n = int(os.environ.get("SFB_SYNTHETIC_VIDEOS", "12"))
            self._n = n * self.views

        @property
        def num_videos(self):
            return self._n

        def __len__(self):
            return self._n

        def __getitem__(self, i):
            cfg = self.cfg
            crop = cfg.DATA.TEST_CROP_SIZE if self.mode == "test" else cfg.DATA.TRAIN_CROP_SIZE
            g = torch.Generator().manual_seed(10007 * i + {"train": 1, "val": 2, "test": 3}[self.mode])
            frames = torch.randn(3, cfg.DATA.NUM_FRAMES, crop, crop, generator=g)
            inputs = dsutils.pack_pathway_output(cfg, frames)
            label = (i // self.views) % cfg.MODEL.NUM_CLASSES
            if cfg.MASK.ENABLE:
                t = cfg.DATA.NUM_FRAMES // cfg.MVIT.PATCH_STRIDE[0]
                mask = (torch.rand(t, 7, 7, generator=g) < cfg.AUG.MASK_RATIO).float()
                inputs = inputs + [torch.Tensor(), mask]
            return inputs, label, i, torch.zeros(1), {}  # index = clip id (TestMeter: video = id // num_clips)

    DATASET_REGISTRY._do_register("Synthetic", Synthetic)


def driver_cfg(yaml, num_gpus, overrides=(), out_dir=None, batch=4, crop=64, frames=None):
    refshim = setup_reference()
    from slowfast.config.defaults import assert_and_infer_cfg, get_cfg
    cfg = get_cfg()
    cfg.merge_from_file(os.path.join(refshim.REFERENCE_ROOT, "configs", yaml))
    base = ["NUM_GPUS", num_gpus, "TRAIN.DATASET", "synthetic", "TEST.DATASET", "synthetic", "TRAIN.BATCH_SIZE", batch,
            "TEST.BATCH_SIZE", batch, "DATA_LOADER.NUM_WORKERS", 0, "DATA_LOADER.PIN_MEMORY", num_gpus > 0,
            "SOLVER.MAX_EPOCH", 1, "SOLVER.WARMUP_EPOCHS", 0.0, "TRAIN.EVAL_PERIOD", 1, "TRAIN.CHECKPOINT_PERIOD", 1,
            "TRAIN.AUTO_RESUME", False, "LOG_MODEL_INFO", False, "BN.USE_PRECISE_STATS", False,
            "TEST.NUM_ENSEMBLE_VIEWS", 2, "TEST.NUM_SPATIAL_CROPS", 1, "TENSORBOARD.ENABLE", False,
            "DATA.TRAIN_CROP_SIZE", crop, "DATA.TEST_CROP_SIZE", crop, "LOG_PERIOD", 1,
            "OUTPUT_DIR", out_dir or tempfile.mkdtemp(prefix="sfb_driver_")]
    if frames is not None:
        base += ["DATA.NUM_FRAMES", frames]
    cfg.merge_from_list(base + list(overrides))
    return assert_and_infer_cfg(cfg)


@contextlib.contextmanager
def recorded_meters():
    """Wrap the reference's TrainMeter / ValMeter / TestMeter ``update_stats`` to record their arguments."""
    from slowfast.utils import meters
    rec = {"train": [], "val": [], "test": []}
    orig = (meters.TrainMeter.update_stats, meters.ValMeter.update_stats, meters.TestMeter.update_stats)

    def train_us(self, top1_err, top5_err, loss, lr, grad_norm, mb_size, multi_loss=None):
        rec["train"].append(dict(loss=float(loss), top1_err=top1_err, lr=lr, grad_norm=float(grad_norm), mb=mb_size))
        return orig[0](self, top1_err, top5_err, loss, lr, grad_norm, mb_size, multi_loss)

    def val_us(self, top1_err, top5_err, mb_size):
        rec["val"].append(dict(top1_err=top1_err, top5_err=top5_err, mb=mb_size))
        return orig[1](self, top1_err, top5_err, mb_size)

    def test_us(self, preds, labels, clip_ids):
        rec["test"].append(dict(preds=preds.detach().clone().cpu(), labels=labels.clone().cpu(), ids=clip_ids.clone().cpu()))
        return orig[2](self, preds, labels, clip_ids)

    meters.TrainMeter.update_stats, meters.ValMeter.update_stats, meters.TestMeter.update_stats = train_us, val_us, test_us
    try:
        yield rec
    finally:
        meters.TrainMeter.update_stats, meters.ValMeter.update_stats, meters.TestMeter.update_stats = orig


def use_engine(on: bool):
    """Point the reference's MODEL_REGISTRY at the engine classes (or back at the stock ones)."""
    import slowfast.models  # noqa: F401  (registers the stock models)
    from slowfast.models.build import MODEL_REGISTRY

    import slowfast_b200.integration as sfb
    stock = getattr(use_engine, "_stock", None)
    if stock is None:
        stock = {k: MODEL_REGISTRY._obj_map[k] for k in sfb.ENGINE_CLASSES if k in MODEL_REGISTRY._obj_map}
        use_engine._stock = stock
    if on:
        return sfb.register(replace=True)
    for k, v in stock.items():
        MODEL_REGISTRY._obj_map[k] = v
    return []


def run_train(cfg):
    from tools.train_net import train
    with recorded_meters() as rec:
        out = train(cfg)
    return rec, out


def run_test(cfg):
    from tools.test_net import test
    with recorded_meters() as rec:
        out = test(cfg)
    return rec, out


def _worker(local_rank, num_proc, func_name, init_method, cfg_args, engine, ret_path):  # pragma: no cover - spawned
    """Body of one DDP process for NUM_GPUS > 1 (mirrors slowfast/utils/multiprocessing.py run(): init the process group,
    set the device, call the unmodified driver function).  ``cfg_args`` = kwargs of ``driver_cfg`` (the stand-in CfgNode
    class is local to the shim and cannot be pickled, so every rank builds its own identical config)."""
    setup_reference()
    use_engine(engine)
    cfg = driver_cfg(**cfg_args)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.distributed.init_process_group(backend="nccl", init_method=init_method, world_size=num_proc, rank=local_rank)
    torch.cuda.set_device(local_rank)
    rec, _ = (run_train if func_name == "train" else run_test)(cfg)
    if local_rank == 0:
        torch.save(rec, ret_path)
    torch.distributed.destroy_process_group()


if __name__ == "__main__":
    # CPU dry run of the harness itself with the STOCK model (NUM_GPUS 0); train_epoch calls torch.cuda.synchronize()
    # unconditionally (train_net.py:269), which needs a driver - stubbed here only.
    torch.cuda.synchronize = lambda *a, **k: None
    torch.cuda.empty_cache = lambda *a, **k: None
    setup_reference()
    yaml = sys.argv[1] if len(sys.argv) > 1 else "Kinetics/C2D_8x8_R50.yaml"
    cfg = driver_cfg(yaml, 0, ["MODEL.DROPOUT_RATE", 0.0], batch=2, frames=8)
    rec, out = run_train(cfg)
    print("train losses", [round(r["loss"], 4) for r in rec["train"]], "val iters", len(rec["val"]))
    if not cfg.MASK.ENABLE:
        rec, out = run_test(cfg)
        print("test batches", len(rec["test"]), out[:80])
