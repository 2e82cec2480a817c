"""TEST INFRASTRUCTURE.  Needs a CUDA device and the unmodified reference (see oracle/refshim.py):

    python oracle/make_golden_autocast.py [OUT_DIR]

Runs the reference's own modules under torch.autocast(bfloat16) on the GPU (what TRAIN.MIXED_PRECISION gives with
bf16) on the fixtures of tests/test_gpu_models.py::test_fast_mode_is_in_the_reference_bf16_autocast_error_class, and
stores what that test compares the engine's fast mode against: the reference's bf16 logits and, per parameter, the
relative L2 error of its bf16 gradient against the fp32 oracle (oracle/torch_oracle.py).  Writes
``reference_bf16_autocast.pt`` to OUT_DIR (default tests/golden).
"""
from __future__ import annotations

import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import refshim, torch_oracle as TO  # noqa: E402
from slowfast_b200.config import get_cfg  # noqa: E402

# family: (golden case giving the config and state layout, engine preset)
FAMILIES = {"mvit": ("mvitv2_s_small", "MVITv2_S_16x4"), "slowfast": ("slowfast_r50_small", "SLOWFAST_8x8_R50")}
STATE_SEED, INPUT_SEED, DLOGITS_SEED = 91, 92, 93


def fixture(family: str):
    """Config, state, inputs and upstream gradient of the fast-mode comparison (shared with the test)."""
    gold = torch.load(os.path.join(ROOT, "tests", "golden", FAMILIES[family][0] + ".pt"))
    cfg = get_cfg(FAMILIES[family][1], B200={"NSPLIT": 1})
    ov = gold["overrides"]
    for k, v in zip(ov[0::2], ov[1::2]):
        sec, key = k.split(".")
        cfg[sec][key] = v
    template = {k: torch.empty(shape, dtype=torch.long if k.endswith("num_batches_tracked") else torch.float32)
                for k, shape in gold["keys"]}
    state = TO.fixture_state(template, STATE_SEED)
    if family == "slowfast":       # weak residual branches: the comparison is about rounding, not chaos
        for k in state:
            if k.endswith("c_bn.weight"):
                state[k] = state[k] * 0.1
    inputs = TO.synthetic_inputs(cfg, 2, INPUT_SEED)
    dlogits = torch.randn(2, 400, generator=torch.Generator().manual_seed(DLOGITS_SEED))
    return gold, cfg, state, inputs, dlogits


def run_family(family: str, dev):
    gold, cfg, state, inputs, dlogits = fixture(family)
    o_logits, o_grads = TO.forward_backward(cfg, state, inputs, dlogits)
    rcfg = refshim.load_cfg(gold["yaml"], ["NUM_GPUS", 1] + list(gold["overrides"]))
    model = refshim.build_reference_model(rcfg)
    model.load_state_dict(state, strict=True)
    model = model.to(dev).train()
    with torch.autocast("cuda", dtype=torch.bfloat16):
        r_logits = model([t.to(dev) for t in inputs])
    r_logits.float().backward(dlogits.to(dev))
    r_logits = r_logits.detach().float().cpu()
    grad_err = {k: ((p.grad.float().cpu() - o_grads[k]).norm() / o_grads[k].norm().clamp_min(1e-20)).item()
                for k, p in model.named_parameters() if k in o_grads}
    e = sorted(grad_err.values())
    print(f"[{family}] reference bf16 autocast vs fp32 oracle: logits rel-L2 "
          f"{((r_logits - o_logits).norm() / o_logits.norm()).item():.2e}, median gradient rel-L2 {e[len(e) // 2]:.2e}")
    return dict(logits=r_logits, grad_err=grad_err)


def main():
    out_dir = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden")
    assert torch.cuda.is_available(), "the reference's bf16 autocast run needs a CUDA device"
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.set_num_threads(min(32, len(os.sched_getaffinity(0))))
    dev = torch.device("cuda:0")
    gold = {f: run_family(f, dev) for f in FAMILIES}
    gold["device"] = torch.cuda.get_device_name(dev)
    gold["torch"] = str(torch.__version__)
    os.makedirs(out_dir, exist_ok=True)
    out = os.path.join(out_dir, "reference_bf16_autocast.pt")
    torch.save(gold, out)
    print(f"wrote {out} ({os.path.getsize(out) / 1024:.1f} KiB)")


if __name__ == "__main__":
    main()
