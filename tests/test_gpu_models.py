"""GPU parity of whole models (forward + backward through the engine) against
  (a) the golden vectors produced by the UNMODIFIED reference in the build container (tests/golden/*.pt), and
  (b) the plain-PyTorch oracle (oracle/torch_oracle.py) on fresh seeds.
Tolerances
  * outputs (logits / probabilities): 1e-3 relative, argmax bit-exact (north star).  Measured 8e-5 (224^2) .. 3e-4
    (64^2 fixture); the reference's OWN fp32-vs-fp64 difference on the same fixture is 2e-5, i.e. the split-bf16
    operands (~2^-17 relative) cost one order of magnitude, amplified ~250x by the 50 train-mode-BN layers exactly as
    an fp64 emulation of hi+lo operand rounding predicts (DESIGN.md section 4).
  * parameter gradients: ReLU masks flip wherever a pre-activation is within the forward error of zero, so a
    relative forward error e shows up as ~sqrt(e) relative L2 error in every gradient BELOW the flip, for any two
    implementations: the reference's own operators in fp32 vs fp64 differ by 1.5e-2 (median) / 3e-2 (max) rel-L2 on
    this fixture.  The engine is held to: gradient NORMS within 0.15 of the reference golden (8-element BN vectors of the fast
    pathway are the noisiest; measured worst 7e-2), per-parameter rel-L2
    median < 0.2 and max < 0.5 vs the oracle, cosine > 0.9.  (Each backward kernel is checked on its own to 2e-5 in
    tests/test_gpu_kernels.py, where no mask can flip.)
"""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
TOL = 1e-3
# parameter-gradient norms (see module docstring)
GRAD_TOL = 0.15


PRESET = {"Kinetics/SLOWFAST_8x8_R50.yaml": "SLOWFAST_8x8_R50", "Kinetics/C2D_8x8_R50.yaml": "C2D_8x8_R50",
          "Kinetics/SLOW_8x8_R50.yaml": "SLOW_8x8_R50", "Kinetics/I3D_8x8_R50.yaml": "I3D_8x8_R50",
          "Kinetics/MVITv2_S_16x4.yaml": "MVITv2_S_16x4", "Kinetics/MVITv2_B_32x3.yaml": "MVITv2_B_32x3",
          "Kinetics/X3D_M.yaml": "X3D_M",
          "masked_ssl/k400_MVITv2_S_16x4_MaskFeat_PT.yaml": "MVITv2_S_16x4_MaskFeat_PT"}


def sample_idx(numel: int, k: int = 256) -> torch.Tensor:
    """The element subset oracle/make_golden.py stores per parameter gradient (``grad_samples``)."""
    return torch.linspace(0, numel - 1, min(numel, k)).round().long()


def _model_class(cfg):
    if cfg.MODEL.MODEL_NAME == "SlowFast":
        from slowfast_b200.nets.resnet import B200SlowFast
        return B200SlowFast
    if cfg.MODEL.MODEL_NAME == "MViT":
        from slowfast_b200.nets.mvit import B200MViT
        return B200MViT
    if cfg.MODEL.MODEL_NAME == "X3D":
        from slowfast_b200.nets.x3d import B200X3D
        return B200X3D
    from slowfast_b200.nets.resnet_single import B200ResNet
    return B200ResNet


def _cfg_for(gold, nsplit=3):
    from slowfast_b200.config import get_cfg
    preset = PRESET[gold["yaml"]]
    if gold["case"].startswith("maskfeat_b"):   # composed config (BASELINE config 5, SURVEY.md section 3.5)
        preset = "MVITv2_B_32x3_MaskFeat_PT"
    cfg = get_cfg(preset, B200={"NSPLIT": nsplit})
    ov = gold["overrides"]
    for k, v in zip(ov[0::2], ov[1::2]):
        sec, key = k.split(".")
        if sec == "AUG":
            continue  # loader-side keys (mask window) are not read by the model
        cfg[sec][key] = v
    return cfg


def _run_engine(cfg, state, inputs, dlogits, dev):
    model = _model_class(cfg)(cfg)
    model.load_state_dict(state, strict=True)
    model = model.to(dev).train()
    logits = model([t.to(dev) for t in inputs])
    logits.backward(dlogits.to(dev))
    torch.cuda.synchronize()
    grads = {k: p.grad.detach().cpu() for k, p in model.named_parameters()}
    return logits.detach().cpu(), grads, {k: v.detach().cpu() for k, v in model.state_dict().items()}


@pytest.mark.parametrize("name", ["slowfast_r50_small", "slowfast_r50_224", "c2d_r50_small", "slow_r50_small",
                                  "i3d_r50_small", "x3d_m_small", "x3d_m_224"])
def test_model_matches_reference_golden(name, cuda_device):
    from oracle import torch_oracle as TO
    gold = torch.load(os.path.join(GOLDEN, name + ".pt"))
    cfg = _cfg_for(gold)
    template = {k: torch.empty(shape, dtype=torch.long if k.endswith("num_batches_tracked") else torch.float32)
                for k, shape in gold["keys"]}
    state = TO.fixture_state(template, gold["st_seed"])
    inputs = TO.synthetic_inputs(cfg, gold["batch"], gold["in_seed"])
    dlogits = torch.randn(gold["logits"].shape, generator=torch.Generator().manual_seed(gold["in_seed"] + 1000))
    logits, grads, new_state = _run_engine(cfg, state, inputs, dlogits, cuda_device)
    ref = gold["logits"]
    rel = ((logits - ref).abs().max() / ref.abs().max()).item()
    assert rel < TOL, f"logits rel err {rel}"
    assert torch.equal(logits.argmax(1), ref.argmax(1))
    errs = {}
    for k, dg in gold["grads"].items():
        g = grads[k].double().flatten()
        assert g.numel() == dg["numel"]
        e = abs(g.norm().item() - dg["norm"]) / max(dg["norm"], 1e-20)
        head = (g[:4] - torch.tensor(dg["head"], dtype=torch.float64)).abs().max().item() / max(dg["norm"] / dg["numel"] ** 0.5, 1e-20)
        errs[k] = (e, head)
    top = sorted(errs.items(), key=lambda kv: -kv[1][0])[:8]
    print(f"{name}: logits rel {rel:.2e}; worst grad-norm errs: " + ", ".join(f"{k}={v[0]:.2e}" for k, v in top))
    worst = top[0][1][0]
    assert worst < GRAD_TOL, f"{top[0][0]}: grad norm rel err {worst}"
    # the 4 leading elements of every gradient, in units of that gradient's RMS element: a wrong layout / transposed
    # filter / shifted tap shows up as O(1) here even when the norm happens to agree
    heads = sorted(v[1] for v in errs.values())
    print(f"{name}: leading-element error / RMS: median {heads[len(heads) // 2]:.2e}, max {heads[-1]:.2e}")
    # (measured on the B200: median 0.07-0.12, max 0.2-0.5 on these deliberately chaotic fixtures, where ReLU mask flips put
    # ~8 % rel-L2 into every gradient of ANY two implementations; a layout error gives a median of ~1.4)
    assert heads[len(heads) // 2] < 0.25 and heads[-1] < 1.5, (heads[len(heads) // 2], heads[-1])
    if "grad_samples" in gold:
        # element-wise: 256 evenly spaced elements of EVERY parameter gradient against the reference's fp32 values, held
        # to a multiple of the reference's own fp32-vs-fp64 error on the same elements (``grad_env``; floor 1e-3)
        env = gold["grad_env"]
        ratio, rels = {}, {}
        for k, ref_s in gold["grad_samples"].items():
            g = grads[k].flatten()[sample_idx(grads[k].numel())].double()
            r = ref_s.double()
            rels[k] = ((g - r).norm() / r.norm().clamp_min(1e-30)).item()
            ratio[k] = rels[k] / max(env[k], 1e-3)
        rs = sorted(rels.values())
        worst_k = max(ratio, key=ratio.get)
        e = sorted(env.values())
        print(f"{name}: sampled gradients vs reference fp32: rel-L2 median {rs[len(rs) // 2]:.2e} max {rs[-1]:.2e} "
              f"(reference fp32-vs-fp64 envelope: median {e[len(e) // 2]:.2e} max {e[-1]:.2e}); worst ratio "
              f"{ratio[worst_k]:.1f} at {worst_k}")
        # Bound: 8x the reference's own fp32-vs-fp64 error where that is the larger number (the 224^2 fixtures: 1-2e-2),
        # else the mask-flip plateau of the split-bf16 operands (2^-17 per operand vs fp32's 2^-24: the engine enters the
        # chaotic regime of a fixture ~100x earlier than fp32 does; measured 6e-2 median on x3d_m_small whose fp32
        # envelope is 4e-5) - the same 0.15 / 0.6 the fresh-seed oracle comparison below uses.  The gentle fixtures pin
        # the wiring to < 1e-2 element-wise.
        assert rs[len(rs) // 2] < max(8 * e[len(e) // 2], 0.15), "median sampled-gradient error above the bound"
        assert rs[-1] < 0.6, (worst_k, rels[worst_k], env[worst_k])
    for k, dr in gold["running"].items():
        v = new_state[k].double().flatten()
        assert abs(v.sum().item() - dr["sum"]) / max(abs(dr["sum"]), dr["norm"], 1e-20) < 1e-3, k
    print(f"{name}: logits rel {rel:.2e}, worst grad-norm rel {worst:.2e}")


@pytest.mark.parametrize("nsplit,tol", [(3, 1e-3), (1, 0.2)])
def test_slowfast_matches_oracle_fresh_seed(nsplit, tol, cuda_device):
    """Fresh inputs / weights vs the oracle evaluated on this box's CPU: every parameter gradient compared in full
    (rel-L2).  The bf16 fast mode is checked against the error class the reference's own bf16 autocast shows
    (BASELINE.md §4: 3e-2 rel-L2 on logits)."""
    from oracle import torch_oracle as TO
    gold = torch.load(os.path.join(GOLDEN, "slowfast_r50_small.pt"))
    cfg = _cfg_for(gold, nsplit)
    template = {k: torch.empty(shape, dtype=torch.long if k.endswith("num_batches_tracked") else torch.float32)
                for k, shape in gold["keys"]}
    state = TO.fixture_state(template, 123)
    inputs = TO.synthetic_inputs(cfg, 3, 321)
    dlogits = torch.randn(3, 400, generator=torch.Generator().manual_seed(9))
    o_logits, o_grads = TO.forward_backward(cfg, state, inputs, dlogits)
    logits, grads, _ = _run_engine(cfg, state, inputs, dlogits, cuda_device)
    rel = ((logits - o_logits).norm() / o_logits.norm()).item()
    assert rel < tol, f"logits rel-L2 {rel}"
    if nsplit == 1:
        # bf16 fast mode: operand rounding of 2^-9 puts the stage-5 activations of this (deliberately chaotic)
        # fixture 40 % off in ANY bf16 implementation; only the output tolerance is meaningful here.
        print(f"nsplit=1: logits rel-L2 {rel:.2e}")
        return
    per = {k: ((grads[k] - o_grads[k]).norm() / o_grads[k].norm().clamp_min(1e-20)).item() for k in o_grads}
    top = sorted(per.items(), key=lambda kv: -kv[1])[:8]
    med = sorted(per.values())[len(per) // 2]
    print(f"nsplit={nsplit}: logits rel-L2 {rel:.2e}, median grad rel-L2 {med:.2e}, worst: " +
          ", ".join(f"{k}={v:.2e}" for k, v in top))
    cos = min(torch.nn.functional.cosine_similarity(grads[k].flatten().double(), o_grads[k].flatten().double(), dim=0).item()
              for k in o_grads)
    assert med < 0.2 and top[0][1] < 0.5 and cos > 0.9, (med, top[0], cos)


def test_slowfast_eval_mode(cuda_device):
    from oracle import torch_oracle as TO
    gold = torch.load(os.path.join(GOLDEN, "slowfast_r50_small.pt"))
    cfg = _cfg_for(gold)
    template = {k: torch.empty(shape, dtype=torch.long if k.endswith("num_batches_tracked") else torch.float32)
                for k, shape in gold["keys"]}
    state = TO.fixture_state(template, 77)
    inputs = TO.synthetic_inputs(cfg, 2, 78)
    from slowfast_b200.nets.resnet import B200SlowFast
    model = B200SlowFast(cfg)
    model.load_state_dict(state)
    model = model.to(cuda_device).eval()
    with torch.no_grad():
        probs = model([t.to(cuda_device) for t in inputs]).cpu()
    ref = TO.forward(cfg, {k: v.clone() for k, v in state.items()}, inputs, training=False)
    assert ((probs - ref).abs().max() / ref.abs().max()).item() < TOL
    assert torch.equal(probs.argmax(1), ref.argmax(1))
    assert torch.allclose(probs.sum(1), torch.ones(2), atol=1e-5)


def test_slowfast_gentle_fixture_tight_gradients(cuda_device):
    """Same network with weak residual branches (c_bn.weight x 0.1): the forward error is no longer amplified, almost
    no ReLU mask flips, and every parameter gradient must agree with the oracle tightly - this is the check that the
    backward WIRING (accumulation order, slices, strided dgrad, stems, lateral fusions) is exact."""
    from oracle import torch_oracle as TO
    gold = torch.load(os.path.join(GOLDEN, "slowfast_r50_small.pt"))
    cfg = _cfg_for(gold)
    template = {k: torch.empty(shape, dtype=torch.long if k.endswith("num_batches_tracked") else torch.float32)
                for k, shape in gold["keys"]}
    state = TO.fixture_state(template, 31)
    for k in state:
        if k.endswith("c_bn.weight"):
            state[k] = state[k] * 0.1
    inputs = TO.synthetic_inputs(cfg, 2, 32)
    dlogits = torch.randn(2, 400, generator=torch.Generator().manual_seed(33))
    o_logits, o_grads = TO.forward_backward(cfg, state, inputs, dlogits)
    logits, grads, _ = _run_engine(cfg, state, inputs, dlogits, cuda_device)
    rel = ((logits - o_logits).norm() / o_logits.norm()).item()
    per = {k: ((grads[k] - o_grads[k]).norm() / o_grads[k].norm().clamp_min(1e-20)).item() for k in o_grads}
    top = sorted(per.items(), key=lambda kv: -kv[1])[:6]
    med = sorted(per.values())[len(per) // 2]
    print(f"gentle fixture: logits rel-L2 {rel:.2e}, median grad rel-L2 {med:.2e}, worst: " +
          ", ".join(f"{k}={v:.2e}" for k, v in top))
    assert rel < 1e-4 and med < 1e-2 and top[0][1] < 5e-2


def test_c2d_gentle_fixture_and_eval(cuda_device):
    """C2D-R50 (single pathway + temporal max-pool after res2): tight gradient check on the gentle fixture and the
    eval-mode (running statistics, softmax) forward."""
    from oracle import torch_oracle as TO
    gold = torch.load(os.path.join(GOLDEN, "c2d_r50_small.pt"))
    cfg = _cfg_for(gold)
    template = {k: torch.empty(shape, dtype=torch.long if k.endswith("num_batches_tracked") else torch.float32)
                for k, shape in gold["keys"]}
    state = TO.fixture_state(template, 41)
    for k in state:
        if k.endswith("c_bn.weight"):
            state[k] = state[k] * 0.1
    inputs = TO.synthetic_inputs(cfg, 2, 42)
    dlogits = torch.randn(2, 400, generator=torch.Generator().manual_seed(43))
    o_logits, o_grads = TO.forward_backward(cfg, state, inputs, dlogits)
    logits, grads, _ = _run_engine(cfg, state, inputs, dlogits, cuda_device)
    rel = ((logits - o_logits).norm() / o_logits.norm()).item()
    per = {k: ((grads[k] - o_grads[k]).norm() / o_grads[k].norm().clamp_min(1e-20)).item() for k in o_grads}
    med = sorted(per.values())[len(per) // 2]
    worst = max(per.items(), key=lambda kv: kv[1])
    print(f"c2d gentle: logits rel-L2 {rel:.2e}, median grad rel-L2 {med:.2e}, worst {worst}")
    assert rel < 1e-4 and med < 1e-2 and worst[1] < 5e-2
    model = _model_class(cfg)(cfg)
    model.load_state_dict(state)
    model = model.to(cuda_device).eval()
    with torch.no_grad():
        probs = model([t.to(cuda_device) for t in inputs]).cpu()
    ref = TO.forward(cfg, {k: v.clone() for k, v in state.items()}, inputs, training=False)
    assert ((probs - ref).abs().max() / ref.abs().max()).item() < TOL


@pytest.mark.parametrize("name", ["mvitv2_s_small", "mvitv2_s_224", "mvitv2_b_small", "mvitv2_b_224"])
def test_mvit_matches_reference_golden(name, cuda_device):
    """MViTv2-S (pooled attention with decomposed rel-pos bias, residual pooling, cls token) forward + backward vs the
    golden vectors of the UNMODIFIED reference.  No ReLU on this path => no mask flips: gradients are held to 2e-2
    on norms (measured 5e-5 median / 1e-2 worst rel-L2 against the oracle)."""
    from oracle import torch_oracle as TO
    gold = torch.load(os.path.join(GOLDEN, name + ".pt"))
    cfg = _cfg_for(gold)
    template = {k: torch.empty(shape, dtype=torch.float32) for k, shape in gold["keys"]}
    state = TO.fixture_state(template, gold["st_seed"])
    inputs = TO.synthetic_inputs(cfg, gold["batch"], gold["in_seed"])
    dlogits = torch.randn(gold["logits"].shape, generator=torch.Generator().manual_seed(gold["in_seed"] + 1000))
    logits, grads, _ = _run_engine(cfg, state, inputs, dlogits, cuda_device)
    ref = gold["logits"]
    rel = ((logits - ref).abs().max() / ref.abs().max()).item()
    assert rel < TOL, f"logits rel err {rel}"
    assert torch.equal(logits.argmax(1), ref.argmax(1))
    floor = gold.get("grad_norm_floor", 0.0)
    errs = {}
    for k, dg in gold["grads"].items():
        g = grads[k].double().flatten()
        errs[k] = abs(g.norm().item() - dg["norm"]) / max(dg["norm"], floor, 1e-20)
    top = sorted(errs.items(), key=lambda kv: -kv[1])[:6]
    print(f"{name}: logits rel {rel:.2e}; worst grad-norm errs: " + ", ".join(f"{k}={v:.2e}" for k, v in top))
    assert top[0][1] < 2e-2


def test_mvit_matches_oracle_every_gradient(cuda_device):
    from oracle import torch_oracle as TO
    gold = torch.load(os.path.join(GOLDEN, "mvitv2_s_small.pt"))
    cfg = _cfg_for(gold)
    template = {k: torch.empty(shape, dtype=torch.float32) for k, shape in gold["keys"]}
    state = TO.fixture_state(template, 51)
    inputs = TO.synthetic_inputs(cfg, 3, 52)
    dlogits = torch.randn(3, 400, generator=torch.Generator().manual_seed(53))
    o_logits, o_grads = TO.forward_backward(cfg, state, inputs, dlogits)
    logits, grads, _ = _run_engine(cfg, state, inputs, dlogits, cuda_device)
    rel = ((logits - o_logits).norm() / o_logits.norm()).item()
    norms = sorted(v.norm().item() for v in o_grads.values())
    floor = 1e-2 * norms[len(norms) // 2]  # gradients that are zero in exact arithmetic (norm_k.bias) are noise
    per = {k: ((grads[k] - o_grads[k]).norm() / o_grads[k].norm().clamp_min(floor)).item() for k in o_grads}
    med = sorted(per.values())[len(per) // 2]
    worst = max(per.items(), key=lambda kv: kv[1])
    print(f"mvit vs oracle: logits rel-L2 {rel:.2e}, median grad rel-L2 {med:.2e}, worst {worst}")
    assert rel < 1e-3 and med < 1e-3 and worst[1] < 5e-2
    # eval mode
    model = _model_class(cfg)(cfg)
    model.load_state_dict(state)
    model = model.to(cuda_device).eval()
    with torch.no_grad():
        probs = model([t.to(cuda_device) for t in inputs]).cpu()
    ref = TO.forward(cfg, {k: v.clone() for k, v in state.items()}, inputs, training=False)
    assert ((probs - ref).abs().max() / ref.abs().max()).item() < TOL


def test_x3d_gentle_fixture_and_eval(cuda_device):
    """X3D-M (channelwise 3x3x3, SE on even blocks, Swish, 54/108-wide bottlenecks padded to 56/112, X3DStem,
    X3DHead): tight per-parameter gradient check on the gentle fixture (weak residual branches => no ReLU mask
    flips) and the eval-mode forward (running statistics, SE on running-stat BN output, softmax)."""
    from oracle import torch_oracle as TO
    gold = torch.load(os.path.join(GOLDEN, "x3d_m_small.pt"))
    cfg = _cfg_for(gold)
    template = {k: torch.empty(shape, dtype=torch.long if k.endswith("num_batches_tracked") else torch.float32)
                for k, shape in gold["keys"]}
    state = TO.fixture_state(template, 61)
    for k in state:
        if k.endswith("c_bn.weight"):
            state[k] = state[k] * 0.1
    inputs = TO.synthetic_inputs(cfg, 3, 62)
    dlogits = torch.randn(3, 400, generator=torch.Generator().manual_seed(63))
    o_logits, o_grads = TO.forward_backward(cfg, state, inputs, dlogits)
    logits, grads, _ = _run_engine(cfg, state, inputs, dlogits, cuda_device)
    rel = ((logits - o_logits).norm() / o_logits.norm()).item()
    per = {k: ((grads[k] - o_grads[k]).norm() / o_grads[k].norm().clamp_min(1e-20)).item() for k in o_grads}
    med = sorted(per.values())[len(per) // 2]
    top = sorted(per.items(), key=lambda kv: -kv[1])[:6]
    print(f"x3d gentle: logits rel-L2 {rel:.2e}, median grad rel-L2 {med:.2e}, worst: " +
          ", ".join(f"{k}={v:.2e}" for k, v in top))
    assert rel < 1e-4 and med < 1e-2 and top[0][1] < 5e-2
    model = _model_class(cfg)(cfg)
    model.load_state_dict(state)
    model = model.to(cuda_device).eval()
    with torch.no_grad():
        probs = model([t.to(cuda_device) for t in inputs]).cpu()
    ref = TO.forward(cfg, {k: v.clone() for k, v in state.items()}, inputs, training=False)
    assert ((probs - ref).abs().max() / ref.abs().max()).item() < TOL
    assert torch.equal(probs.argmax(1), ref.argmax(1))


@pytest.mark.parametrize("name", ["maskfeat_s_small", "maskfeat_s_224", "maskfeat_s_shipped_small", "maskfeat_b_small",
                                  "maskfeat_b_224"])
def test_maskfeat_matches_reference_golden(name, cuda_device):
    """MaskMViT (mask-token substitution, MViTv2 encoder, MSSeparateHead, HOG targets) vs the UNMODIFIED reference:
    predictions for the masked tokens 1e-3 (measured ~1e-5), every parameter-gradient norm 2e-2, HOG regression
    targets: identical up to fp32 rounding of atan2 / the 64-pixel cell sums (a pixel whose orientation sits within
    one ulp of a bin edge may land in the neighbouring bin: at most a handful of the ~70k target values may differ)."""
    from oracle import torch_oracle as TO
    from slowfast_b200.nets.maskfeat import B200MaskMViT
    gold = torch.load(os.path.join(GOLDEN, name + ".pt"))
    cfg = _cfg_for(gold)
    template = {k: torch.empty(shape, dtype=torch.float32) for k, shape in gold["keys"]}
    state = TO.fixture_state(template, gold["st_seed"])
    frames, mask = TO.maskfeat_inputs(cfg, gold["batch"], gold["in_seed"])
    dpred = torch.randn(gold["logits"].shape, generator=torch.Generator().manual_seed(gold["in_seed"] + 1000))
    model = B200MaskMViT(cfg)
    model.load_state_dict(state, strict=True)
    model = model.to(cuda_device).train()
    preds, labels = model([frames.to(cuda_device), torch.Tensor(), mask.to(cuda_device)])
    assert len(preds) == 1 and len(labels) == 1 and labels[0][1] == 1.0 and labels[0][2] == "mse"
    pred = preds[0]
    pred.backward(dpred.to(cuda_device))
    torch.cuda.synchronize()
    ref = gold["logits"]
    assert pred.shape == ref.shape
    rel = ((pred.detach().cpu() - ref).abs().max() / ref.abs().max()).item()
    assert rel < TOL, f"prediction rel err {rel}"
    lab = labels[0][0].cpu()
    dig = gold["labels_digest"]
    assert lab.numel() == dig["numel"]
    # every value through the digest of the whole target; each value of the stored rows (all rows of smaller targets)
    norm_err = abs(lab.double().norm().item() - dig["norm"]) / dig["norm"]
    assert norm_err < 1e-3, norm_err
    if "label_rows" in gold:
        lab = lab[gold["label_rows"]]
    ref_lab = gold["labels"]
    assert lab.shape == ref_lab.shape
    bad = ((lab - ref_lab).abs() > 1e-4).sum().item()
    print(f"{name}: pred rel {rel:.2e}; HOG targets differing by > 1e-4: {bad} of {lab.numel()}, "
          f"max abs {(lab - ref_lab).abs().max().item():.2e}")
    assert bad <= max(4, lab.numel() // 5000)
    floor = gold.get("grad_norm_floor", 0.0)
    grads = {k: p.grad.detach().cpu() for k, p in model.named_parameters()}
    errs = {k: abs(grads[k].double().norm().item() - dg["norm"]) / max(dg["norm"], floor, 1e-20)
            for k, dg in gold["grads"].items()}
    top = sorted(errs.items(), key=lambda kv: -kv[1])[:6]
    print(f"{name}: worst grad-norm errs: " + ", ".join(f"{k}={v:.2e}" for k, v in top))
    assert top[0][1] < 2e-2
    # the reference's loss on the engine's outputs (losses.py:25 MultipleMSELoss): mean squared error per head, summed
    loss = sum(torch.nn.functional.mse_loss(p, l[0]) * l[1] for p, l in zip(preds, labels))
    assert torch.isfinite(loss)


def test_maskfeat_matches_oracle_every_gradient(cuda_device):
    from oracle import torch_oracle as TO
    from slowfast_b200.nets.maskfeat import B200MaskMViT
    gold = torch.load(os.path.join(GOLDEN, "maskfeat_s_small.pt"))
    cfg = _cfg_for(gold)
    template = {k: torch.empty(shape, dtype=torch.float32) for k, shape in gold["keys"]}
    state = TO.fixture_state(template, 71)
    frames, mask = TO.maskfeat_inputs(cfg, 3, 72)
    o_pred0 = TO.forward(cfg, state, [frames, mask], True)
    dpred = torch.randn(o_pred0.shape, generator=torch.Generator().manual_seed(73))
    o_pred, o_grads = TO.forward_backward(cfg, state, [frames, mask], dpred)
    model = B200MaskMViT(cfg)
    model.load_state_dict(state, strict=True)
    model = model.to(cuda_device).train()
    preds, labels = model([frames.to(cuda_device), torch.Tensor(), mask.to(cuda_device)])
    preds[0].backward(dpred.to(cuda_device))
    torch.cuda.synchronize()
    rel = ((preds[0].detach().cpu() - o_pred).norm() / o_pred.norm()).item()
    grads = {k: p.grad.detach().cpu() for k, p in model.named_parameters()}
    norms = sorted(v.norm().item() for v in o_grads.values())
    floor = 1e-2 * norms[len(norms) // 2]
    per = {k: ((grads[k] - o_grads[k]).norm() / o_grads[k].norm().clamp_min(floor)).item() for k in o_grads}
    med = sorted(per.values())[len(per) // 2]
    worst = max(per.items(), key=lambda kv: kv[1])
    print(f"maskfeat vs oracle: pred rel-L2 {rel:.2e}, median grad rel-L2 {med:.2e}, worst {worst}")
    assert rel < 1e-3 and med < 1e-3 and worst[1] < 5e-2
    # labels vs the oracle's CPU HOG on this fresh clip
    o_lab = TO.maskfeat_labels(cfg, frames, mask)
    lab = labels[0][0].cpu()
    assert ((lab - o_lab).abs() > 1e-4).sum().item() <= max(4, lab.numel() // 5000)
    # return_all: predictions for every token; the masked rows are the same numbers
    with torch.no_grad():
        pa, _ = model([frames.to(cuda_device), torch.Tensor(), mask.to(cuda_device)], return_all=True)
    assert pa[0].shape[0] == 3 and pa[0].shape[2] == o_pred.shape[1]


@pytest.mark.parametrize("family", ["mvit", "slowfast"])
def test_fast_mode_is_in_the_reference_bf16_autocast_error_class(family, cuda_device):
    """Fast mode (cfg.B200.NSPLIT = 1: plain bf16 tensor-core operands, fp32 accumulate) is not held to the fp32 tolerance
    but to the error class of the reference's OWN reduced-precision run: the unmodified reference modules on a B200
    under torch.autocast(bfloat16) (what TRAIN.MIXED_PRECISION would give with bf16) against the fp32 oracle, stored by
    oracle/make_golden_autocast.py.  The engine's fast mode must not be worse than 2x that (it keeps fp32 storage, so it
    is usually better)."""
    from oracle import torch_oracle as TO
    from oracle.make_golden_autocast import fixture
    _, cfg, state, inputs, dlogits = fixture(family)
    o_logits, o_grads = TO.forward_backward(cfg, state, inputs, dlogits)
    logits, grads, _ = _run_engine(cfg, state, inputs, dlogits, cuda_device)
    e_log = ((logits - o_logits).norm() / o_logits.norm()).item()
    per = sorted(((grads[k] - o_grads[k]).norm() / o_grads[k].norm().clamp_min(1e-20)).item() for k in o_grads)
    e_grad = per[len(per) // 2]
    ref = torch.load(os.path.join(GOLDEN, "reference_bf16_autocast.pt"))[family]
    r_log = ((ref["logits"] - o_logits).norm() / o_logits.norm()).item()
    rper = sorted(ref["grad_err"][k] for k in o_grads if k in ref["grad_err"])
    r_grad = rper[len(rper) // 2]
    print(f"{family}: fast mode logits rel-L2 {e_log:.2e} (reference bf16 autocast {r_log:.2e}); median gradient rel-L2 "
          f"{e_grad:.2e} (reference {r_grad:.2e})")
    bound_log, bound_grad = max(2 * r_log, 1e-3), max(2 * r_grad, 1e-3)
    assert e_log < bound_log and e_grad < bound_grad, (e_log, bound_log, e_grad, bound_grad)
