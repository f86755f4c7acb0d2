"""GPU: the configuration bench.py times is the configuration proven here.

ResNet-101 224^2 (seeded random init, as bench.py), S = 50 superpixels, k = 20 keep-masks drawn with seed 1 (the first 768 of
the masks bench.py scores), micro-batch 384 over 2 stream copies, fused expansion+reduction launches, the device-side tie
policy on (PerturbationEngine defaults) -- against (a) the oracle's fp32 CPU forward of the reference's `model(x)`
(generate_gp_training_data_imagenet.py:246) on a 256-mask subset and (b) the engine's own fp32 lowering on all 768.

Tolerances (north_star): logits within 1e-2 relative in bf16, stated here element-wise against the row's own scale,
|a - b| <= 1e-2 * max_k |b[n, k]| for every element of every row (stricter than one max-norm over the batch); identical
top-1 on EVERY mask; target-class probability within the bound the logit tolerance implies,
|d ln p| <= 2 * 1e-2 * max|logit|  (p = exp(l_t - lse(l)); both terms move by at most the logit error)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import classifier as ocls
from oracle import masks as om
from oracle import scoring as oscore
from oracle import synthetic

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

TOL_BF16 = 1e-2
N_MASKS = 768
MICRO_BATCH = 384
STREAMS = 2


def _rowwise_err(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float((np.abs(a - b) / np.abs(b).max(axis=1, keepdims=True)).max())


@pytest.fixture(scope="module")
def bench_setup(nib):
    x = synthetic.synthetic_image("imagenet")
    seg = synthetic.voronoi_labels(224, 224, 50)
    model = ocls.build_imagenet_model("resnet101")
    sels = nib.draw_selections("subset_keep", 50, N_MASKS, seed=1)
    bits = nib.selection_bits(sels, 50)
    eng = nib.PerturbationEngine(model, x, seg, target=0, mode=nib.KEEP_MUL, precision="bf16", max_batch=MICRO_BATCH, S=50,
                                 streams=STREAMS)
    assert eng.refine_ties is not None, "the tie policy must be on by default for bf16"
    assert len(eng.classifier._replicas) == STREAMS - 1
    return dict(nib=nib, x=x, seg=seg, model=model, sels=sels, bits=bits, eng=eng)


def test_bench_config_logits_and_top1_vs_engine_fp32_all_masks(bench_setup):
    s = bench_setup
    nib, eng = s["nib"], s["eng"]
    from network_interpretation_imagenet_b200.classifier import Classifier
    d_bits = torch.from_numpy(s["bits"].view(np.int64)).cuda()
    lg16 = eng.classifier.forward_masked(eng.synth, d_bits, nib.KEEP_MUL)
    total, tc = eng.classifier.launch_counts()
    assert tc > 0, "the tcgen05 path did not run"
    f32 = Classifier.from_torch(s["model"], (224, 224), precision="fp32", max_batch=64)
    lg32 = f32.forward_masked(eng.synth, d_bits, nib.KEEP_MUL)
    a, b = lg16.cpu().numpy(), lg32.cpu().numpy()
    err = _rowwise_err(a, b)
    assert err <= TOL_BF16, f"bf16 logits vs fp32 engine: row-wise relative error {err:.3e}"
    # the quantity the tie band is derived from: error of (top1 - other) logit differences, relative to max|logit|
    t1 = b.argmax(1)
    rows = np.arange(len(t1))
    diff_err = np.abs((a[rows, t1][:, None] - a) - (b[rows, t1][:, None] - b)) / np.abs(b).max(axis=1, keepdims=True)
    eps = float(diff_err.max())
    from network_interpretation_imagenet_b200.engine import DEFAULT_TIE_BAND
    print(f"\n[bench-config] bf16 vs fp32 engine: logit err {err:.3e}, top1-difference err {eps:.3e}, band {DEFAULT_TIE_BAND:g}")
    assert eps <= 2 * TOL_BF16, f"top-1 difference error {eps:.3e} exceeds what the logit tolerance allows"
    # the product path (scores with the tie policy) must give the fp32 arg-max on every mask
    out = eng.score_masks(s["bits"])
    s32 = nib.score(lg32, 0)
    assert np.array_equal(out["top1"].cpu().numpy(), s32["top1"].cpu().numpy()), "top-1 differs from the fp32 engine"
    st = eng.tie_stats()
    print(f"[bench-config] tie policy: {st}")
    assert st["overflow"] == 0, st
    amax = float(np.abs(b).max())
    rtol = float(np.expm1(2 * TOL_BF16 * amax))
    p16, p32 = out["target_prob"].cpu().numpy().astype(np.float64), s32["target_prob"].cpu().numpy().astype(np.float64)
    assert np.all(np.abs(p16 - p32) <= rtol * p32), (float((np.abs(p16 - p32) / p32).max()), rtol)


def test_bench_config_vs_oracle_fp32_cpu_subset(bench_setup):
    """256 of the 768 masks (every third) through the oracle: numpy mask ops + torch CPU fp32 forward."""
    s = bench_setup
    nib, eng = s["nib"], s["eng"]
    pick = np.arange(0, N_MASKS, 3)[:256]
    sels = [s["sels"][i] for i in pick]
    batch = om.masked_batch(s["x"], s["seg"], sels, "keep")
    want = np.concatenate([ocls.forward_logits(s["model"], batch[i:i + 32]).numpy() for i in range(0, len(pick), 32)])
    d_bits = torch.from_numpy(s["bits"].view(np.int64)).cuda()
    got = eng.classifier.forward_masked(eng.synth, d_bits, nib.KEEP_MUL).cpu().numpy()[pick]
    err = _rowwise_err(got, want)
    assert err <= TOL_BF16, f"bf16 logits vs oracle: row-wise relative error {err:.3e}"
    top1, tprob, _, _ = oscore.score(want, 0)
    out = eng.score_masks(s["bits"])
    assert np.array_equal(out["top1"].cpu().numpy()[pick], top1), "top-1 differs from the oracle on some mask"
    amax = float(np.abs(want).max())
    rtol = float(np.expm1(2 * TOL_BF16 * amax))
    p = out["target_prob"].cpu().numpy()[pick].astype(np.float64)
    assert np.all(np.abs(p - tprob) <= rtol * tprob), (float((np.abs(p - tprob) / tprob).max()), rtol)


def test_tie_policy_is_device_side_and_bounded(bench_setup):
    """A band wide enough to catch every mask with a 16-row buffer: exactly the first 16 rows (index order) are refined,
    the overflow is counted, refined rows carry the fp32 scores bit for bit, the others keep their bf16 scores."""
    s = bench_setup
    nib = s["nib"]
    from network_interpretation_imagenet_b200.classifier import Classifier
    eng = nib.PerturbationEngine(s["model"], s["x"], s["seg"], target=0, mode=nib.KEEP_MUL, precision="bf16", max_batch=64,
                                 S=50, refine_ties=10.0, tie_capacity=16, tie_precision="fp32")
    bits = s["bits"][:48]
    out = eng.score_masks(bits)
    st = eng.tie_stats()
    assert st["near_ties"] == 48 and st["overflow"] == 32 and st["refined"] == 16, st
    d_bits = torch.from_numpy(bits.view(np.int64)).cuda()
    f32 = Classifier.from_torch(s["model"], (224, 224), precision="fp32", max_batch=16)
    s32 = nib.score(f32.forward_masked(eng.synth, d_bits[:16], nib.KEEP_MUL), 0)
    assert torch.equal(out["target_prob"][:16], s32["target_prob"]) and torch.equal(out["top1"][:16], s32["top1"])
    s16 = nib.score(eng.classifier.forward_masked(eng.synth, d_bits, nib.KEEP_MUL), 0)
    assert torch.equal(out["target_prob"][16:], s16["target_prob"][16:]) and torch.equal(out["top1"][16:], s16["top1"][16:])
    # the default re-score precision (split-bf16 tensor-core products): same rows refined, scores within 1e-4 of the fp32 ones
    engx = nib.PerturbationEngine(s["model"], s["x"], s["seg"], target=0, mode=nib.KEEP_MUL, precision="bf16", max_batch=64,
                                  S=50, refine_ties=10.0, tie_capacity=16)
    assert engx.tie_precision == "split"          # torchvision ResNet: the tcgen05 pair kernel over split-bf16 tensors
    outx = engx.score_masks(bits)
    assert torch.equal(outx["top1"][:16], s32["top1"])
    assert torch.allclose(outx["target_prob"][:16], s32["target_prob"], rtol=1e-4, atol=0)
    assert torch.equal(outx["target_prob"][16:], s16["target_prob"][16:])
    engy = nib.PerturbationEngine(s["model"], s["x"], s["seg"], target=0, mode=nib.KEEP_MUL, precision="bf16", max_batch=64,
                                  S=50, refine_ties=10.0, tie_capacity=16, tie_precision="x3")
    outy = engy.score_masks(bits)
    assert torch.equal(outy["top1"][:16], s32["top1"])
    assert torch.allclose(outy["target_prob"][:16], s32["target_prob"], rtol=1e-4, atol=0)
    # no near-tie at all: nothing is refined, nothing changes
    eng0 = nib.PerturbationEngine(s["model"], s["x"], s["seg"], target=0, mode=nib.KEEP_MUL, precision="bf16", max_batch=64,
                                  S=50, refine_ties=1e-9, tie_capacity=16)
    out0 = eng0.score_masks(bits)
    assert eng0.tie_stats()["near_ties"] == 0
    assert torch.equal(out0["target_prob"], s16["target_prob"]) and torch.equal(out0["top1"], s16["top1"])


def test_bench_dump_outputs_are_the_scores_of_the_last_timed_step(nib, tmp_path):
    """bench.py --dump-outputs writes the score table its timed path produced: the scores the engine gives for the same
    seeded job (the first N masks of seed 1, the seeded ResNet-101, micro-batch and stream copies as passed)."""
    n, mb = 96, 48
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--masks-per-step",
                        str(n), "--micro-batch", str(mb), "--no-cpu-baseline", "--no-library-bar", "--no-gp",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == 2 and line["config"]["masks_per_step_total"] == n
    assert sorted(os.listdir(tmp_path)) == ["target_prob.npy", "top1.npy"]
    prob, top1 = np.load(tmp_path / "target_prob.npy"), np.load(tmp_path / "top1.npy")
    assert prob.dtype == top1.dtype == np.float32 and prob.shape == top1.shape == (n,)
    eng = nib.PerturbationEngine(ocls.build_imagenet_model("resnet101"), synthetic.synthetic_image("imagenet"),
                                 synthetic.voronoi_labels(224, 224, 50), target=0, mode=nib.KEEP_MUL, precision="bf16",
                                 max_batch=mb, S=50, streams=STREAMS)
    out = eng.score_masks(nib.selection_bits(nib.draw_selections("subset_keep", 50, n, seed=1), 50))
    assert np.array_equal(top1, out["top1"].cpu().numpy().astype(np.float32))
    np.testing.assert_allclose(prob, out["target_prob"].cpu().numpy(), rtol=1e-5, atol=0)
