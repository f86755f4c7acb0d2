"""GPU: torchvision VGG and AlexNet on the engine.

The 3x3 first conv on raw input rows (conv_tc.cu tc_conv_is_raw3x3, TC_A_RAW over 16-byte pixels), Linear layers
lowered as convolutions (the first as a valid KxK conv over the final map, the middle ones as 1x1 convs on 1x1 maps),
whole networks in all four precisions against the torch fp32 CPU forward (oracle.classifier.forward_logits), the bench
configuration with the tie policy on, and the ImageNet drop-in with `-a vgg16`.  Tolerances as tests/test_gpu_classifier.py:
element-wise against each row's own scale."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import classifier as ocls
from oracle import synthetic

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

TOL_FP32 = 1e-4
TOL_BF16 = 1e-2


def rel_err(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float((np.abs(a - b) / np.maximum(np.abs(b).max(axis=1, keepdims=True), 1e-30)).max())


# ---- 3x3 first conv on raw input rows --------------------------------------------------------------------------------
def _raw3x3_net(nib, H, Cout, relu, N, seed):
    from network_interpretation_imagenet_b200 import _lib
    from network_interpretation_imagenet_b200.classifier import _Builder, Classifier
    g = torch.Generator().manual_seed(seed)
    w = torch.randn(Cout, 3, 3, 3, generator=g) / np.sqrt(27)
    bias = torch.randn(Cout, generator=g) * 0.1
    x = torch.randn(N, 3, H, H, generator=g)
    b = _Builder(_lib.PREC_BF16, N)
    x_in = b.buffer(H, H, 8, pad=1, pooled=False)     # 8-channel pixels in a 1-pixel zero halo
    out = b.buffer(H, H, Cout, pooled=False)
    b.conv(x_in, 3, out, Cout, w, bias, 3, 1, 1, relu=relu)
    feat = b.buffer(1, 1, Cout)
    b.pool(_lib.POOL_AVG, out, Cout, feat, H, H, 0)
    b.fc(feat, Cout, 4, torch.zeros(4, Cout), None)
    net = Classifier(b, x_in, (3, H, H), 4, "bf16", N, taps={"out": out})
    ref = F.conv2d(x.to(torch.bfloat16).double(), w.to(torch.bfloat16).double(), bias.double(), padding=1)
    if relu:
        ref = ref.clamp_min(0)
    return net, x, ref


@pytest.mark.parametrize("relu", [True, False])
@pytest.mark.parametrize("Cout", [64, 128])
@pytest.mark.parametrize("H", [224, 130, 100, 32])   # two column tiles of 112, two of 65, one tile per row (x2)
def test_raw_row_3x3_first_conv_vs_torch(nib, H, Cout, relu):
    N = 5
    net, x, ref = _raw3x3_net(nib, H, Cout, relu, N, seed=H + Cout + relu)
    net.forward(x.cuda())
    total, tc = net.launch_counts()
    assert tc == 1, "the 3x3 first conv did not take the tcgen05 raw-row path"
    got = net.read_tap("out", N).cpu().double()
    scale = max(ref.abs().max().item(), 1.0)
    err = (got - ref).abs().max().item()
    assert err <= 1.2e-2 * scale, f"max abs err {err} (scale {scale})"
    net.set_tensor_core(False)     # the same buffers through the CUDA-core kernel
    net.forward(x.cuda())
    got2 = net.read_tap("out", N).cpu().double()
    assert (got2 - ref).abs().max().item() <= 1.2e-2 * scale


def test_raw_row_3x3_without_a_column_split_falls_back(nib):
    """131 columns: no split into equal tiles of 64..128 columns, so the CUDA-core kernel runs, and is right."""
    N = 5
    net, x, ref = _raw3x3_net(nib, 131, 64, True, N, seed=131)
    net.forward(x.cuda())
    total, tc = net.launch_counts()
    assert tc == 0
    got = net.read_tap("out", N).cpu().double()
    assert (got - ref).abs().max().item() <= 1.2e-2 * max(ref.abs().max().item(), 1.0)


# ---- Linear layers as convolutions --------------------------------------------------------------------------------------
LINEAR_CASES = [(512, 7, 4096), (256, 6, 4096), (4096, 1, 4096)]    # Cin, K (= map side), Cout: fc6 VGG / AlexNet, fc7


def _linear_as_conv(nib, precision, Cin, K, Cout, N, seed):
    from network_interpretation_imagenet_b200 import _lib
    from network_interpretation_imagenet_b200.classifier import _Builder, Classifier
    g = torch.Generator().manual_seed(seed)
    lin_w = torch.randn(Cout, Cin * K * K, generator=g) / np.sqrt(Cin * K * K)
    lin_b = torch.randn(Cout, generator=g) * 0.1
    x = torch.randn(N, Cin, K, K, generator=g)
    split = precision == "split"
    b = _Builder(_lib.PREC_SPLIT if split else _lib.PREC_BF16, N)
    x_in = b.buffer(K, K, Cin, pooled=False, f32=split)
    src = x_in
    if split:
        src = b.buffer(K, K, Cin, pooled=False)
        b.convert(x_in, src)
    out = b.buffer(1, 1, Cout, pooled=False)
    b.conv(src, Cin, out, Cout, lin_w.view(Cout, Cin, K, K), lin_b, K, 1, 0, relu=True)
    tap = out
    if split:
        tap = b.buffer(1, 1, Cout, pooled=False, f32=True)
        b.convert(out, tap)
    b.fc(tap, Cout, 4, torch.zeros(4, Cout), None)
    net = Classifier(b, x_in, (Cin, K, K), 4, precision, N, taps={"out": tap})
    net.forward(x.cuda())
    got = net.read_tap("out", N).cpu().double().view(N, Cout)
    xs = x if split else x.to(torch.bfloat16)
    ws = lin_w if split else lin_w.to(torch.bfloat16)
    ref = (torch.flatten(xs.double(), 1) @ ws.double().T + lin_b.double()).clamp_min(0)   # torch's NCHW flatten
    return net, got, ref


# split: VGG's fc6 (K = 25088) is not lowered on split tensors: the tensor cores' fp32 accumulation measured 8.4e-5 of scale
# there, so split networks run it on fp32 buffers on the CUDA cores (classifier._FP32_GRADE_TC_MAX_K)
@pytest.mark.parametrize("precision,case", [("bf16", c) for c in LINEAR_CASES] + [("split", c) for c in LINEAR_CASES[1:]],
                         ids=lambda v: v if isinstance(v, str) else "cin%d_k%d_cout%d" % v)
def test_linear_as_conv_vs_torch(nib, case, precision):
    Cin, K, Cout = case
    net, got, ref = _linear_as_conv(nib, precision, Cin, K, Cout, N=5, seed=sum(case))
    total, tc = net.launch_counts()
    assert tc == 1, "the Linear-as-conv did not take the tcgen05 path"
    scale = max(ref.abs().max().item(), 1.0)
    err = (got - ref).abs().max().item()
    assert err <= (1.2e-2 if precision == "bf16" else 5e-5) * scale, f"max abs err {err} (scale {scale})"


# ---- whole networks -------------------------------------------------------------------------------------------------------
ARCHS = ["vgg11", "vgg16", "vgg16_bn", "vgg19_bn", "alexnet"]


@pytest.fixture(scope="module")
def nets():
    """Seeded random-init models (bench.py's weights), four inputs each, and the torch fp32 CPU logits."""
    out = {}
    base = torch.from_numpy(synthetic.synthetic_image("imagenet"))
    g = torch.Generator().manual_seed(3)
    x = base[None].repeat(4, 1, 1, 1)
    x[1] = x[1].flip(2) * 0.5
    x[2:] = x[2:] * (torch.rand(2, 1, 224, 224, generator=g) > 0.5).float()
    for arch in ARCHS:
        m = ocls.build_imagenet_model(arch)
        out[arch] = (m, x, ocls.forward_logits(m, x).numpy())
    return out


@pytest.mark.parametrize("arch", ARCHS)
def test_fp32_whole_network(nib, nets, arch):
    m, x, want = nets[arch]
    net = nib.Classifier.from_torch(m, (224, 224), precision="fp32", max_batch=x.shape[0])
    assert net.arch == "tv_plain"
    err = rel_err(net.forward(x.cuda()).cpu().numpy(), want)
    assert err <= TOL_FP32, f"{arch} fp32: rel err {err:.3e}"


VGG_FP32_GRADE_MEASURED_TOL = 1.5e-4


@pytest.mark.parametrize("arch", ARCHS)
def test_vgg_x3_and_split_are_outside_the_fp32_tolerance_and_say_so(nib, nets, arch):
    """The fp32-grade lowerings (x3: split-bf16 mma.sync products on fp32 tensors; split: the tcgen05 pair kernel on
    split-bf16 tensors, the tie policy's re-score) do NOT meet north_star's 1e-4 on the VGGs: 8 to 16 convolutions in a row,
    each accumulated in the tensor cores' fp32, measured up to 1.17e-4 (x3) and 1.36e-4 (split) row-wise, VGG-11 within
    1e-4 (with fc6 on the CUDA cores; 1.6e-4 .. 1.9e-4 with it on the tensor cores).  AlexNet meets 1e-4.  This pins the measured band, so that a regression or a fix
    shows up; the CUDA-core fp32 lowering meets 1e-4 (test_fp32_whole_network)."""
    m, x, want = nets[arch]
    tol = TOL_FP32 if arch == "alexnet" else VGG_FP32_GRADE_MEASURED_TOL
    got = {"fp32": nib.Classifier.from_torch(m, (224, 224), precision="fp32", max_batch=x.shape[0]).forward(x.cuda()).cpu().numpy()}
    for precision in ("x3", "split"):
        got[precision] = nib.Classifier.from_torch(m, (224, 224), precision=precision,
                                                   max_batch=x.shape[0]).forward(x.cuda()).cpu().numpy()
        err = rel_err(got[precision], want)
        print(f"\n[{arch} {precision}] row-wise relative logit error {err:.3e} (north_star 1e-4; accepted band {tol:g})")
        assert err <= tol, f"{arch} {precision}: rel err {err:.3e}"
    d = rel_err(got["split"], got["fp32"])
    print(f"[{arch}] split vs the fp32 lowering {d:.3e}")
    assert d <= tol
    assert np.array_equal(got["split"].argmax(1), got["fp32"].argmax(1))


@pytest.mark.parametrize("arch", ARCHS)
def test_bf16_whole_network(nib, nets, arch):
    m, x, want = nets[arch]
    net = nib.Classifier.from_torch(m, (224, 224), precision="bf16", max_batch=x.shape[0])
    got = net.forward(x.cuda()).cpu().numpy()
    err = rel_err(got, want)
    print(f"\n[{arch} bf16] row-wise relative logit error {err:.3e}")
    assert err <= TOL_BF16, f"{arch} bf16: rel err {err:.3e}"
    srt = np.sort(want, 1)
    decided = (srt[:, -1] - srt[:, -2]) > 2 * TOL_BF16 * np.abs(want).max(axis=1)
    assert np.array_equal(got.argmax(1)[decided], want.argmax(1)[decided]), "top-1 differs outside the tie band"
    if arch == "vgg16":
        # 13 convs + fc6 + fc7 on tcgen05; the rest is the input staging, 5 max pools and the fc: no conv_simt launch
        total, tc = net.launch_counts()
        assert tc == 15, tc
        assert total - tc == 7, (total, tc)


# ---- the bench configuration with the tie policy on --------------------------------------------------------------------
def test_vgg16_bench_config_top1_identical_to_fp32_on_every_mask(nib):
    """VGG-16 bf16, micro-batch 384 over 2 stream copies, 768 keep-masks of bench.py's seed, default band: top-1 equal
    to the fp32 lowering on every mask, no overflow, target_prob within the bound the 1e-2 logit tolerance implies."""
    from network_interpretation_imagenet_b200.classifier import Classifier
    from network_interpretation_imagenet_b200.engine import TIE_BANDS
    x = synthetic.synthetic_image("imagenet")
    seg = synthetic.voronoi_labels(224, 224, 50)
    model = ocls.build_imagenet_model("vgg16")
    bits = nib.selection_bits(nib.draw_selections("subset_keep", 50, 768, seed=1), 50)
    eng = nib.PerturbationEngine(model, x, seg, target=0, mode=nib.KEEP_MUL, precision="bf16", max_batch=384, S=50,
                                 streams=2)
    assert eng.refine_ties == TIE_BANDS["tv_plain"] and eng.tie_precision == "split"
    out = eng.score_masks(bits)
    d_bits = torch.from_numpy(bits.view(np.int64)).cuda()
    f32 = Classifier.from_torch(model, (224, 224), precision="fp32", max_batch=128)
    lg32 = f32.forward_masked(eng.synth, d_bits, nib.KEEP_MUL)
    s32 = nib.score(lg32, 0)
    st = eng.tie_stats()
    print(f"\n[vgg16 bench-config] tie policy: {st}")
    assert np.array_equal(out["top1"].cpu().numpy(), s32["top1"].cpu().numpy()), "top-1 differs from the fp32 engine"
    assert st["overflow"] == 0, st
    amax = float(lg32.abs().max())
    rtol = float(np.expm1(2 * TOL_BF16 * amax))
    p16, p32 = out["target_prob"].cpu().numpy().astype(np.float64), s32["target_prob"].cpu().numpy().astype(np.float64)
    assert np.all(np.abs(p16 - p32) <= rtol * p32), (float((np.abs(p16 - p32) / p32).max()), rtol)


def test_imagenet_dropin_runs_vgg16(nib, tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "generate_gp_training_data_imagenet.py"), "-a", "vgg16",
                        "--synthetic", "--num_mask_samples", "256", "--no-write"],
                       capture_output=True, text=True, cwd=tmp_path, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "correct_pred_count" in r.stdout, r.stdout[-2000:]
