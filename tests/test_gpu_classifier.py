"""GPU: stage 2 (classifier forward + scoring) through the C ABI.

Floating-point kernels: compared with the oracle's torch fp32 CPU forward (the reference's `model(x)`,
generate_gp_training_data_imagenet.py:246).  Tolerances are north_star's: <= 1e-4 (fp32 mode), <= 1e-2 (bf16 mode),
stated element-wise against each row's own scale: |a - b| <= tol * max_k |b[n, k]| for every logit of every input n
(a logit that crosses zero has no meaningful per-element relative error; the row maximum is the scale its arg-max and
softmax live on).  Identical top-1 on EVERY input is the engine's contract (raw classifier + tie policy) and is tested at
the engine level (tests/test_gpu_engine.py, tests/test_gpu_bench_config.py); here the raw classifier must agree wherever
the reference's own top-2 margin exceeds the band the logit tolerance allows."""
import ctypes as C
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import classifier as ocls
from oracle import scoring as oscore
from oracle import synthetic

pytestmark = pytest.mark.gpu

TOL_FP32 = 1e-4
TOL_BF16 = 1e-2


def rel_err(a, b):
    """Largest |a - b| relative to the row's own max |b| (2-D logits [N, K]; other shapes: the tensor's max |b|)."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    if a.ndim == 2:
        return float((np.abs(a - b) / np.maximum(np.abs(b).max(axis=1, keepdims=True), 1e-30)).max())
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


# ---- tcgen05 GEMM descriptors ---------------------------------------------------------------------
@pytest.mark.parametrize("M,N,K", [(128, 128, 64), (256, 64, 128), (300, 256, 256), (1000, 32, 576), (4096, 128, 1024)])
def test_tc_gemm(nib, M, N, K):
    lib = nib._lib.load()
    g = torch.Generator().manual_seed(M + N + K)
    A = (torch.randn(M, K, generator=g) * 0.5).to(torch.bfloat16).cuda()
    B = (torch.randn(N, K, generator=g) * 0.5).to(torch.bfloat16).cuda()
    Cd = torch.zeros(M, N, dtype=torch.float32, device="cuda")
    nib._lib.check(lib.nib_tc_gemm_bf16(A.data_ptr(), B.data_ptr(), Cd.data_ptr(), M, N, K, nib._lib.stream_handle()),
                   "nib_tc_gemm_bf16")
    torch.cuda.synchronize()
    ref = A.float() @ B.float().t()
    err = (Cd - ref).abs().max().item()
    assert err <= 1e-3 * max(1.0, ref.abs().max().item()), f"max abs err {err}"


# ---- single convolutions through a one-layer network -------------------------------------------------
def _one_conv_net(nib, precision, Cin, Cout, k, stride, pad, H, W, relu, residual, N, seed, tensor_core=True):
    from network_interpretation_imagenet_b200 import _lib
    from network_interpretation_imagenet_b200.classifier import _Builder, Classifier, _out_hw
    g = torch.Generator().manual_seed(seed)
    w = torch.randn(Cout, Cin, k, k, generator=g) / np.sqrt(Cin * k * k)
    bias = torch.randn(Cout, generator=g) * 0.1
    x = torch.randn(N, Cin, H, W, generator=g)
    b = _Builder({"fp32": _lib.PREC_FP32, "bf16": _lib.PREC_BF16, "x3": _lib.PREC_X3}[precision], N)
    x_in = b.buffer(H, W, Cin, pooled=False)
    Ho, Wo = _out_hw(H, k, stride, pad), _out_hw(W, k, stride, pad)
    res_buf = None
    xin2 = x_in
    if residual:   # residual = a 1x1 stride-matched projection of the input computed first (same engine, SIMT-checked separately)
        res_buf = b.buffer(Ho, Wo, Cout, pooled=False)
        wr = torch.randn(Cout, Cin, 1, 1, generator=g) / np.sqrt(Cin)
        b.conv(x_in, Cin, res_buf, Cout, wr, None, 1, stride, 0, relu=False)
    out = b.buffer(Ho, Wo, Cout, pooled=False)
    b.conv(xin2, Cin, out, Cout, w, bias, k, stride, pad, relu=relu, res=res_buf, res_C=Cout if residual else 0)
    feat = b.buffer(1, 1, Cout)
    if Ho == Wo:
        b.pool(_lib.POOL_AVG, out, Cout, feat, Ho, Ho, 0)
    b.fc(feat, Cout, 4, torch.zeros(4, Cout), None)
    net = Classifier(b, x_in, (Cin, H, W), 4, precision, N, taps={"out": out, "res": res_buf})
    net.set_tensor_core(tensor_core)
    net.forward(x.cuda())
    got = net.read_tap("out", N).cpu()
    if precision == "bf16":
        xr, wq = x.to(torch.bfloat16).float(), w.to(torch.bfloat16).float()
    else:
        xr, wq = x, w
    ref = F.conv2d(xr.double(), wq.double(), bias.double(), stride=stride, padding=pad)
    if residual:
        wrq = wr.to(torch.bfloat16).float() if precision == "bf16" else wr
        r = F.conv2d(xr.double(), wrq.double(), None, stride=stride)
        if precision == "bf16":
            r = r.float().to(torch.bfloat16).double()
        ref = ref + r
    if relu:
        ref = ref.clamp_min(0)
    return got.double(), ref, net


CONV_CASES = [
    # Cin, Cout, k, stride, pad, H,  W,  relu, residual
    (64, 64, 1, 1, 0, 16, 16, True, False),
    (64, 256, 1, 1, 0, 14, 14, False, True),
    (256, 64, 1, 1, 0, 14, 14, True, False),
    (64, 64, 3, 1, 1, 16, 16, True, False),
    (128, 128, 3, 1, 1, 14, 14, True, False),
    (128, 128, 3, 2, 1, 28, 28, True, False),
    (256, 512, 1, 2, 0, 28, 28, False, False),
    (128, 32, 3, 1, 1, 7, 7, False, False),
    (512, 512, 3, 1, 1, 7, 7, True, True),
    # 3x3 64 -> 64 on the resident input patch (conv_tc.cu TC_A_HALO): 2 / 4 / 8 image rows per tile; N = 5 images
    # makes the tile count odd, so one CTA of the last pair runs past the batch
    (64, 64, 3, 1, 1, 56, 56, True, False),
    (64, 64, 3, 1, 1, 32, 30, False, False),
    (64, 64, 3, 1, 1, 16, 14, True, False),
    # same mode with two channel blocks and 32 outputs (DenseNet growth convs): 64-byte output rows under the 64B swizzle
    (128, 32, 3, 1, 1, 56, 56, False, False),
    (128, 32, 3, 1, 1, 28, 28, True, False),
    (64, 32, 3, 1, 1, 16, 14, True, False),
    (128, 32, 3, 1, 1, 14, 14, False, False),     # 7 image rows per tile (8 fit, 7 divides the height)
    (128, 32, 3, 1, 1, 7, 7, True, False),        # one 7x7 image per tile
]


@pytest.mark.parametrize("case", CONV_CASES, ids=lambda c: "cin%d_cout%d_k%d_s%d_h%d_w%d" % (c[0], c[1], c[2], c[3], c[5], c[6]))
def test_conv_tcgen05_vs_torch(nib, case):
    Cin, Cout, k, stride, pad, H, W, relu, residual = case
    got, ref, net = _one_conv_net(nib, "bf16", Cin, Cout, k, stride, pad, H, W, relu, residual, N=5, seed=sum(case[:7]))
    total, tc = net.launch_counts()
    assert tc >= 1, "the tcgen05 path did not run for an eligible layer"
    err = (got - ref).abs().max().item()
    scale = max(ref.abs().max().item(), 1.0)
    assert err <= 1.2e-2 * scale, f"max abs err {err} (scale {scale})"   # bf16 output rounding = 2^-9 rel + accum


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("case", [(3, 64, 7, 2, 3, 32, 32, True, False), (16, 32, 3, 2, 1, 16, 16, True, False),
                                  (64, 128, 3, 1, 1, 9, 9, False, True), (1, 32, 3, 1, 1, 28, 28, True, False)],
                         ids=lambda c: "cin%d_cout%d_k%d_s%d" % (c[0], c[1], c[2], c[3]))
def test_conv_simt_vs_torch(nib, precision, case):
    Cin, Cout, k, stride, pad, H, W, relu, residual = case
    got, ref, net = _one_conv_net(nib, precision, Cin, Cout, k, stride, pad, H, W, relu, residual, N=3,
                                  seed=sum(case[:7]), tensor_core=False)
    err = (got - ref).abs().max().item()
    scale = max(ref.abs().max().item(), 1.0)
    assert err <= (1e-5 if precision == "fp32" else 1.2e-2) * scale


def _one_split_conv(nib, Cin, Cout, k, stride, pad, H, relu, residual, N, seed):
    """One conv on split-bf16 tensors (tcgen05 pair kernel, split mode) between two fp32 <-> split converts."""
    from network_interpretation_imagenet_b200 import _lib
    from network_interpretation_imagenet_b200.classifier import _Builder, Classifier, _out_hw
    g = torch.Generator().manual_seed(seed)
    w = torch.randn(Cout, Cin, k, k, generator=g) / np.sqrt(Cin * k * k)
    bias = torch.randn(Cout, generator=g) * 0.1
    x = torch.randn(N, Cin, H, H, generator=g)
    b = _Builder(_lib.PREC_SPLIT, N)
    x_in = b.buffer(H, H, Cin, pooled=False, f32=True)
    xs = b.buffer(H, H, Cin, pooled=False)
    b.convert(x_in, xs)
    Ho = _out_hw(H, k, stride, pad)
    res_buf, wr = None, None
    if residual:
        res_buf = b.buffer(Ho, Ho, Cout, pooled=False)
        wr = torch.randn(Cout, Cin, 1, 1, generator=g) / np.sqrt(Cin)
        b.conv(xs, Cin, res_buf, Cout, wr, None, 1, stride, 0, relu=False)
    out = b.buffer(Ho, Ho, Cout, pooled=False)
    b.conv(xs, Cin, out, Cout, w, bias, k, stride, pad, relu=relu, res=res_buf, res_C=Cout if residual else 0)
    of = b.buffer(Ho, Ho, Cout, pooled=False, f32=True)
    b.convert(out, of)
    feat = b.buffer(1, 1, Cout, f32=True)
    b.pool(_lib.POOL_AVG, of, Cout, feat, Ho, Ho, 0)
    b.fc(feat, Cout, 4, torch.zeros(4, Cout), None)
    net = Classifier(b, x_in, (Cin, H, H), 4, "split", N, taps={"out": of})
    net.forward(x.cuda())
    got = net.read_tap("out", N).cpu().double()
    ref = F.conv2d(x.double(), w.double(), bias.double(), stride=stride, padding=pad)
    if residual:
        ref = ref + F.conv2d(x.double(), wr.double(), None, stride=stride)
    if relu:
        ref = ref.clamp_min(0)
    return got, ref, net


SPLIT_CASES = [
    # Cin, Cout, k, stride, pad, H, relu, residual
    (64, 64, 1, 1, 0, 16, True, False),
    (64, 64, 3, 1, 1, 16, True, False),
    (64, 256, 1, 1, 0, 14, True, True),
    (256, 64, 1, 1, 0, 14, True, False),
    (128, 128, 3, 2, 1, 28, True, False),
    (256, 256, 3, 1, 1, 14, True, False),
    (256, 512, 1, 2, 0, 28, False, False),
    (128, 512, 1, 1, 0, 9, True, True),
    (512, 512, 3, 1, 1, 7, True, True),
    (64, 128, 3, 1, 1, 33, True, True),          # ragged M (5 x 33 x 33 rows), BLOCK_N = 128 with residual
]


@pytest.mark.parametrize("case", SPLIT_CASES, ids=lambda c: "cin%d_cout%d_k%d_s%d_h%d_res%d" % (c[0], c[1], c[2], c[3], c[5], c[7]))
def test_conv_split_tcgen05_vs_torch(nib, case):
    """conv_tc3_kernel in split mode: activations [hi | lo], weights [Wh | Wh | Wl], both halves of the fp32 result stored
    (and both halves of the residual added): fp32-grade against torch fp64."""
    Cin, Cout, k, stride, pad, H, relu, residual = case
    got, ref, net = _one_split_conv(nib, Cin, Cout, k, stride, pad, H, relu, residual, N=5, seed=sum(case[:6]))
    total, tc = net.launch_counts()
    assert tc == (2 if residual else 1), "the split convs did not take the tcgen05 path"
    err = (got - ref).abs().max().item()
    scale = max(ref.abs().max().item(), 1.0)
    assert err <= 3e-5 * scale, f"max abs err {err} (scale {scale})"


def test_split_mode_resnets(nib):
    """The tie policy's re-score lowering for torchvision ResNets: within the fp32 tolerance (1e-4) of the torch fp32 forward
    and 5e-5 of the CUDA-core fp32 lowering, bottleneck (ResNet-101) and basic-block (ResNet-18) bodies."""
    for arch, n in (("resnet101", 3), ("resnet18", 5)):
        m = ocls.build_imagenet_model(arch)
        x = torch.from_numpy(synthetic.synthetic_image("imagenet"))[None].repeat(n, 1, 1, 1)
        x[1] = x[1].flip(2) * 0.5
        x[2] = x[2] * (torch.rand(1, 224, 224, generator=torch.Generator().manual_seed(3)) > 0.5).float()
        net, got, want = _check_net(nib, m, x, "split", TOL_FP32)
        total, tc = net.launch_counts()
        assert tc >= (100 if arch == "resnet101" else 19), (arch, tc)
        ref32 = nib.Classifier.from_torch(m, (224, 224), precision="fp32", max_batch=n).forward(x.cuda()).cpu().numpy()
        assert rel_err(got, ref32) <= 5e-5, arch
        assert np.array_equal(got.argmax(1), ref32.argmax(1))
    with pytest.raises(TypeError):
        nib.Classifier.from_torch(ocls.load_resnet56(), (32, 32), precision="split", max_batch=4)


X3_CASES = [
    # Cin, Cout, k, stride, pad, H,  W,  relu, residual
    (16, 16, 3, 1, 1, 32, 32, True, True),       # ResNet-56 stage 1 (K = 144: half a slab of tail)
    (32, 64, 3, 2, 1, 16, 16, True, False),
    (64, 256, 1, 1, 0, 14, 14, False, True),
    (256, 64, 1, 1, 0, 9, 9, True, False),
    (256, 256, 3, 1, 1, 14, 14, True, False),
    (512, 1000, 1, 1, 0, 3, 3, False, False),    # ragged Cout: 1000 = 7 x 128 + 104
    (128, 32, 3, 1, 1, 7, 7, False, False),
]


@pytest.mark.parametrize("case", X3_CASES, ids=lambda c: "cin%d_cout%d_k%d_s%d_h%d" % (c[0], c[1], c[2], c[3], c[5]))
def test_conv_x3_vs_torch(nib, case):
    """Split-bf16 tensor-core conv (conv_x3.cu): fp32 in / out, products hi*hi + lo*hi + hi*lo, against torch fp64."""
    Cin, Cout, k, stride, pad, H, W, relu, residual = case
    got, ref, net = _one_conv_net(nib, "x3", Cin, Cout, k, stride, pad, H, W, relu, residual, N=5, seed=sum(case[:7]))
    err = (got - ref).abs().max().item()
    scale = max(ref.abs().max().item(), 1.0)
    assert err <= 2e-5 * scale, f"max abs err {err} (scale {scale})"
    got32, _, _ = _one_conv_net(nib, "fp32", Cin, Cout, k, stride, pad, H, W, relu, residual, N=5, seed=sum(case[:7]))
    assert (got - got32).abs().max().item() <= 2e-5 * scale


@pytest.mark.parametrize("cpix", [8, 4])
@pytest.mark.parametrize("H", [224, 64, 50])
def test_stem_7x7_tcgen05_vs_torch(nib, H, cpix):
    """torchvision conv1 (7x7/2, pad 3, Cin=3) through the overlapping-window TMA map: one output row per tile."""
    from network_interpretation_imagenet_b200 import _lib
    from network_interpretation_imagenet_b200.classifier import _Builder, Classifier, _out_hw
    g = torch.Generator().manual_seed(H)
    N, Cout = 3, 64
    w = torch.randn(Cout, 3, 7, 7, generator=g) / np.sqrt(147)
    bias = torch.randn(Cout, generator=g) * 0.1
    x = torch.randn(N, 3, H, H, generator=g)
    b = _Builder(_lib.PREC_BF16, N)
    x_in = b.buffer(H, H, cpix, pad=3, pooled=False)   # 8-channel pixels: one filter row per K block; 4: row pairs
    Ho = _out_hw(H, 7, 2, 3)
    out = b.buffer(Ho, Ho, Cout, pooled=False)
    b.conv(x_in, 3, out, Cout, w, bias, 7, 2, 3, relu=True)
    feat = b.buffer(1, 1, Cout)
    b.pool(_lib.POOL_AVG, out, Cout, feat, Ho, Ho, 0)
    b.fc(feat, Cout, 4, torch.zeros(4, Cout), None)
    net = Classifier(b, x_in, (3, H, H), 4, "bf16", N, taps={"out": out})
    net.forward(x.cuda())
    total, tc = net.launch_counts()
    assert tc == 1, "the stem did not take the tcgen05 path"
    got = net.read_tap("out", N).cpu().double()
    ref = F.conv2d(x.to(torch.bfloat16).double(), w.to(torch.bfloat16).double(), bias.double(), stride=2, padding=3).clamp_min(0)
    err = (got - ref).abs().max().item()
    assert err <= 1.2e-2 * max(ref.abs().max().item(), 1.0), err
    net.set_tensor_core(False)     # same buffers through the CUDA-core kernel
    net.forward(x.cuda())
    got2 = net.read_tap("out", N).cpu().double()
    assert (got2 - ref).abs().max().item() <= 1.2e-2 * max(ref.abs().max().item(), 1.0)


@pytest.mark.parametrize("kind,k,s,p", [("max", 3, 2, 1), ("avg", 2, 2, 0), ("avg", 7, 7, 0)])
def test_pool_bf16_vector_path_vs_torch(nib, kind, k, s, p):
    from network_interpretation_imagenet_b200 import _lib
    from network_interpretation_imagenet_b200.classifier import _Builder, Classifier, _out_hw
    g = torch.Generator().manual_seed(k)
    N, Cc, H = 3, 64, 14
    x = torch.randn(N, Cc, H, H, generator=g)
    b = _Builder(_lib.PREC_BF16, N)
    x_in = b.buffer(H, H, Cc, pooled=False)
    Ho = _out_hw(H, k, s, p)
    out = b.buffer(Ho, Ho, Cc, pooled=False)
    b.pool(_lib.POOL_MAX if kind == "max" else _lib.POOL_AVG, x_in, Cc, out, k, s, p)
    feat = b.buffer(1, 1, Cc)
    b.pool(_lib.POOL_AVG, out, Cc, feat, Ho, Ho, 0)
    b.fc(feat, Cc, 4, torch.zeros(4, Cc), None)
    # a conv must read the input buffer for the NCHW staging to know the channel count: identity-free trick — use Cin=Cc
    net = Classifier(b, x_in, (Cc, H, H), 4, "bf16", N, taps={"out": out})
    net.forward(x.cuda())
    got = net.read_tap("out", N).cpu()
    xb = x.to(torch.bfloat16).float()
    ref = F.max_pool2d(xb, k, s, p) if kind == "max" else F.avg_pool2d(xb, k, s, p)
    assert (got - ref.to(torch.bfloat16).float()).abs().max().item() <= 2e-2 * ref.abs().max().item()


# ---- whole networks ------------------------------------------------------------------------------------
def _check_net(nib, model, x, precision, tol, max_batch=None):
    want = ocls.forward_logits(model, x).numpy()
    net = nib.Classifier.from_torch(model, tuple(x.shape[2:]), precision=precision, max_batch=max_batch or x.shape[0])
    got = net.forward(torch.as_tensor(x).cuda()).cpu().numpy()
    err = rel_err(got, want)
    assert err <= tol, f"{precision}: rel err {err:.3e} > {tol}"
    # top-1 must agree wherever the reference's own top-2 margin is outside the logit tolerance band; inside it
    # the engine's tie policy (PerturbationEngine.refine_ties, tested in test_gpu_engine.py) re-scores in fp32.
    srt = np.sort(want, 1)
    decided = (srt[:, -1] - srt[:, -2]) > 2 * tol * np.abs(want).max(axis=1)
    assert np.array_equal(got.argmax(1)[decided], want.argmax(1)[decided]), "top-1 differs outside the tie band"
    return net, got, want


def test_mnist_net_fp32_with_taps(nib):
    m = ocls.load_mnist_net()
    x = torch.rand(16, 1, 28, 28, generator=torch.Generator().manual_seed(3))
    net, got, want = _check_net(nib, m, x, "fp32", TOL_FP32)
    with torch.no_grad():
        x0, x1, x2, _ = m(x)
    for name, ref in (("x0", x0), ("x1", x1), ("x2", x2)):
        tap = net.read_tap(name, 16).cpu().numpy()
        assert rel_err(tap, ref.numpy()) <= TOL_FP32, name


def test_mnist_net_fp32_golden(nib, golden_dir):
    """Against the output of the reference's own Classification_Net class (tests/golden/make_golden.py make_mnist_net)."""
    g = np.load(os.path.join(golden_dir, "mnist_net.npz"))
    net = nib.Classifier.from_torch(ocls.load_mnist_net(), (28, 28), precision="fp32", max_batch=4)
    got = net.forward(torch.from_numpy(g["x"]).cuda()).cpu().numpy()
    assert rel_err(got, g["pred0"]) <= TOL_FP32
    assert rel_err(net.read_tap("x2", 4).cpu().numpy(), g["x2"]) <= TOL_FP32
    assert np.array_equal(got.argmax(1), g["pred0"].argmax(1))


def test_mnist_net_bf16(nib):
    m = ocls.load_mnist_net()
    x = torch.rand(64, 1, 28, 28, generator=torch.Generator().manual_seed(4))
    _check_net(nib, m, x, "bf16", TOL_BF16)


def test_resnet56_fp32_checkpoint_and_golden(nib, golden_dir):
    g = np.load(os.path.join(golden_dir, "resnet56.npz"))
    m = ocls.load_resnet56()
    net = nib.Classifier.from_torch(m, (32, 32), precision="fp32", max_batch=4)
    got = net.forward(torch.from_numpy(g["x"]).cuda()).cpu().numpy()
    assert rel_err(got, g["logits"]) <= TOL_FP32          # the reference's own module output
    x = torch.rand(32, 3, 32, 32, generator=torch.Generator().manual_seed(9))
    _check_net(nib, m, x, "fp32", TOL_FP32, max_batch=16)  # also exercises chunking over max_batch


RESNET56_BF16_MEASURED_TOL = 3e-2


def test_resnet56_bf16_is_outside_the_stated_tolerance_and_says_so(nib):
    """ResNet-56 in bf16 does NOT meet north_star's 1e-2: 55 sequential layers each round their output to 8 mantissa bits
    and the identity residual stream carries the noise to the end (row-wise error 1e-2 .. 3e-2 on the shipped
    checkpoint).  BASELINE configs[1] is therefore served at fp32 grade (generate_gp_training_data_cifar.py defaults to
    --precision x3: split-bf16 products on the tensor cores, <= 1e-4, test_x3_mode_whole_networks; --precision fp32 is the
    CUDA-core lowering, test_resnet56_fp32_checkpoint_and_golden); bf16 stays available for this net with the band
    below, and this test pins that band so a silent regression (or a fix) shows up."""
    m = ocls.load_resnet56()
    x = torch.rand(64, 3, 32, 32, generator=torch.Generator().manual_seed(10))
    want = ocls.forward_logits(m, x).numpy()
    net = nib.Classifier.from_torch(m, (32, 32), precision="bf16", max_batch=64)
    got = net.forward(x.cuda()).cpu().numpy()
    err = rel_err(got, want)
    print(f"\n[resnet56 bf16] row-wise relative logit error {err:.3e} (north_star 1e-2; accepted band {RESNET56_BF16_MEASURED_TOL:g})")
    assert err <= RESNET56_BF16_MEASURED_TOL
    srt = np.sort(want, 1)
    safe = (srt[:, -1] - srt[:, -2]) > 2 * RESNET56_BF16_MEASURED_TOL * np.abs(want).max(axis=1)
    assert np.array_equal(got.argmax(1)[safe], want.argmax(1)[safe])


def test_x3_mode_whole_networks(nib):
    """The tie policy's re-score precision: every network within the fp32 tolerance (1e-4) of the torch fp32 forward, and
    within 5e-5 of the CUDA-core fp32 lowering."""
    m = ocls.build_imagenet_model("resnet101")
    x = torch.from_numpy(synthetic.synthetic_image("imagenet"))[None].repeat(3, 1, 1, 1)
    x[1] = x[1].flip(2) * 0.5
    x[2] = x[2] * (torch.rand(1, 224, 224, generator=torch.Generator().manual_seed(3)) > 0.5).float()
    net, got, want = _check_net(nib, m, x, "x3", TOL_FP32)
    ref32 = nib.Classifier.from_torch(m, (224, 224), precision="fp32", max_batch=3).forward(x.cuda()).cpu().numpy()
    assert rel_err(got, ref32) <= 5e-5
    assert np.array_equal(got.argmax(1), ref32.argmax(1))
    m56 = ocls.load_resnet56()
    x56 = torch.rand(32, 3, 32, 32, generator=torch.Generator().manual_seed(9))
    _check_net(nib, m56, x56, "x3", TOL_FP32, max_batch=16)
    mm = ocls.load_mnist_net()
    _check_net(nib, mm, torch.rand(16, 1, 28, 28, generator=torch.Generator().manual_seed(3)), "x3", TOL_FP32)
    md = ocls.build_imagenet_model("densenet121")
    xd = torch.from_numpy(synthetic.synthetic_image("imagenet"))[None].repeat(2, 1, 1, 1)
    xd[1] = xd[1].flip(1)
    _check_net(nib, md, xd, "x3", TOL_FP32)


def test_resnet101_fp32(nib):
    m = ocls.build_imagenet_model("resnet101")
    x = torch.from_numpy(synthetic.synthetic_image("imagenet"))[None].repeat(2, 1, 1, 1)
    x[1] = x[1].flip(2) * 0.5
    _check_net(nib, m, x, "fp32", TOL_FP32)


def test_resnet101_bf16_tcgen05(nib):
    m = ocls.build_imagenet_model("resnet101")
    g = torch.Generator().manual_seed(2)
    base = torch.from_numpy(synthetic.synthetic_image("imagenet"))
    x = base[None] * (torch.rand(8, 1, 224, 224, generator=g) > 0.4).float()
    net, got, want = _check_net(nib, m, x, "bf16", TOL_BF16)
    total, tc = net.launch_counts()
    # 104 convs on the tensor path; 29 of the 1x1 reductions ride in the previous expansion's fused launch (NIB_TC_FUSE)
    assert tc >= (100 if os.environ.get("NIB_TC_FUSE") == "0" else 75), f"only {tc} tcgen05 launches for ResNet-101"


def test_densenet121_fp32(nib):
    m = ocls.build_imagenet_model("densenet121")
    x = torch.from_numpy(synthetic.synthetic_image("imagenet"))[None].repeat(2, 1, 1, 1)
    x[1] = x[1].flip(1)
    _check_net(nib, m, x, "fp32", TOL_FP32)


def test_densenet121_bf16(nib):
    m = ocls.build_imagenet_model("densenet121")
    x = torch.from_numpy(synthetic.synthetic_image("imagenet"))[None].repeat(4, 1, 1, 1)
    x = x * torch.rand(4, 1, 1, 1, generator=torch.Generator().manual_seed(1))
    net, got, want = _check_net(nib, m, x, "bf16", TOL_BF16)
    total, tc = net.launch_counts()
    # stem + 58 bottleneck 1x1 (BN-ReLU applied to the A tiles inside the pair kernel) + 58 3x3 + 3 transitions
    assert tc >= 118, f"only {tc} tcgen05 launches for DenseNet-121 (expected 120 convs on the tensor path)"
    # from the op list: input staging + one launch per op that is not a tcgen05 conv.  A pre-activated conv that fell
    # back to the pack pass would add one launch of its own
    kinds = [k for _, k, _, _ in net.profile(4)]
    assert tc == sum(k == 1 for k in kinds)
    assert total - tc == 1 + sum(k not in (1, 4) for k in kinds), f"{total - tc} non-tcgen05 launches: a pack pass ran"


def test_densenet_cifar_fp32(nib):
    torch.manual_seed(5)
    m = ocls.DenseNetCifar(depth=22, growth_rate=12, num_init_features=24, bn_size=4).eval()
    ocls._randomize_bn(m, 6)
    x = torch.rand(8, 3, 32, 32, generator=torch.Generator().manual_seed(7))
    _check_net(nib, m, x, "fp32", TOL_FP32)


def test_graph_replay_matches_eager(nib):
    m = ocls.load_resnet56()
    x = torch.rand(8, 3, 32, 32, generator=torch.Generator().manual_seed(12)).cuda()
    net = nib.Classifier.from_torch(m, (32, 32), precision="fp32", max_batch=8)
    a = net.forward(x).clone()
    net.set_graph(True)
    out = torch.empty_like(a)
    b1 = net.forward(x, out=out).clone()
    b2 = net.forward(x, out=out).clone()
    assert torch.equal(a, b1) and torch.equal(a, b2)


# ---- scoring --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,K", [(1, 10), (257, 1000), (64, 10), (5, 1001)])
def test_score_vs_oracle(nib, N, K):
    g = torch.Generator().manual_seed(N * K)
    logits = torch.randn(N, K, generator=g) * 3
    logits[0, K // 2] = logits[0].max() + 1
    if N > 1:
        logits[1, 3] = logits[1, 7] = logits[1].max() + 2   # a tie: torch.max returns the first index
    target = 3
    top1, tp, mp, corr = oscore.score(logits, target)
    s = nib.score(logits.cuda(), target)
    assert np.array_equal(s["top1"].cpu().numpy(), top1)
    assert np.array_equal(s["correct"].cpu().numpy(), corr)
    np.testing.assert_allclose(s["target_prob"].cpu().numpy(), tp, rtol=2e-5, atol=1e-9)
    np.testing.assert_allclose(s["max_prob"].cpu().numpy(), mp, rtol=2e-5, atol=1e-9)


@pytest.mark.parametrize("K1,N1,N2,H", [(64, 256, 64, 12), (128, 512, 128, 9), (256, 1024, 256, 14), (256, 1024, 256, 5),
                                        (128, 256, 128, 3), (192, 768, 256, 64)])   # M = 63: the pair's second tile is all padding; 224 tiles: several per pair
def test_fused_expand_reduce_vs_torch(nib, K1, N1, N2, H):
    """conv_fused_ca_kernel: 1x1 expansion (+ residual, ReLU) and the next 1x1 reduction in one launch; both outputs (the
    N1-channel tensor that stays in global memory for the next residual, and the reduction) against torch fp32."""
    from network_interpretation_imagenet_b200 import _lib
    from network_interpretation_imagenet_b200.classifier import _Builder, Classifier
    N = 7                                               # M = 7*H*H rows: ragged last tile, odd tile counts
    g = torch.Generator().manual_seed(K1 + H)
    x = torch.randn(N, N1, H, H, generator=g)
    w0 = torch.randn(K1, N1, 1, 1, generator=g) / N1 ** 0.5
    wc = torch.randn(N1, K1, 1, 1, generator=g) / K1 ** 0.5
    bc = torch.randn(N1, generator=g) * 0.1
    wa = torch.randn(N2, N1, 1, 1, generator=g) / N1 ** 0.5
    ba = torch.randn(N2, generator=g) * 0.1
    b = _Builder(_lib.PREC_BF16, N)
    x_in = b.buffer(H, H, N1, pooled=False)
    h = b.buffer(H, H, K1, pooled=False)
    y = b.buffer(H, H, N1, pooled=False)
    o = b.buffer(H, H, N2, pooled=False)
    b.conv(x_in, N1, h, K1, w0, None, 1, 1, 0, relu=True)
    b.conv(h, K1, y, N1, wc, bc, 1, 1, 0, relu=True, res=x_in, res_C=N1)      # expansion + residual
    b.conv(y, N1, o, N2, wa, ba, 1, 1, 0, relu=True)                           # next reduction
    feat = b.buffer(1, 1, N2)
    b.pool(_lib.POOL_AVG, o, N2, feat, H, H, 0)
    b.fc(feat, N2, 4, torch.zeros(4, N2), None)
    net = Classifier(b, x_in, (N1, H, H), 4, "bf16", N, taps={"y": y, "o": o})
    total0, tc0 = net.launch_counts()
    net.forward(x.cuda())
    total1, tc1 = net.launch_counts()
    assert tc1 - tc0 == 2                               # conv0 + ONE fused launch for the two 1x1 convs
    bf = lambda t: t.to(torch.bfloat16).to(torch.float32)
    xr = bf(x)
    hr = bf(F.relu(F.conv2d(xr, bf(w0))))
    yr = bf(F.relu(F.conv2d(hr, bf(wc), bc) + xr))
    orf = F.relu(F.conv2d(yr, bf(wa), ba))
    got_y = net.read_tap("y", N).cpu()
    got_o = net.read_tap("o", N).cpu()
    assert rel_err(got_y.numpy(), yr.numpy()) <= 1.2e-2
    assert rel_err(got_o.numpy(), orf.numpy()) <= 1.2e-2
