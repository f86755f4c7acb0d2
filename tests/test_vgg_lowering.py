"""CPU: the torchvision VGG / AlexNet recipe of classifier.py checks its input before it touches the library, and the
first Linear's weight, handed over as a KxK conv, computes the same product as torch's NCHW flatten."""
import numpy as np
import pytest
import torch
import torch.nn as nn
import torchvision.models as tvm

from network_interpretation_imagenet_b200 import _lib, classifier
from network_interpretation_imagenet_b200.classifier import Classifier


class _NoLibrary(Exception):
    pass


@pytest.fixture
def no_library(monkeypatch):
    """Any attempt to load libnib.so fails loudly: the checks under test must come first."""
    def boom(*a, **k):
        raise _NoLibrary("the library was touched")
    monkeypatch.setattr(_lib, "load", boom)


class _Done(Exception):
    pass


class _Recorder:
    """Stands in for classifier._Builder: records what the recipe hands to each nib_net_* call, stops at the fc op."""

    def __init__(self, precision, max_batch):
        self.n, self.calls = 0, []

    def buffer(self, H, W, Cc, pad=0, pooled=True, f32=False):
        self.n += 1
        self.calls.append(("buffer", self.n, (H, W, Cc, pad, f32)))
        return self.n

    def convert(self, a, b):
        self.calls.append(("convert", a, b))

    def release(self, b):
        pass

    def conv(self, in_buf, Cin, out_buf, Cout, w, b, k, stride, pad, relu, **kw):
        self.calls.append(("conv", dict(Cin=Cin, Cout=Cout, w=w.detach().clone(), k=k, stride=stride, pad=pad, relu=relu,
                                        in_buf=in_buf, out_buf=out_buf)))

    def pool(self, kind, in_buf, Cc, out_buf, k, stride, pad, **kw):
        self.calls.append(("pool", (k, stride, pad)))

    def fc(self, in_buf, Cin, Cout, w, b):
        self.calls.append(("fc", Cin, Cout))
        raise _Done()


def _record(monkeypatch, model, precision, hw=(224, 224)):
    monkeypatch.setattr(classifier, "_Builder", _Recorder)
    rec = {}
    orig = _Recorder.__init__

    def init(self, *a):
        orig(self, *a)
        rec["r"] = self
    monkeypatch.setattr(_Recorder, "__init__", init)
    with pytest.raises(_Done):
        Classifier.from_torch(model, hw, precision=precision, max_batch=4)
    return rec["r"].calls


def test_ceil_mode_pool_is_rejected_before_the_library(no_library):
    m = tvm.vgg11(weights=None)
    m.features[2] = nn.MaxPool2d(2, 2, ceil_mode=True)
    with pytest.raises(TypeError, match="MaxPool2d"):
        Classifier.from_torch(m, (224, 224), precision="bf16")


def test_grouped_conv_is_rejected_before_the_library(no_library):
    m = tvm.vgg11(weights=None)
    m.features[3] = nn.Conv2d(64, 128, 3, padding=1, groups=2)
    with pytest.raises(TypeError, match="Conv2d"):
        Classifier.from_torch(m, (224, 224), precision="bf16")


def test_input_size_without_identity_avgpool_is_rejected_before_the_library(no_library):
    with pytest.raises(ValueError, match="avgpool"):
        Classifier.from_torch(tvm.vgg16(weights=None), (256, 256), precision="bf16")


def test_squeezenet_still_raises_type_error(no_library):
    with pytest.raises(TypeError):
        Classifier.from_torch(tvm.squeezenet1_0(weights=None), (224, 224), precision="bf16")


def test_split_rejects_widths_off_the_64_channel_grid(no_library):
    m = tvm.vgg11(weights=None)
    m.features[3] = nn.Conv2d(64, 96, 3, padding=1)
    m.features[6] = nn.Conv2d(96, 256, 3, padding=1)
    with pytest.raises(TypeError, match="split"):
        Classifier.from_torch(m, (224, 224), precision="split")


@pytest.mark.parametrize("arch,K,C", [("vgg16", 7, 512), ("alexnet", 6, 256)])
def test_fc6_reshape_matches_the_nchw_flatten(monkeypatch, arch, K, C):
    """Repack the weight the recipe hands to nib_net_add_conv as net.cu does ([Cout][Cin][R][S] -> [Cout][R][S][Cin]) and
    apply it to the NHWC-flattened features: the product must equal torch's flatten(x) @ W.T in fp64."""
    model = getattr(tvm, arch)(weights=None).eval()
    calls = _record(monkeypatch, model, "bf16")
    convs = [c[1] for c in calls if c[0] == "conv"]
    fc6 = next(c for c in convs if c["k"] == K and c["Cin"] == C)
    assert (fc6["stride"], fc6["pad"], fc6["Cout"]) == (1, 0, 4096)
    w = fc6["w"].double().numpy()                                        # [Cout][Cin][R][S]
    krsc = np.ascontiguousarray(w.transpose(0, 2, 3, 1)).reshape(w.shape[0], -1)
    g = torch.Generator().manual_seed(0)
    x = torch.randn(3, C, K, K, generator=g, dtype=torch.float64)       # NCHW features
    nhwc = x.permute(0, 2, 3, 1).reshape(3, -1).numpy()
    got = nhwc @ krsc.T
    want = (torch.flatten(x, 1) @ model.classifier[1 if arch == "alexnet" else 0].weight.detach().double().T).numpy()
    np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("arch", ["vgg11", "vgg16_bn", "alexnet"])
@pytest.mark.parametrize("precision", ["bf16", "fp32", "split"])
def test_recipe_op_sequence(monkeypatch, arch, precision):
    """Every conv and Linear becomes one conv op (the last Linear the fc op); the bf16 input is 8-channel pixels in a
    1-pixel halo for a 3x3 first conv; split converts around every pool, around VGG's fc6 and before the fc."""
    model = getattr(tvm, arch)(weights=None).eval()
    calls = _record(monkeypatch, model, precision)
    n_conv = sum(isinstance(m, nn.Conv2d) for m in model.features) + 2
    convs = [c[1] for c in calls if c[0] == "conv"]
    assert len(convs) == n_conv
    assert [c["relu"] for c in convs[-2:]] == [True, True]
    assert calls[-1] == ("fc", 4096, 1000)
    x_in = calls[0][2]
    if precision == "bf16" and arch.startswith("vgg"):
        assert x_in == (224, 224, 8, 1, False)
    else:
        assert x_in[2:4] == (4, 0)
    n_pool = sum(isinstance(m, nn.MaxPool2d) for m in model.features)
    assert sum(c[0] == "pool" for c in calls) == n_pool
    if precision == "split":
        # the first conv and the pools read and write fp32 buffers, every other conv split tensors: a convert sits on each
        # boundary between the two, and before the fc
        seq = [c[0] for c in calls if c[0] != "buffer"]
        kind = {}
        for c in calls:
            if c[0] == "buffer":
                kind[c[1]] = "f32" if c[2][4] else "split"
        assert kind[convs[0]["in_buf"]] == kind[convs[0]["out_buf"]] == "f32"
        for c in convs[1:]:   # a reduction longer than 16384 (VGG's fc6) stays on fp32 buffers: CUDA cores, fp32 accumulate
            want = "f32" if c["Cin"] * c["k"] ** 2 > 16384 else "split"
            assert kind[c["in_buf"]] == kind[c["out_buf"]] == want, (c["Cin"], c["k"])
        assert seq[-2] == "convert"
        for i, s in enumerate(seq):
            if s == "pool":
                assert seq[i - 1] == "convert" or (seq[i - 1] == "conv" and i - 1 == seq.index("conv"))
    else:
        assert not any(c[0] == "convert" for c in calls)
