"""Stage 2 host mirror: lowers the reference's classifiers onto the libnib.so network executor.

The reference builds its models with `import_module('models.'+arch).createModel(**kwargs)`
(generate_gp_training_data_cifar.py:71-79), `Classification_Net()` (generate_gp_training_data_mnist.py:86-107)
and `torchvision.models.__dict__[arch](pretrained=True)` (generate_gp_training_data_imagenet.py:579), then
calls `model(masked_img_tensor)` one image at a time (:246).  `Classifier.from_torch(module, ...)` walks such
a module once, folds eval-mode BatchNorm into the adjacent convolution, hands the weights to the C library
and afterwards `forward(x)` / `forward_masked(...)` run entirely in the hand-written CUDA kernels.

Recognised structures (by attributes, not class identity, so the reference's own classes, the drop-in
`models/` wrappers and torchvision all lower the same way):
  * torchvision ResNet (Bottleneck / BasicBlock)          -> resnet101 of imagenet :579
  * models/resnet.py ResNetCifar (BasicBlockWithDeathRate + DownsampleB, eval path :26-42, :71-76)
  * mnist Classification_Net (conv1..conv6 + fc1, returns (x0, x1, x2, pred0), mnist :97-105)
  * torchvision DenseNet and the CIFAR DenseNet(-BC) of models/densenet.py:44-99
  * torchvision VGG (vgg11/13/16/19, with or without BN) and AlexNet: `features / avgpool / classifier`
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch
import torch.nn as nn

from . import _lib


def _f32(t: torch.Tensor) -> np.ndarray:
    return np.ascontiguousarray(t.detach().to(torch.float32).cpu().numpy())


def fold_bn(conv_w: torch.Tensor, conv_b: torch.Tensor | None, bn: nn.BatchNorm2d | None):
    """conv -> BN(eval) == conv with w*scale, b' = beta + (b - mean)*scale,  scale = gamma/sqrt(var+eps)."""
    w = conv_w.detach().double()
    b = conv_b.detach().double() if conv_b is not None else torch.zeros(w.shape[0], dtype=torch.float64, device=w.device)
    if bn is not None:
        scale = bn.weight.detach().double() / torch.sqrt(bn.running_var.detach().double() + bn.eps)
        w = w * scale.view(-1, 1, 1, 1)
        b = bn.bias.detach().double() + (b - bn.running_mean.detach().double()) * scale
    elif conv_b is None:
        return w.float(), None
    return w.float(), b.float()


def bn_affine(bn: nn.BatchNorm2d):
    """eval BN as per-channel (scale, shift): y = x*scale + shift."""
    scale = bn.weight.detach().double() / torch.sqrt(bn.running_var.detach().double() + bn.eps)
    shift = bn.bias.detach().double() - bn.running_mean.detach().double() * scale
    return scale.float(), shift.float()


class _Builder:
    """Thin object wrapper over the nib_net_* C calls with a shape-keyed buffer pool."""

    def __init__(self, precision: int, max_batch: int):
        self.lib = _lib.load()
        h = C.c_void_p()
        _lib.check(self.lib.nib_net_create(precision, max_batch, C.byref(h)), "nib_net_create")
        self.h = h
        self.shapes: dict[int, tuple[int, int, int]] = {}
        self.free: dict[tuple[int, int, int], list[int]] = {}

    def buffer(self, H, W, Cc, pad=0, pooled=True, f32=False) -> int:
        """f32: an fp32 buffer in a network whose default buffer kind is not fp32 (NIB_PREC_SPLIT: stem, pooled features)."""
        key = (H, W, Cc, bool(f32))
        if pooled and pad == 0 and self.free.get(key):
            return self.free[key].pop()
        b = (self.lib.nib_net_add_buffer_f32 if f32 else self.lib.nib_net_add_buffer)(self.h, H, W, Cc, pad)
        if b < 0:
            _lib.check(b, "nib_net_add_buffer")
        self.shapes[b] = key
        return b

    def convert(self, in_buf: int, out_buf: int):
        """fp32 <-> split bf16 boundary of a NIB_PREC_SPLIT network."""
        _lib.check(self.lib.nib_net_add_convert(self.h, in_buf, out_buf), "nib_net_add_convert")

    def release(self, b: int):
        self.free.setdefault(self.shapes[b], []).append(b)

    def conv(self, in_buf, Cin, out_buf, Cout, w, b, k, stride, pad, relu, in_coff=0, out_coff=0, res=None, res_C=0,
             pre=None):
        d = _lib.ConvDesc()
        d.in_buf, d.in_coff, d.Cin = in_buf, in_coff, Cin
        d.out_buf, d.out_coff, d.Cout = out_buf, out_coff, Cout
        d.res_buf, d.res_coff, d.res_C = (res if res is not None else -1), 0, res_C
        d.R = d.S = k
        d.stride, d.pad = stride, pad
        d.flags = (_lib.CONV_RELU if relu else 0) | (_lib.CONV_PRE_BNRELU if pre is not None else 0)
        wn = _f32(w)
        bn_ = _f32(b) if b is not None else None
        ps = _f32(pre[0]) if pre is not None else None
        pb = _f32(pre[1]) if pre is not None else None
        _lib.check(self.lib.nib_net_add_conv(self.h, C.byref(d), wn.ctypes.data,
                                             bn_.ctypes.data if bn_ is not None else None,
                                             ps.ctypes.data if ps is not None else None,
                                             pb.ctypes.data if pb is not None else None), "nib_net_add_conv")

    def pool(self, kind, in_buf, Cc, out_buf, k, stride, pad, in_coff=0, out_coff=0, pre=None):
        ps = _f32(pre[0]) if pre is not None else None
        pb = _f32(pre[1]) if pre is not None else None
        _lib.check(self.lib.nib_net_add_pool(self.h, kind, in_buf, in_coff, Cc, out_buf, out_coff, k, stride, pad,
                                             ps.ctypes.data if ps is not None else None,
                                             pb.ctypes.data if pb is not None else None), "nib_net_add_pool")

    def fc(self, in_buf, Cin, Cout, w, b):
        wn, bn_ = _f32(w), (_f32(b) if b is not None else None)
        _lib.check(self.lib.nib_net_add_fc(self.h, in_buf, Cin, Cout, wn.ctypes.data,
                                           bn_.ctypes.data if bn_ is not None else None), "nib_net_add_fc")


def _out_hw(H, k, s, p):
    return (H + 2 * p - k) // s + 1


class Classifier:
    """A lowered classifier living in libnib.so.  `forward` returns logits [N, classes] fp32 on the device."""

    def __init__(self, builder: _Builder, in_buf: int, in_shape, num_classes: int, precision: str, max_batch: int,
                 taps=None, arch: str = ""):
        self.lib = builder.lib
        self.h = builder.h
        self.in_buf = in_buf
        self.C, self.H, self.W = in_shape
        self.num_classes = num_classes
        self.precision = precision
        self.max_batch = max_batch
        self.taps = taps or {}
        self.arch = arch
        _lib.check(self.lib.nib_net_set_input(self.h, in_buf), "nib_net_set_input")
        _lib.check(self.lib.nib_net_finalize(self.h), "nib_net_finalize")
        ptr, H, W, Cc, pad, dt = C.c_void_p(), C.c_int(), C.c_int(), C.c_int(), C.c_int(), C.c_int()
        _lib.check(self.lib.nib_net_buffer_info(self.h, in_buf, C.byref(ptr), C.byref(H), C.byref(W), C.byref(Cc),
                                                C.byref(pad), C.byref(dt)), "nib_net_buffer_info")
        self.in_c_stride, self.in_pad = Cc.value, pad.value
        self._replicas: list["Classifier"] = []     # extra copies (own activation buffers) driven from side streams
        self._streams: list = []

    def __del__(self):
        try:
            if getattr(self, "h", None):
                self.lib.nib_net_destroy(self.h)
                self.h = None
        except Exception:
            pass

    # -- construction --------------------------------------------------------------------------
    @staticmethod
    def from_torch(module: nn.Module, input_hw=None, precision: str = "bf16", max_batch: int = 128,
                   streams: int = 1) -> "Classifier":
        """streams > 1: that many copies of the lowered network (weights + activation buffers each), fed round-robin with
        consecutive micro-batches from their own CUDA streams by `forward` / `forward_masked`.  Every conv layer is a
        persistent kernel that fills the GPU, so copies do not run side by side; what overlaps is one kernel's ramp-up
        with the previous kernel's partial last wave and drain (measured +5 % on ResNet-101, tools/overlap_exp.py)."""
        c = Classifier._from_torch_one(module, input_hw, precision, max_batch)
        for _ in range(max(1, int(streams)) - 1):
            c._replicas.append(Classifier._from_torch_one(module, input_hw, precision, max_batch))
        if c._replicas:
            c._streams = [torch.cuda.Stream() for _ in range(len(c._replicas) + 1)]
        return c

    @staticmethod
    def _from_torch_one(module: nn.Module, input_hw, precision: str, max_batch: int) -> "Classifier":
        prec = {"fp32": _lib.PREC_FP32, "bf16": _lib.PREC_BF16, "x3": _lib.PREC_X3, "split": _lib.PREC_SPLIT}[precision]
        m = module.module if isinstance(module, nn.DataParallel) else module  # cifar :75 wraps in DataParallel
        if hasattr(m, "layer4") and hasattr(m, "fc") and hasattr(m, "maxpool"):
            return _lower_tv_resnet(m, input_hw or (224, 224), prec, precision, max_batch)
        if _is_plain_cnn(m):
            return _lower_tv_plain(m, input_hw or (224, 224), prec, precision, max_batch)
        if precision == "split":
            raise TypeError("precision 'split' (split-bf16 tensors on the tcgen05 pair kernel) is lowered for torchvision "
                            "ResNets, VGGs and AlexNet only (every body conv needs Cin % 64 == 0 and Cout % 64 == 0); use "
                            "'x3' for this network")
        if hasattr(m, "layer3") and hasattr(m, "fc") and not hasattr(m, "layer4"):
            return _lower_resnet_cifar(m, input_hw or (32, 32), prec, precision, max_batch)
        if hasattr(m, "conv6") and hasattr(m, "fc1"):
            return _lower_mnist(m, input_hw or (28, 28), prec, precision, max_batch)
        if hasattr(m, "features") and hasattr(m, "classifier") and hasattr(m.features, "denseblock1"):
            return _lower_tv_densenet(m, input_hw or (224, 224), prec, precision, max_batch)
        if hasattr(m, "blocks") and hasattr(m, "norm5") and hasattr(m, "classifier"):
            return _lower_densenet_cifar(m, input_hw or (32, 32), prec, precision, max_batch)
        raise TypeError(f"unsupported classifier structure: {type(m).__name__}")

    # -- execution -----------------------------------------------------------------------------
    def set_tensor_core(self, enable: bool):
        _lib.check(self.lib.nib_net_set_tensor_core(self.h, int(enable)), "nib_net_set_tensor_core")

    def set_graph(self, enable: bool):
        _lib.check(self.lib.nib_net_set_graph(self.h, int(enable)), "nib_net_set_graph")
        for r in self._replicas:
            r.set_graph(enable)

    def launch_counts(self):
        """(all kernel launches, tcgen05 launches) so far, summed over the stream copies."""
        a, b = C.c_longlong(), C.c_longlong()
        _lib.check(self.lib.nib_net_launch_counts(self.h, C.byref(a), C.byref(b)), "nib_net_launch_counts")
        ra = [r.launch_counts() for r in self._replicas]
        return a.value + sum(x[0] for x in ra), b.value + sum(x[1] for x in ra)

    def _round_robin(self, N: int, launch):
        """launch(copy, i, n) for every micro-batch [i, i+n); with stream copies, micro-batch j goes to copy j % K on its
        own stream, fenced against the caller's stream on both sides (inputs are ready, outputs are visible)."""
        if not self._replicas:
            for i in range(0, N, self.max_batch):
                launch(self, i, min(self.max_batch, N - i))
            return
        main = torch.cuda.current_stream()
        copies = [self] + self._replicas
        used = min(len(copies), (N + self.max_batch - 1) // self.max_batch)
        for s in self._streams[:used]:
            s.wait_stream(main)
        for j, i in enumerate(range(0, N, self.max_batch)):
            k = j % len(copies)
            with torch.cuda.stream(self._streams[k]):
                launch(copies[k], i, min(self.max_batch, N - i))
        for s in self._streams[:used]:
            main.wait_stream(s)

    def forward(self, x: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
        """x: [N,C,H,W] fp32 CUDA (the tensor the reference feeds `model(...)`).  Any N; chunks of max_batch."""
        if not x.is_cuda:
            raise RuntimeError("Classifier.forward needs a CUDA tensor: this engine has no CPU path")
        x = x.to(torch.float32).contiguous()
        N = int(x.shape[0])
        if tuple(x.shape[1:]) != (self.C, self.H, self.W):
            raise ValueError(f"input {tuple(x.shape)} does not match network input {(self.C, self.H, self.W)}")
        if out is None:
            out = torch.empty(N, self.num_classes, dtype=torch.float32, device=x.device)

        def launch(c, i, n):
            _lib.check(c.lib.nib_net_forward(c.h, x[i:i + n].data_ptr(), _lib.IN_NCHW_F32, n,
                                             out[i:i + n].data_ptr(), _lib.stream_handle()), "nib_net_forward")

        self._round_robin(N, launch)
        return out

    def forward_masked(self, synth, sel_bits, mode: int, out: torch.Tensor | None = None) -> torch.Tensor:
        """Fused stages 1+2: masks are synthesised directly into the network's input buffer (the masked
        batch never exists as a separate tensor), then scored.  synth: masks.MaskSynth."""
        d_sel = synth.device_bits(sel_bits)
        N = int(d_sel.shape[0])
        if out is None:
            out = torch.empty(N, self.num_classes, dtype=torch.float32, device=d_sel.device)
        if mode == _lib.MASK_REMOVE_MINMAX:
            synth.seg_minmax()   # computed (once) on the caller's stream, before the side streams fork from it

        def launch(c, i, n):
            a = synth.mask_args(d_sel[i:i + n], mode, None, 0, 0)
            _lib.check(c.lib.nib_net_forward_masked(c.h, C.byref(a), out[i:i + n].data_ptr(), _lib.stream_handle()),
                       "nib_net_forward_masked")

        self._round_robin(N, launch)
        return out

    def profile(self, N: int):
        """Per-op (ms, kind, flops) of one forward over the N images currently in the input buffer."""
        cap = 4096
        ms = (C.c_float * cap)()
        kind = (C.c_int * cap)()
        flops = (C.c_double * cap)()
        geom = (C.c_int * (8 * cap))()
        n = C.c_int()
        _lib.check(self.lib.nib_net_profile(self.h, N, ms, kind, flops, geom, cap, C.byref(n), _lib.stream_handle()),
                   "nib_net_profile")
        return [(ms[i], kind[i], flops[i], tuple(geom[8 * i:8 * i + 8])) for i in range(n.value)]

    def read_tap(self, name: str, N: int) -> torch.Tensor:
        """NCHW fp32 copy of a named intermediate (MNIST x0/x1/x2, mnist :97-105) for the last batch."""
        buf = self.taps[name]
        H, W, Cc = C.c_int(), C.c_int(), C.c_int()
        _lib.check(self.lib.nib_net_buffer_info(self.h, buf, None, C.byref(H), C.byref(W), C.byref(Cc), None, None),
                   "nib_net_buffer_info")
        out = torch.empty(N, Cc.value, H.value, W.value, dtype=torch.float32, device="cuda")
        _lib.check(self.lib.nib_net_read_buffer_nchw(self.h, buf, N, out.data_ptr(), _lib.stream_handle()),
                   "nib_net_read_buffer_nchw")
        return out


# ---- lowering recipes --------------------------------------------------------------------------------
def _in_cpad(Cin: int) -> int:
    return 4 if Cin <= 4 else Cin


def _lower_tv_resnet(m, hw, prec, precision, max_batch):
    H, W = hw
    b = _Builder(prec, max_batch)
    cin = m.conv1.in_channels
    c1 = m.conv1
    stem_tc = (precision == "bf16" and c1.kernel_size == (7, 7) and c1.stride == (2, 2) and c1.padding == (3, 3) and cin <= 8)
    # tcgen05 stem: 8-channel-padded pixels (16 B) inside a 3-pixel zero halo, so each filter row of an output pixel
    # is one contiguous 128 B window (conv_tc.cu tc_conv_is_stem)
    # 4-channel pixels (8 B) inside a 3-pixel zero halo when the image has <= 3 channels: the stem's TMA box then covers
    # two filter rows per K block (conv_tc.cu tc_conv_is_stem4); 8-channel pixels otherwise
    split = precision == "split"   # stem and pooled features in fp32 buffers, the body's tensors as bf16 [hi | lo] halves
    x_in = (b.buffer(H, W, 4 if cin <= 4 else 8, pad=3, pooled=False) if stem_tc
            else b.buffer(H, W, _in_cpad(cin), pooled=False, f32=split))
    Hc, Wc = _out_hw(H, c1.kernel_size[0], c1.stride[0], c1.padding[0]), _out_hw(W, c1.kernel_size[0], c1.stride[0], c1.padding[0])
    t = b.buffer(Hc, Wc, c1.out_channels, f32=split)
    w, bias = fold_bn(c1.weight, c1.bias, m.bn1)
    b.conv(x_in, cin, t, c1.out_channels, w, bias, c1.kernel_size[0], c1.stride[0], c1.padding[0], relu=True)
    mp = m.maxpool
    k, s, p = mp.kernel_size, mp.stride, mp.padding
    Hp, Wp = _out_hw(Hc, k, s, p), _out_hw(Wc, k, s, p)
    x = b.buffer(Hp, Wp, c1.out_channels, f32=split)
    b.pool(_lib.POOL_MAX, t, c1.out_channels, x, k, s, p)
    b.release(t)
    if split:
        xs = b.buffer(Hp, Wp, c1.out_channels)
        b.convert(x, xs)
        b.release(x)
        x = xs
    Cx, Hx, Wx = c1.out_channels, Hp, Wp
    for layer in (m.layer1, m.layer2, m.layer3, m.layer4):
        for blk in layer:
            convs = [(blk.conv1, blk.bn1), (blk.conv2, blk.bn2)]
            if hasattr(blk, "conv3"):
                convs.append((blk.conv3, blk.bn3))
            # identity / projection shortcut
            if blk.downsample is not None:
                dc, dbn = blk.downsample[0], blk.downsample[1]
                Hd, Wd = _out_hw(Hx, dc.kernel_size[0], dc.stride[0], dc.padding[0]), _out_hw(Wx, dc.kernel_size[0], dc.stride[0], dc.padding[0])
                idn = b.buffer(Hd, Wd, dc.out_channels)
                w, bias = fold_bn(dc.weight, dc.bias, dbn)
                b.conv(x, Cx, idn, dc.out_channels, w, bias, dc.kernel_size[0], dc.stride[0], dc.padding[0], relu=False)
            else:
                idn = x
            cur, Cc, Hh, Ww = x, Cx, Hx, Wx
            tmp = []
            for i, (cv, bn) in enumerate(convs):
                last = i == len(convs) - 1
                Ho, Wo = _out_hw(Hh, cv.kernel_size[0], cv.stride[0], cv.padding[0]), _out_hw(Ww, cv.kernel_size[0], cv.stride[0], cv.padding[0])
                o = b.buffer(Ho, Wo, cv.out_channels)
                w, bias = fold_bn(cv.weight, cv.bias, bn)
                if last:   # out = relu(bn(conv(.)) + identity)   (torchvision Bottleneck.forward)
                    b.conv(cur, Cc, o, cv.out_channels, w, bias, cv.kernel_size[0], cv.stride[0], cv.padding[0],
                           relu=True, res=idn, res_C=cv.out_channels)
                else:
                    b.conv(cur, Cc, o, cv.out_channels, w, bias, cv.kernel_size[0], cv.stride[0], cv.padding[0], relu=True)
                    tmp.append(o)
                cur, Cc, Hh, Ww = o, cv.out_channels, Ho, Wo
            for tbuf in tmp:
                b.release(tbuf)
            if idn != x:
                b.release(idn)
            b.release(x)
            x, Cx, Hx, Wx = cur, Cc, Hh, Ww
    if split:
        xf = b.buffer(Hx, Wx, Cx, f32=True)
        b.convert(x, xf)
        x = xf
    feat = b.buffer(1, 1, Cx, f32=split)
    assert Hx == Wx, "global average pool expects a square map"
    b.pool(_lib.POOL_AVG, x, Cx, feat, Hx, Hx, 0)   # AdaptiveAvgPool2d((1,1))
    b.fc(feat, Cx, m.fc.out_features, m.fc.weight, m.fc.bias)
    return Classifier(b, x_in, (cin, H, W), m.fc.out_features, precision, max_batch, arch="tv_resnet")


def _lower_resnet_cifar(m, hw, prec, precision, max_batch):
    H, W = hw
    b = _Builder(prec, max_batch)
    # bf16: every activation carries at least 64 physical channels (zero weights / biases for the padding), which puts
    # the 16- and 32-channel stages on the tcgen05 implicit-GEMM path (K atom = 64 channels) instead of the CUDA-core
    # kernel: 4x / 2x redundant MACs on zeros, still ~3.5x faster end to end (profiles/README.md, configs[1]).
    cp = (lambda c: max(c, 64)) if precision == "bf16" else (lambda c: c)

    def padw(w, bias, co, ci):
        if co == w.shape[0] and ci == w.shape[1]:
            return w, bias
        wp = torch.zeros(co, ci, w.shape[2], w.shape[3], dtype=w.dtype, device=w.device)
        wp[:w.shape[0], :w.shape[1]] = w
        bp = None
        if bias is not None:
            bp = torch.zeros(co, dtype=bias.dtype, device=bias.device)
            bp[:bias.shape[0]] = bias
        return wp, bp

    x_in = b.buffer(H, W, _in_cpad(3), pooled=False)
    x = b.buffer(H, W, cp(16))
    w, bias = padw(*fold_bn(m.conv1.weight, None, m.bn1), cp(16), 3)
    b.conv(x_in, 3, x, cp(16), w, bias, 3, 1, 1, relu=True)
    Cx, Hx, Wx = 16, H, W
    for layer in (m.layer1, m.layer2, m.layer3):
        for blk in layer:
            s = blk.conv1.stride[0]
            planes = blk.conv1.out_channels
            Ho, Wo = _out_hw(Hx, 3, s, 1), _out_hw(Wx, 3, s, 1)
            t = b.buffer(Ho, Wo, cp(planes))
            w, bias = padw(*fold_bn(blk.conv1.weight, None, blk.bn1), cp(planes), cp(Cx))
            b.conv(x, cp(Cx), t, cp(planes), w, bias, 3, s, 1, relu=True)  # conv1 takes the un-downsampled x (:33)
            if blk.downsample is not None:                                 # DownsampleB: avgpool + zero channels
                ks = blk.downsample.avg.kernel_size
                ks = ks if isinstance(ks, int) else ks[0]
                idn = b.buffer(_out_hw(Hx, ks, ks, 0), _out_hw(Wx, ks, ks, 0), cp(Cx))
                b.pool(_lib.POOL_AVG, x, cp(Cx), idn, ks, ks, 0)
            else:
                idn = x
            o = b.buffer(Ho, Wo, cp(planes))
            w, bias = padw(*fold_bn(blk.conv2.weight, None, blk.bn2), cp(planes), cp(planes))
            b.conv(t, cp(planes), o, cp(planes), w, bias, 3, 1, 1, relu=True, res=idn, res_C=cp(Cx))
            b.release(t)
            if idn != x:
                b.release(idn)
            b.release(x)
            x, Cx, Hx, Wx = o, planes, Ho, Wo
    ks = m.avgpool.kernel_size
    ks = ks if isinstance(ks, int) else ks[0]
    assert _out_hw(Hx, ks, ks, 0) == 1, "AvgPool2d(8) must reduce to 1x1 (models/resnet.py:103)"
    feat = b.buffer(1, 1, cp(Cx))
    b.pool(_lib.POOL_AVG, x, cp(Cx), feat, ks, ks, 0)
    fw = m.fc.weight
    if cp(Cx) != Cx:
        fw = torch.zeros(fw.shape[0], cp(Cx), dtype=fw.dtype, device=fw.device)
        fw[:, :Cx] = m.fc.weight
    b.fc(feat, cp(Cx), m.fc.out_features, fw, m.fc.bias)
    return Classifier(b, x_in, (3, H, W), m.fc.out_features, precision, max_batch, arch="resnet_cifar")


def _lower_mnist(m, hw, prec, precision, max_batch):
    H, W = hw
    b = _Builder(prec, max_batch)
    x_in = b.buffer(H, W, _in_cpad(1), pooled=False)
    cur, Cc, Hh, Ww = x_in, 1, H, W
    taps = {}
    for name in ("conv1", "conv2", "conv3", "conv4", "conv5"):
        seq = getattr(m, name)
        cv, bn = seq[0], seq[1]
        Ho, Wo = _out_hw(Hh, 3, cv.stride[0], cv.padding[0]), _out_hw(Ww, 3, cv.stride[0], cv.padding[0])
        o = b.buffer(Ho, Wo, cv.out_channels, pooled=False)
        w, bias = fold_bn(cv.weight, cv.bias, bn)
        b.conv(cur, Cc, o, cv.out_channels, w, bias, 3, cv.stride[0], cv.padding[0], relu=True)
        cur, Cc, Hh, Ww = o, cv.out_channels, Ho, Wo
        if name == "conv2":
            taps["x0"] = o
        if name == "conv4":
            taps["x1"] = o
    cv = m.conv6
    o = b.buffer(Hh, Ww, cv.out_channels, pooled=False)
    b.conv(cur, Cc, o, cv.out_channels, cv.weight.detach().float(), cv.bias.detach().float(), 3, 1, 1, relu=False)
    taps["x2"] = o
    feat = b.buffer(1, 1, cv.out_channels)
    assert Hh == Ww
    b.pool(_lib.POOL_AVG, o, cv.out_channels, feat, Hh, Hh, 0)           # x2.mean(3).mean(2)
    b.fc(feat, cv.out_channels, m.fc1.out_features, m.fc1.weight, m.fc1.bias)
    return Classifier(b, x_in, (1, H, W), m.fc1.out_features, precision, max_batch, taps=taps, arch="mnist")


def _dense_block(b: _Builder, layers, blk_buf, C0, H, W, Ctot):
    """BN-ReLU-conv1x1-BN-ReLU-conv3x3, concat == write into the next channel slice of blk_buf."""
    cur = C0
    for lyr in layers:
        n1, c1 = lyr.norm1, lyr.conv1
        has_bottleneck = hasattr(lyr, "conv2") and getattr(lyr, "conv2") is not None
        if has_bottleneck:
            n2, c2 = lyr.norm2, lyr.conv2
            mid = b.buffer(H, W, c1.out_channels)
            w, bias = fold_bn(c1.weight, None, n2)                           # conv1 -> norm2 -> relu2 folds forward
            b.conv(blk_buf, cur, mid, c1.out_channels, w, bias, 1, 1, 0, relu=True, pre=bn_affine(n1))
            b.conv(mid, c1.out_channels, blk_buf, c2.out_channels, c2.weight.detach().float(), None, 3, 1, 1,
                   relu=False, out_coff=cur)
            b.release(mid)
            cur += c2.out_channels
        else:
            b.conv(blk_buf, cur, blk_buf, c1.out_channels, c1.weight.detach().float(), None, 3, 1, 1, relu=False,
                   out_coff=cur, pre=bn_affine(n1))
            cur += c1.out_channels
    assert cur == Ctot
    return cur


def _lower_tv_densenet(m, hw, prec, precision, max_batch):
    H, W = hw
    f = m.features
    b = _Builder(prec, max_batch)
    c0 = f.conv0
    stem_tc = (precision == "bf16" and c0.kernel_size == (7, 7) and c0.stride == (2, 2) and c0.padding == (3, 3))
    x_in = b.buffer(H, W, 4, pad=3, pooled=False) if stem_tc else b.buffer(H, W, _in_cpad(3), pooled=False)
    Hc, Wc = _out_hw(H, 7, 2, 3), _out_hw(W, 7, 2, 3)
    t = b.buffer(Hc, Wc, c0.out_channels)
    w, bias = fold_bn(c0.weight, None, f.norm0)
    b.conv(x_in, 3, t, c0.out_channels, w, bias, 7, 2, 3, relu=True)
    Hx, Wx = _out_hw(Hc, 3, 2, 1), _out_hw(Wc, 3, 2, 1)
    blocks = [getattr(f, n) for n in ("denseblock1", "denseblock2", "denseblock3", "denseblock4")]
    trans = [getattr(f, n) for n in ("transition1", "transition2", "transition3")]
    Cin = c0.out_channels
    prev, prev_is_stem = t, True
    for bi, blk in enumerate(blocks):
        layers = list(blk.children())
        growth = layers[0].conv2.out_channels
        Ctot = Cin + growth * len(layers)
        buf = b.buffer(Hx, Wx, Ctot, pooled=False)
        if prev_is_stem:
            b.pool(_lib.POOL_MAX, prev, Cin, buf, 3, 2, 1)                       # pool0 -> channels [0,Cin)
            b.release(prev)
        else:
            b.pool(_lib.POOL_AVG, prev, Cin, buf, 2, 2, 0)                       # transition avgpool
            b.release(prev)
        _dense_block(b, layers, buf, Cin, Hx, Wx, Ctot)
        if bi < len(trans):
            tr = trans[bi]
            Co = tr.conv.out_channels
            tt = b.buffer(Hx, Wx, Co)
            b.conv(buf, Ctot, tt, Co, tr.conv.weight.detach().float(), None, 1, 1, 0, relu=False, pre=bn_affine(tr.norm))
            prev, prev_is_stem = tt, False
            Cin = Co
            Hx, Wx = Hx // 2, Wx // 2
        else:
            feat = b.buffer(1, 1, Ctot)
            assert Hx == Wx
            b.pool(_lib.POOL_AVG, buf, Ctot, feat, Hx, Hx, 0, pre=bn_affine(f.norm5))   # relu(norm5) -> avgpool
            b.fc(feat, Ctot, m.classifier.out_features, m.classifier.weight, m.classifier.bias)
    return Classifier(b, x_in, (3, H, W), m.classifier.out_features, precision, max_batch, arch="tv_densenet")


def _lower_densenet_cifar(m, hw, prec, precision, max_batch):
    """CIFAR DenseNet(-BC) of models/densenet.py:44-99 in the restated module layout
    (stem, blocks = [dense, transition, dense, transition, dense], norm5, classifier)."""
    H, W = hw
    b = _Builder(prec, max_batch)
    x_in = b.buffer(H, W, _in_cpad(3), pooled=False)
    seq = list(m.blocks.children())
    Cin = m.stem.out_channels
    Hx, Wx = H, W
    prev = None
    for i in range(0, len(seq), 2):
        layers = list(seq[i].children())
        growth = (layers[0].conv2 if hasattr(layers[0], "conv2") else layers[0].conv1).out_channels
        Ctot = Cin + growth * len(layers)
        buf = b.buffer(Hx, Wx, Ctot, pooled=False)
        if prev is None:
            b.conv(x_in, 3, buf, Cin, m.stem.weight.detach().float(), None, 3, 1, 1, relu=False)
        else:
            b.pool(_lib.POOL_AVG, prev, Cin, buf, 2, 2, 0)
            b.release(prev)
        _dense_block(b, layers, buf, Cin, Hx, Wx, Ctot)
        if i + 1 < len(seq):
            tr = list(seq[i + 1].children())   # BN, ReLU, Conv1x1, AvgPool
            Co = tr[2].out_channels
            tt = b.buffer(Hx, Wx, Co)
            b.conv(buf, Ctot, tt, Co, tr[2].weight.detach().float(), None, 1, 1, 0, relu=False, pre=bn_affine(tr[0]))
            prev, Cin = tt, Co
            Hx, Wx = Hx // 2, Wx // 2
        else:
            feat = b.buffer(1, 1, Ctot)
            assert Hx == 8 and Wx == 8, "avg_pool2d(8) expects an 8x8 map (models/densenet.py:96)"
            b.pool(_lib.POOL_AVG, buf, Ctot, feat, 8, 8, 0, pre=bn_affine(m.norm5))
            b.fc(feat, Ctot, m.classifier.out_features, m.classifier.weight, m.classifier.bias)
    return Classifier(b, x_in, (3, H, W), m.classifier.out_features, precision, max_batch, arch="densenet_cifar")


# ---- torchvision VGG / AlexNet: features (conv [BN] ReLU, max pool) / avgpool / classifier (Linear ReLU Dropout) ----------
def _is_plain_cnn(m) -> bool:
    return (isinstance(getattr(m, "features", None), nn.Sequential) and isinstance(getattr(m, "classifier", None), nn.Sequential)
            and not hasattr(m.features, "denseblock1"))


def _pair(v):
    return tuple(v) if isinstance(v, (tuple, list)) else (v, v)


def _plain_cnn_layers(m, hw, precision):
    """Checks the whole module and returns (feature ops, (C, H, W) of the final map, [(Linear, relu)]) without touching the
    library: feature ops are ("conv", Conv2d, BatchNorm2d | None, relu) and ("pool", k, stride, pad).  TypeError names a
    module this lowering does not take, ValueError an input size it cannot serve."""
    H, W = hw
    C = None
    ops = []
    mods = list(m.features.children())
    i = 0
    while i < len(mods):
        mod = mods[i]
        if isinstance(mod, nn.Conv2d):
            k, s, p, d = _pair(mod.kernel_size), _pair(mod.stride), _pair(mod.padding), _pair(mod.dilation)
            if (mod.groups != 1 or d != (1, 1) or k[0] != k[1] or s[0] != s[1] or isinstance(mod.padding, str) or p[0] != p[1]
                    or mod.padding_mode != "zeros"):
                raise TypeError(f"unsupported Conv2d in features[{i}]: {mod} (needs groups 1, dilation 1, square kernel, "
                                "stride and zero padding)")
            if C is not None and mod.in_channels != C:
                raise TypeError(f"features[{i}]: {mod} takes {mod.in_channels} channels, the map has {C}")
            bn = None
            if i + 1 < len(mods) and isinstance(mods[i + 1], nn.BatchNorm2d):
                bn = mods[i + 1]
                i += 1
            relu = i + 1 < len(mods) and isinstance(mods[i + 1], nn.ReLU)
            if relu:
                i += 1
            H, W = _out_hw(H, k[0], s[0], p[0]), _out_hw(W, k[0], s[0], p[0])
            if H < 1 or W < 1:
                raise ValueError(f"input {hw} is too small for features[{i}]")
            C = mod.out_channels
            ops.append(("conv", mod, bn, relu))
        elif isinstance(mod, nn.MaxPool2d):
            k, s, p, d = _pair(mod.kernel_size), _pair(mod.stride), _pair(mod.padding), _pair(mod.dilation)
            if k[0] != k[1] or s[0] != s[1] or p[0] != p[1] or d != (1, 1) or mod.ceil_mode or mod.return_indices:
                raise TypeError(f"unsupported MaxPool2d in features[{i}]: {mod} (needs a square window, dilation 1, "
                                "ceil_mode=False)")
            if C is None:
                raise TypeError("features must start with a Conv2d")
            H, W = _out_hw(H, k[0], s[0], p[0]), _out_hw(W, k[0], s[0], p[0])
            if H < 1 or W < 1:
                raise ValueError(f"input {hw} is too small for features[{i}]")
            ops.append(("pool", k[0], s[0], p[0]))
        else:
            raise TypeError(f"unsupported module in features[{i}]: {type(mod).__name__}")
        i += 1
    if C is None:
        raise TypeError("features holds no Conv2d")
    ap = getattr(m, "avgpool", None)
    if ap is not None and not isinstance(ap, nn.Identity):
        if not isinstance(ap, nn.AdaptiveAvgPool2d):
            raise TypeError(f"unsupported avgpool: {type(ap).__name__}")
        oh, ow = _pair(ap.output_size)
        if (oh is not None and oh != H) or (ow is not None and ow != W):
            # only the identity case is lowered (every 224^2 drop-in); a general adaptive pool is not
            raise ValueError(f"input {hw} gives a {H}x{W} feature map; avgpool wants {ap.output_size} and is lowered "
                             "only where it is an identity")
    lins = []
    for j, mod in enumerate(m.classifier.children()):
        if isinstance(mod, nn.Linear):
            lins.append([mod, False])
        elif isinstance(mod, nn.ReLU):
            if not lins or lins[-1][1]:
                raise TypeError(f"classifier[{j}]: a ReLU must follow a Linear")
            lins[-1][1] = True
        elif not isinstance(mod, nn.Dropout):     # Dropout: identity in eval
            raise TypeError(f"unsupported module in classifier[{j}]: {type(mod).__name__}")
    if len(lins) < 2 or lins[-1][1]:
        raise TypeError("classifier must hold at least two Linear layers and end in a Linear without ReLU")
    if H != W:
        raise ValueError(f"input {hw} gives a non-square {H}x{W} feature map")
    if lins[0][0].in_features != C * H * W:
        raise ValueError(f"input {hw} gives {C}x{H}x{W} features; classifier[0] takes {lins[0][0].in_features}")
    for a, b in zip(lins, lins[1:]):
        if b[0].in_features != a[0].out_features:
            raise TypeError(f"{b[0]} does not take the {a[0].out_features} outputs of {a[0]}")
    if precision == "split":
        body = [op[1] for op in ops[1:] if op[0] == "conv"]
        widths = [(c.in_channels, c.out_channels) for c in body] + [(C, lins[0][0].out_features)]
        widths += [(l.in_features, l.out_features) for l, _ in lins[1:-1]]
        if any(a % 64 or b % 64 for a, b in widths):
            raise TypeError("precision 'split' needs Cin % 64 == 0 and Cout % 64 == 0 for every conv after the first and "
                            "every Linear but the last; use 'x3' for this network")
    return ops, (C, H, W), [(l, r) for l, r in lins]


# Longest reduction an fp32-grade lowering puts on split-bf16 tensor-core products (net.cu NIB_X3_MAX_K): the tensor cores'
# fp32 accumulation drifts with K, so split networks run VGG's fc6 (K = 25088) on fp32 buffers on the CUDA cores.
_FP32_GRADE_TC_MAX_K = 16384


def _lower_tv_plain(m, hw, prec, precision, max_batch):
    """Convs (BN folded) and max pools as they come; the first Linear as a valid KxK conv over the KxK final map (its
    weight viewed [out][C][K][K]: nib_net_add_conv's KRSC repack then matches the NHWC order of the map, so no flatten op
    is needed), the middle Linears as 1x1 convs on 1x1 maps, the last Linear as the fc op.  bf16: a 3x3/1 first conv
    reads 8-channel pixels in a 1-pixel zero halo (the tcgen05 raw-row mode, conv_tc.cu tc_conv_is_raw3x3).  split: the
    first conv, the pools and a Linear longer than _FP32_GRADE_TC_MAX_K run on fp32 buffers, everything else on split-bf16
    tensors, with converts between."""
    ops, (C, Hf, Wf), lins = _plain_cnn_layers(m, hw, precision)   # everything is checked before the library is touched
    H, W = hw
    b = _Builder(prec, max_batch)
    split = precision == "split"
    c1 = ops[0][1]
    cin = c1.in_channels
    raw3 = (precision == "bf16" and _pair(c1.kernel_size) == (3, 3) and _pair(c1.stride) == (1, 1)
            and _pair(c1.padding) == (1, 1) and cin <= 8)
    x_in = b.buffer(H, W, 8, pad=1, pooled=False) if raw3 else b.buffer(H, W, _in_cpad(cin), pooled=False, f32=split)
    x, Cx, Hx, Wx, x_split = x_in, cin, H, W, False

    def to_split(want):
        nonlocal x, x_split
        if split and want != x_split:
            y = b.buffer(Hx, Wx, Cx, f32=not want)
            b.convert(x, y)
            b.release(x)
            x, x_split = y, want

    for op in ops:
        if op[0] == "conv":
            _, cv, bn, relu = op
            if x != x_in:
                to_split(True)
            k, s, p = cv.kernel_size[0], _pair(cv.stride)[0], _pair(cv.padding)[0]
            Ho, Wo = _out_hw(Hx, k, s, p), _out_hw(Wx, k, s, p)
            o = b.buffer(Ho, Wo, cv.out_channels, f32=split and not x_split)
            w, bias = fold_bn(cv.weight, cv.bias, bn)
            b.conv(x, Cx, o, cv.out_channels, w, bias, k, s, p, relu=relu)
            if x != x_in:
                b.release(x)
            x, Cx, Hx, Wx = o, cv.out_channels, Ho, Wo
        else:
            _, k, s, p = op
            to_split(False)
            Ho, Wo = _out_hw(Hx, k, s, p), _out_hw(Wx, k, s, p)
            o = b.buffer(Ho, Wo, Cx, f32=split)
            b.pool(_lib.POOL_MAX, x, Cx, o, k, s, p)
            b.release(x)
            x, Hx, Wx = o, Ho, Wo
    for j, (lin, relu) in enumerate(lins[:-1]):
        K = Hx if j == 0 else 1
        tc = Cx * K * K <= _FP32_GRADE_TC_MAX_K
        to_split(tc)
        wc = lin.weight.detach().reshape(lin.out_features, Cx, K, K)
        o = b.buffer(1, 1, lin.out_features, f32=split and not tc)
        b.conv(x, Cx, o, lin.out_features, wc, lin.bias, K, 1, 0, relu=relu)
        b.release(x)
        x, Cx, Hx, Wx = o, lin.out_features, 1, 1
    to_split(False)
    last = lins[-1][0]
    b.fc(x, Cx, last.out_features, last.weight, last.bias)
    return Classifier(b, x_in, (cin, H, W), last.out_features, precision, max_batch, arch="tv_plain")
