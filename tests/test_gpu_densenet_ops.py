"""DenseNet's engine operators one at a time against float64 references of the operation.

DenseNet lowers onto features no other network uses: BN-ReLU pre-activation on the input of a conv (in-kernel transform
of the CTA-pair kernel's A tiles, the bnrelu pack pass, the CUDA-core gathers), convs and pools writing a channel slice
of a wider concat buffer, and pre-activated pools (norm5).  Each case here builds a one- or two-op network with
classifier._Builder and compares every output element with the fp64 result of the operation

    y = conv(relu(x * scale + shift), w) + bias   (then ReLU when the conv has it),

with x and w rounded where the precision stores them (bf16 nets: bf16 activations and conv weights; fp32 / x3: nothing),
under a per-element bound built from the operand precisions (see _consts):

    |got - ref| <= c_out * |ref| + c_op * (|a| (*) |w|),   a = relu(x * scale + shift),  (*) = the same conv in fp64.

Every case also asserts the path it tests: tcgen05 launches, the extra pack launch, tensor core on or off."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import classifier as ocls

U32 = 2.0 ** -24    # unit roundoff of fp32 (24 significant bits, round to nearest)
U16 = 2.0 ** -8     # unit roundoff of bf16 (8 significant bits, round to nearest): half its 2^-7 ulp at 1
POISONS = ("nan", "inf", "big")


def _gamma(n, u):
    """Bound on the relative error of a sum of n terms in precision u, any order: n u / (1 - n u)."""
    return n * u / (1.0 - n * u)


def _consts(path, K, act_rounded=True):
    """(c_out, c_op) for a conv with reduction length K on one of the engine's paths.

    bf16_tc  : tcgen05, bf16 x bf16 products (exact in fp32), fp32 accumulation inside the tensor core, which may truncate
               rather than round: 2 U32 per addition.  The activated operand fmaf(x, s, h) is rounded once in fp32 and
               once to bf16 before the MMA (U32 + U16, relative to |a|).  Output: bias add in fp32 (U32), bf16 store (U16).
    bf16_simt: CUDA cores, activated operand kept in fp32 (U32), fmaf accumulation (one rounding per term), bf16 store.
    fp32     : as bf16_simt with an fp32 store.
    x3       : split-bf16 tensor-core products a_hi w_hi + a_lo w_hi + a_hi w_lo: each of a, w is hi + lo up to U16^2 of
               its size, and the dropped a_lo w_lo is at most U16^2 |a w|: 3 U16^2 per product, then the tensor core's
               fp32 accumulation (2 U32 per addition) and the fp32 transform (U32); fp32 store.
    act_rounded=False: the conv's input needs no transform (a bf16 tensor read as is), so the operand terms drop out.
    The store rounds the accumulated error too: c_op is scaled by (1 + c_out)."""
    act = 0.0
    if path == "bf16_tc":
        act = U32 + U16 if act_rounded else 0.0
        c_op, c_out = act + _gamma(K, 2 * U32), U16 + U32
    elif path in ("bf16_simt", "fp32"):
        act = U32 if act_rounded else 0.0
        c_op, c_out = act + _gamma(K, U32), (U16 + U32) if path == "bf16_simt" else U32
    elif path == "x3":
        act = U32 if act_rounded else 0.0
        c_op, c_out = act + 3 * U16 * U16 + _gamma(K, 2 * U32), U32
    else:
        raise ValueError(path)
    return c_out, c_op * (1 + c_out)


def _excess(got, ref, mag, c_out, c_op):
    """Elements outside the bound (or not finite) and the worst ratio |got - ref| / bound."""
    got, ref, mag = got.double(), ref.double(), mag.double()
    bound = c_out * ref.abs() + c_op * mag
    err = (got - ref).abs()
    bad = (err > bound) | ~torch.isfinite(got)
    ratio = (err / bound.clamp_min(1e-300)).max().item()
    return int(bad.sum().item()), ratio


def _assert_within(got, ref, mag, c_out, c_op, what):
    n, ratio = _excess(got, ref, mag, c_out, c_op)
    assert n == 0, f"{what}: {n} of {got.numel()} elements outside the bound (worst |err| / bound = {ratio:.3g})"


def _bf(t):
    return t.to(torch.bfloat16).to(torch.float32)


def _preact_ref(x, s, h, w, bias, stride, pad, relu, round_act=False):
    """fp64 conv(relu(x*s+h)) + bias (+ReLU) and the magnitude conv |a| (*) |w|.  round_act: the activated operand
    rounded to bf16 (the tcgen05 path's operand), for the checker's self-test."""
    a = (x.double() * s.double().view(1, -1, 1, 1) + h.double().view(1, -1, 1, 1)).clamp_min(0)
    if round_act:
        a = a.to(torch.bfloat16).double()
    wd = w.double()
    ref = F.conv2d(a, wd, bias.double() if bias is not None else None, stride=stride, padding=pad)
    if relu:
        ref = ref.clamp_min(0)
    mag = F.conv2d(a.abs(), wd.abs(), None, stride=stride, padding=pad)
    return ref, mag


def _bn_params(x, g):
    """Eval-BN scale / shift that reach the edges: scales of both signs, shifts mostly positive (a conv that lets the
    shift into its zero padding shows relu(shift) there), and every 7th channel dead (x*s+h < 0 at every pixel)."""
    Cin = x.shape[1]
    sign = torch.where(torch.rand(Cin, generator=g) < 0.3, -1.0, 1.0)
    s = sign * (0.5 + torch.rand(Cin, generator=g))
    h = 0.1 + 0.9 * torch.rand(Cin, generator=g)
    h = torch.where(torch.rand(Cin, generator=g) < 0.15, -h, h)
    dead = torch.arange(Cin) % 7 == 3
    amax = x.abs().amax(dim=(0, 2, 3))
    s[dead] = 0.1 * sign[dead]
    h[dead] = -(0.1 * amax[dead] + 0.25)
    return s.float(), h.float()


def _poison_fill(kind, shape):
    if kind == "zero":
        return torch.zeros(shape)
    if kind == "nan":
        return torch.full(shape, float("nan"))
    alt = torch.where(torch.arange(int(np.prod(shape))).reshape(shape) % 2 == 0, 1.0, -1.0)
    return alt * (float("inf") if kind == "inf" else 3e38)


# ---- checker self-test (CPU) ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [1, 3])
def test_bound_rejects_indexing_bugs_and_accepts_operand_rounding(k):
    """The bf16 tensor-path bound, Cin = 96 in a 128-channel concat buffer: the references that real indexing bugs
    produce must fail it; the one that differs only by rounding the activated operand to bf16 must pass."""
    g = torch.Generator().manual_seed(40 + k)
    N, Cin, Cbuf, Cout, H = 2, 96, 128, 32, 10
    pad = k // 2
    buf = _bf(torch.randn(N, Cbuf, H, H, generator=g))
    x, stale = buf[:, :Cin], buf[:, Cin:]
    s, h = _bn_params(x, g)
    w = _bf(torch.randn(Cout, Cin, k, k, generator=g) / np.sqrt(Cin * k * k))
    bias = torch.randn(Cout, generator=g) * 0.1
    c_out, c_op = _consts("bf16_tc", Cin * k * k)
    ref, mag = _preact_ref(x, s, h, w, bias, 1, pad, True)

    rounded, _ = _preact_ref(x, s, h, w, bias, 1, pad, True, round_act=True)
    assert _excess(rounded, ref, mag, c_out, c_op)[0] == 0
    assert _excess(_bf(rounded.float()), ref, mag, c_out, c_op)[0] == 0      # and the bf16 store on top

    bugs = {
        "neighbour_scale_shift": _preact_ref(x, s.roll(1), h.roll(1), w, bias, 1, pad, True)[0],
        "no_relu": F.conv2d(x.double() * s.double().view(1, -1, 1, 1) + h.double().view(1, -1, 1, 1), w.double(),
                            bias.double(), padding=pad).clamp_min(0),
        # the last 16-byte chunk of the slice read 8 channels too far: stale channels [Cin, Cin + 8) leak in
        "stale_leak": _preact_ref(torch.cat([x[:, :Cin - 8], stale[:, :8]], 1), s, h, w, bias, 1, pad, True)[0],
    }
    if pad:   # the shift applied at padded taps: padding before the activation instead of after it
        bugs["shift_at_padded_taps"] = _preact_ref(F.pad(x, (pad,) * 4), s, h, w, bias, 1, 0, True)[0]
    for name, bad in bugs.items():
        assert _excess(bad, ref, mag, c_out, c_op)[0] > 0, f"the bound accepts the '{name}' bug"


# ---- one pre-activated conv reading a channel slice of a concat buffer --------------------------------------------------
def _native_forward(net, xn):
    """Public forward with the buffer's own layout (NHWC, net dtype): every channel of the input buffer is written, so the
    channels outside the conv's slice hold whatever the caller put there."""
    from network_interpretation_imagenet_b200 import _lib
    N = xn.shape[0]
    out = torch.empty(N, net.num_classes, dtype=torch.float32, device="cuda")
    _lib.check(net.lib.nib_net_forward(net.h, xn.data_ptr(), _lib.IN_NATIVE, N, out.data_ptr(), _lib.stream_handle()),
               "nib_net_forward")
    torch.cuda.synchronize()
    return out


class _PreactConv:
    """conv(relu(x*s+h)) of channels [in_coff, in_coff + Cin) of a C-channel input buffer into its own output buffer,
    then a global average pool and a 4-way fc (a network must end in an fc)."""

    def __init__(self, precision, C, in_coff, Cin, Cout, k, stride, H, N=5, relu=True, seed=0):
        from network_interpretation_imagenet_b200 import _lib
        from network_interpretation_imagenet_b200.classifier import _Builder, Classifier, _out_hw
        g = torch.Generator().manual_seed(seed)
        self.precision, self.N, self.C, self.in_coff, self.Cin, self.H = precision, N, C, in_coff, Cin, H
        self.stride, self.pad, self.relu, self.K = stride, k // 2, relu, Cin * k * k
        self.w = torch.randn(Cout, Cin, k, k, generator=g) / np.sqrt(Cin * k * k)
        self.bias = torch.randn(Cout, generator=g) * 0.1
        self.x = torch.randn(N, Cin, H, H, generator=g)
        if precision == "bf16":
            self.x, self.wq = _bf(self.x), _bf(self.w)
        else:
            self.wq = self.w
        self.s, self.h = _bn_params(self.x, g)
        b = _Builder({"fp32": _lib.PREC_FP32, "bf16": _lib.PREC_BF16, "x3": _lib.PREC_X3}[precision], N)
        self.x_in = b.buffer(H, H, C, pooled=False)
        Ho = _out_hw(H, k, stride, self.pad)
        out = b.buffer(Ho, Ho, Cout, pooled=False)
        b.conv(self.x_in, Cin, out, Cout, self.w, self.bias, k, stride, self.pad, relu=relu, in_coff=in_coff,
               pre=(self.s, self.h))
        feat = b.buffer(1, 1, Cout)
        b.pool(_lib.POOL_AVG, out, Cout, feat, Ho, Ho, 0)
        b.fc(feat, Cout, 4, torch.zeros(4, Cout), None)
        self.net = Classifier(b, self.x_in, (C, H, H), 4, precision, N, taps={"out": out})

    def run(self, fill="zero", tensor_core=True):
        """One forward with `fill` in every channel outside the slice: (output NCHW fp64, total launches, tcgen05 launches)."""
        self.net.set_tensor_core(tensor_core)
        full = _poison_fill(fill, (self.N, self.C, self.H, self.H))
        full[:, self.in_coff:self.in_coff + self.Cin] = self.x
        dt = torch.bfloat16 if self.precision == "bf16" else torch.float32
        xn = full.permute(0, 2, 3, 1).contiguous().to(dt).cuda()
        t0, c0 = self.net.launch_counts()
        _native_forward(self.net, xn)
        t1, c1 = self.net.launch_counts()
        return self.net.read_tap("out", self.N).cpu().double(), t1 - t0, c1 - c0

    def reference(self):
        return _preact_ref(self.x, self.s, self.h, self.wq, self.bias, self.stride, self.pad, self.relu)

    def check(self, got, path, what):
        ref, mag = self.reference()
        c_out, c_op = _consts(path, self.K)
        _assert_within(got, ref, mag, c_out, c_op, what)

    def check_poison_invariant(self, base, tensor_core=True):
        """NaN, +-Inf and +-3e38 outside the slice change nothing: the output is finite and bitwise the zero-fill one."""
        for kind in POISONS:
            got, _, _ = self.run(kind, tensor_core)
            assert torch.isfinite(got).all(), f"non-finite output with {kind} outside the channel slice"
            assert torch.equal(got, base), f"{kind} outside the channel slice changed the output"


def _cid(c):
    return "_".join(f"{n}{v}" for n, v in zip(("C", "off", "cin", "cout", "h"), c))


# C (buffer channels), in_coff, Cin, Cout, H.  Cin % 64 in {0, 32, 8}; the transform reads [in_coff, in_coff + roundup64(Cin))
XFORM_CASES = [
    (64, 0, 64, 128, 56),
    (128, 0, 96, 128, 14),       # stale channels [96, 128)
    (72, 0, 72, 256, 14),        # in_coff + roundup64(Cin) = 128 > C: the TMA box runs past the pixel's channels
    (96, 0, 72, 128, 7),         # stale [72, 96), then past the row end
    (256, 0, 224, 256, 14),
    (1024, 0, 1024, 128, 7),     # 16 K blocks
    (136, 32, 96, 128, 14),      # in_coff != 0, and in_coff + 128 > C
    # Cout = 64: one N tile; <= 9 K blocks used to select the resident-weights instantiation, which has no transform
    (128, 0, 96, 64, 56),
    (640, 0, 576, 64, 14),       # 9 K blocks
    (704, 0, 640, 64, 14),       # 10 K blocks: streamed weights either way
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", XFORM_CASES, ids=_cid)
def test_preact_1x1_bf16_transform(nib, case):
    """BN-ReLU inside conv_tc3_kernel (transform warps on the A tiles): one tcgen05 launch, no pack launch."""
    C, off, Cin, Cout, H = case
    op = _PreactConv("bf16", C, off, Cin, Cout, 1, 1, H, seed=sum(case))
    got, total, tc = op.run()
    assert (total, tc) == (3, 1), f"launches (total, tcgen05) = {(total, tc)}: expected conv + pool + fc, no pack pass"
    op.check(got, "bf16_tc", "transform")
    op.check_poison_invariant(got)


# C, in_coff, Cin, Cout, k, H.  1x1 with Cout % 64 != 0, and every pre-activated 3x3 (growth convs of the non-bottleneck
# dense layer): 64 / 128 packed channels and 32 outputs at 32x32 and 14x14 land on the resident-patch mode
PACK_CASES = [
    (128, 0, 96, 32, 1, 14),
    (96, 0, 72, 96, 1, 14),
    (64, 0, 64, 32, 3, 32),
    (128, 0, 96, 32, 3, 32),
    (128, 0, 128, 32, 3, 32),
    (64, 0, 64, 32, 3, 14),
    (128, 0, 96, 32, 3, 14),
    (160, 32, 128, 32, 3, 14),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", PACK_CASES, ids=lambda c: "C%d_off%d_cin%d_cout%d_k%d_h%d" % c)
def test_preact_bf16_pack_pass(nib, case):
    """bnrelu_pack_kernel into the scratch tensor, then the tcgen05 conv on it: the pack launch is there."""
    C, off, Cin, Cout, k, H = case
    op = _PreactConv("bf16", C, off, Cin, Cout, k, 1, H, relu=False, seed=sum(case))
    got, total, tc = op.run()
    assert (total, tc) == (4, 1), f"launches (total, tcgen05) = {(total, tc)}: expected pack + conv + pool + fc"
    op.check(got, "bf16_tc", "pack pass")
    op.check_poison_invariant(got)


# precision, C, in_coff, Cin, Cout, k, stride, H.  fp32: Cin 36 takes the scalar gather, 96 the 8-channel vector gather
SIMT_CASES = [
    ("bf16", 128, 0, 96, 128, 1, 1, 14),
    ("bf16", 96, 0, 64, 32, 3, 1, 14),
    ("bf16", 128, 0, 96, 64, 3, 2, 15),
    ("fp32", 40, 0, 36, 32, 3, 1, 14),
    ("fp32", 48, 4, 36, 64, 3, 2, 15),
    ("fp32", 128, 0, 96, 32, 3, 1, 14),
    ("fp32", 128, 0, 96, 64, 3, 2, 15),
    ("fp32", 104, 8, 96, 128, 1, 1, 7),
    ("x3", 128, 0, 96, 32, 3, 1, 14),
    ("x3", 128, 0, 96, 64, 3, 2, 15),
    ("x3", 104, 8, 96, 128, 1, 1, 7),
    ("x3", 40, 0, 36, 32, 3, 1, 14),     # Cin % 16 != 0: the fp32 CUDA-core kernel
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", SIMT_CASES, ids=lambda c: "%s_C%d_off%d_cin%d_cout%d_k%d_s%d_h%d" % c)
def test_preact_conv_cuda_cores(nib, case):
    """Pre-activation in the CUDA-core gathers (conv_simt.cu) and the split-bf16 conv (conv_x3.cu), 3x3 pad 1 at stride
    1 and 2 with positive shifts: padded taps must stay zero, not relu(shift)."""
    prec, C, off, Cin, Cout, k, stride, H = case
    op = _PreactConv(prec, C, off, Cin, Cout, k, stride, H, seed=sum(case[1:]))
    got, total, tc = op.run(tensor_core=False)
    assert (total, tc) == (3, 0), f"launches (total, tcgen05) = {(total, tc)}"
    op.check(got, {"bf16": "bf16_simt", "fp32": "fp32", "x3": "x3" if Cin % 16 == 0 else "fp32"}[prec], prec)
    op.check_poison_invariant(got, tensor_core=False)
    if prec == "x3":   # the same layer in an fp32 net: the fp32 kernel gives the same bits only when x3 fell back to it
        got32, _, _ = _PreactConv("fp32", C, off, Cin, Cout, k, stride, H, seed=sum(case[1:])).run(tensor_core=False)
        if Cin % 16 == 0:
            assert not torch.equal(got, got32), "the x3 net ran the fp32 CUDA-core kernel"
        else:
            assert torch.equal(got, got32), "Cin % 16 != 0 must fall back to the fp32 CUDA-core kernel"


# ---- transform vs pack pass ---------------------------------------------------------------------------------------------
XFORM_VS_PACK_CASES = [c for c in XFORM_CASES if c[3] in (128, 256)]


def preact_outputs_for_ab():
    """{case id: (output, total launches, tcgen05 launches)} of the Cout 128 / 256 transform cases in this process."""
    res = {}
    for case in XFORM_VS_PACK_CASES:
        C, off, Cin, Cout, H = case
        got, total, tc = _PreactConv("bf16", C, off, Cin, Cout, 1, 1, H, seed=sum(case)).run()
        res[_cid(case)] = (got, total, tc)
    return res


@pytest.mark.gpu
def test_preact_transform_matches_pack_pass_bitwise(nib, tmp_path):
    """The transform's arithmetic is the pack kernel's (fmaf, fmaxf, round to nearest) and the MMA sequence is the same,
    so the two paths give the same bits.  NIB_TC_NO_XFORM is read once per process: the pack side runs in a child."""
    out = tmp_path / "pack.pt"
    env = dict(os.environ, NIB_TC_NO_XFORM="1")
    worker = os.path.join(os.path.dirname(os.path.abspath(__file__)), "densenet_ops_worker.py")
    r = subprocess.run([sys.executable, worker, str(out)], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    pack = torch.load(out)
    mine = preact_outputs_for_ab()
    for key, (got, total, tc) in mine.items():
        pgot, ptotal, ptc = pack[key]
        assert (total, tc) == (3, 1) and (ptotal, ptc) == (4, 1), (key, (total, tc), (ptotal, ptc))
        assert torch.equal(got, pgot), f"{key}: transform and pack pass differ (max |diff| {(got - pgot).abs().max().item():.3g})"


# ---- writes into a channel slice leave the rest of the buffer alone ------------------------------------------------------
class _DevArray:
    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (ptr, False), "version": 2,
                                         "strides": None}


def _buffer_view(net, buf, N, bf16):
    """Zero-copy [N, H, W, C] view of an engine buffer (no halo)."""
    ptr, H, W, Cc, pad = C.c_void_p(), C.c_int(), C.c_int(), C.c_int(), C.c_int()
    from network_interpretation_imagenet_b200 import _lib
    _lib.check(net.lib.nib_net_buffer_info(net.h, buf, C.byref(ptr), C.byref(H), C.byref(W), C.byref(Cc), C.byref(pad),
                                           None), "nib_net_buffer_info")
    assert pad.value == 0
    t = torch.as_tensor(_DevArray(ptr.value, (N, H.value, W.value, Cc.value), "<i2" if bf16 else "<f4"), device="cuda")
    return t.view(torch.bfloat16) if bf16 else t


def _bits(t):
    return t.contiguous().view(torch.int16 if t.dtype == torch.bfloat16 else torch.int32)


@pytest.mark.gpu
@pytest.mark.parametrize("prec,tensor_core,H", [("bf16", True, 14), ("bf16", True, 28), ("bf16", True, 7),
                                                ("bf16", False, 14), ("fp32", False, 14)])
def test_dense_layer_writes_only_its_slice(nib, prec, tensor_core, H):
    """The DenseNet pair on one concat buffer: pre-activated 1x1 of [0, cur) into mid, 3x3 of mid into [cur, cur + 32).
    Every other channel of the buffer is bitwise what forward put there; mid and the slice match fp64."""
    from network_interpretation_imagenet_b200 import _lib
    from network_interpretation_imagenet_b200.classifier import _Builder, Classifier
    N, Ctot, cur, mid_c, growth = 5, 256, 160, 128, 32
    g = torch.Generator().manual_seed(H + tensor_core)
    bf16 = prec == "bf16"
    q = _bf if bf16 else (lambda t: t)
    xfull = q(torch.randn(N, Ctot, H, H, generator=g))
    x = xfull[:, :cur]
    s, h = _bn_params(x, g)
    w1 = torch.randn(mid_c, cur, 1, 1, generator=g) / np.sqrt(cur)
    b1 = torch.randn(mid_c, generator=g) * 0.1
    w2 = torch.randn(growth, mid_c, 3, 3, generator=g) / np.sqrt(9 * mid_c)
    b = _Builder(_lib.PREC_BF16 if bf16 else _lib.PREC_FP32, N)
    buf = b.buffer(H, H, Ctot, pooled=False)
    mid = b.buffer(H, H, mid_c, pooled=False)
    b.conv(buf, cur, mid, mid_c, w1, b1, 1, 1, 0, relu=True, pre=(s, h))
    b.conv(mid, mid_c, buf, growth, w2, None, 3, 1, 1, relu=False, out_coff=cur)
    feat = b.buffer(1, 1, Ctot)
    b.pool(_lib.POOL_AVG, buf, Ctot, feat, H, H, 0)
    b.fc(feat, Ctot, 4, torch.zeros(4, Ctot), None)
    net = Classifier(b, buf, (Ctot, H, H), 4, prec, N, taps={"buf": buf, "mid": mid})
    net.set_tensor_core(tensor_core)
    xn = xfull.permute(0, 2, 3, 1).contiguous().to(torch.bfloat16 if bf16 else torch.float32).cuda()
    _native_forward(net, xn)
    total, tc = net.launch_counts()
    assert (total, tc) == ((4, 2) if tensor_core else (4, 0)), (total, tc)
    after = _buffer_view(net, buf, N, bf16).clone()
    keep = torch.ones(Ctot, dtype=torch.bool)
    keep[cur:cur + growth] = False
    assert torch.equal(_bits(after[..., keep]), _bits(xn[..., keep])), "a channel outside [cur, cur + 32) changed"
    path = ("bf16_tc" if tensor_core else "bf16_simt") if bf16 else "fp32"
    ref1, mag1 = _preact_ref(x, s, h, q(w1), b1, 1, 0, True)
    got_mid = net.read_tap("mid", N).cpu().double()
    _assert_within(got_mid, ref1, mag1, *_consts(path, cur), "mid")
    ref2 = F.conv2d(got_mid, q(w2).double(), None, padding=1)           # on the stored mid: no operand rounding left
    mag2 = F.conv2d(got_mid.abs(), q(w2).double().abs(), None, padding=1)
    got2 = after[..., cur:cur + growth].permute(0, 3, 1, 2).double().cpu()
    _assert_within(got2, ref2, mag2, *_consts(path, 9 * mid_c, act_rounded=False), "growth slice")


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["bf16", "fp32"])
@pytest.mark.parametrize("kind", ["pool0_max3s2", "transition_avg2"])
def test_pool_writes_only_its_slice(nib, prec, kind):
    """pool0 (3x3/2 max, pad 1) into channels [0, 64) and the transition's 2x2 average into [0, Co) of a wider dense
    block buffer prefilled with a pattern: the slice matches torch, every other channel keeps its bits."""
    from network_interpretation_imagenet_b200 import _lib
    from network_interpretation_imagenet_b200.classifier import _Builder, Classifier, _out_hw
    N = 5
    Cs, Ctot, H, k, st, pd = (64, 128, 28, 3, 2, 1) if kind.startswith("pool0") else (128, 256, 14, 2, 2, 0)
    bf16 = prec == "bf16"
    q = _bf if bf16 else (lambda t: t)
    g = torch.Generator().manual_seed(k + Ctot)
    x = q(torch.randn(N, Cs, H, H, generator=g))
    Ho = _out_hw(H, k, st, pd)
    b = _Builder(_lib.PREC_BF16 if bf16 else _lib.PREC_FP32, N)
    src = b.buffer(H, H, Cs, pooled=False)
    dst = b.buffer(Ho, Ho, Ctot, pooled=False)
    b.pool(_lib.POOL_MAX if k == 3 else _lib.POOL_AVG, src, Cs, dst, k, st, pd)
    feat = b.buffer(1, 1, Ctot)
    b.pool(_lib.POOL_AVG, dst, Ctot, feat, Ho, Ho, 0)
    b.fc(feat, Ctot, 4, torch.zeros(4, Ctot), None)
    net = Classifier(b, src, (Cs, H, H), 4, prec, N, taps={"dst": dst})
    view = _buffer_view(net, dst, N, bf16)
    pattern = q(torch.randn(N, Ho, Ho, Ctot, generator=g)).to(view.dtype).cuda()
    view.copy_(pattern)
    net.forward(x.cuda())
    torch.cuda.synchronize()
    after = view.clone()
    assert torch.equal(_bits(after[..., Cs:]), _bits(pattern[..., Cs:])), "a channel past the pool's slice changed"
    got = after[..., :Cs].permute(0, 3, 1, 2).double().cpu()
    if k == 3:   # a maximum of stored values is exact
        assert torch.equal(got, F.max_pool2d(x.double(), 3, 2, 1))
    else:
        ref = F.avg_pool2d(x.double(), 2, 2)
        c_out = (U16 + U32) if bf16 else U32
        _assert_within(got, ref, F.avg_pool2d(x.double().abs(), 2, 2), c_out, (_gamma(4, U32) + U32) * (1 + c_out),
                       "transition pool")


# ---- pre-activated pools (norm5 -> ReLU -> global average; BN-ReLU before a padded max pool) -------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["bf16", "fp32"])
@pytest.mark.parametrize("kind,H,Cc", [("gap", 7, 64), ("gap", 8, 36), ("gap", 7, 100), ("max3s2", 14, 64), ("max3s2", 15, 36)])
def test_preact_pool(nib, prec, kind, H, Cc):
    """The scalar pool_kernel with pre_scale: relu(x*s+h) per tap, only at in-bounds taps.  Every 5th channel has
    x < 0, s > 0 and shift 1, so each activation is below relu(shift) and a padded tap that contributed it would win."""
    from network_interpretation_imagenet_b200 import _lib
    from network_interpretation_imagenet_b200.classifier import _Builder, Classifier, _out_hw
    N = 5
    bf16 = prec == "bf16"
    q = _bf if bf16 else (lambda t: t)
    g = torch.Generator().manual_seed(H * Cc)
    x = torch.randn(N, Cc, H, H, generator=g)
    probe = torch.arange(Cc) % 5 == 1
    x[:, probe] = -x[:, probe].abs() - 0.5
    x = q(x)
    s, h = _bn_params(x, g)
    s[probe], h[probe] = 0.5 + torch.rand(int(probe.sum()), generator=g), 1.0
    b = _Builder(_lib.PREC_BF16 if bf16 else _lib.PREC_FP32, N)
    src = b.buffer(H, H, Cc, pooled=False)
    if kind == "gap":
        out = b.buffer(1, 1, Cc)
        b.pool(_lib.POOL_AVG, src, Cc, out, H, H, 0, pre=(s, h))
        b.fc(out, Cc, 4, torch.zeros(4, Cc), None)
    else:
        Ho = _out_hw(H, 3, 2, 1)
        out = b.buffer(Ho, Ho, Cc, pooled=False)
        b.pool(_lib.POOL_MAX, src, Cc, out, 3, 2, 1, pre=(s, h))
        feat = b.buffer(1, 1, Cc)
        b.pool(_lib.POOL_AVG, out, Cc, feat, Ho, Ho, 0)
        b.fc(feat, Cc, 4, torch.zeros(4, Cc), None)
    net = Classifier(b, src, (Cc, H, H), 4, prec, N, taps={"out": out})
    net.forward(x.cuda())
    got = net.read_tap("out", N).cpu().double()
    a = (x.double() * s.double().view(1, -1, 1, 1) + h.double().view(1, -1, 1, 1)).clamp_min(0)
    c_out = (U16 + U32) if bf16 else U32
    if kind == "gap":   # fp32 sum of H*H activations (each rounded once in fp32), one division
        ref = a.mean(dim=(2, 3), keepdim=True)
        c_op = _gamma(H * H, U32) + 2 * U32
    else:               # a maximum of activations rounded once in fp32; torch pads the max pool with -inf
        ref = F.max_pool2d(a, 3, 2, 1)
        c_op = U32
    _assert_within(got, ref, ref, c_out, c_op * (1 + c_out), f"{kind} pool")


# ---- whole networks the suite did not have -----------------------------------------------------------------------------
def _check_net(nib, model, x, precision, tol):
    """test_gpu_classifier._check_net: row-wise |got - want| <= tol * max |want| against the torch fp32 forward."""
    want = ocls.forward_logits(model, x).numpy()
    net = nib.Classifier.from_torch(model, tuple(x.shape[2:]), precision=precision, max_batch=x.shape[0])
    got = net.forward(torch.as_tensor(x).cuda()).cpu().numpy()
    err = float((np.abs(got - want) / np.abs(want).max(axis=1, keepdims=True)).max())
    assert err <= tol, f"{precision}: rel err {err:.3e} > {tol}"
    srt = np.sort(want, 1)
    decided = (srt[:, -1] - srt[:, -2]) > 2 * tol * np.abs(want).max(axis=1)
    assert np.array_equal(got.argmax(1)[decided], want.argmax(1)[decided]), "top-1 differs outside the tie band"
    return net


def _launches_per_forward(net, N):
    """(non-tcgen05 launches, tcgen05 launches) one forward makes if no conv runs a pack pass, from the op list: input
    staging, then one launch per op, tcgen05 for kind 1, nothing for a conv computed in the previous op's fused launch."""
    kinds = [k for _, k, _, _ in net.profile(N)]
    return 1 + sum(k not in (1, 4) for k in kinds), sum(k == 1 for k in kinds)


TOL_FP32, TOL_BF16 = 1e-4, 1e-2


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["bf16", "x3"])
def test_densenet_cifar_bc(nib, precision):
    torch.manual_seed(5)
    m = ocls.DenseNetCifar(depth=22, growth_rate=12, num_init_features=24, bn_size=4).eval()
    ocls._randomize_bn(m, 6)
    x = torch.rand(8, 3, 32, 32, generator=torch.Generator().manual_seed(7))
    _check_net(nib, m, x, precision, TOL_BF16 if precision == "bf16" else TOL_FP32)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "x3", "bf16"])
def test_densenet_cifar_no_bottleneck(nib, precision):
    """bn_size = 0: every dense layer is a pre-activated 3x3 (64 / 96 -> 32).  In bf16 each takes the pack pass and the
    tcgen05 conv on the packed tensor: one extra launch per layer."""
    torch.manual_seed(8)
    m = ocls.DenseNetCifar(depth=10, growth_rate=32, num_init_features=64, bn_size=0).eval()
    ocls._randomize_bn(m, 9)
    x = torch.rand(6, 3, 32, 32, generator=torch.Generator().manual_seed(10))
    net = _check_net(nib, m, x, precision, TOL_BF16 if precision == "bf16" else TOL_FP32)
    if precision == "bf16":
        total, tc = net.launch_counts()
        other, tcs = _launches_per_forward(net, 6)
        n_dense = sum(1 for blk in list(m.blocks.children())[::2] for _ in blk.children())
        assert tc == tcs and total - tc == other + n_dense, (total, tc, other, tcs, n_dense)


@pytest.mark.gpu
def test_tv_densenet_growth16_bf16(nib):
    """torchvision DenseNet-BC with growth 16 and bn_size 4: every bottleneck 1x1 is a pre-activated conv with Cout = 64
    and Cin of 64 .. 112 (one N tile, <= 9 K blocks), and every transition is one 128 -> 64: the transform must run on
    all of them (no pack pass, and no instantiation that skips it)."""
    import torchvision.models as tvm
    torch.manual_seed(11)
    m = tvm.DenseNet(growth_rate=16, block_config=(4, 4, 4, 4), num_init_features=64, bn_size=4, num_classes=10).eval()
    ocls._randomize_bn(m, 12)
    x = torch.rand(4, 3, 64, 64, generator=torch.Generator().manual_seed(13))
    net = _check_net(nib, m, x, "bf16", TOL_BF16)
    total, tc = net.launch_counts()
    other, tcs = _launches_per_forward(net, 4)
    assert tc == tcs and total - tc == other, (total, tc, other, tcs)
    assert tc >= 1 + 16 + 3, tc      # stem, 16 bottlenecks, 3 transitions (the 16-output growth convs: CUDA cores)
