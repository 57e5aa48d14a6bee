"""conv3x3_tc_kernel (csrc/conv3x3.cu) against float64 on its exact operands, across the strip planner's shape contract.

Every operand the kernel feeds its MMAs is a 16-bit value, read back here from the prepared blob; the product of two of
them is exact in float64.  So conv2d in float64 over exactly those operands is the true result, and the kernel may
differ from it only by its fp32 accumulation and epilogue roundings.  Per element that is bounded by

    |got - ref| <= 4 (K / 16) 2^-24 S + 2^-23 (|E + shift| + |shift|)        S = conv2d(|x16|, |Wp|)

a rigorous fp32 chain bound over the K / 16 MMA instructions with a factor 4 for whatever the tensor core does inside one
K step.  The bar is shown to mean something in every case: the output must violate it, by more than 4x, against a
mutated reference that lacks one MMA K step (input channels [0, 16) of the centre tap).  Output buffers start as NaN:
everything inside the written region must be finite and everything outside it must keep its bits."""
import ctypes as C
import math

import pytest
import torch
import torch.nn.functional as F

from pixelspointspolygons_b200 import _lib

pytestmark = pytest.mark.gpu

DT = {"fp16": torch.float16, "bf16": torch.bfloat16}
PREC = {"fp16": _lib.P3P_PRECISION["fp16"], "bf16": _lib.P3P_PRECISION["bf16"]}
NLC, NCHW = _lib.P3P_LAYOUT_NLC, _lib.P3P_LAYOUT_NCHW
NAN_BITS = 0x7FC00000
GUARD = 4099  # fp32 elements after the last image that must keep their bits
EPS = 1e-5


def plan(H, W, Cout):
    """launch_conv3x3_any's planner: (rows, N, acc_stride, strips, co_tiles, stages)."""
    co_tiles = (Cout + 127) // 128
    rows = 0
    r = 1
    while r <= H and r * W <= 256:
        if (r * W) % 16 == 0 and co_tiles * (128 if r * W <= 128 else 256) <= 512:
            rows = r
        r += 1
    N = rows * W
    stage_bytes = co_tiles * 128 * 128 + (N * 128 + 1023) // 1024 * 1024
    return rows, N, 128 if N <= 128 else 256, -(-H // rows), co_tiles, min(8, 200 * 1024 // stage_bytes)


# (B, Cin, Cout, H, W) -> what the planner must pick: (rows, N, acc_stride, strips, co_tiles, stages)
CASES = {
    (2, 768, 384, 28, 28): (4, 112, 128, 7, 3, 3),       # fusion_layer of the early-fusion encoders
    (2, 128, 256, 28, 28): (8, 224, 256, 4, 2, 3),       # last strip of 4 rows
    (2, 64, 128, 28, 28): (8, 224, 256, 4, 1, 4),
    (1, 128, 129, 16, 16): (16, 256, 256, 1, 2, 3),      # 2 tiles x 256 columns = all of TMEM; tile 2 holds 1 channel
    (1, 64, 1, 16, 16): (16, 256, 256, 1, 1, 4),
    (3, 64, 257, 20, 20): (4, 80, 128, 5, 3, 3),         # last tile holds 1 channel
    (1, 64, 96, 17, 15): (16, 240, 256, 2, 1, 4),        # odd width, last strip of 1 row, HW = 255: scalar NCHW stores
    (2, 64, 64, 41, 6): (40, 240, 256, 2, 1, 4),         # HW = 246
    (1, 64, 64, 16, 1): (16, 16, 128, 1, 1, 8),          # W = 1, the smallest N
    (2, 64, 128, 1, 16): (1, 16, 128, 1, 1, 8),          # H = 1: both vertical taps are padding
    (1, 64, 256, 1, 256): (1, 256, 256, 1, 2, 3),        # the widest image
    (1, 1536, 384, 8, 16): (8, 128, 128, 1, 3, 3),       # 216 K iterations through 3 stages
    (24, 64, 384, 28, 28): (4, 112, 128, 7, 3, 3),       # 168 CTAs: more than one wave on 148 SMs
    (1, 384, 256, 224, 224): (1, 224, 256, 224, 2, 3),   # proj tail at its real size
}
SHAPES = list(CASES)
PRODUCTION = (2, 768, 384, 28, 28)


def stream():
    return torch.cuda.current_stream().cuda_stream


class Case:
    """One convolution: parameters, prepared blob, decoded operands, input and float64 references."""

    def __init__(self, dev, shape, prec, seed=0, bn=True, bias=True):
        B, Cin, Cout, H, W = shape
        self.shape, self.prec, self.dev, self.bn, self.has_bias = shape, prec, dev, bn, bias
        g = torch.Generator().manual_seed(1000 * seed + Cin + 7 * Cout + 13 * H + W)
        self.w = torch.randn(Cout, Cin, 3, 3, generator=g) / math.sqrt(9 * Cin)
        self.bias = torch.randn(Cout, generator=g) * 0.1 if bias else None
        if bn:
            self.gamma = torch.rand(Cout, generator=g) + 0.5
            self.gamma[::5] *= -1.0
            self.beta = torch.randn(Cout, generator=g) * 0.1
            self.mean = torch.randn(Cout, generator=g) * 0.1
            self.var = torch.rand(Cout, generator=g) + 0.5
        x = torch.randn(B, H, W, Cin, generator=g)
        x[:, 0] += 1.0  # borders matter (zero padding)
        self.x16 = x.to(DT[prec]).to(dev)
        self.blob = self._prepare()
        cout_pad = (Cout + 127) // 128 * 128
        nw = cout_pad * 9 * Cin
        self.wp = self.blob[: 2 * nw].view(DT[prec]).view(cout_pad, 9 * Cin)
        self.shift = self.blob[2 * nw: 2 * nw + 4 * cout_pad].view(torch.float32)
        # float64 references over the exact operands (on the device: tens of GFLOP at the larger shapes)
        Wd = self.wp[:Cout].double().view(Cout, 3, 3, Cin).permute(0, 3, 1, 2)
        xd = self.x16.double().permute(0, 3, 1, 2)
        self.K = 9 * Cin
        self.E = F.conv2d(xd, Wd, padding=1).view(B, Cout, H * W)
        S = F.conv2d(xd.abs(), Wd.abs(), padding=1).view(B, Cout, H * W)
        # one MMA K step: input channels [0, 16) of the centre tap (never padding, so it counts at every position)
        self.D = torch.einsum("bhwc,oc->bohw", xd.permute(0, 2, 3, 1)[..., :16], Wd[:, :16, 1, 1]).reshape(B, Cout, H * W)
        sh = self.shift[:Cout].double().view(1, Cout, 1)
        self.pre = self.E + sh
        self.bound = 4 * (self.K / 16) * 2.0 ** -24 * S + 2.0 ** -23 * (self.pre.abs() + sh.abs()) + 1e-30

    def _prepare(self):
        B, Cin, Cout, H, W = self.shape
        d = self.dev
        self.dev_params = [t.to(d) if t is not None else None for t in (
            self.w, self.bias, *((self.gamma, self.beta, self.mean, self.var) if self.bn else (None,) * 4))]
        p = _lib.ConvParams()
        for name, t in zip(("weight", "bias", "norm_weight", "norm_bias", "norm_mean", "norm_var"), self.dev_params):
            setattr(p, name, t.data_ptr() if t is not None else None)
        p.eps, p.in_channels, p.out_channels = EPS, Cin, Cout
        l = _lib.lib()
        nbytes = l.p3p_conv3x3_blob_bytes(Cin, Cout)
        blob = torch.empty(nbytes, dtype=torch.uint8, device=d)
        _lib.check(l.p3p_conv3x3_prepare(C.byref(p), PREC[self.prec], blob.data_ptr(), nbytes, stream()), "p3p_conv3x3_prepare")
        torch.cuda.synchronize()
        return blob

    def check_blob(self):
        """Weights: to16(fp32(gamma / sqrt(var + eps)) * w) bit for bit; shift: BN shift + bias, either rounding of the one
        FMA contraction nvcc may make; pad rows and pad shifts 0.  The kernel's fp32 operations are IEEE (no fast-math), so
        each is emulated here as the float64 operation on fp32 values rounded once to fp32, which is the correctly rounded
        fp32 result for +, -, *, / and sqrt.  (torch's own fp32 sqrt on the CPU is not correctly rounded in every case.)"""
        Cout, Cin = self.shape[2], self.shape[1]

        def f32(t):
            return t.double().float()

        if self.bn:
            s = f32(torch.sqrt(f32(self.var.double() + torch.tensor(EPS, dtype=torch.float32).double()).double()))
            a = f32(self.gamma.double() / s.double())
        else:
            a = torch.ones(Cout)
        want = f32(a.double()[:, None, None, None] * self.w.double()).permute(0, 2, 3, 1).reshape(Cout, 9 * Cin).to(DT[self.prec])
        wp = self.wp.cpu()
        bad = wp[:Cout].view(torch.int16) != want.view(torch.int16)
        assert not bad.any(), f"prepared weights differ from to16(scale * w) in {int(bad.sum())} elements"
        assert not wp[Cout:].view(torch.int16).any(), "pad rows of the prepared weights are not 0"
        sh = self.shift.cpu()
        b = self.bias if self.bias is not None else torch.zeros(Cout)
        if self.bn:
            d = f32(b.double() - self.mean.double())
            plain = f32(f32(a.double() * d.double()).double() + self.beta.double())
            fused = f32(a.double() * d.double() + self.beta.double())
            ok = (sh[:Cout] == plain) | (sh[:Cout] == fused)
            assert ok.all(), f"shift differs in channels {torch.nonzero(~ok).flatten().tolist()}"
        else:
            assert torch.equal(sh[:Cout], b), "shift without BatchNorm is not the bias"
        assert not sh[Cout:].any(), "pad shifts are not 0"

    def run(self, layout=NLC, relu=1, c_total=None, c_offset=0, x16=None, B=None):
        _, Cin, Cout, H, W = self.shape
        x16 = self.x16 if x16 is None else x16
        B = x16.shape[0] if B is None else B
        c_total = Cout if c_total is None else c_total
        n = B * H * W * c_total
        out = torch.full((n + GUARD,), float("nan"), device=self.dev)
        rc = _lib.lib().p3p_conv3x3(x16.data_ptr(), B, H, W, Cin, self.blob.data_ptr(), Cout, PREC[self.prec], relu, out.data_ptr(),
                                    layout, c_total, c_offset, stream())
        _lib.check(rc, "p3p_conv3x3")
        torch.cuda.synchronize()
        mask = torch.zeros(n + GUARD, dtype=torch.bool, device=self.dev)
        if layout == NLC:
            mask[:n].view(B, H * W, c_total)[:, :, c_offset:c_offset + Cout] = True
            got = out[:n].view(B, H * W, c_total)[:, :, c_offset:c_offset + Cout].permute(0, 2, 1)
        else:
            mask[:n].view(B, c_total, H * W)[:, c_offset:c_offset + Cout] = True
            got = out[:n].view(B, c_total, H * W)[:, c_offset:c_offset + Cout]
        check_sentinels(out, mask)
        return out, got  # got: (B, Cout, H W)

    def compare(self, got, relu, what):
        ref = self.pre.clamp_min(0) if relu else self.pre  # ReLU is 1-Lipschitz: the same bound holds after it
        mut = (self.pre - self.D).clamp_min(0) if relu else self.pre - self.D
        return compare(got, ref, mut, self.bound, f"{what} {self.shape} {self.prec} relu={relu}")


def check_sentinels(out, mask):
    """Every element of the written region is finite (it was written), every other keeps its NaN bits (no stray store)."""
    assert torch.isfinite(out[mask]).all(), f"{int((~torch.isfinite(out[mask])).sum())} elements of the output were not written"
    outside = out.view(torch.int32)[~mask]
    assert (outside == NAN_BITS).all(), f"{int((outside != NAN_BITS).sum())} elements outside the output were overwritten"


def compare(got, ref, mut, bound, what):
    """max |got - ref| / bound must be <= 1, and against the reference without one MMA K step it must exceed 4."""
    err = (got.double() - ref).abs() / bound
    ratio = err.max().item()
    mratio = ((got.double() - mut).abs() / bound).max().item()
    msg = f"{what}: max |err| / bound = {ratio:.3g}, without one K step {mratio:.3g}"
    print(msg)
    assert ratio <= 1.0, msg + f" at {tuple(int(i) for i in torch.nonzero(err == err.max())[0])}"
    assert mratio > 4.0, msg + " (the bar cannot see one missing K step)"
    return ratio


@pytest.mark.parametrize("prec", ["fp16", "bf16"])
@pytest.mark.parametrize("shape", SHAPES, ids=["x".join(map(str, s)) for s in SHAPES])
def test_conv3x3_exact(cuda_device, shape, prec):
    B, Cin, Cout, H, W = shape
    assert plan(H, W, Cout) == CASES[shape]
    c = Case(cuda_device, shape, prec)
    c.check_blob()
    out_nlc, got_nlc = c.run(NLC)
    c.compare(got_nlc, 1, "NLC")
    _, got_nchw = c.run(NCHW)
    c.compare(got_nchw, 1, "NCHW")
    assert torch.equal(got_nchw, got_nlc), "NCHW and NLC stores of the same accumulators differ"
    again, _ = c.run(NLC)
    assert torch.equal(again.view(torch.int32), out_nlc.view(torch.int32)), "a repeated call is not bit-identical"
    if B > 1:  # each image as a batch of one: bit-identical
        for i in range(B):
            _, one = c.run(NLC, x16=c.x16[i:i + 1])
            assert torch.equal(one[0], got_nlc[i]), f"image {i} differs from the same image run alone"


@pytest.mark.parametrize("prec", ["fp16", "bf16"])
@pytest.mark.parametrize("shape", [(2, 128, 256, 28, 28), (1, 64, 96, 17, 15), (2, 64, 64, 41, 6)],
                         ids=["2x128x256x28x28", "1x64x96x17x15", "2x64x64x41x6"])
def test_conv3x3_channel_offset(cuda_device, shape, prec):
    """Channels [32, 32 + Cout) of a buffer of Cout + 64 channels, as token rows and as NCHW."""
    Cout = shape[2]
    c = Case(cuda_device, shape, prec, seed=1)
    for layout, name in ((NLC, "NLC"), (NCHW, "NCHW")):
        _, got = c.run(layout, c_total=Cout + 64, c_offset=32)
        c.compare(got, 1, f"{name} c_offset=32 c_total={Cout + 64}")


@pytest.mark.parametrize("prec", ["fp16", "bf16"])
def test_conv3x3_relu_off(cuda_device, prec):
    """relu = 0 of the C entry (the Python modules always pass 1): the negative half of the outputs is checked too."""
    c = Case(cuda_device, PRODUCTION, prec, seed=2)
    for layout, name in ((NLC, "NLC"), (NCHW, "NCHW")):
        _, got = c.run(layout, relu=0)
        assert (got < 0).float().mean() > 0.3, "ReLU was applied"
        c.compare(got, 0, name)


@pytest.mark.parametrize("prec", ["fp16", "bf16"])
@pytest.mark.parametrize("shape", [(2, 64, 128, 28, 28), (3, 64, 257, 20, 20)], ids=["2x64x128x28x28", "3x64x257x20x20"])
def test_conv3x3_without_batchnorm_or_bias(cuda_device, shape, prec):
    """p3p_conv_params with norm_weight = NULL and bias = NULL: weights to16(w), shift 0; relu = 0."""
    c = Case(cuda_device, shape, prec, seed=3, bn=False, bias=False)
    c.check_blob()
    _, got = c.run(NCHW, relu=0)
    c.compare(got, 0, "NCHW no BN no bias")
    c2 = Case(cuda_device, shape, prec, seed=4, bn=False, bias=True)
    c2.check_blob()
    _, got = c2.run(NLC, relu=1)
    c2.compare(got, 1, "NLC no BN")


@pytest.mark.parametrize("prec", ["fp16", "bf16"])
def test_conv3x3_vit_tokens_exact(cuda_device, prec):
    """p3p_conv3x3_vit_tokens: row 0 = cls_token + pos_embed[0] bit for bit, row 1 + pos = relu(E + shift) + pos_embed[1 + pos]
    within the conv bound plus the fp32 add's rounding; guard rows after the last image keep their bits."""
    B, Cin, Cout, H, W = PRODUCTION
    c = Case(cuda_device, PRODUCTION, prec, seed=5)
    g = torch.Generator().manual_seed(6)
    cls = torch.randn(Cout, generator=g).to(cuda_device)
    pos = torch.randn(1 + H * W, Cout, generator=g).to(cuda_device)
    n = B * (1 + H * W) * Cout
    out = torch.full((n + GUARD,), float("nan"), device=cuda_device)
    rc = _lib.lib().p3p_conv3x3_vit_tokens(c.x16.data_ptr(), B, H, W, Cin, c.blob.data_ptr(), Cout, PREC[prec], cls.data_ptr(),
                                           pos.data_ptr(), out.data_ptr(), stream())
    _lib.check(rc, "p3p_conv3x3_vit_tokens")
    torch.cuda.synchronize()
    mask = torch.zeros(n + GUARD, dtype=torch.bool, device=cuda_device)
    mask[:n] = True
    check_sentinels(out, mask)
    tok = out[:n].view(B, 1 + H * W, Cout)
    for b in range(B):
        assert torch.equal(tok[b, 0], cls + pos[0]), f"class-token row of image {b}"
    posd = pos[1:].double().t().unsqueeze(0)  # (1, Cout, H W)
    ref = c.pre.clamp_min(0) + posd
    mut = (c.pre - c.D).clamp_min(0) + posd
    compare(tok[:, 1:].permute(0, 2, 1), ref, mut, c.bound + 2.0 ** -23 * ref.abs(), f"vit tokens {PRODUCTION} {prec}")
