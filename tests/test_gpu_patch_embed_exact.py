"""patch_embed_tc_kernel (csrc/patch_embed.cu) against float64 on its exact operands, and the two layout kernels of the
fusion / proj routes (nchw_to_nhwc16_kernel, upsample_bilinear_nhwc16_kernel, csrc/conv3x3.cu) against their definitions.

Patch embed.  The images and weights are rounded here as the kernel rounds them (fp16 / bf16: cvt.rn, torch's `.to`;
tf32: cvt.rna, round to nearest with ties away), then the 8 x 8 / 8 convolution is computed in float64 and the fp32 bias
added.  The kernel may differ only by its fp32 accumulation over K / 16 (tf32: K / 8) MMA instructions and the bias add:

    |got - ref| <= 4 steps 2^-24 S + 2^-23 (|ref| + |bias|)          (+ half a 16-bit ulp for a 16-bit output)

The exact fp32 route would miss this bar by the operand rounding (about 1e-3 of the result), so passing it also shows that
the tensor-core route ran.  Against a reference without one MMA K step the output must miss the bar by more than 4x."""
import pytest
import torch
import torch.nn.functional as F

from pixelspointspolygons_b200 import _lib
from test_gpu_conv3x3_exact import GUARD, check_sentinels, compare, stream

pytestmark = pytest.mark.gpu

NLC, NCHW = _lib.P3P_LAYOUT_NLC, _lib.P3P_LAYOUT_NCHW
F32, BF16, F16 = _lib.P3P_DTYPE_F32, _lib.P3P_DTYPE_BF16, _lib.P3P_DTYPE_F16
TDT = {F16: torch.float16, BF16: torch.bfloat16}
HALF_ULP = {F16: 2.0 ** -11, BF16: 2.0 ** -8}  # relative, normal range
OUT16 = {"fp16": F16, "bf16": BF16, "tf32": F16}


def pe_rows(H, W):
    """launch_patch_embed's row group: the most cell rows r dividing ny with r * nx <= 128 and a multiple of 16."""
    ny, nx = H // 8, W // 8
    for r in range(ny, 0, -1):
        if ny % r == 0 and r * nx <= 128 and (r * nx) % 16 == 0:
            return r
    return 0


# (in_chans, H, W, C) -> rows of the row group
PE_CASES = {
    (3, 224, 224, 384): 4,   # the encoders' image embedding
    (3, 224, 224, 512): 4,   # a second round of 1 tile
    (3, 224, 224, 768): 4,   # two full rounds (ViT-base width)
    (3, 224, 224, 129): 4,
    (1, 224, 224, 384): 4,   # 16-bit tiles of 16 KB: smaller than the fp32 NCHW epilogue's transpose staging
    (1, 224, 224, 512): 4,   # ... and a second round reading the image operand again
    (2, 128, 128, 200): 8,
    (3, 224, 448, 384): 2,
    (3, 160, 160, 384): 4,   # N = 80
}
PE_SHAPES = list(PE_CASES)


def tf32_rna(x):
    """cvt.rna.tf32.f32 of finite values: round the 13 dropped mantissa bits to nearest, ties away from zero."""
    bits = x.view(torch.int32).to(torch.int64) & 0xFFFFFFFF
    r = ((bits + 0x1000) & 0xFFFFE000) & 0xFFFFFFFF
    return torch.where(r >= 2 ** 31, r - 2 ** 32, r).to(torch.int32).view(torch.float32)


def operand(x, prec):
    """The kernel's MMA operand of fp32 x, in float64."""
    if prec == "tf32":
        return tf32_rna(x).double()
    return x.to(torch.float16 if prec == "fp16" else torch.bfloat16).double()


class PeCase:
    def __init__(self, dev, shape, prec, B=2, seed=0):
        ic, H, W, C = shape
        self.shape, self.prec, self.dev, self.B = shape, prec, dev, B
        self.ny, self.nx = H // 8, W // 8
        g = torch.Generator().manual_seed(seed * 1000 + ic + C + H + 3 * W)
        self.img = torch.randn(B, ic, H, W, generator=g).to(dev)
        self.w = (torch.randn(C, ic, 8, 8, generator=g) / (64 * ic) ** 0.5).to(dev)
        self.bias = (torch.randn(C, generator=g) * 0.1).to(dev)
        xd, wd = operand(self.img, prec), operand(self.w, prec)
        self.E = F.conv2d(xd, wd, stride=8).reshape(B, C, -1)
        S = F.conv2d(xd.abs(), wd.abs(), stride=8).reshape(B, C, -1)
        # one MMA K step: k = (c, py, px) in [0, 16) for 16-bit operands (rows py 0, 1 of channel 0), [0, 8) for tf32
        wm = torch.zeros_like(wd)
        kr = 1 if prec == "tf32" else 2
        wm[:, 0, :kr] = wd[:, 0, :kr]
        self.D = F.conv2d(xd, wm, stride=8).reshape(B, C, -1)
        K = ic * 64
        steps = K / 8 if prec == "tf32" else K / 16
        bd = self.bias.double().view(1, C, 1)
        self.ref = self.E + bd
        self.bound = 4 * steps * 2.0 ** -24 * S + 2.0 ** -23 * (self.ref.abs() + bd.abs()) + 1e-30
        l = _lib.lib()
        nbytes = l.p3p_patch_embed_blob_bytes(C, ic, 8)
        self.blob = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        _lib.check(l.p3p_patch_embed_prepare(self.w.data_ptr(), self.bias.data_ptr(), C, ic, 8, _lib.P3P_PRECISION[prec],
                                             self.blob.data_ptr(), nbytes, stream()), "p3p_patch_embed_prepare")

    def run(self, dtype, layout, c_total, c_offset, prepared, img=None):
        """-> (out buffer, (B, C, cells) view of the written channels); buffers start as NaN (16-bit: 0xFFFF)."""
        ic, H, W, C = self.shape
        img = self.img if img is None else img
        B = img.shape[0]
        cells = self.ny * self.nx
        n = B * cells * c_total
        if dtype == F32:
            out = torch.full((n + GUARD,), float("nan"), device=self.dev)
        else:
            out = torch.full((n + GUARD,), -1, dtype=torch.int16, device=self.dev)
        l = _lib.lib()
        p = _lib.P3P_PRECISION[self.prec]
        if prepared:  # no raw weights: only the tensor-core route can run
            rc = l.p3p_patch_embed_prepared(img.data_ptr(), B, ic, H, W, 8, self.blob.data_ptr(), None, None, C, p, out.data_ptr(),
                                            dtype, layout, c_total, c_offset, stream())
        else:
            rc = l.p3p_patch_embed(img.data_ptr(), B, ic, H, W, 8, self.w.data_ptr(), self.bias.data_ptr(), C, p, out.data_ptr(),
                                   dtype, layout, c_total, c_offset, stream())
        _lib.check(rc, "p3p_patch_embed")
        torch.cuda.synchronize()
        mask = torch.zeros(n + GUARD, dtype=torch.bool, device=self.dev)
        if layout == NLC:
            mask[:n].view(B, cells, c_total)[:, :, c_offset:c_offset + C] = True
        else:
            mask[:n].view(B, c_total, cells)[:, c_offset:c_offset + C] = True
        if dtype == F32:
            check_sentinels(out, mask)
            vals = out
        else:
            vals = out.view(TDT[dtype]).float()
            assert torch.isfinite(vals[mask]).all(), "elements of the output were not written"
            assert (out[~mask] == -1).all(), f"{int((out[~mask] != -1).sum())} elements outside the output were overwritten"
        body = vals[:n]
        if layout == NLC:
            got = body.view(B, cells, c_total)[:, :, c_offset:c_offset + C].permute(0, 2, 1)
        else:
            got = body.view(B, c_total, cells)[:, c_offset:c_offset + C]
        return out, got

    def check(self, got, dtype, what):
        bound = self.bound
        if dtype != F32:
            bound = bound + HALF_ULP[dtype] * (self.ref.abs() + bound) + 2.0 ** -25
        return compare(got, self.ref, self.ref - self.D, bound, f"{what} {self.shape} {self.prec}")


def outputs(prec, C):
    """(out dtype, layout, c_total, c_offset): fp32 NCHW (the transpose-staging epilogue), fp32 token rows, 16-bit token rows
    in the second half of a 2 C buffer (the fusion route's concat), 16-bit NCHW."""
    o16 = OUT16[prec]
    return [(F32, NCHW, C, 0), (F32, NLC, C, 0), (o16, NLC, 2 * C, C), (o16, NCHW, C, 0)]


@pytest.mark.parametrize("prec", ["fp16", "bf16", "tf32"])
@pytest.mark.parametrize("shape", PE_SHAPES, ids=["x".join(map(str, s)) for s in PE_SHAPES])
def test_patch_embed_exact(cuda_device, shape, prec):
    ic, H, W, C = shape
    assert pe_rows(H, W) == PE_CASES[shape]
    c = PeCase(cuda_device, shape, prec)
    for dtype, layout, c_total, c_offset in outputs(prec, C):
        what = f"{'fp32' if dtype == F32 else '16-bit'} {'NLC' if layout == NLC else 'NCHW'} c_offset={c_offset}"
        out, got = c.run(dtype, layout, c_total, c_offset, prepared=False)
        c.check(got, dtype, what)
        out_p, _ = c.run(dtype, layout, c_total, c_offset, prepared=True)
        assert torch.equal(out_p.view(torch.int16), out.view(torch.int16)), f"{what}: prepared weights differ from raw weights"
    # determinism and batch invariance (fp32 NCHW)
    out, got = c.run(F32, NCHW, C, 0, prepared=True)
    again, _ = c.run(F32, NCHW, C, 0, prepared=True)
    assert torch.equal(again.view(torch.int32), out.view(torch.int32)), "a repeated call is not bit-identical"
    _, one = c.run(F32, NCHW, C, 0, prepared=True, img=c.img[1:2])
    assert torch.equal(one[0], got[1]), "image 1 differs from the same image run alone"


@pytest.mark.parametrize("prec", ["fp16", "bf16", "tf32"])
def test_patch_embed_exact_batch_24(cuda_device, prec):
    """24 images at 224 x 224: 168 CTAs, more than one wave on 148 SMs; each image equals itself run alone."""
    C = 384
    c = PeCase(cuda_device, (3, 224, 224, C), prec, B=24, seed=1)
    _, got = c.run(F32, NCHW, C, 0, prepared=True)
    c.check(got, F32, "fp32 NCHW B=24")
    _, got16 = c.run(OUT16[prec], NLC, 2 * C, C, prepared=True)
    c.check(got16, OUT16[prec], "16-bit NLC B=24")
    for i in range(24):
        _, one = c.run(F32, NCHW, C, 0, prepared=True, img=c.img[i:i + 1])
        assert torch.equal(one[0], got[i]), f"image {i} differs from the same image run alone"


# ------------------------------------------------------------------------------------------------------------------------
# p3p_nchw_to_nhwc16: x.permute(0, 2, 3, 1).to(dtype) bit for bit
# ------------------------------------------------------------------------------------------------------------------------
SPECIALS = [0.0, -0.0, 1e-40, -1e-40, 6e-8, -3e-5, 65504.0, 65519.0, 65520.0, -7e4, 1e6, 3.0e38, float("inf"), float("-inf"),
            float("nan"), 1 + 2 ** -11, 1 + 3 * 2 ** -11, 1 + 2 ** -8, -(1 + 3 * 2 ** -8), 2.0 ** -24, 2.0 ** -25]


@pytest.mark.parametrize("prec", ["fp16", "bf16"])
@pytest.mark.parametrize("hw", [(1, 1), (3, 11), (28, 28)], ids=["HW1", "HW33", "HW784"])
@pytest.mark.parametrize("C", [1, 33, 768])
def test_nchw_to_nhwc16_bits(cuda_device, prec, hw, C):
    """Conversion as torch's: round to nearest even, subnormals kept, beyond the format's range inf (fp16 above 65504),
    NaN stays NaN (with the device's canonical payload); channels [2, 2 + C) of a C + 5 channel buffer, nothing else."""
    H, W = hw
    B, c_total, c_offset = 2, C + 5, 2
    dt = torch.float16 if prec == "fp16" else torch.bfloat16
    x = torch.randn(B, C, H, W, generator=torch.Generator().manual_seed(C + H))
    flat = x.view(-1)
    idx = torch.arange(0, flat.numel(), 5)
    flat[idx] = torch.tensor(SPECIALS)[torch.arange(idx.numel()) % len(SPECIALS)]
    xd = x.to(cuda_device)
    n = B * H * W * c_total
    out = torch.full((n + GUARD,), -1, dtype=torch.int16, device=cuda_device)
    rc = _lib.lib().p3p_nchw_to_nhwc16(xd.data_ptr(), B, C, H, W, _lib.P3P_PRECISION[prec], out.data_ptr(), c_total, c_offset,
                                       stream())
    _lib.check(rc, "p3p_nchw_to_nhwc16")
    torch.cuda.synchronize()
    out = out.cpu()
    got = out[:n].view(B, H, W, c_total)[..., c_offset:c_offset + C]
    want = x.permute(0, 2, 3, 1).to(dt)
    nan = torch.isnan(want)
    assert torch.equal(torch.isnan(got.view(dt)), nan), "NaN positions differ"
    assert torch.equal(got[~nan], want.view(torch.int16)[~nan]), f"{int((got[~nan] != want.view(torch.int16)[~nan]).sum())} values differ"
    mask = torch.zeros(n + GUARD, dtype=torch.bool)
    mask[:n].view(B, H, W, c_total)[..., c_offset:c_offset + C] = True
    assert (out[~mask] == -1).all(), "elements outside the output were overwritten"


# ------------------------------------------------------------------------------------------------------------------------
# p3p_upsample_bilinear_nhwc16: ATen's upsample_bilinear2d (align_corners = False) of token rows, rounded to 16 bits
# ------------------------------------------------------------------------------------------------------------------------
def source_index(n_out, n_in, fused):
    """ATen's fp32 source index: (dst + 0.5) * (n_in / n_out) - 0.5 clamped at 0 -> (i0, i1, lambda0, lambda1) as the kernel
    computes them, with the multiply-add rounded twice or (an FMA contraction) once."""
    scale = torch.tensor(n_in, dtype=torch.float32) / torch.tensor(n_out, dtype=torch.float32)
    o = torch.arange(n_out, dtype=torch.float32) + 0.5
    f = (o.double() * scale.double() - 0.5).float() if fused else o * scale - 0.5
    f = f.clamp_min(0.0)
    i0 = f.long()
    i1 = i0 + (i0 < n_in - 1).long()
    l1 = f - i0.float()
    return i0, i1, (1.0 - l1).double(), l1.double()


def upsample_ref(src, H, W, fused):
    """src (B, h, w, C) float64 -> (B, H, W, C) float64 weighted sums, and the largest of the four neighbours."""
    _, h, w, _ = src.shape
    y0, y1, hy, ly = (t.to(src.device) for t in source_index(H, h, fused))
    x0, x1, hx, lx = (t.to(src.device) for t in source_index(W, w, fused))
    r0, r1 = src[:, y0], src[:, y1]
    v00, v01, v10, v11 = r0[:, :, x0], r0[:, :, x1], r1[:, :, x0], r1[:, :, x1]
    hy, ly, hx, lx = hy.view(1, -1, 1, 1), ly.view(1, -1, 1, 1), hx.view(1, 1, -1, 1), lx.view(1, 1, -1, 1)
    v = hy * (hx * v00 + lx * v01) + ly * (hx * v10 + lx * v11)
    m = torch.stack([v00.abs(), v01.abs(), v10.abs(), v11.abs()]).amax(0)
    return v, m


def ordered(bits16):
    """16-bit float bit patterns -> integers in value order (adjacent values differ by 1, +0 == -0)."""
    b = bits16.int()
    return torch.where(b < 0, -(b & 0x7FFF), b)


UPS = [((28, 28), (224, 224)), ((5, 7), (24, 32)), ((28, 28), (14, 14)), ((1, 1), (8, 8)), ((1, 7), (3, 5)), ((7, 1), (4, 9)),
       ((28, 28), (28, 28)), ((13, 9), (100, 3))]


# 28 x 28 -> 224 x 224 at the proj tails' width; the other sizes at odd and tiny widths
UPS_CASES = [(UPS[0], 384)] + [(u, C) for u in UPS[1:] for C in (1, 3, 385)]


def ups_id(case):
    ((h, w), (H, W)), C = case
    return f"{h}x{w}-{H}x{W}-C{C}"


@pytest.mark.parametrize("prec", ["fp16", "bf16"])
@pytest.mark.parametrize("sizes, C", UPS_CASES, ids=[ups_id(u) for u in UPS_CASES])
def test_upsample_bilinear_exact(cuda_device, sizes, C, prec):
    """Token rows (B, 1 + h w, C) with the class token skipped through the batch stride; the float64 weighted sum of the
    kernel's fp32 weights, within half a 16-bit ulp + 2^-20 of the largest neighbour; within 1 ulp of F.interpolate in
    fp32 + .to(dtype) and equal to it in >= 99.9 % of elements; 16-bit sentinels after the output intact."""
    (h, w), (H, W) = sizes
    B, skip = 2, 1
    dt = torch.float16 if prec == "fp16" else torch.bfloat16
    o16 = F16 if prec == "fp16" else BF16
    tokens = torch.randn(B, skip + h * w, C, generator=torch.Generator().manual_seed(h * 31 + w + C)).to(cuda_device)
    n = B * H * W * C
    out = torch.full((n + GUARD,), -1, dtype=torch.int16, device=cuda_device)
    src = tokens.view(-1)[skip * C:]
    rc = _lib.lib().p3p_upsample_bilinear_nhwc16(src.data_ptr(), B, h, w, C, (skip + h * w) * C, H, W, _lib.P3P_PRECISION[prec],
                                                 out.data_ptr(), stream())
    _lib.check(rc, "p3p_upsample_bilinear_nhwc16")
    torch.cuda.synchronize()
    assert (out[n:] == -1).all(), "elements after the output were overwritten"
    got16 = out[:n].view(B, H, W, C)
    got = got16.view(dt).double()
    assert torch.isfinite(got).all(), "elements of the output were not written"
    x = tokens[:, skip:].double().view(B, h, w, C)
    errs = []
    for fused in (False, True):
        v, m = upsample_ref(x, H, W, fused)
        bound = HALF_ULP[o16] * v.abs() + 2.0 ** -20 * m + 2.0 ** -25
        errs.append((got - v).abs() / bound)
    ratio = torch.minimum(*errs).max().item()
    print(f"upsample {sizes} C={C} {prec}: max |err| / bound = {ratio:.3g}")
    assert ratio <= 1.0, f"upsample {sizes} C={C} {prec}: max |err| / bound = {ratio:.3g}"
    xi = tokens[:, skip:].view(B, h, w, C).permute(0, 3, 1, 2)
    ti = F.interpolate(xi, size=(H, W), mode="bilinear", align_corners=False).permute(0, 2, 3, 1).to(dt)
    d = (ordered(got16) - ordered(ti.view(torch.int16))).abs()
    # Where the four neighbours nearly cancel, one 16-bit ulp of the result is far below the fp32 differences of two
    # implementations (summation order, FMA contraction of the index and of the weighted sum): there the two may differ by
    # up to 2^-16 of the largest neighbour instead.
    _, m = upsample_ref(x, H, W, False)
    far = (d > 1) & ((got - ti.double()).abs() > 2.0 ** -16 * m)
    print(f"  vs F.interpolate: {int((d > 1).sum())} elements > 1 ulp, {(d == 0).double().mean().item():.5%} equal")
    assert not far.any(), f"{int(far.sum())} elements more than 1 ulp and 2^-16 of the largest neighbour from F.interpolate"
    assert (d == 0).double().mean().item() >= 0.999, f"only {(d == 0).double().mean().item():.4%} equal to F.interpolate"
