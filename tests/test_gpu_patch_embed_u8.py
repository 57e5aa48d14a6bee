"""The uint8 image route of the patch embedding (p3p_patch_embed_u8, `PatchEmbed` / `EarlyFusionFrontEnd` on uint8
(B, H, W, in_chans), `HostPipeline(image_dtype=torch.uint8)`) against the fp32 route fed the image the pixel table stands
for, x[b][c][y][x] = lut[c][u8[b][y][x][c]].  The table is applied exactly, so every comparison is bit for bit (int32 /
int16 patterns: inf and NaN compare too)."""
import pytest
import torch

from oracle import pillars_oracle as po
from pixelspointspolygons_b200 import HostPipeline, PatchEmbed
from pixelspointspolygons_b200 import _lib
from pixelspointspolygons_b200.fusion import default_pixel_lut
from test_gpu_conv3x3_exact import GUARD, stream
from test_gpu_fusion_vit_tokens import front_end, tiles_for, vit_params
from test_gpu_parity import TOL, assert_close, to_nested
from test_gpu_patch_embed_exact import pe_rows
from test_gpu_pipeline import TOTAL, direct_points, fill, las_batch

pytestmark = pytest.mark.gpu

NLC, NCHW = _lib.P3P_LAYOUT_NLC, _lib.P3P_LAYOUT_NCHW
F32, BF16, F16 = _lib.P3P_DTYPE_F32, _lib.P3P_DTYPE_BF16, _lib.P3P_DTYPE_F16
OUT16 = {"fp16": F16, "bf16": BF16, "tf32": F16, "fp32": BF16}
PRECS = ["fp16", "bf16", "tf32", "fp32"]


def route(ic, H, W, P, C, prec):
    """launch_patch_embed's planner: "tc" (tensor cores) or "simt" (exact kernel) -- the same for both image formats."""
    if prec == "fp32" or P != 8:
        return "simt"
    rows, nx, ny = pe_rows(H, W), W // 8, H // 8
    tf32 = prec == "tf32"
    K, esize = ic * 64, (4 if tf32 else 2)
    smem = 1024 + ((1 if tf32 else 3) * 128 + rows * nx) * K * esize
    k_ok = K % (32 if tf32 else 64) == 0
    aligned = all((ny * nx * e) % 16 == 0 for e in (4, 2))
    return "tc" if rows > 0 and k_ok and smem <= 200 * 1024 and aligned else "simt"


def random_lut(ic, seed, big=False):
    """(ic, 256) fp32 with negative values, subnormals, +-0 (and, for `big`, values beyond fp16's 65504)."""
    g = torch.Generator().manual_seed(seed)
    lut = torch.randn(ic, 256, generator=g)
    specials = [0.0, -0.0, 1e-40, -1e-40, 2.0 ** -130, -3.5, 6e-8]
    if big:
        specials += [7e4, -1e5, 65520.0]
    for c in range(ic):
        for i, v in enumerate(specials):
            lut[c, (37 * c + 11 * i) % 256] = v
    return lut


def expand(img8, lut):
    """uint8 (B, H, W, ic) + (ic, 256) -> fp32 (B, ic, H, W): lut[c][u]."""
    ic = img8.shape[3]
    idx = img8.permute(0, 3, 1, 2).long() + 256 * torch.arange(ic, device=img8.device).view(1, -1, 1, 1)
    return lut.to(img8.device).reshape(-1)[idx].contiguous()


# (in_chans, H, W, C, P): every in_chans at every image size, the three widths in turn; P = 4 (exact route); in_chans 4 on
# the tensor cores (tf32 at 64 x 64: the only precision whose operands fit)
SHAPES = [(ic, H, W, (200, 384, 512)[(i + ic) % 3], 8) for ic in (1, 2, 3, 4)
          for i, (H, W) in enumerate([(224, 224), (160, 160), (128, 128), (224, 448)])] + [(3, 224, 224, 384, 4), (4, 64, 64, 384, 8)]


class U8Case:
    def __init__(self, dev, shape, prec, seed=0, big=False, B=2):
        ic, H, W, C, P = shape
        self.shape, self.prec, self.dev, self.B = shape, prec, dev, B
        g = torch.Generator().manual_seed(seed * 7919 + ic * 101 + H + W + C + P)
        self.img8 = torch.randint(0, 256, (B, H, W, ic), dtype=torch.uint8, generator=g).to(dev)
        self.lut = random_lut(ic, seed + ic, big).to(dev)
        self.x = expand(self.img8, self.lut)
        scale = 8.0 if big else 1.0
        self.w = (torch.randn(C, ic, P, P, generator=g) / (P * P * ic) ** 0.5 * scale).to(dev)
        self.bias = (torch.randn(C, generator=g) * 0.1).to(dev)
        l = _lib.lib()
        nbytes = l.p3p_patch_embed_blob_bytes(C, ic, P)
        self.blob = torch.zeros(nbytes, dtype=torch.uint8, device=dev)
        _lib.check(l.p3p_patch_embed_prepare(self.w.data_ptr(), self.bias.data_ptr(), C, ic, P, _lib.P3P_PRECISION[prec],
                                             self.blob.data_ptr(), nbytes, stream()), "p3p_patch_embed_prepare")

    def buffer(self, dtype, c_total):
        ic, H, W, C, P = self.shape
        n = self.B * (H // P) * (W // P) * c_total
        if dtype == F32:
            return torch.full((n + GUARD,), float("nan"), device=self.dev), n
        return torch.full((n + 2 * GUARD,), -1, dtype=torch.int16, device=self.dev), n

    def call(self, u8, weights, dtype, layout, c_total, c_offset, check=True):
        """weights: "raw" (weight + bias, no blob), "blob" (prepared weights + raw) or "blob_only" (no raw weights: only the
        tensor-core route can run).  -> (return code, output buffer)."""
        ic, H, W, C, P = self.shape
        out, _ = self.buffer(dtype, c_total)
        l = _lib.lib()
        p = _lib.P3P_PRECISION[self.prec]
        blob = None if weights == "raw" else self.blob.data_ptr()
        w = None if weights == "blob_only" else self.w.data_ptr()
        b = None if weights == "blob_only" else self.bias.data_ptr()
        if u8:
            rc = l.p3p_patch_embed_u8(self.img8.data_ptr(), self.lut.data_ptr(), self.B, ic, H, W, P, blob, w, b, C, p,
                                      out.data_ptr(), dtype, layout, c_total, c_offset, stream())
        elif weights == "raw":
            rc = l.p3p_patch_embed(self.x.data_ptr(), self.B, ic, H, W, P, w, b, C, p, out.data_ptr(), dtype, layout, c_total,
                                   c_offset, stream())
        else:
            rc = l.p3p_patch_embed_prepared(self.x.data_ptr(), self.B, ic, H, W, P, blob, w, b, C, p, out.data_ptr(), dtype, layout,
                                            c_total, c_offset, stream())
        if check:
            _lib.check(rc, "patch embed")
        torch.cuda.synchronize()
        return rc, out

    def mask(self, dtype, layout, c_total, c_offset):
        ic, H, W, C, P = self.shape
        out, n = self.buffer(dtype, c_total)
        cells = (H // P) * (W // P)
        m = torch.zeros(out.numel(), dtype=torch.bool, device=self.dev)
        if layout == NLC:
            m[:n].view(self.B, cells, c_total)[:, :, c_offset:c_offset + C] = True
        else:
            m[:n].view(self.B, c_total, cells)[:, c_offset:c_offset + C] = True
        return m


def bits(out):
    return out.view(torch.int32) if out.dtype == torch.float32 else out


def outputs(prec, C):
    o16 = OUT16[prec]
    return [(F32, NCHW, C, 0), (F32, NLC, C, 0), (o16, NLC, 2 * C, C), (o16, NCHW, C, 0)]


def check_case(c):
    ic, H, W, C, P = c.shape
    r = route(ic, H, W, P, C, c.prec)
    for dtype, layout, c_total, c_offset in outputs(c.prec, C):
        what = f"{c.shape} {c.prec} out={dtype} layout={layout} c_offset={c_offset}"
        mask = c.mask(dtype, layout, c_total, c_offset)
        sentinel = bits(c.buffer(dtype, c_total)[0])
        for weights in ("raw", "blob"):
            _, want = c.call(False, weights, dtype, layout, c_total, c_offset)
            _, got = c.call(True, weights, dtype, layout, c_total, c_offset)
            assert torch.equal(bits(got), bits(want)), f"{what} {weights}: {int((bits(got) != bits(want)).sum())} elements differ"
            assert torch.equal(bits(got)[~mask], sentinel[~mask]), f"{what} {weights}: elements outside the channels were written"
            assert not torch.equal(bits(got)[mask], sentinel[mask]), f"{what} {weights}: nothing was written"
        # the route: with the prepared weights alone only the tensor-core route runs; both formats take the same one
        rc8, _ = c.call(True, "blob_only", dtype, layout, c_total, c_offset, check=False)
        rc32, _ = c.call(False, "blob_only", dtype, layout, c_total, c_offset, check=False)
        if r == "tc":
            assert rc8 == 0 and rc32 == 0, f"{what}: the tensor-core route was expected ({_lib.lib().p3p_last_error()})"
        else:
            assert rc8 == rc32 == -2, f"{what}: the exact route was expected"  # P3P_ERR_UNSUPPORTED: it needs the raw weights
            assert b"exact route" in _lib.lib().p3p_last_error()


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("shape", SHAPES, ids=["ic{}-{}x{}-C{}-P{}".format(*s) for s in SHAPES])
def test_u8_route_equals_fp32_route_on_the_expanded_image(cuda_device, shape, prec):
    check_case(U8Case(cuda_device, shape, prec))


def test_u8_route_fp16_operands_beyond_65504(cuda_device):
    """Table values above fp16's range become inf operands (and NaN / inf outputs) in both routes alike."""
    c = U8Case(cuda_device, (3, 224, 224, 384, 8), "fp16", seed=3, big=True)
    _, out = c.call(True, "blob", F32, NCHW, 384, 0)
    assert not torch.isfinite(out[:-GUARD]).all(), "no value beyond 65504 reached an operand"
    check_case(c)


def test_planner_routes_of_the_covered_shapes():
    """The shapes above reach both routes: in_chans 4 at 16-bit and at tf32 exceeds the operand budget, P = 4 is exact."""
    assert route(4, 224, 224, 8, 384, "fp16") == "simt" and route(4, 224, 224, 8, 384, "tf32") == "simt"
    assert route(3, 224, 224, 8, 384, "fp16") == "tc" and route(3, 224, 448, 8, 384, "tf32") == "tc"
    assert route(3, 224, 224, 4, 384, "fp16") == "simt"
    assert route(4, 64, 64, 8, 384, "tf32") == "tc" and route(4, 64, 64, 8, 384, "fp16") == "simt"


# ------------------------------------------------------------------------------------------------------------------------
# PatchEmbed: the table
# ------------------------------------------------------------------------------------------------------------------------
def test_default_table_and_set_pixel_lut(cuda_device):
    pe = PatchEmbed(embed_dim=384, precision="fp16").to(cuda_device).eval()
    want = torch.arange(256).float().div(255)
    assert torch.equal(pe.pixel_lut.view(torch.int32), want.expand(3, 256).contiguous().view(torch.int32))
    assert torch.equal(default_pixel_lut(3), pe.pixel_lut)
    assert set(pe.state_dict()) == {"proj.weight", "proj.bias"}
    g = torch.Generator().manual_seed(4)
    img8 = torch.randint(0, 256, (2, 224, 224, 3), dtype=torch.uint8, generator=g).to(cuda_device)

    def pair():
        with torch.no_grad():
            got = pe(img8)
            want = pe(expand(img8, pe.pixel_lut))
        torch.cuda.synchronize()
        return got, want

    got, want = pair()
    assert torch.equal(got.view(torch.int32), want.view(torch.int32))
    blob = pe._blob(cuda_device, "fp16")
    # albumentations-style Normalize (ImageNet mean / std, max_pixel_value 255) as a table, per channel
    mean, std = torch.tensor([0.485, 0.456, 0.406]), torch.tensor([0.229, 0.224, 0.225])
    lut = (torch.arange(256).float().view(1, 256) - mean.view(3, 1) * 255) / (std.view(3, 1) * 255)
    pe.set_pixel_lut(lut)
    assert torch.equal(pe.pixel_lut, lut)
    got2, want2 = pair()
    assert torch.equal(got2.view(torch.int32), want2.view(torch.int32))
    assert not torch.equal(got2, got), "the new table was not used"
    assert pe._blob(cuda_device, "fp16") is blob, "the prepared weights were re-made by a table change"
    pe.set_pixel_lut(torch.arange(256).float())  # (256,): every channel
    assert torch.equal(pe.pixel_lut, torch.arange(256).float().expand(3, 256))
    with pytest.raises(ValueError):
        pe.set_pixel_lut(torch.zeros(4, 256))
    with pytest.raises(TypeError):
        pe(img8.permute(0, 3, 1, 2).contiguous())  # uint8 NCHW
    with pytest.raises(TypeError):
        pe(img8.to(torch.int16))


# ------------------------------------------------------------------------------------------------------------------------
# EarlyFusionFrontEnd
# ------------------------------------------------------------------------------------------------------------------------
def imagenet_lut():
    mean, std = torch.tensor([0.485, 0.456, 0.406]), torch.tensor([0.229, 0.224, 0.225])
    return (torch.arange(256).float().view(1, 256) / 255 - mean.view(3, 1)) / std.view(3, 1)


@pytest.mark.parametrize("prec", ["fp16", "bf16"])
def test_front_end_eval_u8_equals_expanded(cuda_device, prec):
    fe, _, _, _ = front_end(cuda_device, prec)
    fe.image_embed.set_pixel_lut(imagenet_lut())
    B = 3
    x_lid = to_nested(tiles_for(B), cuda_device)
    img8 = torch.randint(0, 256, (B, 224, 224, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(8)).to(cuda_device)
    x32 = expand(img8, fe.image_embed.pixel_lut)
    cls, pos = vit_params(9, device=cuda_device)
    le = fe.lidar_embed
    with torch.no_grad():
        pairs = [(fe(img8, x_lid), fe(x32, x_lid), "forward"),
                 (fe.forward_tokens(img8, x_lid, lidar_zero=False), fe.forward_tokens(x32, x_lid, lidar_zero=False), "forward_tokens"),
                 (fe.forward_tokens(img8, x_lid, lidar_zero=False, cls_token=cls, pos_embed=pos),
                  fe.forward_tokens(x32, x_lid, lidar_zero=False, cls_token=cls, pos_embed=pos), "forward_tokens cls / pos")]
        outs = [torch.empty(B, 2 * fe.channels, le.ny, le.nx, device=cuda_device) for _ in range(2)]
        pairs.append((fe.forward_into(img8, x_lid, outs[0], lidar_zero=True), fe.forward_into(x32, x_lid, outs[1], lidar_zero=True),
                      "forward_into"))
        x16 = [torch.empty(B, le.ny, le.nx, 2 * fe.channels, dtype=fe.fusion_layer.operand_dtype, device=cuda_device) for _ in range(2)]
        toks = [torch.empty(B, le.ny * le.nx, fe.channels, device=cuda_device) for _ in range(2)]
        pairs.append((fe.forward_tokens_into(img8, x_lid, x16[0], toks[0], lidar_zero=False),
                      fe.forward_tokens_into(x32, x_lid, x16[1], toks[1], lidar_zero=False), "forward_tokens_into"))
    torch.cuda.synchronize()
    for got, want, what in pairs:
        assert got.shape == want.shape, what
        assert torch.equal(got.view(torch.int32), want.view(torch.int32)), what
    assert torch.equal(x16[0].view(torch.int16), x16[1].view(torch.int16))


def test_front_end_train_u8_equals_expanded(cuda_device, monkeypatch):
    """Train mode: the uint8 image goes through the same table into a contiguous fp32 NCHW tensor and `image_embed.proj`.
    The image half (train-mode PatchEmbed, forward and backward) and the whole token route (fusion_layer with BatchNorm
    batch statistics, class token, pos_embed): output and the gradients of image_embed.proj are bit for bit those of the
    expanded fp32 image, cuDNN deterministic.  One LiDAR half, computed once, feeds both (the fused LiDAR training step sums
    with atomics)."""
    fe, _, _, _ = front_end(cuda_device, "fp16")
    fe.image_embed.set_pixel_lut(imagenet_lut())
    fe.train()
    B = 2
    x_lid = to_nested(tiles_for(B), cuda_device)
    img8 = torch.randint(0, 256, (B, 224, 224, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(10)).to(cuda_device)
    x32 = expand(img8, fe.image_embed.pixel_lut)
    cls, pos = (torch.nn.Parameter(t) for t in vit_params(11, device=cuda_device))
    gy = torch.randn(B, 1 + 784, 384, generator=torch.Generator().manual_seed(13)).to(cuda_device)
    gi = torch.randn(B, 384, 28, 28, generator=torch.Generator().manual_seed(14)).to(cuda_device)
    lidar_half = fe.lidar_embed(x_lid, return_flattened=False).detach()
    monkeypatch.setattr(fe, "forward", lambda x_image, x_lidar: torch.cat((fe.image_embed(x_image), lidar_half), dim=1))
    proj = fe.image_embed.proj

    def image_half(img):
        fe.zero_grad(set_to_none=True)
        y = fe.image_embed(img)
        (y * gi).sum().backward()
        return y.detach().clone(), proj.weight.grad.clone(), proj.bias.grad.clone()

    def token_route(img):
        fe.zero_grad(set_to_none=True)
        y = fe.forward_tokens(img, x_lid, cls_token=cls, pos_embed=pos)
        (y * gy).sum().backward()
        return y.detach().clone(), proj.weight.grad.clone(), proj.bias.grad.clone()

    deterministic, benchmark = torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = True, False
    try:
        half8, half32 = image_half(img8), image_half(x32)
        got, want = token_route(img8), token_route(x32)
    finally:
        torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = deterministic, benchmark
    assert fe.image_embed.expand_pixels(img8).is_contiguous()
    names = ("output", "proj.weight.grad", "proj.bias.grad")
    for a, b, what in zip(half8, half32, names):
        assert torch.count_nonzero(b) > 0, what
        assert torch.equal(a.view(torch.int32), b.view(torch.int32)), f"image half: {what}"
    for a, b, what in zip(got, want, names):
        assert torch.count_nonzero(b) > 0, what
        assert torch.equal(a.view(torch.int32), b.view(torch.int32)), f"token route: {what}: max |u8 - fp32| = {(a - b).abs().max().item():.3g}"


# ------------------------------------------------------------------------------------------------------------------------
# HostPipeline(image_dtype=torch.uint8)
# ------------------------------------------------------------------------------------------------------------------------
def run_pipeline(pipe, batches):
    done = []
    for batch, img in batches:
        fill(pipe, pipe.staging(), batch, img)
        prev = pipe.submit()
        if prev is not None:
            prev.done.synchronize()
            done.append(prev.out.clone())
    last = pipe.flush()
    last.done.synchronize()
    done.append(last.out.clone())
    return done


@pytest.mark.parametrize("mode, slots", [("concat", 2), ("tokens", 3), ("vit_tokens", 2)])
def test_pipeline_u8_equals_fp32_pipeline_and_direct_calls(cuda_device, mode, slots):
    from test_gpu_pipeline import B

    fe, _, _, _ = front_end(cuda_device, "fp16")
    fe.image_embed.set_pixel_lut(imagenet_lut())
    kw = {}
    if mode == "vit_tokens":
        cls, pos = vit_params(21, device=cuda_device)
        kw = dict(cls_token=cls, pos_embed=pos)
    p8 = HostPipeline(fe, B, TOTAL, slots=slots, mode=mode, image_dtype=torch.uint8, **kw)
    p32 = HostPipeline(fe, B, TOTAL, slots=slots, mode=mode, **kw)
    assert p8.slots[0].image.dtype == torch.uint8 and p8.slots[0].image.shape == (B, 224, 224, 3)
    assert p8.slots[0].image.is_pinned()
    img_bytes = B * 3 * 224 * 224

    def align(n):
        return (n + 255) // 256 * 256

    assert p32.h2d_bytes_per_step - p8.h2d_bytes_per_step == align(4 * img_bytes) - align(img_bytes)
    g = torch.Generator().manual_seed(22)
    imgs = [torch.randint(0, 256, (B, 224, 224, 3), dtype=torch.uint8, generator=g) for _ in range(6)]
    batches = [las_batch(40 + s) for s in range(6)]
    got = run_pipeline(p8, list(zip(batches, imgs)))
    want = run_pipeline(p32, [(b, expand(i, fe.image_embed.pixel_lut)) for b, i in zip(batches, imgs)])
    assert len(got) == len(want) == 6
    for i, (batch, img, a, b) in enumerate(zip(batches, imgs, got, want)):
        assert torch.equal(a.view(torch.int32), b.view(torch.int32)), f"batch {i}: uint8 and fp32 pipelines differ"
        x, img_d = direct_points(batch, cuda_device), img.to(cuda_device)
        with torch.no_grad():
            if mode == "concat":
                d = fe(img_d, x)
            elif mode == "tokens":
                d = fe.forward_tokens(img_d, x, lidar_zero=False)
            else:
                d = fe.forward_tokens(img_d, x, lidar_zero=False, **kw)
        assert torch.equal(a.view(torch.int32), d.view(torch.int32)), f"batch {i}: the pipeline differs from the direct call"
    # an in-place table update (set_pixel_lut) is seen by the captured graphs
    fe.image_embed.set_pixel_lut(default_pixel_lut(3))
    again = run_pipeline(p8, [(batches[0], imgs[0]), (batches[1], imgs[1])])
    with torch.no_grad():
        x, img_d = direct_points(batches[1], cuda_device), imgs[1].to(cuda_device)
        d = fe(img_d, x) if mode == "concat" else fe.forward_tokens(img_d, x, lidar_zero=False, **kw)
    assert torch.equal(again[1].view(torch.int32), d.view(torch.int32)), "the graphs did not read the updated table"
    assert not torch.equal(again[1], got[1])


def test_pipeline_refuses_other_image_dtypes(cuda_device):
    fe, _, _, _ = front_end(cuda_device, "fp16")
    with pytest.raises(ValueError, match="image_dtype"):
        HostPipeline(fe, 2, 1000, slots=2, mode="concat", image_dtype=torch.float16)


def test_oracle_patch_embed_agrees_on_the_default_table(cuda_device):
    """The default table is the fp32 image the CPU oracle consumes (u / 255): the uint8 route within the fp16 contract of it."""
    pe = PatchEmbed(embed_dim=384, precision="fp16").to(cuda_device).eval()
    _, sdi = po.synth_weights(2)
    pe.load_state_dict(sdi)
    img8 = torch.randint(0, 256, (1, 224, 224, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(3))
    ref = po.OraclePatchEmbed().eval()
    ref.load_state_dict(sdi)
    with torch.no_grad():
        want = ref(img8.permute(0, 3, 1, 2).float() / 255)
        got = pe(img8.to(cuda_device)).cpu()
    assert_close(got, want, TOL["fp16"], "uint8 patch embed, default table")
