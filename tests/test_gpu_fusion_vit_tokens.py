"""GPU tests of the early-fusion ViT input (p3p_conv3x3_vit_tokens, `EarlyFusionFrontEnd.forward_tokens(...,
cls_token=, pos_embed=)`, `HostPipeline(mode="vit_tokens")`): what `EarlyFusionViT.forward` hands the ViT blocks --
fusion_layer -> flatten / transpose -> timm `_pos_embed` (cat class token, + pos_embed; early_fusion_vit.py:96-125).

Checkers: the real torch modules on the CPU in fp32 (oracle front end -> fusion_layer -> flatten / transpose -> cat cls ->
+ pos), with the bars of test_gpu_fusion_layer.py; and, bit for bit, the token route without the class token followed by
the same fp32 add in torch (the epilogue adds pos_embed to the fp32 value that route stores)."""
import pytest
import torch
import torch.nn as nn

from oracle import pillars_oracle as po
from pixelspointspolygons_b200 import HostPipeline, default_cfg
from pixelspointspolygons_b200._lib import P3P_LAYOUT_NLC
from pixelspointspolygons_b200.fusion import ConvBnRelu3x3, EarlyFusionFrontEnd
from test_gpu_fusion_layer import TOL, torch_fusion_layer
from test_gpu_parity import assert_close, to_nested
from test_gpu_pipeline import TOTAL, direct_points, fill, las_batch

pytestmark = pytest.mark.gpu

FRONT_TOL = {"fp16": 2e-3, "bf16": 2e-2}  # two 16-bit roundings in series (activations, then the convolution's operands)
C, HW = 384, 784


def vit_params(seed, hw=HW, c=C, device="cpu"):
    g = torch.Generator().manual_seed(seed)
    cls = torch.randn(1, 1, c, generator=g) * 0.02
    pos = torch.randn(1, 1 + hw, c, generator=g) * 0.02
    return cls.to(device), pos.to(device)


def with_pos_embed(tokens, cls, pos):
    """timm `_pos_embed` on fp32 token rows (B, hw, C)."""
    B = tokens.shape[0]
    return torch.cat((cls.expand(B, -1, -1).to(tokens), tokens), dim=1) + pos.to(tokens)


def front_end(dev, prec, seed=3):
    cfg = default_cfg(device=str(dev), p3p_precision=prec)
    fe = EarlyFusionFrontEnd(cfg).eval()
    sd, sdi = po.synth_weights(seed)
    fe.lidar_embed.load_state_dict(sd)
    fe.image_embed.load_state_dict(sdi)
    ref_fl = torch_fusion_layer(768, 384, 9)
    fe.fusion_layer.load_state_dict(ref_fl.state_dict())
    return fe.to(dev), sd, sdi, ref_fl


def tiles_for(B):
    tiles = [po.synth_tile(20000 if i % 4 == 0 else 5000, 41 + i, clustered=(i % 2 == 1)) for i in range(B)]
    if B == 3:
        tiles[2] = po.synth_tile(0, 43)  # one empty tile
    return tiles


@pytest.mark.parametrize("prec", ["fp16", "bf16"])
@pytest.mark.parametrize("B", [1, 3, 16])
def test_fusion_vit_tokens_match_reference_modules(cuda_device, prec, B):
    fe, sd, sdi, ref_fl = front_end(cuda_device, prec)
    tiles = tiles_for(B)
    imgs = torch.rand(B, 3, 224, 224, generator=torch.Generator().manual_seed(2))
    cls, pos = vit_params(5)
    ref_enc = po.OraclePointPillarsEncoder(po.GridSpec()).eval()
    ref_enc.load_state_dict(sd)
    ref_pe = po.OraclePatchEmbed().eval()
    ref_pe.load_state_dict(sdi)
    x_img, x_lid = imgs.to(cuda_device), to_nested(tiles, cuda_device)
    cls_d, pos_d = cls.to(cuda_device), pos.to(cuda_device)
    for lidar_zero in (False, True):
        with torch.no_grad():
            concat = po.early_fusion_front(ref_pe, ref_enc, imgs, tiles, apply_lidar_dropout=lidar_zero)
            want = with_pos_embed(ref_fl(concat).flatten(2).transpose(1, 2), cls, pos)
            got = fe.forward_tokens(x_img, x_lid, lidar_zero=lidar_zero, cls_token=cls_d, pos_embed=pos_d)
            plain = fe.forward_tokens(x_img, x_lid, lidar_zero=lidar_zero)
        torch.cuda.synchronize()
        what = f"fusion ViT tokens B={B} {prec} lidar_zero={lidar_zero}"
        assert got.shape == (B, 1 + HW, C) and got.dtype == torch.float32
        assert_close(got, want, FRONT_TOL[prec], what)
        # row 0: cls_token + pos_embed[0] in fp32, bit for bit
        assert torch.equal(got[:, 0], (cls_d[0, 0] + pos_d[0, 0]).expand(B, -1)), what
        # rows 1..: the token route without the class token, + pos_embed in torch, bit for bit
        assert torch.equal(got[:, 1:], plain + pos_d[:, 1:]), what


def test_vit_params_are_converted_and_checked(cuda_device):
    fe, _, _, _ = front_end(cuda_device, "fp16")
    tiles = tiles_for(2)
    x_img = torch.rand(2, 3, 224, 224, generator=torch.Generator().manual_seed(4)).to(cuda_device)
    x_lid = to_nested(tiles, cuda_device)
    cls, pos = vit_params(6, device=cuda_device)
    with torch.no_grad():
        want = fe.forward_tokens(x_img, x_lid, lidar_zero=False, cls_token=cls, pos_embed=pos)
        # float64 on the host: converted to fp32 on the device, as PointPillarsEncoder.forward_tokens does
        got = fe.forward_tokens(x_img, x_lid, lidar_zero=False, cls_token=cls.double().cpu(), pos_embed=pos.double().cpu())
        assert torch.equal(got, want)
        with pytest.raises(ValueError, match="both or neither"):
            fe.forward_tokens(x_img, x_lid, cls_token=cls)
        with pytest.raises(ValueError, match="both or neither"):
            fe.forward_tokens(x_img, x_lid, pos_embed=pos)
        with pytest.raises(ValueError, match="pos_embed"):
            fe.forward_tokens(x_img, x_lid, cls_token=cls, pos_embed=pos[:, 1:])


@pytest.mark.parametrize("prec", ["fp16", "bf16"])
@pytest.mark.parametrize("shape", [(2, 768, 384, 28, 28), (1, 128, 200, 12, 20), (3, 64, 64, 8, 16),
                                   (2, 128, 384, 30, 28), (2, 64, 96, 13, 20)])
def test_conv_vit_tokens_matches_torch(cuda_device, prec, shape):
    """The convolution alone.  28 x 28 / 384: 7 strips of 4 rows; 30 x 28: the last of 8 strips ends mid-image; 13 x 20: a
    12-row strip and a 1-row one; 12 x 20 and 8 x 16: one strip per image.  The class-token row of every image comes from
    its strip-0 CTA."""
    B, cin, cout, H, W = shape
    ref = torch_fusion_layer(cin, cout, 5)
    mod = ConvBnRelu3x3(cin, cout, precision=prec).eval()
    mod.load_state_dict(ref.state_dict())
    mod = mod.to(cuda_device)
    x = torch.randn(B, cin, H, W, generator=torch.Generator().manual_seed(1))
    x[:, :, 0, :] += 2.0
    cls, pos = vit_params(7, H * W, cout)
    cls_d, pos_d = cls.to(cuda_device).reshape(-1), pos.to(cuda_device).reshape(-1)
    x16 = x.to(cuda_device).permute(0, 2, 3, 1).contiguous().to(mod.operand_dtype)
    got = torch.full((B, 1 + H * W, cout), float("nan"), device=cuda_device)
    plain = torch.empty(B, H * W, cout, device=cuda_device)
    with torch.no_grad():
        want = with_pos_embed(ref(x).flatten(2).transpose(1, 2), cls, pos)
        mod._runner.run_vit_tokens(x16, cls_d, pos_d, got)
        mod.forward_nhwc(x16, plain, P3P_LAYOUT_NLC)
    torch.cuda.synchronize()
    assert_close(got, want, TOL[prec], f"conv3x3 ViT tokens {shape} {prec}")  # (NaN left anywhere fails here)
    assert torch.equal(got[:, 0], (cls_d + pos_d[:cout]).expand(B, -1))
    assert torch.equal(got[:, 1:], plain + pos_d.view(1 + H * W, cout)[1:])


def test_two_lanes_in_flight_equal_the_serial_result(cuda_device):
    fe, _, _, _ = front_end(cuda_device, "fp16")
    cls, pos = vit_params(8, device=cuda_device)
    g = torch.Generator().manual_seed(9)
    batches = [(torch.rand(4, 3, 224, 224, generator=g).to(cuda_device), to_nested(tiles_for(4)[::-1] if i % 2 else tiles_for(4), cuda_device))
               for i in range(4)]
    with torch.no_grad():
        want = [fe.forward_tokens(img, x, lidar_zero=bool(i == 3), cls_token=cls, pos_embed=pos).clone() for i, (img, x) in enumerate(batches)]
    torch.cuda.synchronize()
    le = fe.lidar_embed
    streams = [torch.cuda.Stream(cuda_device), torch.cuda.Stream(cuda_device)]
    x16 = [torch.empty(4, le.ny, le.nx, 2 * C, dtype=fe.fusion_layer.operand_dtype, device=cuda_device) for _ in range(4)]
    outs = [torch.empty_like(w) for w in want]
    with torch.no_grad():
        for rep in range(3):
            for i, (img, x) in enumerate(batches):
                with torch.cuda.stream(streams[i % 2]):
                    fe.forward_tokens_into(img, x, x16[i], outs[i], lidar_zero=bool(i == 3), lane=i % 2, cls_token=cls, pos_embed=pos)
    torch.cuda.synchronize()
    for o, w in zip(outs, want):
        assert torch.equal(o, w)


def test_host_pipeline_vit_tokens_mode(cuda_device):
    B = 4
    fe, _, _, _ = front_end(cuda_device, "fp16")
    cls, pos = (nn.Parameter(t) for t in vit_params(10, device=cuda_device))
    pipe = HostPipeline(fe, B, TOTAL, slots=2, mode="vit_tokens", cls_token=cls, pos_embed=pos, host_result="full")
    g = torch.Generator().manual_seed(5)
    batches = [(las_batch(20 + s), torch.rand(B, 3, 224, 224, generator=g)) for s in range(5)]

    def run(some):
        done = []
        for batch, img in some:
            fill(pipe, pipe.staging(), batch, img)
            prev = pipe.submit()
            if prev is not None:
                prev.done.synchronize()
                done.append(prev.out.clone())
        last = pipe.flush()
        last.host_done.synchronize()
        done.append(last.out.clone())
        assert torch.equal(last.host_out, last.out.cpu())
        return done

    def direct(some):
        with torch.no_grad():
            return [fe.forward_tokens(img.to(cuda_device), direct_points(batch, cuda_device), lidar_zero=False, cls_token=cls,
                                      pos_embed=pos) for batch, img in some]

    first = run(batches[:3])
    for out, want in zip(first, direct(batches[:3])):
        assert out.shape == (B, 1 + HW, C)
        assert torch.equal(out, want)
    # an in-place update of the parameters (what an optimizer step does) is seen by the next replay
    torch.cuda.synchronize()
    with torch.no_grad():
        pos.mul_(-2.0).add_(0.5)
        cls.add_(1.0)
    torch.cuda.synchronize()
    second = run(batches[3:])
    for out, want in zip(second, direct(batches[3:])):
        assert torch.equal(out, want)
        assert torch.equal(out[:, 0], (cls[0, 0] + pos[0, 0]).detach().expand(B, -1))
    with pytest.raises(ValueError, match="cls_token and pos_embed"):
        HostPipeline(fe, B, TOTAL, slots=2, mode="vit_tokens")
    with pytest.raises(ValueError, match="vit_tokens"):
        HostPipeline(fe, B, TOTAL, slots=2, mode="tokens", cls_token=cls, pos_embed=pos)
    with pytest.raises(TypeError, match="float32"):
        HostPipeline(fe, B, TOTAL, slots=2, mode="vit_tokens", cls_token=cls.detach().half(), pos_embed=pos)


def test_train_mode_matches_reference_expression(cuda_device, monkeypatch):
    """Train mode: the torch route + `torch.cat` + add.  Output and gradients equal those of the reference's expression on
    the same module and the same input.  The fused LiDAR training step sums its batch moments with atomics, so two passes
    through it differ in the last bits (amplified by the BatchNorm batch statistics downstream): both expressions are fed
    one LiDAR half, computed once, next to the live image half; cuDNN in deterministic mode for both.  A separate pass
    through the whole train route checks that every parameter it reaches gets a gradient."""
    fe, _, _, _ = front_end(cuda_device, "fp16")
    fe.train()
    B = 2
    tiles = tiles_for(B)
    imgs = torch.rand(B, 3, 224, 224, generator=torch.Generator().manual_seed(12)).to(cuda_device)
    x_lid = to_nested(tiles, cuda_device)
    cls, pos = (nn.Parameter(t) for t in vit_params(11, device=cuda_device))
    gy = torch.randn(B, 1 + HW, C, generator=torch.Generator().manual_seed(13)).to(cuda_device)
    names = [n for n, _ in fe.named_parameters() if n.startswith(("fusion_layer.", "image_embed."))]
    assert names

    def step(fn):
        fe.zero_grad(set_to_none=True)
        cls.grad = pos.grad = None
        y = fn()
        (y * gy).sum().backward()
        grads = {n: p.grad.clone() for n, p in fe.named_parameters() if p.grad is not None}
        return y.detach().clone(), cls.grad.clone(), pos.grad.clone(), grads

    # the whole train route: gradients reach cls_token, pos_embed and every parameter of the three submodules
    whole = step(lambda: fe.forward_tokens(imgs, x_lid, cls_token=cls, pos_embed=pos))
    assert whole[0].shape == (B, 1 + HW, C)
    assert torch.count_nonzero(whole[1]) > 0 and torch.count_nonzero(whole[2]) > 0
    for n, p in fe.named_parameters():
        assert n in whole[3] and torch.isfinite(whole[3][n]).all(), n
        # (the conv bias ahead of a BatchNorm in batch-statistics mode has a zero gradient up to rounding)
        assert n == "fusion_layer.0.bias" or torch.count_nonzero(whole[3][n]) > 0, n

    lidar_half = fe.lidar_embed(x_lid, return_flattened=False).detach()
    monkeypatch.setattr(fe, "forward", lambda x_image, x_lidar: torch.cat((fe.image_embed(x_image), lidar_half), dim=1))

    def reference():
        x = fe(imgs, x_lid)
        x = fe.fusion_layer(x).flatten(2).transpose(1, 2)
        return torch.cat((cls.expand(x.shape[0], -1, -1), x), dim=1) + pos

    deterministic, benchmark = torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = True, False
    try:
        got = step(lambda: fe.forward_tokens(imgs, x_lid, cls_token=cls, pos_embed=pos))
        want = step(reference)
    finally:
        torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = deterministic, benchmark
    for a, b, what in ((got[0], want[0], "output"), (got[1], want[1], "cls_token.grad"), (got[2], want[2], "pos_embed.grad")):
        torch.testing.assert_close(a, b, rtol=1e-5, atol=1e-6 * b.abs().max().item(), msg=what)
    scale = max(want[3][n].abs().max().item() for n in names)
    for n in names:
        assert n in got[3], n
        torch.testing.assert_close(got[3][n], want[3][n], rtol=1e-5, atol=1e-6 * scale, msg=n)


def test_without_vit_params_forward_tokens_is_the_parent_route(cuda_device):
    """No cls_token / pos_embed: the output is bit for bit the three-kernel route of the token rows (image half, LiDAR half,
    p3p_conv3x3 into (B, ny nx, C)), issued here by hand."""
    for prec in ("fp16", "bf16"):
        fe, _, _, _ = front_end(cuda_device, prec)
        tiles = tiles_for(3)
        imgs = torch.rand(3, 3, 224, 224, generator=torch.Generator().manual_seed(14)).to(cuda_device)
        x_lid = to_nested(tiles, cuda_device)
        le, fl = fe.lidar_embed, fe.fusion_layer
        with torch.no_grad():
            got = fe.forward_tokens(imgs, x_lid, lidar_zero=False)
            x16 = torch.empty(3, le.ny, le.nx, 2 * C, dtype=fl.operand_dtype, device=cuda_device)
            fe.image_embed.forward_into(imgs, x16, 2 * C, 0, layout=P3P_LAYOUT_NLC)
            le.encode_into(x_lid, x16, P3P_LAYOUT_NLC, c_total=2 * C, c_offset=C, lidar_zero=False)
            want = fl.forward_nhwc(x16, torch.empty(3, HW, C, device=cuda_device), P3P_LAYOUT_NLC)
        torch.cuda.synchronize()
        assert got.shape == (3, HW, C)
        assert torch.equal(got, want), prec
