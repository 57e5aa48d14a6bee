"""Early-fusion front end: image patch embedding + LiDAR pillar encoder -> one (B, 2C, ny, nx) concat buffer.

Mirrors the part of the reference's fusion encoders that is on the hot path
(R:pixelspointspolygons/models/fusion_layers/early_fusion_vit.py:43-52,69-72,96-121 and
early_fusion_vit_cnn.py:41-50,67-70,90-92):

    x_image = self.image_embed(x_image)                          # timm PatchEmbed, flatten=False -> (B, C, ny, nx)
    x_lidar = self.lidar_embed(x_lidar, return_flattened=False)  # PointPillarsEncoder          -> (B, C, ny, nx)
    if cfg.experiment.lidar_dropout is not None and rand <= p:  x_lidar = x_lidar * 0.0
    x = torch.cat((x_image, x_lidar), dim=1)                     # image channels first

Submodule and parameter names are the reference's (`image_embed.proj.{weight,bias}`,
`lidar_embed.voxel_encoder.pfn_layers.*`; SURVEY Appendix C), so a checkpoint's `encoder.image_embed.*` /
`encoder.lidar_embed.*` entries load unchanged.  In eval mode both halves are written by libp3p.so kernels directly
into the concat buffer (no intermediate tensors, no cat copy); everything after the concat (`fusion_layer`, the
ViT) is outside this package (SURVEY 8f).
"""
from __future__ import annotations

import ctypes as C
import logging
from typing import Optional

import torch
import torch.nn as nn

from . import _lib
from ._lib import P3P_LAYOUT_NCHW, P3P_LAYOUT_NLC, P3P_PRECISION
from .encoder import PointPillarsEncoder, _get, _out_dtype_code


def default_pixel_lut(in_chans: int = 3) -> torch.Tensor:
    """(in_chans, 256) fp32: byte u -> u / 255 in every channel, torchvision's `ToTensor` arithmetic -- with the reference's
    `image_mean 0, std 1` (config/encoder/early_fusion_vit.yaml:48-50) the whole of its normalisation."""
    return torch.arange(256, dtype=torch.float32).div(255).expand(int(in_chans), 256).contiguous()


class PatchEmbed(nn.Module):
    """timm.layers.PatchEmbed as the reference uses it (`flatten = False`, norm = Identity, NCHW output).

    Besides the fp32 NCHW image (B, in_chans, H, W) the module takes the decoded image as the loader holds it before its
    normalisation: uint8 channels-last (B, H, W, in_chans), in_chans <= 4.  A pixel table maps every byte to the value the
    loader's normalisation would give it (`set_pixel_lut`; default `default_pixel_lut`), and the kernel applies it while it
    builds its operand, so the result is the one of the fp32 image expanded through the table, bit for bit.  The table is
    neither a parameter nor a buffer (state_dict keys stay timm's); each device keeps one copy, updated in place."""

    def __init__(self, img_size=224, patch_size=8, in_chans=3, embed_dim=384, bias=True, precision: str = "fp16"):
        super().__init__()
        self.img_size, self.patch_size, self.in_chans, self.embed_dim = int(img_size), int(patch_size), int(in_chans), int(embed_dim)
        self.flatten = False
        self.proj = nn.Conv2d(in_chans, embed_dim, kernel_size=patch_size, stride=patch_size, bias=bias)
        self.norm = nn.Identity()
        self.precision = precision
        self._blobs = {}  # (device, precision) -> (parameter stamp, prepared weights)
        self._pixel_lut = default_pixel_lut(self.in_chans)  # host copy of the table
        self._luts = {}   # device -> (in_chans, 256) fp32 copy the kernels read

    @property
    def pixel_lut(self) -> torch.Tensor:
        """The pixel table (in_chans, 256) fp32 of the uint8 route (a copy on the CPU)."""
        return self._pixel_lut.clone()

    def set_pixel_lut(self, lut) -> None:
        """Install the table `lut[c][u]` = the value the loader's normalisation gives byte u of channel c: (in_chans, 256),
        or (256,) for every channel.  Takes effect on the next call; the device copies are updated in place, so CUDA graphs
        that captured this module (HostPipeline) read the new table too."""
        t = torch.as_tensor(lut).detach().to(device="cpu", dtype=torch.float32)
        if t.shape == (256,):
            t = t.expand(self.in_chans, 256)
        if t.shape != (self.in_chans, 256):
            raise ValueError(f"the pixel table must be ({self.in_chans}, 256) or (256,), got {tuple(t.shape)}")
        self._pixel_lut = t.contiguous().clone()
        for dev, d in self._luts.items():
            with torch.cuda.device(dev):
                d.copy_(self._pixel_lut)
                torch.cuda.current_stream(dev).synchronize()  # in place before any stream's next kernel reads it

    def _lut(self, device) -> torch.Tensor:
        d = self._luts.get(device)
        if d is None:
            d = self._luts[device] = self._pixel_lut.to(device)
        return d

    def expand_pixels(self, x: torch.Tensor) -> torch.Tensor:
        """uint8 (B, H, W, in_chans) -> the fp32 (B, in_chans, H, W) image it stands for: lut[c][x[b, y, x, c]]."""
        if x.dtype != torch.uint8 or x.dim() != 4 or x.shape[3] != self.in_chans:
            raise TypeError(f"x_image must be uint8 (B, H, W, {self.in_chans})")
        lut = self._lut(x.device) if x.is_cuda else self._pixel_lut
        idx = x.permute(0, 3, 1, 2).long() + 256 * torch.arange(self.in_chans, device=x.device).view(1, -1, 1, 1)
        # (the gather keeps the index's channels-last strides; a contiguous NCHW tensor, as the loader's ToTensorV2 + collate
        # give, makes cuDNN pick the same convolution algorithms as for the fp32 image)
        return lut.reshape(-1)[idx].contiguous()

    def _blob(self, device, precision: str) -> torch.Tensor:
        """The weights as tensor-core operand tiles (p3p_patch_embed_prepare), re-made when a parameter changes."""
        tensors = [self.proj.weight, self.proj.bias]
        stamp = tuple((t._version, t.data_ptr()) if t is not None else None for t in tensors)
        hit = self._blobs.get((device, precision))
        if hit is not None and hit[0] == stamp:
            return hit[1]
        w = self.proj.weight.detach().contiguous()
        b = self.proj.bias.detach().contiguous() if self.proj.bias is not None else None
        nbytes = _lib.lib().p3p_patch_embed_blob_bytes(self.embed_dim, self.in_chans, self.patch_size)
        blob = torch.empty(nbytes, dtype=torch.uint8, device=device)
        with torch.cuda.device(device):
            _lib.check(_lib.lib().p3p_patch_embed_prepare(w.data_ptr(), b.data_ptr() if b is not None else None, self.embed_dim,
                                                          self.in_chans, self.patch_size, P3P_PRECISION[precision], blob.data_ptr(),
                                                          nbytes, torch.cuda.current_stream(device).cuda_stream),
                       "p3p_patch_embed_prepare")
        self._blobs[(device, precision)] = (stamp, blob)
        return blob

    def _image_hw(self, x: torch.Tensor):
        """(B, H, W) of an fp32 NCHW or a uint8 NHWC image; anything else is a TypeError."""
        if x.dim() == 4 and x.dtype == torch.float32 and x.shape[1] == self.in_chans:
            return x.shape[0], x.shape[2], x.shape[3]
        if x.dim() == 4 and x.dtype == torch.uint8 and x.shape[3] == self.in_chans:
            return x.shape[0], x.shape[1], x.shape[2]
        raise TypeError(f"x_image must be float32 (B, {self.in_chans}, H, W) or uint8 (B, H, W, {self.in_chans})")

    def forward_into(self, x: torch.Tensor, out: torch.Tensor, c_total: int, c_offset: int, precision: Optional[str] = None,
                     layout: int = P3P_LAYOUT_NCHW):
        """Conv2d(P x P / P) of `x` into channels [c_offset, c_offset + C) of `out`: NCHW (B, c_total, H/P, W/P) or
        channels-last rows (B, H/P * W/P, c_total); fp32, bf16 or fp16.  x: fp32 (B, in_chans, H, W), or uint8
        (B, H, W, in_chans) mapped through the pixel table."""
        if not x.is_cuda:
            raise RuntimeError("PatchEmbed runs on CUDA only (sm_100a); x_image is on " + str(x.device))
        B, H, W = self._image_hw(x)
        x = x.contiguous()
        w = self.proj.weight.detach().contiguous()
        b = self.proj.bias.detach().contiguous() if self.proj.bias is not None else None
        dt = _out_dtype_code(out)
        need = B * (H // self.patch_size) * (W // self.patch_size) * c_total
        if out.device != x.device or not out.is_contiguous() or out.numel() < need:
            raise ValueError(f"out must be a contiguous tensor of at least {need} elements on {x.device}")
        precision = precision or self.precision
        if w.device != x.device or w.dtype != torch.float32:
            raise RuntimeError("PatchEmbed parameters must be float32 on the device of x_image")
        with torch.cuda.device(x.device):
            blob = self._blob(x.device, precision)
            st = torch.cuda.current_stream(x.device).cuda_stream
            if x.dtype == torch.uint8:
                rc = _lib.lib().p3p_patch_embed_u8(x.data_ptr(), self._lut(x.device).data_ptr(), B, self.in_chans, H, W,
                                                   self.patch_size, blob.data_ptr(), w.data_ptr(),
                                                   b.data_ptr() if b is not None else None, self.embed_dim, P3P_PRECISION[precision],
                                                   out.data_ptr(), dt, layout, c_total, c_offset, st)
                _lib.check(rc, "p3p_patch_embed_u8")
                return out
            rc = _lib.lib().p3p_patch_embed_prepared(x.data_ptr(), B, self.in_chans, H, W, self.patch_size, blob.data_ptr(),
                                                     w.data_ptr(), b.data_ptr() if b is not None else None, self.embed_dim,
                                                     P3P_PRECISION[precision], out.data_ptr(), dt, layout, c_total, c_offset, st)
        _lib.check(rc, "p3p_patch_embed_prepared")
        return out

    def forward(self, x):
        if self.training and torch.is_grad_enabled():
            if x.dtype == torch.uint8:  # the same table, then the autograd route
                x = self.expand_pixels(x)
            y = self.proj(x)  # autograd route of the optional training step
        else:
            B, H, W = self._image_hw(x) if x.dtype == torch.uint8 else (x.shape[0], x.shape[2], x.shape[3])
            y = torch.empty(B, self.embed_dim, H // self.patch_size, W // self.patch_size, dtype=torch.float32, device=x.device)
            self.forward_into(x, y, self.embed_dim, 0)
        if self.flatten:
            y = y.flatten(2).transpose(1, 2)
        return self.norm(y)


class _Conv3x3Runner:
    """Kernel side of a Conv2d(3x3, padding 1) + eval-mode BatchNorm2d + ReLU triple whose torch modules live elsewhere:
    prepared-weights blob per device (re-made when a parameter changes) and the call into libp3p.so."""

    def __init__(self, conv: nn.Conv2d, bn: nn.BatchNorm2d, precision: str):
        if conv.kernel_size != (3, 3) or conv.padding != (1, 1) or conv.stride != (1, 1) or conv.groups != 1:
            raise NotImplementedError("the kernel implements Conv2d(kernel_size=3, padding=1, stride=1, groups=1)")
        self.conv, self.bn = conv, bn
        self.in_channels, self.out_channels = conv.in_channels, conv.out_channels
        self.precision = "bf16" if precision == "bf16" else "fp16"  # operand type of the kernel (fp32 accumulate)
        self._blobs = {}

    @property
    def operand_dtype(self) -> torch.dtype:
        return torch.bfloat16 if self.precision == "bf16" else torch.float16

    def _tensors(self):
        return [self.conv.weight, self.conv.bias, self.bn.weight, self.bn.bias, self.bn.running_mean, self.bn.running_var]

    def blob(self, device) -> torch.Tensor:
        tensors = self._tensors()
        stamp = tuple((t._version, t.data_ptr()) if t is not None else None for t in tensors) + (self.precision,)
        hit = self._blobs.get(device)
        if hit is not None and hit[0] == stamp:
            return hit[1]
        keep = [t.detach().to(device=device, dtype=torch.float32).contiguous() if t is not None else None for t in tensors]
        p = _lib.ConvParams()
        for name, t in zip(("weight", "bias", "norm_weight", "norm_bias", "norm_mean", "norm_var"), keep):
            setattr(p, name, t.data_ptr() if t is not None else None)
        p.eps, p.in_channels, p.out_channels = float(self.bn.eps), self.in_channels, self.out_channels
        nbytes = _lib.lib().p3p_conv3x3_blob_bytes(self.in_channels, self.out_channels)
        blob = torch.empty(nbytes, dtype=torch.uint8, device=device)
        with torch.cuda.device(device):
            _lib.check(_lib.lib().p3p_conv3x3_prepare(C.byref(p), P3P_PRECISION[self.precision], blob.data_ptr(), nbytes,
                                                      torch.cuda.current_stream(device).cuda_stream), "p3p_conv3x3_prepare")
        self._blobs[device] = (stamp, blob)
        return blob

    def run(self, x16: torch.Tensor, out: torch.Tensor, layout: int, c_total: Optional[int] = None, c_offset: int = 0):
        """x16: (B, H, W, Cin) 16-bit channels-last (operand_dtype) -> out fp32: token rows (B, H W, c_total) or NCHW."""
        if x16.dtype != self.operand_dtype or x16.dim() != 4 or x16.shape[3] != self.in_channels or not x16.is_contiguous():
            raise TypeError(f"x must be a contiguous {self.operand_dtype} tensor (B, H, W, {self.in_channels})")
        if not x16.is_cuda:
            raise RuntimeError("the 3x3 convolution kernel runs on CUDA only (sm_100a); x is on " + str(x16.device))
        B, H, W, _ = x16.shape
        c_total = self.out_channels if c_total is None else int(c_total)
        if out.dtype != torch.float32 or not out.is_contiguous() or out.device != x16.device or out.numel() < B * H * W * c_total:
            raise ValueError("out must be a contiguous float32 tensor of B * H * W * c_total elements on the device of x")
        with torch.cuda.device(x16.device):
            blob = self.blob(x16.device)
            rc = _lib.lib().p3p_conv3x3(x16.data_ptr(), B, H, W, self.in_channels, blob.data_ptr(), self.out_channels,
                                        P3P_PRECISION[self.precision], 1, out.data_ptr(), layout, c_total, c_offset,
                                        torch.cuda.current_stream(x16.device).cuda_stream)
        _lib.check(rc, "p3p_conv3x3")
        return out

    def run_vit_tokens(self, x16: torch.Tensor, cls_token: torch.Tensor, pos_embed: torch.Tensor, out: torch.Tensor):
        """x16 as in `run` -> out (B, 1 + H W, Cout) fp32, the ViT input (p3p_conv3x3_vit_tokens): row 0 of every image
        cls_token + pos_embed[0], row 1 + pos the convolution + BN + ReLU at pos + pos_embed[1 + pos].  cls_token (Cout) and
        pos_embed ((1 + H W) Cout values) are contiguous float32 on the device of x; the kernel reads them in place."""
        if x16.dtype != self.operand_dtype or x16.dim() != 4 or x16.shape[3] != self.in_channels or not x16.is_contiguous():
            raise TypeError(f"x must be a contiguous {self.operand_dtype} tensor (B, H, W, {self.in_channels})")
        if not x16.is_cuda:
            raise RuntimeError("the 3x3 convolution kernel runs on CUDA only (sm_100a); x is on " + str(x16.device))
        B, H, W, _ = x16.shape
        Cc, rows = self.out_channels, H * W + 1
        for name, t, n in (("cls_token", cls_token, Cc), ("pos_embed", pos_embed, rows * Cc)):
            if t.dtype != torch.float32 or not t.is_contiguous() or t.device != x16.device or t.numel() != n:
                raise ValueError(f"{name} must be a contiguous float32 tensor of {n} elements on the device of x")
        if out.dtype != torch.float32 or not out.is_contiguous() or out.device != x16.device or out.numel() < B * rows * Cc:
            raise ValueError("out must be a contiguous float32 tensor of B * (1 + H * W) * Cout elements on the device of x")
        with torch.cuda.device(x16.device):
            blob = self.blob(x16.device)
            rc = _lib.lib().p3p_conv3x3_vit_tokens(x16.data_ptr(), B, H, W, self.in_channels, blob.data_ptr(), Cc,
                                                   P3P_PRECISION[self.precision], cls_token.data_ptr(), pos_embed.data_ptr(),
                                                   out.data_ptr(), torch.cuda.current_stream(x16.device).cuda_stream)
        _lib.check(rc, "p3p_conv3x3_vit_tokens")
        return out


class ConvBnRelu3x3(nn.Sequential):
    """`nn.Sequential(nn.Conv2d(cin, cout, kernel_size=3, padding=1), nn.BatchNorm2d(cout), nn.ReLU(inplace=True))` -- the
    reference's `fusion_layer` (early_fusion_vit.py:75-79, early_fusion_vit_cnn.py:72-76) -- with the same child indices,
    hence the same state_dict keys (`0.weight`, `0.bias`, `1.weight`, `1.running_mean`, ...).  In eval mode the three run as
    one implicit-GEMM tensor-core kernel on 16-bit channels-last input (csrc/conv3x3.cu); train mode takes the torch modules
    (the optional training step)."""

    def __init__(self, in_channels: int, out_channels: int, precision: str = "fp16"):
        super().__init__(nn.Conv2d(in_channels, out_channels, kernel_size=3, padding=1), nn.BatchNorm2d(out_channels),
                         nn.ReLU(inplace=True))
        self._runner = _Conv3x3Runner(self[0], self[1], precision)

    @property
    def operand_dtype(self) -> torch.dtype:
        return self._runner.operand_dtype

    def forward_nhwc(self, x16, out, layout, c_total=None, c_offset=0):
        return self._runner.run(x16, out, layout, c_total, c_offset)

    def forward(self, x):
        """Drop-in for the reference's call `self.fusion_layer(x)`: x (B, Cin, H, W) fp32 -> (B, Cout, H, W) fp32."""
        if self.training:
            return super().forward(x)
        r = self._runner
        B, Cin, H, W = x.shape
        x = x.contiguous()
        x16 = torch.empty(B, H, W, Cin, dtype=r.operand_dtype, device=x.device)
        with torch.cuda.device(x.device):
            rc = _lib.lib().p3p_nchw_to_nhwc16(x.data_ptr(), B, Cin, H, W, P3P_PRECISION[r.precision], x16.data_ptr(), Cin, 0,
                                               torch.cuda.current_stream(x.device).cuda_stream)
        _lib.check(rc, "p3p_nchw_to_nhwc16")
        out = torch.empty(B, r.out_channels, H, W, dtype=torch.float32, device=x.device)
        return r.run(x16, out, P3P_LAYOUT_NCHW)


class ProjTail(nn.Sequential):
    """The reference's `proj` (pointpillars_vit_cnn.py:20-25, early_fusion_vit_cnn.py:78-83):
    `nn.Sequential(nn.Upsample(size, mode='bilinear', align_corners=False), nn.Conv2d(cin, cout, 3, padding=1),
    nn.BatchNorm2d(cout), nn.ReLU(inplace=True))`, same child indices (`1.weight`, `2.running_mean`, ...).  Eval mode:
    a bilinear-upsampling kernel that reads the ViT tokens in place and writes 16-bit channels-last, then the implicit-GEMM
    convolution kernel."""

    def __init__(self, in_channels: int, out_channels: int, size, precision: str = "fp16"):
        size = (int(size), int(size)) if isinstance(size, int) else (int(size[0]), int(size[1]))
        super().__init__(nn.Upsample(size=size, mode="bilinear", align_corners=False),
                         nn.Conv2d(in_channels, out_channels, kernel_size=3, padding=1), nn.BatchNorm2d(out_channels),
                         nn.ReLU(inplace=True))
        self.size = size
        self._runner = _Conv3x3Runner(self[1], self[2], precision)

    def forward_tokens(self, tokens: torch.Tensor, h: int, w: int, skip_rows: int = 0):
        """tokens: (B, skip_rows + h w, C) fp32 (the ViT output; skip_rows = 1 drops the class token in place, as
        `x[:, 1:, :]` + permute + view do in the reference) -> (B, Cout, H, W) fp32."""
        if self.training:
            B, _, Cc = tokens.shape
            x = tokens[:, skip_rows:, :].permute(0, 2, 1).reshape(B, Cc, h, w)
            return super().forward(x)
        if not tokens.is_cuda or tokens.dtype != torch.float32:
            raise TypeError("tokens must be a float32 CUDA tensor")
        tokens = tokens.contiguous()
        B, rows, Cc = tokens.shape
        H, W = self.size
        r = self._runner
        x16 = torch.empty(B, H, W, Cc, dtype=r.operand_dtype, device=tokens.device)
        src = tokens.view(-1)[skip_rows * Cc:]
        with torch.cuda.device(tokens.device):
            rc = _lib.lib().p3p_upsample_bilinear_nhwc16(src.data_ptr(), B, h, w, Cc, rows * Cc, H, W, P3P_PRECISION[r.precision],
                                                         x16.data_ptr(), torch.cuda.current_stream(tokens.device).cuda_stream)
        _lib.check(rc, "p3p_upsample_bilinear_nhwc16")
        out = torch.empty(B, r.out_channels, H, W, dtype=torch.float32, device=tokens.device)
        return r.run(x16, out, P3P_LAYOUT_NCHW)

    def forward(self, x):
        """Drop-in for `self.proj(x)`: x (B, C, h, w) fp32 -> (B, Cout, H, W) fp32."""
        if self.training:
            return super().forward(x)
        B, Cc, h, w = x.shape
        tokens = x.flatten(2).transpose(1, 2).contiguous()  # (B, h w, C)
        return self.forward_tokens(tokens, h, w)


class EarlyFusionFrontEnd(nn.Module):
    """`EarlyFusionViT.forward` / `EarlyFusionViTCNN.forward` up to and including the concat."""

    def __init__(self, cfg, local_rank: int = 0):
        super().__init__()
        self.cfg = cfg
        self.local_rank = local_rank
        verbosity = getattr(logging, str(_get(_get(cfg, "run_type"), "logging", "INFO")).upper(), logging.INFO)
        self.logger = logging.getLogger(f"{self.__class__.__name__}[{local_rank}]")
        self.logger.setLevel(verbosity)
        enc = cfg.experiment.encoder
        dim = int(enc.patch_feature_dim)
        # early_fusion_vit.py:43-52
        output_shape = [int(enc.patch_feature_width), int(enc.patch_feature_height)]
        self.lidar_embed = PointPillarsEncoder(cfg, voxel_encoder={"in_channels": 3, "feat_channels": [64, dim]},
                                               scatter={"in_channels": dim, "output_shape": output_shape}, local_rank=local_rank)
        # early_fusion_vit.py:69-70: the ViT's own PatchEmbed, re-parented, flatten switched off
        self.image_embed = PatchEmbed(img_size=int(_get(enc, "in_size", enc.in_height)), patch_size=int(_get(enc, "patch_size", 8)),
                                      in_chans=3, embed_dim=dim, precision=self.lidar_embed.precision)
        self.channels = dim
        # early_fusion_vit.py:75-79
        self.fusion_layer = ConvBnRelu3x3(2 * dim, dim, precision=self.lidar_embed.precision)
        self._side_streams = {}

    def _dropout_now(self, device=None) -> bool:
        """early_fusion_vit.py:113-119: one draw per forward for the whole batch, `torch.rand(1, device=x_lidar.device)` --
        i.e. from the generator of the LiDAR tensor's device, so that a seeded run drops the same batches as the reference
        -- then `.item() <= p` (one host sync, as in the reference)."""
        p = _get(_get(self.cfg, "experiment"), "lidar_dropout", None)
        if p is None:
            return False
        return bool(torch.rand(1, device=device).item() <= float(p))

    def forward_into(self, x_image, x_lidar, out: torch.Tensor, lidar_zero: Optional[bool] = None, lane: int = 0):
        """Eval-mode fused path: both halves written in place into `out` (B, 2C, ny, nx); returns `out`.  `lane`: see
        `PointPillarsEncoder.encode_into` (one lane per stream when several batches are in flight)."""
        dim = self.channels
        lidar_zero = self._dropout_now(out.device) if lidar_zero is None else bool(lidar_zero)
        # the two halves are independent until the concat: the patch embedding runs on a side stream next to the
        # voxelizer + PFN (fork / join by events, so a CUDA graph captures them as parallel branches)
        dev = out.device
        cur = torch.cuda.current_stream(dev)
        side = self._side_stream(dev, lane)
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            self.image_embed.forward_into(x_image, out, 2 * dim, 0)
        self.lidar_embed.encode_into(x_lidar, out, P3P_LAYOUT_NCHW, c_total=2 * dim, c_offset=dim, lidar_zero=lidar_zero, lane=lane)
        cur.wait_stream(side)
        return out

    def _side_stream(self, dev, lane: int = 0):
        side = self._side_streams.get((dev, lane))
        if side is None:
            side = self._side_streams[(dev, lane)] = torch.cuda.Stream(dev)
        return side

    def _vit_params(self, cls_token, pos_embed, device):
        """cls_token (1, 1, C) / pos_embed (1, 1 + ny nx, C) as contiguous fp32 on `device` -- the parameters themselves
        when they already are -- or (None, None) when neither is given."""
        if (cls_token is None) != (pos_embed is None):
            raise ValueError("cls_token and pos_embed go together: pass both or neither")
        if cls_token is None:
            return None, None
        hw, Cc = self.lidar_embed.ny * self.lidar_embed.nx, self.channels
        if cls_token.numel() != Cc or pos_embed.numel() != (hw + 1) * Cc:
            raise ValueError(f"cls_token must hold {Cc} and pos_embed {(hw + 1) * Cc} values")
        return (cls_token.detach().to(device=device, dtype=torch.float32).contiguous(),
                pos_embed.detach().to(device=device, dtype=torch.float32).contiguous())

    def forward_tokens(self, x_image, x_lidar, lidar_zero: Optional[bool] = None, *, cls_token: Optional[torch.Tensor] = None,
                       pos_embed: Optional[torch.Tensor] = None) -> torch.Tensor:
        """`EarlyFusionViT.forward` through `self.fusion_layer(x).flatten(2).transpose(1, 2)` (early_fusion_vit.py:96-123):
        (B, ny nx, C) fp32 tokens, the ViT's input.  Eval mode: the two producers write their halves of ONE 16-bit
        channels-last buffer (B, ny, nx, 2C) -- the reference's fp32 NCHW concat tensor never exists -- and the implicit-GEMM
        kernel turns it into token rows.

        With `cls_token` (1, 1, C) and `pos_embed` (1, 1 + ny nx, C) -- the ViT's own parameters -- the result is also
        passed through timm's `_pos_embed` (early_fusion_vit.py:124, `vit.forward_features` with `patch_embed = Identity`;
        one class token, `no_embed_class = False`): (B, 1 + ny nx, C) fp32, row 0 = cls_token + pos_embed[0], row 1 + cell =
        token + pos_embed[1 + cell].  Eval mode writes it from the convolution's epilogue (no cat, no add kernel); train mode
        runs the torch route above followed by `torch.cat` + add, so gradients reach cls_token and pos_embed."""
        if self.training:
            if (cls_token is None) != (pos_embed is None):
                raise ValueError("cls_token and pos_embed go together: pass both or neither")
            x = self.forward(x_image, x_lidar)
            t = self.fusion_layer(x).flatten(2).transpose(1, 2)
            if cls_token is None:
                return t
            B, hw, Cc = t.shape
            if cls_token.numel() != Cc or pos_embed.numel() != (hw + 1) * Cc:
                raise ValueError(f"cls_token must hold {Cc} and pos_embed {(hw + 1) * Cc} values")
            cls = cls_token.to(device=t.device, dtype=torch.float32).reshape(1, 1, Cc).expand(B, -1, -1)
            return torch.cat((cls, t), dim=1) + pos_embed.to(device=t.device, dtype=torch.float32).reshape(1, hw + 1, Cc)
        dim, le, fl = self.channels, self.lidar_embed, self.fusion_layer
        B, dev = x_image.shape[0], x_image.device
        x16 = torch.empty(B, le.ny, le.nx, 2 * dim, dtype=fl.operand_dtype, device=dev)
        rows = le.ny * le.nx + (0 if cls_token is None else 1)
        out = torch.empty(B, rows, dim, dtype=torch.float32, device=dev)
        return self.forward_tokens_into(x_image, x_lidar, x16, out, lidar_zero, cls_token=cls_token, pos_embed=pos_embed)

    def forward_tokens_into(self, x_image, x_lidar, x16: torch.Tensor, out: torch.Tensor, lidar_zero: Optional[bool] = None,
                            lane: int = 0, *, cls_token: Optional[torch.Tensor] = None, pos_embed: Optional[torch.Tensor] = None):
        """forward_tokens with caller-owned buffers: x16 (B, ny, nx, 2C) 16-bit scratch, out (B, ny nx, C) fp32 -- or
        (B, 1 + ny nx, C) with cls_token / pos_embed, which the kernel reads in place when they are fp32 on the device
        (otherwise from a converted copy)."""
        dim, le, fl = self.channels, self.lidar_embed, self.fusion_layer
        dev = x_image.device
        cls, pos = self._vit_params(cls_token, pos_embed, dev)
        lidar_zero = self._dropout_now(dev) if lidar_zero is None else bool(lidar_zero)
        cur = torch.cuda.current_stream(dev)
        side = self._side_stream(dev, lane)
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            self.image_embed.forward_into(x_image, x16, 2 * dim, 0, layout=P3P_LAYOUT_NLC)
        le.encode_into(x_lidar, x16, P3P_LAYOUT_NLC, c_total=2 * dim, c_offset=dim, lidar_zero=lidar_zero, lane=lane)
        cur.wait_stream(side)
        if cls is not None:
            return fl._runner.run_vit_tokens(x16, cls, pos, out)
        return fl.forward_nhwc(x16, out, P3P_LAYOUT_NLC)

    def forward(self, x_image, x_lidar):
        if self.training:  # BatchNorm batch statistics: the dense autograd route of the optional training step
            xi = self.image_embed(x_image)
            xl = self.lidar_embed(x_lidar, return_flattened=False)
            if self._dropout_now(xl.device):
                xl = xl * 0.0
            return torch.cat((xi, xl), dim=1)
        B = x_image.shape[0]
        le = self.lidar_embed
        out = torch.empty(B, 2 * self.channels, le.ny, le.nx, dtype=le.out_dtype, device=x_image.device)
        return self.forward_into(x_image, x_lidar, out)
