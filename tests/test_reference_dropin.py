"""The module as the PixelsPointsPolygons project's encoders use it (CPU, plus the shapes of the real forward on the GPU).

On every checkout the module is checked against what the project expects of it, recorded from its source in
tests/golden/reference_dropin.json: the constructor call and the cfg fields it reads (its encoder YAMLs), the Open3D-ML
kwargs the constructor derives, the state-dict key names and shapes its checkpoints store, the `forward` arguments its
encoders pass and the shapes they consume.

Where the environment variable P3P_REFERENCE_DIR names a checkout of the project, the same tests also import its
encoder classes unmodified with the single swap INTEGRATION.md describes -- `pixelspointspolygons.models.pointpillars.
pointpillars_o3d` provided by this package instead of the Open3D subclass -- and a stub `timm` (the ViT blocks are out of
scope), with cfg from the project's own YAML through PyYAML: the reference constructors accept our module, it lands where
the reference puts it (`vit.patch_embed`, `lidar_embed`), the reference's `forward` drives it with the arguments we
implement, shapes flow through the reference's own post-processing, and the reference's key names load.  (The
arithmetic of the module is covered by the -m gpu parity tests; this file pins the boundary.)"""
import importlib.util
import inspect
import json
import os
import sys
import types

import numpy as np
import pytest
import torch
import torch.nn as nn

REF = os.environ.get("P3P_REFERENCE_DIR", "")
LIVE = bool(REF) and os.path.isdir(os.path.join(REF, "pixelspointspolygons"))
with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_dropin.json")) as f:
    FACTS = json.load(f)


class StubViT(nn.Module):
    """timm VisionTransformer reduced to what the reference's encoders touch: `patch_embed`, `cls_token`, `pos_embed`,
    forward = patch_embed -> class token + positional embedding -> (blocks omitted) -> (B, 1 + N, C)."""

    def __init__(self, dim=384, n=784):
        super().__init__()
        self.patch_embed = nn.Identity()
        self.cls_token = nn.Parameter(torch.zeros(1, 1, dim))
        self.pos_embed = nn.Parameter(torch.zeros(1, n + 1, dim))
        self.seen = None

    def forward(self, x):
        x = self.patch_embed(x)
        self.seen = tuple(x.shape)
        x = torch.cat([self.cls_token.expand(x.shape[0], -1, -1), x], dim=1)
        return x + self.pos_embed


def load_reference(monkeypatch, tmp_path):
    import pixelspointspolygons_b200 as ours

    created = []

    def pkg(name, path=None):
        m = types.ModuleType(name)
        m.__path__ = [path] if path else []
        monkeypatch.setitem(sys.modules, name, m)
        return m

    base = os.path.join(REF, "pixelspointspolygons")
    pkg("pixelspointspolygons", base)
    pkg("pixelspointspolygons.models", os.path.join(base, "models"))
    pkg("pixelspointspolygons.models.pointpillars", os.path.join(base, "models", "pointpillars"))
    pkg("pixelspointspolygons.models.fusion_layers", os.path.join(base, "models", "fusion_layers"))
    pkg("pixelspointspolygons.misc")
    logger_mod = types.ModuleType("pixelspointspolygons.misc.logger")
    import logging

    logger_mod.make_logger = lambda name, level=logging.INFO, local_rank=0, **kw: logging.getLogger(name)
    monkeypatch.setitem(sys.modules, "pixelspointspolygons.misc.logger", logger_mod)
    head = types.ModuleType("pixelspointspolygons.models.multitask_head")
    head.MultitaskHead = nn.Identity
    monkeypatch.setitem(sys.modules, "pixelspointspolygons.models.multitask_head", head)
    # THE swap (INTEGRATION.md): the module the reference imports `PointPillarsEncoder` from
    swap = types.ModuleType("pixelspointspolygons.models.pointpillars.pointpillars_o3d")
    swap.PointPillarsEncoder = ours.PointPillarsEncoder
    monkeypatch.setitem(sys.modules, "pixelspointspolygons.models.pointpillars.pointpillars_o3d", swap)
    timm = types.ModuleType("timm")

    def create_model(model_name, num_classes=0, global_pool="", **kw):
        created.append(model_name)
        return StubViT()

    timm.create_model = create_model
    monkeypatch.setitem(sys.modules, "timm", timm)

    def load(rel, name):
        spec = importlib.util.spec_from_file_location(name, os.path.join(base, rel))
        mod = importlib.util.module_from_spec(spec)
        monkeypatch.setitem(sys.modules, name, mod)
        spec.loader.exec_module(mod)
        return mod

    ppvit = load("models/pointpillars/pointpillars_vit.py", "pixelspointspolygons.models.pointpillars.pointpillars_vit")
    efvit = load("models/fusion_layers/early_fusion_vit.py", "pixelspointspolygons.models.fusion_layers.early_fusion_vit")
    (tmp_path / "backbones").mkdir()
    torch.save({}, tmp_path / "backbones" / "dino_deitsmall8_pretrain.pth")
    return ppvit, efvit, created, str(tmp_path)


def fake_kernel(monkeypatch, calls):
    """The CUDA call replaced by a recorder (there is no GPU here and the module has no CPU path by design)."""
    from pixelspointspolygons_b200 import PointPillarsEncoder

    def forward(self, x_lidar, return_flattened=True):
        B = len(x_lidar) if isinstance(x_lidar, (list, tuple)) else x_lidar.shape[0]
        calls.append((type(x_lidar).__name__, B, return_flattened))
        hw = self.ny * self.nx
        return torch.zeros(B, hw, self.channels) if return_flattened else torch.zeros(B, self.channels, self.ny, self.nx)

    monkeypatch.setattr(PointPillarsEncoder, "forward", forward)


def live_pointpillars_vit(monkeypatch, tmp_path):
    from pixelspointspolygons_b200 import PointPillarsEncoder
    from pixelspointspolygons_b200.config import cfg_from_encoder_yaml

    ppvit, _, created, out_path = load_reference(monkeypatch, tmp_path)
    cfg = cfg_from_encoder_yaml(os.path.join(REF, "config", "encoder", "pointpillars_vit.yaml"), device="cpu", out_path=out_path)
    model = ppvit.PointPillarsViT(cfg, bottleneck=True)
    assert created == ["vit_small_patch8_224.dino"]
    enc = model.vit.patch_embed
    assert isinstance(enc, PointPillarsEncoder)
    # the reference's cfg -> Open3D-ML kwargs mapping (pointpillars_o3d.py:39-60), reproduced by our constructor
    assert enc.point_cloud_range == [0, 0, 0, 224, 224, 100] and enc.voxel_size == [8, 8, 100]
    assert enc.max_num_points == 64 and enc.max_voxels == [784, 784] and (enc.ny, enc.nx, enc.channels) == (28, 28, 384)
    # checkpoint keys as the reference's models save them (SURVEY Appendix C)
    keys = [k for k in model.state_dict() if "patch_embed" in k]
    assert "vit.patch_embed.voxel_encoder.pfn_layers.0.linear.weight" in keys
    assert "vit.patch_embed.voxel_encoder.pfn_layers.1.norm.running_var" in keys
    calls = []
    fake_kernel(monkeypatch, calls)
    x = torch.nested.nested_tensor([torch.rand(50, 3), torch.rand(7, 3)], layout=torch.jagged)
    y = model.eval()(x)  # reference forward: vit(x) -> drop the class token -> AdaptiveAvgPool1d(out_feature_dim)
    assert calls == [("NestedTensor", 2, True)] or calls == [("Tensor", 2, True)]
    assert model.vit.seen == (2, 784, 384) and tuple(y.shape) == (2, 784, 256)


def live_early_fusion_vit(monkeypatch, tmp_path):
    from pixelspointspolygons_b200 import ConvBnRelu3x3, PointPillarsEncoder
    from pixelspointspolygons_b200.config import cfg_from_encoder_yaml

    _, efvit, _, out_path = load_reference(monkeypatch, tmp_path)
    cfg = cfg_from_encoder_yaml(os.path.join(REF, "config", "encoder", "early_fusion_vit.yaml"), device="cpu", out_path=out_path)
    model = efvit.EarlyFusionViT(cfg)
    assert isinstance(model.lidar_embed, PointPillarsEncoder)
    # our fused-layer module has the reference's state_dict keys: its weights load into it and back
    ours = ConvBnRelu3x3(768, 384)
    assert list(ours.state_dict().keys()) == list(model.fusion_layer.state_dict().keys())
    ours.load_state_dict(model.fusion_layer.state_dict(), strict=True)
    model.fusion_layer = ours.train()  # (train mode = the torch modules; the kernel needs a GPU)
    calls = []
    fake_kernel(monkeypatch, calls)
    # the stub ViT's patch_embed is re-parented as image_embed by the reference; give it the conv timm would have
    model.image_embed = nn.Conv2d(3, 384, 8, 8)
    x_lidar = torch.nested.nested_tensor([torch.rand(50, 3), torch.rand(7, 3)], layout=torch.jagged)
    y = model(torch.rand(2, 3, 224, 224), x_lidar)
    assert calls and calls[0][1:] == (2, False)  # lidar_embed(x_lidar, return_flattened=False)
    assert tuple(y.shape) == (2, 784, 256)


def stored_cfg(device="cpu"):
    from pixelspointspolygons_b200.config import AttrDict

    enc = {k: v for k, v in FACTS["encoder_cfg"].items() if k != "source"}
    return AttrDict.wrap(dict(host=dict(device=device), run_type=dict(logging="WARNING"),
                              experiment=dict(encoder=enc, lidar_dropout=None)))


def stored_encoder(device="cpu"):
    from pixelspointspolygons_b200 import PointPillarsEncoder

    ctor = FACTS["constructor"]
    return PointPillarsEncoder(stored_cfg(device), voxel_encoder=ctor["voxel_encoder"], scatter=ctor["scatter"],
                               local_rank=ctor["local_rank"])


def keys_and_shapes(module):
    """name -> shape (a checkpoint loads by name: the order of the keys is not part of the format)"""
    return {k: list(t.shape) for k, t in module.state_dict().items()}


def stored(entry):
    return {k: s for k, s in FACTS[entry]["keys"]}


def check_stored_encoder():
    """The constructor call of the reference's encoders, the kwargs it derives, its checkpoint keys, its forward signature."""
    from pixelspointspolygons_b200 import PointPillarsEncoder

    enc = stored_encoder()
    for name, value in FACTS["constructed"].items():
        if name != "source":
            assert getattr(enc, name) == value, name
    assert keys_and_shapes(enc) == stored("state_dict")
    # a checkpoint with the reference's names and shapes loads strictly, and comes back under the same names
    sd = {k: torch.zeros(s, dtype=torch.long) if k.endswith("num_batches_tracked") else torch.rand(s)
          for k, s in stored("state_dict").items()}
    enc.load_state_dict(sd, strict=True)
    assert all(torch.equal(enc.state_dict()[k], v) for k, v in sd.items())
    params = inspect.signature(PointPillarsEncoder.forward).parameters
    assert list(params)[1:3] == ["x_lidar", "return_flattened"] and params["return_flattened"].default is True


def test_reference_pointpillars_vit_accepts_the_module(monkeypatch, tmp_path):
    check_stored_encoder()
    if LIVE:
        live_pointpillars_vit(monkeypatch, tmp_path)


def test_reference_early_fusion_vit_accepts_the_module(monkeypatch, tmp_path):
    from pixelspointspolygons_b200 import ConvBnRelu3x3
    from pixelspointspolygons_b200.fusion import EarlyFusionFrontEnd

    check_stored_encoder()
    fe = EarlyFusionFrontEnd(stored_cfg())
    assert keys_and_shapes(fe.fusion_layer) == stored("fusion_layer_state_dict")
    assert keys_and_shapes(fe.image_embed) == stored("image_embed_state_dict")
    assert keys_and_shapes(fe.lidar_embed) == stored("state_dict")
    ours = ConvBnRelu3x3(768, 384)
    sd = {k: torch.zeros(s, dtype=torch.long) if k.endswith("num_batches_tracked") else torch.rand(s)
          for k, s in stored("fusion_layer_state_dict").items()}
    ours.load_state_dict(sd, strict=True)
    if LIVE:
        live_early_fusion_vit(monkeypatch, tmp_path)


@pytest.mark.gpu
@pytest.mark.parametrize("encoder", ["pointpillars_vit", "early_fusion_vit"])
def test_forward_hands_the_reference_the_shapes_it_consumes(cuda_device, encoder):
    from tools.synth import synth_tile

    want = FACTS["forward"][encoder]
    enc = stored_encoder(str(cuda_device)).to(cuda_device).eval()
    x = torch.nested.nested_tensor([torch.from_numpy(synth_tile(n, 70 + n)) for n in (50, 7)], layout=torch.jagged).to(cuda_device)
    with torch.no_grad():
        y = enc(x, return_flattened=want["return_flattened"])
    assert list(y.shape) == [2] + want["shape_per_tile"] and y.dtype == torch.float32 and y.is_cuda
    assert np.isfinite(y.cpu().numpy()).all()
