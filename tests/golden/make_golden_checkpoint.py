"""Golden parameter names and shapes for tests/test_checkpoint_cpu.py: the reference's own classes (read in place from the
reference tree, never copied) are constructed over the torch-backed paddle shim; no weights are needed, only the keys and
shapes of their state_dicts, which go to tests/golden/reference_checkpoint_names.npz.

    python tests/golden/make_golden_checkpoint.py          (needs the reference tree; the tests read the committed .npz)

Stored entries:
    moco:<name>     shape (int64 vector) of the MoCo v2 checkpoint entry `encoder_q.{0,1}.*`: ResNet-50 (resnetimagenet.py) and
                    NonLinearNeckV1 (base_neck.py) with in 2048, hidden 2048, out 128
    mocov3:<name>   shape of the MoCoV3Pretrain state_dict entry (passl/models/mocov3.py; ViT img 32, patch 8, dim 64, depth 1,
                    2 heads, qkv bias, projector dim 32, mlp 48), the CosineEMA wrapper's `momentum_encoder.model.*` / `steps` included
    mocov3_pos      the fixed 2-D sin-cos position table that model builds, float32 [1, 17, 64]
"""
import functools
import importlib
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import paddle_shim  # noqa: E402,F401
import make_golden  # noqa: E402
import make_golden_models as M  # noqa: E402


def moco_names():
    nn = sys.modules["paddle.nn"]

    class Conv2D(nn.Layer):
        def __init__(self, i, o, kernel_size, stride=1, padding=0, dilation=1, groups=1, bias_attr=None, **kw):
            super().__init__()
            self.weight = torch.nn.Parameter(torch.zeros(o, i, kernel_size, kernel_size))

    class BatchNorm2D(nn.Layer):
        def __init__(self, c, **kw):
            super().__init__()
            self.weight, self.bias = torch.nn.Parameter(torch.ones(c)), torch.nn.Parameter(torch.zeros(c))
            self.register_buffer("_mean", torch.zeros(c))
            self.register_buffer("_variance", torch.ones(c))

    class MaxPool2D(nn.Layer):
        def __init__(self, *a, **k):
            super().__init__()
    saved = {k: getattr(nn, k, None) for k in ("Conv2D", "BatchNorm2D", "MaxPool2D")}
    nn.Conv2D, nn.BatchNorm2D, nn.MaxPool2D = Conv2D, BatchNorm2D, MaxPool2D
    try:
        rn = importlib.import_module("passl_v110.modeling.backbones.resnetimagenet")
        necks = importlib.import_module("passl_v110.modeling.necks.base_neck")
        ref_backbone = rn.ResNet(rn.BottleneckBlock, 50, num_classes=0, with_pool=False)
        ref_neck = necks.NonLinearNeckV1(in_channels=2048, hid_channels=2048, out_channels=128)
    finally:
        for k, v in saved.items():
            if v is not None:
                setattr(nn, k, v)
    out = {}
    for pre, mod in (("encoder_q.0.", ref_backbone), ("encoder_q.1.", ref_neck)):
        for k, v in mod.state_dict().items():
            out["moco:" + pre + k] = np.array(v.shape, dtype=np.int64)
    return out


def mocov3_names():
    import paddle
    nn = sys.modules["paddle.nn"]
    paddle.meshgrid = lambda *xs: torch.meshgrid(*xs, indexing="ij")
    paddle.sin, paddle.cos = torch.sin, torch.cos

    class Conv2D(nn.Layer):
        def __init__(self, i, o, kernel_size, stride=1, padding=0, bias_attr=None, **kw):
            super().__init__()
            k = kernel_size if isinstance(kernel_size, (tuple, list)) else (kernel_size, kernel_size)
            self.weight = torch.nn.Parameter(torch.zeros(o, i, k[0], k[1]))
            self.bias = None if bias_attr is False else torch.nn.Parameter(torch.zeros(o))

    class BatchNorm1D(nn.Layer):                 # Paddle keeps (frozen) weight / bias entries when weight_attr / bias_attr are False
        def __init__(self, c, weight_attr=None, bias_attr=None, **kw):
            super().__init__()
            self.weight, self.bias = torch.nn.Parameter(torch.ones(c)), torch.nn.Parameter(torch.zeros(c))
            self.register_buffer("_mean", torch.zeros(c))
            self.register_buffer("_variance", torch.ones(c))
    saved = {k: getattr(nn, k, None) for k in ("Conv2D", "BatchNorm1D", "LayerList")}
    nn.Conv2D, nn.BatchNorm1D, nn.LayerList = Conv2D, BatchNorm1D, torch.nn.ModuleList
    torch.Tensor._share_buffer_to = lambda self, other: None
    torch.Tensor.set_value = lambda self, v: self.data.copy_(v)
    nn.Layer.create_parameter = lambda self, shape, **kw: torch.nn.Parameter(torch.zeros(tuple(shape)), requires_grad=False)
    nn.Layer.named_sublayers = lambda self: self.named_modules()

    class _NoInit(types.ModuleType):
        def __getattr__(self, n):
            return lambda *a, **k: None
    try:
        vt = importlib.import_module("passl.models.vision_transformer")
        vt.init = _NoInit("init")
        mv = importlib.import_module("passl.models.mocov3")
        mv.init = _NoInit("init")
        ref = mv.MoCoV3Pretrain(functools.partial(mv.MoCoV3ViT, img_size=32, patch_size=8, embed_dim=64, depth=1, num_heads=2,
                                                  mlp_ratio=4, qkv_bias=True), dim=32, mlp_dim=48)
        out = {"mocov3:" + k: np.array(v.shape, dtype=np.int64) for k, v in ref.state_dict().items()}
        out["mocov3_pos"] = ref.base_encoder.pos_embed.detach().numpy().astype(np.float32)
    finally:
        for k, v in saved.items():
            if v is not None:
                setattr(nn, k, v)
    return out


def main():
    make_golden.setup()
    M.extend_shim()
    out = moco_names()
    out.update(mocov3_names())
    np.savez_compressed(os.path.join(HERE, "reference_checkpoint_names.npz"), **out)
    print("wrote reference_checkpoint_names.npz: %d MoCo v2 entries, %d MoCo v3 entries" %
          (sum(k.startswith("moco:") for k in out), sum(k.startswith("mocov3:") for k in out)))


if __name__ == "__main__":
    main()
