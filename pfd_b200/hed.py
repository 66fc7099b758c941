"""HED soft-edge annotator of ControlNet.preprocess(type='hed' / 'softedge_v11p') on the pfd_b200 kernels.

Mirrors lib/model_zoo/controlnet_annotator/hed/__init__.py (ControlNetHED_Apache2 + apply_hed) and the
'hed' branch of lib/model_zoo/controlnet.py:370-376.  ``ControlNetHED`` is a parameter holder with the reference's
state-dict keys, so ``load_state_dict(torch.load('ControlNetHED.pth'), strict=True)`` works.  The network is a
module-level singleton, like the reference's ``netNetwork``, and deliberately not a sub-module of ControlNet, so
ControlNet's state dict keeps the reference layout.  It is loaded lazily from the reference's locations (never
downloaded) or injected with ``set_network``.

Numerics: activations are fp16 channel-last with fp32 accumulation.  The reference feeds the raw 0-255 image, so
every conv bias and the input are multiplied by the power-of-two ``SCALE`` (ReLU and max-pool commute with a positive
scale, so every activation is exactly SCALE times the reference's) and the fp32 projections divide it out again.
The projections, resizes, mean, sigmoid and quantisation are fp32 / fp64.  A non-finite logit raises RuntimeError.
"""
from __future__ import annotations

import os
from typing import List, Mapping, Optional, Union

import torch
import torch.nn as nn

from . import native as nv
from .graphs import weights_signature
from .modules import Conv2d, IndexedSequential, pack_conv3x3, pad_cols

SCALE = 2.0 ** -8
MODEL_RELPATH = os.path.join("pretrained", "controlnet", "preprocess", "hed", "ControlNetHED.pth")
_HERE = os.path.dirname(os.path.abspath(__file__))


class DoubleConvBlock(nn.Module):
    """hed/__init__.py:23-39: `layer_number` 3x3 convs (+ ReLU) and a 1x1 projection to one channel."""

    def __init__(self, input_channel: int, output_channel: int, layer_number: int):
        super().__init__()
        self.convs = IndexedSequential(*[Conv2d(input_channel if i == 0 else output_channel, output_channel, 3,
                                                padding=1) for i in range(layer_number)])
        self.projection = Conv2d(output_channel, 1, 1)


class ControlNetHED(nn.Module):
    """Parameter holder of ControlNetHED_Apache2 (hed/__init__.py:42-49); computed by `run`."""

    def __init__(self):
        super().__init__()
        self.norm = nn.Parameter(torch.zeros(size=(1, 3, 1, 1)))
        self.block1 = DoubleConvBlock(3, 64, 2)
        self.block2 = DoubleConvBlock(64, 128, 2)
        self.block3 = DoubleConvBlock(128, 256, 3)
        self.block4 = DoubleConvBlock(256, 512, 3)
        self.block5 = DoubleConvBlock(512, 512, 3)

    def blocks(self) -> List[DoubleConvBlock]:
        return [self.block1, self.block2, self.block3, self.block4, self.block5]

    def forward(self, *a, **k):  # pragma: no cover
        raise RuntimeError("ControlNetHED is a parameter holder: use pfd_b200.hed.run / ControlNet.preprocess")


_network: Optional[ControlNetHED] = None
_pack = None            # (key, packed weights) of the last network run


def model_paths() -> List[str]:
    """Where `get_network` looks for ControlNetHED.pth: the reference's model directory under the working directory,
    then next to this module."""
    return [os.path.join(os.getcwd(), MODEL_RELPATH), os.path.join(_HERE, "ControlNetHED.pth")]


def set_network(net: Union[nn.Module, Mapping[str, torch.Tensor], None]) -> Optional[ControlNetHED]:
    """Use `net` for every later HED run: a ControlNetHED (kept as is, so a later load_state_dict on it is seen), any
    module or state dict with the reference's keys (loaded strictly into a new ControlNetHED), or None to forget the
    network (the next run loads it from `model_paths()` again)."""
    global _network, _pack
    if net is not None and not isinstance(net, ControlNetHED):
        sd = net.state_dict() if isinstance(net, nn.Module) else net
        net = ControlNetHED()
        net.load_state_dict(sd, strict=True)
    _network, _pack = net, None
    return net


def get_network() -> ControlNetHED:
    """The network set by `set_network`, else ControlNetHED.pth from the first of `model_paths()` that exists."""
    if _network is None:
        for path in model_paths():
            if os.path.exists(path):
                set_network(torch.load(path, map_location="cpu", weights_only=True))
                break
        else:
            raise FileNotFoundError("HED annotator weights ControlNetHED.pth not found; looked in "
                                    + ", ".join(model_paths()) + " (nothing is downloaded: place the file there or "
                                    "call pfd_b200.hed.set_network)")
    return _network


def _packed(net: ControlNetHED, device: torch.device, scale: float):
    """fp16 GEMM weights with biases multiplied by `scale`, fp32 projections and norm, on `device` (the network itself
    may stay on the CPU); re-built whenever a weight of `net` changes (load_state_dict, in-place writes, .to())."""
    global _pack
    key = (weights_signature(net), str(device), scale)
    if _pack is not None and _pack[0] == key:
        return _pack[1]

    def f16(t):
        return t.detach().to(device=device, dtype=torch.float16).contiguous()

    def f32(t):
        return t.detach().to(device=device, dtype=torch.float32).reshape(-1).contiguous()

    with torch.no_grad():
        blocks = []
        for blk in net.blocks():
            convs = []
            for conv in blk.convs:
                w = pad_cols(pack_conv3x3(conv.weight.to(device)))          # [Cout, 9*Cin (padded to 8)], k = tap*Cin + c
                convs.append((w, f16(conv.bias.detach().float() * scale)))
            blocks.append((convs, f32(blk.projection.weight), f32(blk.projection.bias)))
        pk = {"norm": f32(net.norm), "blocks": blocks}
    _pack = (key, pk)
    return pk


def run(x: torch.Tensor, net: Optional[ControlNetHED] = None, scale: float = SCALE) -> torch.Tensor:
    """HED edge map of a CUDA [B,3,H,W] fp16/fp32 image in [0,1] -> float32 [B,3,H,W] (apply_hed per image +
    ToTensor + repeat, controlnet.py:370-376), as one batched network pass.  H, W >= 16."""
    if x.dim() != 4 or x.shape[1] != 3:
        raise ValueError(f"HED expects a [B,3,H,W] image, got {tuple(x.shape)}")
    B, _, H, W = x.shape
    if H < 16 or W < 16:
        raise ValueError(f"HED needs an image of at least 16x16 (four 2x2 max-pools), got {H}x{W}")
    net = net if net is not None else get_network()
    pk = _packed(net, x.device, scale)
    h = nv.hed_input(x, pk["norm"], scale)
    maps = []
    for k, (convs, pw, pb) in enumerate(pk["blocks"]):
        if k > 0:
            h = nv.maxpool2x2(h)
        for w, b in convs:
            if h.shape[3] % 8:                                          # the 3-channel stem: im2col + GEMM
                Bh, Hh, Wh, _ = h.shape
                col = nv.im2col3x3(h, w.shape[1])
                h = nv.linear(col.reshape(Bh * Hh * Wh, w.shape[1]), w, b, act=nv.ACT_RELU).reshape(Bh, Hh, Wh, -1)
            else:
                h = nv.conv3x3(h, w, b, act=nv.ACT_RELU)
        maps.append(nv.hed_project(h, pw, pb, 1.0 / scale))
    out, nonfinite = nv.hed_fuse(maps, H, W)
    bad = int(nonfinite.item())
    if bad:
        raise RuntimeError(f"HED: {bad} of {B * H * W} edge logits are not finite: the network's activations "
                           f"overflowed fp16 at activation scale {scale:g}; use a smaller scale (pfd_b200.hed.run)")
    return out
