"""CPU fp32 restatement of the HED soft-edge annotator behind ControlNet.preprocess(type='hed' / 'softedge_v11p').
TEST INFRASTRUCTURE — only tests/ and tools/ may import this module.

Reference path: lib/model_zoo/controlnet.py:370-376 (tensor -> ToPILImage -> apply_hed -> ToTensor -> repeat(1,3,1,1)
-> float32) and lib/model_zoo/controlnet_annotator/hed/__init__.py:102-128.  Written from the maths:
  1. u8 = floor(x*255) (ToPILImage; the product is rounded in the tensor's dtype first);
  2. h = u8 - norm, then five VGG blocks (2x2 floor max-pool before blocks 2-5, 3x3 pad-1 convs + ReLU) each
     followed by a 1x1 projection to one channel;
  3. every projection resized to HxW with cv2's INTER_LINEAR (half-pixel centres, clamped borders, float32),
     averaged in float32, sigmoid in float64, (e*255).clip(0,255) truncated to uint8.
The resize is restated in numpy (cv2 is not needed); tests/test_hed_cpu.py pins it against cv2.resize and the whole
chain against tests/golden/hed_reference.npz, which the unmodified reference produced (tools/make_golden_hed.py).
"""
import math

import numpy as np
import torch
import torch.nn.functional as F

BLOCKS = ((3, 64, 2), (64, 128, 2), (128, 256, 3), (256, 512, 3), (512, 512, 3))   # (Cin, Cout, convs)
PREFIX = "hed."

# Gain schedule of the synthetic weights (on top of synth_tensor's unit-fan-in scaling): He gain on every conv keeps
# the activations at the input's 0-255 scale through all 13 ReLU convs; projection k is divided by that block's
# typical activation so each logit map is O(1) and their mean spreads over the sigmoid's steep part (>= 64 output
# levels, no saturated pixels) without using every level: a steeper map puts more pixels next to a quantisation step.  norm is an ImageNet-like per-channel mean.
CONV_GAIN = math.sqrt(2.0)
PROJ_GAIN = (1 / 20.0, 1 / 40.0, 1 / 60.0, 1 / 60.0, 1 / 60.0)


def state_dict_shapes():
    """Keys and shapes of the reference's ControlNetHED_Apache2 state dict (hed/__init__.py:23-49)."""
    shapes = {"norm": (1, 3, 1, 1)}
    for k, (cin, cout, n) in enumerate(BLOCKS, 1):
        for i in range(n):
            shapes[f"block{k}.convs.{i}.weight"] = (cout, cin if i == 0 else cout, 3, 3)
            shapes[f"block{k}.convs.{i}.bias"] = (cout,)
        shapes[f"block{k}.projection.weight"] = (1, cout, 1, 1)
        shapes[f"block{k}.projection.bias"] = (1,)
    return shapes


def synth_state_dict(seed=0, amplify_log2=0):
    """Seeded HED weights under the reference key names (pfd_b200.weights.synth_tensor with PREFIX + the gain schedule
    above).  amplify_log2 = a scales every activation by exactly 2**a: the first conv's weight and every conv bias by
    2**a, every projection weight by 2**-a.  ReLU and max-pool commute with a positive scale, so the logits (and the
    edge map) are unchanged while the activations' range grows."""
    from pfd_b200.weights import synth_tensor
    amp = 2.0 ** amplify_log2
    sd = {}
    for name, shape in state_dict_shapes().items():
        t = synth_tensor(PREFIX + name, shape, seed)
        if name == "norm":
            t = 120.0 + 16.0 * torch.randn(shape, generator=torch.Generator().manual_seed(seed + 17))
        elif ".convs." in name and name.endswith("weight"):
            t = t * CONV_GAIN * (amp if name.startswith("block1.convs.0.") else 1.0)
        elif ".convs." in name:
            t = t * amp
        elif name.endswith("projection.weight"):
            t = t * (PROJ_GAIN[int(name[5]) - 1] / amp)
        sd[name] = t.contiguous()
    return sd


# Golden cases (tests/golden/hed_reference.npz): (name, H, W, images, seed).  512^2; a non-square size not divisible by
# 16 with two images (the batched case); 33x31, where block 5 is 2x1.
CASES = (("512x512", 512, 512, 1, 100), ("200x328", 200, 328, 2, 101), ("33x31", 33, 31, 1, 102))


def case_images(name):
    """The uint8 [n, H, W, 3] input images of golden case `name`: uniform noise smoothed by a 17x17 and then a 9x9 box
    filter, stretched to 0..255 per image.  Integer arithmetic only, so every machine builds the same images and the
    golden file needs to hold only the edge maps."""
    _, H, W, n, seed = next(c for c in CASES if c[0] == name)
    v = np.random.RandomState(seed).randint(0, 256, size=(n, H, W, 3)).astype(np.int64)
    for r in (8, 4):
        p = np.pad(v, ((0, 0), (r, r), (r, r), (0, 0)), mode="reflect")
        c = np.cumsum(np.cumsum(np.pad(p, ((0, 0), (1, 0), (1, 0), (0, 0))), axis=1), axis=2)
        k = 2 * r + 1
        v = c[:, k:, k:] - c[:, :-k, k:] - c[:, k:, :-k] + c[:, :-k, :-k]
    lo = v.min(axis=(1, 2, 3), keepdims=True)
    hi = v.max(axis=(1, 2, 3), keepdims=True)
    return ((v - lo) * 256 // (hi - lo + 1)).astype(np.uint8)


def encode_edges(edges):
    """uint8 [..., W] edge maps -> row-wise differences mod 256 (smooth maps compress better that way)."""
    return np.diff(edges.astype(np.int16), axis=-1, prepend=0).astype(np.uint8)


def golden_edges(golden, name):
    """The reference's uint8 [n, H, W] edge maps of case `name` from tests/golden/hed_reference.npz."""
    return np.cumsum(golden[f"edge_delta_{name}"], axis=-1, dtype=np.uint8)


def to_u8(x):
    """ToPILImage on a float [3,H,W] tensor: x.mul(255).byte() in x's dtype -> HxWx3 uint8."""
    return x.mul(255).byte().permute(1, 2, 0).contiguous().cpu().numpy()


def logits(sd, img_u8):
    """Five fp32 projection maps [H_k, W_k] of an HxWx3 uint8 image, plus the maximum activation of each block."""
    sd = {k: v.detach().float().cpu() for k, v in sd.items()}
    h = torch.from_numpy(np.ascontiguousarray(img_u8)).float().permute(2, 0, 1)[None] - sd["norm"]
    maps, amax = [], []
    for k, (_, _, n) in enumerate(BLOCKS, 1):
        if k > 1:
            h = F.max_pool2d(h, 2, 2)
        for i in range(n):
            h = F.relu(F.conv2d(h, sd[f"block{k}.convs.{i}.weight"], sd[f"block{k}.convs.{i}.bias"], padding=1))
        amax.append(float(h.max()))
        p = F.conv2d(h, sd[f"block{k}.projection.weight"], sd[f"block{k}.projection.bias"])
        maps.append(p[0, 0].numpy().astype(np.float32))
    return maps, amax


def _linear_taps(n_src, n_dst):
    """INTER_LINEAR source indices and weights of each destination index: half-pixel centres
    f = (d + 0.5) * n_src / n_dst - 0.5 in float64, weight f - floor(f) rounded to float32, clamped to the first / last
    source index with weight 0 outside (this matches cv2.resize on float32 maps to ~1e-7 relative)."""
    scale = 1.0 / (float(n_dst) / n_src)
    f = (np.arange(n_dst) + 0.5) * scale - 0.5
    i0 = np.floor(f).astype(np.int64)
    w1 = f - i0
    lo = i0 < 0
    i0[lo], w1[lo] = 0, 0.0
    hi = i0 >= n_src - 1
    i0[hi], w1[hi] = n_src - 1, 0.0
    i1 = np.minimum(i0 + 1, n_src - 1)
    return i0, i1, (1.0 - w1).astype(np.float32), w1.astype(np.float32)


def resize_linear(src, H, W):
    """cv2.resize(src, (W, H), interpolation=cv2.INTER_LINEAR) of a float32 [h, w] map: rows first, then columns."""
    src = np.asarray(src, dtype=np.float32)
    if src.shape == (H, W):
        return src.copy()
    x0, x1, a0, a1 = _linear_taps(src.shape[1], W)
    y0, y1, b0, b1 = _linear_taps(src.shape[0], H)
    rows = src[:, x0] * a0 + src[:, x1] * a1
    return (rows[y0] * b0[:, None] + rows[y1] * b1[:, None]).astype(np.float32)


def edge_u8(maps, H, W):
    """Resize, float32 mean, float64 sigmoid, x255, clip and truncate -> HxW uint8."""
    acc = resize_linear(maps[0], H, W)
    for m in maps[1:]:
        acc = acc + resize_linear(m, H, W)
    mean = acc / np.float32(len(maps))
    e = 1.0 / (1.0 + np.exp(-mean.astype(np.float64)))
    return (e * 255.0).clip(0, 255).astype(np.uint8)


def apply_hed(sd, img_u8):
    H, W = img_u8.shape[:2]
    return edge_u8(logits(sd, img_u8)[0], H, W)


def preprocess_hed(sd, x):
    """ControlNet.preprocess(x, type='hed') for a float [B,3,H,W] tensor -> float32 [B,3,H,W] on the CPU."""
    ys = [torch.from_numpy(apply_hed(sd, to_u8(xi))).float().div(255)[None] for xi in x]
    return torch.stack(ys).repeat(1, 3, 1, 1)
