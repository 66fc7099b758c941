"""ControlNet (model part) on the pfd_b200 kernels — mirrors lib/model_zoo/controlnet.py:66-324.

Same constructor arguments / state-dict keys as the reference (spatial-transformer configuration,
`legacy=False`).  ``forward`` returns the 13 residuals as channel-last tensors for
``UNetModel2D_Next.apply(control=...)``.  The hint stem (controlnet.py:165-181) depends only on the
control image, so its output is cached per hint tensor instead of being recomputed every DDIM step.
``preprocess`` provides the annotator-free types on the GPU ('input', 'canny' — bit-exact cv2.Canny,
SURVEY.md §8 f1) and the HED soft-edge network ('hed', pfd_b200/hed.py); the other annotator networks
(controlnet.py:361-503) are outside the path.
"""
from __future__ import annotations

from typing import List, Optional, Tuple

import torch
import torch.nn as nn

from . import native as nv
from .modules import Conv2d, IndexedSequential, Linear, pk_conv3, pk_conv3_small, pk_lin
from .unet import (Downsample, ResBlock, SpatialTransformer, batched_emb_layers, context_kv, run_resblock,
                   run_spatial_transformer, time_embed_silu)

_HINT_STEM = [(16, 1), (16, 1), (32, 2), (32, 1), (96, 2), (96, 1), (256, 2)]


class ControlNet(nn.Module):
    def __init__(self, image_size, in_channels, model_channels, hint_channels, num_res_blocks,
                 attention_resolutions, dropout=0, channel_mult=(1, 2, 4, 8), conv_resample=True, dims=2,
                 use_checkpoint=False, use_fp16=False, num_heads=-1, num_head_channels=-1,
                 num_heads_upsample=-1, use_scale_shift_norm=False, resblock_updown=False,
                 use_new_attention_order=False, use_spatial_transformer=False, transformer_depth=1,
                 context_dim=None, n_embed=None, legacy=True, disable_self_attentions=None,
                 num_attention_blocks=None, disable_middle_self_attn=False, use_linear_in_transformer=False):
        super().__init__()
        if not use_spatial_transformer or context_dim is None or dims != 2 or use_scale_shift_norm or \
                resblock_updown or transformer_depth != 1 or use_linear_in_transformer:
            raise NotImplementedError("pfd_b200.ControlNet supports the configuration of "
                                      "configs/model/controlnet.yaml (spatial transformer, depth 1)")
        if isinstance(context_dim, (list, tuple)):
            context_dim = context_dim[0]
        if num_heads == -1:
            assert num_head_channels != -1
        self.dims, self.image_size = dims, image_size
        self.in_channels, self.model_channels = in_channels, model_channels
        if isinstance(num_res_blocks, int):
            num_res_blocks = len(channel_mult) * [num_res_blocks]
        self.num_res_blocks = list(num_res_blocks)
        self.attention_resolutions = list(attention_resolutions)
        self.channel_mult = list(channel_mult)
        self.num_heads, self.num_head_channels = num_heads, num_head_channels
        ted = model_channels * 4
        self.time_embed = IndexedSequential(Linear(model_channels, ted), nn.SiLU(), Linear(ted, ted))
        self.input_blocks = nn.ModuleList([IndexedSequential(Conv2d(in_channels, model_channels, 3, padding=1))])
        self.zero_convs = nn.ModuleList([self.make_zero_conv(model_channels)])
        stem, cin = [], hint_channels
        for cout, s in _HINT_STEM:
            stem += [Conv2d(cin, cout, 3, padding=1, stride=s), nn.SiLU()]
            cin = cout
        stem.append(Conv2d(cin, model_channels, 3, padding=1))
        self.input_hint_block = IndexedSequential(*stem)

        def heads_of(ch):
            if num_head_channels == -1:
                return num_heads, ch // num_heads
            return ch // num_head_channels, num_head_channels

        ch, ds = model_channels, 1
        for level, mult in enumerate(channel_mult):
            for _ in range(self.num_res_blocks[level]):
                layers = [ResBlock(ch, ted, dropout, out_channels=mult * model_channels)]
                ch = mult * model_channels
                if ds in attention_resolutions:
                    nh, dh = heads_of(ch)
                    layers.append(SpatialTransformer(ch, nh, dh, context_dim=context_dim))
                self.input_blocks.append(IndexedSequential(*layers))
                self.zero_convs.append(self.make_zero_conv(ch))
            if level != len(channel_mult) - 1:
                self.input_blocks.append(IndexedSequential(Downsample(ch, out_channels=ch)))
                self.zero_convs.append(self.make_zero_conv(ch))
                ds *= 2
        nh, dh = heads_of(ch)
        self.middle_block = IndexedSequential(ResBlock(ch, ted, dropout),
                                              SpatialTransformer(ch, nh, dh, context_dim=context_dim),
                                              ResBlock(ch, ted, dropout))
        self.middle_block_out = self.make_zero_conv(ch)

    def make_zero_conv(self, channels):
        return IndexedSequential(Conv2d(channels, channels, 1, padding=0))

    # -------------------------------------------------------------------------------------------
    def _all_resblocks(self) -> List[ResBlock]:
        rbs = [l for blk in self.input_blocks for l in blk if isinstance(l, ResBlock)]
        return rbs + [self.middle_block[0], self.middle_block[2]]

    def _transformers(self) -> List[SpatialTransformer]:
        sts = [l for blk in self.input_blocks for l in blk if isinstance(l, SpatialTransformer)]
        return sts + [self.middle_block[1]]

    def prepare_context(self, context: torch.Tensor) -> List[Tuple[torch.Tensor, torch.Tensor]]:
        return [context_kv(st, context) for st in self._transformers()]

    def hint_features(self, hint: torch.Tensor) -> torch.Tensor:
        """input_hint_block(hint) -> channel-last [1|B, H/8, W/8, model_channels] (controlnet.py:165-181)."""
        h = nv.nchw_to_nhwc(hint.to(torch.float16) if hint.dtype != torch.float32 else hint)
        convs = [m for m in self.input_hint_block if isinstance(m, Conv2d)]
        for i, conv in enumerate(convs):
            act = nv.ACT_SILU if i < len(convs) - 1 else nv.ACT_NONE
            s = conv.stride[0]
            B, H, W, C = h.shape
            if C % 8 == 0 and C >= 16:
                w, b = pk_conv3(conv)
                h = nv.conv3x3(h, w, b, stride=s, act=act)
            else:
                w, b, kpad = pk_conv3_small(conv)
                col = nv.im2col3x3(h, kpad, stride=s)
                Ho, Wo = col.shape[1], col.shape[2]
                h = nv.linear(col.reshape(B * Ho * Wo, kpad), w, b, act=act).reshape(B, Ho, Wo, w.shape[0])
        return h

    def forward(self, x, hint, timesteps, context, kv=None, hint_feat=None, **kwargs) -> List[torch.Tensor]:
        """controlnet.py:302-324.  x NCHW latents; returns 13 channel-last residuals."""
        nv.gn_reset()
        x = x.to(torch.float16)
        context = context.to(torch.float16).contiguous()
        silu_emb = time_embed_silu(self.time_embed, timesteps, self.model_channels)
        rbs = self._all_resblocks()
        embs = {id(rb): e for rb, e in zip(rbs, batched_emb_layers(self, rbs, silu_emb))}
        if kv is None:
            kv = self.prepare_context(context)
        kv_of = {id(st): kvi for st, kvi in zip(self._transformers(), kv)}
        guided = hint_feat if hint_feat is not None else self.hint_features(hint)
        outs = []
        h = nv.nchw_to_nhwc(x)
        for bi, blk in enumerate(self.input_blocks):
            for layer in blk:
                if isinstance(layer, ResBlock):
                    h = run_resblock(layer, h, None, embs[id(layer)])
                elif isinstance(layer, SpatialTransformer):
                    h = run_spatial_transformer(layer, h, context, kv_of[id(layer)])
                elif isinstance(layer, Downsample):
                    w, b = pk_conv3(layer.op)
                    h = nv.conv3x3(h, w, b, stride=2)
                elif isinstance(layer, Conv2d):
                    w, b, kpad = pk_conv3_small(layer)
                    B, H, W, _ = h.shape
                    col = nv.im2col3x3(h, kpad)
                    h = nv.linear(col.reshape(B * H * W, kpad), w, b).reshape(B, H, W, w.shape[0])
            if guided is not None:
                B = h.shape[0]
                if guided.shape[0] == B:
                    h = nv.axpby(h, 1.0, guided, 1.0)
                else:                                                   # hint batch 1 broadcast (controlnet.py:315)
                    for i in range(B):
                        nv.axpby(h[i], 1.0, guided[0], 1.0, out=h[i])
                guided = None
            w, b = pk_lin(self.zero_convs[bi][0])
            outs.append(nv.conv1x1(h, w, b))
        h = run_resblock(self.middle_block[0], h, None, embs[id(self.middle_block[0])])
        h = run_spatial_transformer(self.middle_block[1], h, context, kv_of[id(self.middle_block[1])])
        h = run_resblock(self.middle_block[2], h, None, embs[id(self.middle_block[2])])
        w, b = pk_lin(self.middle_block_out[0])
        outs.append(nv.conv1x1(h, w, b))
        return outs

    @torch.no_grad()
    def preprocess(self, x, type="canny", **kwargs):
        """controlnet.py:332-376 on the GPU for the types: 'none', 'input' / 'shuffle_v11e' (the uint8 round
        trip of ToPILImage -> ToTensor), 'canny' / 'canny_v11p' (cv2.Canny(rgb_u8, low, high), reproduced
        bit-exactly by pfd_canny_f32) and 'hed' / 'softedge_v11p' (the HED soft-edge network, pfd_b200.hed; its
        weights ControlNetHED.pth are read from the reference's locations or set with pfd_b200.hed.set_network;
        images must be at least 16x16).  x: [B,3,H,W] tensor in [0,1] or an image path.  Returns float32
        [B,3,H,W] on x's device.  The other annotators (midas, mlsd, openpose, ...) raise NotImplementedError."""
        if type == "none" or type is None:
            return None
        if isinstance(x, str):
            import numpy as np
            import PIL.Image
            arr = np.array(PIL.Image.open(x).convert("RGB"))
            x = torch.from_numpy(arr).permute(2, 0, 1)[None].to(self.get_device()).to(torch.float32) / 255.0
        elif not isinstance(x, torch.Tensor):
            raise AssertionError("preprocess expects a tensor or an image path")
        if x.shape[1] == 1:
            x = x.repeat(1, 3, 1, 1)
        if not x.is_cuda:
            x = x.to(self.get_device())
        if x.dtype not in (torch.float16, torch.float32):
            x = x.to(torch.float32)
        if type in ("input", "shuffle_v11e"):
            return nv.image_u8_roundtrip(x)
        if type in ("canny", "canny_v11p"):
            low = kwargs.pop("low_threshold", 100)
            high = kwargs.pop("high_threshold", 200)
            out, _ = nv.canny(x, int(low), int(high))
            return out
        if type in ("hed", "softedge_v11p"):
            from . import hed
            return hed.run(x)
        raise NotImplementedError(f"controlnet annotator '{type}' is a separate network outside the pfd_b200 "
                                  "hot path; feed a ready control map (do_preprocess=False)")

    def get_device(self):
        return self.time_embed[0].weight.device

    def get_dtype(self):
        return self.time_embed[0].weight.dtype
