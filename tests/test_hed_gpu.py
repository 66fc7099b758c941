"""GPU tests of ControlNet.preprocess(type='hed' / 'softedge_v11p') (pfd_b200/hed.py, csrc/hed.cu): parity with the
reference's recorded output (tests/golden/hed_reference.npz), the fp16 range fold, the overflow and size guards,
re-packing on load_state_dict, and the new kernels against their CPU restatements."""
import os

import numpy as np
import pytest
import torch

from oracle import hed_oracle as O

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def golden():
    return dict(np.load(os.path.join(ROOT, "tests", "golden", "hed_reference.npz")))


@pytest.fixture(scope="module")
def net():
    from pfd_b200 import get_model, model_cfg_bank
    n = get_model()(model_cfg_bank()("pfd_seecoder_with_controlnet")).half()
    n.to("cuda")
    n.eval()
    return n


@pytest.fixture
def hed_weights():
    from pfd_b200 import hed
    hed.set_network(O.synth_state_dict(seed=0))
    yield hed
    hed.set_network(None)


def _images(name, dtype):
    """The golden case's uint8 images as [B,3,H,W] tensors in [0,1] whose ToPILImage quantisation gives them back."""
    u8 = torch.from_numpy(O.case_images(name)).permute(0, 3, 1, 2)
    x = ((u8.double() + 0.5) / 255).to(dtype)
    assert torch.equal(x.mul(255).byte(), u8)
    return x.cuda()


def _check(out, ref_u8, what):
    """float32 [B,3,H,W] CUDA output against uint8 [B,H,W] reference maps: all channels equal, every pixel within 1/255,
    at most 3 % of the pixels different (per image)."""
    assert out.dtype == torch.float32 and out.is_cuda and out.shape == (ref_u8.shape[0], 3) + ref_u8.shape[1:], what
    out = out.cpu()
    assert torch.equal(out[:, 0], out[:, 1]) and torch.equal(out[:, 0], out[:, 2]), what
    for b in range(out.shape[0]):
        d = (out[b, 0] * 255 - torch.from_numpy(ref_u8[b]).float()).abs()
        frac = float((d > 0.5).float().mean())
        print(f"[hed] {what} image {b}: max |diff| {float(d.max()):.3f}/255, {100 * frac:.2f}% of pixels differ")
        assert float(d.max()) <= 1.0 + 1e-3, what
        assert frac <= 0.03, what


@pytest.mark.parametrize("name", ["512x512", "200x328", "33x31"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
def test_hed_matches_reference_golden(net, hed_weights, golden, name, dtype):
    x = _images(name, dtype)                                  # 200x328 holds two images: one B=2 call
    for kind in ("hed", "softedge_v11p"):
        _check(net.ctl.preprocess(x, type=kind), O.golden_edges(golden, name), f"{kind} {name} {dtype}")


def test_hed_fold_keeps_amplified_activations_in_fp16(net, hed_weights, golden):
    sd = O.synth_state_dict(seed=0, amplify_log2=12)
    _, amax = O.logits(sd, O.case_images("200x328")[0])
    assert amax[0] > 65504                                            # an unscaled fp16 run would overflow in block 1
    hed_weights.set_network(sd)
    out = net.ctl.preprocess(_images("200x328", torch.float32), type="hed")
    assert torch.isfinite(out).all()
    _check(out, O.golden_edges(golden, "200x328"), "amplified 2^12")


@pytest.mark.parametrize("amplify_log2", [16, 20])
def test_hed_overflow_raises(net, hed_weights, golden, amplify_log2):
    """2^16: activations overflow fp16 even after the 2^-8 fold; 2^20: the first conv's weights do not fit fp16."""
    hed_weights.set_network(O.synth_state_dict(seed=0, amplify_log2=amplify_log2))
    with pytest.raises(RuntimeError, match="not finite"):
        net.ctl.preprocess(_images("33x31", torch.float32), type="hed")


def test_hed_small_images_raise(net, hed_weights):
    for shape in ((1, 3, 15, 40), (2, 3, 40, 8)):
        with pytest.raises(ValueError):
            net.ctl.preprocess(torch.rand(shape, device="cuda"), type="hed")


def test_hed_repacks_after_load_state_dict(net, golden):
    from pfd_b200 import hed
    module = hed.ControlNetHED()
    module.load_state_dict(O.synth_state_dict(seed=0))
    hed.set_network(module)
    try:
        x = _images("33x31", torch.float32)
        a = net.ctl.preprocess(x, type="hed")
        _check(a, O.golden_edges(golden, "33x31"), "seed 0")
        sd1 = O.synth_state_dict(seed=1)
        module.load_state_dict(sd1)
        b = net.ctl.preprocess(x, type="hed")
        assert not torch.equal(a, b)
        _check(b, O.apply_hed(sd1, O.case_images("33x31")[0])[None], "seed 1 after load_state_dict")
    finally:
        hed.set_network(None)


def test_hed_kernels_match_cpu():
    from pfd_b200 import native as nv
    g = torch.Generator().manual_seed(0)
    # max-pool: odd sizes drop the last row / column
    x = torch.randn((2, 9, 13, 64), generator=g).half()
    ref = torch.nn.functional.max_pool2d(x.float().permute(0, 3, 1, 2), 2, 2).permute(0, 2, 3, 1)
    assert torch.equal(nv.maxpool2x2(x.cuda()).float().cpu(), ref)
    # projection: fp32 dot product (+ the inverse activation scale)
    for C in (64, 128, 256, 512):
        x = torch.randn((1, 7, 11, C), generator=g).half()
        w, b = torch.randn(C, generator=g), torch.randn(1, generator=g)
        out = nv.hed_project(x.cuda(), w.cuda(), b.cuda(), 4.0).cpu()
        ref = (x.double() @ w.double()) * 4.0 + b.double()
        assert torch.allclose(out.double(), ref, rtol=1e-5, atol=1e-5), C
    # input: ToPILImage quantisation in the input's dtype, then (u8 - norm) * scale
    x = torch.rand((2, 3, 17, 19), generator=g)
    norm = torch.tensor([120.5, 100.25, 90.0])
    for dt in (torch.float32, torch.float16):
        ref = ((x.to(dt).mul(255).byte().float() - norm[:, None, None]) * 2 ** -8).half().permute(0, 2, 3, 1)
        assert torch.equal(nv.hed_input(x.to(dt).cuda(), norm.cuda(), 2 ** -8).cpu(), ref)
    # fuse: the same fp32 logits give the oracle's edge map
    maps, _ = O.logits(O.synth_state_dict(seed=0), (torch.rand((37, 45, 3), generator=g) * 255).byte().numpy())
    out, bad = nv.hed_fuse([torch.from_numpy(m)[None].cuda() for m in maps], 37, 45)
    ref = O.edge_u8(maps, 37, 45)
    d = (out[0, 0].cpu() * 255 - torch.from_numpy(ref).float()).abs()
    assert int(bad.item()) == 0 and float(d.max()) <= 1.0 + 1e-3 and float((d > 0.5).float().mean()) <= 0.001
