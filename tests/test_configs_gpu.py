"""GPU parity at the BASELINE configs' OWN sizes (VERDICT r1 "next round" item 1) against outputs of the UNMODIFIED
reference (fp32, CPU) committed as tests/golden/config_outputs.npz by tools/make_golden_configs.py; the seeded
inputs are regenerated here by oracle/golden_inputs.config_inputs().  Everything goes through the public,
reference-shaped API and therefore through the C-ABI.

Tolerances (BASELINE.json: fp16 path, latent MSE < 1e-3): one network evaluation must agree to relative rms
5e-3 (measured 1-2e-3 = the reference's own fp16-vs-fp32 floor, printed by test_reference_fp16_floor from the
recorded fp16 run of the reference); multi-step / end-to-end results compound that and get 2e-2.
"""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
REL_EVAL, REL_E2E, MSE_TOL = 5e-3, 2e-2, 1e-3


def _metrics(out, ref):
    out, ref = torch.as_tensor(out).detach().float().cpu(), torch.as_tensor(np.asarray(ref)).float()
    mse = (out - ref).pow(2).mean().item()
    return mse, (mse / max(ref.pow(2).mean().item(), 1e-20)) ** 0.5


def _check(name, out, ref, rel_tol=REL_EVAL, mse_tol=MSE_TOL):
    """MSE bar of BASELINE.json (1e-3) is stated for unit-variance SD latents; with the synthetic weights some
    tensors have a larger scale (e.g. 10-step latents rms ~9.5), so the bar is applied to the MSE normalised by
    max(1, mean(ref^2)); the relative rms bound is the sharper assertion either way."""
    mse, rel = _metrics(out, ref)
    ref_ms = float(torch.as_tensor(np.asarray(ref)).float().pow(2).mean())
    nmse = mse / max(1.0, ref_ms)
    print(f"[parity] {name}: mse={mse:.3e} normalised_mse={nmse:.3e} rel_rms={rel:.3e} (tol {rel_tol:.0e}, ref rms {ref_ms ** 0.5:.3f})")
    assert np.isfinite(mse) and nmse < mse_tol and rel < rel_tol, f"{name}: mse={mse:.3e} nmse={nmse:.3e} rel_rms={rel:.3e}"
    return mse, rel


@pytest.fixture(scope="module")
def env():
    from oracle.golden_inputs import config_inputs
    from pfd_b200 import get_model, model_cfg_bank
    from pfd_b200.weights import SCHEDULE_BUFFERS, fill_module_
    net = get_model()(model_cfg_bank()("pfd_seecoder_with_controlnet"))
    fill_module_(net, seed=0, skip=SCHEDULE_BUFFERS)
    net = net.half()
    net.to("cuda")
    net.eval()
    gold = dict(np.load(os.path.join(GOLD, "config_outputs.npz")))
    return net, gold, config_inputs()


def _eps(net, x, t, c, control=None):
    tt = torch.full((x.shape[0],), int(t), dtype=torch.long, device="cuda")
    return net.apply_model({"type": "image", "x": x.cuda().half()}, tt,
                           {"type": "image", "c": c.cuda().half(), "control": control})


def test_config1_end_to_end(env):
    """BASELINE configs[0]: 256x256 reference image -> SeeCoder -> 10 DDIM steps, CFG 2.0, [1,4,64,64] -> VAE 512x512."""
    net, gold, inp = env
    from pfd_b200 import DDIMSampler
    ctx = net.ctx_encode(inp["c1_img"].cuda(), "image")
    _check("cfg1 SeeCoder context (256x256)", ctx, gold["c1_ctx"].astype(np.float32))
    x, inter = DDIMSampler(net).sample(
        steps=10, x_info={"type": "image", "xt": inp["c1_xT"].cuda().half()},
        c_info={"type": "image", "conditioning": ctx, "unconditional_conditioning": torch.zeros_like(ctx),
                "unconditional_guidance_scale": 2.0, "control": None},
        shape=[1, 4, 64, 64], verbose=False, eta=0.0)
    assert len(inter["pred_x0"]) == 2                                     # index 9 and index 0 (ddim.py:122)
    _check("cfg1 latent after 10 steps (own context)", x, gold["c1_latent"], rel_tol=REL_E2E)
    im = net.vae_decode(x, "image")
    assert im.shape == (1, 3, 512, 512) and im.min() >= 0 and im.max() <= 1
    _check("cfg1 image 512x512 (end to end)", im, gold["c1_image"].astype(np.float32), rel_tol=REL_E2E)
    im2 = net.vae_decode(torch.as_tensor(gold["c1_latent"]).cuda().half(), "image")
    _check("cfg1 VAE decode of the reference latent", im2, gold["c1_image"].astype(np.float32))


def test_config2_teacher_forced_eps(env):
    """configs[1] size: B=4 (CFG batch 8) at 64x64 latents, three timesteps across the schedule."""
    net, gold, inp = env
    x = torch.cat([inp["c2_x"]] * 2)
    cond = inp["c2_cond"].repeat(4, 1, 1)
    c = torch.cat([torch.zeros_like(cond), cond])
    for t in inp["c2_t"]:
        _check(f"cfg2 eps B=4 64x64 t={t}", _eps(net, x, t, c), gold[f"c2_eps_t{t}"])


def test_config3_zero_padded_unconditional(env):
    """configs[2]: the anime unconditional context is a [77,768] tensor zero-padded to 148 tokens (app.py:238-241)."""
    net, gold, inp = env
    x = torch.cat([inp["c3_x"]] * 2)
    c = torch.cat([inp["c3_uncond"].repeat(2, 1, 1), inp["c3_cond"].repeat(2, 1, 1)])
    _check("cfg3 eps with padded uncond", _eps(net, x, inp["c3_t"], c), gold["c3_eps"])


def test_config4_controlnet_at_64(env):
    """configs[3]: ControlNet at 64x64 latents with a 512x512 canny-like hint, B=2 (CFG batch 4)."""
    net, gold, inp = env
    x = torch.cat([inp["c4_x"]] * 2).cuda().half()
    cond = inp["c4_cond"].repeat(2, 1, 1)
    c = torch.cat([torch.zeros_like(cond), cond]).cuda().half()
    hint = inp["c4_hint"].cuda().half()
    tt = torch.full((4,), int(inp["c4_t"]), dtype=torch.long, device="cuda")
    outs = net.ctl(x, hint=hint, timesteps=tt, context=c)
    assert len(outs) == 13
    for i, o in enumerate(outs):
        nchw = o.permute(0, 3, 1, 2).float().cpu().reshape(-1)[::97]
        _check(f"cfg4 controlnet residual[{i}]", nchw, gold[f"c4_ctl_{i}_sub"])
    e = net.apply_model({"type": "image", "x": x}, tt, {"type": "image", "c": c, "control": hint})
    _check("cfg4 controlled eps 64x64", e, gold["c4_eps"])


def test_config5_position_aware_768_two_steps(env):
    """configs[4]: PPE_MLP installed (app.py:166-175), 768x768 reference image, 96x96 latents, steps=30 -> 31-entry
    schedule; two teacher-forced p_sample_ddim steps (the second starts from the reference's x after step 0)."""
    net, gold, inp = env
    from pfd_b200 import DDIMSampler
    from pfd_b200.seecoder import PPE_MLP
    from pfd_b200.weights import fill_module_
    pe = PPE_MLP(freq_num=20, freq_max=None, out_channel=768, mlp_layer=3)
    fill_module_(pe, seed=0, prefix="ctx.image.qtransformer.pe_layer.")
    qt = net.ctx["image"].qtransformer
    qt.pe_layer = pe.half().cuda()
    try:
        ctx = net.ctx_encode(inp["c5_img"].cuda(), "image")
    finally:
        qt.pe_layer = None
    _check("cfg5 SeeCoder-PA context (768x768)", ctx, gold["c5_ctx"].astype(np.float32))
    sampler = DDIMSampler(net)
    sampler.make_schedule(ddim_num_steps=30, ddim_eta=0.0, verbose=False)
    ts = sampler.ddim_timesteps
    assert len(ts) == 31
    cref = torch.as_tensor(gold["c5_ctx"].astype(np.float32)).cuda().half()
    x = inp["c5_xT"].cuda().half()
    for i in range(2):
        index = len(ts) - i - 1
        tt = torch.full((1,), int(ts[index]), dtype=torch.long, device="cuda")
        x_info = {"type": "image", "x": x}
        c_info = {"type": "image", "conditioning": cref, "unconditional_conditioning": torch.zeros_like(cref),
                  "unconditional_guidance_scale": 2.0, "control": None}
        x_prev, p0 = sampler.p_sample_ddim(x_info, c_info, tt, index)
        _check(f"cfg5 x after step {i} (96x96 latents, index {index})", x_prev, gold[f"c5_x_step{i}"])
        _check(f"cfg5 pred_x0 step {i}", p0, gold[f"c5_x0_step{i}"])
        x = torch.as_tensor(gold[f"c5_x_step{i}"]).cuda().half()         # teacher forcing


def test_seecoder_512_matches_reference(env):
    """512x512 reference image: feature maps 128/64/32/16 -> padded 12x12 windows at every Swin stage."""
    net, gold, inp = env
    img = inp["c6_img"].cuda()
    fea = net.ctx["image"].imencoder(img)
    for k in ("res3", "res4", "res5"):
        nchw = fea[k].permute(0, 3, 1, 2).contiguous().float().cpu()
        _check(f"cfg2 swin {k} (512x512)", nchw.reshape(-1)[::31], gold[f"c6_swin_{k}_sub"])
    c = net.ctx_encode(img, "image")
    _check("cfg2 SeeCoder context (512x512)", c, gold["c6_ctx"].astype(np.float32))
    c2 = net.ctx_encode(img, "image")                                    # cached-graph replay path
    assert (c.float() - c2.float()).abs().max().item() < 2e-2


class _patched_randn_like:
    def __init__(self, tensors):
        self.q = [t.clone() for t in tensors]

    def __enter__(self):
        self.orig = torch.randn_like
        torch.randn_like = lambda x, *a, **k: self.q.pop(0).to(device=x.device, dtype=x.dtype)
        return self

    def __exit__(self, *e):
        torch.randn_like = self.orig


@pytest.mark.parametrize("graph", [True, False])
def test_eta_sampler_matches_reference(env, graph):
    """eta = 0.5 (ddim.py:168-170): sigma_t * noise added every step, with the reference's noise tensors injected."""
    net, gold, inp = env
    from pfd_b200 import DDIMSampler
    cond = inp["c7_cond"].cuda().half()
    with _patched_randn_like(inp["c7_noise"]):
        x, _ = DDIMSampler(net, use_cuda_graph=graph).sample(
            steps=4, x_info={"type": "image", "xt": inp["c7_xT"].cuda().half()},
            c_info={"type": "image", "conditioning": cond, "unconditional_conditioning": torch.zeros_like(cond),
                    "unconditional_guidance_scale": 2.0, "control": None},
            shape=[1, 4, 16, 16], verbose=False, eta=0.5)
    _check(f"eta=0.5 4-step latent (graph={graph})", x, gold["c7_latent"], rel_tol=REL_E2E)


def test_vae_encode_matches_reference(env):
    """SURVEY §8 f4: AutoencoderKL.encode (asymmetric-pad stride-2 convs) -> posterior mean / logvar / sample."""
    net, gold, inp = env
    img = inp["c8_img"].cuda()
    post = net.vae["image"].encode(img, out_posterior=True)
    _check("vae encode posterior mean (256x256)", post.mean, gold["c8_mean"])
    _check("vae encode posterior logvar", post.logvar, gold["c8_logvar"], rel_tol=2e-2)
    torch.manual_seed(5)
    z = net.vae_encode(img, "image")
    torch.manual_seed(5)
    nz = torch.randn(tuple(z.shape))                                     # the reference's CPU draw (distributions.py:36)
    ref = 0.18215 * (torch.as_tensor(gold["c8_mean"]) + torch.exp(0.5 * torch.as_tensor(gold["c8_logvar"])) * nz)
    _check("vae_encode sample (scaled)", z, ref)


def test_sample_multicontext_matches_reference(env):
    """SURVEY §8 f4: DDIMSampler.sample_multicontext (ddim.py:174-299) / apply_model_multicontext (pfd.py:367-439)."""
    net, gold, inp = env
    from pfd_b200 import DDIMSampler
    ca, cb = inp["c9_cond_a"].cuda().half(), inp["c9_cond_b"].cuda().half()
    mk = lambda c, r: {"type": "image", "conditioning": c, "unconditional_conditioning": torch.zeros_like(c),
                       "unconditional_guidance_scale": 2.0, "ratio": r}
    x, _ = DDIMSampler(net).sample_multicontext(
        steps=4, x_info={"type": "image", "xt": inp["c9_xT"].cuda().half()}, c_info_list=[mk(ca, 0.3), mk(cb, 0.7)],
        shape=[1, 4, 16, 16], verbose=False, eta=0.0)
    _check("multicontext 4-step latent", x, gold["c9_latent"], rel_tol=REL_E2E)


def test_reference_fp16_floor(env):
    """Three-way comparison on config 1's inputs: the UNMODIFIED reference in eager fp16 on a B200 (recorded by
    tools/make_golden_fp16.py in tests/golden/reference_fp16_c1.npz) vs the reference in fp32 (the floor), ours vs
    the fp32 golden, ours vs the reference in fp16 (the north-star's parity statement)."""
    net, gold, inp = env
    x_r = torch.as_tensor(np.load(os.path.join(GOLD, "reference_fp16_c1.npz"))["c1_latent"])
    img, xT = inp["c1_img"].cuda().half(), inp["c1_xT"].cuda().half()
    from pfd_b200 import DDIMSampler
    ctx = net.ctx_encode(img, "image")
    x, _ = DDIMSampler(net).sample(
        steps=10, x_info={"type": "image", "xt": xT},
        c_info={"type": "image", "conditioning": ctx, "unconditional_conditioning": torch.zeros_like(ctx),
                "unconditional_guidance_scale": 2.0, "control": None}, shape=[1, 4, 64, 64], verbose=False, eta=0.0)
    f_mse, f_rel = _metrics(x_r, gold["c1_latent"])
    o_mse, o_rel = _metrics(x, gold["c1_latent"])
    p_mse, p_rel = _metrics(x, x_r.float().cpu())
    print(f"[floor] cfg1 10-step latent: reference fp16 (CUDA eager) vs reference fp32: mse={f_mse:.3e} rel={f_rel:.3e}; "
          f"pfd_b200 vs reference fp32: mse={o_mse:.3e} rel={o_rel:.3e}; pfd_b200 vs reference fp16: mse={p_mse:.3e} rel={p_rel:.3e}")
    ref_ms = max(1.0, float(torch.as_tensor(gold["c1_latent"]).pow(2).mean()))
    assert p_mse / ref_ms < MSE_TOL and o_mse / ref_ms < MSE_TOL
    assert o_rel < max(3.0 * f_rel, REL_EVAL), "pfd_b200 is further from the fp32 reference than 3x the reference's own fp16 error"
