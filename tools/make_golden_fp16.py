"""Golden output of the UNMODIFIED reference in eager fp16 on the GPU, config 1 (tests/golden/reference_fp16_c1.npz).

tests/test_configs_gpu.py::test_reference_fp16_floor compares the CUDA path with the reference's fp32 result
(config_outputs.npz) and with the reference's own fp16 result on the same inputs.  The fp16 run needs the reference
tree and a CUDA device, so it is recorded once here: SeeCoder on the 256x256 image of config_inputs(), then 10 DDIM
steps with CFG 2.0 from the seeded x_T, in the reference's modules with the name-seeded synthetic weights in fp16.

    python tools/make_golden_fp16.py [OUT.npz]      # needs the reference tree (tools/ref_harness.py) and a GPU
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import ref_harness as rh  # noqa: E402
from oracle.golden_inputs import config_inputs  # noqa: E402


def main():
    out = os.path.abspath(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden",
                                                                           "reference_fp16_c1.npz"))
    inp = config_inputs()
    cwd = os.getcwd()
    try:
        ref, _ = rh.build_reference_net("pfd_seecoder", fast=True)
        rh.fill_reference_net(ref)
        ref = ref.half()
        ref.to("cuda")
        from lib.model_zoo.ddim import DDIMSampler as RefSampler
        img, xT = inp["c1_img"].cuda().half(), inp["c1_xT"].cuda().half()
        with torch.no_grad():
            ctx = ref.ctx_encode(img, "image")
            real = torch.randn
            torch.randn = lambda *a, **k: xT.clone()
            try:
                x, _ = RefSampler(ref).sample(
                    steps=10, x_info={"type": "image"},
                    c_info={"type": "image", "conditioning": ctx, "unconditional_conditioning": torch.zeros_like(ctx),
                            "unconditional_guidance_scale": 2.0, "control": None},
                    shape=[1, 4, 64, 64], verbose=False, eta=0.0)
            finally:
                torch.randn = real
    finally:
        os.chdir(cwd)
    os.makedirs(os.path.dirname(out), exist_ok=True)
    np.savez_compressed(out, c1_latent=x.cpu().numpy().astype(np.float16),
                        device=np.array(torch.cuda.get_device_name()), torch=np.array(torch.__version__))
    print(f"wrote {out}: latent rms {x.float().pow(2).mean().sqrt():.3f} on {torch.cuda.get_device_name()}", flush=True)


if __name__ == "__main__":
    main()
