"""Time ControlNet.preprocess(type='hed') per image on the GPU at 512^2, 768x1024 and 1536^2 against an eager fp32
stand-in of the reference's path, in the same process:
  pfd    pfd_b200.hed.run: fp16 tcgen05 convs, GPU projections / resize / sigmoid (includes the overflow check's sync);
  eager  the same network as torch fp32 nn.Conv2d on the GPU (torch defaults, so cuDNN may use TF32), the five maps
         copied to the host, then cv2.resize (numpy INTER_LINEAR if cv2 is absent), mean, sigmoid and uint8 on the CPU,
         one image at a time, as apply_hed does (hed/__init__.py:115-128).
Both use the seeded synthetic weights of oracle/hed_oracle.py.  Reports ms/image, achieved TFLOP/s of the network's
convolutions (2 FLOP per MAC, computed from the shapes) and the pixel agreement of the two arms.

    python tools/hed_perf.py [--iters N] [--out result.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import hed_oracle as O  # noqa: E402
from pfd_b200 import hed  # noqa: E402

SIZES = ((512, 512), (768, 1024), (1536, 1536))


def flops(H, W):
    total = 0
    for k, (cin, cout, n) in enumerate(O.BLOCKS):
        h, w = H >> k, W >> k
        for i in range(n):
            total += 2 * 9 * (cin if i == 0 else cout) * cout * h * w
        total += 2 * cout * h * w
    return total


class Eager(torch.nn.Module):
    def __init__(self, sd):
        super().__init__()
        self.sd = {k: v.cuda().float() for k, v in sd.items()}

    def forward(self, u8):
        h = u8 - self.sd["norm"]
        maps = []
        for k, (_, _, n) in enumerate(O.BLOCKS, 1):
            if k > 1:
                h = F.max_pool2d(h, 2, 2)
            for i in range(n):
                h = F.relu(F.conv2d(h, self.sd[f"block{k}.convs.{i}.weight"], self.sd[f"block{k}.convs.{i}.bias"],
                                    padding=1))
            maps.append(F.conv2d(h, self.sd[f"block{k}.projection.weight"], self.sd[f"block{k}.projection.bias"]))
        return maps


def eager_preprocess(model, x, resize):
    """controlnet.py:370-376 with apply_hed's body: per image, network on the GPU, tail on the host."""
    ys = []
    for xi in x:
        u8 = xi.mul(255).byte().float()[None]                          # ToPILImage -> np.array -> float
        H, W = u8.shape[2:]
        maps = [m.cpu().numpy().astype(np.float32)[0, 0] for m in model(u8)]
        e = np.stack([resize(m, H, W) for m in maps], axis=2)
        e = 1 / (1 + np.exp(-np.mean(e, axis=2).astype(np.float64)))
        ys.append(torch.from_numpy((e * 255.0).clip(0, 255).astype(np.uint8)).float().div(255)[None])
    return torch.stack(ys).repeat(1, 3, 1, 1).to(x.device)


def timed(fn, iters):
    fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(iters):
        out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / iters * 1e3, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("hed_perf.py needs a CUDA device")
    try:
        import cv2
        resize = lambda m, H, W: cv2.resize(m, (W, H), interpolation=cv2.INTER_LINEAR)  # noqa: E731
        tail = "cv2.resize"
    except ImportError:
        resize, tail = O.resize_linear, "numpy INTER_LINEAR"
    gpu = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    sd = O.synth_state_dict(seed=0)
    hed.set_network(sd)
    model = Eager(sd)
    rows = []
    print(f"[hed_perf] {gpu}, power limit {power}; eager host tail: {tail}; {args.iters} timed iterations per arm")
    for H, W in SIZES:
        g = torch.Generator().manual_seed(H + W)
        x = F.avg_pool2d(torch.rand((1, 3, H, W), generator=g), 7, 1, 3).cuda()
        x = (x - x.min()) / (x.max() - x.min())
        # alternate the arms so drift on a shared machine hits both alike
        t_pfd, t_eager = [], []
        for _ in range(2):
            t, a = timed(lambda: hed.run(x), args.iters)
            t_pfd.append(t)
            t, b = timed(lambda: eager_preprocess(model, x, resize), max(2, args.iters // 4))
            t_eager.append(t)
        tp, te = min(t_pfd), min(t_eager)
        d = (a - b).abs().mul(255)
        row = {"H": H, "W": W, "gflop": flops(H, W) / 1e9, "pfd_ms": tp, "eager_ms": te,
               "pfd_tflops": flops(H, W) / tp / 1e9, "eager_tflops": flops(H, W) / te / 1e9, "speedup": te / tp,
               "max_diff_lsb": float(d.max()), "pixels_differ": float((d > 0.5).float().mean())}
        rows.append(row)
        print(f"[hed_perf] {H}x{W}: {row['gflop']:.0f} GFLOP  pfd {tp:.2f} ms ({row['pfd_tflops']:.0f} TFLOP/s)  "
              f"eager fp32 {te:.2f} ms ({row['eager_tflops']:.0f} TFLOP/s)  speed-up {row['speedup']:.1f}x  "
              f"outputs: max {row['max_diff_lsb']:.0f} LSB, {100 * row['pixels_differ']:.2f}% of pixels differ")
    hed.set_network(None)
    if args.out:
        with open(args.out, "w") as f:
            json.dump({"gpu": gpu, "power_limit": power, "eager_tail": tail, "rows": rows}, f, indent=1)


if __name__ == "__main__":
    main()
