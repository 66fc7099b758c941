"""Record tests/golden/hed_reference.npz: the reference's own apply_hed (lib/model_zoo/controlnet_annotator/hed/
__init__.py:102-128, loaded unmodified by file path) on the seeded images of oracle/hed_oracle.case_images with the
seeded synthetic HED weights of oracle/hed_oracle.synth_state_dict.  The file holds the uint8 edge maps (row-wise differences, oracle/hed_oracle.golden_edges decodes them), a digest of
each case's input images (the tests rebuild the images and check the digest), and the reference model's state-dict
keys and shapes; not the images or the weights.  Needs the reference tree, cv2 and einops; run from the repository
root:  python tools/make_golden_hed.py <reference_root>
"""
import hashlib
import importlib.util
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle.hed_oracle import CASES, case_images, encode_edges, synth_state_dict  # noqa: E402


def main():
    if len(sys.argv) != 2:
        sys.exit("usage: python tools/make_golden_hed.py <root of the original Prompt-Free-Diffusion checkout>")
    path = os.path.join(sys.argv[1], "lib", "model_zoo", "controlnet_annotator", "hed", "__init__.py")
    spec = importlib.util.spec_from_file_location("reference_hed", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    net = mod.ControlNetHED_Apache2()
    ref_sd = net.state_dict()
    net.load_state_dict(synth_state_dict(seed=0), strict=True)
    mod.netNetwork = net
    out = {"sd_keys": np.array(list(ref_sd)),
           "sd_shapes": np.array(json.dumps({k: list(v.shape) for k, v in ref_sd.items()}))}
    for name, *_ in CASES:
        imgs = case_images(name)
        edges = np.stack([mod.apply_hed(img, device="cpu") for img in imgs])
        out[f"edge_delta_{name}"] = encode_edges(edges)
        out[f"img_sha256_{name}"] = np.array(hashlib.sha256(imgs.tobytes()).hexdigest())
        e = edges.astype(np.int64)
        print(f"{name}: {len(imgs)} image(s), {len(np.unique(e))} levels, "
              f"{100 * np.mean((e == 0) | (e == 255)):.2f}% at 0/255, mean {e.mean():.1f}")
    dst = os.path.join(ROOT, "tests", "golden", "hed_reference.npz")
    np.savez_compressed(dst, **out)
    print(f"wrote {dst} ({os.path.getsize(dst)} bytes)")


if __name__ == "__main__":
    main()
