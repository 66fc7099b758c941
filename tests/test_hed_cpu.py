"""CPU checks of the HED annotator (ControlNet.preprocess type 'hed' / 'softedge_v11p'): the oracle's cv2-style resize
against cv2 itself, the oracle against the reference's recorded output (tests/golden/hed_reference.npz, written by
tools/make_golden_hed.py from the unmodified apply_hed), the fixture's spread, and the parameter holder's layout."""
import hashlib
import json
import os

import numpy as np
import pytest
import torch

from oracle import hed_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "hed_reference.npz")
CASES = [c[0] for c in O.CASES]


@pytest.fixture(scope="module")
def golden():
    return dict(np.load(GOLDEN))


@pytest.mark.parametrize("src,dst", [((7, 5), (33, 31)), ((12, 20), (200, 328)), ((100, 82), (200, 328)),
                                     ((64, 64), (512, 512)), ((200, 328), (77, 123)), ((33, 31), (16, 15)),
                                     ((2, 1), (33, 31)), ((40, 40), (40, 40))])
def test_resize_matches_cv2_inter_linear(src, dst):
    cv2 = pytest.importorskip("cv2")
    rng = np.random.RandomState(sum(src) + sum(dst))
    m = (rng.randn(*src) * 3).astype(np.float32)
    ref = cv2.resize(m, (dst[1], dst[0]), interpolation=cv2.INTER_LINEAR)
    out = O.resize_linear(m, *dst)
    assert out.shape == ref.shape and out.dtype == np.float32
    assert np.max(np.abs(out - ref)) <= 1e-6 * np.max(np.abs(ref))


def test_golden_images_are_rebuilt_exactly(golden):
    for name in CASES:
        imgs = O.case_images(name)
        assert hashlib.sha256(imgs.tobytes()).hexdigest() == str(golden[f"img_sha256_{name}"]), name
        assert imgs.shape[1:3] == O.golden_edges(golden, name).shape[1:], name


def test_oracle_reproduces_reference_golden(golden):
    sd = O.synth_state_dict(seed=0)
    for name in CASES:
        for img, ref in zip(O.case_images(name), O.golden_edges(golden, name)):
            out = O.apply_hed(sd, img)
            d = np.abs(out.astype(np.int64) - ref)
            assert d.max() <= 1 and np.mean(d == 0) >= 0.999, (name, int(d.max()), float(np.mean(d > 0)))


def test_amplified_weights_keep_the_logits_and_widen_the_range():
    img = O.case_images("33x31")[0]
    maps, amax = O.logits(O.synth_state_dict(seed=0), img)
    maps_a, amax_a = O.logits(O.synth_state_dict(seed=0, amplify_log2=12), img)
    assert amax_a[0] > 65504 > 64 * amax[0]
    assert np.array_equal(O.edge_u8(maps, 33, 31), O.edge_u8(maps_a, 33, 31))


def test_golden_fixture_is_not_degenerate(golden):
    for name in CASES:
        for e in O.golden_edges(golden, name):
            assert len(np.unique(e)) >= 64, name
            assert np.mean((e == 0) | (e == 255)) < 0.05, name


def test_state_dict_layout_matches_reference(golden):
    from pfd_b200.hed import ControlNetHED
    sd = ControlNetHED().state_dict()
    ref_shapes = json.loads(str(golden["sd_shapes"]))
    assert list(sd) == list(golden["sd_keys"])
    assert {k: list(v.shape) for k, v in sd.items()} == ref_shapes
    assert {k: list(v) for k, v in O.state_dict_shapes().items()} == ref_shapes
    ControlNetHED().load_state_dict(O.synth_state_dict(seed=3), strict=True)


def test_controlnet_state_dict_is_unchanged():
    from pfd_b200 import get_model, hed, model_cfg_bank
    with torch.device("meta"):
        before = get_model()(model_cfg_bank()("pfd_seecoder_with_controlnet")).ctl.state_dict()
    try:
        hed.set_network(O.synth_state_dict(seed=0))
        with torch.device("meta"):
            after = get_model()(model_cfg_bank()("pfd_seecoder_with_controlnet")).ctl.state_dict()
    finally:
        hed.set_network(None)
    assert list(after) == list(before)
    assert not any(k.startswith(("norm", "block")) or "projection" in k for k in after)


def test_loader_reads_the_reference_location_and_never_downloads(tmp_path, monkeypatch):
    from pfd_b200 import hed
    monkeypatch.chdir(tmp_path)
    hed.set_network(None)
    with pytest.raises(FileNotFoundError) as e:
        hed.get_network()
    assert os.path.join(str(tmp_path), hed.MODEL_RELPATH) in str(e.value)
    path = tmp_path / hed.MODEL_RELPATH
    path.parent.mkdir(parents=True)
    sd = O.synth_state_dict(seed=2)
    torch.save(sd, str(path))
    try:
        net = hed.get_network()
        assert torch.equal(net.block3.convs[1].weight, sd["block3.convs.1.weight"])
        assert hed.get_network() is net
    finally:
        hed.set_network(None)


def test_small_images_are_rejected():
    from pfd_b200 import hed
    for shape in ((1, 3, 15, 64), (1, 3, 64, 15)):
        with pytest.raises(ValueError):
            hed.run(torch.zeros(shape))
