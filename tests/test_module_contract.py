"""CPU: the drop-in TriPlaneGenerator keeps the reference's state-dict contract and API, and refuses to run on CPU."""
import json
import os

import pytest
import torch

from next3d_b200 import config, weights
from oracle import generator as og
from tests.helpers import GOLDEN_DIR


def _tiny():
    from next3d_b200.triplane_next3d import TriPlaneGenerator
    cfg = config.tiny_config(512)
    sd = weights.make_state_dict(cfg, seed=2)
    G = TriPlaneGenerator.from_config(cfg, sd, device='cpu')
    return cfg, sd, G


def test_state_dict_names_and_shapes():
    cfg, sd, G = _tiny()
    got = G.state_dict()
    assert sorted(got.keys()) == sorted(s[0] for s in config.param_spec(cfg)) and len(got) == 674
    for k, v in sd.items():
        assert tuple(got[k].shape) == tuple(v.shape), k
        assert torch.equal(got[k].float(), v.float()), k


def test_mapping_matches_oracle():
    cfg, sd, G = _tiny()
    z, c_cond, _, _ = weights.demo_inputs(cfg, 3, seed=2)
    ws = G.mapping(z, c_cond, truncation_psi=0.7, truncation_cutoff=14)
    ref = og.mapping(sd, cfg, z, c_cond, 0.7, 14)
    assert ws.shape == (3, 28, 512)
    assert (ws - ref).abs().max().item() < 1e-5


def test_no_cpu_fallback():
    cfg, sd, G = _tiny()
    z, c_cond, c_cam, v = weights.demo_inputs(cfg, 1, seed=2)
    ws = G.mapping(z, c_cond)
    with pytest.raises(RuntimeError, match='CUDA'):
        G.synthesis(ws, c_cam, v, noise_mode='const')


def test_reference_state_dict_round_trip():
    """The reference's own loader path: copy_params_and_buffers(G_ref, G_new, require_all=True) (gen_samples_next3d.py:153), then
    G_new.load_state_dict(G_ref.state_dict()), against the names and shapes the reference's TriPlaneGenerator of the same config
    reports (tests/golden/reference_state_dict.json, written by tests/golden/make_golden.py)."""
    cfg, sd, G = _tiny()
    with open(os.path.join(GOLDEN_DIR, 'reference_state_dict.json')) as f:
        ref = {k: {n: tuple(shape) for n, shape in v} for k, v in json.load(f).items()}
    for name, t in list(G.named_parameters()) + list(G.named_buffers()):      # misc.copy_params_and_buffers, require_all=True
        assert name in ref['params_and_buffers'], name
        assert tuple(t.shape) == ref['params_and_buffers'][name], name
    assert {n: tuple(t.shape) for n, t in G.state_dict().items()} == ref['state_dict']
    G.load_state_dict({n: sd[n] for n in ref['state_dict']})


def test_engine_cache_key_tracks_weights_mask_and_options():
    """The packed engine must not go stale: in-place weight updates (load_state_dict / copy_params_and_buffers), a new UV mask and
    pack-time rendering options all change the cache key (checked on CPU through the key alone; the GPU test re-runs synthesis)."""
    cfg, sd, G = _tiny()
    v0 = G._state_version()
    G.load_state_dict(weights.make_state_dict(cfg, seed=5))
    assert G._state_version() != v0
    v1 = G._state_version()
    with torch.no_grad():
        G.state_dict(keep_vars=True)['decoder.net.0.bias'].add_(1.0)
    assert G._state_version() != v1


def test_uv_face_mask_loaded_when_present(tmp_path, monkeypatch):
    """triplane_next3d.py:91-92: channel 0 of cv2.imread (blue) / 255, nearest-resized to 256^2; all ones + a warning when absent."""
    import numpy as np
    from PIL import Image
    from next3d_b200.triplane_next3d import TriPlaneGenerator
    d = tmp_path / 'data' / 'ffhq'
    d.mkdir(parents=True)
    rgb = np.zeros((512, 512, 3), np.uint8)
    rgb[:256, :, 2] = 255                                 # blue channel on in the upper half
    Image.fromarray(rgb).save(d / 'uv_face_eye_mask.png')
    monkeypatch.chdir(tmp_path)
    m = TriPlaneGenerator._load_uv_face_mask()
    assert m.shape == (1, 1, 256, 256) and float(m[0, 0, :128].min()) == 1.0 and float(m[0, 0, 128:].max()) == 0.0
    monkeypatch.chdir(d)                                   # no data/ffhq below this directory
    with pytest.warns(UserWarning, match='all-ones'):
        m = TriPlaneGenerator._load_uv_face_mask()
    assert torch.equal(m, torch.ones(1, 1, 256, 256))
