"""Row f1 of SURVEY.md section 8 (batched frame drivers): the frame schedule and the batching logic against the reference's own
per-frame code (gen_videos_next3d.py:96-171, camera_utils.py:68-86), through what that code returned for the same inputs
(tests/golden/reference_checks.npz, written by tests/golden/make_golden.py).  CPU only; the generator is a stub here, the real one
is covered by tests/test_gpu_generator.py (batch invariance)."""
import numpy as np
import pytest
import torch

from next3d_b200 import camera, drivers
from tests.golden.make_golden import CAMERA_VIEWS, ORBIT_FRAMES, grid_sample_index, grid_slices, key
from tests.helpers import load_golden


@pytest.fixture(scope='module')
def ref():
    return {k: torch.from_numpy(v) for k, v in load_golden('reference_checks').items()}


def test_cameras_match_reference_sampler(ref):
    lookat = torch.tensor([0, 0, 0.2])
    for i, (h, v) in enumerate(CAMERA_VIEWS):
        assert torch.equal(camera.look_at_pose(h, v, lookat, 2.7), ref[key('look_at', i)])
    assert torch.equal(camera.fov_to_intrinsics(18.837), ref['fov_intrinsics'])
    # the orbit of gen_videos_next3d.py:128-140, frame by frame
    F = ORBIT_FRAMES
    c = drivers.orbit_camera_params(F, lookat, 2.7)
    intr = torch.tensor([[4.2647, 0, 0.5], [0, 4.2647, 0.5], [0, 0, 1]])
    for f in range(F):
        pose = ref['orbit_poses'][f:f + 1]
        assert torch.equal(c[f], torch.cat([pose.reshape(-1, 16), intr.reshape(-1, 9)], 1)[0])


def test_interpolated_latents_match_per_frame_calls():
    import scipy.interpolate
    g = torch.Generator().manual_seed(0)
    K, w_frames, wraps = 3, 5, 2
    ws = torch.randn(K, 28, 16, generator=g)
    got = drivers.interpolate_ws(ws, w_frames, wraps)
    x = np.arange(-K * wraps, K * (wraps + 1))                            # gen_videos_next3d.py:112-114
    interp = scipy.interpolate.interp1d(x, np.tile(ws.numpy(), [wraps * 2 + 1, 1, 1]), kind='cubic', axis=0)
    for f in range(K * w_frames):
        assert np.array_equal(got[f].numpy(), interp(f / w_frames))      # :143-144
    assert np.allclose(got[::w_frames].numpy(), ws.numpy(), atol=1e-6)    # passes through the key frames


def test_uint8_conversion_is_layout_grid(ref):
    img = ref['layout_grid_x']
    got = drivers.to_uint8_hwc(img)
    for k in range(2):
        assert np.array_equal(got[k].numpy(), ref['layout_grid'][k].numpy())     # gen_videos_next3d.py:35-49, one image per grid


class _StubG(torch.nn.Module):
    """Deterministic stand-in with the generator's call signature: pixel = f(ws, c, v) per sample, independent of the batch."""
    def __init__(self):
        super().__init__()
        self.p = torch.nn.Parameter(torch.zeros(1))
        self.calls = []

    def synthesis(self, ws, c, v, noise_mode='const', seed=None):
        self.calls.append(ws.shape[0])
        s = ws.mean(dim=(1, 2)) + c.mean(dim=1) + v.mean(dim=(1, 2))
        img = torch.tanh(s)[:, None, None, None] * torch.linspace(-1, 1, 48).reshape(1, 3, 4, 4)
        return {'image': img, 'image_depth': s[:, None, None, None].expand(-1, 1, 4, 4) + torch.arange(16.).reshape(1, 1, 4, 4)}


@pytest.mark.parametrize('F,batch,mesh', [(10, 4, 'static'), (8, 8, 'per_frame'), (5, 3, 'iter'), (1, 8, 'static')])
def test_batched_frames_equal_per_frame_loop(F, batch, mesh):
    g = torch.Generator().manual_seed(2)
    ws, cams = torch.randn(F, 28, 16, generator=g), torch.randn(F, 25, generator=g)
    vf = torch.randn(F, 7, 3, generator=g)
    G = _StubG()
    verts = {'static': vf[:1], 'per_frame': vf, 'iter': (vf[i:i + 1] for i in range(F))}[mesh]
    got = list(drivers.render_frames(G, ws, cams, verts, batch=batch, device='cpu'))
    assert len(got) == F and all(n == batch for n in G.calls) and len(G.calls) == -(-F // batch)
    for f in range(F):
        v = vf[:1] if mesh == 'static' else vf[f:f + 1]
        ref = drivers.to_uint8_hwc(_StubG().synthesis(ws[f:f + 1], cams[f:f + 1], v)['image'])[0].numpy()
        assert np.array_equal(got[f], ref)
    depth = list(drivers.render_frames(_StubG(), ws, cams, vf[:1], batch=batch, image_mode='image_depth', device='cpu'))
    assert len(depth) == F and depth[0].shape == (4, 4, 3) and depth[0].max() == 255


# ------------------------------------------------------------------------------------------------ row f2: shape extraction
@pytest.mark.parametrize('N', [17, 64])
def test_chunked_samples_are_slices_of_the_reference_grid(ref, N):
    """gen_samples_next3d.create_samples, stored at the points make_golden.grid_sample_index lists: the whole 17^3 grid, and
    every 61st point of the 64^3 grid plus the chunks checked below."""
    idx = torch.from_numpy(grid_sample_index(N))
    grid = ref[key('create_samples', N)]
    assert torch.equal(drivers.create_samples(N, 1.0)[:, idx], grid)
    for head, n in grid_slices(N):
        pos = torch.searchsorted(idx, torch.arange(head, head + n))
        assert torch.equal(drivers.create_samples(N, 1.0, head, n), grid[:, pos])


def test_large_index_rounding_like_the_reference():
    """Indices above 2^24 are rounded by .float() in the reference; the chunked generator must reproduce that, not fix it."""
    N, head, n = 512, 2 ** 26 + 12345, 4096
    idx = torch.arange(head, head + n, dtype=torch.int64)
    y = (idx.float() / N) % N
    got = drivers.create_samples(N, 1.0, head, n)[0]
    assert torch.equal(got[:, 1], y * (1.0 / (N - 1)) + (-0.5))
    assert (idx.float().long() != idx).any()                              # the rounding really happens in this range


def test_trim_matches_script():
    """flip along axis 0, then a border of int(30 * R / 256) voxels on all six faces set to -1000 (gen_samples_next3d.py:226-238)."""
    R = 64
    g = torch.Generator().manual_seed(3)
    sig = torch.randn(R, R, R, generator=g)
    ref = sig.numpy()[::-1].copy()
    pad = int(30 * R / 256)
    inner = np.zeros((R, R, R), bool)
    inner[pad:R - pad, pad:R - pad, pad:R - pad] = True
    ref[~inner] = -1000
    assert np.array_equal(drivers.trim_sigma_grid(sig.clone(), R).numpy(), ref)


def _make_drive_root(tmp_path, n=6, with_lms=True):
    import json
    rng = np.random.RandomState(0)
    labels = []
    for k in range(n):
        name = f'{k:04d}'
        (tmp_path / f'{name}.png').write_bytes(b'')
        v = rng.randn(11, 3)
        (tmp_path / f'{name}.obj').write_text(''.join(f'v {a:.6f} {b:.6f} {c:.6f}\n' for a, b, c in v) + 'f 1 2 3\n')
        if with_lms:
            (tmp_path / f'{name}_kpt2d.txt').write_text('\n'.join(f'{a:.5f} {b:.5f} {c:.5f}' for a, b, c in rng.randn(68, 3)) + '\n')
        labels.append([f'{name}.png', rng.randn(25).tolist()])
    (tmp_path / 'dataset.json').write_text(json.dumps({'labels': labels}))
    return labels


def test_reenact_schedule_matches_the_script(tmp_path):
    """reenact_avatar_next3d.py:125-160 restated with its own expressions: frame selection, file names, smoothed cameras."""
    import glob
    import os
    labels = _make_drive_root(tmp_path, n=6)
    root = str(tmp_path)
    num_frames = 4
    sch = drivers.reenact_schedule(root, num_frames)
    img_list = sorted(glob.glob(root + '/*.png'))
    want_ids, want_cams = [], []
    for k, img_path in enumerate([img for img in img_list]):                      # the script's loop (:125-131, :159-160)
        if k > num_frames:
            break
        if k < 1:
            continue
        if k + 1 >= len(labels):
            continue
        want_ids.append(os.path.basename(img_list[k]).split('.')[0])
        camera_params = (np.array(labels[k - 1][1]) + np.array(labels[k][1]) + np.array(labels[k + 1][1])) / 3
        want_cams.append(torch.tensor(camera_params).unsqueeze(0).float())
    assert sch['ids'] == want_ids and sch['obj_paths'] == [root + f'/{i}.obj' for i in want_ids]
    assert sch['lms_paths'] == [root + f'/{i}_kpt2d.txt' for i in want_ids]
    assert torch.equal(sch['cams'], torch.cat(want_cams))


def test_frame_pack_round_trip(tmp_path):
    from next3d_b200 import inputs
    _make_drive_root(tmp_path, n=5)
    root = str(tmp_path)
    sch = drivers.reenact_schedule(root, 10)
    verts = np.stack([inputs.load_frame(o, l)[0].numpy() for o, l in zip(sch['obj_paths'], sch['lms_paths'])])
    path = str(tmp_path / 'clip.n3dpack')
    inputs.write_frame_pack(path, verts, sch['cams'].numpy(), ids=sch['ids'])
    pack = inputs.FramePack(path, pin=False)
    assert len(pack) == len(sch['ids']) and pack.ids == sch['ids']
    assert np.array_equal(pack.verts, verts) and np.array_equal(pack.cams, sch['cams'].numpy())
    frames = list(pack)
    assert frames[1].shape == (1, verts.shape[1], 3) and np.array_equal(frames[1][0].numpy(), verts[1])
