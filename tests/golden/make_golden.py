"""Generate golden fixtures by running the REAL reference (imported through oracle/ref_shim.py, which needs a checkout of
the reference project) on seeded synthetic weights and inputs:

    python tests/golden/make_golden.py [name ...]

What the reference executes: its own TriPlaneGenerator.mapping + .synthesis on CPU (every torch_utils.ops call
takes its `_ref` branch, fp32), with (a) our seeded state dict loaded via load_state_dict, (b) the sampler's
uniforms injected, (c) our CPU restatement standing in for the absent pytorch3d rasterizer, (d) a synthetic
all-ones eye mask.  Outputs are stored subsampled so the fixtures stay small:
  image_raw, image_depth (full), image[..., ::4, ::4], face index buffer of sample 0 (int16, -1 = empty),
  alpha planes checksum, mouth boxes, and strided samples of the blended tri-planes (hooked from the renderer).

`reference_checks` stores, for the tests that pin the oracle and the drivers against the reference's own functions, the inputs
those tests feed and what the reference returned for them, plus the reference's parameter / buffer / state-dict names and shapes
and its demo FLAME frame (demo.obj.gz, demo_kpt2d.txt), so that the comparisons run without the reference.
"""
import math
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from next3d_b200 import config, weights  # noqa: E402
from oracle import ref_shim  # noqa: E402
from tests.helpers import save_golden  # noqa: E402

CASES = {
    # name: (config factory, img_resolution, batch, seed)
    'tiny512_b2': (config.tiny_config, 512, 2, 0),
    'tiny256_b1': (config.tiny_config, 256, 1, 1),      # BASELINE.json configs[0]: 64^2 -> 256^2 (4X SR head)
    'full512_b1': (config.full_config, 512, 1, 0),      # BASELINE.json configs[1] shapes, batch 1
}


def run_case(name):
    factory, res, batch, seed = CASES[name]
    cfg = factory(res)
    G = ref_shim.build_reference_generator(cfg)
    sd = weights.make_state_dict(cfg, seed=seed)
    G.load_state_dict(sd)
    z, c_cond, c_cam, v = weights.demo_inputs(cfg, batch, seed=seed)
    u_c, u_f = weights.sampler_noise(cfg, batch, seed=seed)
    captured = {}
    orig = G.renderer.forward

    def hook(planes, *a, **k):
        captured['planes'] = planes.detach().clone()
        return orig(planes, *a, **k)

    G.renderer.forward = hook
    with torch.no_grad():
        ws = G.mapping(z, c_cond, truncation_psi=0.7, truncation_cutoff=14)
        with ref_shim.injected_sampler_noise(u_c, u_f):
            out = G.synthesis(ws, c_cam, v, noise_mode='const')
    planes = captured['planes']
    save_golden(
        name,
        ws=ws.numpy(),
        image_raw=out['image_raw'].numpy(),
        image_depth=out['image_depth'].numpy(),
        image_s4=out['image'][..., ::4, ::4].numpy(),
        image_absmax=np.float32(out['image'].abs().max().item()),
        image_sum=np.float64(out['image'].double().sum().item()),
        planes_s8=planes[..., ::8, ::8].numpy(),
        planes_sum=np.float64(planes.double().sum().item()),
    )
    print(name, 'image', tuple(out['image'].shape), 'range', out['image'].min().item(), out['image'].max().item())


# parameters of the op checks in tests/test_oracle_vs_reference.py
UPFIRDN_CASES = [(1, 1, [1, 1, 1, 1]), (2, 1, [2, 1, 2, 1]), (1, 2, [1, 1, 1, 1]), (1, 1, [2, 2, 2, 2]), (2, 2, [3, 0, 1, 2]),
                 (1, 1, [-1, 0, 0, -1])]
CONV_RESAMPLE_CASES = [(3, 2, 1, False), (3, 1, 2, True), (3, 1, 1, True), (1, 1, 1, True)]
CAMERA_VIEWS = [(math.pi / 2, math.pi / 2), (math.pi / 2 + 0.4, math.pi / 2 - 0.2), (0.3, 1e-7), (3.0, 3.2)]
ORBIT_FRAMES = 24
SAMPLE_GRIDS = {17: 1, 64: 61}                      # N -> stride of the stored sample of the N^3 grid


def grid_slices(N):
    """(head, count) chunks of the N^3 sample grid that the chunked generator is checked on."""
    return [(head, min(n, N ** 3 - head)) for head, n in [(0, 1000), (N ** 3 - 777, 777), (12345 % N ** 3, 2048)]]


def grid_sample_index(N):
    idx = set(range(0, N ** 3, SAMPLE_GRIDS[N]))
    for head, n in grid_slices(N):
        idx.update(range(head, head + n))
    return np.array(sorted(idx), np.int64)
SYNTH_SEED = 3                                      # tiny 512^2 config, batch 2, mesh jittered by 1e-4


def key(*parts):
    return '_'.join(str(p).replace('-', 'm') for p in parts)


def fill_mouth_input():
    a = torch.zeros(3, 1, 64, 64)
    a[:, :, 10:50, 12:52] = 1.0
    a[0, :, 25:30, 20:40] = 0.0                      # hole
    a[1, :, 20:24, 20:24] = 0.5                      # interior fractional patch
    a[1, :, 40:44, 30:34] = 0.0
    a[2, :, :5, :5] = 1.0                            # corner covered
    a[2, :, 30:33, 30:36] = 0.0
    return (a + torch.nn.functional.avg_pool2d(a, 3, 1, 1)) / 2   # fractional edges


def run_reference_checks():
    import gzip
    import json
    import shutil
    from oracle import ops as oo
    ref_shim.import_reference()
    from torch_utils import misc
    from torch_utils.ops import bias_act, upfirdn2d, conv2d_resample, filtered_lrelu
    import training_avatar_texture.networks_stylegan2 as sg2
    import training_avatar_texture.volumetric_rendering.renderer as rr
    import camera_utils
    with ref_shim.in_scratch():
        import gen_samples_next3d
        import gen_videos_next3d
    out = {}

    g = torch.Generator().manual_seed(0)
    x = torch.randn(3, 7, 5, 6, generator=g) * 3
    b = torch.randn(7, generator=g)
    out.update(bias_act_x=x, bias_act_b=b)
    for act in oo.ACTIVATIONS:
        for i, (gain, clamp) in enumerate([(None, None), (0.7, 0.5)]):
            out[key('bias_act', act, i)] = bias_act.bias_act(x, b, act=act, gain=gain, clamp=clamp, impl='ref')

    g = torch.Generator().manual_seed(1)
    x = torch.randn(2, 5, 9, 12, generator=g)
    f = upfirdn2d.setup_filter([1, 3, 3, 1])
    out.update(upfirdn2d_x=x, filter=f, upsample2d=upfirdn2d.upsample2d(x, f, impl='ref'),
               downsample2d=upfirdn2d.downsample2d(x[..., :8, :], f, impl='ref'))
    for up, down, pad in UPFIRDN_CASES:
        out[key('upfirdn2d', up, down, *pad)] = upfirdn2d.upfirdn2d(x, f, up=up, down=down, padding=pad, gain=up * up, impl='ref')

    for k, up, down, flip in CONV_RESAMPLE_CASES:
        g = torch.Generator().manual_seed(2)
        x = out['conv2d_resample_x'] = torch.randn(2, 6, 8, 8, generator=g)
        w = torch.randn(4, 6, k, k, generator=g)
        out[key('conv2d_resample_w', k, up, down, flip)] = w
        out[key('conv2d_resample', k, up, down, flip)] = conv2d_resample.conv2d_resample(x, w, f=f, up=up, down=down, padding=k // 2,
                                                                                        flip_weight=flip)

    g = torch.Generator().manual_seed(3)
    x, w, s = torch.randn(2, 6, 8, 8, generator=g), torch.randn(4, 6, 3, 3, generator=g), torch.randn(2, 6, generator=g)
    noise = torch.randn(16, 16, generator=g)
    out.update(modconv_x=x, modconv_w=w, modconv_s=s, modconv_noise=noise,
               modulated_conv2d=sg2.modulated_conv2d(x, w, s, noise=noise, up=2, padding=1, resample_filter=f, flip_weight=False))

    g = torch.Generator().manual_seed(4)
    x, b = torch.randn(2, 3, 10, 10, generator=g), torch.randn(3, generator=g)
    out.update(filtered_lrelu_x=x, filtered_lrelu_b=b,
               filtered_lrelu=filtered_lrelu.filtered_lrelu(x, fu=f, fd=f, b=b, up=2, down=2, padding=3, impl='ref'))

    a = fill_mouth_input()
    out.update(fill_mouth_alpha=a, fill_mouth=rr.fill_mouth(a))

    # cameras (camera_utils.py:68-86, 140-151) and the orbit of gen_videos_next3d.py:128-140
    lookat = torch.tensor([0, 0, 0.2])
    for i, (h, v) in enumerate(CAMERA_VIEWS):
        out[key('look_at', i)] = camera_utils.LookAtPoseSampler.sample(h, v, lookat, radius=2.7)[0]
    out['fov_intrinsics'] = camera_utils.FOV_to_intrinsics(18.837)
    F = ORBIT_FRAMES
    out['orbit_poses'] = torch.cat([camera_utils.LookAtPoseSampler.sample(3.14 / 2 + 0.35 * np.sin(2 * 3.14 * f / (F // 2)),
                                                                          3.14 / 2 - 0.05 + 0.25 * np.cos(2 * 3.14 * f / (F // 2)),
                                                                          lookat, radius=2.7) for f in range(F)])

    g = torch.Generator().manual_seed(1)
    img = torch.randn(2, 3, 8, 8, generator=g) * 1.5
    out['layout_grid_x'] = img
    out['layout_grid'] = np.stack([gen_videos_next3d.layout_grid(img[k:k + 1], grid_w=1, grid_h=1) for k in range(2)])
    for N in SAMPLE_GRIDS:
        idx = grid_sample_index(N)
        out[key('create_samples', N)] = gen_samples_next3d.create_samples(N=N, voxel_origin=[0, 0, 0], cube_length=1.0)[0][:, idx]

    # the reference's full synthesis on the oracle's inputs (tiny config, batch 2)
    cfg = config.tiny_config(512)
    G = ref_shim.build_reference_generator(cfg)
    sd = weights.make_state_dict(cfg, seed=SYNTH_SEED)
    G.load_state_dict(sd)
    z, c_cond, c_cam, v = weights.demo_inputs(cfg, 2, seed=SYNTH_SEED, jitter=1e-4)
    u_c, u_f = weights.sampler_noise(cfg, 2, seed=SYNTH_SEED)
    with torch.no_grad():
        ws = G.mapping(z, c_cond, truncation_psi=0.7, truncation_cutoff=14)
        with ref_shim.injected_sampler_noise(u_c, u_f):
            r = G.synthesis(ws, c_cam, v, noise_mode='const')
    out.update(synthesis_ws=ws, synthesis_image_s4=r['image'][..., ::4, ::4], synthesis_image_absmax=np.float32(r['image'].abs().max()),
               synthesis_image_raw=r['image_raw'], synthesis_image_depth=r['image_depth'])
    save_golden('reference_checks', **{k: (t.numpy() if isinstance(t, torch.Tensor) else t) for k, t in out.items()})

    # names and shapes the reference's loaders see (torch_utils/misc.py:153-167, module.state_dict())
    G_ref = ref_shim.build_reference_generator(cfg)
    names = {'params_and_buffers': [[n, list(t.shape)] for n, t in misc.named_params_and_buffers(G_ref)],
             'state_dict': [[n, list(t.shape)] for n, t in G_ref.state_dict().items()]}
    with open(os.path.join(ROOT, 'tests', 'golden', 'reference_state_dict.json'), 'w') as fh:
        json.dump(names, fh, indent=0)
        fh.write('\n')

    demo = os.path.join(ref_shim.REF_ROOT, 'data', 'demo')
    with open(os.path.join(demo, 'demo.obj'), 'rb') as src, gzip.GzipFile(os.path.join(ROOT, 'tests', 'golden', 'demo.obj.gz'), 'wb', 9, mtime=0) as dst:
        shutil.copyfileobj(src, dst)
    shutil.copyfile(os.path.join(demo, 'demo_kpt2d.txt'), os.path.join(ROOT, 'tests', 'golden', 'demo_kpt2d.txt'))


if __name__ == '__main__':
    for n in (sys.argv[1:] or list(CASES) + ['reference_checks']):
        if n == 'reference_checks':
            run_reference_checks()
        else:
            run_case(n)
