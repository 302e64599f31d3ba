"""TEST INFRASTRUCTURE ONLY (container-side): import the *real* reference from /root/reference.

The reference (MrTornado24/Next3D) does not import as-is in this image (SURVEY.md Appendix D):
  * `from pydantic import NoneStr`            dnnlib/util.py:26              (removed in pydantic 2)
  * `from turtle import update`               triplane_next3d.py:20          (needs tkinter)
  * `from matplotlib.image import ...`        volumetric_rendering/ray_marcher.py:17
  * `pytorch3d` (io.load_obj, structures.Meshes, renderer.mesh.rasterize_meshes)  renderer.py:25-27
  * `cv2.imread('data/ffhq/uv_face_eye_mask.png')` triplane_next3d.py:91 -- file not shipped
This module installs sys.modules stubs for those, plugs OUR CPU rasterizer restatement
(oracle/rasterize.py, pytorch3d semantics per SURVEY.md Appendix C) in place of pytorch3d, writes
a synthetic eye mask into a scratch cwd, and returns the reference's own TriPlaneGenerator.

It is used ONLY by tests/golden/make_golden.py, which stores what the reference's own code returns
so that the tests pin the oracle restatement against it without a checkout of the reference.
"""
import os
import sys
import types
import contextlib
import tempfile

import numpy as np
import torch

REF_ROOT = '/root/reference'


def available():
    return os.path.isdir(os.path.join(REF_ROOT, 'training_avatar_texture'))


def _install_stubs():
    import pydantic
    pydantic.__dict__.setdefault('NoneStr', type(None))

    def stub(name, **attrs):
        if name in sys.modules and not getattr(sys.modules[name], '_n3d_stub', False):
            return sys.modules[name]
        m = types.ModuleType(name)
        m._n3d_stub = True
        for k, v in attrs.items():
            setattr(m, k, v)
        sys.modules[name] = m
        return m

    stub('turtle', update=None)
    try:
        import matplotlib.image  # noqa: F401
    except Exception:
        stub('matplotlib')
        stub('matplotlib.image', composite_images=None)
    for name in ('imageio', 'mrcfile'):
        try:
            __import__(name)
        except Exception:
            stub(name)

    from collections import namedtuple
    Faces = namedtuple('Faces', 'verts_idx textures_idx')
    Aux = namedtuple('Aux', 'verts_uvs')

    def load_obj(path):
        v, vt, fv, ft = [], [], [], []
        with open(path) as f:
            for line in f:
                if line.startswith('v '):
                    v.append([float(x) for x in line.split()[1:4]])
                elif line.startswith('vt '):
                    vt.append([float(x) for x in line.split()[1:3]])
                elif line.startswith('f '):
                    toks = [t.split('/') for t in line.split()[1:4]]
                    fv.append([int(t[0]) - 1 for t in toks])
                    ft.append([int(t[1]) - 1 for t in toks])
        return (torch.tensor(v, dtype=torch.float32),
                Faces(torch.tensor(fv, dtype=torch.int64), torch.tensor(ft, dtype=torch.int64)),
                Aux(torch.tensor(vt, dtype=torch.float32)))

    class Meshes:
        def __init__(self, verts, faces):
            self.verts, self.faces = verts, faces

    def rasterize_meshes(meshes, image_size, blur_radius, faces_per_pixel, bin_size, max_faces_per_bin,
                         perspective_correct, cull_backfaces):
        from oracle import rasterize as orast
        assert blur_radius == 0.0 and faces_per_pixel == 1 and not perspective_correct and cull_backfaces
        H, W = (image_size, image_size) if isinstance(image_size, int) else image_size
        p2f, zbuf, bary = orast.rasterize_meshes(meshes.verts.numpy(), meshes.faces.numpy(), H, W)
        return (torch.from_numpy(p2f)[..., None], torch.from_numpy(zbuf)[..., None],
                torch.from_numpy(bary)[:, :, :, None, :], None)

    stub('pytorch3d')
    stub('pytorch3d.io', load_obj=load_obj)
    stub('pytorch3d.structures', Meshes=Meshes)
    stub('pytorch3d.renderer')
    stub('pytorch3d.renderer.mesh', rasterize_meshes=rasterize_meshes)


_scratch = None


def scratch_cwd():
    """Scratch dir holding data/ffhq/uv_face_eye_mask.png (synthetic all-255) and data/demo -> reference."""
    global _scratch
    if _scratch is None:
        import cv2
        _scratch = tempfile.mkdtemp(prefix='n3d_refshim_')
        os.makedirs(os.path.join(_scratch, 'data', 'ffhq'))
        cv2.imwrite(os.path.join(_scratch, 'data', 'ffhq', 'uv_face_eye_mask.png'),
                    np.full((256, 256, 3), 255, np.uint8))
        os.symlink(os.path.join(REF_ROOT, 'data', 'demo'), os.path.join(_scratch, 'data', 'demo'))
    return _scratch


@contextlib.contextmanager
def in_scratch():
    old = os.getcwd()
    os.chdir(scratch_cwd())
    try:
        yield
    finally:
        os.chdir(old)


def import_reference():
    assert available(), 'reference tree not present (GPU box?)'
    sys.dont_write_bytecode = True
    _install_stubs()
    if REF_ROOT not in sys.path:
        sys.path.insert(0, REF_ROOT)
    with in_scratch():
        import training_avatar_texture.triplane_next3d as tp
    return tp


def build_reference_generator(cfg):
    """cfg: next3d_b200.config.GeneratorConfig -> reference TriPlaneGenerator (eval, no grad, CPU)."""
    tp = import_reference()
    sr_cls = {'8XDC': 'SuperresolutionHybrid8XDC', '4X': 'SuperresolutionHybrid4X'}[cfg.sr_module]
    rk = dict(cfg.rendering_kwargs)
    rk['superresolution_module'] = f'training_avatar_texture.superresolution.{sr_cls}'
    common = dict(channel_base=cfg.channel_base, channel_max=cfg.channel_max,
                  fused_modconv_default='inference_only')
    with in_scratch():
        G = tp.TriPlaneGenerator(
            z_dim=512, c_dim=25, w_dim=512, img_resolution=cfg.img_resolution, img_channels=3,
            topology_path='data/demo/demo.obj', sr_num_fp16_res=4,
            mapping_kwargs=dict(num_layers=2), rendering_kwargs=rk, sr_kwargs=dict(common),
            num_fp16_res=0, conv_clamp=None, **common)
    return G.eval().requires_grad_(False)


@contextlib.contextmanager
def injected_sampler_noise(u_coarse, u_fine):
    """Replace torch.rand_like / torch.rand inside the reference renderer module by pre-generated uniforms
    (renderer.py:205 `torch.rand_like(depths_coarse)` [N,M,D,1]; renderer.py:252 `torch.rand(N_rays, N_importance)`)."""
    import training_avatar_texture.volumetric_rendering.renderer as rr
    real_torch = rr.torch

    class _T:
        def __getattr__(self, k):
            return getattr(real_torch, k)

        @staticmethod
        def rand_like(x):
            assert tuple(x.shape) == tuple(u_coarse.shape), (x.shape, u_coarse.shape)
            return u_coarse.to(x.dtype)

        @staticmethod
        def rand(*shape, device=None):
            assert tuple(shape) == tuple(u_fine.shape), (shape, u_fine.shape)
            return u_fine

    rr.torch = _T()
    try:
        yield
    finally:
        rr.torch = real_torch
