"""CPU: pin the oracle restatement against the reference's own functions, through what those functions returned for the same
inputs (tests/golden/reference_checks.npz, written by tests/golden/make_golden.py from the reference's code)."""
import pytest
import torch

from next3d_b200 import config, weights
from oracle import ops as oo, generator as og
from tests.golden.make_golden import CONV_RESAMPLE_CASES, SYNTH_SEED, UPFIRDN_CASES, key
from tests.helpers import load_golden


@pytest.fixture(scope='module')
def ref():
    return {k: torch.from_numpy(v) for k, v in load_golden('reference_checks').items()}


def test_bias_act_all_activations(ref):
    x, b = ref['bias_act_x'], ref['bias_act_b']
    for act in oo.ACTIVATIONS:
        for i, (gain, clamp) in enumerate([(None, None), (0.7, 0.5)]):
            o = oo.bias_act(x, b, act=act, gain=gain, clamp=clamp)
            assert torch.equal(ref[key('bias_act', act, i)], o), act


@pytest.mark.parametrize('up,down,pad', UPFIRDN_CASES)
def test_upfirdn2d(ref, up, down, pad):
    x, f = ref['upfirdn2d_x'], ref['filter']
    assert torch.equal(f, oo.setup_filter())
    o = oo.upfirdn2d(x, oo.setup_filter(), up=up, down=down, padding=pad, gain=up * up)
    assert torch.equal(ref[key('upfirdn2d', up, down, *pad)], o)
    assert torch.equal(ref['upsample2d'], oo.upsample2d(x, f))
    assert torch.equal(ref['downsample2d'], oo.downsample2d(x[..., :8, :], f))


@pytest.mark.parametrize('k,up,down,flip', CONV_RESAMPLE_CASES)
def test_conv2d_resample(ref, k, up, down, flip):
    x, w = ref['conv2d_resample_x'], ref[key('conv2d_resample_w', k, up, down, flip)]
    f = oo.setup_filter()
    o = oo.conv2d_resample(x, w, f=f, up=up, down=down, padding=k // 2, flip_weight=flip)
    assert torch.equal(ref[key('conv2d_resample', k, up, down, flip)], o)


def test_modulated_conv2d(ref):
    x, w, s, noise = ref['modconv_x'], ref['modconv_w'], ref['modconv_s'], ref['modconv_noise']
    f = oo.setup_filter()
    o = oo.modulated_conv2d(x, w, s, noise=noise, up=2, padding=1, resample_filter=f, flip_weight=False)
    assert torch.equal(ref['modulated_conv2d'], o)


def test_filtered_lrelu(ref):
    x, b, fu = ref['filtered_lrelu_x'], ref['filtered_lrelu_b'], ref['filter']
    o = oo.filtered_lrelu(x, fu=fu, fd=fu, b=b, up=2, down=2, padding=3)
    assert torch.equal(ref['filtered_lrelu'], o)


def test_fill_mouth_vs_cv2(ref):
    """Our BFS restatement == the reference's cv2.floodFill-based fill_mouth, including fractional alphas (the input:
    make_golden.fill_mouth_input)."""
    assert torch.equal(ref['fill_mouth'], og.fill_mouth(ref['fill_mouth_alpha']))


def test_full_synthesis_bit_exact(ref):
    """The reference's mapping + synthesis on the same weights, latents, mesh and sampler uniforms; its image is stored at every
    4th pixel in both directions, together with its largest magnitude."""
    cfg = config.tiny_config(512)
    sd = weights.make_state_dict(cfg, seed=SYNTH_SEED)
    z, c_cond, c_cam, v = weights.demo_inputs(cfg, 2, seed=SYNTH_SEED, jitter=1e-4)
    u_c, u_f = weights.sampler_noise(cfg, 2, seed=SYNTH_SEED)
    with torch.no_grad():
        ws = og.mapping(sd, cfg, z, c_cond, 0.7, 14)
        assert torch.equal(ws, ref['synthesis_ws'])
        o = og.synthesis(sd, cfg, ws, c_cam, v, u_c, u_f)
    image_max = ref['synthesis_image_absmax'].item()
    assert (o['image'][..., ::4, ::4] - ref['synthesis_image_s4']).abs().max().item() <= 1e-6 * image_max
    assert abs(o['image'].abs().max().item() - image_max) <= 1e-6 * image_max
    for k in ('image_raw', 'image_depth'):
        r = ref['synthesis_' + k]
        assert (o[k] - r).abs().max().item() <= 1e-6 * r.abs().max().item(), k


def test_view_transform_is_the_blas_fma_chain():
    """oracle.generator._bmm3_fma (explicit k = 0,1,2 fused chain, float64-emulated) == torch.bmm bit for bit: pins the summation
    order the reference's bmm (renderer.py:505-514) takes on this machine, which the CUDA transform kernel reproduces."""
    g = torch.Generator().manual_seed(0)
    p = torch.randn(3, 5023, 3, generator=g)
    R = torch.randn(3, 3, 3, generator=g)
    assert torch.equal(og._bmm3_fma(p, R), torch.bmm(p, R))
    for view in ((0, 0, 0), (0, 90, 0), (0, -90, 0), (90, 0, 0)):
        Rv = og.angle2matrix(torch.tensor(view, dtype=torch.float32))[None].expand(3, -1, -1)
        assert torch.equal(og._bmm3_fma(p, Rv), torch.bmm(p, Rv))
