"""Row f3 of SURVEY.md section 8: native .obj / landmark parsers vs the reference's own parsing code (gen_samples_next3d.py:165-178,
restated below as the oracle), bit-exact in float32.  CPU only."""
import gzip
import os

import numpy as np
import pytest
import torch

from next3d_b200 import inputs
from tests.helpers import GOLDEN_DIR


def ref_parse_obj(path):
    """What gen_samples_next3d.py:165-174 computes, restated: the numbers after the tag of every line whose first two characters
    are 'v ', through float(), flattened to [V, 3] float64, then .float()."""
    rows = [[float(tok) for tok in ln.split()[1:]] for ln in open(path, 'r').read().split('\n') if ln[:2] == 'v ']
    return torch.from_numpy(np.array(rows, dtype=np.float64).reshape(-1, 3)).float()[None]


def _write_obj(path, rng, n=500):
    fmts = ['%.6f', '%.9e', '%g', '%.17g', '%+.3f']
    with open(path, 'w', newline='') as f:
        f.write('# synthetic mesh\nmtllib x.mtl\no face\n')
        for i in range(n):
            xyz = rng.standard_normal(3) * (10.0 ** rng.integers(-6, 6))
            sep = ['  ', ' ', '\t'][i % 3]
            eol = '\r\n' if i % 7 == 0 else '\n'
            f.write('v ' + sep.join(fmts[(i + k) % len(fmts)] % xyz[k] for k in range(3)) + eol)
            if i % 5 == 0:
                f.write('vt %.4f %.4f\nvn 0 0 1\n' % (rng.random(), rng.random()))
        f.write('v -0.0 0 1e-45\nv 1e39 -1e39 3.4028235e38\n')           # signed zero, float32 denormal / overflow to inf
        f.write('f 1/1 2/2 3/3\n')
        f.write('v 1 2 3')                                                # last line without a newline


def test_obj_vertices_bit_exact(tmp_path):
    rng = np.random.default_rng(0)
    p = tmp_path / 'm.obj'
    _write_obj(p, rng)
    ref = ref_parse_obj(p)[0].numpy()
    got = inputs.load_obj_vertices(str(p))
    assert got.dtype == np.float32 and got.shape == ref.shape
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))
    assert np.array_equal(inputs.load_obj_vertices(open(p, 'rb').read()).view(np.uint32), ref.view(np.uint32))


def test_reference_demo_frame(tmp_path):
    """The reference's demo FLAME frame (data/demo/demo.obj, stored gzipped, and data/demo/demo_kpt2d.txt)."""
    obj, lms = tmp_path / 'demo.obj', os.path.join(GOLDEN_DIR, 'demo_kpt2d.txt')
    with gzip.open(os.path.join(GOLDEN_DIR, 'demo.obj.gz'), 'rb') as f:
        obj.write_bytes(f.read())
    obj = str(obj)
    v = ref_parse_obj(obj)
    l = torch.from_numpy(np.loadtxt(lms)).float().unsqueeze(0)
    ref = torch.cat((v, l), 1)                                            # gen_samples_next3d.py:176-178
    got = inputs.load_frame(obj, lms)
    assert got.shape == ref.shape == (1, 5023 + 68, 3)
    assert torch.equal(got, ref)


def test_float_table_like_loadtxt(tmp_path):
    p = tmp_path / 'k.txt'
    p.write_text('# header\n1.5 2.25 -3e-3\n\n  4 5 6   # trailing comment\n7\t8\t9\n')
    ref = np.loadtxt(p).astype(np.float32)
    got = inputs.load_float_table(str(p))
    assert got.shape == ref.shape and np.array_equal(got, ref)
    one = tmp_path / 'one.txt'
    one.write_text('1 2 3\n')
    assert inputs.load_float_table(str(one)).shape == np.loadtxt(one).shape == (3,)


def test_malformed_inputs_raise(tmp_path):
    with pytest.raises(ValueError):
        inputs.load_obj_vertices(b'v 1 2 x3\n')                          # float('x3') raises in the reference too
    with pytest.raises(ValueError):
        inputs.load_obj_vertices(b'v 1 2\n')                             # reshape((-1, 3)) fails in the reference
    with pytest.raises(ValueError):
        inputs.load_float_table(b'1 2 3\n4 5\n')                         # ragged rows: np.loadtxt raises
    assert inputs.load_obj_vertices(b'').shape == (0, 3)


def test_prefetcher_order_and_content(tmp_path):
    rng = np.random.default_rng(1)
    frames = []
    for i in range(7):
        o, k = tmp_path / f'{i}.obj', tmp_path / f'{i}_kpt2d.txt'
        _write_obj(o, rng, n=20 + i)
        np.savetxt(k, rng.standard_normal((68, 3)))
        frames.append((str(o), str(k)))
    got = list(inputs.FramePrefetcher(frames, depth=3, workers=2, pin=False))
    assert len(got) == 7
    for (o, k), t in zip(frames, got):
        ref = torch.cat((ref_parse_obj(o), torch.from_numpy(np.loadtxt(k)).float().unsqueeze(0)), 1)
        assert torch.equal(t, ref)
