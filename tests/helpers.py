"""Shared helpers for the parity tests."""
import os

import numpy as np
import torch

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


def save_golden(name, **arrays):
    """Write a fixture.  float32 arrays are stored byte-transposed (all first bytes, then all second bytes, ...): the exponent and
    high mantissa bytes then sit together and deflate ~15 % better, which keeps the fixtures under 1 MB each, losslessly."""
    packed = {}
    for k, a in arrays.items():
        a = np.asarray(a)
        if a.dtype == np.float32 and a.ndim > 0:
            packed[k + '__bytes'] = np.ascontiguousarray(a).view(np.uint8).reshape(-1, 4).T.copy()
            packed[k + '__shape'] = np.array(a.shape, np.int64)
        else:
            packed[k] = a
    np.savez_compressed(os.path.join(GOLDEN_DIR, f'{name}.npz'), **packed)


def load_golden(name):
    with np.load(os.path.join(GOLDEN_DIR, f'{name}.npz')) as z:
        out = {k: z[k] for k in z.files}
    for k in [k for k in out if k.endswith('__bytes')]:
        base = k[:-len('__bytes')]
        out[base] = np.ascontiguousarray(out.pop(k).T).view(np.float32).reshape(tuple(out.pop(base + '__shape')))
    return out


def range_rel_err(a, ref):
    """max|a - ref| / max|ref| -- the parity metric used everywhere in this repo (SURVEY.md section 7: per-pixel
    relative error is ill-conditioned at zero crossings, so errors are normalised by the reference's range)."""
    a = torch.as_tensor(a, dtype=torch.float64)
    ref = torch.as_tensor(ref, dtype=torch.float64)
    return ((a - ref).abs().max() / ref.abs().max().clamp_min(1e-30)).item()


def pixel_rel_err(a, ref, floor=1e-3):
    """north_star's literal metric: max over elements of |a - ref| / max(|ref|, floor * max|ref|) -- per-pixel relative error with an
    absolute floor so that zero crossings do not divide by ~0.  Returned together with the fraction of elements above 1e-3."""
    a = torch.as_tensor(a, dtype=torch.float64)
    ref = torch.as_tensor(ref, dtype=torch.float64)
    den = ref.abs().clamp_min(floor * ref.abs().max().clamp_min(1e-30))
    e = (a - ref).abs() / den
    return e.max().item(), (e > 1e-3).double().mean().item()


def report_parity(name, a, ref):
    """Both parity metrics of one output; appended to gpurun_out/parity_report.jsonl when that directory exists (so a GPU run
    leaves the numbers behind for profiles/).  -> (range_rel, pixel_rel_max, pixel_rel_frac_above_1e-3)."""
    import json
    r = range_rel_err(a, ref)
    pmax, pfrac = pixel_rel_err(a, ref)
    out = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'gpurun_out')
    if os.path.isdir(out):
        with open(os.path.join(out, 'parity_report.jsonl'), 'a') as f:
            f.write(json.dumps({'case': name, 'range_rel_err': r, 'pixel_rel_err_max_floor1e-3': pmax, 'pixel_frac_above_1e-3': pfrac}) + '\n')
    return r, pmax, pfrac
