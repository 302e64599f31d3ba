#!/usr/bin/env python
"""Benchmark of the hot path: Next3D generator forward (TriPlaneGenerator.synthesis) images/sec on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config c2|c3|c4|c5] [--batch B] [--dump-outputs DIR]

Workloads (BASELINE.json `configs`; seeded random-init weights of the FFHQ-512 architecture (172.8 M parameters), synthetic
latents, the demo FLAME mesh, synthetic all-ones eye mask, noise_mode='const', sampler uniforms from the in-kernel RNG):
  c2 (default, the headline): 64^2 neural render, 48+48 samples per ray -> 512^2 SR, batch 8 per GPU, weak scaling.
  c3: 128^2 neural render, 96+96 samples per ray (gen_videos_next3d.py --sample_mult 2 --nrr 128), batch 16 per GPU.
  c4: one 240-frame clip (gen_videos_next3d.py:128-171: orbit camera, cubic w interpolation, 96+96 samples, 64^2 render) split
      over the N GPUs through drivers.render_frames_sharded (uint8 frames gathered to rank 0, read back to the host): STRONG scaling.
  c5: shape extraction, 256^3 density grid (gen_samples_next3d.py:208-238): tri-plane fetch + decoder only.
A "step" = one synthesis() call on one batch per GPU (c4: the whole clip; c5: one grid).
`value` = whole-job images/s with inputs resident in HBM; `e2e` = the same through the public API with pinned HOST
inputs (H2D inside the timed region) and the final images read back to the host (D2H inside the timed region).
The default N=1 run also reports c3 / c4 / c5 under `other_configs` (short runs; the headline stays c2).
`--dump-outputs DIR` writes what the timed path returned in its last timed step as DIR/<name>.npy (see _dump_outputs); the inputs,
weights and sampler seeds depend only on the arguments, so two builds run with the same arguments can be compared output for output.
`--impl reference` times the CPU oracle port (the reference itself is Python that cannot travel to the GPU box; the oracle
is pinned bit-exactly against it, tests/test_oracle_vs_reference.py) on the host cores.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

UNIT = 'img/s'
CONFIGS = {
    'c2': dict(res=64, depth=48, batch=8,
               metric='generator images/sec at 512^2 (64^2 neural render, 48+48 samples/ray)',
               workload='FFHQ-512 generator forward (TriPlaneGenerator.synthesis): 64^2 neural render -> 512^2 SR, 48+48 depth samples, '),
    'c3': dict(res=128, depth=96, batch=16,
               metric='generator images/sec at 512^2 (128^2 neural render, 96+96 samples/ray)',
               workload='FFHQ-512 generator forward (TriPlaneGenerator.synthesis): 128^2 neural render -> 512^2 SR, 96+96 depth samples (ray-MLP-bound), '),
    'c4': dict(res=64, depth=96, batch=8, frames=240,
               metric='video frames/sec at 512^2 (240-frame clip, 64^2 neural render, 96+96 samples/ray)',
               workload='gen_videos_next3d.py clip: 240 frames (orbit camera, interpolated w, static demo mesh), 96+96 depth samples, frames sharded over the GPUs, '),
    'c5': dict(grid=256,
               metric='shape-extraction density grids/sec (256^3 voxels, tri-plane fetch + decoder)',
               workload='gen_samples_next3d.py --shapes: 256^3 density grid from cached tri-planes, flip + trim fused, '),
}
METRIC = CONFIGS['c2']['metric']
WORKLOAD = CONFIGS['c2']['workload']


def config_for(name):
    """GeneratorConfig of a benchmark configuration (full FFHQ-512 widths)."""
    import copy
    import dataclasses
    from next3d_b200 import config
    base = config.full_config(512)
    rk = copy.deepcopy(base.rendering_kwargs)
    spec = CONFIGS[name]
    if 'depth' in spec:
        rk.update(depth_resolution=spec['depth'], depth_resolution_importance=spec['depth'])
    return dataclasses.replace(base, neural_rendering_resolution=spec.get('res', 64), rendering_kwargs=rk)


_JSON_OUT = None


def _guard_stdout():
    """The contract is ONE JSON line on stdout.  Libraries print to file descriptor 1 behind Python's back (NCCL's version banner,
    for one): keep a private duplicate of the real stdout for the JSON line and point fd 1 at stderr for everything else."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), 'w')
        os.dup2(2, 1)


def _emit(line):
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(line) + '\n')
    out.flush()


DUMP_BYTES = 60 * 10 ** 6       # data of all dumped arrays together; with the .npy headers the dump stays under 64 MB


def _dump_outputs(dirname, arrays):
    """Write {name: tensor or array} as dirname/<name>.npy, float32 (float64 where the output is float64).  The smallest arrays are
    written whole; an array larger than its share of DUMP_BYTES is replaced by a sample of its flattened elements at positions drawn
    from a generator seeded with 0 (sorted; the same positions for the same shape in every run)."""
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    items = sorted(((k, np.asarray(v.detach().cpu() if hasattr(v, 'detach') else v)) for k, v in arrays.items()), key=lambda kv: kv[1].size)
    left = DUMP_BYTES
    for i, (name, a) in enumerate(items):
        dtype = np.float64 if a.dtype == np.float64 else np.float32
        n = left // (len(items) - i) // np.dtype(dtype).itemsize
        if a.size > n:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).integers(0, a.size, n))]
        a = a.astype(dtype)
        np.save(os.path.join(dirname, name + '.npy'), a)
        left -= a.nbytes


def _traffic(kernel):
    """Measured DRAM bytes per launch of `kernel` (dram__bytes_read + dram__bytes_write, ncu capture of one forward at the bench
    batch size, summarised by tools/dram_table.py into profiles/): (bytes, source) or (None, None)."""
    for fname in ('r02_dram_traffic.json', 'r01_dram_traffic.json'):
        path = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'profiles', fname)
        try:
            with open(path) as f:
                ks = json.load(f)['kernels']
            k = ks[kernel] if kernel in ks else next(v for n, v in ks.items() if n.startswith(kernel + '<'))     # template instances
            return k['dram_bytes_per_launch'], 'profiles/%s (ncu, %d launches of one batch-8 forward)' % (fname, k['launches'])
        except (OSError, KeyError, ValueError, StopIteration):
            continue
    return None, None


def _peaks():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            p = json.load(f)
        return dict(hbm=float(p['hbm_gbs']), tf=float(p.get('bf16_tflops_sustained', p['bf16_tflops'])), src='measured (MEASURED_PEAKS.json, sustained)')
    except Exception:
        return dict(hbm=6650.0, tf=1400.0, src='fallback (B200_PROFILING.md)')


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = 'index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, gpu_index):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-lms', '20', '-i', str(self.idx)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([time.perf_counter()] + [x.strip() for x in line.split(',')])

    def stop(self, window=None, scope='timed region + e2e loop (same load)'):
        """Median SM clock / throttle reasons of the samples that arrived inside `window` = (t0, t1) perf_counter times of the
        timed region; if nvidia-smi delivered none in there (the region is a few hundred ms), of all samples taken under the same
        load (timed region + end-to-end loop), and says which."""
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        rows = self.rows
        if window is not None:
            inside = [r for r in self.rows if window[0] <= r[0] <= window[1]]
            if inside:
                rows, scope = inside, 'timed region'
        sm, mx, reasons = [], [], set()
        for r in rows:
            r = r[1:]
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, val in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), r[4:8]):
                    if val.lower().startswith('active'):
                        reasons.add(name)
            except Exception:
                pass
        return {'sm_mhz': statistics.median(sm) if sm else None, 'sm_max_mhz': max(mx) if mx else None, 'reasons': sorted(reasons),
                'samples': len(sm), 'window': scope}


def _cpu_threads():
    """Threads for the CPU arm.  Measured on the GPU box's 128-core host (tools/cpu_probe.py, batch 1): 8 threads 2.30 s/img,
    16 -> 1.98, 32 -> 2.41, 64 -> 3.75, 128 -> 101.9 (oversubscription of many small convolutions): use the fastest setting."""
    return int(os.environ.get('N3D_CPU_THREADS', min(os.cpu_count() or 1, 16)))


def run_reference(args):
    """CPU arm: the oracle port of the reference's CPU path on the host cores; one image (c5: one 64^3 block of the grid) per step."""
    import torch
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    from next3d_b200 import weights
    from oracle import generator as og, renderer as orr
    cores = _cpu_threads()
    torch.set_num_threads(cores)
    name = args.config
    spec = CONFIGS[name]
    cfg = config_for(name)
    sd = weights.make_state_dict(cfg, seed=0)
    z, c_cond, c_cam, v = weights.demo_inputs(cfg, 1, seed=0)
    u_c, u_f = weights.sampler_noise(cfg, 1, seed=0)
    with torch.no_grad():
        ws = og.mapping(sd, cfg, z, c_cond, 0.7, 14)
        if name == 'c5':
            from next3d_b200 import drivers
            planes = og.synthesis(sd, cfg, ws, c_cam, v, u_c, u_f, return_intermediates=True)['planes']
            pts = drivers.create_samples(256, 1.0, head=256 ** 3 // 2, count=64 ** 3)
            step = lambda: dict(zip(('rgb', 'sigma'), orr.run_model(sd, planes, pts, cfg.rendering_kwargs)))
            units_per_step, unit = (64 ** 3) / (256 ** 3), 'grids/s'
            sample = 'each step = 64^3 consecutive voxels (1/64) of the 256^3 grid through run_model (tri-plane fetch + decoder), planes precomputed'
        else:
            step = lambda: og.synthesis(sd, cfg, ws, c_cam, v, u_c, u_f)
            units_per_step, unit = 1.0, UNIT
            sample = 'each step = 1 image (batch 1) of that workload (bounded sample: the CPU path takes seconds per image)'
        for _ in range(args.warmup):
            step()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            out = step()
        dt = time.perf_counter() - t0
    if args.dump_outputs:
        _dump_outputs(args.dump_outputs, out)
    val = args.steps * units_per_step / dt
    desc = f'{args.steps} steps, fp32 torch CPU ops (oracle port of the reference path), {cores} threads (of {os.cpu_count()} host cores; more threads are slower, see bench.py::_cpu_threads); {sample}'
    _emit({
        'impl': 'reference', 'metric': spec['metric'], 'value': val, 'unit': unit, 'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': 1e3 * dt / args.steps, 'higher_is_better': True, 'scaling': 'strong' if name == 'c4' else 'weak', 'vs_baseline': None, 'dtype': 'f32',
        'data': 'synthetic',
        'config': {'workload': spec['workload'] + (f'batch {args.batch or spec["batch"]} per GPU' if 'batch' in spec else 'one GPU'), 'sample': sample + ', host cores only'},
        'cpu_baseline': {'value': val, 'unit': unit, 'cores': cores, 'kind': 'port', 'sample': desc},
        'e2e': {'value': val, 'unit': unit, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}})


def cpu_baseline_sample():
    """Bounded CPU sample for the N=1 line: 1 warm-up + 3 images, batch 1, all host threads."""
    import torch
    from next3d_b200 import config, weights
    from oracle import generator as og
    cores = _cpu_threads()
    torch.set_num_threads(cores)
    cfg = config.full_config(512)
    sd = weights.make_state_dict(cfg, seed=0)
    z, c_cond, c_cam, v = weights.demo_inputs(cfg, 1, seed=0)
    u_c, u_f = weights.sampler_noise(cfg, 1, seed=0)
    times = []
    with torch.no_grad():
        ws = og.mapping(sd, cfg, z, c_cond, 0.7, 14)
        og.synthesis(sd, cfg, ws, c_cam, v, u_c, u_f)
        for _ in range(3):
            t0 = time.perf_counter()
            og.synthesis(sd, cfg, ws, c_cam, v, u_c, u_f)
            times.append(time.perf_counter() - t0)
    med = statistics.median(times)
    return {'value': 1.0 / med, 'unit': UNIT, 'cores': cores, 'kind': 'port',
            'sample': f'1 warm-up + median of 3 synthesis() calls, batch 1, same weights/config, CPU oracle port (fp32 torch ops), {cores} of {os.cpu_count()} host threads (fastest setting)'}


def _barrier(dist, world, dev):
    import torch
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)


def _renderer_roofline(name, cfg, B, ms_r, step_ms, pk):
    """Roofline entry of the fused renderer for config `name` (SURVEY.md section 8d): C2 is HBM-bound by the formula (planes read
    once + rays + outputs), C3 tensor-bound (decoder FLOPs).  The reachable ceilings are lower than either: see `limits`."""
    M = cfg.neural_rendering_resolution ** 2
    Dt = cfg.rendering_kwargs['depth_resolution'] + cfg.rendering_kwargs['depth_resolution_importance']
    bytes_img = 3 * 32 * 256 * 256 * 4 + M * 6 * 4 + M * 34 * 4            # planes once + rays + rgb32/depth/wsum out (RNG in kernel)
    flops_img = M * Dt * 8320
    t_hbm, t_tc = bytes_img / (pk['hbm'] * 1e9), flops_img / (pk['tf'] * 1e12)
    samples = B * M * Dt
    # hard per-SM limits of a per-sample gather + MLP (DESIGN.md section 3.2): 12 x 128-byte L1 wavefronts per sample at one per
    # clock, and 192 MUFU operations per sample (64 softplus = ex2 + lg2, 32 sigmoid = ex2 + rcp) at 16 per clock and SM
    clk = 1.85e9
    limits = {'l1_wavefront_floor_ms': 1e3 * samples * 12 / (148 * clk), 'mufu_floor_ms': 1e3 * samples * 192 / (148 * 16 * clk),
              'note': 'floors at 148 SMs x 1.85 GHz; a per-sample bilinear gather cannot read each texel once, and the activations are SFU-bound'}
    if t_hbm >= t_tc:
        ach = bytes_img * B / (ms_r * 1e-3) / 1e9
        r = {'bound': 'hbm', 'achieved': ach, 'peak': pk['hbm'], 'unit': 'GB/s', 'frac': ach / pk['hbm'], 'algorithmic_bytes_per_launch': bytes_img * B}
    else:
        ach = flops_img * B / (ms_r * 1e-3) / 1e12
        r = {'bound': 'tensor', 'achieved': ach, 'peak': pk['tf'], 'unit': 'TFLOP/s', 'frac': ach / pk['tf'], 'algorithmic_flops_per_launch': flops_img * B}
    r.update({'kernel': 'render_fused_kernel (ray sampler + tri-plane fetch + tcgen05 MLP + importance resampling + compositing)', 'config': name,
              'ms_per_step': ms_r, 'share_of_step': ms_r / step_ms if step_ms else None, 'flops_per_image': flops_img, 'peak_source': pk['src'],
              'limits': limits})
    return r


def _measured_floors(eng, planes, cam, intr, R):
    """Gather-only and activations-only micro-kernels on the same rays / samples as the renderer (n3d_render_floor): ms each."""
    import torch
    from next3d_b200 import kernels as K
    out = {}
    for kind, key in ((0, 'gather_only_ms'), (1, 'activations_only_ms')):
        for _ in range(2):
            K.render_floor(planes, cam, intr, R, eng.rk, kind)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(5):
            K.render_floor(planes, cam, intr, R, eng.rk, kind, seed=i)
        e1.record()
        torch.cuda.synchronize()
        out[key] = e0.elapsed_time(e1) / 5
    out['note'] = ('measured on this GPU, same rays and sample positions: the tri-plane gather alone on all 16 warps per SM (no MLP) and the '
                   "decoder's 192 MUFU operations per sample alone -- what a per-sample gather + MLP can reach at best; the HBM formula above assumes "
                   'every plane texel is read once, which no per-sample bilinear fetch does')
    return out


def _kernel_profile(G, eng, ws_d, c_d, v_d):
    """Per-kernel device times of one eager, single-stream forward (CUDA events around every launch of the graded kernels)."""
    eng.prof = []
    graph, conc = G.use_cuda_graph, eng.concurrent
    G.use_cuda_graph = False                             # events around every launch need the eager path ...
    eng.concurrent = False                               # ... and one stream: a kernel sharing the SMs with another branch is not its own time
    G.synthesis(ws_d, c_d, v_d, noise_mode='const', seed=5)
    summ = eng.profile_summary()
    eng.prof = None
    G.use_cuda_graph, eng.concurrent = graph, conc
    return summ


def _time_c5(G, ws, v, steps, warmup):
    """256^3 density grid from cached planes: (ms per grid, roofline dict, the grid of the last timed step)."""
    import torch
    from next3d_b200 import kernels as K
    eng = G._get_engine()
    R = CONFIGS['c5']['grid']
    planes = eng.compute_planes(ws[:1], v[:1], 'const')
    out = torch.empty(R, R, R, device=planes.device)
    box = G.rendering_kwargs['box_warp']
    pad = int(30 * R / 256)
    for _ in range(max(warmup, 2)):
        K.sample_grid(planes[0], R, box, box, eng.dec, out, pad=pad)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        K.sample_grid(planes[0], R, box, box, eng.dec, out, pad=pad)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    pk = _peaks()
    interior = (R - 2 * pad) ** 3
    flops = R ** 3 * 8320                                  # SURVEY.md 8d counts every voxel: 139.6 GFLOP
    ach = flops / (ms * 1e-3) / 1e12
    roof = {'kernel': 'points_fused_kernel (in-kernel voxel coordinates + tri-plane fetch + tcgen05 MLP, sigma only, flip + trim fused)',
            'bound': 'tensor', 'achieved': ach, 'peak': pk['tf'], 'unit': 'TFLOP/s', 'frac': ach / pk['tf'], 'peak_source': pk['src'],
            'algorithmic_flops_per_launch': flops, 'decoded_voxels': interior,
            'note': 'algorithmic FLOPs of the full 256^3 grid; the %d border voxels the script overwrites with -1000 are not decoded '
                    '(%.0f %% of the grid), so the executed FLOPs are lower' % (R ** 3 - interior, 100.0 * (1 - interior / R ** 3)),
            'limits': {'mufu_floor_ms': 1e3 * interior * 128 / (148 * 16 * 1.85e9), 'l1_wavefront_floor_ms': 1e3 * interior * 12 / (148 * 1.85e9)}}
    return ms, roof, out


def _time_c4(G, dev, rank, world, steps, warmup):
    """One 240-frame clip split over the ranks: seconds for the whole clip (max over ranks), frames, whether the frames look sane,
    and the clip of the last timed step (uint8 [F, 512, 512, 3] host tensor on rank 0, None elsewhere)."""
    import torch
    import torch.distributed as dist
    from next3d_b200 import drivers, weights, distributed as D
    spec = CONFIGS['c4']
    cfg = G.cfg
    F = spec['frames']
    z, c_cond, _, v = weights.demo_inputs(cfg, 1, seed=0)
    with torch.no_grad():
        ws = G.mapping(z.to(dev), c_cond.to(dev), truncation_psi=0.7, truncation_cutoff=14)
        wsf = drivers.interpolate_ws(ws.cpu(), F, wraps=2).float()               # one keyframe -> constant w, as in the script
        cams = drivers.orbit_camera_params(F, torch.tensor(G.rendering_kwargs['avg_camera_pivot']), G.rendering_kwargs['avg_camera_radius'])
        host = torch.empty(F, 512, 512, 3, dtype=torch.uint8).pin_memory() if rank == 0 else None      # the video writer's frame buffer
        for _ in range(max(1, min(warmup, 2))):
            drivers.render_frames_sharded(G, wsf, cams, v[:1], batch=spec['batch'], seed=1, out=host)
        _barrier(dist, world, dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            frames = drivers.render_frames_sharded(G, wsf, cams, v[:1], batch=spec['batch'], seed=100 + i, out=host)
        e1.record()
        _barrier(dist, world, dev)
    dt = D.max_over_ranks(e0.elapsed_time(e1) / 1e3, dev) / steps
    ok = frames is None or (frames.shape == (F, 512, 512, 3) and int(frames.float().std()) > 0)
    return dt, F, ok, frames


def run_ours(args):
    import torch
    import torch.distributed as dist
    from next3d_b200 import weights, distributed as D
    from next3d_b200.triplane_next3d import TriPlaneGenerator

    rank, world, local = D.init_from_env()
    assert torch.cuda.is_available(), 'bench.py needs a CUDA device (no CPU fallback)'
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    name = args.config
    spec = CONFIGS[name]
    cfg = config_for(name)
    sd = weights.make_state_dict(cfg, seed=0)
    G = TriPlaneGenerator.from_config(cfg, sd, device=dev)
    G.use_cuda_graph = not args.no_graph
    del sd
    pk = _peaks()

    if name == 'c5':                                       # one GPU: a single grid (N replicas for N > 1, no collective)
        z, c_cond, _, v = weights.demo_inputs(cfg, 1, seed=0)
        with torch.no_grad():
            ws = G.mapping(z.to(dev), c_cond.to(dev), truncation_psi=0.7, truncation_cutoff=14)
            sampler = ClockSampler(local) if rank == 0 else None
            if sampler:
                sampler.start()
            ms, roof, grid = _time_c5(G, ws, v.to(dev), args.steps, args.warmup)
            clocks = sampler.stop(scope='warm-up + timed region (same load)') if sampler else None
        ms = 1e3 * D.max_over_ranks(ms / 1e3, dev)
        if rank == 0 and args.dump_outputs:
            _dump_outputs(args.dump_outputs, {'sigma_grid': grid})
        if rank == 0:
            _emit({'metric': spec['metric'], 'value': world * 1e3 / ms, 'unit': 'grids/s', 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
                   'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'bf16x3 decoder (fp32 accumulate), f32 elsewhere',
                   'data': 'synthetic', 'config': {'workload': spec['workload'] + 'one grid per GPU (replicas only: a single grid does not shard in the script)'},
                   'roofline': roof, 'clocks': clocks, 'gpu_launches': args.steps})
        if world > 1:
            dist.destroy_process_group()
        return

    if name == 'c4':
        G.use_cuda_graph = not args.no_graph
        sampler = ClockSampler(local) if rank == 0 else None
        if sampler:
            sampler.start()
        dt, F, ok, frames = _time_c4(G, dev, rank, world, args.steps, args.warmup)
        clocks = sampler.stop(scope='warm-up + timed region (same load)') if sampler else None
        if rank == 0 and args.dump_outputs:
            _dump_outputs(args.dump_outputs, {'frames': frames})
        if rank == 0:
            _emit({'metric': spec['metric'], 'value': F / dt, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
                   'ms_per_step': 1e3 * dt, 'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None,
                   'dtype': 'bf16x3 (hi/lo split operands, fp32 accumulate) for convs; f32 elsewhere', 'data': 'synthetic',
                   'config': {'workload': spec['workload'] + f'batches of {spec["batch"]} frames per GPU', 'frames': F,
                              'parallelism': f'frames sharded x{world}, uint8 frames gathered to rank 0 on a side stream, read back to pinned host memory',
                              'step': 'one step = the whole clip'},
                   'frames_ok': ok, 'clocks': clocks,
                   'e2e': {'value': F / dt, 'unit': UNIT, 'h2d_bytes_per_step': int(F * (28 * 512 + 25) * 4),
                           'd2h_bytes_per_step': int(F * 512 * 512 * 3), 'ms_per_step': 1e3 * dt,
                           'note': 'this configuration IS end to end: host schedule -> H2D per batch -> synthesis -> uint8 -> gather -> D2H'},
                   'gpu_launches': G._get_engine().launches * -(-F // (spec['batch'] * world)) * args.steps})
        if world > 1:
            dist.destroy_process_group()
        return

    # ------------------------------------------------------------------------------------------------ c2 / c3
    B = args.batch or spec['batch']
    # global sample ids: rank r owns [r*B, (r+1)*B)
    z, c_cond, c_cam, v = weights.demo_inputs(cfg, B * world, seed=0)
    a, b = D.shard_range(B * world, rank, world)
    z, c_cond, c_cam, v = z[a:b], c_cond[a:b], c_cam[a:b], v[a:b]
    with torch.no_grad():
        ws_host = G.mapping(z.to(dev), c_cond.to(dev), truncation_psi=0.7, truncation_cutoff=14).cpu().pin_memory()
    c_host, v_host = c_cam.pin_memory(), v.pin_memory()
    ws_d, c_d, v_d = ws_host.to(dev), c_host.to(dev), v_host.to(dev)
    eng = G._get_engine()
    side = torch.cuda.Stream(dev)
    gstage, gdone = [None, None], [None, None]
    gather_ev = []

    def step_device(i):
        """synthesis, then (N > 1) the one collective of the path: the images are copied into a ping-pong staging buffer and
        gathered on rank 0 from there on a side stream, so the next replay overwrites the graph's static output while NCCL is still
        draining the previous batch; the main stream only waits for the gather of step i-2 (same staging buffer)."""
        main = torch.cuda.current_stream(dev)
        out = G.synthesis(ws_d, c_d, v_d, noise_mode='const', seed=1000 + i)
        if world > 1:
            k = i & 1
            if gdone[k] is not None:
                main.wait_event(gdone[k])
            if gstage[k] is None:
                gstage[k] = torch.empty_like(out['image'])
            gstage[k].copy_(out['image'])
            side.wait_stream(main)
            with torch.cuda.stream(side):
                g0 = torch.cuda.Event(enable_timing=True); g0.record(side)
                D.gather_images(gstage[k], dst=0)
                gdone[k] = torch.cuda.Event(enable_timing=True); gdone[k].record(side)
                gather_ev.append((g0, gdone[k]))
        return out

    copy_s = torch.cuda.Stream(dev)
    stage, drained = [None, None], [None, None]

    def step_e2e(i, host_out):
        """One end-to-end step the way a serving loop would run it: H2D of the inputs, synthesis, and the D2H of the images on a
        copy stream from a ping-pong staging buffer, so that the read-back of step i overlaps the compute of step i+1
        (the graph's static output buffer is free again after a few-us device copy)."""
        main = torch.cuda.current_stream(dev)
        w = ws_host.to(dev, non_blocking=True)
        c = c_host.to(dev, non_blocking=True)
        vv = v_host.to(dev, non_blocking=True)
        out = G.synthesis(w, c, vv, noise_mode='const', seed=2000 + i)
        img = out['image']
        if world > 1:
            img = D.gather_images(img, dst=0)
        if img is not None:
            k = i & 1
            if drained[k] is not None:
                main.wait_event(drained[k])                 # the D2H of step i-2 has left this staging buffer
            if stage[k] is None:
                stage[k] = torch.empty_like(img)
            stage[k].copy_(img)
            copy_s.wait_stream(main)
            with torch.cuda.stream(copy_s):
                host_out[: img.shape[0]].copy_(stage[k], non_blocking=True)
                drained[k] = torch.cuda.Event()
                drained[k].record(copy_s)
        return out

    with torch.no_grad():
        for i in range(args.warmup):
            step_device(i)
        _barrier(dist, world, dev)
        gather_ev.clear()
        launches_per_step = eng.launches
        sampler = ClockSampler(local) if rank == 0 else None
        if sampler:
            sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        _barrier(dist, world, dev)
        t_begin = time.perf_counter()
        e0.record()
        for i in range(args.steps):
            out = step_device(i)
        if world > 1:
            torch.cuda.current_stream(dev).wait_stream(side)
        e1.record()
        _barrier(dist, world, dev)
        t_end = time.perf_counter()
        dt = D.max_over_ranks(e0.elapsed_time(e1) / 1e3, dev)
        if rank == 0 and args.dump_outputs:                    # before the loops below overwrite the graph's static outputs
            _dump_outputs(args.dump_outputs, out)
        gather_ms = statistics.median([x.elapsed_time(y) for x, y in gather_ev]) if gather_ev else None

        # ---- end to end through the public API: pinned host inputs -> synthesis -> images on the host
        host_out = torch.empty(B * world if rank == 0 else B, 3, 512, 512).pin_memory()
        for i in range(min(args.warmup, 3)):
            step_e2e(i, host_out)
        _barrier(dist, world, dev)
        e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e2.record()
        for i in range(args.steps):
            step_e2e(i, host_out)
        torch.cuda.current_stream(dev).wait_stream(copy_s)   # the last read-back is inside the timed region
        e3.record()
        _barrier(dist, world, dev)
        dt_e2e = D.max_over_ranks(e2.elapsed_time(e3) / 1e3, dev)
        clocks = sampler.stop((t_begin, t_end)) if sampler else None

        # ---- per-kernel device times (CUDA events around every launch of the two graded kernels), one extra step
        roof = roof_r = None
        step_ms = 1e3 * dt / args.steps
        if rank == 0:
            summ = _kernel_profile(G, eng, ws_d, c_d, v_d)
            n_g, ms_g, fl_g = summ['conv_gemm']
            ach = fl_g / (ms_g * 1e-3) / 1e12
            tr_g, tr_src = _traffic('conv_gemm_kernel') if (B == 8 and name == 'c2') else (None, None)
            roof = {'kernel': 'conv_gemm_kernel (tcgen05 implicit GEMM, all conv layers)', 'bound': 'tensor', 'achieved': ach, 'peak': pk['tf'],
                    'unit': 'TFLOP/s', 'frac': ach / pk['tf'], 'traffic': tr_g, 'traffic_unit': 'DRAM bytes per launch (mean)', 'traffic_source': tr_src,
                    'peak_source': pk['src'], 'launches_per_step': n_g,
                    'ms_per_step': ms_g, 'share_of_step': ms_g / step_ms,
                    'note': 'algorithmic FLOPs (one product per MAC: %.1f GFLOP/img); the bf16x3 scheme executes 3x that on the tensor pipe; '
                            'launches and time include the fixed-order reduction passes of the split-K 4^2-16^2 layers' % (fl_g / B / 1e9)}
            n_r, ms_r, _ = summ['render_rays']
            roof_r = _renderer_roofline(name, cfg, B, ms_r, step_ms, pk)
            tr_r, tr_rsrc = _traffic('render_fused_kernel') if (B == 8 and name == 'c2') else (None, None)
            roof_r['traffic'], roof_r['traffic_source'] = tr_r, tr_rsrc
            try:
                planes_b = eng.compute_planes(ws_d, v_d, 'const')
                roof_r['limits']['measured'] = _measured_floors(eng, planes_b, c_d[:, :16].contiguous(), c_d[:, 16:25].contiguous(), cfg.neural_rendering_resolution)
                del planes_b
            except Exception as e:
                roof_r['limits']['measured'] = {'error': repr(e)}

        # ---- the other BASELINE.json configurations, short runs (N = 1 only; the headline stays this config)
        others = None
        if rank == 0 and world == 1 and name == 'c2' and not args.no_other_configs:
            others = {}
            try:
                ms5, roof5, _ = _time_c5(G, ws_d, v_d, 5, 2)
                others['c5'] = {'metric': CONFIGS['c5']['metric'], 'value': 1e3 / ms5, 'unit': 'grids/s', 'ms_per_step': ms5, 'steps': 5,
                                'config': {'workload': CONFIGS['c5']['workload'] + 'one GPU'}, 'roofline': roof5}
            except Exception as e:                                              # an extra must never take the headline down
                others['c5'] = {'error': repr(e)}
            del G, eng
            torch.cuda.empty_cache()
            for oname in ('c3', 'c4'):
                try:
                    ocfg = config_for(oname)
                    G2 = TriPlaneGenerator.from_config(ocfg, weights.make_state_dict(ocfg, seed=0), device=dev)
                    G2.use_cuda_graph = not args.no_graph
                    if oname == 'c3':
                        B3 = CONFIGS['c3']['batch']
                        z3, cc3, cam3, v3 = weights.demo_inputs(ocfg, B3, seed=0)
                        ws3 = G2.mapping(z3.to(dev), cc3.to(dev), truncation_psi=0.7, truncation_cutoff=14)
                        cam3, v3 = cam3.to(dev), v3.to(dev)
                        for i in range(3):
                            G2.synthesis(ws3, cam3, v3, noise_mode='const', seed=i)
                        torch.cuda.synchronize(dev)
                        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        f0.record()
                        for i in range(5):
                            G2.synthesis(ws3, cam3, v3, noise_mode='const', seed=10 + i)
                        f1.record()
                        torch.cuda.synchronize(dev)
                        ms3 = f0.elapsed_time(f1) / 5
                        summ3 = _kernel_profile(G2, G2._get_engine(), ws3, cam3, v3)
                        roof3 = _renderer_roofline('c3', ocfg, B3, summ3['render_rays'][1], ms3, pk)
                        eng3 = G2._get_engine()
                        planes3 = eng3.compute_planes(ws3, v3, 'const')
                        roof3['limits']['measured'] = _measured_floors(eng3, planes3, cam3[:, :16].contiguous(), cam3[:, 16:25].contiguous(), 128)
                        del planes3
                        others['c3'] = {'metric': CONFIGS['c3']['metric'], 'value': B3 * 1e3 / ms3, 'unit': UNIT, 'ms_per_step': ms3, 'steps': 5,
                                        'config': {'workload': CONFIGS['c3']['workload'] + f'batch {B3}, one GPU', 'global_batch': B3},
                                        'roofline_renderer': roof3}
                    else:
                        dt4, F4, ok4, _ = _time_c4(G2, dev, 0, 1, 1, 1)
                        others['c4'] = {'metric': CONFIGS['c4']['metric'], 'value': F4 / dt4, 'unit': UNIT, 'ms_per_step': 1e3 * dt4, 'steps': 1,
                                        'config': {'workload': CONFIGS['c4']['workload'] + 'one GPU', 'frames': F4}, 'frames_ok': ok4, 'scaling': 'strong'}
                    del G2
                    torch.cuda.empty_cache()
                except Exception as e:
                    others[oname] = {'error': repr(e)}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    imgs = B * world * args.steps
    line = {
        'metric': spec['metric'], 'value': imgs / dt, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': 1e3 * dt / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'bf16x3 (hi/lo split operands, fp32 accumulate) for convs; f32 elsewhere', 'data': 'synthetic',
        'config': {'workload': spec['workload'] + f'batch {B} per GPU', 'global_batch': B * world,
                   'parallelism': f'batch-sharded x{world}, one gather of images (from a staging buffer on a side stream, overlapped with the next step)',
                   'launch': 'eager' if args.no_graph else 'one CUDA graph replay per step',
                   'l2': 'no explicit flush: per-step working set (0.7 GB packed weights + >4 GB activations) >> 126 MB L2'},
        'clocks': clocks,
        'e2e': {'value': imgs / dt_e2e, 'unit': UNIT, 'h2d_bytes_per_step': int(ws_host.numel() * 4 + c_host.numel() * 4 + v_host.numel() * 4),
                'd2h_bytes_per_step': int(B * 3 * 512 * 512 * 4), 'ms_per_step': 1e3 * dt_e2e / args.steps},
        'gpu_launches': launches_per_step * args.steps,
        'roofline': roof, 'roofline_renderer': roof_r,
    }
    if gather_ms is not None:
        line['collective'] = {'op': 'ncclGather of [B,3,512,512] fp32 images to rank 0 (side stream)', 'median_ms_on_rank0': gather_ms,
                              'bytes_per_rank': int(B * 3 * 512 * 512 * 4)}
    if others:
        line['other_configs'] = others
    if world == 1 and not args.no_cpu_baseline:
        line['cpu_baseline'] = cpu_baseline_sample()
    _emit(line)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--batch', type=int, default=None, help='samples per GPU per step (default: the configuration\'s: c2 8, c3 16)')
    ap.add_argument('--config', default='c2', choices=['c2', 'c3', 'c4', 'c5'], help='BASELINE.json configuration (c2 = the headline)')
    ap.add_argument('--no-other-configs', action='store_true', help='default N=1 run: skip the short c3 / c4 / c5 runs')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-graph', action='store_true', help='launch kernels eagerly instead of replaying the captured CUDA graph')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the outputs of the last timed step as DIR/<name>.npy (float32, at most 64 MB in all)')
    args = ap.parse_args()
    _guard_stdout()
    args.warmup = max(args.warmup, 3) if args.impl == 'ours' else args.warmup
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
