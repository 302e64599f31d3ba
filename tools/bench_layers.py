"""Micro-benchmark of the up-conv building blocks at the generator's layer shapes (batch 8): transposed-conv GEMM launch,
FIR-up epilogue, FIR-down split.  CUDA-event timing, L2 flushed (256 MB write) before every timed launch.
Usage (GPU box): python tools/bench_layers.py [tag]"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from next3d_b200 import kernels as K

DEV = 'cuda'
N = 8
flush = torch.empty(256 << 20, dtype=torch.uint8, device=DEV)


def timeit(fn, reps=5):
    fn(); torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    ts.sort()
    return ts[len(ts) // 2]


def main(tag):
    g = torch.Generator(device=DEV).manual_seed(1)
    print(f'# {tag}')
    for cin, cout, res in [(256, 128, 256), (32, 256, 128), (256, 128, 128), (512, 256, 64), (512, 512, 32), (512, 512, 16)]:
        x = torch.randn(N, res, res, cin, device=DEV, generator=g)
        hi, lo = K.split_bf16(x)
        w = torch.randn(cout, cin, 3, 3, device=DEV, generator=g) / (cin * 9) ** 0.5
        w_hi, w_lo = K.pack_conv_weight(w)
        raw = torch.empty(N, 2 * res + 1, 2 * res + 1, cout, device=DEV)
        us = timeit(lambda: K.conv_transposed_gemm(hi, lo, w_hi, w_lo, N, res, res, raw))
        fl = 2.0 * cin * cout * N * (3 * res + 2) ** 2
        print(f'convT   {cin:4d}->{cout:4d} @{res:3d}^2  {us:8.1f} us  {fl / us * 1e-6:6.1f} TF/s')
        o_hi = torch.empty(N, 2 * res, 2 * res, cout, device=DEV, dtype=torch.bfloat16)
        o_lo = torch.empty_like(o_hi)
        d = torch.rand(N, cout, device=DEV) + 0.5
        b = torch.randn(cout, device=DEV)
        nz = torch.randn(2 * res, 2 * res, device=DEV)
        st = torch.randn(N, cout, device=DEV)
        outs = [K.make_split_out(o_hi, o_lo, st, cout, 0)]
        gb = raw.numel() * 4 + o_hi.numel() * 4
        for mode in ('0', '1'):                      # 0: register-tiled kernel, 1: streamed kernel where eligible
            os.environ['N3D_FIR_STREAM'] = mode
            us = timeit(lambda: K.fir_up_epilogue(raw, cout, d, b, nz, 2 ** 0.5, 0.2, 256.0, outs=outs))
            print(f'fir_up  C={cout:4d} out {2 * res:3d}^2 stream={mode} {us:8.1f} us  {gb / us * 1e-3:6.0f} GB/s')
        os.environ.pop('N3D_FIR_STREAM')
    if os.environ.get('FIR_ONLY'):
        return
    for cin, cout, res in [(128, 128, 512), (128, 128, 256), (256, 256, 128), (512, 512, 64), (512, 512, 32), (512, 512, 16), (512, 512, 8), (512, 512, 4),
                           (1024, 512, 32), (1024, 512, 16), (1024, 512, 8)]:
        x = torch.randn(N, res, res, cin, device=DEV, generator=g)
        hi, lo = K.split_bf16(x)
        del x
        w = torch.randn(cout, cin, 3, 3, device=DEV, generator=g) / (cin * 9) ** 0.5
        w_hi, w_lo = K.pack_conv_weight(w)
        o_hi = torch.empty(N, res, res, cout, device=DEV, dtype=torch.bfloat16)
        o_lo = torch.empty_like(o_hi)
        d = torch.rand(N, cout, device=DEV) + 0.5
        b = torch.randn(cout, device=DEV)
        st = torch.randn(N, cout, device=DEV)
        outs = [K.make_split_out(o_hi, o_lo, st, cout, 0)]
        us = timeit(lambda: K.conv_gemm(hi, lo, w_hi, w_lo, K.taps_conv3x3(), N, res, res, dcoef=d, bias=b, gain=2 ** 0.5, slope=0.2, clamp=256.0, outs=outs))
        fl = 2.0 * cin * cout * 9 * N * res * res
        print(f'conv3x3 {cin:4d}->{cout:4d} @{res:3d}^2  {us:8.1f} us  {fl / us * 1e-6:6.1f} TF/s')
        del hi, lo, o_hi, o_lo
    for c, res in [(128, 256), (256, 128), (512, 64)]:
        x = torch.randn(N, res, res, c, device=DEV, generator=g)
        sh = (res + 2) // 2
        hi = torch.empty(4, N, sh, sh, c, device=DEV, dtype=torch.bfloat16)
        lo = torch.empty_like(hi)
        us = timeit(lambda: K.fir_down_split(x, hi, lo))
        gb = x.numel() * 4 + hi.numel() * 4
        print(f'fir_dn  C={c:4d} in  {res:3d}^2      {us:8.1f} us  {gb / us * 1e-3:6.0f} GB/s')


if __name__ == '__main__':
    main(sys.argv[1] if len(sys.argv) > 1 else 'default')
