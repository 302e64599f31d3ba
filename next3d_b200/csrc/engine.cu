// Memory-bound glue kernels of the generator engine (everything between two tensor-core convolutions that could not be
// folded into a GEMM epilogue).  All tensors NHWC; 128-bit accesses along the channel dimension; grids sized in
// multiples of the SM count.
#include <cstdlib>
#include "common.cuh"
#include "../../include/next3d_b200.h"
#include <cuda.h>
#include "tc_ptx.cuh"

namespace {
constexpr int kSMs = 148;
inline int grid_for(int64_t work_items, int threads, int per_sm = 8) {
    int64_t g = (work_items + threads - 1) / threads;
    int64_t cap = (int64_t)kSMs * per_sm;
    return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---------------------------------------------------------------------------------------------- styles / demod
// one warp per (row, n): 512-long dot product with float4 loads
// output layout: every layer owns a dense [N, Cin] block: styles[ooff[r] + n * cin[r]]
__global__ void __launch_bounds__(256) styles_kernel(const float* __restrict__ ws, int N, int num_ws, int wdim,
                                                     const float* __restrict__ A, const float* __restrict__ b,
                                                     const int* __restrict__ widx, const float* __restrict__ scale,
                                                     const int64_t* __restrict__ ooff, const int* __restrict__ cin,
                                                     float* __restrict__ styles, int rows) {
    const int lane = threadIdx.x & 31;
    const int64_t warp_global = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const float inv = rsqrtf((float)wdim);
    for (int64_t r = warp_global; r < rows; r += nwarps) {
        const float4* a4 = reinterpret_cast<const float4*>(A + r * wdim);
        const int wi = widx[r];
        for (int n = 0; n < N; ++n) {
            const float4* w4 = reinterpret_cast<const float4*>(ws + ((int64_t)n * num_ws + wi) * wdim);
            float acc = 0.f;
            for (int i = lane; i < wdim / 4; i += 32) {
                const float4 a = __ldg(a4 + i), w = __ldg(w4 + i);
                acc += a.x * w.x + a.y * w.y + a.z * w.z + a.w * w.w;
            }
            acc = warp_sum(acc);
            if (lane == 0) styles[ooff[r] + (int64_t)n * cin[r]] = (acc * inv + b[r]) * scale[r];
        }
    }
}

// one warp per output channel row r of some layer: styles of that layer at styles[soff[r] + n*cin[r] + i],
// result at dcoef[ooff[r] + n*cout[r]] (dense [N, Cout] block per layer)
__global__ void __launch_bounds__(256) demod_kernel(const float* __restrict__ styles, const float* __restrict__ wsq,
                                                    const int64_t* __restrict__ woff, const int* __restrict__ cin,
                                                    const int64_t* __restrict__ soff, const int64_t* __restrict__ ooff,
                                                    const int* __restrict__ cout, float* __restrict__ dcoef, int rows, int N) {
    const int lane = threadIdx.x & 31;
    const int64_t warp_global = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = warp_global; r < rows; r += nwarps) {
        const float* w = wsq + woff[r];
        const int c = cin[r];
        for (int n = 0; n < N; ++n) {
            const float* s = styles + soff[r] + (int64_t)n * c;
            float acc = 0.f;
            for (int i = lane; i < c; i += 32) { const float sv = s[i]; acc += sv * sv * __ldg(w + i); }
            acc = warp_sum(acc);
            if (lane == 0) dcoef[ooff[r] + (int64_t)n * cout[r]] = rsqrtf(acc + 1e-8f);
        }
    }
}

// ---------------------------------------------------------------------------------------------- modulate + split
__global__ void __launch_bounds__(256) modulate_split_kernel(const float* __restrict__ x, int64_t npix, int N, int C,
                                                             const float* __restrict__ style, __nv_bfloat16* __restrict__ hi,
                                                             __nv_bfloat16* __restrict__ lo, int cstride, int coff) {
    const int c4n = C >> 2;
    const int64_t total = (int64_t)N * npix * c4n;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int c4 = (int)(i % c4n);
        const int64_t pix = i / c4n;
        const int n = (int)(pix / npix);
        float4 v = __ldg(reinterpret_cast<const float4*>(x) + i);
        if (style) {
            const float4 s = __ldg(reinterpret_cast<const float4*>(style + (int64_t)n * C) + c4);
            v.x *= s.x; v.y *= s.y; v.z *= s.z; v.w *= s.w;
        }
        uint2 h, l;
        split_bf16x2(v.x, v.y, h.x, l.x); split_bf16x2(v.z, v.w, h.y, l.y);
        const int64_t o = pix * cstride + coff + c4 * 4;
        *reinterpret_cast<uint2*>(hi + o) = h;
        *reinterpret_cast<uint2*>(lo + o) = l;
    }
}

// ---------------------------------------------------------------------------------------------- FIR helpers
// [1,3,3,1]/8 per axis; upfirdn2d's 2-D filter is the outer product / 64 (setup_filter, upfirdn2d.py:101-111)
__device__ __constant__ float kFir1[4] = {0.125f, 0.375f, 0.375f, 0.125f};   // immutable constants (not runtime state)

struct EpiParams {
    const float* dcoef; const float* bias; const float* noise; int64_t noise_nstride;
    float gain, slope, clamp;
    N3DSplitOut out[2];
    float* out_f32; int f32_cstride, f32_coff;
};

// float4 arithmetic on the packed fp32x2 pipe (FFMA2 / FMUL2 / FADD2, sm_100): half the issue slots of scalar code.
__device__ __forceinline__ float2 f4lo(const float4& v) { return make_float2(v.x, v.y); }
__device__ __forceinline__ float2 f4hi(const float4& v) { return make_float2(v.z, v.w); }
__device__ __forceinline__ float4 f4_join(const float2& a, const float2& b) { return make_float4(a.x, a.y, b.x, b.y); }
__device__ __forceinline__ float4 f4_fma(float w, const float4& v, const float4& a) {
    const float2 ww = make_float2(w, w);
    return f4_join(__ffma2_rn(ww, f4lo(v), f4lo(a)), __ffma2_rn(ww, f4hi(v), f4hi(a)));
}
__device__ __forceinline__ float4 f4_fma4(const float4& w, const float4& v, const float4& a) {
    return f4_join(__ffma2_rn(f4lo(w), f4lo(v), f4lo(a)), __ffma2_rn(f4hi(w), f4hi(v), f4hi(a)));
}
__device__ __forceinline__ float4 f4_mul4(const float4& w, const float4& v) { return f4_join(__fmul2_rn(f4lo(w), f4lo(v)), __fmul2_rn(f4hi(w), f4hi(v))); }
__device__ __forceinline__ float4 f4_scale(float w, const float4& v) {
    const float2 ww = make_float2(w, w);
    return f4_join(__fmul2_rn(ww, f4lo(v)), __fmul2_rn(ww, f4hi(v)));
}

// Per-thread epilogue constants of one (image, 4-channel group): demodulation and bias pre-multiplied by the activation gain
// (lrelu(a) * g == lrelu(a * g) for g > 0), the two consumers' styles.
struct EpiVec { float4 dcg, bsg, st[2]; };

__device__ __forceinline__ EpiVec epi_load(const EpiParams& E, int n, int C, int c0) {
    EpiVec V;
    float4 dc = make_float4(1.f, 1.f, 1.f, 1.f), bs = make_float4(0.f, 0.f, 0.f, 0.f);
    if (E.dcoef) dc = __ldg(reinterpret_cast<const float4*>(E.dcoef + (int64_t)n * C + c0));
    if (E.bias) bs = __ldg(reinterpret_cast<const float4*>(E.bias + c0));
    V.dcg = f4_scale(E.gain, dc); V.bsg = f4_scale(E.gain, bs);
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        V.st[k] = make_float4(1.f, 1.f, 1.f, 1.f);
        if (E.out[k].hi && E.out[k].style) V.st[k] = __ldg(reinterpret_cast<const float4*>(E.out[k].style + (int64_t)n * C + c0));
    }
    return V;
}

// Output cursors of one thread: element offsets of its current 2x2 block's top-left pixel in the fp32 output and in the two split
// outputs (channel offset included), advanced by two rows per strip step -- no 64-bit multiplies in the loop.
struct EpiCursor { int64_t f32, sp[2]; };

__device__ __forceinline__ EpiCursor epi_cursor(const EpiParams& E, int64_t pix, int c0) {
    EpiCursor P;
    P.f32 = pix * E.f32_cstride + E.f32_coff + c0;
    P.sp[0] = pix * E.out[0].cstride + E.out[0].coff + c0;
    P.sp[1] = pix * E.out[1].cstride + E.out[1].coff + c0;
    return P;
}

// bias_act (lrelu with 0 <= slope <= 1: max(t, slope * t)) + clamp + the fp32 / modulated split-bf16 stores of one pixel.
// nzg = noise * gain; dpix = pixel offset from the cursor (0, 1, W2, W2 + 1).
__device__ __forceinline__ void epi_store(const EpiParams& E, const EpiVec& V, const EpiCursor& P, const float4& acc, float nzg, int dpix) {
    float4 t = f4_fma4(acc, V.dcg, make_float4(V.bsg.x + nzg, V.bsg.y + nzg, V.bsg.z + nzg, V.bsg.w + nzg));
    const float4 ts = f4_scale(E.slope, t);
    t = make_float4(fmaxf(t.x, ts.x), fmaxf(t.y, ts.y), fmaxf(t.z, ts.z), fmaxf(t.w, ts.w));
    if (E.clamp >= 0.f) {
        const float c = E.clamp;
        t = make_float4(fminf(fmaxf(t.x, -c), c), fminf(fmaxf(t.y, -c), c), fminf(fmaxf(t.z, -c), c), fminf(fmaxf(t.w, -c), c));
    }
    if (E.out_f32) *reinterpret_cast<float4*>(E.out_f32 + P.f32 + dpix * E.f32_cstride) = t;
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        const N3DSplitOut o = E.out[k];
        if (!o.hi) continue;
        const float4 m = f4_mul4(t, V.st[k]);
        uint2 h, l;
        split_bf16x2(m.x, m.y, h.x, l.x); split_bf16x2(m.z, m.w, h.y, l.y);
        const int64_t off = P.sp[k] + dpix * o.cstride;
        *reinterpret_cast<uint2*>((__nv_bfloat16*)o.hi + off) = h;
        *reinterpret_cast<uint2*>((__nv_bfloat16*)o.lo + off) = l;
    }
}

// ---------------------------------------------------------------------------------------------- FIR passes
// Both FIR passes (up: after every up-conv, with the epilogue; down: before every stride-2 conv) evaluate the separable 4x4 FIR one
// 2x2 output block and one 4-channel group per thread: a horizontal pass over the raw rows of a five-column window, then a vertical
// pass over five filtered rows.  Consecutive blocks down a column share 3 of the 5 rows, so the filtered rows stay in registers and
// slide down: 2 row reads per block instead of 5 (the unshared form is bound by L2->L1 traffic, 2.5x the raw tensor).
// Each direction has a register-tiled kernel (rows read from global memory) and a streamed one (rows read from a shared-memory ring
// filled by bulk copies).  Both call the functions below for every arithmetic instruction, so they round identically and the
// batch-size-dependent choice between them never shows in the results.

// 1-D taps [1, 3, 3, 1] * s: s = 1/4 for up (upfirdn2d's gain 4 spread over both axes), 1/8 for down.
constexpr float kFirUpS = 0.25f, kFirDownS = 0.125f;

__device__ __forceinline__ float4 fir4(float s, const float4& a, const float4& b, const float4& c, const float4& d) {
    return f4_fma(s, d, f4_fma(3.f * s, c, f4_fma(3.f * s, b, f4_scale(s, a))));
}

// Horizontal pass over raw row r: the two outputs that start at window columns 0 and 1.  A window column with ok[q] == false lies
// outside the image and reads as zero; so does a row outside [0, src.rows).  `Src` is where the rows come from (GlobalRows, RowRing).
template <class Src>
__device__ __forceinline__ void fir_hrow(Src& src, int r, float s, const bool (&ok)[5], float4 (&h)[2]) {
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    h[0] = z; h[1] = z;
    if (r < 0 || r >= src.rows) return;
    const float4* p = src.acquire(r);
    float4 v[5];
#pragma unroll
    for (int q = 0; q < 5; ++q) v[q] = ok[q] ? src.ld(p, q) : z;
    h[0] = fir4(s, v[0], v[1], v[2], v[3]);
    h[1] = fir4(s, v[1], v[2], v[3], v[4]);
    src.release();
}

// Up: window = raw columns x0-1 .. x0+3 of the 2-column block at x0; only the first / last can fall outside the image (vl / vr).
template <class Src>
__device__ __forceinline__ void fir_hrow_up(Src& src, int r, bool vl, bool vr, float4 (&h)[2]) {
    fir_hrow(src, r, kFirUpS, {vl, true, true, true, vr}, h);
}

// Down: window = input columns x0-2 .. x0+2, x0 even in [0, W]: the first two are outside together (x0 == 0: vl), the next two
// together (x0 == W: vm), the last one when x0 + 2 >= W (vr).
template <class Src>
__device__ __forceinline__ void fir_hrow_down(Src& src, int r, bool vl, bool vm, bool vr, float4 (&h)[2]) {
    fir_hrow(src, r, kFirDownS, {vl, vl, vm, vm, vr}, h);
}

// Vertical pass of output row a, column b of the block from the filtered rows a .. a+3.
__device__ __forceinline__ float4 fir_vert(float s, const float4 (&h)[5][2], int a, int b) {
    return fir4(s, h[a][b], h[a + 1][b], h[a + 2][b], h[a + 3][b]);
}

// The window moves down two rows: filtered rows 2 .. 4 become rows 0 .. 2.
__device__ __forceinline__ void fir_slide(float4 (&h)[5][2]) {
#pragma unroll
    for (int r = 0; r < 3; ++r) { h[r][0] = h[r + 2][0]; h[r][1] = h[r + 2][1]; }
}

// Raw noise of the 2x2 block at (y0, x0) of an image's [H2, W2] noise plane nzp (null: no noise), as {(0,0), (0,1), (1,0), (1,1)}.
__device__ __forceinline__ float4 fir_up_noise(const float* nzp, int y0, int W2) {
    if (!nzp) return make_float4(0.f, 0.f, 0.f, 0.f);
    const float* p = nzp + (int64_t)y0 * W2;
    return make_float4(__ldg(p), __ldg(p + 1), __ldg(p + W2), __ldg(p + W2 + 1));
}

// One step of the FIR-up epilogue: the 2x2 output block at cursor P from the filtered rows h and its raw noise nz, then window and
// cursor move down two rows.
__device__ __forceinline__ void fir_up_block(const EpiParams& E, const EpiVec& V, EpiCursor& P, int W2, float4 nz, float4 (&h)[5][2]) {
    // explicit: no FMA contraction into the bias add
    const float nzg[4] = {__fmul_rn(E.gain, nz.x), __fmul_rn(E.gain, nz.y), __fmul_rn(E.gain, nz.z), __fmul_rn(E.gain, nz.w)};
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int b = 0; b < 2; ++b) epi_store(E, V, P, fir_vert(kFirUpS, h, a, b), nzg[2 * a + b], a * W2 + b);
    fir_slide(h);
    P.f32 += 2 * (int64_t)W2 * E.f32_cstride;
    P.sp[0] += 2 * (int64_t)W2 * E.out[0].cstride;
    P.sp[1] += 2 * (int64_t)W2 * E.out[1].cstride;
}

// One step of the FIR-down pass: the 2x2 FIR outputs (y0 + a, x0 + b) of one sub-pixel, zero beyond the (H+1)x(W+1) FIR output, as
// bf16 hi / lo into parity image a * 2 + b (hi, lo: the sub-pixel in parity image 0), written only when `active`; then the window
// moves down two rows.
__device__ __forceinline__ void fir_down_block(float4 (&h)[5][2], bool active, int y0, int x0, int H, int W, int64_t par_stride,
                                               __nv_bfloat16* hi, __nv_bfloat16* lo) {
    if (active) {
#pragma unroll
        for (int a = 0; a < 2; ++a)
#pragma unroll
            for (int b = 0; b < 2; ++b) {
                float4 v = fir_vert(kFirDownS, h, a, b);
                if (y0 + a > H || x0 + b > W) v = make_float4(0.f, 0.f, 0.f, 0.f);
                uint2 hh, l;
                split_bf16x2(v.x, v.y, hh.x, l.x); split_bf16x2(v.z, v.w, hh.y, l.y);
                const int64_t off = (int64_t)(a * 2 + b) * par_stride;
                *reinterpret_cast<uint2*>(hi + off) = hh;
                *reinterpret_cast<uint2*>(lo + off) = l;
            }
    }
    fir_slide(h);
}

// Raw rows of the register-tiled kernels, read from global memory on the read-only path.  col: the thread's first window column in
// row 0; stride, cs: row and column stride in float4; rows: image height.
struct GlobalRows {
    const float4* col; int64_t stride; int rows, cs;
    __device__ const float4* acquire(int r) const { return col + r * stride; }
    __device__ float4 ld(const float4* p, int q) const { return __ldg(p + q * cs); }
    __device__ void release() const {}
};

// Raw rows of the streamed kernels.  A CTA's tile needs a window of ncols raw columns of one image; a producer lane streams the
// window's rows -- each a CONTIGUOUS ncols * C * 4-byte segment of the NHWC tensor -- through NR shared-memory stages with 1-D
// bulk copies (TMA engine, mbarrier full / empty pair per stage), and the kFsConsumers consumer threads read their five columns from
// the stages.  Loads are in flight NR rows ahead of the arithmetic and cost no registers.  Each thread counts its own stage / phase.
constexpr int kFsConsumers = 256, kFsThreads = kFsConsumers + 32;
constexpr int kFsSmemLimit = 112 * 1024;          // dynamic shared memory limit of both streamed kernels: 2 CTAs per SM

struct RowRing {
    int NR, rows, ncols, c4n;      // rows: image height; rows outside [0, rows) are zero padding, neither copied nor waited for
    const float4* win;             // consumers: the thread's first window column in stage 0
    uint32_t ring, bars;           // shared addresses: NR stages of ncols * c4n float4, then NR full and NR empty barriers
    int s = 0; uint32_t ph = 0;

    // smem: the CTA's dynamic shared memory; off: float4 offset of the thread's first window column within a stage
    __device__ RowRing(uint8_t* smem, int NR, int rows, int ncols, int c4n, int off)
        : NR(NR), rows(rows), ncols(ncols), c4n(c4n), win(reinterpret_cast<const float4*>(smem) + off), ring(n3d_tc::smem_u32(smem)),
          bars(ring + (uint32_t)(NR * ncols * c4n) * 16u) {}
    __device__ uint32_t stage(int k) const { return ring + (uint32_t)(k * ncols * c4n) * 16u; }
    __device__ uint32_t full(int k) const { return bars + 8u * (uint32_t)k; }
    __device__ uint32_t empty(int k) const { return bars + 8u * (uint32_t)(NR + k); }
    __device__ void advance() { if (++s == NR) { s = 0; ph ^= 1u; } }

    __device__ void init() const {          // every thread of the CTA
        if (threadIdx.x == 0) {
            for (int k = 0; k < NR; ++k) { n3d_tc::mbar_init(full(k), 1); n3d_tc::mbar_init(empty(k), kFsConsumers / 32); }
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncthreads();
    }

    // Producer lane: rows first .. last of the window that starts at column col0 of an image (img: its pixel (0, 0); `width` pixels
    // per row), each clipped to the image's columns (the consumers' edge flags zero the clipped ones).
    __device__ void produce(const float* img, int width, int col0, int first, int last) {
        const int C = 4 * c4n;
        const int col_lo = max(col0, 0), col_hi = min(col0 + ncols - 1, width - 1);
        const uint32_t bytes = (uint32_t)(col_hi - col_lo + 1) * (uint32_t)C * 4u;
        const uint32_t dst_off = (uint32_t)(col_lo - col0) * (uint32_t)C * 4u;
        const float* src = img + (int64_t)col_lo * C;
        for (int r = first; r <= last; ++r) {
            if (r < 0 || r >= rows) continue;
            n3d_tc::mbar_wait_short(empty(s), ph ^ 1u);
            n3d_tc::mbar_expect_tx(full(s), bytes);
            n3d_tc::bulk_load_1d(stage(s) + dst_off, src + (int64_t)r * width * C, bytes, full(s));
            advance();
        }
    }

    // Consumers (the row source of fir_hrow): wait for the next row's stage, read it, hand it back.
    __device__ const float4* acquire(int) {
        n3d_tc::mbar_wait_short(full(s), ph);
        return win + s * ncols * c4n;
    }
    __device__ float4 ld(const float4* p, int q) const { return p[q * c4n]; }
    __device__ void release() {
        __syncwarp();                      // every lane has consumed its values: the stage may be refilled
        if ((threadIdx.x & 31) == 0) n3d_tc::mbar_arrive(empty(s));
        advance();
    }
};

// FIR-up epilogue, register-tiled: thread = (image, strip of S output row pairs, 2 output columns, 4-channel group).  2 columns per
// thread measured best on B200 (1 column: +23 % time despite 1.5x the occupancy, 4 columns: +15 %).
__global__ void __launch_bounds__(256) fir_up_epilogue_kernel(const float* __restrict__ raw, int N, int H2, int W2, int C, int S, EpiParams E) {
    const int RH = H2 + 1, RW = W2 + 1, c4n = C >> 2, BH = H2 >> 1, BW = W2 >> 1, nstrip = (BH + S - 1) / S;
    const int64_t total = (int64_t)N * nstrip * BW * c4n;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int c4 = (int)(i % c4n);
        int64_t t = i / c4n;
        const int bx = (int)(t % BW); t /= BW;
        const int st = (int)(t % nstrip);
        const int n = (int)(t / nstrip);
        const int x0 = bx * 2, c0 = c4 * 4;
        const int by_begin = st * S, by_end = min(by_begin + S, BH);
        const bool vl = x0 > 0, vr = x0 + 3 < RW;
        GlobalRows rows{reinterpret_cast<const float4*>(raw) + ((int64_t)n * RH * RW + (x0 - 1)) * c4n + c4, (int64_t)RW * c4n, RH, c4n};
        const EpiVec V = epi_load(E, n, C, c0);
        const float* nzp = E.noise ? E.noise + (int64_t)n * E.noise_nstride + x0 : nullptr;
        float4 h[5][2];
#pragma unroll
        for (int r = 0; r < 3; ++r) fir_hrow_up(rows, 2 * by_begin - 1 + r, vl, vr, h[r]);
        EpiCursor P = epi_cursor(E, ((int64_t)n * H2 + 2 * by_begin) * W2 + x0, c0);
        for (int y0 = 2 * by_begin; y0 < 2 * by_end; y0 += 2) {
            fir_hrow_up(rows, y0 + 2, vl, vr, h[3]);
            fir_hrow_up(rows, y0 + 3, vl, vr, h[4]);
            fir_up_block(E, V, P, W2, fir_up_noise(nzp, y0, W2), h);
        }
    }
}

// FIR-up epilogue, streamed.  The register-tiled kernel is bound by load latency at 16 warps/SM (DRAM 42-62 % of peak,
// profiles/r02_ncu_glue.txt): every strip step waits for its own ten 16-byte loads.  Here a CTA owns a (TR output rows) x (TC output
// columns) x (all C channels) tile of one image and reads its raw rows through a RowRing.  thread = (column pair, 4-channel group):
// (TC / 2) * (C / 4) == 256.
__global__ void __launch_bounds__(kFsThreads, 2) fir_up_stream_kernel(const float* __restrict__ raw, int N, int H2, int W2, int C, int TC, int TR, int NR,
                                                                       EpiParams E) {
    extern __shared__ __align__(128) uint8_t fs_smem[];
    const int RH = H2 + 1, RW = W2 + 1, c4n = C >> 2;
    const int tiles_x = W2 / TC, tiles_y = H2 / TR;
    const int bx = blockIdx.x % tiles_x, by = (blockIdx.x / tiles_x) % tiles_y, n = blockIdx.x / (tiles_x * tiles_y);
    const int X0 = bx * TC, Y0 = by * TR;
    const int c4 = threadIdx.x % c4n, j = threadIdx.x / c4n;
    RowRing ring(fs_smem, NR, RH, TC + 3, c4n, 2 * j * c4n + c4);
    ring.init();
    if (threadIdx.x >= kFsConsumers) {      // producer: raw rows Y0-1 .. Y0+TR+1, columns X0-1 .. X0+TC+1
        if (threadIdx.x == kFsConsumers) ring.produce(raw + (int64_t)n * RH * RW * C, RW, X0 - 1, Y0 - 1, Y0 + TR + 1);
        return;
    }
    const int x0 = X0 + 2 * j, c0 = c4 * 4;
    const bool vl = x0 > 0, vr = x0 + 3 < RW;
    const EpiVec V = epi_load(E, n, C, c0);
    const float* nzp = E.noise ? E.noise + (int64_t)n * E.noise_nstride + x0 : nullptr;
    float4 h[5][2];
#pragma unroll
    for (int r = 0; r < 3; ++r) fir_hrow_up(ring, Y0 - 1 + r, vl, vr, h[r]);
    EpiCursor P = epi_cursor(E, ((int64_t)n * H2 + Y0) * W2 + x0, c0);
    // the noise of a block is fetched one step ahead: its global-load latency was 26 % of all stall samples when it sat between the
    // FIR and the stores (ncu source page of the first version)
    float4 nz_next = fir_up_noise(nzp, Y0, W2);
    for (int y0 = Y0; y0 < Y0 + TR; y0 += 2) {
        const float4 nz = nz_next;
        if (y0 + 2 < Y0 + TR) nz_next = fir_up_noise(nzp, y0 + 2, W2);
        fir_hrow_up(ring, y0 + 2, vl, vr, h[3]);
        fir_hrow_up(ring, y0 + 3, vl, vr, h[4]);
        fir_up_block(E, V, P, W2, nz, h);
    }
}

// Second pass of a split-K convolution: sum the S raw partial tensors in a fixed order, then the usual epilogue.
// thread = (pixel, 4-channel group).
__global__ void __launch_bounds__(256) splitk_epilogue_kernel(const float* __restrict__ part, int S, int64_t stride, int N, int H, int W, int C, EpiParams E) {
    const int c4n = C >> 2;
    const int64_t total = (int64_t)N * H * W * c4n;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int c4 = (int)(i % c4n);
        const int64_t pix = i / c4n;
        const int n = (int)(pix / ((int64_t)H * W));
        const int64_t yx = pix - (int64_t)n * H * W;
        float4 acc = __ldg(reinterpret_cast<const float4*>(part) + i);
        for (int s = 1; s < S; ++s) {
            const float4 v = __ldg(reinterpret_cast<const float4*>(part + (int64_t)s * stride) + i);
            acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
        }
        const EpiVec V = epi_load(E, n, C, c4 * 4);
        const EpiCursor P = epi_cursor(E, pix, c4 * 4);
        const float nzg = E.noise ? __fmul_rn(E.gain, __ldg(E.noise + (int64_t)n * E.noise_nstride + yx)) : 0.f;
        epi_store(E, V, P, acc, nzg, 0);
    }
}

// FIR (pad 2,2,2,2) -> [(H+1),(W+1)] -> parity-split bf16 hi/lo, layout [4 parities][N][SH][SW][C], register-tiled.
// thread = (image, strip of S sub-pixel rows, sub-pixel column sx, 4-channel group) -> per sub-pixel the 2x2 block of FIR outputs
// (2sy+a, 2sx+b), one per parity image.
__global__ void __launch_bounds__(256) fir_down_split_kernel(const float* __restrict__ x, int N, int H, int W, int C, int S,
                                                             __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo) {
    const int SH = (H + 2) / 2, SW = (W + 2) / 2, c4n = C >> 2, nstrip = (SH + S - 1) / S;
    const int64_t total = (int64_t)N * nstrip * SW * c4n;
    const int64_t par_stride = (int64_t)N * SH * SW * C;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int c4 = (int)(i % c4n);
        int64_t t = i / c4n;
        const int sx = (int)(t % SW); t /= SW;
        const int st = (int)(t % nstrip);
        const int n = (int)(t / nstrip);
        const int x0 = sx * 2;                               // FIR output (y, x) reads input rows y-2 .. y+1, columns x-2 .. x+1
        const int sy_begin = st * S, sy_end = min(sy_begin + S, SH);
        const bool vl = x0 >= 2, vm = x0 < W, vr = x0 + 2 < W;
        GlobalRows rows{reinterpret_cast<const float4*>(x) + ((int64_t)n * H * W + (x0 - 2)) * c4n + c4, (int64_t)W * c4n, H, c4n};
        float4 h[5][2];
#pragma unroll
        for (int r = 0; r < 3; ++r) fir_hrow_down(rows, 2 * sy_begin - 2 + r, vl, vm, vr, h[r]);
        for (int sy = sy_begin; sy < sy_end; ++sy) {
            const int y0 = sy * 2;
            fir_hrow_down(rows, y0 + 1, vl, vm, vr, h[3]);
            fir_hrow_down(rows, y0 + 2, vl, vm, vr, h[4]);
            const int64_t o = (((int64_t)n * SH + sy) * SW + sx) * C + c4 * 4;
            fir_down_block(h, true, y0, x0, H, W, par_stride, hi + o, lo + o);
        }
    }
}

// FIR-down pass, streamed (same construction as fir_up_stream_kernel): a CTA owns TS sub-pixel rows x TSC sub-pixel columns x all
// channels of one image ((TSC) * (C / 4) == 256 consumer threads) and reads its 2 TS + 3 input rows through a RowRing.
__global__ void __launch_bounds__(kFsThreads, 2) fir_down_stream_kernel(const float* __restrict__ x, int N, int H, int W, int C, int TSC, int TS, int NR,
                                                                         __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo) {
    extern __shared__ __align__(128) uint8_t fs_smem[];
    const int SH = (H + 2) / 2, SW = (W + 2) / 2, c4n = C >> 2;
    const int tiles_x = (SW + TSC - 1) / TSC, tiles_y = (SH + TS - 1) / TS;
    const int bx = blockIdx.x % tiles_x, by = (blockIdx.x / tiles_x) % tiles_y, n = blockIdx.x / (tiles_x * tiles_y);
    const int SX0 = bx * TSC, SY0 = by * TS, rows_here = min(TS, SH - SY0);
    const int iy_first = 2 * SY0 - 2, iy_last = 2 * (SY0 + rows_here - 1) + 2;
    const int c4 = threadIdx.x % c4n, j = threadIdx.x / c4n;
    RowRing ring(fs_smem, NR, H, 2 * TSC + 3, c4n, 2 * j * c4n + c4);
    ring.init();
    if (threadIdx.x >= kFsConsumers) {      // producer: input columns 2 SX0 - 2 .. 2 SX0 + 2 TSC
        if (threadIdx.x == kFsConsumers) ring.produce(x + (int64_t)n * H * W * C, W, 2 * SX0 - 2, iy_first, iy_last);
        return;
    }
    const int sx = SX0 + j, x0 = 2 * sx;
    const bool active = sx < SW;                                // the last column tile is ragged (SW = W / 2 + 1)
    const bool vl = active && x0 >= 2, vm = active && x0 < W, vr = active && x0 + 2 < W;
    const int64_t par_stride = (int64_t)N * SH * SW * C;
    float4 h[5][2];
#pragma unroll
    for (int r = 0; r < 3; ++r) fir_hrow_down(ring, iy_first + r, vl, vm, vr, h[r]);
    for (int sy = SY0; sy < SY0 + rows_here; ++sy) {
        const int y0 = sy * 2;
        fir_hrow_down(ring, y0 + 1, vl, vm, vr, h[3]);
        fir_hrow_down(ring, y0 + 2, vl, vm, vr, h[4]);
        const int64_t o = (((int64_t)n * SH + sy) * SW + sx) * C + c4 * 4;
        fir_down_block(h, active, y0, x0, H, W, par_stride, hi + o, lo + o);
    }
}

// upsample2d: zero-insert x2, pad (2,1), 4x4 FIR * 4.  Polyphase form: out[2i] = .25 x[i-1] + .75 x[i], out[2i+1] = .75 x[i] + .25 x[i+1]
// per axis.  thread = (input pixel (i,j), VEC channels) -> the 2x2 output block from the 3x3 input neighbourhood.
template <int VEC>
__global__ void __launch_bounds__(256) upsample2d_kernel(const float* __restrict__ x, int N, int H, int W, int C, float* __restrict__ y, int nchw) {
    const int OH = 2 * H, OW = 2 * W, cvn = C / VEC;
    const int64_t total = (int64_t)N * H * W * cvn;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
        const int cv = (int)(idx % cvn);
        int64_t t = idx / cvn;
        const int j = (int)(t % W); t /= W;
        const int i = (int)(t % H);
        const int n = (int)(t / H);
        float v[3][3][VEC];
#pragma unroll
        for (int a = 0; a < 3; ++a)
#pragma unroll
            for (int b = 0; b < 3; ++b) {
                const int yy = i - 1 + a, xx = j - 1 + b;
                const bool ok = yy >= 0 && yy < H && xx >= 0 && xx < W;
                const float* src = x + (((int64_t)n * H + (ok ? yy : 0)) * W + (ok ? xx : 0)) * C + cv * VEC;
                if (VEC == 4) {
                    const float4 q = ok ? __ldg(reinterpret_cast<const float4*>(src)) : make_float4(0.f, 0.f, 0.f, 0.f);
                    v[a][b][0] = q.x; v[a][b][1 % VEC] = q.y; v[a][b][2 % VEC] = q.z; v[a][b][3 % VEC] = q.w;
                } else {
                    v[a][b][0] = ok ? __ldg(src) : 0.f;
                }
            }
        const float wa[2][3] = {{0.25f, 0.75f, 0.f}, {0.f, 0.75f, 0.25f}};
#pragma unroll
        for (int a = 0; a < 2; ++a)
#pragma unroll
            for (int b = 0; b < 2; ++b) {
                float o[VEC];
#pragma unroll
                for (int e = 0; e < VEC; ++e) {
                    float acc = 0.f;
#pragma unroll
                    for (int p = 0; p < 3; ++p)
#pragma unroll
                        for (int q = 0; q < 3; ++q) acc += (wa[a][p] * wa[b][q]) * v[p][q][e];
                    o[e] = acc;
                }
                const int oy = 2 * i + a, ox = 2 * j + b;
                if (nchw) {
#pragma unroll
                    for (int e = 0; e < VEC; ++e) y[(((int64_t)n * C + cv * VEC + e) * OH + oy) * OW + ox] = o[e];
                } else {
                    float* dst = y + (((int64_t)n * OH + oy) * OW + ox) * C + cv * VEC;
                    if (VEC == 4) *reinterpret_cast<float4*>(dst) = make_float4(o[0], o[1 % VEC], o[2 % VEC], o[3 % VEC]);
                    else dst[0] = o[0];
                }
            }
    }
}

// downsample2d: pad (1,1), 4x4 FIR, keep every 2nd pixel
__global__ void __launch_bounds__(256) downsample2d_kernel(const float* __restrict__ x, int N, int H, int W, int C, float* __restrict__ y) {
    const int OH = H / 2, OW = W / 2;
    const int64_t total = (int64_t)N * OH * OW * C;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % C);
        int64_t t = i / C;
        const int ox = (int)(t % OW); t /= OW;
        const int oy = (int)(t % OH);
        const int n = (int)(t / OH);
        float acc = 0.f;
#pragma unroll
        for (int fy = 0; fy < 4; ++fy) {
            const int iy = oy * 2 + fy - 1;
            if (iy < 0 || iy >= H) continue;
#pragma unroll
            for (int fx = 0; fx < 4; ++fx) {
                const int ix = ox * 2 + fx - 1;
                if (ix < 0 || ix >= W) continue;
                acc += (kFir1[fy] * kFir1[fx]) * __ldg(x + (((int64_t)n * H + iy) * W + ix) * C + c);
            }
        }
        y[i] = acc;
    }
}
}  // namespace

extern "C" int n3d_styles(const float* ws, int N, int num_ws, int wdim, const float* affine_w, const float* affine_b,
                          const int32_t* row_widx, const float* row_scale, const int64_t* row_ooff, const int32_t* row_cin,
                          float* styles, int rows, void* stream) {
    N3D_CHECK_ARG(ws && affine_w && affine_b && row_widx && row_scale && row_ooff && row_cin && styles, "n3d_styles: null pointer");
    N3D_CHECK_ARG(wdim % 4 == 0 && rows > 0 && N > 0, "n3d_styles: bad sizes");
    styles_kernel<<<grid_for((int64_t)rows * 32, 256), 256, 0, (cudaStream_t)stream>>>(ws, N, num_ws, wdim, affine_w, affine_b, row_widx,
                                                                                      row_scale, row_ooff, row_cin, styles, rows);
    N3D_CHECK_LAUNCH("n3d_styles");
    return N3D_OK;
}

extern "C" int n3d_demod(const float* styles, const float* wsq, const int64_t* row_woff, const int32_t* row_cin,
                         const int64_t* row_soff, const int64_t* row_ooff, const int32_t* row_cout, float* dcoef, int rows, int N,
                         void* stream) {
    N3D_CHECK_ARG(styles && wsq && row_woff && row_cin && row_soff && row_ooff && row_cout && dcoef, "n3d_demod: null pointer");
    demod_kernel<<<grid_for((int64_t)rows * 32, 256), 256, 0, (cudaStream_t)stream>>>(styles, wsq, row_woff, row_cin, row_soff, row_ooff,
                                                                                     row_cout, dcoef, rows, N);
    N3D_CHECK_LAUNCH("n3d_demod");
    return N3D_OK;
}

// Rows per thread strip of the register-tiled FIR kernels: 16 (3 re-read halo rows per strip) for launches with >= 1024 threads per
// SM, halved down to 4 for smaller ones.  Measured on B200 (tools/bench_layers.py): S=1 is 1.3-1.6x slower than S=4 at every size,
// S=64 loses on everything below 256^2.
static int fir_strip_rows(int64_t threads_per_row, int rows, int num_sms) {
    int S = 16;
    while (S > 4 && threads_per_row * n3d_div_up(rows, S) < (int64_t)num_sms * 1024) S >>= 1;
    return min(S, rows);
}

extern "C" int n3d_modulate_split(const float* x, int64_t npix_per_img, int N, int C, const float* style, void* hi, void* lo,
                                  int out_cstride, int out_coff, void* stream) {
    N3D_CHECK_ARG(x && hi && lo, "n3d_modulate_split: null pointer");
    N3D_CHECK_ARG(C % 4 == 0 && out_cstride % 4 == 0 && out_coff % 4 == 0, "n3d_modulate_split: channels must be multiples of 4");
    const int64_t total = (int64_t)N * npix_per_img * (C / 4);
    modulate_split_kernel<<<grid_for(total, 256, 16), 256, 0, (cudaStream_t)stream>>>(x, npix_per_img, N, C, style, (__nv_bfloat16*)hi,
                                                                                     (__nv_bfloat16*)lo, out_cstride, out_coff);
    N3D_CHECK_LAUNCH("n3d_modulate_split");
    return N3D_OK;
}

// The streamed FIR kernels may run on this input: 16-byte aligned, and not switched off by N3D_FIR_STREAM=0 (register-tiled kernels
// for every shape: A/B runs, and the reference the tests hold the streamed kernels to).  Read at every call, so that one process can
// compare both forms.
static bool fir_streamable(const float* x) {
    const char* e = getenv("N3D_FIR_STREAM");
    return (!e || atoi(e) != 0) && ((uintptr_t)x & 15) == 0;
}

// Kernel and geometry of one FIR launch.  rows > 0: the streamed kernel, tiles of `rows` x `cols` (output rows x columns up,
// sub-pixel rows x columns down) through a ring of NR stages in `smem` bytes of dynamic shared memory.  rows == 0: the register-tiled
// kernel in strips of S rows.
struct FirPlan { int grid, rows, cols, NR, smem, S; };

// FIR-up epilogue: streamed for the large layers -- (TC / 2) * (C / 4) == 256 consumer threads, at least one CTA per SM.
static FirPlan fir_up_plan(const float* raw, int N, int H2, int W2, int C, int num_sms) {
    FirPlan P{};
    const int TC = (C >= 64 && C <= 512 && (2048 % C) == 0) ? 2048 / C : 0;
    if (TC >= 4 && W2 % TC == 0 && fir_streamable(raw)) {
        // rows per tile: the candidate with the best (fill of the last wave of 2 CTAs per SM) x (1 - vertical halo); measured sweep in
        // DESIGN.md section 3.3.  The tiling does not change the arithmetic (results are bit-identical for every tile height).
        double best = 0.0;
        for (int tr = 32; tr <= 128; tr *= 2) {
            if (H2 % tr) continue;
            const int64_t ctas = (int64_t)N * (W2 / TC) * (H2 / tr);
            if (ctas < num_sms) continue;
            const double eff = (double)ctas / (double)(n3d_div_up(ctas, 2 * num_sms) * 2 * num_sms) * tr / (tr + 3);
            if (eff > best) { best = eff; P.rows = tr; P.grid = (int)ctas; }
        }
    }
    if (P.rows) {
        const int row_bytes = (TC + 3) * C * 4;
        P.cols = TC;
        P.NR = min(4, (100 * 1024) / row_bytes);               // deeper rings measured 1-3 % slower (sweep 4 / 6 / 8 / 10)
        P.smem = P.NR * row_bytes + 16 * P.NR;
    } else {
        P.S = fir_strip_rows((int64_t)N * (W2 / 2) * (C / 4), H2 / 2, num_sms);
        P.grid = grid_for((int64_t)N * n3d_div_up(H2 / 2, P.S) * (W2 / 2) * (C / 4), 256, 16);
    }
    return P;
}

// FIR-down split: streamed for the large layers -- TSC * (C / 4) == 256 consumer threads, at least one CTA per SM.
static FirPlan fir_down_plan(const float* x, int N, int H, int W, int C, int num_sms) {
    FirPlan P{};
    const int c4n = C / 4, SH = (H + 2) / 2, SW = (W + 2) / 2;
    const int TSC = (c4n >= 8 && c4n <= 128 && 256 % c4n == 0) ? 256 / c4n : 0;
    if (TSC && fir_streamable(x)) {
        for (int ts = 32; ts >= 16; ts >>= 1) {
            const int64_t ctas = (int64_t)N * n3d_div_up(SW, TSC) * n3d_div_up(SH, ts);
            if (ctas >= num_sms) { P.rows = ts; P.grid = (int)ctas; break; }
        }
    }
    if (P.rows) {
        P.cols = TSC;
        P.NR = 4;
        P.smem = P.NR * (2 * TSC + 3) * C * 4 + 16 * P.NR;
    } else {
        P.S = fir_strip_rows((int64_t)N * SW * c4n, SH, num_sms);
        P.grid = grid_for((int64_t)N * n3d_div_up(SH, P.S) * SW * c4n, 256, 16);
    }
    return P;
}

// EpiParams of one epilogue launch, after the checks the epilogue relies on: an lrelu / linear activation and float4-aligned outputs.
// Errors name the entry point `who`.
static int epi_params(EpiParams& E, const char* who, const float* dcoef, const float* bias, const float* noise, int64_t noise_nstride,
                      float gain, float slope, float clamp, const N3DSplitOut out[2], float* out_f32, int f32_cstride, int f32_coff) {
    N3D_CHECK_ARG(gain > 0.f && slope >= 0.f && slope <= 1.f, "%s: needs gain > 0 and 0 <= slope <= 1 (lrelu / linear)", who);
    for (int k = 0; k < 2; ++k)
        N3D_CHECK_ARG(!out[k].hi || (out[k].cstride % 4 == 0 && out[k].coff % 4 == 0), "%s: unaligned split output", who);
    N3D_CHECK_ARG(!out_f32 || (f32_cstride % 4 == 0 && f32_coff % 4 == 0), "%s: unaligned fp32 output", who);
    E = EpiParams{dcoef, bias, noise, noise_nstride, gain, slope, clamp, {out[0], out[1]}, out_f32, f32_cstride, f32_coff};
    return N3D_OK;
}

extern "C" int n3d_fir_up_epilogue(const float* raw, int N, int H2, int W2, int C, const float* dcoef, const float* bias,
                                   const float* noise, int64_t noise_nstride, float gain, float slope, float clamp,
                                   const N3DSplitOut out[2], float* out_f32, int f32_cstride, int f32_coff, void* stream) {
    N3D_CHECK_ARG(raw && out, "n3d_fir_up_epilogue: null pointer");
    N3D_CHECK_ARG(C % 4 == 0, "n3d_fir_up_epilogue: C must be a multiple of 4");
    EpiParams E;
    if (int e = epi_params(E, "n3d_fir_up_epilogue", dcoef, bias, noise, noise_nstride, gain, slope, clamp, out, out_f32, f32_cstride, f32_coff))
        return e;
    N3D_CHECK_ARG(H2 % 2 == 0 && W2 % 2 == 0, "n3d_fir_up_epilogue: output size must be even");
    N3DDeviceState* D = n3d_device_state();
    if (!D) return N3D_ERR_CUDA;
    const FirPlan P = fir_up_plan(raw, N, H2, W2, C, D->num_sms);
    if (P.rows) {
        if (int e = n3d_smem_optin(D, N3D_CFG_FIR_STREAM, (const void*)fir_up_stream_kernel, kFsSmemLimit, "n3d_fir_up_epilogue")) return e;
        fir_up_stream_kernel<<<P.grid, kFsThreads, P.smem, (cudaStream_t)stream>>>(raw, N, H2, W2, C, P.cols, P.rows, P.NR, E);
    } else {
        fir_up_epilogue_kernel<<<P.grid, 256, 0, (cudaStream_t)stream>>>(raw, N, H2, W2, C, P.S, E);
    }
    N3D_CHECK_LAUNCH("n3d_fir_up_epilogue");
    return N3D_OK;
}

extern "C" int n3d_splitk_epilogue(const float* partial, int S, int64_t split_stride, int N, int H, int W, int C, const float* dcoef,
                                   const float* bias, const float* noise, int64_t noise_nstride, float gain, float slope, float clamp,
                                   const N3DSplitOut out[2], float* out_f32, int f32_cstride, int f32_coff, void* stream) {
    N3D_CHECK_ARG(partial && out && S >= 1 && N > 0 && H > 0 && W > 0, "n3d_splitk_epilogue: bad args");
    N3D_CHECK_ARG(C % 4 == 0 && split_stride % 4 == 0 && ((uintptr_t)partial & 15) == 0, "n3d_splitk_epilogue: C and the split stride must be multiples of 4");
    EpiParams E;
    if (int e = epi_params(E, "n3d_splitk_epilogue", dcoef, bias, noise, noise_nstride, gain, slope, clamp, out, out_f32, f32_cstride, f32_coff))
        return e;
    const int64_t total = (int64_t)N * H * W * (C / 4);
    splitk_epilogue_kernel<<<grid_for(total, 256, 16), 256, 0, (cudaStream_t)stream>>>(partial, S, split_stride, N, H, W, C, E);
    N3D_CHECK_LAUNCH("n3d_splitk_epilogue");
    return N3D_OK;
}

extern "C" int n3d_fir_down_split(const float* x, int N, int H, int W, int C, void* hi, void* lo, void* stream) {
    N3D_CHECK_ARG(x && hi && lo, "n3d_fir_down_split: null pointer");
    N3D_CHECK_ARG(C % 4 == 0 && H % 2 == 0 && W % 2 == 0, "n3d_fir_down_split: C %% 4 and even H, W required");
    N3DDeviceState* D = n3d_device_state();
    if (!D) return N3D_ERR_CUDA;
    const FirPlan P = fir_down_plan(x, N, H, W, C, D->num_sms);
    if (P.rows) {
        if (int e = n3d_smem_optin(D, N3D_CFG_FIR_DOWN_STREAM, (const void*)fir_down_stream_kernel, kFsSmemLimit, "n3d_fir_down_split")) return e;
        fir_down_stream_kernel<<<P.grid, kFsThreads, P.smem, (cudaStream_t)stream>>>(x, N, H, W, C, P.cols, P.rows, P.NR, (__nv_bfloat16*)hi,
                                                                                      (__nv_bfloat16*)lo);
    } else {
        fir_down_split_kernel<<<P.grid, 256, 0, (cudaStream_t)stream>>>(x, N, H, W, C, P.S, (__nv_bfloat16*)hi, (__nv_bfloat16*)lo);
    }
    N3D_CHECK_LAUNCH("n3d_fir_down_split");
    return N3D_OK;
}

extern "C" int n3d_upsample2d_nhwc(const float* x, int N, int H, int W, int C, float* y, int y_nchw, void* stream) {
    N3D_CHECK_ARG(x && y, "n3d_upsample2d_nhwc: null pointer");
    if (C % 4 == 0)
        upsample2d_kernel<4><<<grid_for((int64_t)N * H * W * (C / 4), 256, 16), 256, 0, (cudaStream_t)stream>>>(x, N, H, W, C, y, y_nchw);
    else
        upsample2d_kernel<1><<<grid_for((int64_t)N * H * W * C, 256, 16), 256, 0, (cudaStream_t)stream>>>(x, N, H, W, C, y, y_nchw);
    N3D_CHECK_LAUNCH("n3d_upsample2d_nhwc");
    return N3D_OK;
}

extern "C" int n3d_downsample2d_nhwc(const float* x, int N, int H, int W, int C, float* y, void* stream) {
    N3D_CHECK_ARG(x && y && H % 2 == 0 && W % 2 == 0, "n3d_downsample2d_nhwc: bad args");
    downsample2d_kernel<<<grid_for((int64_t)N * (H / 2) * (W / 2) * C, 256, 16), 256, 0, (cudaStream_t)stream>>>(x, N, H, W, C, y);
    N3D_CHECK_LAUNCH("n3d_downsample2d_nhwc");
    return N3D_OK;
}
