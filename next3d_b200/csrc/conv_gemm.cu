// Implicit-GEMM convolution on tcgen05 tensor cores (sm_100a) -- the dense contraction of every conv layer of the
// generator (modulated 3x3 / 1x1, transposed-conv parity classes, stride-2 convs, ToRGB).
//
//   M = 128 output pixels per tile (TN x TH x TW patch), N = block_n output channels, K = taps x Cin.
//   A (activations, NHWC bf16, split hi/lo) is fetched per (tap, 64-channel chunk) as one 4-D TMA box whose
//   coordinates are shifted by the tap offset; out-of-range rows/columns are zero-filled by TMA, which *is* the
//   convolution padding.  B (weights [T, Cout, Cin] bf16 hi/lo) is a 3-D TMA box.  Both land in shared memory in the
//   K-major SWIZZLE_128B layout that tcgen05.mma consumes directly.
//   Precision: fp32 = hi + lo with bf16 hi, lo; acc += Ahi*Bhi + Ahi*Blo + Alo*Bhi (3 MMAs, fp32 accumulate in TMEM)
//   reproduces an fp32 convolution to ~2^-16 relative -- inside the 1e-3 end-to-end budget where single-pass
//   bf16/fp16/tf32 is not (SURVEY.md section 7 "Precision vs tensor cores").
//   Warp roles (256 threads, persistent over tiles): warp 0 = TMA producer, warp 1 = MMA issuer (one elected lane),
//   warp 2 = TMEM allocator, warps 4-7 = epilogue (TMEM -> registers -> fused demod/noise/bias/lrelu/clamp ->
//   next layer's modulation -> bf16 split / fp32 stores).  Two TMEM accumulator buffers overlap the epilogue of
//   tile i with the MMAs of tile i+1.
#include <cstdlib>
#include "common.cuh"
#include "../../include/next3d_b200.h"
#include <cuda.h>
#include "tc_ptx.cuh"

namespace {
using namespace n3d_tc;

constexpr int kBlockM = 128;
// K per pipeline stage: 64 bf16 (128-byte rows, SWIZZLE_128B) or, for Cin % 64 == 32 (the 32-channel feature images),
// 32 bf16 (64-byte rows, SWIZZLE_64B) so that no TMA box hangs over the channel extent.
constexpr int kThreads = 384;                 // warps 0-3: producer / MMA / TMEM alloc / spare; 4-7 and 8-11: two epilogue groups
constexpr int kMaxBlockN = 256;
constexpr int kMinTiles = 64;                 // see the block_n choice in launch_conv
constexpr int kMinTilesSplit = 128;           // same for split-K launches
constexpr int kStageArrays = 8;               // dcoef | bias | style0 | style1 | up to 4 modulated ToRGB weight rows

struct KParams {
    CUtensorMap tmA_hi, tmA_lo, tmB_hi, tmB_lo;
    int N, MH, MW, Cout;
    int TW, TH, TN;                  // TW*TH*TN == 128, all powers of two
    int tiles_i, tiles_n;
    // up to 4 sub-problems sharing operands / tile shape / epilogue (the 4 output-parity classes of a stride-2 transposed conv)
    int nsub;
    struct Sub { int tap_begin, ntaps, MH, MW, tiles_x, tiles_y, oy_off, ox_off, tile_end; } sub[4];
    int splits; long long split_stride;   // split-K: work item = (tile, K slice); slice s writes its raw partial sums to out_f32 + s * split_stride
    int pair, tile_h, acc_half;        // pair = 1: a CTA tile is two vertically stacked 128-row sub-tiles (M = 256) sharing one weight tile
    int block_n, acc_stride, tmem_cols, stages, stage_bytes, b_bytes, a_bytes, block_k;
    int cin_chunks, ntaps, nprod, a_img_stride;
    N3DConvTap taps[9];
    int mode;
    const float* dcoef; const float* bias; const float* noise; int64_t noise_nstride;
    float gain, slope, clamp;
    N3DSplitOut out[2];
    float* out_f32; int f32_cstride, f32_coff, f32_nchw, f32_accumulate;
    N3DFusedRgb rgb;                 // optional fused ToRGB (<= 4 image channels), see include/next3d_b200.h
    int oy_mul, ox_mul, OH, OW;
    int* err_flag;
};

__device__ __forceinline__ int staged_rgb_channels(const KParams& P) { return (P.rgb.out && P.TN == 1 && P.mode == 0 && P.tiles_n == 1) ? P.rgb.channels : 0; }

struct TileInfo { int sub, tn, x0, y0, n0, split; };
// Tiles are numbered sub-problem-major (all tiles of parity class 0, then class 1, ...), n-tile minor.  Interleaving the classes
// of one spatial tile across neighbouring CTAs (better L2 re-use of the shared activation tile) was measured 0-35 % slower on
// B200: the kernel is bound by L2->SM fill bandwidth, not DRAM, and the interleaved schedule balances the 4/2/2/1-tap classes worse.
__device__ __forceinline__ TileInfo decode_tile(const KParams& P, int tile) {
    const int split = tile % P.splits;                         // K slices of one tile are neighbouring work items (run concurrently)
    tile /= P.splits;
    int sidx = 0, begin = 0;
    while (sidx + 1 < P.nsub && tile >= P.sub[sidx].tile_end) { begin = P.sub[sidx].tile_end; ++sidx; }
    const int local = tile - begin;
    TileInfo t;
    t.sub = sidx;
    t.tn = local % P.tiles_n;
    const int tm = local / P.tiles_n, tx = P.sub[sidx].tiles_x, ty = P.sub[sidx].tiles_y;
    t.x0 = (tm % tx) * P.TW;
    t.y0 = ((tm / tx) % ty) * P.tile_h;
    t.n0 = (tm / (tx * ty)) * P.TN;
    t.split = split;
    return t;
}

// K-step range [kb, ke) of a work item: all taps x channel chunks, or the item's slice of them under split-K.
__device__ __forceinline__ void k_range(const KParams& P, const TileInfo& t, int& kb, int& ke) {
    const int nsteps = P.sub[t.sub].ntaps * P.cin_chunks, per = (nsteps + P.splits - 1) / P.splits;
    kb = t.split * per;
    ke = min(nsteps, kb + per);
}

// ---------------------------------------------------------------------------------------------- the kernel
__global__ void __launch_bounds__(kThreads, 1) conv_gemm_kernel(const __grid_constant__ KParams P) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    // dynamic smem base is only guaranteed 16-B aligned: round up to 1024 (SWIZZLE_128B atoms)
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t bar_base = smem_base + (uint32_t)P.stages * (uint32_t)P.stage_bytes;   // 8-byte aligned
    // barriers: full[stages], empty[stages], tmem_full[2], tmem_empty[2]; then the TMEM base address word
    auto full_bar = [&](int s) { return bar_base + 8u * (uint32_t)s; };
    auto empty_bar = [&](int s) { return bar_base + 8u * (uint32_t)(P.stages + s); };
    auto tfull_bar = [&](int a) { return bar_base + 8u * (uint32_t)(2 * P.stages + a); };
    auto tempty_bar = [&](int a) { return bar_base + 8u * (uint32_t)(2 * P.stages + 2 + a); };
    const uint32_t tmem_slot = bar_base + 8u * (uint32_t)(2 * P.stages + 4);
    const uint32_t stage_area_off = ((tmem_slot + 16u + 15u) & ~15u) - smem_u32(smem_raw);   // byte offset of the epilogue staging area

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&P.tmA_hi); tma_prefetch_desc(&P.tmB_hi);
        if (P.nprod == 3) { tma_prefetch_desc(&P.tmA_lo); tma_prefetch_desc(&P.tmB_lo); }
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < P.stages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), 4); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"((uint32_t)P.tmem_cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

    const int total_tiles = P.sub[P.nsub - 1].tile_end * P.splits;

    if (warp == 0) {
        // ===================================================== TMA producer
        if (lane == 0) {
            int s = 0; uint32_t ph = 0;
            const uint32_t tx_bytes = (uint32_t)(P.nprod == 3 ? 2 : 1) * (uint32_t)(P.a_bytes + P.b_bytes);
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                const TileInfo ti = decode_tile(P, tile);
                const int tn = ti.tn, x0 = ti.x0, y0 = ti.y0, n0 = ti.n0;
                const int tap_begin = P.sub[ti.sub].tap_begin;
                int kb, ke;
                k_range(P, ti, kb, ke);
                for (int idx = kb; idx < ke; ++idx) {
                    const int t = idx / P.cin_chunks, kc = idx - t * P.cin_chunks;
                    const N3DConvTap tap = P.taps[tap_begin + t];
                    mbar_wait(empty_bar(s), ph ^ 1u, P.err_flag, 1);
                    const uint32_t sa = smem_base + (uint32_t)s * (uint32_t)P.stage_bytes;
                    const uint32_t fb = full_bar(s);
                    mbar_expect_tx(fb, tx_bytes);
                    const int img = n0 + (int)tap.img_off * P.a_img_stride;
                    tma_load_4d(sa, &P.tmA_hi, fb, kc * P.block_k, x0 + tap.dx, y0 + tap.dy, img);
                    tma_load_3d(sa + 2 * P.a_bytes, &P.tmB_hi, fb, kc * P.block_k, tn * P.block_n, tap.wtap);
                    if (P.nprod == 3) {
                        tma_load_4d(sa + P.a_bytes, &P.tmA_lo, fb, kc * P.block_k, x0 + tap.dx, y0 + tap.dy, img);
                        tma_load_3d(sa + 2 * P.a_bytes + P.b_bytes, &P.tmB_lo, fb, kc * P.block_k, tn * P.block_n, tap.wtap);
                    }
                    if (++s == P.stages) { s = 0; ph ^= 1u; }
                }
            }
        }
    } else if (warp == 1) {
        // ===================================================== MMA issuer
        if (lane == 0) {
            // instruction descriptor (cute::UMMA::InstrDescriptor): D=f32 [4,6)=1, A=bf16 [7,10)=1, B=bf16 [10,13)=1,
            // both K-major, N>>3 at [17,23), M>>4 at [24,29)
            const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(P.block_n >> 3) << 17) | ((uint32_t)(kBlockM >> 4) << 24);
            const uint64_t dhi = umma_desc_hi(P.block_k);
            const int k16 = P.block_k / 16;
            int s = 0; uint32_t ph = 0; int cnt = 0;            // cnt: tiles of this CTA so far -> accumulator buffer (parity) + barrier phase
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                int kb, ke;
                k_range(P, decode_tile(P, tile), kb, ke);
                const int ksteps = ke - kb;
                const int acc = cnt & 1;
                const uint32_t acc_ph = (uint32_t)(cnt >> 1) & 1u;
                ++cnt;
                mbar_wait(tempty_bar(acc), acc_ph ^ 1u, P.err_flag, 2);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(acc * P.acc_stride);
                for (int ks = 0; ks < ksteps; ++ks) {
                    mbar_wait(full_bar(s), ph, P.err_flag, 3);
                    tc_fence_after();
                    const uint32_t sa = smem_base + (uint32_t)s * (uint32_t)P.stage_bytes;
                    const uint32_t a_hi = sa, a_lo = sa + (uint32_t)P.a_bytes, b_hi = sa + 2u * (uint32_t)P.a_bytes, b_lo = b_hi + (uint32_t)P.b_bytes;
                    for (int u = 0; u <= P.pair; ++u) {            // pair mode: both sub-tiles consume the same weight tile
                        const uint32_t du = d_tmem + (uint32_t)(u * P.acc_half), au = (uint32_t)u * (uint32_t)(kBlockM * P.block_k * 2);
                        for (int k = 0; k < k16; ++k) {
                            const uint32_t koff = (uint32_t)k * 32u;     // 16 bf16 = 32 bytes inside the swizzle row
                            umma_bf16(du, umma_desc(a_hi + au + koff, dhi), umma_desc(b_hi + koff, dhi), idesc, (ks | k) != 0);
                            if (P.nprod == 3) {
                                umma_bf16(du, umma_desc(a_hi + au + koff, dhi), umma_desc(b_lo + koff, dhi), idesc, 1u);
                                umma_bf16(du, umma_desc(a_lo + au + koff, dhi), umma_desc(b_hi + koff, dhi), idesc, 1u);
                            }
                        }
                    }
                    umma_commit(empty_bar(s));                 // frees the smem stage once these MMAs retire
                    if (++s == P.stages) { s = 0; ph ^= 1u; }
                }
                umma_commit(tfull_bar(acc));                   // accumulator complete -> epilogue
            }
        }
    } else if (warp >= 4) {
        // ===================================================== epilogue: 2 groups x 4 warps; group g drains TMEM accumulator g
        const int g = (warp - 4) >> 2;                         // epilogue group == accumulator buffer it serves
        const int q = warp & 3;                                // TMEM lane quarter this warp may access
        const int row = q * 32 + lane;                         // tile row = TMEM lane
        const int gtid = (warp - 4 - 4 * g) * 32 + lane;       // thread index inside the group (0..127)
        const int tw = row % P.TW, th = (row / P.TW) % P.TH, tnn = row / (P.TW * P.TH);
        // per-group staging of the per-channel epilogue vectors of the current tile: [dcoef | bias | style0 | style1][block_n]
        float* stg = reinterpret_cast<float*>(smem_raw + (stage_area_off + (uint32_t)g * (uint32_t)kStageArrays * (uint32_t)kMaxBlockN * 4u));
        const int nrgb = staged_rgb_channels(P);
        const bool staged = (P.TN == 1) && (P.mode == 0);
        int cnt = 0;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
            const TileInfo ti = decode_tile(P, tile);
            const bool mine = (cnt & 1) == g;                  // this CTA's tiles alternate between the two accumulators / groups
            const uint32_t acc_ph = (uint32_t)(cnt >> 1) & 1u;
            ++cnt;
            if (!mine) continue;
            const int tn = ti.tn, n0 = ti.n0;
            const int x = ti.x0 + tw;
            const int n = n0 + tnn;
            const int ox = x * P.ox_mul + P.sub[ti.sub].ox_off;
            if (staged) {
                // all 4 warps of the group are done with the previous tile's vectors before they are overwritten
                asm volatile("bar.sync %0, 128;" ::"r"(1 + g) : "memory");
                for (int i = gtid; i < 4 * P.block_n; i += 128) {
                    const int arr = i / P.block_n, c = i - arr * P.block_n, co = tn * P.block_n + c;
                    float val = arr == 1 ? 0.f : 1.f;
                    if (co < P.Cout && n0 < P.N) {
                        const float* src = arr == 0 ? P.dcoef : arr == 1 ? P.bias : (arr == 2 ? P.out[0].style : P.out[1].style);
                        if (src) val = __ldg(src + (arr == 1 ? (int64_t)co : (int64_t)n0 * P.Cout + co));
                    }
                    stg[arr * kMaxBlockN + c] = val;
                }
                for (int i = gtid; i < nrgb * P.block_n; i += 128) {          // fused ToRGB: W_rgb[c, co] * style_rgb[n, co]
                    const int c = i / P.block_n, co = i - c * P.block_n;
                    float val = 0.f;
                    if (co < P.Cout && n0 < P.N) val = __ldg(P.rgb.weight + (int64_t)c * P.Cout + co) * __ldg(P.rgb.style + (int64_t)n0 * P.Cout + co);
                    stg[(4 + c) * kMaxBlockN + co] = val;
                }
                asm volatile("bar.sync %0, 128;" ::"r"(1 + g) : "memory");
            }

            mbar_wait(tfull_bar(g), acc_ph, P.err_flag, 4);
            tc_fence_after();
            for (int u = 0; u <= P.pair; ++u) {
            const int y = ti.y0 + u * P.TH + th;
            const int oy = y * P.oy_mul + P.sub[ti.sub].oy_off;
            const bool valid = (n < P.N) && (y < P.sub[ti.sub].MH) && (x < P.sub[ti.sub].MW) && (oy < P.OH) && (ox < P.OW);
            const int64_t opix = ((int64_t)n * P.OH + oy) * P.OW + ox;
            float nz = 0.f;
            if (valid && P.noise) nz = __ldg(P.noise + (int64_t)n * P.noise_nstride + (int64_t)oy * P.OW + ox);
            const uint32_t t_row = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(g * P.acc_stride + u * P.acc_half);
            float racc[4] = {0.f, 0.f, 0.f, 0.f};
            for (int c16 = 0; c16 < P.block_n; c16 += 16) {
                uint32_t r[16];
                __syncwarp();                                  // tcgen05.ld is warp-collective (.sync.aligned)
                tmem_ld16(t_row + (uint32_t)c16, r);
                const int co0 = tn * P.block_n + c16;
                if (!valid || co0 >= P.Cout) continue;
                const int nco = min(16, P.Cout - co0);
                float v[16], s0[16], s1[16];
                if (staged) {
                    const float4* d4 = reinterpret_cast<const float4*>(stg + c16);
                    const float4* b4 = reinterpret_cast<const float4*>(stg + kMaxBlockN + c16);
                    const float4* p4 = reinterpret_cast<const float4*>(stg + 2 * kMaxBlockN + c16);
                    const float4* q4 = reinterpret_cast<const float4*>(stg + 3 * kMaxBlockN + c16);
#pragma unroll
                    for (int j4 = 0; j4 < 4; ++j4) {
                        const float4 d = d4[j4], bb = b4[j4], ps = p4[j4], qs = q4[j4];
                        const float dd[4] = {d.x, d.y, d.z, d.w}, bv[4] = {bb.x, bb.y, bb.z, bb.w};
                        const float pv[4] = {ps.x, ps.y, ps.z, ps.w}, qv[4] = {qs.x, qs.y, qs.z, qs.w};
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const int j = j4 * 4 + e;
                            float a = __uint_as_float(r[j]) * dd[e] + nz + bv[e];
                            a = (a > 0.f ? a : a * P.slope) * P.gain;
                            if (P.clamp >= 0.f) a = fminf(fmaxf(a, -P.clamp), P.clamp);
                            v[j] = a; s0[j] = pv[e]; s1[j] = qv[e];
                        }
                    }
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        if (c < nrgb) {
                            const float4* w4 = reinterpret_cast<const float4*>(stg + (4 + c) * kMaxBlockN + c16);
#pragma unroll
                            for (int j4 = 0; j4 < 4; ++j4) {
                                const float4 w = w4[j4];
                                racc[c] = fmaf(v[j4 * 4], w.x, racc[c]); racc[c] = fmaf(v[j4 * 4 + 1], w.y, racc[c]);
                                racc[c] = fmaf(v[j4 * 4 + 2], w.z, racc[c]); racc[c] = fmaf(v[j4 * 4 + 3], w.w, racc[c]);
                            }
                        }
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        float a = __uint_as_float(r[j]);
                        s0[j] = 1.f; s1[j] = 1.f;
                        if (P.mode == 0 && j < nco) {
                            const int co = co0 + j;
                            if (P.dcoef) a *= __ldg(P.dcoef + (int64_t)n * P.Cout + co);
                            a += nz;
                            if (P.bias) a += __ldg(P.bias + co);
                            a = (a > 0.f ? a : a * P.slope) * P.gain;
                            if (P.clamp >= 0.f) a = fminf(fmaxf(a, -P.clamp), P.clamp);
                            if (P.out[0].style) s0[j] = __ldg(P.out[0].style + (int64_t)n * P.Cout + co);
                            if (P.out[1].style) s1[j] = __ldg(P.out[1].style + (int64_t)n * P.Cout + co);
                        }
                        v[j] = a;
                    }
                }
                // ---- fp32 output (loads of the accumulate path are issued together, before any store, so they overlap)
                if (P.out_f32) {
                    if (P.f32_nchw) {
                        float* dst = P.out_f32 + (((int64_t)n * P.f32_cstride + P.f32_coff + co0) * P.OH + oy) * P.OW + ox;
                        const int64_t cs = (int64_t)P.OH * P.OW;
                        if (P.f32_accumulate) {
                            float old[16];
#pragma unroll
                            for (int j = 0; j < 16; ++j) old[j] = j < nco ? dst[j * cs] : 0.f;
#pragma unroll
                            for (int j = 0; j < 16; ++j) v[j] += old[j];
                        }
#pragma unroll
                        for (int j = 0; j < 16; ++j) if (j < nco) dst[j * cs] = v[j];
                    } else {
                        float* dst = P.out_f32 + (int64_t)ti.split * P.split_stride + opix * P.f32_cstride + P.f32_coff + co0;
                        if (nco == 16 && (((uintptr_t)dst & 31) == 0)) {                 // two full 32-byte sectors per thread
                            if (P.f32_accumulate) {
                                float old[16];
                                ld_global_256(dst, old); ld_global_256(dst + 8, old + 8);
#pragma unroll
                                for (int j = 0; j < 16; ++j) v[j] += old[j];
                            }
                            st_global_256(dst, v); st_global_256(dst + 8, v + 8);
                        } else if (nco == 16 && (((P.f32_cstride | (P.f32_coff + co0)) & 3) == 0)) {
                            if (P.f32_accumulate) {
                                float4 old[4];
#pragma unroll
                                for (int j = 0; j < 4; ++j) old[j] = *reinterpret_cast<const float4*>(dst + 4 * j);
#pragma unroll
                                for (int j = 0; j < 4; ++j) { v[4 * j] += old[j].x; v[4 * j + 1] += old[j].y; v[4 * j + 2] += old[j].z; v[4 * j + 3] += old[j].w; }
                            }
#pragma unroll
                            for (int j = 0; j < 16; j += 4) *reinterpret_cast<float4*>(dst + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
                        } else {
                            if (P.f32_accumulate) {
                                float old[16];
#pragma unroll
                                for (int j = 0; j < 16; ++j) old[j] = j < nco ? dst[j] : 0.f;
#pragma unroll
                                for (int j = 0; j < 16; ++j) v[j] += old[j];
                            }
#pragma unroll
                            for (int j = 0; j < 16; ++j) if (j < nco) dst[j] = v[j];
                        }
                    }
                }
                // ---- split bf16 outputs (next layers' pre-modulated operands)
#pragma unroll
                for (int k = 0; k < 2; ++k) {
                    const N3DSplitOut o = P.out[k];
                    if (!o.hi) continue;
                    uint32_t h[8], l[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        split_bf16x2(v[2 * j] * (k == 0 ? s0[2 * j] : s1[2 * j]), v[2 * j + 1] * (k == 0 ? s0[2 * j + 1] : s1[2 * j + 1]), h[j], l[j]);
                    __nv_bfloat16* dh = (__nv_bfloat16*)o.hi + opix * o.cstride + o.coff + co0;
                    __nv_bfloat16* dl = (__nv_bfloat16*)o.lo + opix * o.cstride + o.coff + co0;
                    if (nco == 16 && ((((uintptr_t)dh | (uintptr_t)dl) & 31) == 0)) {           // one full 32-byte sector per array
                        st_global_256(dh, h); st_global_256(dl, l);
                    } else if (nco == 16 && (((o.cstride | (o.coff + co0)) & 7) == 0)) {
#pragma unroll
                        for (int j = 0; j < 8; j += 4) {
                            *reinterpret_cast<uint4*>(dh + 2 * j) = make_uint4(h[j], h[j + 1], h[j + 2], h[j + 3]);
                            *reinterpret_cast<uint4*>(dl + 2 * j) = make_uint4(l[j], l[j + 1], l[j + 2], l[j + 3]);
                        }
                    } else {
#pragma unroll
                        for (int j = 0; j < 16; ++j)
                            if (j < nco) {
                                dh[j] = __ushort_as_bfloat16((unsigned short)(h[j >> 1] >> ((j & 1) * 16)));
                                dl[j] = __ushort_as_bfloat16((unsigned short)(l[j >> 1] >> ((j & 1) * 16)));
                            }
                    }
                }
            }
            if (nrgb > 0 && valid) {                       // ToRGBLayer: linear bias (+ clamp), added to the up-sampled skip image
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    if (c < nrgb) {
                        float o = racc[c] + __ldg(P.rgb.bias + c);
                        if (P.rgb.clamp >= 0.f) o = fminf(fmaxf(o, -P.rgb.clamp), P.rgb.clamp);
                        float* dst = P.rgb.nchw ? P.rgb.out + (((int64_t)n * nrgb + c) * P.OH + oy) * P.OW + ox : P.rgb.out + opix * nrgb + c;
                        *dst = P.rgb.accumulate ? (*dst + o) : o;
                    }
                }
            }
            }   // u
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty_bar(g));
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)P.tmem_cols) : "memory");
    }
}

// ---------------------------------------------------------------------------------------------- host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess || !p) return nullptr;
        fn = (EncodeTiledFn)p;
    }
    return fn;
}

int make_tmap(CUtensorMap* tm, const void* base, int rank, const uint64_t* dims, const uint32_t* box, int block_k) {
    EncodeTiledFn enc = get_encode_fn();
    if (!enc) { n3d_set_error("cuTensorMapEncodeTiled unavailable (no CUDA driver?)"); return N3D_ERR_CUDA; }
    cuuint64_t gdim[5], gstr[5];
    cuuint32_t bdim[5], estr[5];
    uint64_t stride = 2;
    for (int i = 0; i < rank; ++i) {
        gdim[i] = dims[i]; bdim[i] = box[i]; estr[i] = 1;
        stride *= dims[i];
        if (i < rank - 1) gstr[i] = stride;      // byte stride of dim i+1
    }
    CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), gdim, gstr, bdim, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, block_k == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { n3d_set_error("cuTensorMapEncodeTiled failed with CUresult %d", (int)r); return N3D_ERR_CUDA; }
    return N3D_OK;
}

int pow2_ceil(int v) { int p = 1; while (p < v) p <<= 1; return p; }


}  // namespace

namespace {
struct SubSpec { int ntaps; N3DConvTap taps[9]; int MH, MW, oy_off, ox_off; };

int launch_conv(const N3DConvGemm* p, int nsub, const SubSpec* specs, void* stream) {
    N3D_CHECK_ARG(p && p->a_hi && p->w_hi, "n3d_conv_gemm: null operand");
    N3D_CHECK_ARG(p->nprod == 1 || p->nprod == 3, "n3d_conv_gemm: nprod must be 1 or 3");
    N3D_CHECK_ARG(p->nprod == 1 || (p->a_lo && p->w_lo), "n3d_conv_gemm: nprod 3 needs lo operands");
    N3D_CHECK_ARG(p->Cin >= 8 && p->Cin % 8 == 0, "n3d_conv_gemm: Cin %d must be a multiple of 8 (TMA 16-byte strides)", p->Cin);
    N3D_CHECK_ARG(p->Cout >= 1 && p->N >= 1, "n3d_conv_gemm: bad sizes");
    N3D_CHECK_ARG(((uintptr_t)p->a_hi & 15) == 0 && ((uintptr_t)p->w_hi & 15) == 0, "n3d_conv_gemm: operands must be 16-byte aligned");
    N3D_CHECK_ARG(p->mode == 0 || (p->mode == 1 && p->out_f32), "n3d_conv_gemm: bad mode");
    const int splits = p->splits > 1 ? p->splits : 1;
    N3D_CHECK_ARG(splits == 1 || (p->mode == 1 && nsub == 1 && !p->f32_nchw && !p->f32_accumulate && p->split_stride > 0),
                  "n3d_conv_gemm: split-K needs mode 1 (raw NHWC fp32 partial sums) and a split stride");
    cudaStream_t st = (cudaStream_t)stream;

    KParams K;
    memset(&K, 0, sizeof(K));
    K.N = p->N; K.Cout = p->Cout;
    K.splits = splits; K.split_stride = p->split_stride;
    int maxH = 1, maxW = 1;
    for (int i = 0; i < nsub; ++i) { maxH = max(maxH, specs[i].MH); maxW = max(maxW, specs[i].MW); }
    K.TW = min(16, pow2_ceil(maxW));
    K.TH = min(kBlockM / K.TW, pow2_ceil(maxH));
    K.TN = kBlockM / (K.TW * K.TH);
    K.tiles_i = n3d_div_up(p->N, K.TN);
    K.nsub = nsub;
    int tiles_m = 0, tap_total = 0;
    for (int i = 0; i < nsub; ++i) {
        N3D_CHECK_ARG(specs[i].ntaps >= 1 && specs[i].MH >= 1 && specs[i].MW >= 1, "n3d_conv_gemm: bad sub-problem %d", i);
        K.sub[i].tap_begin = tap_total; K.sub[i].ntaps = specs[i].ntaps;
        for (int t = 0; t < specs[i].ntaps; ++t) {
            N3D_CHECK_ARG(tap_total < 9, "n3d_conv_gemm: more than 9 taps in total");
            N3D_CHECK_ARG(specs[i].taps[t].wtap >= 0 && specs[i].taps[t].wtap < p->T, "n3d_conv_gemm: tap weight slab out of range");
            K.taps[tap_total++] = specs[i].taps[t];
        }
        K.sub[i].MH = specs[i].MH; K.sub[i].MW = specs[i].MW; K.sub[i].oy_off = specs[i].oy_off; K.sub[i].ox_off = specs[i].ox_off;
        K.sub[i].tiles_x = n3d_div_up(specs[i].MW, K.TW); K.sub[i].tiles_y = n3d_div_up(specs[i].MH, K.TH);
        tiles_m += K.sub[i].tiles_x * K.sub[i].tiles_y * K.tiles_i;
    }
    // block_n: the largest legal UMMA N (M=128 needs N % 16 == 0) not exceeding Cout, halved while the launch has fewer than
    // kMinTiles tiles.  Narrow tiles re-fetch the activation tile once per n-tile, so filling all 148 SMs with block_n = 32 tiles is
    // slower than 64 SMs with block_n = 128 (512->512 @16^2, batch 8: 107 -> 60 us; 1024->512 @16^2: 206 -> 110 us; thresholds 64
    // and 96 measured equal, 32 and 148 worse; tools/bench_layers.py).
    const int cout16 = ((p->Cout + 15) / 16) * 16;
    int bn = 16;
    {
        const int cands[6] = {256, 128, 96, 64, 32, 16};
        for (int i = 0; i < 6; ++i) {
            if (cands[i] > cout16) continue;
            if (cands[i] == 96 && cout16 % 96 != 0) continue;
            bn = cands[i];
            break;
        }
        int min_tiles = kMinTiles;
        if (splits > 1) {                                   // split launches: short K loops, so spread over (nearly) all SMs
            min_tiles = kMinTilesSplit;
            if (const char* e = getenv("N3D_SPLITK_MINTILES")) min_tiles = atoi(e);      // A/B diagnostics (tools/bench_splitk.py)
        }
        while (bn > 32 && tiles_m * splits * n3d_div_up(p->Cout, bn) < min_tiles) bn = (bn == 96) ? 32 : bn / 2;
        if (p->rgb.out) {                                   // fused ToRGB needs every output channel of a pixel in one tile
            N3D_CHECK_ARG(cout16 <= 256 && cout16 % 16 == 0, "n3d_conv_gemm: fused ToRGB needs Cout <= 256");
            N3D_CHECK_ARG(p->rgb.channels >= 1 && p->rgb.channels <= 4 && p->rgb.weight && p->rgb.style && p->rgb.bias, "n3d_conv_gemm: bad fused ToRGB descriptor");
            N3D_CHECK_ARG(p->mode == 0 && nsub == 1 && K.TN == 1, "n3d_conv_gemm: fused ToRGB needs mode 0 and >= 128 output positions per image");
            bn = cout16;
        }
    }
    K.block_n = bn;
    K.tiles_n = n3d_div_up(p->Cout, bn);
    // Pair mode (M = 256 per CTA tile): with block_n = 128 the kernel is bound by the L2 -> shared-memory fill rate (measured
    // 12.3 TB/s chip-wide, profiles/r01_ncu_convsr.txt), not by the tensor pipe; two sub-tiles sharing each weight tile cut the
    // bytes per MMA by 25 %.  Only for launches with several waves of tiles.
    K.pair = (bn == 128 && K.TN == 1 && splits == 1 && tiles_m * K.tiles_n >= 8 * 148) ? 1 : 0;
    {
        static int force = -2;
        if (force == -2) { const char* e = getenv("N3D_CONV_PAIR"); force = e ? atoi(e) : -1; }
        if (force == 0) K.pair = 0;
    }
    K.tile_h = K.TH * (1 + K.pair);
    if (K.pair) {
        tiles_m = 0;
        for (int i = 0; i < nsub; ++i) { K.sub[i].tiles_y = n3d_div_up(specs[i].MH, K.tile_h); tiles_m += K.sub[i].tiles_x * K.sub[i].tiles_y * K.tiles_i; }
    }
    K.acc_half = max(32, pow2_ceil(bn));
    K.acc_stride = K.acc_half * (1 + K.pair);
    K.tmem_cols = 2 * K.acc_stride;
    K.block_k = (p->Cin % 64 == 0 || p->Cin % 32 != 0) ? 64 : 32;
    K.a_bytes = (1 + K.pair) * kBlockM * K.block_k * 2;
    K.b_bytes = bn * K.block_k * 2;
    K.stage_bytes = 2 * K.a_bytes + 2 * K.b_bytes;
    K.stages = min(6, (200 * 1024) / K.stage_bytes);      // + 16 KiB epilogue staging + barriers + 1 KiB alignment slack <= 227 KiB
    K.cin_chunks = n3d_div_up(p->Cin, K.block_k);
    if (splits > 1) {                                        // every K slice must own at least one step
        const int nsteps = tap_total * K.cin_chunks, per = n3d_div_up(nsteps, splits);
        N3D_CHECK_ARG(per * (splits - 1) < nsteps, "n3d_conv_gemm: %d K slices for %d K steps", splits, nsteps);
    }
    K.ntaps = tap_total; K.nprod = p->nprod; K.a_img_stride = p->a_img_mul;
    {
        int end = 0;
        for (int i = 0; i < nsub; ++i) { end += K.sub[i].tiles_x * K.sub[i].tiles_y * K.tiles_i * K.tiles_n; K.sub[i].tile_end = end; }
    }
    K.mode = p->mode; K.dcoef = p->dcoef; K.bias = p->bias; K.noise = p->noise; K.noise_nstride = p->noise_nstride;
    K.gain = p->gain; K.slope = p->slope; K.clamp = p->clamp;
    K.out[0] = p->out[0]; K.out[1] = p->out[1];
    K.out_f32 = p->out_f32; K.f32_cstride = p->f32_cstride; K.f32_coff = p->f32_coff; K.f32_nchw = p->f32_nchw;
    K.f32_accumulate = p->f32_accumulate;
    K.rgb = p->rgb;
    K.oy_mul = p->oy_mul; K.ox_mul = p->ox_mul; K.OH = p->OH; K.OW = p->OW;
    K.err_flag = nullptr;       // a protocol timeout traps (the launch fails with an error); no device-side flag is kept

    const uint64_t adims[4] = {(uint64_t)p->Cin, (uint64_t)p->AW, (uint64_t)p->AH, (uint64_t)p->NI};
    const uint32_t abox[4] = {(uint32_t)K.block_k, (uint32_t)K.TW, (uint32_t)K.tile_h, (uint32_t)K.TN};
    const uint64_t wdims[3] = {(uint64_t)p->Cin, (uint64_t)p->Cout, (uint64_t)p->T};
    const uint32_t wbox[3] = {(uint32_t)K.block_k, (uint32_t)bn, 1u};
    int rc;
    if ((rc = make_tmap(&K.tmA_hi, p->a_hi, 4, adims, abox, K.block_k)) != N3D_OK) return rc;
    if ((rc = make_tmap(&K.tmB_hi, p->w_hi, 3, wdims, wbox, K.block_k)) != N3D_OK) return rc;
    if (p->nprod == 3) {
        if ((rc = make_tmap(&K.tmA_lo, p->a_lo, 4, adims, abox, K.block_k)) != N3D_OK) return rc;
        if ((rc = make_tmap(&K.tmB_lo, p->w_lo, 3, wdims, wbox, K.block_k)) != N3D_OK) return rc;
    }

    const int smem = K.stages * K.stage_bytes + 8 * (2 * K.stages + 4) + 32 + 2 * kStageArrays * kMaxBlockN * 4 + 1024;
    N3DDeviceState* D = n3d_device_state();
    if (!D) return N3D_ERR_CUDA;
    if (int e = n3d_smem_optin(D, N3D_CFG_CONV, (const void*)conv_gemm_kernel, 227 * 1024, "n3d_conv_gemm")) return e;
    const int total_tiles = tiles_m * K.tiles_n * splits;
    const int num_sms = D->num_sms;
    const int grid = min(total_tiles, num_sms);
    conv_gemm_kernel<<<grid, kThreads, smem, st>>>(K);
    N3D_CHECK_LAUNCH("n3d_conv_gemm");
    return N3D_OK;
}
}  // namespace

extern "C" int n3d_conv_gemm(const N3DConvGemm* p, void* stream) {
    N3D_CHECK_ARG(p, "n3d_conv_gemm: null descriptor");
    N3D_CHECK_ARG(p->ntaps >= 1 && p->ntaps <= 9, "n3d_conv_gemm: ntaps %d", p->ntaps);
    N3D_CHECK_ARG(p->MH >= 1 && p->MW >= 1, "n3d_conv_gemm: bad M-space");
    SubSpec sp;
    sp.ntaps = p->ntaps;
    for (int i = 0; i < p->ntaps; ++i) sp.taps[i] = p->taps[i];
    sp.MH = p->MH; sp.MW = p->MW; sp.oy_off = p->oy_off; sp.ox_off = p->ox_off;
    return launch_conv(p, 1, &sp, stream);
}

// Stride-2 transposed 3x3 convolution (conv_transpose2d(stride 2), conv2d_resample.py:114-127) as ONE launch: the four
// output-parity classes (a, b) -- out[2p+a, 2q+b] = sum_{ky = a mod 2, kx = b mod 2} W[ky,kx] x[p-(ky-a)/2, q-(kx-b)/2] -- become four
// sub-problems (4 / 2 / 2 / 1 taps) of the same persistent kernel, heaviest first.  p->MH, p->MW = INPUT height/width; the raw fp32
// result [(2H+1), (2W+1)] goes to p->out_f32 (mode 1); taps / offsets / OH / OW of the descriptor are ignored and derived here.
extern "C" int n3d_conv_transposed_gemm(const N3DConvGemm* p, void* stream) {
    N3D_CHECK_ARG(p && p->out_f32, "n3d_conv_transposed_gemm: null descriptor / output");
    N3D_CHECK_ARG(p->T == 9, "n3d_conv_transposed_gemm: needs 3x3 weights (T == 9)");
    N3DConvGemm q = *p;
    q.mode = 1; q.oy_mul = 2; q.ox_mul = 2; q.OH = 2 * p->MH + 1; q.OW = 2 * p->MW + 1; q.a_img_mul = 0;
    SubSpec sp[4];
    const int order[4][2] = {{0, 0}, {0, 1}, {1, 0}, {1, 1}};
    for (int c = 0; c < 4; ++c) {
        const int a = order[c][0], b = order[c][1];
        sp[c].ntaps = 0;
        for (int ky = 0; ky < 3; ++ky)
            for (int kx = 0; kx < 3; ++kx)
                if ((ky - a) % 2 == 0 && (kx - b) % 2 == 0) {
                    N3DConvTap t;
                    t.dy = (int8_t)(-(ky - a) / 2); t.dx = (int8_t)(-(kx - b) / 2); t.img_off = 0; t.wtap = ky * 3 + kx;
                    sp[c].taps[sp[c].ntaps++] = t;
                }
        sp[c].MH = p->MH + 1 - a; sp[c].MW = p->MW + 1 - b; sp[c].oy_off = a; sp[c].ox_off = b;
    }
    return launch_conv(&q, 4, sp, stream);
}
