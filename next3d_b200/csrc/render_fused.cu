// Fused volume renderer for sm_100a, warp-specialised: ray generation, stratified depths, tri-plane bilinear fetch (+ mean over
// planes), MLP decoder (32 -> 64 softplus -> 1 + 32, sigmoid) on tcgen05 tensor cores, coarse compositing weights, importance
// resampling, sort-merge of coarse + fine samples and final alpha compositing in ONE persistent kernel.  Replaces
// RaySampler.forward (ray_sampler.py:24-63), ImportanceRenderer.forward (renderer.py:95-268), OSGDecoder.forward
// (triplane_next3d.py:359-371) and MipRayMarcher2.run_forward (ray_marcher.py:27-66).
//
// One CTA per SM, 16 warps:
//   warps  0-7   E ("epilogue") : two sets of four; warp w owns TMEM lanes 32*(w%4).., set s = w/4 owns hidden units 32s..32s+31 and
//                colour channels 16s..16s+15.  Thread = tile row = one depth sample of one ray in every tile of its group.
//   warps  8-14  G ("gather")   : build the layer-1 A operand in shared memory; work item = 32 rows (a quarter) of a tile, items
//                dealt round-robin to the seven warps; 12 bilinear taps per sample fetched as 128-bit loads, 8 lanes x 4
//                channels per sample.
//   warp  15     MMA issuer (one lane) + TMEM allocation.
// Work unit: a GROUP = 128/L rays (a 4x2 or 2x2 pixel block) x L lanes each, L = 16 (<= 48 samples per pass) or 32 (<= 96).
// A pass of a group is T = ceil(D / L) <= 3 tiles of 128 rows; row = ray_slot * L + j holds sample k = tile * L + j of that ray,
// so a ray's samples always sit in the same L lanes of the same warp and every per-ray phase (transmittance scan, PDF/CDF,
// inverse-CDF sampling, rank merge, weighted colour sum) runs on registers + warp shuffles, no CTA-wide barrier anywhere.
// Tile stream of a CTA: C(0) | C(1) F(0) | C(2) F(1) | ...  (coarse tiles of group r+1 are issued before the fine tiles of
// group r, so the importance sampling of a group never stalls the gather warps).
//
// TMEM (512 columns): [0,64) layer-1 accumulator; [64,192) two hidden-activation buffers (bf16 hi words | lo words) that are the
// A operand of layer 2 (tcgen05.mma with A in tensor memory: no shared-memory round trip, no swizzle); [192,224) two sigma
// accumulators (N = 16, column 0 used); [224,512) nine colour-logit slots of 32 columns (coarse of two groups + fine of one):
// the colour logits never leave TMEM until the final weights are known, then each thread applies the sigmoid and accumulates
// coefficient x colour for its own rows.  Decoder arithmetic: bf16x3 (hi*hi + hi*lo + lo*hi), fp32 accumulate.
#include "common.cuh"
#include "../../include/next3d_b200.h"
#include "tc_ptx.cuh"
#include "render_common.cuh"

namespace {
using namespace n3d_tc;
using namespace n3d_rc;

constexpr int kEWarps = 8, kGWarps = 7;
constexpr int kWarps = kEWarps + kGWarps + 1;
constexpr int kThreads = kWarps * 32;           // 512 (16 warps -> 128 registers per thread)
constexpr int kMaxT = 3;                        // tiles per pass
constexpr unsigned FULL = 0xffffffffu;

constexpr uint32_t kColL1 = 0, kColH = 64, kColSig = 192, kColSlot = 224;

// shared-memory byte offsets (base 1024-aligned)
constexpr int kOffW0hi = 0, kOffW0lo = 4096, kOffWchi = 8192, kOffWclo = 12288, kOffWshi = 16384, kOffWslo = 18432;
constexpr int kNF = 3;                                          // layer-1 A-operand buffers
constexpr int kOffF = 20480;                                    // kNF x (hi 8 KiB | lo 8 KiB)
constexpr int kOffTaps = kOffF + kNF * 16384;                     // 8 warps x [12][32] x (offset, weight)
constexpr int kTapBytesPerWarp = 12 * 32 * 8;
constexpr int kOffEscr = kOffTaps + kGWarps * kTapBytesPerWarp; // per-E-warp scratch
constexpr int kEscrFloats = 960;
constexpr int kOffTfine = kOffEscr + kEWarps * kEscrFloats * 4; // [2][rays per group][Df] fine depths for the gather warps
constexpr int kTfineFloats = 384;
constexpr int kOffBias = kOffTfine + 2 * kTfineFloats * 4;      // b0 * log2e [64] | b1 colour [32] | b1 sigma [1] (+pad)
constexpr int kOffBar = kOffBias + (64 + 32 + 16) * 4;
constexpr int kNumBars = 20;
constexpr int kSmemBytes = kOffBar + kNumBars * 8 + 16;

enum { BAR_FFULL = 0, BAR_FEMPTY = 3, BAR_L1DONE = 6, BAR_L1FREE = 7, BAR_HFULL = 8, BAR_L2DONE = 10, BAR_CFREE = 12, BAR_FFREE = 14,
       BAR_FINE = 15 };

struct FusedK {
    N3DRender p;
    int M;                       // rays per image
    float delta_coarse, scale;
    int Tc, Tf;                  // tiles per coarse / fine pass
    int gw, log2gw;              // pixel block of a group: gw x 2
    int blocks_x, gpi;           // group map: blocks of 4 x 8 groups, groups per image (padded)
    long long total_groups;
    int mode;                    // diagnostics: bit 0 = all taps read texel 0 (no cache misses)
};

// ---------------------------------------------------------------------------------------------------------------- group -> rays
struct RayId {
    int n, row, col;
    bool ok;
    long long gr;
};
__device__ __forceinline__ RayId ray_of(const FusedK& K, int gg, int rs) {
    RayId r;
    const int n = gg / K.gpi;
    const int q = gg - n * K.gpi;
    const int blk = q >> 5, inb = q & 31;
    const int byi = blk / K.blocks_x, bxi = blk - byi * K.blocks_x;
    const int tx = bxi * 4 + (inb & 3), ty = byi * 8 + (inb >> 2);
    r.col = tx * K.gw + (rs & (K.gw - 1));
    r.row = ty * 2 + (rs >> K.log2gw);
    r.n = n;
    r.ok = r.col < K.p.res && r.row < K.p.res;
    r.gr = (long long)n * K.M + (long long)r.row * K.p.res + r.col;
    return r;
}

struct Ray {
    float ox, oy, oz, dx, dy, dz;
    uint32_t img4;
    long long gr;
    bool ok;
};
// ray_sampler.py:43-63 for pixel (row i, column j)
__device__ __forceinline__ Ray make_ray(const FusedK& K, int gg, int rs) {
    const N3DRender& P = K.p;
    const RayId id = ray_of(K, gg, rs);
    Ray r;
    r.ok = id.ok;
    r.gr = id.gr;
    r.img4 = (uint32_t)id.n * (uint32_t)(3 * P.PH * P.PW * 128);       // byte offset of the image's planes
    r.ox = r.oy = r.oz = r.dx = r.dy = r.dz = 0.f;
    if (id.ok) {
        const float inv = 1.f / (float)P.res, half = 0.5f / (float)P.res;
        const float xc = (float)id.col * inv + half, yc = (float)id.row * inv + half;
        const float* I = P.intrinsics + id.n * 9;
        const float fx = __ldg(I), sk = __ldg(I + 1), cx = __ldg(I + 2), fy = __ldg(I + 4), cy = __ldg(I + 5);
        const float xl = (xc - cx + cy * sk / fy - sk * yc / fy) / fx;
        const float yl = (yc - cy) / fy;
        const float* C = P.cam2world + id.n * 16;
        float wv[3], o[3];
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            wv[a] = __ldg(C + a * 4) * xl + __ldg(C + a * 4 + 1) * yl + __ldg(C + a * 4 + 2) + __ldg(C + a * 4 + 3);
            o[a] = __ldg(C + a * 4 + 3);
            wv[a] -= o[a];
        }
        const float nrm = fmaxf(sqrtf(wv[0] * wv[0] + wv[1] * wv[1] + wv[2] * wv[2]), 1e-12f);
        r.ox = o[0]; r.oy = o[1]; r.oz = o[2];
        r.dx = wv[0] / nrm; r.dy = wv[1] / nrm; r.dz = wv[2] / nrm;
    }
    return r;
}

__device__ __forceinline__ float coarse_depth(const FusedK& K, uint64_t seed, long long gr, int k) {
    const N3DRender& P = K.p;
    const float u = P.u_coarse ? __ldg(P.u_coarse + gr * P.depth_coarse + k) : hash_uniform(seed, (uint64_t)(gr * P.depth_coarse + k));
    return linspace_at(P.ray_start, P.ray_end, P.depth_coarse, k) + u * K.delta_coarse;
}

// ---------------------------------------------------------------------------------------------------------------- gather warps
// 12 bilinear taps of one sample (3 planes x 4 corners; plane 0 <- (x,y), 1 <- (x,z), 2 <- (z,y); grid_sample zeros padding,
// align_corners=False): byte offset of the texel + weight / 3.  Zero-weight taps all point at texel 0.
__device__ __forceinline__ void setup_taps(uint2* __restrict__ taps, int lane, float px, float py, float pz, bool valid, uint32_t img4, int PH,
                                           int PW, float scale) {
    const float x = scale * px, y = scale * py, z = scale * pz;
#pragma unroll
    for (int pl = 0; pl < 3; ++pl) {
        const float gx = pl == 2 ? z : x, gy = pl == 1 ? z : y;
        const float ix = ((gx + 1.f) * (float)PW - 1.f) * 0.5f, iy = ((gy + 1.f) * (float)PH - 1.f) * 0.5f;
        const float flx = floorf(ix), fly = floorf(iy);
        const float fx = ix - flx, fy = iy - fly;
        const int x0 = (int)fminf(fmaxf(flx, -2.f), (float)PW), y0 = (int)fminf(fmaxf(fly, -2.f), (float)PH);
        const uint32_t pbase = img4 + (uint32_t)(pl * PH * PW) * 128u;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int xi = x0 + (c & 1), yi = y0 + (c >> 1);
            const float wx = (c & 1) ? fx : 1.f - fx, wy = (c >> 1) ? fy : 1.f - fy;
            const bool inside = valid && xi >= 0 && xi < PW && yi >= 0 && yi < PH;
            const float w = inside ? wx * wy * (1.f / 3.f) : 0.f;            // 1/3: mean over the three planes
            const uint32_t off = inside ? pbase + (uint32_t)(yi * PW + xi) * 128u : 0u;
            taps[(pl * 4 + c) * 32 + lane] = make_uint2(off, __float_as_uint(w));
        }
    }
}

// 32 samples whose taps sit in `taps`: lanes = 8 samples x 4 channel octets per step (4 steps); every tap is one 256-bit load per
// lane (four lanes cover the texel's 128-byte line), accumulated with packed fp32x2 FMAs; the mean feature goes straight into the
// K-major SWIZZLE_64B bf16 (hi, lo) A-operand tile rows row0..row0+31 as one 16-byte store per lane and operand half.
// Weights already carry the 1/3 of the plane mean.
__device__ __forceinline__ void gather_rows(const float* __restrict__ planes, const uint2* __restrict__ taps, uint8_t* __restrict__ f_hi,
                                            uint8_t* __restrict__ f_lo, int row0, int lane) {
    const int c8 = lane & 3, s8 = lane >> 2;
    const char* const base = reinterpret_cast<const char*>(planes) + c8 * 32;
    const uint2* const tl = taps + s8;                          // + tap * 32 + step * 8
#pragma unroll 1
    for (int step = 0; step < 4; ++step) {
        float2 acc[4];
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            uint2 tp[6];
            float v[6][8];
#pragma unroll
            for (int i = 0; i < 6; ++i) tp[i] = tl[(half * 6 + i) * 32 + step * 8];
#pragma unroll
            for (int i = 0; i < 6; ++i) ldg_nc_256(reinterpret_cast<const float*>(base + tp[i].x), v[i]);
#pragma unroll
            for (int i = 0; i < 6; ++i) {
                const float wt = __uint_as_float(tp[i].y);
                const float2 w2 = make_float2(wt, wt);
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const float2 x = make_float2(v[i][2 * c], v[i][2 * c + 1]);
                    acc[c] = (half == 0 && i == 0) ? __fmul2_rn(w2, x) : __ffma2_rn(w2, x, acc[c]);
                }
            }
        }
        uint32_t h[4], l[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) split_bf16x2(acc[c].x, acc[c].y, h[c], l[c]);
        const uint32_t off = sw64_off(row0 + step * 8 + s8, c8 * 16);
        *reinterpret_cast<uint4*>(f_hi + off) = make_uint4(h[0], h[1], h[2], h[3]);
        *reinterpret_cast<uint4*>(f_lo + off) = make_uint4(l[0], l[1], l[2], l[3]);
    }
}

// ---------------------------------------------------------------------------------------------------------------- per-ray math
// A ray's samples live in the L lanes [lane & ~(L-1), +L) of one warp, sample k = t * L + j in register slot t of lane j.
template <int L>
__device__ __forceinline__ float seg_next(float v, float v_next_slot, int lane) {      // value of sample k + 1
    const float a = __shfl_down_sync(FULL, v, 1);
    const float b = __shfl_sync(FULL, v_next_slot, lane & ~(L - 1));
    return ((lane & (L - 1)) == L - 1) ? b : a;
}
template <int L>
__device__ __forceinline__ float seg_prev(float v, float v_prev_slot, int lane) {      // value of sample k - 1
    const float a = __shfl_up_sync(FULL, v, 1);
    const float b = __shfl_sync(FULL, v_prev_slot, lane | (L - 1));
    return ((lane & (L - 1)) == 0) ? b : a;
}
template <int L>
__device__ __forceinline__ float seg_sum(float v) {
#pragma unroll
    for (int o = L / 2; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}
template <int L, int NT, bool MUL>
__device__ __forceinline__ void seg_scan(float (&x)[NT], int lane) {                  // inclusive scan in sample order
    float carry = MUL ? 1.f : 0.f;
    const int j = lane & (L - 1);
#pragma unroll
    for (int t = 0; t < NT; ++t) {
        float v = x[t];
#pragma unroll
        for (int o = 1; o < L; o <<= 1) {
            const float up = __shfl_up_sync(FULL, v, o);
            if (j >= o) v = MUL ? v * up : v + up;
        }
        v = MUL ? v * carry : v + carry;
        x[t] = v;
        carry = __shfl_sync(FULL, v, lane | (L - 1));
    }
}

// MipRayMarcher2 weights (ray_marcher.py:27-46) of a depth-sorted list of `cnt` samples (d, sg):
//   alpha_k = 1 - exp(-softplus((s_k + s_k+1)/2 - 1) * (t_k+1 - t_k)),  T_k = prod_{i<k} (1 - alpha_i + 1e-10),  w_k = alpha_k T_k
// w_k = 0 for k >= cnt - 1.  tmid_k = (t_k + t_k+1) / 2.
template <int L, int NT>
__device__ __forceinline__ void march_weights(const float (&d)[NT], const float (&sg)[NT], int cnt, int lane, float (&w)[NT], float (&tmid)[NT]) {
    const int j = lane & (L - 1);
    float fac[NT], al[NT];
#pragma unroll
    for (int t = 0; t < NT; ++t) {
        const float dn = seg_next<L>(d[t], t + 1 < NT ? d[t + 1] : 0.f, lane);
        const float sn = seg_next<L>(sg[t], t + 1 < NT ? sg[t + 1] : 0.f, lane);
        const int k = t * L + j;
        float alpha = 0.f;
        if (k < cnt - 1) {
            const float delta = dn - d[t];
            const float dens = softplus_fast((sg[t] + sn) * 0.5f - 1.f);
            // 1 - exp(-x): the MUFU exponential is ~2e-7 off near 1, a BIAS that adds up over ~190 thin intervals; below 1/16 the
            // alternating series is exact to 1e-8 relative
            const float xx = dens * delta;
            const float ser = xx * (1.f - xx * (0.5f - xx * (0.16666667f - xx * (0.041666668f - xx * 0.0083333338f))));
            alpha = xx < 0.0625f ? ser : 1.f - ex2_approx(-kLog2e * xx);
        }
        al[t] = alpha;
        fac[t] = k < cnt - 1 ? (1.f - alpha + 1e-10f) : 1.f;
        tmid[t] = (d[t] + dn) * 0.5f;
    }
    seg_scan<L, NT, true>(fac, lane);
#pragma unroll
    for (int t = 0; t < NT; ++t) {
        const float ex = seg_prev<L>(fac[t], t > 0 ? fac[t - 1] : 1.f, lane);
        w[t] = al[t] * ((t == 0 && j == 0) ? 1.f : ex);
    }
}

// Tile stream of a CTA with n groups: C(0) | C(1) F(0) | ... | C(n-1) F(n-2) | F(n-1); every role walks it with the same iterator.
struct TileIter {
    int n, Tc, Tf;
    int r, kind, t;                 // round, 0 coarse / 1 fine, tile of the pass
    __device__ __forceinline__ TileIter(int n_, int Tc_, int Tf_) : n(n_), Tc(Tc_), Tf(Tf_), r(0), kind(0), t(-1) {}
    __device__ __forceinline__ bool next() {
        ++t;
        for (;;) {
            if (kind == 0) {
                if (r < n && t < Tc) return true;
                kind = 1; t = 0;
            }
            if (r >= 1 && t < Tf) return true;
            kind = 0; t = 0; ++r;
            if (r > n) return false;
        }
    }
    __device__ __forceinline__ int group() const { return kind == 0 ? r : r - 1; }
};

struct Smem {
    uint8_t* base;
    __device__ __forceinline__ uint32_t bar(int i) const { return smem_u32(base + kOffBar + i * 8); }
};

// Decoder weights -> bf16 (hi, lo) B-operand tiles in shared memory, with the activation scalings folded in: layer 1 produces
// x * log2(e); hidden units are kept as softplus / ln2; colour logits as -(x) * log2(e) (the argument of ex2 in the sigmoid).
__device__ __forceinline__ void stage_decoder(uint8_t* sb, const float* __restrict__ w0, const float* __restrict__ b0, const float* __restrict__ w1,
                                              const float* __restrict__ b1, int tid) {
    float* const sB0 = reinterpret_cast<float*>(sb + kOffBias);
    float* const sB1c = sB0 + 64;
    float* const sB1s = sB1c + 32;
    for (int i = tid; i < kHidden * kFeat; i += kThreads) {               // W0 [64][32]: row = hidden unit, K = 32 (SWIZZLE_64B)
        const int n = i / kFeat, k = i - n * kFeat;
        __nv_bfloat16 h, l;
        split_bf16(__ldg(w0 + i) * kLog2e, h, l);        // layer 1 produces x * log2(e) (the argument of ex2)
        *reinterpret_cast<__nv_bfloat16*>(sb + kOffW0hi + sw64_off(n, k * 2)) = h;
        *reinterpret_cast<__nv_bfloat16*>(sb + kOffW0lo + sw64_off(n, k * 2)) = l;
    }
    for (int i = tid; i < 32 * kHidden; i += kThreads) {                  // colour rows of W1 (outputs 1..32) [32][64] (SWIZZLE_128B)
        const int n = i / kHidden, k = i - n * kHidden;
        __nv_bfloat16 h, l;
        split_bf16(-__ldg(w1 + (n + 1) * kHidden + k), h, l);   // hidden units are kept as softplus / ln2; colour logits as -x * log2(e)
        *reinterpret_cast<__nv_bfloat16*>(sb + kOffWchi + sw128_off(n, k * 2)) = h;
        *reinterpret_cast<__nv_bfloat16*>(sb + kOffWclo + sw128_off(n, k * 2)) = l;
    }
    for (int i = tid; i < 16 * kHidden; i += kThreads) {                  // sigma row of W1 (output 0) padded to N = 16
        const int n = i / kHidden, k = i - n * kHidden;
        __nv_bfloat16 h, l;
        split_bf16(n == 0 ? __ldg(w1 + k) * kLn2 : 0.f, h, l);
        *reinterpret_cast<__nv_bfloat16*>(sb + kOffWshi + sw128_off(n, k * 2)) = h;
        *reinterpret_cast<__nv_bfloat16*>(sb + kOffWslo + sw128_off(n, k * 2)) = l;
    }
    for (int i = tid; i < kHidden; i += kThreads) sB0[i] = __ldg(b0 + i) * kLog2e;
    for (int i = tid; i < 32; i += kThreads) sB1c[i] = -kLog2e * __ldg(b1 + 1 + i);
    if (tid == 0) sB1s[0] = __ldg(b1);
}

// layer 1 of tile ti: [128 x 32] x [32 x 64] -> TMEM [kColL1, +64), bf16x3; frees the A buffer and publishes the accumulator
__device__ __forceinline__ void mma_layer1(const Smem& S, uint32_t tmem, int ti) {
    uint8_t* const sb = S.base;
    const uint64_t dhi64 = umma_desc_hi(32);
    const uint32_t id64 = umma_idesc_bf16(64);
    const uint32_t w0h = smem_u32(sb + kOffW0hi), w0l = smem_u32(sb + kOffW0lo);
    const int b = ti % kNF;
    mbar_wait_sleep(S.bar(BAR_FFULL + b), (uint32_t)((ti / kNF) & 1));
    if (ti > 0) mbar_wait_sleep(S.bar(BAR_L1FREE), (uint32_t)((ti - 1) & 1));
    tc_fence_after();
    const uint32_t a_hi = smem_u32(sb + kOffF + b * 16384), a_lo = a_hi + 8192;
#pragma unroll
    for (int k16 = 0; k16 < kFeat / 16; ++k16) {
        const uint32_t ko = (uint32_t)k16 * 32u;
        umma_bf16(tmem + kColL1, umma_desc(a_hi + ko, dhi64), umma_desc(w0h + ko, dhi64), id64, k16 != 0);
        umma_bf16(tmem + kColL1, umma_desc(a_hi + ko, dhi64), umma_desc(w0l + ko, dhi64), id64, 1u);
        umma_bf16(tmem + kColL1, umma_desc(a_lo + ko, dhi64), umma_desc(w0h + ko, dhi64), id64, 1u);
    }
    umma_commit(S.bar(BAR_FEMPTY + b));
    umma_commit(S.bar(BAR_L1DONE));
}
// layer 2 of the tile in hidden buffer b: A from tensor memory; sigma -> [kColSig + 16 b, +16), colour logits -> column col_c
__device__ __forceinline__ void mma_layer2_issue(const Smem& S, uint32_t tmem, int b, uint32_t col_c, bool colours) {
    uint8_t* const sb = S.base;
    const uint64_t dhi128 = umma_desc_hi(64);
    const uint32_t id32 = umma_idesc_bf16(32), id16 = umma_idesc_bf16(16);
    const uint32_t wch = smem_u32(sb + kOffWchi), wcl = smem_u32(sb + kOffWclo), wsh = smem_u32(sb + kOffWshi), wsl = smem_u32(sb + kOffWslo);
    const uint32_t hA = tmem + kColH + 64u * b;
    const uint32_t dC = tmem + col_c, dS = tmem + kColSig + 16u * b;
#pragma unroll
    for (int k16 = 0; k16 < kHidden / 16; ++k16) {
        const uint32_t ko = (uint32_t)k16 * 32u, ka = (uint32_t)k16 * 8u;
        if (colours) {
            umma_bf16_ts(dC, hA + ka, umma_desc(wch + ko, dhi128), id32, k16 != 0);
            umma_bf16_ts(dC, hA + ka, umma_desc(wcl + ko, dhi128), id32, 1u);
            umma_bf16_ts(dC, hA + 32u + ka, umma_desc(wch + ko, dhi128), id32, 1u);
        }
        umma_bf16_ts(dS, hA + ka, umma_desc(wsh + ko, dhi128), id16, k16 != 0);
        umma_bf16_ts(dS, hA + ka, umma_desc(wsl + ko, dhi128), id16, 1u);
        umma_bf16_ts(dS, hA + 32u + ka, umma_desc(wsh + ko, dhi128), id16, 1u);
    }
    umma_commit(S.bar(BAR_L2DONE + b));
}
// layer-1 epilogue of tile ti (thread = row, this set's 32 hidden units): softplus -> bf16 (hi, lo) words -> hidden buffer
__device__ __forceinline__ void epi1_tile(const Smem& S, uint32_t tlane, int eset, int lane, int ti) {
    const float* const sB0 = reinterpret_cast<const float*>(S.base + kOffBias);
    mbar_wait_sleep(S.bar(BAR_L1DONE), (uint32_t)(ti & 1), 20u);
    tc_fence_after();
    uint32_t a[32];
    tmem_ld16_nowait(tlane + kColL1 + 32u * eset, a);
    tmem_ld16_nowait(tlane + kColL1 + 32u * eset + 16u, a + 16);
    tmem_wait_ld();
    reg_fence16(a);
    reg_fence16(a + 16);
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(S.bar(BAR_L1FREE));
    // hidden unit / ln2 = max(log2(1 + 2^min(y, 126)), y) with y = (x + b0) * log2(e): exact softplus for every finite input
    // (for y > 24 the sum rounds to 2^y); ln2 is folded into the layer-2 weights
    uint32_t hi[16], lo[16];
    const float4* b4 = reinterpret_cast<const float4*>(sB0 + 32 * eset);
    float y[32];
#pragma unroll
    for (int c4 = 0; c4 < 8; ++c4) {
        const float4 bb = b4[c4];
        y[c4 * 4] = __uint_as_float(a[c4 * 4]) + bb.x; y[c4 * 4 + 1] = __uint_as_float(a[c4 * 4 + 1]) + bb.y;
        y[c4 * 4 + 2] = __uint_as_float(a[c4 * 4 + 2]) + bb.z; y[c4 * 4 + 3] = __uint_as_float(a[c4 * 4 + 3]) + bb.w;
    }
    // explicit stages over the 32 independent values: the MUFU operations issue back to back instead of one dependent chain per value
    float e[32];
#pragma unroll
    for (int c = 0; c < 32; ++c) e[c] = ex2_approx(fminf(y[c], 126.f));
#pragma unroll
    for (int c = 0; c < 32; ++c) e[c] = lg2_approx(1.f + e[c]);
#pragma unroll
    for (int c = 0; c < 32; ++c) y[c] = fmaxf(e[c], y[c]);
#pragma unroll
    for (int c = 0; c < 16; ++c) split_bf16x2(y[2 * c], y[2 * c + 1], hi[c], lo[c]);
    const uint32_t hb = tlane + kColH + 64u * (ti & 1);
    tmem_st16(hb + 16u * eset, hi);
    tmem_st16(hb + 32u + 16u * eset, lo);
    tmem_wait_st();
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(S.bar(BAR_HFULL + (ti & 1)));
}
__device__ __forceinline__ float read_sigma_tile(const Smem& S, uint32_t tlane, int tj) {
    const float* const sB1s = reinterpret_cast<const float*>(S.base + kOffBias) + 96;
    mbar_wait_sleep(S.bar(BAR_L2DONE + (tj & 1)), (uint32_t)((tj >> 1) & 1), 20u);
    tc_fence_after();
    uint32_t v;
    tmem_ld1_nowait(tlane + kColSig + 16u * (tj & 1), v);
    tmem_wait_ld();
    reg_fence1(v);
    return __uint_as_float(v) + sB1s[0];
}
__device__ __forceinline__ void init_pipeline_barriers(const Smem& S) {
    for (int b = 0; b < kNF; ++b) { mbar_init(S.bar(BAR_FFULL + b), 4); mbar_init(S.bar(BAR_FEMPTY + b), 1); }
    mbar_init(S.bar(BAR_L1DONE), 1);
    mbar_init(S.bar(BAR_L1FREE), kEWarps);
    mbar_init(S.bar(BAR_HFULL + 0), kEWarps); mbar_init(S.bar(BAR_HFULL + 1), kEWarps);
    mbar_init(S.bar(BAR_L2DONE + 0), 1); mbar_init(S.bar(BAR_L2DONE + 1), 1);
}

// ---------------------------------------------------------------------------------------------------------------- the kernel
template <int L>
__global__ void __launch_bounds__(kThreads, 1) render_fused_kernel(const __grid_constant__ FusedK K) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    constexpr int RPW = 32 / L;                 // rays per warp
    const N3DRender& P = K.p;
    Smem S;
    S.base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);       // pointer arithmetic keeps the shared address space
    uint8_t* const sb = S.base;
    float* const sB0 = reinterpret_cast<float*>(sb + kOffBias);         // b0 * log2(e)
    float* const sB1c = sB0 + 64;                                        // colour biases (outputs 1..32)
    float* const sB1s = sB1c + 32;                                       // sigma bias
    float* const sTfine = reinterpret_cast<float*>(sb + kOffTfine);
    uint32_t* const sTmem = reinterpret_cast<uint32_t*>(sb + kOffBar + kNumBars * 8);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int Dc = P.depth_coarse, Df = P.depth_fine, Dt = Dc + Df;
    const int Tc = K.Tc, Tf = K.Tf;
    const uint64_t seed = P.seed_ptr ? (P.seed + __ldg(reinterpret_cast<const unsigned long long*>(P.seed_ptr))) : P.seed;

    // this CTA's contiguous chunk of groups
    const int g_begin = (int)((K.total_groups * blockIdx.x) / gridDim.x);
    const int n_groups = (int)((K.total_groups * (blockIdx.x + 1)) / gridDim.x) - g_begin;

    // ---- one-time setup
    if (tid == 0) {
        init_pipeline_barriers(S);
        mbar_init(S.bar(BAR_CFREE + 0), kEWarps); mbar_init(S.bar(BAR_CFREE + 1), kEWarps);
        mbar_init(S.bar(BAR_FFREE), kEWarps);
        mbar_init(S.bar(BAR_FINE + 0), 4); mbar_init(S.bar(BAR_FINE + 1), 4);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == kWarps - 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(sTmem)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    stage_decoder(sb, P.w0, P.b0, P.w1, P.b1, tid);
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *sTmem;

    // ============================================================================================================ MMA warp
    if (warp == kWarps - 1) {
        if (lane == 0) {
            // slot of the tile before the current one (its layer 2 is issued after the current tile's layer 1)
            int prev_slot = -1, prev_wait = 0, prev_r = 0;      // prev_wait: 0 none, 1 coarse-slot reuse, 2 fine-slot reuse
            int i = 0;
            auto layer1 = [&](int ti) { mma_layer1(S, tmem, ti); };
            auto layer2 = [&](int tj, int slot, int wait_kind, int r) {
                const int b = tj & 1;
                mbar_wait_sleep(S.bar(BAR_HFULL + b), (uint32_t)((tj >> 1) & 1));
                if (wait_kind == 1) mbar_wait_sleep(S.bar(BAR_CFREE + (r & 1)), (uint32_t)(((r >> 1) - 1) & 1));
                if (wait_kind == 2) mbar_wait_sleep(S.bar(BAR_FFREE), (uint32_t)((r - 1) & 1));
                tc_fence_after();
                mma_layer2_issue(S, tmem, b, kColSlot + 32u * slot, true);
            };
            TileIter it(n_groups, Tc, Tf);
            for (;;) {
                const bool has = it.next();
                const int g = it.group();
                // a fine tile directly behind its own group's coarse tiles (single-group CTA): the gather of this tile waits for
                // the importance sampling, which waits for the previous tile's layer 2 -> issue that first
                const bool early = has && it.kind == 1 && prev_slot >= 0 && prev_slot < 6 && prev_r == g;
                if (has && !early) layer1(i);
                if (prev_slot >= 0) layer2(i - 1, prev_slot, prev_wait, prev_r);
                if (has && early) layer1(i);
                if (!has) break;
                prev_slot = it.kind == 0 ? (g & 1) * 3 + it.t : 6 + it.t;
                prev_wait = it.t != 0 ? 0 : (it.kind == 0 ? (g >= 2 ? 1 : 0) : (g >= 1 ? 2 : 0));
                prev_r = g;
                ++i;
            }
        }
    }
    // ============================================================================================================ gather warps
    else if (warp >= kEWarps) {
        const int gw = warp - kEWarps;
        uint2* const taps = reinterpret_cast<uint2*>(sb + kOffTaps + gw * kTapBytesPerWarp);
        int next_item = gw;                                   // item = tile * 4 + quarter
        auto item = [&](int ti, int q, bool fine, int r, int t) {
            const int row = q * 32 + lane, rs = row / L, j = row & (L - 1);
            const Ray ray = make_ray(K, g_begin + r, rs);
            const int k = t * L + j;
            const bool valid = ray.ok && k < (fine ? Df : Dc);
            float depth = 0.f;
            if (fine) {
                mbar_wait_sleep(S.bar(BAR_FINE + (r & 1)), (uint32_t)((r >> 1) & 1), 40u);
                if (valid) depth = sTfine[(r & 1) * kTfineFloats + rs * Df + k];
            } else if (valid) {
                depth = coarse_depth(K, seed, ray.gr, k);
            }
            setup_taps(taps, lane, ray.ox + depth * ray.dx, ray.oy + depth * ray.dy, ray.oz + depth * ray.dz, valid && !(K.mode & 1), ray.img4, P.PH, P.PW,
                       K.scale);
            __syncwarp();
            const int b = ti % kNF;
            if (ti >= kNF) mbar_wait_sleep(S.bar(BAR_FEMPTY + b), (uint32_t)((ti / kNF - 1) & 1), 40u);
            gather_rows(P.planes, taps, sb + kOffF + b * 16384, sb + kOffF + b * 16384 + 8192, q * 32, lane);
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(S.bar(BAR_FFULL + b));
        };
        auto tile = [&](int ti, bool fine, int r, int t) {
            while (next_item < ti * 4 + 4) {
                item(ti, next_item - ti * 4, fine, r, t);
                next_item += kGWarps;
            }
        };
        TileIter it(n_groups, Tc, Tf);
        for (int i = 0; it.next(); ++i) tile(i, it.kind == 1, it.group(), it.t);
    }
    // ============================================================================================================ epilogue warps
    else {
        const int eset = warp >> 2, q = warp & 3;
        const int row = q * 32 + lane, rs = row / L, j = row & (L - 1), rw = lane / L;
        const uint32_t tlane = tmem + ((uint32_t)(q * 32) << 16);
        float* const es = reinterpret_cast<float*>(sb + kOffEscr) + warp * kEscrFloats;
        // per-warp scratch (floats): region A [0, 640) = sd | sg | wb (RPW x (Dt + 2) each), aliased by the cdf during importance sampling
        // and by the u-bucket tables during ranking; tcs at 640 (RPW x Dc), tfs at 736 (RPW x Df), hist at 832 (RPW x (Dc + 1))
        constexpr int NB = 8 * L;                                   // u-buckets per ray (8 per lane)
        const int strD = Dt + 2;
        float* const s_sd = es + rw * strD;                         // sorted depths
        float* const s_sg = es + RPW * strD + rw * strD;
        float* const s_wb = es + 2 * RPW * strD + rw * strD;
        int* const s_ub = reinterpret_cast<int*>(es) + rw * 2 * NB; // [NB] count | prefix << 8, then [NB] member indices (4 bytes)
        float* const s_tc = es + 640 + rw * Dc;
        float* const s_tf = es + 736 + rw * Df;
        int* const s_hist = reinterpret_cast<int*>(es + 832) + rw * (Dc + 1);

        // state of the group in its fine phase (cur) and of the group in its coarse phase (nxt)
        float cur_tc[kMaxT], cur_sc[kMaxT], cur_tf[kMaxT], cur_sf[kMaxT];
        float nxt_tc[kMaxT], nxt_sc[kMaxT], nxt_tf[kMaxT];
        int cur_pk[kMaxT] = {0, 0, 0}, nxt_pk[kMaxT] = {0, 0, 0};     // per fine sample: u-bucket | cdf bin << 16
        long long cur_gr = 0, nxt_gr = 0;
        bool cur_ok = false, nxt_ok = false;
#pragma unroll
        for (int t = 0; t < kMaxT; ++t) { cur_tc[t] = cur_sc[t] = cur_tf[t] = cur_sf[t] = nxt_tc[t] = nxt_sc[t] = nxt_tf[t] = 0.f; }
        float dmin = INFINITY, dmax = -INFINITY;

        // ---- layer-1 epilogue of tile ti: softplus(acc + b0) -> bf16 (hi, lo) words -> hidden buffer (A operand of layer 2)
        auto epi1 = [&](int ti) { epi1_tile(S, tlane, eset, lane, ti); };
        auto read_sigma = [&](int tj) -> float { return read_sigma_tile(S, tlane, tj); };

        // ---- coarse weights -> smoothed pdf -> cdf -> inverse-CDF fine depths (renderer.py:209-268) for the group in `nxt`
        auto importance = [&](int r) {
            float w[kMaxT], tm[kMaxT];
            march_weights<L, kMaxT>(nxt_tc, nxt_sc, Dc, lane, w, tm);
            // max_pool1d(k2,s1,pad1) -> avg_pool1d(k2,s1) -> + 0.01; entries [1:-1] => pdf weights at k = 1 .. Dc-3, + 1e-5
            const int nw = Dc - 3;
            float c[kMaxT];
            float part = 0.f;
#pragma unroll
            for (int t = 0; t < kMaxT; ++t) {
                const float wp = seg_prev<L>(w[t], t > 0 ? w[t - 1] : 0.f, lane);
                const float wn = seg_next<L>(w[t], t + 1 < kMaxT ? w[t + 1] : 0.f, lane);
                const int k = t * L + j;
                c[t] = (k >= 1 && k <= nw) ? (fmaxf(wp, w[t]) + fmaxf(w[t], wn)) * 0.5f + 0.01f + 1e-5f : 0.f;
                part += c[t];
            }
            const float total = seg_sum<L>(part);
#pragma unroll
            for (int t = 0; t < kMaxT; ++t) c[t] = c[t] / total;
            seg_scan<L, kMaxT, false>(c, lane);                     // c[t] = cdf[k], k = 0 .. nw
            float* const cdf = s_sd;
#pragma unroll
            for (int t = 0; t < kMaxT; ++t) {
                const int k = t * L + j;
                if (k <= nw) cdf[k] = c[t];
                if (k < Dc) s_tc[k] = nxt_tc[t];
            }
            __syncwarp();
            float uu[kMaxT];
            int lo[kMaxT], hi[kMaxT];
#pragma unroll
            for (int t = 0; t < kMaxT; ++t) {
                const int jf = t * L + j;
                const bool act = jf < Df && nxt_ok;
                uu[t] = !act ? 0.f : P.u_fine ? __ldg(P.u_fine + nxt_gr * Df + jf) : hash_uniform(seed ^ 0xA5A5A5A5DEADBEEFull, (uint64_t)(nxt_gr * Df + jf));
                lo[t] = 0;
                hi[t] = act ? nw + 1 : 0;                            // searchsorted(cdf, u, right=True): first index with cdf[idx] > u
            }
            const int nit = 32 - __clz(nw + 1);
            for (int it = 0; it < nit; ++it) {                       // the three searches of a lane advance together (independent chains)
#pragma unroll
                for (int t = 0; t < kMaxT; ++t)
                    if (lo[t] < hi[t]) { const int mid = (lo[t] + hi[t]) >> 1; if (cdf[mid] <= uu[t]) lo[t] = mid + 1; else hi[t] = mid; }
            }
#pragma unroll
            for (int t = 0; t < kMaxT; ++t) {
                const int jf = t * L + j;
                float tf = 0.f;
                int below = 0;
                if (jf < Df && nxt_ok) {
                    below = max(lo[t] - 1, 0);
                    const int above = min(lo[t], nw);
                    const float cb = cdf[below], ca = cdf[above];
                    const float bb = 0.5f * (s_tc[below] + s_tc[below + 1]), ba = 0.5f * (s_tc[above] + s_tc[above + 1]);
                    float denom = ca - cb;
                    if (denom < 1e-5f) denom = 1.f;
                    tf = bb + (uu[t] - cb) / denom * (ba - bb);
                }
                nxt_tf[t] = tf;
                nxt_pk[t] = min(NB - 1, (int)(uu[t] * (float)NB)) | (below << 16);
                if (eset == 0 && jf < Df) sTfine[(r & 1) * kTfineFloats + rs * Df + jf] = tf;
            }
            __syncwarp();
            if (eset == 0 && lane == 0) mbar_arrive(S.bar(BAR_FINE + (r & 1)));
        };

        // ---- final weights + colour composite of group r (state in cur_*).  use_fine: merge coarse + fine; else coarse only.
        auto composite = [&](int r, bool use_fine) {
            const float (&tc)[kMaxT] = cur_tc;
            const float (&sc)[kMaxT] = cur_sc;
            const long long gr = cur_gr;
            const bool ok = cur_ok;
            const int cnt = use_fine ? Dt : Dc;
            float coef_c[kMaxT], coef_f[kMaxT];
            float wsum, dacc;
            float d_first, d_last;
            if (use_fine) {
                // stable sort-merge of coarse (sorted) + fine depths by rank (torch.sort of the concatenation, renderer.py:164-182)
#pragma unroll
                for (int t = 0; t < kMaxT; ++t) {
                    const int k = t * L + j;
                    if (k < Dc) s_tc[k] = tc[t];
                    if (k < Df) s_tf[k] = cur_tf[t];
                    if (k <= Dc) s_hist[k] = 0;
                }
                if (j == 0 && L * kMaxT <= Dc) s_hist[Dc] = 0;
                __syncwarp();
                // zero the u-bucket tables (they alias the sorted arrays, which are written after the ranks are known)
                for (int i = j; i < 2 * NB; i += L) s_ub[i] = 0;
                __syncwarp();
                // Rank of a fine sample among the fine ones.  Fine depths are the inverse CDF of iid uniforms u, a monotone map, so the
                // order of the depths is the order of the u's: bucket the samples by u (NB uniform buckets, ~0.4 samples each), take
                // the bucket prefix count and order the few members of a bucket by (depth, index).  The number of coarse samples <= v
                // follows from the CDF bin the sample was drawn from (its depth lies between the midpoints around that bin).
                int pos_f[kMaxT], pos_c[kMaxT], cntc[kMaxT];
                bool overflow = false;
#pragma unroll
                for (int t = 0; t < kMaxT; ++t) {
                    const int jf = t * L + j;
                    cntc[t] = 0;
                    if (jf < Df) {
                        const float v = cur_tf[t];
                        const int key = cur_pk[t] & 0xffff, below = cur_pk[t] >> 16;
                        const int slot = atomicAdd(&s_ub[key], 1);
                        if (slot < 4) atomicOr(&s_ub[NB + key], jf << (8 * slot));
                        int c = below + 1 + (s_tc[below + 1] <= v ? 1 : 0);
                        if (c == below + 2 && c < Dc && s_tc[c] <= v) ++c;
                        if (!(s_tc[c - 1] <= v && (c == Dc || s_tc[c] > v))) {       // never taken unless the bracket argument fails: search
                            int lo = 0, hi = Dc;
                            while (lo < hi) { const int mid = (lo + hi) >> 1; if (s_tc[mid] <= v) lo = mid + 1; else hi = mid; }
                            c = lo;
                        }
                        cntc[t] = c;
                        atomicAdd(&s_hist[c], 1);
                    }
                }
                __syncwarp();
                {   // exclusive prefix over the buckets: lane j owns buckets 8j .. 8j+7; count and prefix share a word
                    int cn[8], run = 0;
#pragma unroll
                    for (int i = 0; i < 8; ++i) { cn[i] = s_ub[8 * j + i]; run += cn[i]; }
                    int inc = run;
#pragma unroll
                    for (int o = 1; o < L; o <<= 1) { const int up = __shfl_up_sync(FULL, inc, o); if (j >= o) inc += up; }
                    int pre = inc - run;
#pragma unroll
                    for (int i = 0; i < 8; ++i) { s_ub[8 * j + i] = cn[i] | (pre << 8); pre += cn[i]; }
                }
                __syncwarp();
#pragma unroll
                for (int t = 0; t < kMaxT; ++t) {
                    const int jf = t * L + j;
                    pos_f[t] = 0;
                    if (jf < Df) {
                        const float v = cur_tf[t];
                        const int key = cur_pk[t] & 0xffff;
                        const int word = s_ub[key], cn = word & 255;
                        const int mem = s_ub[NB + key];
                        int within = 0;
                        if (cn > 4) overflow = true;
                        else {
#pragma unroll
                            for (int m = 0; m < 4; ++m) {
                                const int idx = (mem >> (8 * m)) & 255;
                                if (m < cn && idx != jf) { const float x = s_tf[idx]; within += (x < v || (x == v && idx < jf)) ? 1 : 0; }
                            }
                        }
                        pos_f[t] = cntc[t] + (word >> 8) + within;
                    }
                }
                if (__any_sync(FULL, overflow)) {                    // a crowded bucket (degenerate u's): full O(Df^2) rank count
#pragma unroll
                    for (int t = 0; t < kMaxT; ++t) {
                        const int jf = t * L + j;
                        if (jf < Df) {
                            const float v = cur_tf[t];
                            int cntf = 0;
                            for (int i = 0; i < Df; ++i) { const float x = s_tf[i]; cntf += (x < v || (x == v && i < jf)) ? 1 : 0; }
                            pos_f[t] = cntc[t] + cntf;
                        }
                    }
                }
                __syncwarp();
                // coarse sample a lands after every fine sample with fewer than a+1 coarse samples <= it: a + #{fine: cnt_c <= a}
                float hc[kMaxT];
#pragma unroll
                for (int t = 0; t < kMaxT; ++t) { const int k = t * L + j; hc[t] = k < Dc ? (float)s_hist[k] : 0.f; }
                seg_scan<L, kMaxT, false>(hc, lane);
#pragma unroll
                for (int t = 0; t < kMaxT; ++t) {
                    const int k = t * L + j;
                    pos_c[t] = k + (int)hc[t];
                    if (k < Dc) { s_sd[pos_c[t]] = tc[t]; s_sg[pos_c[t]] = sc[t]; }
                    if (k < Df) { s_sd[pos_f[t]] = cur_tf[t]; s_sg[pos_f[t]] = cur_sf[t]; }
                }
                __syncwarp();
                float d6[2 * kMaxT], s6[2 * kMaxT], w6[2 * kMaxT], tm6[2 * kMaxT];
#pragma unroll
                for (int t = 0; t < 2 * kMaxT; ++t) {
                    const int p = t * L + j;
                    d6[t] = p < cnt ? s_sd[p] : 0.f;
                    s6[t] = p < cnt ? s_sg[p] : 0.f;
                }
                march_weights<L, 2 * kMaxT>(d6, s6, cnt, lane, w6, tm6);
                float ws = 0.f, da = 0.f;
                if (j == 0) s_wb[0] = 0.f;
#pragma unroll
                for (int t = 0; t < 2 * kMaxT; ++t) {
                    const int p = t * L + j;
                    if (p < cnt) s_wb[p + 1] = w6[t];
                    ws += w6[t];
                    da += w6[t] * tm6[t];
                }
                wsum = seg_sum<L>(ws);
                dacc = seg_sum<L>(da);
                d_first = __shfl_sync(FULL, d6[0], lane & ~(L - 1));
                __syncwarp();
                d_last = s_sd[cnt - 1];
#pragma unroll
                for (int t = 0; t < kMaxT; ++t) {
                    const int k = t * L + j;
                    coef_c[t] = k < Dc ? 0.5f * (s_wb[pos_c[t]] + s_wb[pos_c[t] + 1]) : 0.f;
                    coef_f[t] = k < Df ? 0.5f * (s_wb[pos_f[t]] + s_wb[pos_f[t] + 1]) : 0.f;
                }
            } else {
                float w3[kMaxT], tm3[kMaxT];
                march_weights<L, kMaxT>(tc, sc, cnt, lane, w3, tm3);
                float ws = 0.f, da = 0.f;
#pragma unroll
                for (int t = 0; t < kMaxT; ++t) { ws += w3[t]; da += w3[t] * tm3[t]; }
                wsum = seg_sum<L>(ws);
                dacc = seg_sum<L>(da);
#pragma unroll
                for (int t = 0; t < kMaxT; ++t) {
                    const float wp = seg_prev<L>(w3[t], t > 0 ? w3[t - 1] : 0.f, lane);
                    const int k = t * L + j;
                    coef_c[t] = k < Dc ? 0.5f * ((k > 0 ? wp : 0.f) + w3[t]) : 0.f;
                    coef_f[t] = 0.f;
                }
                d_first = __shfl_sync(FULL, tc[0], lane & ~(L - 1));
                if (j == 0) s_wb[0] = 0.f;                          // keep the scratch race-free across phases
#pragma unroll
                for (int t = 0; t < kMaxT; ++t) { const int k = t * L + j; if (k < Dc) s_sd[k] = tc[t]; }
                __syncwarp();
                d_last = s_sd[Dc - 1];
            }
            // colours: acc[c] += coef * sigmoid(logit + b1) over this thread's rows, channels 16*eset .. +15 (sigmoid * 1.002 - 0.001,
            // triplane_next3d.py:369-370, is affine: applied once to the sum)
            float acc[16];
#pragma unroll
            for (int c = 0; c < 16; ++c) acc[c] = 0.f;
            const float4* bc4 = reinterpret_cast<const float4*>(sB1c + 16 * eset);
            auto add_tile = [&](int slot, float coef) {
                uint32_t v[16];
                tmem_ld16_nowait(tlane + kColSlot + 32u * slot + 16u * eset, v);
                tmem_wait_ld();
                reg_fence16(v);
                float z[16];
#pragma unroll
                for (int c4 = 0; c4 < 4; ++c4) {
                    const float4 bb = bc4[c4];
                    z[c4 * 4] = __uint_as_float(v[c4 * 4]) + bb.x; z[c4 * 4 + 1] = __uint_as_float(v[c4 * 4 + 1]) + bb.y;
                    z[c4 * 4 + 2] = __uint_as_float(v[c4 * 4 + 2]) + bb.z; z[c4 * 4 + 3] = __uint_as_float(v[c4 * 4 + 3]) + bb.w;
                }
#pragma unroll
                for (int c = 0; c < 16; ++c) z[c] = ex2_approx(z[c]);
#pragma unroll
                for (int c = 0; c < 16; ++c) z[c] = rcp_approx(1.f + z[c]);
#pragma unroll
                for (int c = 0; c < 16; ++c) acc[c] = fmaf(coef, z[c], acc[c]);
            };
#pragma unroll
            for (int t = 0; t < kMaxT; ++t)
                if (t < Tc) add_tile((r & 1) * 3 + t, coef_c[t]);
            if (use_fine) {
#pragma unroll
                for (int t = 0; t < kMaxT; ++t)
                    if (t < Tf) add_tile(6 + t, coef_f[t]);
            }
            // the colour slots (and the fine slots) of this group may be overwritten from here on
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                mbar_arrive(S.bar(BAR_CFREE + (r & 1)));
                if (use_fine) mbar_arrive(S.bar(BAR_FFREE));
            }
            // segment reduce-scatter: lane j ends with channel (j & 15) summed over the L lanes
            if (L == 32) {
#pragma unroll
                for (int c = 0; c < 16; ++c) acc[c] += __shfl_xor_sync(FULL, acc[c], 16);
            }
#pragma unroll
            for (int h = 8; h >= 1; h >>= 1) {
                const bool up = (j & h) != 0;
#pragma unroll
                for (int c = 0; c < h; ++c) {
                    const float send = up ? acc[c] : acc[c + h];
                    const float keep = up ? acc[c + h] : acc[c];
                    acc[c] = keep + __shfl_xor_sync(FULL, send, h);
                }
            }
            if (ok && j < 16) {
                float v = fmaf(acc[0], 1.002f, -0.001f * wsum);     // sum_k coef_k (1.002 sigmoid_k - 0.001), sum_k coef_k = wsum
                if (P.white_back) v = v + 1.f - wsum;
                P.rgb[gr * kFeat + 16 * eset + j] = v * 2.f - 1.f;
            }
            if (ok && eset == 0 && j == 0) {
                float depth = dacc / wsum;
                if (isnan(depth)) depth = INFINITY;                  // nan_to_num(nan=inf); the clamp kernel finishes the job
                P.depth[gr] = depth;
                P.wsum[gr] = wsum;
                dmin = fminf(dmin, d_first);
                dmax = fmaxf(dmax, d_last);
            }
        };

        // ---- sigma of tile (kind, r, t) arrived: store it; the last tile of a pass triggers the per-ray phases
        int pend_kind = -1, pend_r = 0, pend_t = 0, pend_i = 0;      // kind: 0 coarse, 1 fine
        auto epi2 = [&]() {
            const float sg = read_sigma(pend_i);
            bool do_composite = false, shift = false;
            if (pend_kind == 0) {
#pragma unroll
                for (int t = 0; t < kMaxT; ++t) if (t == pend_t) nxt_sc[t] = sg;
                if (pend_t == Tc - 1) {
                    // depths + ray of the coarse group
                    const RayId id = ray_of(K, g_begin + pend_r, rs);
                    nxt_ok = id.ok; nxt_gr = id.gr;
#pragma unroll
                    for (int t = 0; t < kMaxT; ++t) { const int k = t * L + j; nxt_tc[t] = (id.ok && k < Dc) ? coarse_depth(K, seed, id.gr, k) : 0.f; }
                    if (Tf > 0) {
                        importance(pend_r);
                        shift = pend_r == 0;                        // the first group moves to its fine phase right away
                    } else {
                        shift = true;                               // coarse-only rendering: composite straight from the coarse pass
                        do_composite = true;
                    }
                }
            } else {
#pragma unroll
                for (int t = 0; t < kMaxT; ++t) if (t == pend_t) cur_sf[t] = sg;
                do_composite = pend_t == Tf - 1;
            }
            if (shift) {
#pragma unroll
                for (int t = 0; t < kMaxT; ++t) { cur_tc[t] = nxt_tc[t]; cur_sc[t] = nxt_sc[t]; cur_tf[t] = nxt_tf[t]; cur_pk[t] = nxt_pk[t]; }
                cur_gr = nxt_gr; cur_ok = nxt_ok;
            }
            if (do_composite) {
                composite(pend_r, pend_kind == 1);
                if (pend_kind == 1) {                               // the next group (already importance-sampled) enters its fine phase
#pragma unroll
                    for (int t = 0; t < kMaxT; ++t) { cur_tc[t] = nxt_tc[t]; cur_sc[t] = nxt_sc[t]; cur_tf[t] = nxt_tf[t]; cur_pk[t] = nxt_pk[t]; }
                    cur_gr = nxt_gr; cur_ok = nxt_ok;
                }
            }
        };

        TileIter it(n_groups, Tc, Tf);
        for (int i = 0;; ++i) {
            const bool has = it.next();
            // a fine tile directly behind the coarse tiles of its own group (single-group CTA): its depths come out of the pending
            // coarse epilogue, which therefore cannot be deferred behind this tile's layer-1 epilogue
            const bool early = has && it.kind == 1 && pend_kind == 0 && pend_r == it.group();
            if (has && !early) epi1(i);
            if (pend_kind >= 0) epi2();
            if (has && early) epi1(i);
            if (!has) break;
            pend_kind = it.kind; pend_r = it.group(); pend_t = it.t; pend_i = i;
        }

        // batch-global depth range (ray_marcher.py:54): one atomic pair per warp of set 0
        if (eset == 0 && P.depth_minmax) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                dmin = fminf(dmin, __shfl_xor_sync(FULL, dmin, o));
                dmax = fmaxf(dmax, __shfl_xor_sync(FULL, dmax, o));
            }
            if (lane == 0) {       // depths are positive (ray_start > 0): IEEE ordering == signed-int ordering
                if (dmin < INFINITY) atomicMin(reinterpret_cast<int*>(P.depth_minmax), __float_as_int(dmin));
                if (dmax > -INFINITY) atomicMax(reinterpret_cast<int*>(P.depth_minmax) + 1, __float_as_int(dmax));
            }
        }
    }

    // ---- teardown
    tc_fence_before();
    __syncthreads();
    if (warp == kWarps - 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u) : "memory");
    }
}

// ---------------------------------------------------------------------------------------------------------------- run_model
// Decoder on arbitrary points (renderer.run_model, renderer.py:149-155; TriPlaneGenerator.sample, triplane_next3d.py:232-276) with the
// same gather / tcgen05 / epilogue roles as the renderer, minus the per-ray phases.  Tile = 128 consecutive points.  In grid mode
// (coords == nullptr) the points are the voxel centres of create_samples (gen_samples_next3d.py:80-102), generated in the kernel
// with the script's own float32 operations, and the flip + border trim of gen_samples_next3d.py:226-238 is applied on the way
// out: voxels in the trimmed border get pad_value and are never decoded.
struct PointsK {
    const float* planes;
    int N, PH, PW;
    const float* coords;         // [N, Pn, 3] or nullptr (grid mode, N = 1)
    long long Pn, total;         // points per image, N * Pn
    float scale;
    const float* w0; const float* b0; const float* w1; const float* b1;
    float* sigma;                // [N, Pn]  (grid mode: [R, R, R] already flipped + trimmed)
    float* rgb;                  // [N, Pn, 32] or nullptr
    int grid_n, pad;             // grid mode: voxels per side, trimmed border width
    float voxel_size, org0, org1, org2, pad_value;
    long long head;              // grid mode: flat index of the first point
};

// voxel centre of flat index idx, bit-identical to the reference's float32 expression chain (float, not floor, division)
__device__ __forceinline__ void grid_point(const PointsK& K, long long idx, float& x, float& y, float& z) {
    const float fn = (float)K.grid_n;
    const float fi = (float)idx;                                   // int64 -> float32, round to nearest (indices above 2^24 lose bits)
    const float s2 = (float)(idx % K.grid_n);
    const float q1 = __fdiv_rn(fi, fn);
    const float s1 = fmodf(q1, fn);
    const float s0 = fmodf(__fdiv_rn(q1, fn), fn);
    x = __fadd_rn(__fmul_rn(s0, K.voxel_size), K.org2);
    y = __fadd_rn(__fmul_rn(s1, K.voxel_size), K.org1);
    z = __fadd_rn(__fmul_rn(s2, K.voxel_size), K.org0);
}
// destination of flat index idx after flip(dims=[0]) and whether it lies in the trimmed border
__device__ __forceinline__ long long grid_dest(const PointsK& K, long long idx, bool& border) {
    const long long n = K.grid_n;
    const long long a = idx / (n * n), rem = idx - a * n * n;
    const long long b = rem / n, c = rem - b * n;
    const long long fa = n - 1 - a;
    border = fa < K.pad || fa >= n - K.pad || b < K.pad || b >= n - K.pad || c < K.pad || c >= n - K.pad;
    return (fa * n + b) * n + c;
}

template <bool RGB>
__global__ void __launch_bounds__(kThreads, 1) points_fused_kernel(const __grid_constant__ PointsK K) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    Smem S;
    S.base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* const sb = S.base;
    uint32_t* const sTmem = reinterpret_cast<uint32_t*>(sb + kOffBar + kNumBars * 8);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const bool grid = K.coords == nullptr;

    const long long n_tiles_all = (K.total + 127) / 128;
    // tiles are dealt round-robin: the skipped border tiles of a trimmed grid are spread evenly over the CTAs
    const long long t_begin = blockIdx.x, t_end = n_tiles_all, t_step = gridDim.x;
    // a tile of the voxel grid is skipped when every one of its points falls into the trimmed border
    auto tile_skipped = [&](long long tile) -> bool {
        if (!grid || K.pad <= 0) return false;
        const long long first = K.head + tile * 128, last = min(K.head + K.total, first + 128) - 1;
        const long long n = K.grid_n, r0 = first / n, r1 = last / n;           // rows (a, b) touched: at most r0 .. r1
        for (long long r = r0; r <= r1; ++r) {
            const long long a = r / n, b = r - a * n, fa = n - 1 - a;
            if (!(fa < K.pad || fa >= n - K.pad || b < K.pad || b >= n - K.pad)) return false;
        }
        return true;
    };

    if (tid == 0) {
        init_pipeline_barriers(S);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == kWarps - 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(sTmem)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    stage_decoder(sb, K.w0, K.b0, K.w1, K.b1, tid);
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *sTmem;

    if (warp == kWarps - 1) {                                      // ---- MMA issuer
        if (lane == 0) {
            int i = 0;
            for (long long tile = t_begin; tile < t_end; tile += t_step) {
                if (tile_skipped(tile)) continue;
                mma_layer1(S, tmem, i);
                if (i > 0) {
                    mbar_wait_sleep(S.bar(BAR_HFULL + ((i - 1) & 1)), (uint32_t)(((i - 1) >> 1) & 1));
                    tc_fence_after();
                    mma_layer2_issue(S, tmem, (i - 1) & 1, kColSlot + 32u * ((i - 1) & 1), RGB);
                }
                ++i;
            }
            if (i > 0) {
                mbar_wait_sleep(S.bar(BAR_HFULL + ((i - 1) & 1)), (uint32_t)(((i - 1) >> 1) & 1));
                tc_fence_after();
                mma_layer2_issue(S, tmem, (i - 1) & 1, kColSlot + 32u * ((i - 1) & 1), RGB);
            }
        }
    } else if (warp >= kEWarps) {                                  // ---- gather warps
        const int gw = warp - kEWarps;
        uint2* const taps = reinterpret_cast<uint2*>(sb + kOffTaps + gw * kTapBytesPerWarp);
        int next_item = gw, i = 0;
        for (long long tile = t_begin; tile < t_end; tile += t_step) {
            if (tile_skipped(tile)) continue;
            while (next_item < i * 4 + 4) {
                const int q = next_item - i * 4;
                const long long g = tile * 128 + q * 32 + lane;
                bool valid = g < K.total;
                float px = 0.f, py = 0.f, pz = 0.f;
                uint32_t img = 0;
                if (valid) {
                    if (grid) {
                        bool border;
                        grid_dest(K, K.head + g, border);
                        valid = !border;
                        grid_point(K, K.head + g, px, py, pz);
                    } else {
                        const float* c = K.coords + g * 3;
                        px = __ldg(c); py = __ldg(c + 1); pz = __ldg(c + 2);
                        img = (uint32_t)(g / K.Pn) * (uint32_t)(3 * K.PH * K.PW * 128);
                    }
                }
                setup_taps(taps, lane, px, py, pz, valid, img, K.PH, K.PW, K.scale);
                __syncwarp();
                const int b = i % kNF;
                if (i >= kNF) mbar_wait_sleep(S.bar(BAR_FEMPTY + b), (uint32_t)((i / kNF - 1) & 1), 40u);
                gather_rows(K.planes, taps, sb + kOffF + b * 16384, sb + kOffF + b * 16384 + 8192, q * 32, lane);
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(S.bar(BAR_FFULL + b));
                next_item += kGWarps;
            }
            ++i;
        }
    } else {                                                       // ---- epilogue warps
        const int eset = warp >> 2, q = warp & 3;
        const uint32_t tlane = tmem + ((uint32_t)(q * 32) << 16);
        const float* const sB1c = reinterpret_cast<const float*>(sb + kOffBias) + 64;
        long long pend_tile = -1;
        int pend_i = 0;
        auto epi2 = [&]() {
            const float sg = read_sigma_tile(S, tlane, pend_i);
            const long long g = pend_tile * 128 + q * 32 + lane;
            if (RGB) {
                uint32_t v[16];
                tmem_ld16_nowait(tlane + kColSlot + 32u * (pend_i & 1) + 16u * eset, v);
                tmem_wait_ld();
                reg_fence16(v);
                if (g < K.total) {
                    const float4* bc4 = reinterpret_cast<const float4*>(sB1c + 16 * eset);
                    float4* dst = reinterpret_cast<float4*>(K.rgb + g * kFeat + 16 * eset);
#pragma unroll
                    for (int c4 = 0; c4 < 4; ++c4) {
                        const float4 bb = bc4[c4];
                        float4 o;                                   // sigmoid(x) * 1.002 - 0.001 (triplane_next3d.py:369-370)
                        o.x = fmaf(rcp_approx(1.f + ex2_approx(__uint_as_float(v[c4 * 4]) + bb.x)), 1.002f, -0.001f);
                        o.y = fmaf(rcp_approx(1.f + ex2_approx(__uint_as_float(v[c4 * 4 + 1]) + bb.y)), 1.002f, -0.001f);
                        o.z = fmaf(rcp_approx(1.f + ex2_approx(__uint_as_float(v[c4 * 4 + 2]) + bb.z)), 1.002f, -0.001f);
                        o.w = fmaf(rcp_approx(1.f + ex2_approx(__uint_as_float(v[c4 * 4 + 3]) + bb.w)), 1.002f, -0.001f);
                        dst[c4] = o;
                    }
                }
            }
            if (eset == 0 && g < K.total) {
                if (grid) {
                    bool border;
                    const long long d = grid_dest(K, K.head + g, border);
                    K.sigma[d] = border ? K.pad_value : sg;
                } else {
                    K.sigma[g] = sg;
                }
            }
        };
        int i = 0;
        for (long long tile = t_begin; tile < t_end; tile += t_step) {
            if (tile_skipped(tile)) {                              // whole tile in the trimmed border: only the pad value is written
                const long long g = tile * 128 + q * 32 + lane;
                if (eset == 0 && g < K.total) { bool border; K.sigma[grid_dest(K, K.head + g, border)] = K.pad_value; }
                continue;
            }
            epi1_tile(S, tlane, eset, lane, i);
            if (pend_tile >= 0) epi2();
            pend_tile = tile; pend_i = i;
            ++i;
        }
        if (pend_tile >= 0) epi2();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == kWarps - 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u) : "memory");
    }
}

}  // namespace

// ---------------------------------------------------------------------------------------------------------------- ceilings
// Two micro-kernels that isolate the hard per-SM limits of the renderer's formulation on the SAME workload (same rays, same sample
// positions, same tap arithmetic), used by bench.py / DESIGN.md to say how far render_fused_kernel is from what the hardware
// allows for a per-sample gather + MLP -- as opposed to the "every texel read once" HBM figure of the survey's formula:
//   kind 0  gather only : all 16 warps of a CTA run the gather role (ray -> depth -> 12 taps -> 256-bit loads -> weighted sum ->
//           bf16 split -> shared-memory tile).  No MMA, no epilogue.  Ceiling of the tri-plane fetch (L1 wavefronts + L2 misses).
//   kind 1  activations only : 192 MUFU operations per sample (64 x (ex2 + lg2), 32 x (ex2 + rcp)) on register operands with the
//           epilogue's surrounding arithmetic.  Ceiling of the SFU pipe.
namespace {
__global__ void __launch_bounds__(kThreads, 1) gather_floor_kernel(const __grid_constant__ FusedK K, float* __restrict__ sink) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* const sb = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    const N3DRender& P = K.p;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int L = P.depth_coarse <= 48 ? 16 : 32;
    uint2* const taps = reinterpret_cast<uint2*>(sb + 32768 + warp * kTapBytesPerWarp);
    uint8_t* const f_hi = sb, * const f_lo = sb + 8192;          // one shared tile: the stores are part of the cost, the data is not used
    const int g_begin = (int)((K.total_groups * blockIdx.x) / gridDim.x);
    const int n_groups = (int)((K.total_groups * (blockIdx.x + 1)) / gridDim.x) - g_begin;
    const int passes = P.depth_fine > 0 ? 2 : 1;
    const int T = K.Tc;
    // item = (group, pass, tile, quarter): the same 32-row work unit the gather warps of the renderer process
    const int items = n_groups * passes * T * 4;
    for (int it = warp; it < items; it += kWarps) {
        const int q = it & 3, t = (it >> 2) % T, pass = (it / (4 * T)) % passes, r = it / (4 * T * passes);
        const int row = q * 32 + lane, rs = row / L, j = row & (L - 1);
        const Ray ray = make_ray(K, g_begin + r, rs);
        const int k = t * L + j;
        const bool valid = ray.ok && k < P.depth_coarse;
        // second pass: the fine samples sit near the coarse ones (shifted by half a step) -- same count, same locality
        const float depth = valid ? coarse_depth(K, P.seed + pass, ray.gr, k) + (pass ? 0.5f * K.delta_coarse : 0.f) : 0.f;
        setup_taps(taps, lane, ray.ox + depth * ray.dx, ray.oy + depth * ray.dy, ray.oz + depth * ray.dz, valid && !(K.mode & 1), ray.img4, P.PH, P.PW,
                   K.scale);
        __syncwarp();
        gather_rows(P.planes, taps, f_hi, f_lo, q * 32, lane);
        __syncwarp();
    }
    if (sink && threadIdx.x == 0 && blockIdx.x == 0) sink[0] = (float)f_hi[0];
}

__global__ void __launch_bounds__(kThreads, 1) mufu_floor_kernel(long long samples, float* __restrict__ sink) {
    // every thread evaluates whole samples: 64 hidden activations (softplus as in epi1) and 32 colour sigmoids
    const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x, nthreads = (long long)gridDim.x * blockDim.x;
    float acc = 0.f;
    for (long long s = tid; s < samples; s += nthreads) {
        float y[32];
#pragma unroll 1
        for (int half = 0; half < 2; ++half) {
#pragma unroll
            for (int c = 0; c < 32; ++c) y[c] = (float)(s & 1023) * 1e-3f + (float)(c + 32 * half) * 0.01f - 0.3f;
            float e[32];
#pragma unroll
            for (int c = 0; c < 32; ++c) e[c] = ex2_approx(fminf(y[c], 126.f));
#pragma unroll
            for (int c = 0; c < 32; ++c) e[c] = lg2_approx(1.f + e[c]);
#pragma unroll
            for (int c = 0; c < 32; ++c) acc += fmaxf(e[c], y[c]);
        }
#pragma unroll
        for (int c = 0; c < 32; ++c) y[c] = (float)(s & 511) * 2e-3f - (float)c * 0.02f;
#pragma unroll
        for (int c = 0; c < 32; ++c) y[c] = ex2_approx(y[c]);
#pragma unroll
        for (int c = 0; c < 32; ++c) y[c] = rcp_approx(1.f + y[c]);
#pragma unroll
        for (int c = 0; c < 32; ++c) acc = fmaf(0.5f, y[c], acc);
    }
    if (sink && acc == 123.456f) sink[0] = acc;
}
}  // namespace

int n3d_render_floor_launch(const N3DRender* p, int kind, float* sink, void* stream) {
    N3DDeviceState* D = n3d_device_state();
    if (!D) return N3D_ERR_CUDA;
    const int dmaxv = p->depth_coarse > p->depth_fine ? p->depth_coarse : p->depth_fine;
    const int L = dmaxv <= 48 ? 16 : 32;
    FusedK K;
    K.p = *p;
    K.M = p->res * p->res;
    K.delta_coarse = (float)(((double)p->ray_end - (double)p->ray_start) / (double)(p->depth_coarse - 1));
    K.scale = 2.f / p->box_warp;
    K.Tc = (p->depth_coarse + L - 1) / L;
    K.Tf = (p->depth_fine + L - 1) / L;
    K.gw = L == 16 ? 4 : 2;
    K.log2gw = L == 16 ? 2 : 1;
    const int tiles_x = (p->res + K.gw - 1) / K.gw, tiles_y = (p->res + 1) / 2;
    K.blocks_x = (tiles_x + 3) / 4;
    K.gpi = K.blocks_x * ((tiles_y + 7) / 8) * 32;
    K.total_groups = (long long)p->N * K.gpi;
    K.mode = 0;
    const int grid = (int)(K.total_groups < D->num_sms ? K.total_groups : D->num_sms);
    if (kind == 0) {
        const size_t smem = 32768 + kWarps * kTapBytesPerWarp + 1024;
        if (int e = n3d_smem_optin(D, N3D_CFG_FLOOR_GATHER, (const void*)gather_floor_kernel, (int)smem, "n3d_render_floor")) return e;
        gather_floor_kernel<<<grid, kThreads, smem, (cudaStream_t)stream>>>(K, sink);
    } else {
        const long long samples = (long long)p->N * K.M * (p->depth_coarse + p->depth_fine);
        mufu_floor_kernel<<<D->num_sms, kThreads, 0, (cudaStream_t)stream>>>(samples, sink);
    }
    N3D_CHECK_LAUNCH("n3d_render_floor");
    return N3D_OK;
}

int n3d_render_fused_launch(const N3DRender* p, void* stream, int mode) {
    const int dmaxv = p->depth_coarse > p->depth_fine ? p->depth_coarse : p->depth_fine;
    const int L = dmaxv <= 48 ? 16 : 32;
    FusedK K;
    K.p = *p;
    K.M = p->res * p->res;
    K.delta_coarse = (float)(((double)p->ray_end - (double)p->ray_start) / (double)(p->depth_coarse - 1));
    K.scale = 2.f / p->box_warp;
    K.Tc = (p->depth_coarse + L - 1) / L;
    K.Tf = (p->depth_fine + L - 1) / L;
    K.gw = L == 16 ? 4 : 2;
    K.log2gw = L == 16 ? 2 : 1;
    const int tiles_x = (p->res + K.gw - 1) / K.gw, tiles_y = (p->res + 1) / 2;
    K.blocks_x = (tiles_x + 3) / 4;
    const int blocks_y = (tiles_y + 7) / 8;
    K.gpi = K.blocks_x * blocks_y * 32;
    K.total_groups = (long long)p->N * K.gpi;
    K.mode = mode;
    N3DDeviceState* D = n3d_device_state();
    if (!D) return N3D_ERR_CUDA;
    const size_t smem = (size_t)kSmemBytes + 1024;
    if (int e = L == 16 ? n3d_smem_optin(D, N3D_CFG_RENDER16, (const void*)render_fused_kernel<16>, (int)smem, "n3d_render_rays")
                        : n3d_smem_optin(D, N3D_CFG_RENDER32, (const void*)render_fused_kernel<32>, (int)smem, "n3d_render_rays"))
        return e;
    const int grid = (int)(K.total_groups < D->num_sms ? K.total_groups : D->num_sms);
    if (L == 16) render_fused_kernel<16><<<grid, kThreads, smem, (cudaStream_t)stream>>>(K);
    else render_fused_kernel<32><<<grid, kThreads, smem, (cudaStream_t)stream>>>(K);
    N3D_CHECK_LAUNCH("n3d_render_rays");
    return N3D_OK;
}

// coords != nullptr: arbitrary points [N, Pn, 3].  coords == nullptr: voxel grid of `grid_n`^3 points (image 0), flat indices
// head .. head + Pn - 1, sigma written flipped + trimmed into the [grid_n]^3 output.
int n3d_points_fused_launch(const float* planes, int N, int PH, int PW, const float* coords, long long Pn, float box_warp, const float* w0,
                            const float* b0, const float* w1, const float* b1, float* sigma, float* rgb, int grid_n, float cube_length, long long head,
                            int pad, float pad_value, void* stream) {
    PointsK K;
    K.planes = planes; K.N = N; K.PH = PH; K.PW = PW; K.coords = coords; K.Pn = Pn; K.total = (long long)N * Pn;
    K.scale = 2.f / box_warp;
    K.w0 = w0; K.b0 = b0; K.w1 = w1; K.b1 = b1; K.sigma = sigma; K.rgb = rgb;
    K.grid_n = grid_n; K.pad = pad; K.pad_value = pad_value; K.head = head;
    K.voxel_size = 0.f; K.org0 = K.org1 = K.org2 = 0.f;
    if (!coords) {       // create_samples: voxel_origin = [0,0,0] - cube_length / 2 (float64), voxel_size = cube_length / (N - 1); both enter
                         // the float32 tensor expression as scalars, i.e. rounded to float32
        K.voxel_size = (float)((double)cube_length / (double)(grid_n - 1));
        K.org0 = K.org1 = K.org2 = (float)(0.0 - (double)cube_length / 2.0);
    }
    N3DDeviceState* D = n3d_device_state();
    if (!D) return N3D_ERR_CUDA;
    const size_t smem = (size_t)kSmemBytes + 1024;
    if (int e = rgb ? n3d_smem_optin(D, N3D_CFG_POINTS_RGB, (const void*)points_fused_kernel<true>, (int)smem, "n3d_sample_points")
                    : n3d_smem_optin(D, N3D_CFG_POINTS, (const void*)points_fused_kernel<false>, (int)smem, "n3d_sample_points"))
        return e;
    const long long tiles = (K.total + 127) / 128;
    const int grid = (int)(tiles < D->num_sms ? tiles : D->num_sms);
    if (rgb) points_fused_kernel<true><<<grid, kThreads, smem, (cudaStream_t)stream>>>(K);
    else points_fused_kernel<false><<<grid, kThreads, smem, (cudaStream_t)stream>>>(K);
    N3D_CHECK_LAUNCH("n3d_sample_points");
    return N3D_OK;
}
