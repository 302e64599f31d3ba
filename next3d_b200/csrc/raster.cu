// Mesh path: view transform, triangle rasterizer (pytorch3d semantics, bit-exact with oracle/oracle_c.c), UV texture
// lookup, mouth flood fill, mouth box, antialiased resize (crop / paste / SR pre-scale) and plane blending.
// These replace pytorch3d.rasterize_meshes, F.grid_sample, cv2.floodFill (host round trip), numpy (host round trip)
// and F.interpolate(antialias=True) on the reference's path (triplane_next3d.py:146-174, 190-230, 330-344).
#include "common.cuh"
#include "../../include/next3d_b200.h"

namespace {
constexpr int kSMs = 148;
inline int grid_for(int64_t work_items, int threads, int per_sm = 8) {
    int64_t g = (work_items + threads - 1) / threads;
    int64_t cap = (int64_t)kSMs * per_sm;
    return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

// ---------------------------------------------------------------------------------------------- transform
// p' = ((p*[1,-1,1]) @ R + [0,-.01,-.01]) * 5 ; y,z negated ; z += zoff ; optional NDC x,y negation.  The 3-term dot products
// are evaluated as the fused chain fma(z, R2j, fma(y, R1j, x * R0j)) -- what torch.bmm's CPU kernel computes for K = 3 -- so the
// view-space vertices, and with them the rasterizer's index buffer, are bit-identical to the oracle's.
__global__ void __launch_bounds__(256) transform_kernel(const float* __restrict__ pts, int N, int P, const float* __restrict__ rot,
                                                        int nviews, float zoff, int ndc_flip, float* __restrict__ out) {
    const int64_t total = (int64_t)N * nviews * P;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int pi = (int)(i % P);
        const int view = (int)((i / P) % nviews);
        const int n = (int)(i / ((int64_t)P * nviews));
        const float* p = pts + ((int64_t)n * P + pi) * 3;
        const float* R = rot + view * 9;
        const float x = p[0], y = -p[1], z = p[2];
        float r[3];
#pragma unroll
        for (int j = 0; j < 3; ++j)
            r[j] = __fmaf_rn(z, R[6 + j], __fmaf_rn(y, R[3 + j], __fmul_rn(x, R[j])));       // k = 0, 1, 2 FMA chain (see oracle.transform_view)
        float ox = __fmul_rn(__fadd_rn(r[0], 0.f), 5.f);
        float oy = -__fmul_rn(__fadd_rn(r[1], -0.01f), 5.f);
        float oz = __fadd_rn(-__fmul_rn(__fadd_rn(r[2], -0.01f), 5.f), zoff);
        if (ndc_flip) { ox = -ox; oy = -oy; }
        float* o = out + i * 3;
        o[0] = ox; o[1] = oy; o[2] = oz;
    }
}

// ---------------------------------------------------------------------------------------------- rasterizer
// One CTA per 16x16-pixel bin of one image, one thread per pixel.  Faces stream through shared memory in chunks of 256:
// every thread sets up one face (culling + bbox exactly as oracle_c.c), faces whose bbox misses the bin are dropped by an
// order-free compaction, and each pixel thread then tests the survivors.  The nearest hit wins; equal depth keeps the
// lower face index (explicit tie-break, so the result does not depend on processing order).  All fp32 arithmetic uses
// round-to-nearest intrinsics in the oracle's expression order (no FMA contraction) -> bit-identical index buffers.
struct FaceSetup {
    float x0, y0, z0, x1, y1, z1, x2, y2, z2, area;
    float xmin, xmax, ymin, ymax;
    int id;
};

__device__ __forceinline__ float edge_fn(float px, float py, float ax, float ay, float bx, float by) {
    return __fsub_rn(__fmul_rn(__fsub_rn(px, ax), __fsub_rn(by, ay)), __fmul_rn(__fsub_rn(py, ay), __fsub_rn(bx, ax)));
}

constexpr int kBin = 16;
constexpr int kChunk = 256;
constexpr int kSetupFloats = 16;     // per (image, face) workspace record: bbox (xmin,xmax,ymin,ymax) | x0 y0 z0 x1 y1 z1 x2 y2 z2 area | pad

// Pass 1: one thread per (image, face): culling + bounding box + barycentric denominator exactly as oracle_c.c, stored once
// instead of being recomputed by every 16x16-pixel bin.  Culled faces get an empty bbox (xmin = +inf).
__global__ void __launch_bounds__(256) raster_setup_kernel(const float* __restrict__ verts, const int* __restrict__ faces, int NM, int V, int F,
                                                           float* __restrict__ ws) {
    const int64_t total = (int64_t)NM * F;
    const float kEps = 1e-8f;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int f = (int)(i % F);
        const int img = (int)(i / F);
        const float* vb = verts + (int64_t)img * V * 3;
        const int i0 = faces[f * 3 + 0], i1 = faces[f * 3 + 1], i2 = faces[f * 3 + 2];
        FaceSetup s;
        s.x0 = vb[i0 * 3]; s.y0 = vb[i0 * 3 + 1]; s.z0 = vb[i0 * 3 + 2];
        s.x1 = vb[i1 * 3]; s.y1 = vb[i1 * 3 + 1]; s.z1 = vb[i1 * 3 + 2];
        s.x2 = vb[i2 * 3]; s.y2 = vb[i2 * 3 + 1]; s.z2 = vb[i2 * 3 + 2];
        s.xmin = fminf(s.x0, fminf(s.x1, s.x2)); s.xmax = fmaxf(s.x0, fmaxf(s.x1, s.x2));
        s.ymin = fminf(s.y0, fminf(s.y1, s.y2)); s.ymax = fmaxf(s.y0, fmaxf(s.y1, s.y2));
        const float zmax = fmaxf(s.z0, fmaxf(s.z1, s.z2));
        const float face_area = edge_fn(s.x0, s.y0, s.x1, s.y1, s.x2, s.y2);
        bool keep = !(zmax < 0.f);
        keep = keep && !(face_area <= kEps && face_area >= -kEps);
        keep = keep && !(face_area < 0.f);
        s.area = __fadd_rn(edge_fn(s.x2, s.y2, s.x0, s.y0, s.x1, s.y1), kEps);
        float4* o = reinterpret_cast<float4*>(ws + i * kSetupFloats);
        o[0] = keep ? make_float4(s.xmin, s.xmax, s.ymin, s.ymax) : make_float4(INFINITY, -INFINITY, INFINITY, -INFINITY);
        o[1] = make_float4(s.x0, s.y0, s.z0, s.x1);
        o[2] = make_float4(s.y1, s.z1, s.x2, s.y2);
        o[3] = make_float4(s.z2, s.area, 0.f, 0.f);
    }
}

// Pass 2: one CTA per 16x16-pixel bin of one image, one thread per pixel.  Face records stream through in chunks of 256: each
// thread tests one face's bbox against the bin (one coalesced float4), survivors are compacted into shared memory (order-free),
// then every pixel thread tests the survivors.  The nearest hit wins; equal depth keeps the lower face index (explicit
// tie-break, so the result does not depend on processing order).  All fp32 arithmetic uses round-to-nearest intrinsics in the
// oracle's expression order (no FMA contraction) -> bit-identical index buffers and barycentrics.
__global__ void __launch_bounds__(256) rasterize_kernel(const float* __restrict__ ws, int F, int H, int W, int* __restrict__ pix_to_face,
                                                        float* __restrict__ bary) {
    __shared__ FaceSetup sf[kChunk];
    __shared__ int s_count;
    const int bins_x = (W + kBin - 1) / kBin;
    const int img = blockIdx.y;
    const int bx = blockIdx.x % bins_x, by = blockIdx.x / bins_x;
    const int xi = bx * kBin + (threadIdx.x % kBin), yi = by * kBin + (threadIdx.x / kBin);
    const float* wb = ws + (int64_t)img * F * kSetupFloats;

    const float xf = __fadd_rn(-1.f, __fdiv_rn(__fadd_rn(__fmul_rn(2.f, (float)(W - 1 - xi)), 1.f), (float)W));
    const float yf = __fadd_rn(-1.f, __fdiv_rn(__fadd_rn(__fmul_rn(2.f, (float)(H - 1 - yi)), 1.f), (float)H));
    // NDC extent of this bin's pixel centres (xf decreases with xi)
    const int xi_hi = min(bx * kBin + kBin - 1, W - 1), yi_hi = min(by * kBin + kBin - 1, H - 1);
    const float bin_xmax = __fadd_rn(-1.f, __fdiv_rn(__fadd_rn(__fmul_rn(2.f, (float)(W - 1 - bx * kBin)), 1.f), (float)W));
    const float bin_xmin = __fadd_rn(-1.f, __fdiv_rn(__fadd_rn(__fmul_rn(2.f, (float)(W - 1 - xi_hi)), 1.f), (float)W));
    const float bin_ymax = __fadd_rn(-1.f, __fdiv_rn(__fadd_rn(__fmul_rn(2.f, (float)(H - 1 - by * kBin)), 1.f), (float)H));
    const float bin_ymin = __fadd_rn(-1.f, __fdiv_rn(__fadd_rn(__fmul_rn(2.f, (float)(H - 1 - yi_hi)), 1.f), (float)H));

    int best_f = -1;
    float best_z = 0.f, bw0 = -1.f, bw1 = -1.f, bw2 = -1.f;

    for (int f0 = 0; f0 < F; f0 += kChunk) {
        if (threadIdx.x == 0) s_count = 0;
        __syncthreads();
        const int f = f0 + threadIdx.x;
        if (f < F) {
            const float4* rec = reinterpret_cast<const float4*>(wb + (int64_t)f * kSetupFloats);
            const float4 bb = __ldg(rec);
            if (!(bb.y < bin_xmin || bb.x > bin_xmax || bb.w < bin_ymin || bb.z > bin_ymax)) {     // also false for culled faces
                const float4 r1 = __ldg(rec + 1), r2 = __ldg(rec + 2), r3 = __ldg(rec + 3);
                FaceSetup s;
                s.xmin = bb.x; s.xmax = bb.y; s.ymin = bb.z; s.ymax = bb.w;
                s.x0 = r1.x; s.y0 = r1.y; s.z0 = r1.z; s.x1 = r1.w;
                s.y1 = r2.x; s.z1 = r2.y; s.x2 = r2.z; s.y2 = r2.w;
                s.z2 = r3.x; s.area = r3.y; s.id = f;
                sf[atomicAdd(&s_count, 1)] = s;
            }
        }
        __syncthreads();
        const int cnt = s_count;
        if (xi < W && yi < H) {
            for (int k = 0; k < cnt; ++k) {
                const FaceSetup& s = sf[k];
                if (xf < s.xmin || xf > s.xmax || yf < s.ymin || yf > s.ymax) continue;
                const float w0 = __fdiv_rn(edge_fn(xf, yf, s.x1, s.y1, s.x2, s.y2), s.area);
                const float w1 = __fdiv_rn(edge_fn(xf, yf, s.x2, s.y2, s.x0, s.y0), s.area);
                const float w2 = __fdiv_rn(edge_fn(xf, yf, s.x0, s.y0, s.x1, s.y1), s.area);
                const float pz = __fadd_rn(__fadd_rn(__fmul_rn(w0, s.z0), __fmul_rn(w1, s.z1)), __fmul_rn(w2, s.z2));
                if (pz < 0.f) continue;
                if (!(w0 > 0.f && w1 > 0.f && w2 > 0.f)) continue;
                if (best_f < 0 || pz < best_z || (pz == best_z && s.id < best_f)) {
                    best_f = s.id; best_z = pz; bw0 = w0; bw1 = w1; bw2 = w2;
                }
            }
        }
        __syncthreads();
    }
    if (xi < W && yi < H) {
        const int64_t p = ((int64_t)img * H + yi) * W + xi;
        pix_to_face[p] = best_f;
        bary[p * 3 + 0] = bw0; bary[p * 3 + 1] = bw1; bary[p * 3 + 2] = bw2;
    }
}

// ---------------------------------------------------------------------------------------------- UV lookup
// bilinear grid_sample, zeros padding, align_corners=False (ATen grid_sampler_2d): ix = ((gx + 1) * W - 1) / 2
__device__ __forceinline__ void bilinear_setup(float gx, float gy, int W, int H, int& x0, int& y0, float& fx, float& fy) {
    const float ix = ((gx + 1.f) * (float)W - 1.f) * 0.5f, iy = ((gy + 1.f) * (float)H - 1.f) * 0.5f;
    const float flx = floorf(ix), fly = floorf(iy);
    x0 = (int)flx; y0 = (int)fly; fx = ix - flx; fy = iy - fly;
}

// One warp per output pixel, lanes = channels for the texture loads.  The per-tap arithmetic (face lookup, barycentric UV,
// bilinear corner offset + weight) is done ONCE: lane l < 16 owns texture tap (view l/4, corner l%4), lane 16 + l owns the
// corresponding eye-mask tap; offsets / weights are then broadcast with shuffles and the 16 texture loads (one coalesced
// 128-byte line each) are issued together.
__global__ void __launch_bounds__(256) uv_sample_kernel(const int* __restrict__ p2f, const float* __restrict__ bary, const float* __restrict__ face_uv,
                                                        const float* __restrict__ tex, const float* __restrict__ mask, int N, int H, int W, int TH,
                                                        int TW, int C, int MH, int MW, float* __restrict__ planes, float* __restrict__ alpha) {
    const int lane = threadIdx.x & 31;
    const int64_t warp_global = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t HW = (int64_t)H * W, total = (int64_t)N * HW;
    const int view = (lane >> 2) & 3, corner = lane & 3;
    const bool is_mask = lane >= 16;
    const int GW = is_mask ? MW : TW, GH = is_mask ? MH : TH;
    for (int64_t pi = warp_global; pi < total; pi += nwarps) {
        const int n = (int)(pi / HW);
        const int64_t pix = pi - (int64_t)n * HW;
        const int64_t src = ((int64_t)(n * 4 + view)) * HW + pix;
        const int f = __ldg(p2f + src);
        float u = 0.f, v = 0.f;
        if (f >= 0) {
            const float b0 = __ldg(bary + src * 3), b1 = __ldg(bary + src * 3 + 1), b2 = __ldg(bary + src * 3 + 2);
            const float* fu = face_uv + (int64_t)f * 6;
            u = __fadd_rn(__fadd_rn(__fmul_rn(b0, __ldg(fu)), __fmul_rn(b1, __ldg(fu + 2))), __fmul_rn(b2, __ldg(fu + 4)));
            v = __fadd_rn(__fadd_rn(__fmul_rn(b0, __ldg(fu + 1)), __fmul_rn(b1, __ldg(fu + 3))), __fmul_rn(b2, __ldg(fu + 5)));
        }
        int x0, y0; float fx, fy;
        bilinear_setup(u, v, GW, GH, x0, y0, fx, fy);
        const int xi = x0 + (corner & 1), yi = y0 + (corner >> 1);
        const float wx = (corner & 1) ? fx : 1.f - fx, wy = (corner >> 1) ? fy : 1.f - fy;
        const bool inside = xi >= 0 && xi < GW && yi >= 0 && yi < GH;
        const float my_w = inside ? wx * wy : 0.f;
        const int cy = min(max(yi, 0), GH - 1), cx = min(max(xi, 0), GW - 1);
        const int my_off = is_mask ? cy * GW + cx : (cy * GW + cx) * C;
        // ---- eye mask: lanes 16..31 fetch their tap, reduce the 4 corners of each view, alpha = mask * visible
        float m = is_mask ? my_w * __ldg(mask + my_off) : 0.f;
        m += __shfl_xor_sync(0xffffffffu, m, 1);
        m += __shfl_xor_sync(0xffffffffu, m, 2);
        if (is_mask && corner == 0 && view != 2) {
            const int aplane = view == 0 ? 0 : (view == 1 ? 1 : 2);
            alpha[((int64_t)aplane * N + n) * HW + pix] = m * (f >= 0 ? 1.f : 0.f);
        }
        // ---- texture: 16 taps broadcast from lanes 0..15
        const float* tb = tex + (int64_t)n * TH * TW * C;
        float val[16], wgt[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const int off = __shfl_sync(0xffffffffu, my_off, i);
            wgt[i] = __shfl_sync(0xffffffffu, my_w, i);
            val[i] = lane < C ? __ldg(tb + (unsigned)(off + lane)) : 0.f;
        }
        float acc[4];
#pragma unroll
        for (int vw = 0; vw < 4; ++vw) {
            float a = 0.f;
#pragma unroll
            for (int c = 0; c < 4; ++c) a += wgt[vw * 4 + c] * val[vw * 4 + c];
            acc[vw] = a;
        }
        if (lane < C) {
            planes[(((int64_t)0 * N + n) * HW + pix) * C + lane] = acc[0];
            planes[(((int64_t)1 * N + n) * HW + pix) * C + lane] = acc[1] + acc[2];
            planes[(((int64_t)2 * N + n) * HW + pix) * C + lane] = acc[3];
        }
    }
}

// ---------------------------------------------------------------------------------------------- fill_mouth
// One CTA per image.  state[p]: 0 = not fillable, 1 = fillable, 2 = reached from the corner.  Alternating row / column
// sweeps (one thread per row resp. column, forward + backward) until a pass changes nothing -- a few passes for
// face-silhouette masks.  Then res = clip(alpha + 1 - (filled/127.5 - 1)) in the reference's op order.
__global__ void __launch_bounds__(1024) fill_mouth_kernel(float* __restrict__ alpha, int H, int W) {
    extern __shared__ unsigned char st[];
    __shared__ int s_changed;
    const int SW = W + 4;                  // row pitch in bytes: (W+4)/4 is odd -> row sweeps (one thread per row) are bank-conflict free
    float* a = alpha + (int64_t)blockIdx.x * H * W;
    const float seed = __fmul_rn(a[0], 255.f);
    const float vmin = seed, vmax = __fadd_rn(seed, 254.f);
    for (int i = threadIdx.x; i < H * W; i += blockDim.x) {
        const float v = __fmul_rn(a[i], 255.f);
        st[(i / W) * SW + (i % W)] = (v >= vmin && v <= vmax) ? 1 : 0;
    }
    __syncthreads();
    if (threadIdx.x == 0) st[0] = 2;      // the seed pixel itself is always filled
    __syncthreads();
    // Four sweep directions run concurrently on disjoint thread groups (state only ever goes 1 -> 2, byte stores: benign races
    // merely delay propagation to the next pass); repeat until a pass changes nothing.
    const int group = threadIdx.x >> 8, gi = threadIdx.x & 255;
    for (int iter = 0; iter < 4 * (H + W); ++iter) {
        if (threadIdx.x == 0) s_changed = 0;
        __syncthreads();
        int changed = 0;
        if (group == 0) {
            for (int y = gi; y < H; y += 256) { unsigned char* r = st + y * SW; bool reach = false;
                for (int x = 0; x < W; ++x) { const unsigned char s = r[x]; if (s == 0) reach = false; else if (s == 2) reach = true; else if (reach) { r[x] = 2; changed = 1; } } }
        } else if (group == 1) {
            for (int y = gi; y < H; y += 256) { unsigned char* r = st + y * SW; bool reach = false;
                for (int x = W - 1; x >= 0; --x) { const unsigned char s = r[x]; if (s == 0) reach = false; else if (s == 2) reach = true; else if (reach) { r[x] = 2; changed = 1; } } }
        } else if (group == 2) {
            for (int x = gi; x < W; x += 256) { bool reach = false;
                for (int y = 0; y < H; ++y) { const unsigned char s = st[y * SW + x]; if (s == 0) reach = false; else if (s == 2) reach = true; else if (reach) { st[y * SW + x] = 2; changed = 1; } } }
        } else {
            for (int x = gi; x < W; x += 256) { bool reach = false;
                for (int y = H - 1; y >= 0; --y) { const unsigned char s = st[y * SW + x]; if (s == 0) reach = false; else if (s == 2) reach = true; else if (reach) { st[y * SW + x] = 2; changed = 1; } } }
        }
        if (changed) atomicOr(&s_changed, 1);
        __syncthreads();
        const int any = s_changed;
        __syncthreads();
        if (!any) break;
    }
    for (int i = threadIdx.x; i < H * W; i += blockDim.x) {
        const float al = a[i];
        const float filled = st[(i / W) * SW + (i % W)] == 2 ? 255.f : __fmul_rn(al, 255.f);
        const float m = __fsub_rn(__fdiv_rn(filled, 127.5f), 1.f);
        const float t = __fdiv_rn(__fadd_rn(__fmul_rn(__fsub_rn(__fmul_rn(m, 2.f), 1.f), -1.f), 1.f), 2.f);
        a[i] = fminf(fmaxf(__fadd_rn(al, t), 0.f), 1.f);
    }
}

// ---------------------------------------------------------------------------------------------- mouth box
__global__ void mouth_box_kernel(const float* __restrict__ lm2d, int N, int* __restrict__ boxes) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const float* lm = lm2d + (int64_t)n * 68 * 2;
    float mx0 = -INFINITY, mn0 = INFINITY, mx1 = -INFINITY, mn1 = INFINITY;
    float l0 = 0.f, l1 = 0.f, r0 = 0.f, r1 = 0.f;
    for (int k = 48; k < 60; ++k) {
        const float a = __fadd_rn(__fmul_rn(lm[k * 2], 128.f), 128.f), b = __fadd_rn(__fmul_rn(lm[k * 2 + 1], 128.f), 128.f);
        mx0 = fmaxf(mx0, a); mn0 = fminf(mn0, a); mx1 = fmaxf(mx1, b); mn1 = fminf(mn1, b);
        if (k == 48) { l0 = a; l1 = b; }
        if (k == 54) { r0 = a; r1 = b; }
    }
    const float avg0 = __fmul_rn(__fadd_rn(l0, r0), 0.5f), avg1 = __fmul_rn(__fadd_rn(l1, r1), 0.5f);
    const float ext = fmaxf(__fsub_rn(mx0, mn0), __fsub_rn(mx1, mn1));
    const int side = (int)__fmul_rn(ext, 1.2f);                 // float32 * 1.2 -> astype(int): truncation
    const int half = side >= 0 ? side / 2 : -((-side + 1) / 2);  // python floor division
    boxes[n * 4 + 0] = (int)((double)avg1 - (double)half);
    boxes[n * 4 + 1] = (int)((double)avg1 + (double)half);
    boxes[n * 4 + 2] = (int)((double)avg0 - (double)half);
    boxes[n * 4 + 3] = (int)((double)avg0 + (double)half);
}

// ---------------------------------------------------------------------------------------------- antialiased resize
// ATen _upsample_bilinear2d_aa weights for one axis (SURVEY.md A.10), fp32 like ATen's accscalar path.
struct AxisTaps { int lo, n; float scale, center, inv, total; };
__device__ __forceinline__ AxisTaps aa_axis(int out_i, int in_size, int out_size) {
    AxisTaps t;
    t.scale = (float)in_size / (float)out_size;
    const float support = t.scale >= 1.f ? t.scale : 1.f;
    t.inv = t.scale >= 1.f ? 1.f / t.scale : 1.f;
    t.center = t.scale * ((float)out_i + 0.5f);
    t.lo = max((int)(t.center - support + 0.5f), 0);
    const int hi = min((int)(t.center + support + 0.5f), in_size);
    t.n = hi - t.lo;
    float tot = 0.f;
    for (int j = 0; j < t.n; ++j) tot += fmaxf(0.f, 1.f - fabsf(((float)(j + t.lo) - t.center + 0.5f) * t.inv));
    t.total = tot;
    return t;
}
__device__ __forceinline__ float aa_weight(const AxisTaps& t, int j) {
    const float w = fmaxf(0.f, 1.f - fabsf(((float)(j + t.lo) - t.center + 0.5f) * t.inv));
    return t.total != 0.f ? w / t.total : w;
}

// Source / destination windows of image n (python slicing semantics: boxes clipped to the image).  Returns false when the
// destination pixel (dy, dx) lies outside the paste window or a window is empty.
struct ResizeWin { int sy0, sx0, ih, iw, ty0, tx0, oh, ow; };
__device__ __forceinline__ bool resize_window(const int* __restrict__ src_box, const int* __restrict__ dst_box, int n, int SH, int SW, int DH, int DW,
                                              int dy, int dx, ResizeWin& w) {
    int sy0 = 0, sy1 = SH, sx0 = 0, sx1 = SW, ty0 = 0, ty1 = DH, tx0 = 0, tx1 = DW;
    if (src_box) { sy0 = src_box[n * 4]; sy1 = src_box[n * 4 + 1]; sx0 = src_box[n * 4 + 2]; sx1 = src_box[n * 4 + 3]; }
    if (dst_box) { ty0 = dst_box[n * 4]; ty1 = dst_box[n * 4 + 1]; tx0 = dst_box[n * 4 + 2]; tx1 = dst_box[n * 4 + 3]; }
    sy0 = max(sy0, 0); sx0 = max(sx0, 0); sy1 = min(sy1, SH); sx1 = min(sx1, SW);
    w.sy0 = sy0; w.sx0 = sx0; w.ih = sy1 - sy0; w.iw = sx1 - sx0; w.ty0 = ty0; w.tx0 = tx0; w.oh = ty1 - ty0; w.ow = tx1 - tx0;
    if (dy < ty0 || dy >= ty1 || dx < tx0 || dx >= tx1) return false;
    return w.ih > 0 && w.iw > 0 && w.oh > 0 && w.ow > 0;
}

__device__ __forceinline__ void resize_store(float acc, int64_t o, int n, int C, int c, float* __restrict__ dst, const float* __restrict__ style,
                                             __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo) {
    if (dst) dst[o] = acc;
    if (hi) {
        float s = acc;
        if (style) s *= __ldg(style + (int64_t)n * C + c);
        __nv_bfloat16 h, l;
        split_bf16(s, h, l);
        hi[o] = h; lo[o] = l;
    }
}

// Wide channels (C = 4 * 2^k <= 128): one warp per destination pixel; the lanes are split into C/4 float4 channel groups x
// 32/(C/4) tap lanes, each tap lane walks every (32/(C/4))-th tap of the window, then the tap lanes are summed with shuffles.
// A warp owns `ppw` consecutive destination pixels per step: their window tests run in parallel on the lanes (ballot), the
// pixels inside are then filtered one after the other.
__global__ void __launch_bounds__(256) resize_aa_kernel(const float* __restrict__ src, int N, int SH, int SW, int C, const int* __restrict__ src_box,
                                                        float* __restrict__ dst, int DH, int DW, const int* __restrict__ dst_box, const float* __restrict__ style,
                                                        __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo, int ppw) {
    const int lane = threadIdx.x & 31;
    const int64_t warp_global = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t total = (int64_t)N * DH * DW;
    const int c4n = C >> 2, ntl = 32 / c4n, tl = lane / c4n, c4 = lane - tl * c4n;
    for (int64_t base = warp_global * ppw; base < total; base += nwarps * ppw) {
        // lane l < ppw tests destination pixel base + l; the warp then visits the pixels that are inside their paste window
        bool inside = false;
        {
            const int64_t pi = base + lane;
            if (lane < ppw && pi < total) {
                ResizeWin w;
                inside = resize_window(src_box, dst_box, (int)(pi / ((int64_t)DH * DW)), SH, SW, DH, DW, (int)((pi / DW) % DH), (int)(pi % DW), w);
            }
        }
        unsigned todo = __ballot_sync(0xffffffffu, inside);
        while (todo) {
            const int l = __ffs(todo) - 1;
            todo &= todo - 1;
            const int64_t pi = base + l;
            const int n = (int)(pi / ((int64_t)DH * DW)), dy = (int)((pi / DW) % DH), dx = (int)(pi % DW);
            ResizeWin w;
            resize_window(src_box, dst_box, n, SH, SW, DH, DW, dy, dx, w);
            const AxisTaps ay = aa_axis(dy - w.ty0, w.ih, w.oh), ax = aa_axis(dx - w.tx0, w.iw, w.ow);
            const int nt = ay.n * ax.n;
            const float4* win0 = reinterpret_cast<const float4*>(src + (((int64_t)n * SH + w.sy0 + ay.lo) * SW + w.sx0 + ax.lo) * C);
            const int64_t o = (((int64_t)n * DH + dy) * DW + dx) * C;
            if (nt >= 64 && c4n <= 8) {
                // Strong minification (the 256^2 -> ~40^2 mouth paste: ~200 taps): every lane is a tap lane and fetches all
                // channels of its taps (independent 128-byte loads), then one butterfly reduction over the warp.
                float4 acc[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) acc[k] = make_float4(0.f, 0.f, 0.f, 0.f);
                for (int t = lane; t < nt; t += 32) {
                    const int j = t / ax.n, i = t - j * ax.n;
                    const float wt = aa_weight(ay, j) * aa_weight(ax, i);
                    const float4* tp = win0 + ((int64_t)j * SW + i) * c4n;
#pragma unroll
                    for (int k = 0; k < 8; ++k) {
                        if (k < c4n) {
                            const float4 v = __ldg(tp + k);
                            acc[k].x = fmaf(wt, v.x, acc[k].x); acc[k].y = fmaf(wt, v.y, acc[k].y);
                            acc[k].z = fmaf(wt, v.z, acc[k].z); acc[k].w = fmaf(wt, v.w, acc[k].w);
                        }
                    }
                }
                float4 mine = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    if (k < c4n) {
                        float4 a = acc[k];
#pragma unroll
                        for (int off = 16; off >= 1; off >>= 1) {
                            a.x += __shfl_xor_sync(0xffffffffu, a.x, off); a.y += __shfl_xor_sync(0xffffffffu, a.y, off);
                            a.z += __shfl_xor_sync(0xffffffffu, a.z, off); a.w += __shfl_xor_sync(0xffffffffu, a.w, off);
                        }
                        if (lane == k) mine = a;
                    }
                }
                if (lane < c4n) {
                    const float a[4] = {mine.x, mine.y, mine.z, mine.w};
#pragma unroll
                    for (int e = 0; e < 4; ++e) resize_store(a[e], o + lane * 4 + e, n, C, lane * 4 + e, dst, style, hi, lo);
                }
                continue;
            }
            const float4* win = win0 + c4;
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
            for (int t = tl; t < nt; t += ntl) {
                const int j = t / ax.n, i = t - j * ax.n;
                const float wt = aa_weight(ay, j) * aa_weight(ax, i);
                const float4 v = __ldg(win + ((int64_t)j * SW + i) * c4n);
                acc.x = fmaf(wt, v.x, acc.x); acc.y = fmaf(wt, v.y, acc.y); acc.z = fmaf(wt, v.z, acc.z); acc.w = fmaf(wt, v.w, acc.w);
            }
            for (int off = c4n; off < 32; off <<= 1) {
                acc.x += __shfl_xor_sync(0xffffffffu, acc.x, off); acc.y += __shfl_xor_sync(0xffffffffu, acc.y, off);
                acc.z += __shfl_xor_sync(0xffffffffu, acc.z, off); acc.w += __shfl_xor_sync(0xffffffffu, acc.w, off);
            }
            if (tl == 0) {
                const float a[4] = {acc.x, acc.y, acc.z, acc.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) resize_store(a[e], o + c4 * 4 + e, n, C, c4 * 4 + e, dst, style, hi, lo);
            }
        }
    }
}

// Any other channel count (the 3-channel raw image): one thread per (destination pixel, channel).
__global__ void __launch_bounds__(256) resize_aa_scalar_kernel(const float* __restrict__ src, int N, int SH, int SW, int C, const int* __restrict__ src_box,
                                                               float* __restrict__ dst, int DH, int DW, const int* __restrict__ dst_box,
                                                               const float* __restrict__ style, __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo) {
    const int64_t total = (int64_t)N * DH * DW * C;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(idx % C);
        const int64_t pi = idx / C;
        const int n = (int)(pi / ((int64_t)DH * DW)), dy = (int)((pi / DW) % DH), dx = (int)(pi % DW);
        ResizeWin w;
        if (!resize_window(src_box, dst_box, n, SH, SW, DH, DW, dy, dx, w)) continue;
        const AxisTaps ay = aa_axis(dy - w.ty0, w.ih, w.oh), ax = aa_axis(dx - w.tx0, w.iw, w.ow);
        float acc = 0.f;
        for (int j = 0; j < ay.n; ++j) {
            const float* row = src + (((int64_t)n * SH + w.sy0 + ay.lo + j) * SW + w.sx0 + ax.lo) * C + c;
            float racc = 0.f;
            for (int i = 0; i < ax.n; ++i) racc += aa_weight(ax, i) * __ldg(row + (int64_t)i * C);
            acc += aa_weight(ay, j) * racc;
        }
        resize_store(acc, idx, n, C, c, dst, style, hi, lo);
    }
}

// ---------------------------------------------------------------------------------------------- plane blend
// planes[n,p,y,x,c] = tex[n,p,y,x,c]*a + static[n,y,x,p*32+c]*(1-a); plane 0's texture comes from the neural-blending output
__global__ void __launch_bounds__(256) blend_kernel(const float* __restrict__ front, const float* __restrict__ tex, const float* __restrict__ alpha,
                                                    const float* __restrict__ stat, int N, int HW, float* __restrict__ planes) {
    const int64_t total = (int64_t)N * 3 * HW * 8;     // float4 groups of the 32 channels
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int c4 = (int)(i & 7);
        int64_t t = i >> 3;
        const int64_t pix = t % HW; t /= HW;
        const int p = (int)(t % 3);
        const int n = (int)(t / 3);
        const float a = __ldg(alpha + ((int64_t)p * N + n) * HW + pix);
        const float4 tv = p == 0 ? __ldg(reinterpret_cast<const float4*>(front + ((int64_t)n * HW + pix) * 32) + c4)
                                 : __ldg(reinterpret_cast<const float4*>(tex + (((int64_t)p * N + n) * HW + pix) * 32) + c4);
        const float4 sv = __ldg(reinterpret_cast<const float4*>(stat + ((int64_t)n * HW + pix) * 96 + p * 32) + c4);
        const float b = 1.f - a;
        float4 o;
        o.x = tv.x * a + sv.x * b; o.y = tv.y * a + sv.y * b; o.z = tv.z * a + sv.z * b; o.w = tv.w * a + sv.w * b;
        reinterpret_cast<float4*>(planes)[i] = o;
    }
}
}  // namespace

extern "C" int n3d_transform_points(const float* pts, int N, int P, const float* rot, int nviews, float zoff, int ndc_flip,
                                    float* out, void* stream) {
    N3D_CHECK_ARG(pts && rot && out && N > 0 && P > 0 && nviews > 0, "n3d_transform_points: bad args");
    transform_kernel<<<grid_for((int64_t)N * nviews * P, 256), 256, 0, (cudaStream_t)stream>>>(pts, N, P, rot, nviews, zoff, ndc_flip, out);
    N3D_CHECK_LAUNCH("n3d_transform_points");
    return N3D_OK;
}

extern "C" int n3d_rasterize(const float* verts, const int32_t* faces, int NM, int V, int F, int H, int W, int32_t* pix_to_face,
                             float* bary, float* workspace, void* stream) {
    N3D_CHECK_ARG(verts && faces && pix_to_face && bary && workspace && NM > 0 && F > 0 && H > 0 && W > 0, "n3d_rasterize: bad args");
    N3D_CHECK_ARG(NM <= 65535, "n3d_rasterize: too many images (%d)", NM);
    N3D_CHECK_ARG(((uintptr_t)workspace & 15) == 0, "n3d_rasterize: workspace must be 16-byte aligned");
    raster_setup_kernel<<<grid_for((int64_t)NM * F, 256), 256, 0, (cudaStream_t)stream>>>(verts, faces, NM, V, F, workspace);
    dim3 grid(((W + kBin - 1) / kBin) * ((H + kBin - 1) / kBin), NM);
    rasterize_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(workspace, F, H, W, pix_to_face, bary);
    N3D_CHECK_LAUNCH("n3d_rasterize");
    return N3D_OK;
}

extern "C" int n3d_uv_sample(const int32_t* pix_to_face, const float* bary, const float* face_uv, const float* texture,
                             const float* eye_mask, int N, int H, int W, int TH, int TW, int C, int MH, int MW,
                             float* tex_planes, float* alpha, void* stream) {
    N3D_CHECK_ARG(pix_to_face && bary && face_uv && texture && eye_mask && tex_planes && alpha, "n3d_uv_sample: null pointer");
    N3D_CHECK_ARG(C <= 32, "n3d_uv_sample: C %d > 32 not supported", C);
    uv_sample_kernel<<<grid_for((int64_t)N * H * W * 32, 256, 16), 256, 0, (cudaStream_t)stream>>>(pix_to_face, bary, face_uv, texture, eye_mask, N, H,
                                                                                                W, TH, TW, C, MH, MW, tex_planes, alpha);
    N3D_CHECK_LAUNCH("n3d_uv_sample");
    return N3D_OK;
}

extern "C" int n3d_fill_mouth(float* alpha, int NI, int H, int W, void* stream) {
    N3D_CHECK_ARG(alpha && NI > 0 && H > 0 && W > 0, "n3d_fill_mouth: bad args");
    N3D_CHECK_ARG((int64_t)H * (W + 4) <= 200 * 1024, "n3d_fill_mouth: image %dx%d too large for the shared-memory state map", H, W);
    N3DDeviceState* D = n3d_device_state();
    if (!D) return N3D_ERR_CUDA;
    if (int e = n3d_smem_optin(D, N3D_CFG_FILL_MOUTH, (const void*)fill_mouth_kernel, 200 * 1024, "n3d_fill_mouth")) return e;
    fill_mouth_kernel<<<NI, 1024, (size_t)H * (W + 4), (cudaStream_t)stream>>>(alpha, H, W);
    N3D_CHECK_LAUNCH("n3d_fill_mouth");
    return N3D_OK;
}

extern "C" int n3d_mouth_box(const float* lm2d, int N, int32_t* boxes, void* stream) {
    N3D_CHECK_ARG(lm2d && boxes && N > 0, "n3d_mouth_box: bad args");
    mouth_box_kernel<<<(N + 63) / 64, 64, 0, (cudaStream_t)stream>>>(lm2d, N, boxes);
    N3D_CHECK_LAUNCH("n3d_mouth_box");
    return N3D_OK;
}

extern "C" int n3d_resize_aa(const float* src, int N, int SH, int SW, int C, const int32_t* src_box, float* dst, int DH, int DW,
                             const int32_t* dst_box, const float* style, void* hi, void* lo, void* stream) {
    N3D_CHECK_ARG(src && (dst || hi) && N > 0 && C > 0, "n3d_resize_aa: bad args");
    N3D_CHECK_ARG(!hi || lo, "n3d_resize_aa: hi without lo");
    const bool wide = (C % 4 == 0) && C <= 128 && (32 % (C / 4) == 0) && ((uintptr_t)src % 16 == 0);
    const int ppw = 4;
    if (wide)
        resize_aa_kernel<<<grid_for((int64_t)N * DH * DW * 32 / ppw, 256, 16), 256, 0, (cudaStream_t)stream>>>(
            src, N, SH, SW, C, src_box, dst, DH, DW, dst_box, style, (__nv_bfloat16*)hi, (__nv_bfloat16*)lo, ppw);
    else
        resize_aa_scalar_kernel<<<grid_for((int64_t)N * DH * DW * C, 256, 16), 256, 0, (cudaStream_t)stream>>>(
            src, N, SH, SW, C, src_box, dst, DH, DW, dst_box, style, (__nv_bfloat16*)hi, (__nv_bfloat16*)lo);
    N3D_CHECK_LAUNCH("n3d_resize_aa");
    return N3D_OK;
}

extern "C" int n3d_blend_planes(const float* blended_front, const float* tex_planes, const float* alpha, const float* static_planes,
                                int N, int H, int W, float* planes, void* stream) {
    N3D_CHECK_ARG(blended_front && tex_planes && alpha && static_planes && planes, "n3d_blend_planes: null pointer");
    blend_kernel<<<grid_for((int64_t)N * 3 * H * W * 8, 256, 16), 256, 0, (cudaStream_t)stream>>>(blended_front, tex_planes, alpha, static_planes, N, H * W, planes);
    N3D_CHECK_LAUNCH("n3d_blend_planes");
    return N3D_OK;
}
