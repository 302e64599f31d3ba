// Shared helpers for libnext3d_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>

// Error codes returned by every extern "C" entry point (include/next3d_b200.h).
#define N3D_OK 0
#define N3D_ERR_INVALID_ARG (-1)
#define N3D_ERR_UNSUPPORTED (-2)
#define N3D_ERR_CUDA (-3)

void n3d_set_error(const char* fmt, ...);

#define N3D_CHECK_ARG(cond, ...)                        \
    do {                                                \
        if (!(cond)) {                                  \
            n3d_set_error(__VA_ARGS__);                 \
            return N3D_ERR_INVALID_ARG;                 \
        }                                               \
    } while (0)

#define N3D_CHECK_LAUNCH(name)                                                       \
    do {                                                                             \
        cudaError_t e__ = cudaGetLastError();                                        \
        if (e__ != cudaSuccess) {                                                    \
            n3d_set_error("%s: launch failed: %s", name, cudaGetErrorString(e__));   \
            return N3D_ERR_CUDA;                                                     \
        }                                                                            \
    } while (0)

static inline int n3d_div_up(long long a, long long b) { return (int)((a + b - 1) / b); }

// Host-side facts cached PER DEVICE (the library holds no device memory and no device-global state): SM count and which kernels
// already had their dynamic shared-memory limit raised on that device.  Indexed by the current device at call time.
struct N3DDeviceState {
    int num_sms;
    unsigned configured;     // bit per kernel, see N3D_CFG_*
};
enum { N3D_CFG_CONV = 1u, N3D_CFG_FILL_MOUTH = 2u, N3D_CFG_RENDER16 = 4u, N3D_CFG_RENDER32 = 8u, N3D_CFG_POINTS = 16u, N3D_CFG_FIR_STREAM = 32u, N3D_CFG_FIR_DOWN_STREAM = 64u,
       N3D_CFG_POINTS_RGB = 128u, N3D_CFG_FLOOR_GATHER = 256u };
N3DDeviceState* n3d_device_state(void);      // api.cu; nullptr (+ error message) when the current device cannot be queried
// api.cu: raises `kernel`'s dynamic shared-memory limit to `bytes` once per device (bit `cfg_bit` of D->configured).  N3D_OK, or
// N3D_ERR_CUDA with an error message naming `who`.
int n3d_smem_optin(N3DDeviceState* D, unsigned cfg_bit, const void* kernel, int bytes, const char* who);

// fp32 -> (hi, lo) bf16 pair with hi + lo ~= x to ~16 mantissa bits (used by the 3-product tensor-core scheme).
__device__ __forceinline__ void split_bf16(float x, __nv_bfloat16& hi, __nv_bfloat16& lo) {
    hi = __float2bfloat16_rn(x);
    lo = __float2bfloat16_rn(x - __bfloat162float(hi));
}

// Two values at once -> packed bf16x2 words (element a in the low half): one cvt.rn.bf16x2.f32 per word instead of two scalar
// conversions plus a byte permute.  Bit-identical to split_bf16 on each element.
__device__ __forceinline__ void split_bf16x2(float a, float b, uint32_t& hi, uint32_t& lo) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    hi = *reinterpret_cast<const uint32_t*>(&h);
    const float2 r = __fadd2_rn(make_float2(a, b), make_float2(-__uint_as_float(hi << 16), -__uint_as_float(hi & 0xffff0000u)));   // exact
    const __nv_bfloat162 l = __floats2bfloat162_rn(r.x, r.y);
    lo = *reinterpret_cast<const uint32_t*>(&l);
}

// 256-bit global accesses (sm_100: LDG/STG.E.ENL2.256): one full 32-byte sector per thread and instruction.  `p` must be
// 32-byte aligned.
__device__ __forceinline__ void st_global_256(void* p, const uint32_t (&w)[8]) {
    asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(w[0]), "r"(w[1]), "r"(w[2]), "r"(w[3]), "r"(w[4]), "r"(w[5]),
                 "r"(w[6]), "r"(w[7])
                 : "memory");
}
__device__ __forceinline__ void st_global_256(float* p, const float* v) {
    asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]),
                 "f"(v[6]), "f"(v[7])
                 : "memory");
}
__device__ __forceinline__ void ld_global_256(const float* p, float* v) {
    asm volatile("ld.global.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7])
                 : "l"(p)
                 : "memory");
}

// read-only variant (non-coherent path, freely schedulable: no volatile, no memory clobber)
__device__ __forceinline__ void ldg_nc_256(const float* p, float* v) {
    asm("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
        : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7])
        : "l"(p));
}

__device__ __forceinline__ uint32_t pack_bf16x2(__nv_bfloat16 a, __nv_bfloat16 b) {
    return (uint32_t)__bfloat16_as_ushort(a) | ((uint32_t)__bfloat16_as_ushort(b) << 16);
}
