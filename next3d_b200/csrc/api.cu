// Library-level entry points: error reporting and version.
#include "common.cuh"
#include "../../include/next3d_b200.h"
#include <stdarg.h>

static thread_local char g_err[512] = "";

void n3d_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

extern "C" const char* n3d_last_error(void) { return g_err; }
extern "C" int n3d_version(void) { return 100; }

static N3DDeviceState g_dev_state[128];

N3DDeviceState* n3d_device_state(void) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 128) {
        n3d_set_error("cannot query the current CUDA device");
        return nullptr;
    }
    N3DDeviceState* d = &g_dev_state[dev];
    if (!d->num_sms) {
        int n = 0;
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        d->num_sms = n > 0 ? n : 148;
    }
    return d;
}

int n3d_smem_optin(N3DDeviceState* D, unsigned cfg_bit, const void* kernel, int bytes, const char* who) {
    if (D->configured & cfg_bit) return N3D_OK;
    const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e != cudaSuccess) {
        n3d_set_error("%s: cannot raise dynamic shared memory to %d bytes: %s", who, bytes, cudaGetErrorString(e));
        return N3D_ERR_CUDA;
    }
    D->configured |= cfg_bit;
    return N3D_OK;
}
