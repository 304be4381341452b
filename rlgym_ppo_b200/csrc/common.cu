#include <stdarg.h>

#include <stdlib.h>

#include "common.cuh"

namespace rlppo {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

static int g_dev_ok[64];  // 0 unknown, 1 ok, -1 bad
static int g_dev_sms[64];

int check_device() {
    int dev = -1;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess || dev < 0 || dev >= 64) {
        set_error("no CUDA device available (%s); librlppo_b200 has no CPU fallback",
                  e == cudaSuccess ? "bad device index" : cudaGetErrorString(e));
        cudaGetLastError();
        return RLPPO_ERR_DEVICE;
    }
    if (g_dev_ok[dev] == 0) {
        cudaDeviceProp p;
        e = cudaGetDeviceProperties(&p, dev);
        if (e != cudaSuccess) {
            set_error("cudaGetDeviceProperties: %s", cudaGetErrorString(e));
            return RLPPO_ERR_DEVICE;
        }
        g_dev_sms[dev] = p.multiProcessorCount;
        g_dev_ok[dev] = (p.major == 10) ? 1 : -1;
    }
    if (g_dev_ok[dev] < 0) {
        set_error("device %d is not compute capability 10.x; the kernels are built for sm_100a only", dev);
        return RLPPO_ERR_DEVICE;
    }
    return RLPPO_OK;
}

int pdl_mode() {
    static int mode = -1;
    if (mode < 0) {
        const char* e = getenv("RLPPO_PDL");
        mode = (e != nullptr && e[0] == '0') ? 0 : 1;
    }
    return mode;
}

int num_sms() {
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64 || g_dev_sms[dev] == 0) return 148;
    return g_dev_sms[dev];
}

}  // namespace rlppo

extern "C" {
int rlppo_version(void) { return 101; }
const char* rlppo_last_error(void) { return rlppo::g_err; }
int rlppo_device_check(void) { return rlppo::check_device(); }
}
