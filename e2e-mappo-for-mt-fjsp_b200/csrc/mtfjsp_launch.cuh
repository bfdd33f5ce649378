// mtfjsp_launch.cuh -- host-side launch and error helpers shared by every CUDA source of the library (no device code).
//
// fail() keeps the one per-thread message mtfjsp_last_error returns, so whichever entry point failed last on a thread is
// the one it describes.  The caches below are per device, not per thread: a thread may drive several GPUs, and several
// threads one GPU.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <map>
#include <mutex>

#include "../../include/mtfjsp.h"

// one copy for the whole library, none exported from it
#pragma GCC visibility push(hidden)

inline thread_local char g_err[512] = "";

// records why the call fails (`what` names the entry point) and returns its code
inline int fail(int code, const char* what, cudaError_t e = cudaSuccess) {
    if (e != cudaSuccess) snprintf(g_err, sizeof g_err, "%s: %s", what, cudaGetErrorString(e));
    else snprintf(g_err, sizeof g_err, "%s", what);
    return code;
}

#define CK(call, msg)                                               \
    do {                                                            \
        cudaError_t e_ = (call);                                    \
        if (e_ != cudaSuccess) return fail(MTFJSP_E_CUDA, msg, e_); \
    } while (0)

// the tail of a launch: MTFJSP_OK, or MTFJSP_E_CUDA with the launch error
inline int launched(const char* what) {
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? MTFJSP_OK : fail(MTFJSP_E_CUDA, what, e);
}

// keys of the caches below; being types of this header, they keep the std::map code out of the exports too
struct KernelOnDevice {
    const void* kernel;
    int dev;
    bool operator<(const KernelOnDevice& o) const { return kernel != o.kernel ? kernel < o.kernel : dev < o.dev; }
};
struct Device {
    int dev;
    bool operator<(const Device& o) const { return dev < o.dev; }
};

// Lets `kernel` take `bytes` of dynamic shared memory on the current device.  The runtime applies the attribute to the
// current device only, so it is set once per (kernel, device), and again only when a larger size is asked for there.  At
// or below 48 KB no opt-in is needed: every kernel launched through here declares no static shared memory.
inline cudaError_t opt_in_smem(const void* kernel, size_t bytes) {
    if (bytes <= 48 * 1024) return cudaSuccess;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    static std::mutex mu;
    static std::map<KernelOnDevice, size_t> granted;
    std::lock_guard<std::mutex> lock(mu);
    size_t& have = granted[{kernel, dev}];
    if (have >= bytes) return cudaSuccess;
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e == cudaSuccess) have = bytes;
    return e;
}
template <class... A>
cudaError_t opt_in_smem(void (*kernel)(A...), size_t bytes) {
    return opt_in_smem(reinterpret_cast<const void*>(kernel), bytes);
}

// SMs of the current device (148 on a B200, and the fallback when the query fails)
inline int sm_count() {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    static std::mutex mu;
    static std::map<Device, int> known;
    std::lock_guard<std::mutex> lock(mu);
    const auto it = known.find(Device{dev});
    if (it != known.end()) return it->second;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess) known[Device{dev}] = sms;
    return sms;
}

// one persistent CTA per SM, fewer when there are fewer tiles
inline int persistent_grid(long long tiles) {
    const int sms = sm_count();
    return (int)(tiles < sms ? tiles : sms);
}

// Operand alignment, checked on the host before any launch: cp.async, TMA and the float4 loads / stores move 16 bytes at a
// time, adj_w and fea1 are read as float2.  NULL passes (optional pointers are checked for presence separately).
template <class... P>
bool al16(P... p) { return ((((uintptr_t)p & 15) == 0) && ...); }
inline bool al8(const void* p) { return ((uintptr_t)p & 7) == 0; }

#pragma GCC visibility pop
