// capi.cu — library plumbing of libtrl_b200.so: version, errors, workspace.
#include <cuda_runtime.h>
#include <mutex>
#include <stdio.h>
#include <string.h>

#include "trl_common.cuh"

static thread_local char g_err[256] = "";
static std::mutex g_ws_mutex;
// per device: workspace slots and host streams, created under that device
struct DeviceSlots {
    void* ws_ptr[TRL_WS_SLOTS];
    size_t ws_size[TRL_WS_SLOTS];
    cudaStream_t host_stream[TRL_HOST_STREAMS];
};
static DeviceSlots g_dev[TRL_MAX_DEVICES] = {};

int trl_check(cudaError_t e) {
    if (e == cudaSuccess) return TRL_OK;
    strncpy(g_err, cudaGetErrorString(e), sizeof(g_err) - 1);
    g_err[sizeof(g_err) - 1] = 0;
    return TRL_E_CUDA;
}

int trl_device() {
    int dev = -1;
    if (trl_check(cudaGetDevice(&dev)) != TRL_OK) return -1;
    if (dev < 0 || dev >= TRL_MAX_DEVICES) {
        snprintf(g_err, sizeof(g_err), "device %d lies past the library's per-device tables (%d entries)", dev, TRL_MAX_DEVICES);
        return -1;
    }
    return dev;
}

void* trl_workspace(int slot, size_t bytes) {
    std::lock_guard<std::mutex> lock(g_ws_mutex);
    if (slot < 0 || slot >= TRL_WS_SLOTS) return nullptr;
    const int dev = trl_device();
    if (dev < 0) return nullptr;
    void*& ptr = g_dev[dev].ws_ptr[slot];
    size_t& size = g_dev[dev].ws_size[slot];
    if (size >= bytes && ptr) return ptr;
    if (ptr) { cudaFree(ptr); ptr = nullptr; size = 0; }
    void* p = nullptr;
    if (trl_check(cudaMalloc(&p, bytes)) != TRL_OK) return nullptr;
    // counters start at zero.  cudaMemset runs on the legacy default stream, which the library's non-blocking
    // streams do not wait for: without the synchronisation the memset can land AFTER the first H2D copy into
    // the new buffer (seen as wrong answers for the first calls after a re-allocation).
    if (trl_check(cudaMemset(p, 0, bytes)) != TRL_OK || trl_check(cudaDeviceSynchronize()) != TRL_OK) { cudaFree(p); return nullptr; }
    ptr = p;
    size = bytes;
    return p;
}

cudaStream_t trl_host_stream(int which) {
    std::lock_guard<std::mutex> lock(g_ws_mutex);
    const int dev = trl_device();
    if (dev < 0) return nullptr;
    cudaStream_t& s = g_dev[dev].host_stream[which & (TRL_HOST_STREAMS - 1)];
    if (!s) {
        if (trl_check(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking)) != TRL_OK) return nullptr;
    }
    return s;
}

int g_trl_pdl = 1;
extern "C" void trl_set_pdl(int enabled) { g_trl_pdl = enabled ? 1 : 0; }

extern "C" int trl_abi_version(void) { return 10; }
extern "C" const char* trl_last_error(void) { return g_err; }
extern "C" int trl_sizeof_player(void) { return (int)sizeof(TrlPlayer); }
extern "C" int trl_sizeof_game(void) { return (int)sizeof(TrlGame); }

// One-thread kernel that records the GPU's global nanosecond timer: put between the kernels of a
// captured step to get the in-graph timeline (tools/step_timeline.py).
__global__ void stamp_kernel(unsigned long long* slot) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    *slot = t;
}
extern "C" int trl_stamp_globaltimer(unsigned long long* slot, void* stream) {
    if (!slot) return TRL_E_ARG;
    stamp_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(slot);
    return trl_check(cudaGetLastError());
}
