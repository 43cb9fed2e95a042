// trl_common.cuh — error plumbing and the library-owned device workspace.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include "../../include/trl.h"

// Records the error text for trl_last_error(); returns TRL_OK or TRL_E_CUDA.
int trl_check(cudaError_t e);

// Every call runs on the current device.  State the library keeps between calls (workspace, host streams, kernel
// attributes, SM counts, pushed debug switches) is kept per device, in tables of TRL_MAX_DEVICES entries.
#define TRL_MAX_DEVICES 64
// Index of the current device; -1 (error text set, the caller returns TRL_E_CUDA) if it cannot be read or lies past
// the tables.
int trl_device();

// Library-owned, grow-only device scratch of the current device (used only by the *_host entry points, the trunk work
// counters and trl_movegen when the caller passes no mask buffer).  Returns nullptr on failure.
enum TrlWorkspaceSlot { TRL_WS_MOVEGEN_MASK = 0, TRL_WS_HOST_STAGE = 1, TRL_WS_TRUNK_COUNTER = 2, TRL_WS_TRUNK_COUNTER_TAPS = 3, TRL_WS_TRUNK_COUNTER_WIDE = 4, TRL_WS_HOST_BOARDS = 5, TRL_WS_SLOTS = 6 };
void* trl_workspace(int slot, size_t bytes);

// Streams (0 .. TRL_HOST_STREAMS - 1) of the current device used by the *_host entry points (created on first use,
// non-blocking).  nullptr on failure.
#ifndef TRL_HOST_STREAMS
#define TRL_HOST_STREAMS 4
#endif
cudaStream_t trl_host_stream(int which = 0);

// Programmatic dependent launch (PDL).  A kernel launched with the attribute may become resident and run
// its prologue while the previous kernel of the stream is still draining; it must execute
// trl_grid_dep_wait() before it touches anything that kernel wrote.  The previous kernel allows this by
// executing trl_grid_dep_launch() in every CTA (without it the dependent simply starts when it exits).
// Both instructions are no-ops for kernels launched without the attribute.
extern int g_trl_pdl;   // capi.cu; trl_set_pdl()
#ifdef __CUDACC__
__device__ __forceinline__ void trl_grid_dep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void trl_grid_dep_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// cudaLaunchKernelEx with optional PDL and launch priority (0 = stream default).
template <typename... KP, typename... A>
static inline int trl_launch_ex(void (*kernel)(KP...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                                bool pdl, bool high_priority, A... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    cudaLaunchAttribute attr[2];
    unsigned n = 0;
    if (pdl && g_trl_pdl) {
        attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[n].val.programmaticStreamSerializationAllowed = 1;
        ++n;
    }
    if (high_priority) {
        int lo = 0, hi = 0;
        cudaDeviceGetStreamPriorityRange(&lo, &hi);
        attr[n].id = cudaLaunchAttributePriority;
        attr[n].val.priority = hi;
        ++n;
    }
    cfg.attrs = attr; cfg.numAttrs = n;
    return trl_check(cudaLaunchKernelEx(&cfg, kernel, static_cast<KP>(args)...));
}
#endif
