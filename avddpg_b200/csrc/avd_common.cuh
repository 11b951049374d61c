// avd_common.cuh -- error plumbing and launch helpers shared by the C-ABI translation units.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/avddpg_b200.h"

namespace avd {

void set_error(const char* fmt, ...);           // defined in avd_lib.cu
void count_launch(int n = 1);                    // kernels launched by this library so far (avd_kernel_launches)
int sm_count();                                  // cached multiprocessor count of the current device

#define AVD_REQUIRE(cond, ...)                    \
    do {                                          \
        if (!(cond)) {                            \
            ::avd::set_error(__VA_ARGS__);        \
            return AVD_ERR_INVALID_ARG;           \
        }                                         \
    } while (0)

#define AVD_CUDA_OK(expr)                                                                   \
    do {                                                                                    \
        cudaError_t _e = (expr);                                                            \
        if (_e != cudaSuccess) {                                                            \
            ::avd::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            return AVD_ERR_CUDA;                                                            \
        }                                                                                   \
    } while (0)

// A run table must cover the batch exactly: the kernels index runs->seed with p / platoons_per_run for every platoon p < P.
#define AVD_REQUIRE_RUNS(r, P)                                                                                               \
    AVD_REQUIRE((r)->seed && (r)->runs >= 1 && (r)->platoons_per_run >= 1 && (int64_t)(r)->runs * (r)->platoons_per_run == (P), \
                "run table of %d runs x %lld platoons (seed %p) does not cover the batch of %lld platoons", (int)(r)->runs,  \
                (long long)(r)->platoons_per_run, (const void*)(r)->seed, (long long)(P))

#define AVD_LAUNCH_OK()                                                                     \
    do {                                                                                    \
        ::avd::count_launch();                                                              \
        cudaError_t _e = cudaGetLastError();                                                \
        if (_e != cudaSuccess) {                                                            \
            ::avd::set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e), __FILE__, __LINE__); \
            return AVD_ERR_CUDA;                                                            \
        }                                                                                   \
    } while (0)

// Programmatic dependent launch (PDL).  A kernel launched through launch_pdl() may become resident while the previous
// kernel of the stream is still running -- SM by SM, as that kernel's CTAs exit -- and run its prologue (barrier init, TMEM
// allocation, weight tables) there; it must execute pdl_wait() before it touches anything an earlier kernel wrote, and calls
// pdl_launch_dependents() to allow the same for its successor.  AVD_PDL=0 in the environment restores plain launches.
bool pdl_enabled();                              // defined in avd_lib.cu
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}
#endif

// Persistent-style grid: enough 256-thread CTAs to fill every SM to 2048 threads, never more than
// the work needs (B200: 148 SMs x 8 CTAs).
inline int grid_for(int64_t work_items, int threads = 256, int ctas_per_sm = 8) {
    int64_t need = (work_items + threads - 1) / threads;
    int64_t cap = (int64_t)sm_count() * ctas_per_sm;
    if (need < 1) need = 1;
    return (int)(need < cap ? need : cap);
}

// Grid for a grid-stride kernel: exactly the number of CTAs that are co-resident (SMs x occupancy), so
// there is a single wave and no tail, capped by the work available.
template <class Kernel>
inline int resident_grid(Kernel kernel, int64_t work_items, int threads = 256, size_t smem = 0) {
    int occ = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, threads, smem) != cudaSuccess || occ < 1) {
        cudaGetLastError();
        occ = 1;
    }
    int64_t need = (work_items + threads - 1) / threads;
    int64_t cap = (int64_t)sm_count() * occ;
    if (need < 1) need = 1;
    return (int)(need < cap ? need : cap);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

}  // namespace avd
