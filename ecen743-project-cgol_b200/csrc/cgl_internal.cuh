// cgl_internal.cuh -- helpers shared by the translation units of libcgl_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/cgl_b200.h"
#include "cgl_bits.cuh"

namespace cgl {

void set_error(const char *fmt, ...);
int sm_count();

#define CGL_REQUIRE(cond, code, ...)            \
    do {                                        \
        if (!(cond)) {                          \
            cgl::set_error(__VA_ARGS__);        \
            return (code);                      \
        }                                       \
    } while (0)

#define CGL_CUDA(expr)                                                                       \
    do {                                                                                     \
        cudaError_t _e = (expr);                                                             \
        if (_e != cudaSuccess) {                                                             \
            cgl::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, \
                           __LINE__);                                                        \
            return (int)_e;                                                                  \
        }                                                                                    \
    } while (0)

#define CGL_LAUNCH_CHECK()                                                                  \
    do {                                                                                    \
        cudaError_t _e = cudaGetLastError();                                                \
        if (_e != cudaSuccess) {                                                            \
            cgl::set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e),      \
                           __FILE__, __LINE__);                                             \
            return (int)_e;                                                                 \
        }                                                                                   \
    } while (0)

// Kernel attributes (cudaFuncSetAttribute) belong to the device that is current when they are set: a
// process that drives several GPUs has to configure each of them once.
struct PerDeviceOnce {
    bool done[64] = {};
    bool first()
    {
        int d = 0;
        if (cudaGetDevice(&d) != cudaSuccess || d < 0 || d >= 64) return true;
        if (done[d]) return false;
        done[d] = true;
        return true;
    }
};

static inline cudaStream_t as_stream(cgl_stream_t s) { return (cudaStream_t)s; }

// grid size for a grid-stride kernel over `n` items with `threads` per block:
// enough blocks to cover n once, capped at a multiple of the SM count (148 on B200).
static inline unsigned grid_for(uint64_t n, unsigned threads, unsigned blocks_per_sm = 16)
{
    uint64_t need = (n + threads - 1) / threads;
    uint64_t cap = (uint64_t)sm_count() * blocks_per_sm;
    if (need < 1) need = 1;
    return (unsigned)(need < cap ? need : cap);
}

// Alarm words (host-mapped int[CGL_ALARM_WORDS], owned by cgl_api.cu): a kernel that gives up on a wait or sees an
// invalid action stores 1 into its word, which the host can read at any time WITHOUT synchronising.
enum { ALARM_BAD_ACTION = 0, ALARM_ENV_TOKEN = 1, ALARM_LIFE_TOKEN = 2, ALARM_HALO = 3 };

// Every translation unit that waits on device-side tokens gets its own copy of the two symbols below (the
// library is built without relocatable device code) and registers a setter with CGL_DEFINE_TU_HOOKS; cgl_api.cu
// calls all setters for the current device (cgl_alarm_words, cgl_set_wait_timeout_ms).
int set_hooks_env(int *alarm_dev, unsigned long long wait_ns);
int set_hooks_life_tb(int *alarm_dev, unsigned long long wait_ns);
int set_hooks_api(int *alarm_dev, unsigned long long wait_ns);

#if defined(__CUDACC__)
__device__ __forceinline__ uint32_t ld_nc_u32(const uint32_t *p) { return __ldg(p); }

static __device__ int *g_alarm = nullptr;                            // device pointer of the host-mapped alarm words
static __device__ unsigned long long g_wait_ns = 2000000000ull;     // how long a device-side wait may last

#define CGL_DEFINE_TU_HOOKS(name)                                                                   \
    int set_hooks_##name(int *alarm_dev, unsigned long long wait_ns)                                \
    {                                                                                               \
        CGL_CUDA(cudaMemcpyToSymbol(g_alarm, &alarm_dev, sizeof(alarm_dev)));                       \
        CGL_CUDA(cudaMemcpyToSymbol(g_wait_ns, &wait_ns, sizeof(wait_ns)));                         \
        return 0;                                                                                   \
    }

__device__ __forceinline__ unsigned long long globaltimer_ns()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

__device__ __forceinline__ void raise_alarm(int word)
{
    int *a = g_alarm;
    if (a != nullptr) {
        *reinterpret_cast<volatile int *>(a + word) = 1;
        __threadfence_system();
    }
}

// Slow path of every bounded device-side wait: called every few hundred failed polls.  True = give up (the
// deadline passed, or another waiter already raised the same alarm: fail fast instead of one timeout per launch).
__device__ __forceinline__ bool wait_expired(unsigned long long t0, int word)
{
    if (globaltimer_ns() - t0 > g_wait_ns) return true;
    const int *a = g_alarm;
    return a != nullptr && *reinterpret_cast<const volatile int *>(a + word) != 0;
}
#endif

}  // namespace cgl
