// common.cuh -- shared helpers for libagrl_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../../include/agrl_b200.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libagrl_b200 is written for sm_100a only (compile with -gencode arch=compute_100a,code=sm_100a)"
#endif

namespace agrl {

// ---- host-side error plumbing --------------------------------------------------------------
void        set_cuda_error(cudaError_t e, const char *what, const char *file, int line);
void        after_launch(cudaStream_t st, const char *name);   // counts; records a profiling event when enabled
// Optional: marks the start of the next launch on `st` (profiling only).  Launch sites that run kernels of
// one call on several streams use it so that a kernel's time is begin->end on ITS stream; without it the
// kernel is timed from the previous event (consecutive launches on one busy stream).
void        before_launch(cudaStream_t st);

#define AGRL_CUDA_TRY(expr)                                                            \
    do {                                                                               \
        cudaError_t _e = (expr);                                                       \
        if (_e != cudaSuccess) {                                                       \
            ::agrl::set_cuda_error(_e, #expr, __FILE__, __LINE__);                     \
            return AGRL_E_CUDA;                                                        \
        }                                                                              \
    } while (0)

// check the launch that just happened (configuration errors surface here without a sync)
#define AGRL_LAUNCH_BEGIN(stream) ::agrl::before_launch(stream)
#define AGRL_LAUNCH_CHECK(stream, name)                                                \
    do {                                                                               \
        AGRL_CUDA_TRY(cudaGetLastError());                                             \
        ::agrl::after_launch(stream, name);                                            \
    } while (0)

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// carve sub-buffers out of a caller-provided workspace
struct Carver {
    char  *base;
    size_t off;
    explicit Carver(void *p) : base(static_cast<char *>(p)), off(0) {}
    template <class T> T *take(size_t n) {
        off = align_up(off, 256);
        T *r = reinterpret_cast<T *>(base ? base + off : nullptr);
        off += n * sizeof(T);
        return r;
    }
    size_t total() const { return align_up(off, 256); }
};

// ---- device helpers -------------------------------------------------------------------------
#ifdef __CUDACC__
constexpr int kNumSMs = 148;

// Monotone map float -> uint32 so that unsigned order == numpy's sort order:
// -inf < ... < -0 == +0 < ... < +inf < NaN (all NaNs equal; ties are then broken by index).
__device__ __forceinline__ uint32_t mono_key(float d) {
    if (d != d) return 0xFFFFFFFFu;
    uint32_t u = __float_as_uint(d + 0.0f);          // -0.0f + 0.0f == +0.0f
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
// Inverse of mono_key: the bits of the distance that was ranked.  A -0 was ranked as +0 and comes back as +0; every NaN
// was ranked as 0xFFFFFFFF and comes back as the NaN 0x7FFFFFFF.
__device__ __forceinline__ float mono_key_value(uint32_t k) {
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7FFFFFFFu) : ~k);
}
__device__ __forceinline__ uint64_t rank_key(float d, uint32_t idx) {
    return (static_cast<uint64_t>(mono_key(d)) << 32) | idx;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ int warp_sum(int v) { return __reduce_add_sync(0xffffffffu, v); }
#endif

}  // namespace agrl
