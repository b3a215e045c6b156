// planes.cuh -- the operand formats of the tcgen05 GEMMs (DESIGN.md section 2), defined once.
//
// Every GEMM of the library reads its operands as planes [P][rows][K] of 16-bit values (the fp16 + E4M3 mode's second
// plane holds E4M3 bytes instead).  For every AGRL_SPLIT_* mode this header decides how many planes there are, which power
// of two scales an fp32 value first, how the value becomes the bytes of each plane and where those bytes go:
//   BF16X2 / BF16X3  x = p0 + p1 (+ p2), each plane the bf16 of what the planes before it left (exact residuals in fp32,
//                    so three planes carry all 24 significand bits)
//   FP16X1           ONE plane fp16(x s), s = 2^k per tensor (f16_scales)
//   FP16_E4M3        plane 0 fp16(x s); plane 1, per 64-element k-block, 64 residuals e4m3((x s - h) 2^6) and 64 value
//                    copies e4m3(x s 2^-6) -- residuals first in the A operand, value copies first in the B operand
//                    (e4m3_offset), so that ONE K-concatenated 8-bit product gives r_a.b + a.r_b
//   FP16X2           h = fp16(x s), l = fp16((x s - h) 2^11), s = 2^k per row (f16x2_scales)
// The encoders take N values (an even count) and return 32-bit words of the 16-bit planes (value 2i in the low half of
// word i) and 16-bit words of the E4M3 plane (value 2i in the low byte).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_fp8.h>

#include "common.cuh"

namespace agrl {
namespace planes {

// ---- mode facts --------------------------------------------------------------------------------
constexpr int count(int split) { return split == AGRL_SPLIT_FP16_E4M3 || split == AGRL_SPLIT_FP16X2 ? 2 : split; }
constexpr bool scaled(int split) { return split == AGRL_SPLIT_FP16X1 || split == AGRL_SPLIT_FP16_E4M3; }   // 2^k per tensor
constexpr bool has_e4m3(int split) { return split == AGRL_SPLIT_FP16_E4M3; }
constexpr bool row_scaled(int split) { return split == AGRL_SPLIT_FP16X2; }                                // 2^k per row
constexpr bool head_ok(int split) {
    return split == AGRL_SPLIT_BF16X2 || split == AGRL_SPLIT_BF16X3 || split == AGRL_SPLIT_FP16X1 || split == AGRL_SPLIT_FP16_E4M3;
}
constexpr bool distance_ok(int split) {
    return split == AGRL_SPLIT_BF16X2 || split == AGRL_SPLIT_BF16X3 || split == AGRL_SPLIT_FP16X2;
}
// column tile of the graph-layer GEMM: three bf16 planes leave room for 128 columns only
constexpr int head_bn(int split) { return split == AGRL_SPLIT_BF16X3 ? 128 : 256; }

// compile-time tag of a mode: the GEMM's plane count, the head GEMM's tile width, the epilogue's flags
template <int kSplit>
struct Mode {
    static constexpr int kP = count(kSplit);
    static constexpr int kHeadBN = head_bn(kSplit);
    static constexpr bool kScaled = scaled(kSplit);
    static constexpr bool kFp8 = has_e4m3(kSplit);
    static constexpr bool kRowScaled = row_scaled(kSplit);
};

// f(Mode<split>{}) for a split that head_ok / distance_ok has accepted
template <class F>
auto with_head_mode(int split, F &&f) {
    switch (split) {
        case AGRL_SPLIT_FP16X1: return f(Mode<AGRL_SPLIT_FP16X1>{});
        case AGRL_SPLIT_FP16_E4M3: return f(Mode<AGRL_SPLIT_FP16_E4M3>{});
        case AGRL_SPLIT_BF16X3: return f(Mode<AGRL_SPLIT_BF16X3>{});
        default: return f(Mode<AGRL_SPLIT_BF16X2>{});
    }
}
template <class F>
auto with_distance_mode(int split, F &&f) {
    switch (split) {
        case AGRL_SPLIT_FP16X2: return f(Mode<AGRL_SPLIT_FP16X2>{});
        case AGRL_SPLIT_BF16X3: return f(Mode<AGRL_SPLIT_BF16X3>{});
        default: return f(Mode<AGRL_SPLIT_BF16X2>{});
    }
}

// byte offset of element k's E4M3 residual (or value copy) in its row of the 8-bit plane
__host__ __device__ constexpr int e4m3_offset(int k, bool b_operand, bool residual) {
    return (k >> 6) * 128 + (k & 63) + (residual == b_operand ? 64 : 0);
}

#ifdef __CUDACC__
// ---- power-of-two scales -----------------------------------------------------------------------
// FP16X1 / FP16_E4M3: the power of two that puts `bound` (max |x| of the tensor) in [2^13, 2^14) -- fp16 keeps 11
// significant bits only between 2^-14 and 2^15 -- and its inverse for the epilogue.  bound 0: 2^0.
__device__ __forceinline__ void f16_scales(float bound, float *up, float *down) {
    int e = 0;
    if (bound > 0.f) frexpf(bound, &e);                // bound = m * 2^e, m in [0.5, 1)
    else e = 14;
    e = max(-100, min(100, e));
    *up = ldexpf(1.0f, 14 - e);
    *down = ldexpf(1.0f, e - 14);
}

// FP16X2: the power of two that puts the row's largest magnitude `mx` in [2^7, 2^8), and its inverse.  Rows that are all
// zero, or hold Inf / NaN (`sumsq`, the row's sum of squares, is NaN then or mx is), stay unscaled.
__device__ __forceinline__ void f16x2_scales(float mx, float sumsq, float *up, float *down) {
    int e = 7;
    if (mx > 0.f && mx < 3.0e38f && sumsq == sumsq) e = ilogbf(mx);
    e = max(-110, min(120, e));
    *up = ldexpf(1.0f, 7 - e);
    *down = ldexpf(1.0f, e - 7);
}

// ---- encoders ----------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t bits(__half2 h) { return *reinterpret_cast<const uint32_t *>(&h); }
__device__ __forceinline__ float2 f16_values(uint32_t w) { return __half22float2(*reinterpret_cast<const __half2 *>(&w)); }
__device__ __forceinline__ uint16_t e4m3x2(float lo, float hi) {
    return __nv_cvt_float2_to_fp8x2(make_float2(lo, hi), __NV_SATFINITE, __NV_E4M3);
}

// one bf16 plane of the residual chain: r -> its bf16 words, and r - bf16(r) (exact) left in r for the next plane
template <int N>
__device__ __forceinline__ void bf16_plane(float (&r)[N], uint32_t (&w)[N / 2]) {
#pragma unroll
    for (int i = 0; i < N / 2; ++i) {
        const __nv_bfloat162 b = __floats2bfloat162_rn(r[2 * i], r[2 * i + 1]);
        w[i] = *reinterpret_cast<const uint32_t *>(&b);
        r[2 * i] = __fsub_rn(r[2 * i], __uint_as_float(w[i] << 16));
        r[2 * i + 1] = __fsub_rn(r[2 * i + 1], __uint_as_float(w[i] & 0xffff0000u));
    }
}

// BF16X2 / BF16X3: all P planes
template <int P, int N>
__device__ __forceinline__ void encode_bf16(const float (&v)[N], uint32_t (&w)[P][N / 2]) {
    float r[N];
#pragma unroll
    for (int i = 0; i < N; ++i) r[i] = v[i];
#pragma unroll
    for (int p = 0; p < P; ++p) bf16_plane(r, w[p]);
}

// FP16X1: fp16(v s)
template <int N>
__device__ __forceinline__ void encode_f16(const float (&v)[N], float s, uint32_t (&h)[N / 2]) {
#pragma unroll
    for (int i = 0; i < N / 2; ++i) h[i] = bits(__floats2half2_rn(v[2 * i] * s, v[2 * i + 1] * s));
}

// FP16_E4M3: h = fp16(v s), the residuals e4m3((v s - h) 2^6) and the value copies e4m3(v s 2^-6).  The residual is ONE
// fma: v s - h is exact in fp32 and 64 a power of two, so fma(v s, 64, -64 h) is the same number as (v s - h) 64.
template <int N>
__device__ __forceinline__ void encode_f16_e4m3(const float (&v)[N], float s, uint32_t (&h)[N / 2], uint16_t (&res)[N / 2],
                                                uint16_t (&val)[N / 2]) {
#pragma unroll
    for (int i = 0; i < N / 2; ++i) {
        const float x0 = v[2 * i] * s, x1 = v[2 * i + 1] * s;
        h[i] = bits(__floats2half2_rn(x0, x1));
        const float2 hf = f16_values(h[i]);
        res[i] = e4m3x2(fmaf(x0, 64.0f, -64.0f * hf.x), fmaf(x1, 64.0f, -64.0f * hf.y));
        val[i] = e4m3x2(x0 * 0.015625f, x1 * 0.015625f);
    }
}

// FP16X2: h = fp16(v s), l = fp16((v s - h) 2^11) -- v s - h is exact in fp32, 2^11 lifts it into fp16's normal range
template <int N>
__device__ __forceinline__ void encode_f16x2(const float (&v)[N], float s, uint32_t (&h)[N / 2], uint32_t (&l)[N / 2]) {
#pragma unroll
    for (int i = 0; i < N / 2; ++i) {
        const float x0 = v[2 * i] * s, x1 = v[2 * i + 1] * s;
        h[i] = bits(__floats2half2_rn(x0, x1));
        const float2 hf = f16_values(h[i]);
        l[i] = bits(__floats2half2_rn(__fsub_rn(x0, hf.x) * 2048.0f, __fsub_rn(x1, hf.y) * 2048.0f));
    }
}
#endif

}  // namespace planes
}  // namespace agrl
