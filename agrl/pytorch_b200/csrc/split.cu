// split.cu -- fp32 rows -> operand planes for the tcgen05 GEMMs in any split format (planes.cuh), plus the TMA
// descriptors.  Rows are B operands (and both operands of the distance GEMM); the E4M3 plane is written in B order.
// The same pass produces what the distance epilogues need: the per-row sum of squares
// (euclidean_squared_distance, distance.py:70-71) or the L2-normalised row x / max(||x||, 1e-12)
// (cosine_distance, distance.py:86-87: F.normalize then mm).
#include "gemm_sm100.cuh"
#include "planes.cuh"

#include <mutex>

namespace agrl {
namespace gemm {

constexpr int kSplitThreads = 256;

// one CTA per row; two passes over the row (the second one hits L1/L2)
__global__ void __launch_bounds__(kSplitThreads)
split_planes_kernel(SplitArgs a) {
    __shared__ float s_part[kSplitThreads / 32], s_maxp[kSplitThreads / 32];
    __shared__ float s_inv, s_ps;
    const int64_t row = blockIdx.x;
    const int tid = threadIdx.x;
    const float *src = a.src + row * a.ld;
    const bool vec = ((reinterpret_cast<uintptr_t>(src) & 15u) == 0) && (a.dim % 4 == 0);
    const bool row_scaled = planes::row_scaled(a.split);

    float inv = 1.0f, ps = 1.0f;
    if (a.sumsq != nullptr || a.normalize || row_scaled) {
        float s = 0.f, m = 0.f;
        if (vec) {
            const float4 *s4 = reinterpret_cast<const float4 *>(src);
            for (int i = tid; i < a.dim / 4; i += kSplitThreads) {
                const float4 v = __ldg(s4 + i);
                s = fmaf(v.x, v.x, s); s = fmaf(v.y, v.y, s); s = fmaf(v.z, v.z, s); s = fmaf(v.w, v.w, s);
                m = fmaxf(fmaxf(m, fmaxf(fabsf(v.x), fabsf(v.y))), fmaxf(fabsf(v.z), fabsf(v.w)));
            }
        } else {
            for (int i = tid; i < a.dim; i += kSplitThreads) { const float v = src[i]; s = fmaf(v, v, s); m = fmaxf(m, fabsf(v)); }
        }
        s = warp_sum(s);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        if ((tid & 31) == 0) { s_part[tid >> 5] = s; s_maxp[tid >> 5] = m; }
        __syncthreads();
        if (tid == 0) {
            float t = 0.f, mx = 0.f;
#pragma unroll
            for (int w = 0; w < kSplitThreads / 32; ++w) { t += s_part[w]; mx = fmaxf(mx, s_maxp[w]); }
            if (a.sumsq) a.sumsq[row] = t;
            const float nrm = fmaxf(sqrtf(t), 1e-12f);       // F.normalize: x / max(||x||_2, eps)
            s_inv = nrm;
            if (row_scaled) planes::f16x2_scales(a.normalize ? __fdiv_rn(mx, nrm) : mx, t, &s_ps, a.unscale + row);
        }
        __syncthreads();
        inv = s_inv;
        if (row_scaled) ps = s_ps;
    }

    const size_t plane_stride = static_cast<size_t>(a.rows) * a.k_pad;
    __nv_bfloat16 *dst = a.planes + row * a.k_pad;
    // pairs of elements -> one 32-bit store per plane
    for (int i = 2 * tid; i < a.k_pad; i += 2 * kSplitThreads) {
        float x[2] = {(i < a.dim) ? src[i] : 0.f, (i + 1 < a.dim) ? src[i + 1] : 0.f};
        if (a.normalize) { x[0] = __fdiv_rn(x[0], inv); x[1] = __fdiv_rn(x[1], inv); }
        uint32_t *w0 = reinterpret_cast<uint32_t *>(dst + i), *w1 = reinterpret_cast<uint32_t *>(dst + plane_stride + i);
        if (row_scaled) {
            uint32_t h[1], l[1];
            planes::encode_f16x2(x, ps, h, l);
            *w0 = h[0]; *w1 = l[0];
        } else if (planes::has_e4m3(a.split)) {
            uint32_t h[1];
            uint16_t res[1], val[1];
            planes::encode_f16_e4m3(x, __ldg(a.prescale), h, res, val);
            *w0 = h[0];
            unsigned char *row8 = reinterpret_cast<unsigned char *>(dst + plane_stride);
            *reinterpret_cast<uint16_t *>(row8 + planes::e4m3_offset(i, true, true)) = res[0];
            *reinterpret_cast<uint16_t *>(row8 + planes::e4m3_offset(i, true, false)) = val[0];
        } else if (planes::scaled(a.split)) {
            uint32_t h[1];
            planes::encode_f16(x, __ldg(a.prescale), h);
            *w0 = h[0];
        } else {
#pragma unroll
            for (int p = 0; p < 3; ++p) {
                if (p < planes::count(a.split)) {
                    uint32_t w[1];
                    planes::bf16_plane(x, w);
                    *reinterpret_cast<uint32_t *>(dst + p * plane_stride + i) = w[0];
                }
            }
        }
    }
}

int launch_split_planes(const SplitArgs &a, cudaStream_t st) {
    if (a.rows <= 0) return AGRL_OK;
    AGRL_LAUNCH_BEGIN(st);
    split_planes_kernel<<<static_cast<unsigned>(a.rows), kSplitThreads, 0, st>>>(a);
    AGRL_LAUNCH_CHECK(st, "split_planes");
    return AGRL_OK;
}

// ---- TMA descriptors ---------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
        else
            (void)cudaGetLastError();
    });
    return fn;
}

int make_plane_tensor_map(CUtensorMap *map, const void *planes, int64_t rows, int64_t k_pad, int P, int box_rows,
                          int64_t plane_rows) {
    EncodeTiledFn fn = encode_tiled_fn();
    if (!fn) return AGRL_E_NO_DEVICE;
    const cuuint64_t dims[3] = {static_cast<cuuint64_t>(k_pad), static_cast<cuuint64_t>(rows), static_cast<cuuint64_t>(P)};
    const cuuint64_t strides[2] = {static_cast<cuuint64_t>(k_pad) * 2, static_cast<cuuint64_t>(plane_rows) * k_pad * 2};
    const cuuint32_t box[3] = {BK, static_cast<cuuint32_t>(box_rows), 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    const CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void *>(planes), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                          CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_cuda_error(cudaErrorInvalidValue, "cuTensorMapEncodeTiled", __FILE__, __LINE__);
        return AGRL_E_CUDA;
    }
    return AGRL_OK;
}

// 3-D tensor map over fp32 node rows (batch, V, C): box = (box_channels <= 256, V rows, 1 tracklet), no swizzle -- one
// bulk tensor copy lands a [V][64] fp32 tile (256-byte rows) of one tracklet in shared memory (graph_kernel_tc, head.cu).
int make_rows_tensor_map_f32(CUtensorMap *map, const float *x, int64_t batch, int V, int C, int box_channels) {
    EncodeTiledFn fn = encode_tiled_fn();
    if (!fn) return AGRL_E_NO_DEVICE;
    const cuuint64_t dims[3] = {static_cast<cuuint64_t>(C), static_cast<cuuint64_t>(V), static_cast<cuuint64_t>(batch)};
    const cuuint64_t strides[2] = {static_cast<cuuint64_t>(C) * 4, static_cast<cuuint64_t>(V) * C * 4};
    const cuuint32_t box[3] = {static_cast<cuuint32_t>(box_channels), static_cast<cuuint32_t>(V), 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    const CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float *>(x), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                          CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_cuda_error(cudaErrorInvalidValue, "cuTensorMapEncodeTiled", __FILE__, __LINE__);
        return AGRL_E_CUDA;
    }
    return AGRL_OK;
}

}  // namespace gemm
}  // namespace agrl
