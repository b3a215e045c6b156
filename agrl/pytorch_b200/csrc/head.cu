// head.cu -- the VMGN adaptive graph head, eval mode (torchreid/models/vmgn.py:296-321).
//
// Per batch of B tracklets (S frames, P = 7 pyramid strips, V = S*P region nodes, C channels):
//
//   pool_tma_kernel    one pass over both layer4 maps (the only HBM-heavy step, 2 x S*C*h*w*4 B per tracklet, half that
//                      for the bf16 / fp16 maps of an autocast backbone, read as they are and summed in fp32): strip
//                      means -> node tensor X0 (B,V,C) written directly in node order (vmgn.py:304-308, no cat / transpose
//                      copies, x4_2 read once instead of three times) and the global mean -> BN neck -> out[:, :C]
//                      (vmgn.py:299-301).  Persistent CTAs, loads kept in flight in a shared-memory ring by cp.async.bulk;
//                      runs at the measured HBM copy peak.  pool_kernel (register loads) covers maps that are not 16x8 or
//                      unaligned, pool_nhwc_kernel channels-last maps.
//   graph_kernel_tc    one CTA per tracklet: Gram matrix of the centred nodes and the message passing Y = G.X (vmgn.py:168,
//                      re-associated as (G.X).W^T) as tcgen05 MMAs on operands the CTA converts itself in shared memory;
//                      affinity 2/(exp(d)+1) (vmgn.py:114-120), L1 row normalisation of affinity and pose graph (:157,:162),
//                      average (:164) on CUDA cores in between.  Y leaves as operand planes for the GEMM.  First layer:
//                      the nodes of a frame are T.(its four quarter strips), so G.X.W^T = (G.T).(Q.W^T): the kernel stops
//                      after the graph, emits G.T and the planes of the 4S quarter rows; graph_mix_kernel applies G.T and
//                      the layer's element-wise part after the GEMM.
//   split_gemm_kernel  (gemm_sm100.cuh) Y.W^T on tcgen05 with the layer's epilogue fused:
//                      0.9*X + 0.1*LeakyReLU(BN(.)) (vmgn.py:169-172).
//   attn_kernel        temporal attention (vmgn.py:276-277), part mean, BN neck -> out[:, C:] (:317-321).
//   clip_pool_kernel   mean / max over the clips of a tracklet (train_vidreid_xent_htri.py:471-476).
#include "gemm_sm100.cuh"

#include <cuda_fp16.h>
#include <cuda_fp8.h>

namespace agrl {

constexpr int kParts = 7;              // calc_splits(4) = [4,2,1] (utils/reidtools.py:13-15)
constexpr int kMaxNodes = 64;
constexpr int kHeadThreads = 256;

// operand planes of a GEMM mode: bf16 x2 / x3, ONE scaled fp16 plane, or the fp16 plane + one plane of E4M3 pairs
static inline int planes_of(int split) { return split == AGRL_SPLIT_FP16_E4M3 ? 2 : split; }
static inline bool scaled_mode(int split) { return split == AGRL_SPLIT_FP16X1 || split == AGRL_SPLIT_FP16_E4M3; }

// ------------------------------------------------------------------------------------------------
// weight preparation: folded BN vectors
// ------------------------------------------------------------------------------------------------
struct FoldArgs {
    const float *w[AGRL_HEAD_MAX_LAYERS + 2], *b[AGRL_HEAD_MAX_LAYERS + 2];
    const float *mean[AGRL_HEAD_MAX_LAYERS + 2], *var[AGRL_HEAD_MAX_LAYERS + 2];
    float *scale[AGRL_HEAD_MAX_LAYERS + 2], *shift[AGRL_HEAD_MAX_LAYERS + 2];
    int channels;
    float eps;
};

__global__ void fold_bn_kernel(FoldArgs a) {
    const int which = blockIdx.y;
    for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < a.channels; c += gridDim.x * blockDim.x) {
        const float s = __fdiv_rn(a.w[which][c], sqrtf(a.var[which][c] + a.eps));
        a.scale[which][c] = s;
        a.shift[which][c] = fmaf(-a.mean[which][c], s, a.b[which][c]);
    }
}

// fp16 mode: W is multiplied by the power of two that puts max|W| just below 2^14 before it is rounded to fp16
// (fp16 keeps 11 significant bits only between 2^-14 and 2^15), and the GEMM epilogue multiplies by its inverse.
__global__ void absmax_kernel(const float *__restrict__ w, size_t n, float *slot) {
    float m = 0.f;
    for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n; i += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const float v = fabsf(w[i]);
        if (v < 3.0e38f) m = fmaxf(m, v);              // ignore inf / NaN
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<unsigned int *>(slot + 2), __float_as_uint(m));
}
__device__ __forceinline__ void pow2_scales(float bound, float *up, float *down) {
    int e = 0;
    if (bound > 0.f) frexpf(bound, &e);                // bound = m * 2^e, m in [0.5, 1)
    else e = 14;
    e = max(-100, min(100, e));
    *up = ldexpf(1.0f, 14 - e);
    *down = ldexpf(1.0f, e - 14);
}
__global__ void w_scale_kernel(float *slot) { pow2_scales(slot[2], slot, slot + 1); }

struct Prepared {                       // layout of the caller-owned "prepared" buffer
    __nv_bfloat16 *w_planes[AGRL_HEAD_MAX_LAYERS];     // [P][C][C]
    float *scale[AGRL_HEAD_MAX_LAYERS + 2], *shift[AGRL_HEAD_MAX_LAYERS + 2];   // layers.., global, att
    float *w_scale;                                    // fp16 mode: per layer {2^k, 2^-k, max|W| bits}
    size_t bytes;
};

static Prepared carve_prepared(const agrl_head_params *p, void *buf) {
    Carver c(buf);
    Prepared r;
    const size_t C = static_cast<size_t>(p->channels);
    for (int l = 0; l < p->num_layers; ++l) r.w_planes[l] = c.take<__nv_bfloat16>(planes_of(p->split) * C * C);
    for (int l = 0; l < p->num_layers + 2; ++l) { r.scale[l] = c.take<float>(C); r.shift[l] = c.take<float>(C); }
    r.w_scale = c.take<float>(4 * AGRL_HEAD_MAX_LAYERS);
    r.bytes = c.total();
    return r;
}

// ------------------------------------------------------------------------------------------------
// element types of the layer4 maps (agrl_head_params.maps_dtype): fp32, or the bf16 / fp16 maps an autocast backbone
// returns.  Every pooling kernel converts on load (exact: both 16-bit formats, inf and NaN included, are subsets of fp32)
// and then sums exactly as it does for fp32, so 16-bit maps give the bits that their .float() copy gives.
// Vec4 is four consecutive elements: one 16-byte load at fp32, one 8-byte load at 16 bits.
// ------------------------------------------------------------------------------------------------
template <class T> struct MapElem;
template <> struct MapElem<float> {
    using Vec4 = float4;
    static __device__ __forceinline__ float cvt(float v) { return v; }
    static __device__ __forceinline__ float4 cvt4(const float4 &v) { return v; }
};
template <> struct MapElem<__nv_bfloat16> {
    using Vec4 = uint2;
    static __device__ __forceinline__ float cvt(__nv_bfloat16 v) { return __bfloat162float(v); }
    static __device__ __forceinline__ float4 cvt4(const uint2 &v) {
        const float2 lo = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162 *>(&v.x));
        const float2 hi = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162 *>(&v.y));
        return make_float4(lo.x, lo.y, hi.x, hi.y);
    }
};
template <> struct MapElem<__half> {
    using Vec4 = uint2;
    static __device__ __forceinline__ float cvt(__half v) { return __half2float(v); }
    static __device__ __forceinline__ float4 cvt4(const uint2 &v) {
        const float2 lo = __half22float2(*reinterpret_cast<const __half2 *>(&v.x));
        const float2 hi = __half22float2(*reinterpret_cast<const __half2 *>(&v.y));
        return make_float4(lo.x, lo.y, hi.x, hi.y);
    }
};

// ------------------------------------------------------------------------------------------------
// pooling: grid (C/64, B), 8 warps x 8 channels, loop over the S frames
// ------------------------------------------------------------------------------------------------
template <class T>
struct PoolArgs {
    const T *x41, *x42;                // (B*S, C, hw)
    float *nodes;                      // (B, V, C)
    float *out; int64_t ld_out;        // (B, 2C): global branch -> [:, :C]
    const float *g_scale, *g_shift;    // folded global_bottleneck
    int S, C, hw;
};

constexpr int kPoolCh = 64;            // channels per CTA

template <bool kVec, class T>
__global__ void __launch_bounds__(kHeadThreads)
pool_kernel(PoolArgs<T> a) {
    using E = MapElem<T>;
    using Vec4 = typename E::Vec4;
    extern __shared__ float s_nodes[];                 // [S][7][kPoolCh]
    const int b = blockIdx.y, c0 = blockIdx.x * kPoolCh;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int grp = lane >> 3, sub = lane & 7;         // 8-lane group <-> quarter strip
    const int hw = a.hw, qlen = hw >> 2;
    const float inv_q = 1.0f / static_cast<float>(qlen), inv_h = 1.0f / static_cast<float>(2 * qlen);
    const float inv_w = 1.0f / static_cast<float>(hw);

    float gsum[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) gsum[i] = 0.f;

    for (int s = 0; s < a.S; ++s) {
        const size_t frame = (static_cast<size_t>(b) * a.S + s) * a.C;
        float q1[8], q2[8];
        if (kVec) {
            // hw == 128: four elements per lane cover a (frame, channel) plane; 16 loads in flight per lane
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const size_t off = (frame + c0 + warp * 8 + i) * hw + lane * 4;
                const float4 v1 = E::cvt4(__ldcs(reinterpret_cast<const Vec4 *>(a.x41 + off)));
                const float4 v2 = E::cvt4(__ldcs(reinterpret_cast<const Vec4 *>(a.x42 + off)));
                q1[i] = (v1.x + v1.y) + (v1.z + v1.w);
                q2[i] = (v2.x + v2.y) + (v2.z + v2.w);
            }
        } else {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const size_t off = (frame + c0 + warp * 8 + i) * hw + grp * qlen;
                float s1 = 0.f, s2 = 0.f;
                for (int e = sub; e < qlen; e += 8) { s1 += E::cvt(a.x41[off + e]); s2 += E::cvt(a.x42[off + e]); }
                q1[i] = s1; q2[i] = s2;
            }
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            float v1 = q1[i], v2 = q2[i];
            // quarter sums: reduce inside each 8-lane group
            v1 += __shfl_xor_sync(0xffffffffu, v1, 4); v2 += __shfl_xor_sync(0xffffffffu, v2, 4);
            v1 += __shfl_xor_sync(0xffffffffu, v1, 2); v2 += __shfl_xor_sync(0xffffffffu, v2, 2);
            v1 += __shfl_xor_sync(0xffffffffu, v1, 1); v2 += __shfl_xor_sync(0xffffffffu, v2, 1);
            const float h2 = v2 + __shfl_xor_sync(0xffffffffu, v2, 8);       // half strips
            const float w2 = h2 + __shfl_xor_sync(0xffffffffu, h2, 16);      // whole map
            v1 += __shfl_xor_sync(0xffffffffu, v1, 8);
            v1 += __shfl_xor_sync(0xffffffffu, v1, 16);
            gsum[i] += v1;
            float *dst = s_nodes + (s * kParts) * kPoolCh + warp * 8 + i;
            if (sub == 0) dst[grp * kPoolCh] = v2 * inv_q;                   // parts 0..3
            if (lane == 0) { dst[4 * kPoolCh] = h2 * inv_h; dst[6 * kPoolCh] = w2 * inv_w; }
            if (lane == 16) dst[5 * kPoolCh] = h2 * inv_h;
        }
    }
    // global branch: mean over (S, h, w), BN neck
    if (lane == 0) {
        const float inv_all = 1.0f / (static_cast<float>(a.S) * static_cast<float>(hw));
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int c = c0 + warp * 8 + i;
            a.out[static_cast<size_t>(b) * a.ld_out + c] = fmaf(gsum[i] * inv_all, a.g_scale[c], a.g_shift[c]);
        }
    }
    __syncthreads();
    // node rows: V rows of kPoolCh contiguous floats
    const int V = a.S * kParts;
    float *nodes = a.nodes + static_cast<size_t>(b) * V * a.C + c0;
    for (int i = threadIdx.x; i < V * kPoolCh; i += kHeadThreads) {
        const int v = i / kPoolCh, c = i % kPoolCh;
        nodes[static_cast<size_t>(v) * a.C + c] = s_nodes[i];
    }
}

// ------------------------------------------------------------------------------------------------
// pooling, channels-last maps (SURVEY.md section 8f row 4, the part that stays on our side of the cuDNN boundary):
// a backbone run in torch.channels_last hands over (B*S, h, w, C)-ordered memory; converting it back to NCHW would
// cost a second pass over the 16 MiB per tracklet.  Here a thread owns 4 consecutive channels (one 16-byte load per
// pixel at fp32, 8 bytes at 16 bits, fully coalesced across the CTA), keeps the four quarter-strip sums in registers and
// writes node rows straight from them.  grid (C / 1024, B), 256 threads.  Needs maps aligned to 4 elements.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void add4(float4 &a, const float4 &b) { a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w; }
__device__ __forceinline__ float4 scale4(const float4 &a, float s) { return make_float4(a.x * s, a.y * s, a.z * s, a.w * s); }

template <class T>
__global__ void __launch_bounds__(kHeadThreads)
pool_nhwc_kernel(PoolArgs<T> a) {
    using E = MapElem<T>;
    using Vec4 = typename E::Vec4;
    const int b = blockIdx.y;
    const int c = (blockIdx.x * kHeadThreads + threadIdx.x) * 4;
    if (c >= a.C) return;
    const int hw = a.hw, qlen = hw >> 2, V = a.S * kParts;
    const float inv_q = 1.0f / static_cast<float>(qlen), inv_h = 1.0f / static_cast<float>(2 * qlen);
    const float inv_w = 1.0f / static_cast<float>(hw);
    float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
    float *nodes = a.nodes + static_cast<size_t>(b) * V * a.C + c;
    for (int s = 0; s < a.S; ++s) {
        const size_t frame = (static_cast<size_t>(b) * a.S + s) * hw * a.C + c;
        float4 q[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            float4 s1 = make_float4(0.f, 0.f, 0.f, 0.f), s2 = s1;
            const size_t base = frame + static_cast<size_t>(k) * qlen * a.C;
#pragma unroll 8
            for (int p = 0; p < qlen; ++p) {
                add4(s1, E::cvt4(__ldcs(reinterpret_cast<const Vec4 *>(a.x41 + base + static_cast<size_t>(p) * a.C))));
                add4(s2, E::cvt4(__ldcs(reinterpret_cast<const Vec4 *>(a.x42 + base + static_cast<size_t>(p) * a.C))));
            }
            add4(g, s1);
            q[k] = s2;
        }
        float4 h0 = q[0], h1 = q[2];
        add4(h0, q[1]); add4(h1, q[3]);
        float4 w = h0;
        add4(w, h1);
        float *row = nodes + static_cast<size_t>(s) * kParts * a.C;
#pragma unroll
        for (int k = 0; k < 4; ++k) *reinterpret_cast<float4 *>(row + static_cast<size_t>(k) * a.C) = scale4(q[k], inv_q);
        *reinterpret_cast<float4 *>(row + 4 * static_cast<size_t>(a.C)) = scale4(h0, inv_h);
        *reinterpret_cast<float4 *>(row + 5 * static_cast<size_t>(a.C)) = scale4(h1, inv_h);
        *reinterpret_cast<float4 *>(row + 6 * static_cast<size_t>(a.C)) = scale4(w, inv_w);
    }
    const float inv_all = 1.0f / (static_cast<float>(a.S) * static_cast<float>(hw));
    const float4 sc = *reinterpret_cast<const float4 *>(a.g_scale + c), sh = *reinterpret_cast<const float4 *>(a.g_shift + c);
    float4 o;
    o.x = fmaf(g.x * inv_all, sc.x, sh.x); o.y = fmaf(g.y * inv_all, sc.y, sh.y);
    o.z = fmaf(g.z * inv_all, sc.z, sh.z); o.w = fmaf(g.w * inv_all, sc.w, sh.w);
    float *dst = a.out + static_cast<size_t>(b) * a.ld_out + c;
    dst[0] = o.x; dst[1] = o.y; dst[2] = o.z; dst[3] = o.w;      // ld_out need not be a multiple of 4
}

// ------------------------------------------------------------------------------------------------
// pooling, bulk-copy (TMA) flavour: a persistent, deliberately small CTA (1 producer + 4 consumer
// warps, < 64 registers, two per SM) that keeps its loads in flight in a shared-memory ring instead of in
// registers.
//   work unit   (tracklet b, 32-channel chunk): 2*S ring stages, each one frame of one map (32 channels x
//               128 elements are contiguous in NCHW: 16 KiB at fp32, 8 KiB at 16 bits), fetched with one
//               cp.async.bulk (L2 evict-first) that completes on the stage's mbarrier
//   consumers   warp w owns channels 8w..8w+7 of the chunk: one conflict-free LDS.128 (fp32) or LDS.64 (16 bits)
//               per lane covers a 16x8 plane, strip sums by shuffles exactly as in pool_kernel
//   output      node rows staged in (double-buffered) smem -> full 128-byte row segments
// Requires h*w == 128 (the canonical 16x8 maps) and 16-byte aligned maps; otherwise pool_kernel runs.
// ------------------------------------------------------------------------------------------------
constexpr int kTpCh = 32;
constexpr int kTpConsumerWarps = 4;
constexpr int kTpThreads = 32 * (1 + kTpConsumerWarps);
template <class T> constexpr int tp_stage_bytes() { return kTpCh * 128 * static_cast<int>(sizeof(T)); }
// default ring depth: 4 stages (64 KiB in flight per CTA) at fp32; 12 of 8 KiB at 16 bits, where 4 stages are 5 % slower
// and 8 to 12 within 1-3 % of each other (profiles/half_maps/half_maps_bench.json, DESIGN.md section 3); at S <= 8 two
// CTAs still fit on an SM
template <class T> constexpr int tp_default_stages() { return sizeof(T) == 4 ? 4 : 12; }

template <class T>
struct PoolTmaArgs {
    const T *x41, *x42;                // (batch*S, C, 128), already offset to this sub-batch
    float *nodes;                      // (batch, V, C)
    float *out; int64_t ld_out;        // (batch, 2C)
    const float *g_scale, *g_shift;
    int S, C, stages;
    int unit0, unit1;                  // work units [unit0, unit1) of this launch (unit = tracklet * C/32 + chunk)
    int l2_hint;                       // 1: evict-first cache hint on the bulk copies
};

// dynamic shared memory: ring | two node tiles | barriers (+ alignment slack)
static size_t pool_tma_smem(int S, int stages, int stage_bytes) {
    const size_t b = static_cast<size_t>(stages) * stage_bytes + 2 * static_cast<size_t>(S) * kParts * kTpCh * sizeof(float) +
                     2 * static_cast<size_t>(stages) * 8;
    return ((b + 127) & ~static_cast<size_t>(127)) + 128;
}

__device__ __forceinline__ void bulk_load_evict_first(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar,
                                                      uint64_t policy) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
        ::"r"(dst), "l"(src), "r"(bytes), "r"(bar), "l"(policy) : "memory");
}

// Sum 8 per-lane values over the 8 lanes of each 8-lane group in 7 shuffles (instead of 24): after the xor-4 / 2 / 1
// exchange steps lane `sub` of a group holds the group's total of a[sub].  Pairing order == plain butterflies.
__device__ __forceinline__ float group8_transpose_sum(const float (&a)[8], int sub) {
    float b[4], c[2];
    const bool h4 = (sub & 4) != 0, h2 = (sub & 2) != 0, h1 = (sub & 1) != 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const float send = h4 ? a[j] : a[j + 4], keep = h4 ? a[j + 4] : a[j];
        b[j] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
    }
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        const float send = h2 ? b[j] : b[j + 2], keep = h2 ? b[j + 2] : b[j];
        c[j] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
    }
    const float send = h1 ? c[0] : c[1], keep = h1 ? c[1] : c[0];
    return keep + __shfl_xor_sync(0xffffffffu, send, 1);
}

__device__ __forceinline__ void bulk_load(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}

template <class T>
__global__ void __maxnreg__(48)
pool_tma_kernel(PoolTmaArgs<T> a) {
    using E = MapElem<T>;
    using Vec4 = typename E::Vec4;
    constexpr int kStageBytes = tp_stage_bytes<T>();
    constexpr int kStageVec4 = kTpCh * 128 / 4;                   // 4-element loads per stage
    extern __shared__ __align__(16) unsigned char tp_smem_dyn[];
    const int stages = a.stages, S = a.S, C = a.C, V = S * kParts;
    // align to 128 B by OFFSET (not by casting through an integer) so that the compiler keeps emitting LDS / STS
    unsigned char *smem = tp_smem_dyn + ((128u - (gemm::smem_u32(tp_smem_dyn) & 127u)) & 127u);
    const Vec4 *ring_v = reinterpret_cast<const Vec4 *>(smem);
    float *s_nodes = reinterpret_cast<float *>(smem + stages * kStageBytes);     // [2][V][32]
    uint64_t *bars = reinterpret_cast<uint64_t *>(s_nodes + 2 * V * kTpCh);
    const uint32_t ring = gemm::smem_u32(smem);
    const uint32_t bar_full = gemm::smem_u32(bars), bar_empty = bar_full + 8 * stages;
    const int tid = static_cast<int>(threadIdx.x);
    const int warp = tid >> 5, lane = tid & 31;
    const int chunks = C / kTpCh;
    const int units = a.unit1;
    const int first = a.unit0 + static_cast<int>(blockIdx.x);
    const int stride = static_cast<int>(gridDim.x);

    if (tid == 0) {
        for (int i = 0; i < stages; ++i) { gemm::mbar_init(bar_full + 8 * i, 1); gemm::mbar_init(bar_empty + 8 * i, kTpConsumerWarps); }
        gemm::fence_barrier_init();
    }
    __syncthreads();

    if (warp == 0) {
        // ================= producer: one thread issues every bulk copy of this CTA =================
        if (lane == 0) {
            uint64_t policy;
            asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));
            int stage = 0; uint32_t phase = 0;
            for (int u = first; u < units; u += stride) {
                const int b = u / chunks, cc = u % chunks;
                for (int s = 0; s < S; ++s) {
                    const size_t off = ((static_cast<size_t>(b) * S + s) * C + static_cast<size_t>(cc) * kTpCh) * 128;
#pragma unroll
                    for (int m = 0; m < 2; ++m) {
                        gemm::mbar_wait(bar_empty + 8 * stage, phase ^ 1);
                        const uint32_t full = bar_full + 8 * stage;
                        gemm::mbar_arrive_expect_tx(full, kStageBytes);
                        if (a.l2_hint) bulk_load_evict_first(ring + stage * kStageBytes, (m ? a.x42 : a.x41) + off, kStageBytes, full, policy);
                        else bulk_load(ring + stage * kStageBytes, (m ? a.x42 : a.x41) + off, kStageBytes, full);
                        if (++stage == stages) { stage = 0; phase ^= 1; }
                    }
                }
            }
        }
    } else {
        // ================= consumers =================
        const int cw = warp - 1, ct = tid - 32;                   // consumer warp / thread index
        const int grp = lane >> 3, sub = lane & 7;                // 8-lane group <-> quarter strip (4 rows of 8)
        const float inv_all = 1.0f / (static_cast<float>(S) * 128.0f);
        int stage = 0; uint32_t phase = 0; int it = 0;
        for (int u = first; u < units; u += stride, ++it) {
            const int b = u / chunks, c0 = (u % chunks) * kTpCh;
            float *sn = s_nodes + (it & 1) * V * kTpCh;
            float gsum[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) gsum[i] = 0.f;
            for (int s = 0; s < S; ++s) {
                // ---- layer4_1 frame: only the global mean needs it -> per-lane partial sums ----
                gemm::mbar_wait(bar_full + 8 * stage, phase);
                {
                    const Vec4 *p = ring_v + stage * kStageVec4 + (cw * 8) * 32 + lane;
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const float4 v = E::cvt4(p[i * 32]);
                        gsum[i] += (v.x + v.y) + (v.z + v.w);
                    }
                }
                // the stage is handed back only when its values have ARRIVED in registers: the next bulk copy into it comes
                // from another proxy, and an arrive right behind the shared-memory loads does not wait for them (this
                // ordering cost graph_kernel_tc a 1e-3 error once) -- the empty asm makes the sums, hence the loads, precede it
                asm volatile("" ::"f"(gsum[0]), "f"(gsum[1]), "f"(gsum[2]), "f"(gsum[3]), "f"(gsum[4]), "f"(gsum[5]), "f"(gsum[6]), "f"(gsum[7]) : "memory");
                __syncwarp();
                if (lane == 0) gemm::mbar_arrive(bar_empty + 8 * stage);
                if (++stage == stages) { stage = 0; phase ^= 1; }
                // ---- layer4_2 frame: quarter / half / whole strip means -> node rows ----
                gemm::mbar_wait(bar_full + 8 * stage, phase);
                {
                    const Vec4 *p = ring_v + stage * kStageVec4 + (cw * 8) * 32 + lane;
                    float q[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const float4 v = E::cvt4(p[i * 32]);
                        q[i] = (v.x + v.y) + (v.z + v.w);
                    }
                    asm volatile("" ::"f"(q[0]), "f"(q[1]), "f"(q[2]), "f"(q[3]), "f"(q[4]), "f"(q[5]), "f"(q[6]), "f"(q[7]) : "memory");
                    __syncwarp();
                    if (lane == 0) gemm::mbar_arrive(bar_empty + 8 * stage);      // values are in registers (see above)
                    // lane (grp, sub) ends with channel `sub`'s sum over quarter strip `grp`
                    const float v2 = group8_transpose_sum(q, sub);
                    const float h2 = v2 + __shfl_xor_sync(0xffffffffu, v2, 8);       // half strips
                    const float w2 = h2 + __shfl_xor_sync(0xffffffffu, h2, 16);      // whole map
                    float *dst = sn + (s * kParts) * kTpCh + cw * 8 + sub;
                    dst[grp * kTpCh] = v2 * (1.0f / 32.0f);                          // parts 0..3
                    if ((grp & 1) == 0) dst[(4 + (grp >> 1)) * kTpCh] = h2 * (1.0f / 64.0f);
                    if (grp == 0) dst[6 * kTpCh] = w2 * (1.0f / 128.0f);
                }
                if (++stage == stages) { stage = 0; phase ^= 1; }
            }
            // global branch: mean over (S, h, w), BN neck; lane (grp, sub) ends with channel `sub`'s total
            {
                float t = group8_transpose_sum(gsum, sub);
                t += __shfl_xor_sync(0xffffffffu, t, 8);
                t += __shfl_xor_sync(0xffffffffu, t, 16);
                if (grp == 0) {
                    const int c = c0 + cw * 8 + sub;
                    a.out[static_cast<size_t>(b) * a.ld_out + c] = fmaf(t * inv_all, a.g_scale[c], a.g_shift[c]);
                }
            }
            // node tile complete (named barrier of the consumer warps)
            asm volatile("bar.sync 1, %0;" ::"n"(32 * kTpConsumerWarps) : "memory");
            float *nodes = a.nodes + static_cast<size_t>(b) * V * C + c0;
            for (int v = ct >> 5; v < V; v += kTpConsumerWarps) nodes[static_cast<size_t>(v) * C + lane] = sn[v * kTpCh + lane];
            // (the other s_nodes buffer is used next; this one is rewritten only after the next unit's barrier)
        }
    }
}



// ------------------------------------------------------------------------------------------------
// graph kernel: one CTA per tracklet
// ------------------------------------------------------------------------------------------------
constexpr int kChunk = 128;                 // channel granularity of the graph kernel (C % 128 == 0)
constexpr int kGLd = kMaxNodes + 4;         // graph row stride: float4-aligned rows

struct GraphArgs {
    const float *x;                    // (B, V, C) layer input
    const float *adj;                  // (B, V, V) or null
    const uint64_t *masks;             // (B, 3) part-membership masks instead of adj (pose.cu), or null
    __nv_bfloat16 *y_planes;           // [P][B*V][C]
    int64_t plane_stride;              // B*V*C
    int V, C, P;
    int use_pose, learn_graph;
    int fp16;                          // P == 1: one fp16 plane of y * 2^k, k per tracklet
    float *y_unscale;                  // (B): 2^-k
    // low-rank first layer (graph_kernel_tc only): instead of Y = G.X the kernel writes G.T (B, V, 4S) and the planes of
    // the quarter-strip rows -- y_planes / plane_stride then describe [P][B*4S][C]
    int lowrank = 0;
    float *gt = nullptr;
    // with fp16: second plane of E4M3 pairs (AGRL_SPLIT_FP16_E4M3), per 64-channel k-block 64 bytes
    // e4m3((y s - fp16(y s)) 2^6) then 64 bytes e4m3(y s 2^-6) -- the A-operand order, W has them swapped (split.cu)
    int fp8 = 0;
};

// element (r, c) of the pose graph: the dense matrix, or the three membership masks it is made of
// (dataset_loader.py:373-387: every ordered pair of DISTINCT nodes that share a body-part class)
struct PoseGraph {
    const float *adj;
    uint64_t m0, m1, m2;
    int V;
    __device__ __forceinline__ PoseGraph(const GraphArgs &a, int b) : adj(nullptr), m0(0), m1(0), m2(0), V(a.V) {
        if (!a.use_pose) return;
        if (a.adj) adj = a.adj + static_cast<size_t>(b) * a.V * a.V;
        else { m0 = a.masks[3 * b]; m1 = a.masks[3 * b + 1]; m2 = a.masks[3 * b + 2]; }
    }
    __device__ __forceinline__ float at(int r, int c) const {
        if (adj) return adj[r * V + c];
        const uint64_t hit = ((m0 >> r) & (m0 >> c)) | ((m1 >> r) & (m1 >> c)) | ((m2 >> r) & (m2 >> c));
        return (r != c && (hit & 1ull)) ? 1.0f : 0.0f;
    }
};

// ------------------------------------------------------------------------------------------------
// graph kernel on the tensor cores: the two 56 x 56 x 2048 products of a graph layer -- the Gram
// matrix X.X^T and the message passing Y = G.X -- as tcgen05 MMAs whose operands the CTA converts itself in shared
// memory (no extra HBM traffic: X is read twice, Y planes written once, exactly as in the CUDA-core kernels).
//   Gram   of the CENTRED nodes x_v - x_ref (x_ref = the whole-frame strip of frame 0): distances are translation
//          invariant, and with the common part removed d2 = |xi'|^2 + |xj'|^2 - 2 xi'.xj' no longer cancels 99 % of its
//          terms, so TWO bf16 planes (3 plane products instead of the 6 an fp32-exact Gram of the raw rows needs)
//          keep the affinity within 1e-6.  Per 64-channel block the [node][channel] tile in the 128-byte-swizzled
//          K-major layout is multiplied with itself: M = 128 (rows 64.. are don't-care), N = 64, accumulated over all
//          blocks in TMEM with the dominant product in its own accumulator (as the distance GEMM does).
//   G      affinity, L1 rows, pose mixing on CUDA cores exactly as in graph_kernel; then G as two bf16 planes.
//   Y      per 128-channel block the TRANSPOSED tile [channel][node] (K = nodes) as two bf16 planes; D = G.X^T block,
//          3 plane products (same 16-bit operand class as the planes Y is rounded to anyway), 128 x 128 x 16 MMAs,
//          double-buffered accumulator.
//   input  a loader warp fetches the node rows as raw fp32 tiles [V][64 channels] with ONE bulk tensor copy per tile
//          (3-D tensor map over (tracklet, node, channel), completion on an mbarrier); the converters read shared memory.
//   roles  14 warps: 0..11 workers, 12 issues the MMAs, 13 loads.  Gram: workers 0..7 convert (three operand buffers,
//          three tiles in flight).  Y: workers 2,3,6..11 convert, workers 0,1,4,5 (the ones that may read TMEM lanes
//          0..63) drain accumulators into operand planes with 32-byte stores (st.global.v8.b32: whole sectors).  Inside
//          a phase the roles are coupled by mbarriers only (tile landed / stage free / operands ready / MMAs retired /
//          accumulator drained).
//   clock64 timeline of one tracklet, 2 CTAs per SM (tools/graph_timeline.py, profiles/r2/graph_timeline.txt):
//          with register loads Gram 63-70 k cycles, graph build 23-28 k, Y 125-143 k -- every Gram block and every 64
//          channels of Y waited 2-4 k cycles on its own global loads.  With the staged tiles: Gram 75 k, build 23 k,
//          Y 99 k.  The Gram phase receives one 14 KiB tile per ~2 k cycles whether two, three or four are in flight
//          (request-to-landed grows from 2.2 k to 5 k cycles instead): that is the memory system's rate for this
//          kernel's pattern -- 296 CTAs reading 256-byte pieces 8 KiB apart while their neighbours write 128-byte pieces
//          4 KiB apart -- about 3-3.7 TB/s chip-wide, so the phase is memory-bound at that efficiency.  Y is bound by
//          the four drain warps (TMEM -> conversion -> stores, ~6 k cycles per 128 channels).
//          Tried without gain: staging the output planes through padded shared memory for 64-byte-contiguous stores,
//          eight drain + six convert warps at 64 registers, UMMA M = 64 (other TMEM row layout), 64-channel Y blocks,
//          two or four accumulators per product class, three CTAs per SM, 56 row copies per tile instead of the tensor
//          map (4-5 k cycles of issue overhead per tile), four tile stages with two operand buffers, four operand
//          buffers with two stages, walking the channels of Y in reverse (to reuse the Gram's tail from L2).
// Measured: 30 % faster than the CUDA-core kernel of round 1 (11.5 vs 16.3 ms per pass), another 5-10 % from the staged
// tiles and the 32-byte stores; a Gram on the CUDA cores with only Y on tcgen05 was slower than either (17.1 ms).
// One CTA per tracklet, 448 threads, 2 CTAs per SM (109 KiB smem at V = 56, 256 TMEM columns each).
// ------------------------------------------------------------------------------------------------
constexpr int kTcPlane = 64 * 128;                     // 8 KiB: 64 rows x 128 B
constexpr int kTcGPlanes = 0;                          // two G planes; the 128-row A descriptor of plane 1 runs into the ring
constexpr int kTcRingOff = 2 * kTcPlane;               // Gram: 3 buffers x 2 planes x 8 KiB, then the third tile stage;
constexpr int kTcRingBytes = 8 * kTcPlane;             // Y: 2 buffers x 2 planes x 16 KiB; in between: g[64][68], sq[64]
constexpr int kTcBars = kTcRingOff + kTcRingBytes;
constexpr int kTcRawOff = kTcBars + 256;                // message-passing phase: 2 stages of raw fp32 node rows, [V][64 channels] each
constexpr int kTcSmem = kTcRawOff + 1024;              // + 2 * V * 256 bytes of raw stages (full layer only)
constexpr int kTcThreads = 448;                        // 12 workers, the MMA issuer, the bulk-copy loader
static_assert((kMaxNodes * kGLd + kMaxNodes) * 4 <= kTcRingBytes, "g[] fits the ring");

__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// 8 fp32 -> `P` bf16 planes of 8 values (16 bytes each): p0 = bf16(x), p1 = bf16(x - p0), ...
template <int P>
__device__ __forceinline__ void split8(const float (&v)[8], uint4 (&out)[P]) {
    float r[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) r[i] = v[i];
#pragma unroll
    for (int p = 0; p < P; ++p) {
        uint32_t w[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const __nv_bfloat162 b = __floats2bfloat162_rn(r[2 * i], r[2 * i + 1]);
            w[i] = *reinterpret_cast<const uint32_t *>(&b);
            r[2 * i] = __fsub_rn(r[2 * i], __uint_as_float(w[i] << 16));
            r[2 * i + 1] = __fsub_rn(r[2 * i + 1], __uint_as_float(w[i] & 0xffff0000u));
        }
        out[p] = make_uint4(w[0], w[1], w[2], w[3]);
    }
}

// 8 scaled fp32 -> 8 fp16 (16 B), their residuals x 2^6 as E4M3 (8 B), the values x 2^-6 as E4M3 (8 B)
__device__ __forceinline__ void split8_f16e4(const float (&v)[8], uint4 &h16, uint2 &res8, uint2 &val8) {
    uint32_t hw[4], r[4], c[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const __half2 h = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
        hw[i] = *reinterpret_cast<const uint32_t *>(&h);
        const float2 hf = __half22float2(h);
        // (v - h) * 64 as ONE fma: v - h is exact in fp32 and 64 a power of two, so the result is the same number
        r[i] = __nv_cvt_float2_to_fp8x2(make_float2(fmaf(v[2 * i], 64.0f, -64.0f * hf.x), fmaf(v[2 * i + 1], 64.0f, -64.0f * hf.y)),
                                        __NV_SATFINITE, __NV_E4M3);
        c[i] = __nv_cvt_float2_to_fp8x2(make_float2(v[2 * i] * 0.015625f, v[2 * i + 1] * 0.015625f), __NV_SATFINITE, __NV_E4M3);
    }
    h16 = make_uint4(hw[0], hw[1], hw[2], hw[3]);
    res8 = make_uint2(r[0] | (r[1] << 16), r[2] | (r[3] << 16));
    val8 = make_uint2(c[0] | (c[1] << 16), c[2] | (c[3] << 16));
}

// one 32-byte store per lane (STG.256): full 32-byte sectors instead of two half-written ones
__device__ __forceinline__ void st256(void *p, const uint4 &a, const uint4 &b) {
    asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                 ::"l"(p), "r"(a.x), "r"(a.y), "r"(a.z), "r"(a.w), "r"(b.x), "r"(b.y), "r"(b.z), "r"(b.w) : "memory");
}

// clock64 timeline of the kernel's phases (tools/graph_timeline.py): compiled in only with -DAGRL_TIMELINE
// (AGRL_NVCC_EXTRA=-DAGRL_TIMELINE python -m agrl.pytorch_b200.build --force), never in the product library
#ifdef AGRL_TIMELINE
__device__ long long *g_timeline = nullptr;
#define AGRL_TL_DECL                                                                                         \
    const bool tl_on = g_timeline != nullptr && (blockIdx.x % 97 == 5) && !a.lowrank;                        \
    const long long tl_base = static_cast<long long>(blockIdx.x / 97) * 256
#define AGRL_TL(slot) do { if (tl_on && (threadIdx.x & 31) == 0) g_timeline[tl_base + (slot)] = clock64(); } while (0)
#else
#define AGRL_TL_DECL
#define AGRL_TL(slot) do { } while (0)
#endif

__global__ void __launch_bounds__(kTcThreads, 2)
graph_kernel_tc(const __grid_constant__ CUtensorMap map_x, GraphArgs a) {
    AGRL_TL_DECL;
    extern __shared__ __align__(16) unsigned char tc_smem_dyn[];
    unsigned char *smem = tc_smem_dyn + ((1024u - (gemm::smem_u32(tc_smem_dyn) & 1023u)) & 1023u);
    unsigned char *ring_p = smem + kTcRingOff;
    float *g = reinterpret_cast<float *>(ring_p);                      // [64][68], between the two MMA phases
    float *sq = g + kMaxNodes * kGLd;                                  // [64]
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + kTcBars);     // done[2], gfull[3], gdone[3], yfull[2], accfree[2], tmem slot, rfull[3], rempty[3]
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 14);
    const uint32_t gplanes = gemm::smem_u32(smem) + kTcGPlanes, ring = gemm::smem_u32(ring_p), bar0 = gemm::smem_u32(bars);
    const uint32_t b_done = bar0, b_gfull = bar0 + 16, b_gdone = bar0 + 48, b_yfull = bar0 + 80, b_accfree = bar0 + 96;
    const uint32_t b_rfull = bar0 + 128, b_rempty = bar0 + 160;         // three stages each
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const bool worker = warp < 12, issuer = warp == 12, loader = warp == 13, gram_worker = warp < 8;
    const int V = a.V, C = a.C, b = blockIdx.x;
    const float *x = a.x + static_cast<size_t>(b) * V * C;

    if (tid == 0) {
        for (int i = 0; i < 2; ++i) {
            gemm::mbar_init(b_done + 8 * i, 1);
            gemm::mbar_init(b_yfull + 8 * i, 8); gemm::mbar_init(b_accfree + 8 * i, 4);
        }
        for (int i = 0; i < 3; ++i) {
            gemm::mbar_init(b_rfull + 8 * i, 1); gemm::mbar_init(b_rempty + 8 * i, 8);
            gemm::mbar_init(b_gfull + 8 * i, 8); gemm::mbar_init(b_gdone + 8 * i, 1);
        }
        gemm::fence_barrier_init();
    }
    if (warp == 0) { gemm::tmem_alloc(gemm::smem_u32(tmem_slot), 256); gemm::tmem_relinquish(); }
    if (!a.learn_graph && gram_worker) for (int i = tid; i < kMaxNodes * kGLd; i += kHeadThreads) g[i] = 0.f;
    gemm::tc_fence_before();
    __syncthreads();
    gemm::tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    const bool epi_warp = gram_worker && (warp & 3) < 2;               // warps 0,1,4,5 may read TMEM lanes 0..63; row = node
    const int erow = (warp & 3) * 32 + lane, ehalf = warp >> 2;
    const uint32_t tlane = tmem + (static_cast<uint32_t>((warp & 3) * 32) << 16);
    auto wait_bar = [&](uint32_t bar, int use) { gemm::mbar_wait(bar, static_cast<uint32_t>(use & 1)); };
    const int ref_row = (V > 6) ? 6 : V - 1;                           // centre of the Gram: the whole-frame strip of frame 0
    const int n_gblocks = C / 64;                                      // even (C % 128 == 0)
    if (warp == 0) AGRL_TL(0);
    // Input staging: the node rows reach both tensor-core phases as raw fp32 tiles, [V][64 channels] each, fetched by ONE
    // bulk tensor copy per tile (completion on an mbarrier) by the loader warp -- the converters read shared memory
    // instead of waiting on global loads (clock64 timeline of the register-load version: 2 k cycles per Gram block and
    // 3-4 k per 64 channels of the message-passing phase, all of it exposed load latency).  A tile takes ~2.2 k cycles to
    // arrive, so the Gram phase keeps THREE in flight (the third stage sits in the operand ring's last quarter, next to
    // its three operand buffers); the message-passing phase, bound by its accumulator drain, uses stages 0 and 1.
    const int raw_stage = V * 256;
    auto stage_off = [&](int st) { return st < 2 ? kTcRawOff + st * raw_stage : kTcRingOff + 6 * kTcPlane; };
    // (L2 eviction hints on the tile copies -- keep the Gram phase's tiles, stream the message passing's -- cut the layer-2
    // launch's DRAM reads from 0.82 to 0.72 GB and changed neither its time nor the head's: A/B on one box, tools/build_alt.sh,
    // before and after the drain rework.)
    auto load_raw = [&](int piece, int st) {          // loader: tile of channels [64 piece, +64) -> stage st
        if (lane == 0) {
            const uint32_t full = b_rfull + 8 * st;
            gemm::mbar_arrive_expect_tx(full, static_cast<uint32_t>(raw_stage));
            gemm::tma_load_3d(gemm::smem_u32(smem) + stage_off(st), &map_x, full, piece * 64, 0, b);
        }
    };
    // (No L2 prefetch ahead of the tile copies: per-line prefetches and one tensor-map prefetch per four tiles were both
    // measured -- 0.341 instead of 0.313 ms for the layer-2 launch and 1.05 instead of 0.82 GB of DRAM reads, the prefetched
    // lines being evicted again before their tile copy arrives.)
    // uses of stage st by the Gram phase (tiles st, st + 3, ...): the message passing continues each barrier's phase count
    auto gram_uses_of = [&](int st) { return a.learn_graph ? (n_gblocks + 2 - st) / 3 : 0; };
    if (loader && lane == 0) gemm::prefetch_tensormap(&map_x);

    if (a.learn_graph) {
        // ================= Gram =================
        if (gram_worker) {
            // item = (row, 8-channel slot): 64 rows x 8 slots, two items per thread, read from the staged tile
            for (int kb = 0; kb < n_gblocks; ++kb) {
                const int buf = kb % 3, use = kb / 3;                  // three operand buffers, three tile stages
                wait_bar(b_rfull + 8 * buf, use);                      // the tile has landed
                if (warp == 0) AGRL_TL(96 + kb);
                if (kb >= 3) wait_bar(b_gdone + 8 * buf, use - 1);     // the MMAs that read this operand buffer have retired
                if (warp == 0) AGRL_TL(192 + kb);
                const float *rs = reinterpret_cast<const float *>(smem + stage_off(buf));
                const float4 *rsrc = reinterpret_cast<const float4 *>(rs + ref_row * 64 + (tid & 7) * 8);   // slot is the same for both items
                const float4 rlo = rsrc[0], rhi = rsrc[1];
                unsigned char *dst = ring_p + buf * 2 * kTcPlane;
#pragma unroll
                for (int t = 0; t < 2; ++t) {
                    const int item = tid + kHeadThreads * t, row = item >> 3, slot = item & 7;
                    float c[8];
                    if (row < V) {
                        const float4 *src = reinterpret_cast<const float4 *>(rs + row * 64 + slot * 8);
                        const float4 lo = src[0], hi = src[1];
                        c[0] = __fsub_rn(lo.x, rlo.x); c[1] = __fsub_rn(lo.y, rlo.y); c[2] = __fsub_rn(lo.z, rlo.z); c[3] = __fsub_rn(lo.w, rlo.w);
                        c[4] = __fsub_rn(hi.x, rhi.x); c[5] = __fsub_rn(hi.y, rhi.y); c[6] = __fsub_rn(hi.z, rhi.z); c[7] = __fsub_rn(hi.w, rhi.w);
                    } else {
#pragma unroll
                        for (int i = 0; i < 8; ++i) c[i] = 0.f;
                    }
                    uint4 pl[2];
                    split8<2>(c, pl);
                    const int off = row * 128 + ((slot ^ (row & 7)) << 4);
#pragma unroll
                    for (int p = 0; p < 2; ++p) *reinterpret_cast<uint4 *>(dst + p * kTcPlane + off) = pl[p];
                }
                fence_proxy_async_smem();
                __syncwarp();
                // (the stage is released only after its values have been converted and stored: an arrive right after the
                // shared-memory loads would let the next bulk copy -- another proxy -- overtake them)
                if (lane == 0) { gemm::mbar_arrive(b_gfull + 8 * buf); gemm::mbar_arrive(b_rempty + 8 * buf); }
                if (warp == 0) AGRL_TL(128 + kb);
            }
            for (int i = 0; i < 3; ++i)                                // every Gram MMA has retired
                if (i < n_gblocks) wait_bar(b_gdone + 8 * i, (n_gblocks + 2 - i) / 3 - 1);
            gemm::tc_fence_after();
            if (epi_warp) {
                uint32_t m[32], c[32];
                gemm::tmem_ld_32x32(tlane + ehalf * 32, m);
                gemm::tmem_ld_32x32(tlane + 64 + ehalf * 32, c);
                gemm::tmem_ld_wait();
                // (all 64 x 64 entries: rows / columns >= V are products of zero rows, i.e. zeros)
#pragma unroll
                for (int j = 0; j < 32; ++j)
                    g[erow * kGLd + ehalf * 32 + j] = __fadd_rn(__uint_as_float(m[j]), __uint_as_float(c[j]));
            }
            gemm::tc_fence_before();
        } else if (issuer && lane == 0) {
            constexpr uint32_t idesc = gemm::make_idesc(128, 64);
            for (int kb = 0; kb < n_gblocks; ++kb) {
                const int buf = kb % 3;
                wait_bar(b_gfull + 8 * buf, kb / 3);
                gemm::tc_fence_after();
                const uint32_t base = ring + buf * 2 * kTcPlane;
#pragma unroll
                for (int i = 0; i < 3; ++i) {
                    int pa, pb;
                    gemm::pair_of(2, i, pa, pb);
                    const uint64_t da = gemm::make_smem_desc(base + pa * kTcPlane), db = gemm::make_smem_desc(base + pb * kTcPlane);
                    const bool main_acc = (i == 2);                    // a0.b0 alone in columns 0..63, corrections in 64..127
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        gemm::tc_mma_bf16(tmem + (main_acc ? 0 : 64), da + 2 * k, db + 2 * k, idesc,
                                          main_acc ? ((kb | k) != 0) : ((kb | i | k) != 0));
                }
                gemm::tc_commit(b_gdone + 8 * buf);
                AGRL_TL(160 + kb);
            }
        } else if (loader) {
            for (int kb = 0; kb < n_gblocks; ++kb) {
                if (kb >= 3) wait_bar(b_rempty + 8 * (kb % 3), kb / 3 - 1);
                load_raw(kb, kb % 3);
            }
            if (!a.lowrank)                                            // the first two tiles of the message-passing phase
                for (int hh = 0; hh < 2; ++hh) {
                    if (gram_uses_of(hh) > 0) wait_bar(b_rempty + 8 * hh, gram_uses_of(hh) - 1);
                    load_raw(hh, hh);
                }
        }
        __syncthreads();
        if (warp == 0) AGRL_TL(1);
        if (gram_worker && tid < V) sq[tid] = g[tid * kGLd + tid];
        __syncthreads();
        if (worker) {
            for (int i = tid; i < V * V; i += 32 * 12) {                // affinity (vmgn.py:116-120), all 12 worker warps
                const int r = i / V, c = i % V;
                float d2 = __fadd_rn(sq[c], sq[r]);
                d2 = fmaf(-2.0f, g[r * kGLd + c], d2);
                const float d = sqrtf(fmaxf(d2, 1e-12f));
                g[r * kGLd + c] = __fdiv_rn(2.0f, expf(d) + 1.0f);
            }
        }
        __syncthreads();
    }
    // ---- L1 row normalisation + mixing: one worker warp per row (as graph_kernel) ----
    if (worker) {
        const PoseGraph pose(a, b);
        for (int r = warp; r < V; r += 12) {
            float s0 = 0.f, s1 = 0.f, a0 = 0.f, a1 = 0.f, ra = 0.f, rs = 0.f;
            const int c1 = lane + 32;
            if (a.learn_graph) { s0 = (lane < V) ? g[r * kGLd + lane] : 0.f; s1 = (c1 < V) ? g[r * kGLd + c1] : 0.f; rs = warp_sum(fabsf(s0) + fabsf(s1)); }
            if (a.use_pose) { a0 = (lane < V) ? pose.at(r, lane) : 0.f; a1 = (c1 < V) ? pose.at(r, c1) : 0.f; ra = warp_sum(fabsf(a0) + fabsf(a1)); }
            rs = fmaxf(rs, 1e-12f); ra = fmaxf(ra, 1e-12f);
            float m0, m1;
            if (a.learn_graph && a.use_pose) {
                m0 = __fdiv_rn(__fdiv_rn(a0, ra) + __fdiv_rn(s0, rs), 2.0f);
                m1 = __fdiv_rn(__fdiv_rn(a1, ra) + __fdiv_rn(s1, rs), 2.0f);
            } else if (a.learn_graph) { m0 = __fdiv_rn(s0, rs); m1 = __fdiv_rn(s1, rs); }
            else { m0 = __fdiv_rn(a0, ra); m1 = __fdiv_rn(a1, ra); }
            __syncwarp();
            g[r * kGLd + lane] = (lane < V) ? m0 : 0.f;
            g[r * kGLd + c1] = (c1 < V) ? m1 : 0.f;
        }
    }
    __syncthreads();
    __shared__ float s_scale[2];
    float y_scale = 1.0f;
    if (a.fp16) {                                                      // see graph_kernel
        if (!a.learn_graph) {
            if (worker) {
                for (int r = warp; r < V; r += 12) {
                    const float4 *row = reinterpret_cast<const float4 *>(x + static_cast<size_t>(r) * C);
                    float t = 0.f;
                    for (int i = lane; i < C / 4; i += 32) {
                        const float4 v = __ldg(row + i);
                        t = fmaf(v.x, v.x, t); t = fmaf(v.y, v.y, t); t = fmaf(v.z, v.z, t); t = fmaf(v.w, v.w, t);
                    }
                    t = warp_sum(t);
                    if (lane == 0) sq[r] = t;
                }
            }
            __syncthreads();
        }
        if (warp == 0) {
            float m = fmaxf(lane < V ? sq[lane] : 0.f, lane + 32 < V ? sq[lane + 32] : 0.f);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
            float refn = 0.f;                                          // the Gram was centred: |x_v| <= |x_ref| + |x_v - x_ref|
            if (a.learn_graph) {
                const float4 *row = reinterpret_cast<const float4 *>(x + static_cast<size_t>(ref_row) * C);
                for (int i = lane; i < C / 4; i += 32) {
                    const float4 v = __ldg(row + i);
                    refn = fmaf(v.x, v.x, refn); refn = fmaf(v.y, v.y, refn); refn = fmaf(v.z, v.z, refn); refn = fmaf(v.w, v.w, refn);
                }
                refn = warp_sum(refn);
            }
            if (lane == 0) {
                m = (m < 3.0e38f && refn < 3.0e38f) ? sqrtf(m) + sqrtf(refn) : 0.f;
                pow2_scales(m, &s_scale[0], &s_scale[1]);
                a.y_unscale[b] = s_scale[1];
            }
        }
        __syncthreads();
        y_scale = s_scale[0];
    }
    if (a.lowrank) {
        // ---- low-rank first layer: the nodes of a frame are T.(its four quarter strips), so G.X.W^T = (G.T).(Q.W^T).
        // Emit G.T (V x 4S) and the quarter-strip rows Q as GEMM operand planes; the message passing happens after the
        // GEMM, on 4S instead of 7S rows (graph_mix_kernel). ----
        if (worker) {
            const int S4 = (V / kParts) * 4;
            float *gt = a.gt + static_cast<size_t>(b) * V * S4;
            for (int i = tid; i < V * S4; i += 32 * 12) {
                const int r = i / S4, j = i - r * S4, k = j & 3;
                const float *gr = g + r * kGLd + (j >> 2) * kParts;         // frame j / 4 of row r
                gt[i] = fmaf(0.25f, gr[6], fmaf(0.5f, gr[4 + (k >> 1)], gr[k]));
            }
            const int groups = C / 8;
            for (int i = tid; i < S4 * groups; i += 32 * 12) {
                const int qr = i / groups, cg = i - qr * groups;
                const int row = (qr >> 2) * kParts + (qr & 3);
                const float4 *src = reinterpret_cast<const float4 *>(x + static_cast<size_t>(row) * C + cg * 8);
                const float4 lo = __ldg(src), hi = __ldg(src + 1);
                const float v[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
                __nv_bfloat16 *dst = a.y_planes + (static_cast<size_t>(b) * S4 + qr) * C + cg * 8;
                if (a.fp8) {
                    float vs[8];
#pragma unroll
                    for (int t = 0; t < 8; ++t) vs[t] = v[t] * y_scale;
                    uint4 h16; uint2 r8, c8;
                    split8_f16e4(vs, h16, r8, c8);
                    *reinterpret_cast<uint4 *>(dst) = h16;
                    unsigned char *row8 = reinterpret_cast<unsigned char *>(a.y_planes + a.plane_stride + (static_cast<size_t>(b) * S4 + qr) * C) +
                                          (cg >> 3) * 128 + (cg & 7) * 8;
                    *reinterpret_cast<uint2 *>(row8) = r8;
                    *reinterpret_cast<uint2 *>(row8 + 64) = c8;
                } else if (a.fp16) {
                    uint32_t w[4];
#pragma unroll
                    for (int t = 0; t < 4; ++t) {
                        const __half2 h = __floats2half2_rn(v[2 * t] * y_scale, v[2 * t + 1] * y_scale);
                        w[t] = *reinterpret_cast<const uint32_t *>(&h);
                    }
                    *reinterpret_cast<uint4 *>(dst) = make_uint4(w[0], w[1], w[2], w[3]);
                } else if (a.P == 3) {
                    uint4 pl[3];
                    split8<3>(v, pl);
#pragma unroll
                    for (int pp = 0; pp < 3; ++pp) *reinterpret_cast<uint4 *>(dst + pp * a.plane_stride) = pl[pp];
                } else {
                    uint4 pl[2];
                    split8<2>(v, pl);
#pragma unroll
                    for (int pp = 0; pp < 2; ++pp) *reinterpret_cast<uint4 *>(dst + pp * a.plane_stride) = pl[pp];
                }
            }
        }
        gemm::tc_fence_before();
        __syncthreads();
        if (warp == 0) gemm::tmem_dealloc(tmem, 256);
        return;
    }
    // ---- G as two bf16 planes, K-major [row = output node][k = input node] ----
    if (gram_worker) {
#pragma unroll
        for (int t = 0; t < 2; ++t) {
            const int item = tid + kHeadThreads * t, row = item >> 3, slot = item & 7;
            float v[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = (row < V) ? g[row * kGLd + slot * 8 + i] : 0.f;    // columns >= V hold zeros
            uint4 pl[2];
            split8<2>(v, pl);
            const int off = row * 128 + ((slot ^ (row & 7)) << 4);
            *reinterpret_cast<uint4 *>(smem + kTcGPlanes + off) = pl[0];
            *reinterpret_cast<uint4 *>(smem + kTcGPlanes + kTcPlane + off) = pl[1];
        }
        fence_proxy_async_smem();
    }
    __syncthreads();                                                   // g[] (in the ring) is dead from here on

    // ================= Y = G . X, 128 channels per block =================
    const int n_blocks = C / 128;
    if (warp == 0) AGRL_TL(2);
    if (issuer) {
        if (lane == 0) {
            constexpr uint32_t idesc = gemm::make_idesc(128, 128);
            for (int cb = 0; cb < n_blocks; ++cb) {
                const int buf = cb & 1;
                wait_bar(b_yfull + 8 * buf, cb >> 1);
                if (cb >= 2) wait_bar(b_accfree + 8 * buf, (cb >> 1) - 1);   // the epilogue has drained this accumulator
                gemm::tc_fence_after();
                const uint32_t bbase = ring + buf * 4 * kTcPlane;
#pragma unroll
                for (int i = 0; i < 3; ++i) {
                    int pa, pb;
                    gemm::pair_of(2, i, pa, pb);
                    const uint64_t da = gemm::make_smem_desc(gplanes + pa * kTcPlane), db = gemm::make_smem_desc(bbase + pb * 2 * kTcPlane);
#pragma unroll
                    for (int k = 0; k < 4; ++k) gemm::tc_mma_bf16(tmem + buf * 128, da + 2 * k, db + 2 * k, idesc, (i | k) != 0);
                }
                gemm::tc_commit(b_done + 8 * buf);
                AGRL_TL(16 + cb);
            }
        }
    } else if (loader) {
        // tile hh as soon as every converter warp has released the stage of tile hh - 2 (tiles 0 and 1 were requested at the end
        // of the Gram phase when there is one)
        const int n_halves = 2 * n_blocks;
        for (int hh = a.learn_graph ? 2 : 0; hh < n_halves; ++hh) {
            const int use = gram_uses_of(hh & 1) + (hh >> 1);
            if (use > 0) wait_bar(b_rempty + 8 * (hh & 1), use - 1);
            load_raw(hh, hh & 1);
        }
    } else if (!epi_warp) {
        // converters (workers 2,3,6..11 -> 256 threads), 64 channels at a time: item = (channel, 8-node group), lane =
        // channel, so every shared-memory read is conflict-free (32 consecutive floats of one node row); two items per
        // thread; two such pieces fill one operand buffer
        const int cw = warp < 8 ? ((warp >> 2) * 2 + (warp & 1)) : warp - 4;   // 0..7
        const int ctid = cw * 32 + lane, ch = ctid & 63, g0 = ctid >> 6, n_halves = 2 * n_blocks;
        float nx[2][8];
        for (int hh = 0; hh < n_halves; ++hh) {
            wait_bar(b_rfull + 8 * (hh & 1), gram_uses_of(hh & 1) + (hh >> 1));   // the tile has landed
            {
                const float *rs = reinterpret_cast<const float *>(smem + stage_off(hh & 1)) + ch;
#pragma unroll
                for (int t = 0; t < 2; ++t) {
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const int v = (g0 + 4 * t) * 8 + i;
                        nx[t][i] = (v < V) ? rs[v * 64] : 0.f;
                    }
                }
            }
            const int cb = hh >> 1, buf = cb & 1, prev = (cb >> 1) - 1;
            if ((hh & 1) == 0 && prev >= 0) wait_bar(b_done + 8 * buf, prev);   // the MMAs that read this buffer have retired
            if ((hh & 1) == 0 && cw == 0) AGRL_TL(48 + cb);
            unsigned char *dst = ring_p + buf * 4 * kTcPlane;
            const int row = (hh & 1) * 64 + ch;
#pragma unroll
            for (int t = 0; t < 2; ++t) {
                uint4 pl[2];
                split8<2>(nx[t], pl);
                const int off = row * 128 + (((g0 + 4 * t) ^ (row & 7)) << 4);
                *reinterpret_cast<uint4 *>(dst + off) = pl[0];
                *reinterpret_cast<uint4 *>(dst + 2 * kTcPlane + off) = pl[1];
            }
            // the stage may be refilled only now: the shared-memory reads above have certainly completed once their values
            // have been converted and stored (an arrive right after the loads lets the bulk copy -- another proxy -- overtake them)
            __syncwarp();
            if (lane == 0) gemm::mbar_arrive(b_rempty + 8 * (hh & 1));
            if (hh & 1) {
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) gemm::mbar_arrive(b_yfull + 8 * buf);
                if (cw == 0) AGRL_TL(32 + cb);
            }
        }
    } else {
        // epilogue (workers 0,1,4,5): accumulator -> registers (frees it for block cb + 2) -> planes -> global
        for (int cb = 0; cb < n_blocks; ++cb) {
            const int acc = cb & 1;
            wait_bar(b_done + 8 * acc, cb >> 1);
            if (warp == 0) AGRL_TL(64 + cb);
            gemm::tc_fence_after();
            // 32 channels at a time (64 accumulator values at once do not fit the 72 registers of a thread next to the
            // conversion's temporaries); the accumulator is released after the second read -- the drain, not the MMAs of
            // the next block, paces this phase, so an earlier release would buy nothing
#pragma unroll
            for (int hq = 0; hq < 2; ++hq) {
                uint32_t r[1][32];
                gemm::tmem_ld_32x32(tlane + acc * 128 + ehalf * 64 + hq * 32, r[0]);
                gemm::tmem_ld_wait();
                if (hq == 1) {
                    gemm::tc_fence_before();
                    __syncwarp();
                    if (lane == 0) gemm::mbar_arrive(b_accfree + 8 * acc);
                    if (warp == 0) AGRL_TL(80 + cb);
                }
                if (erow < V) {
                    __nv_bfloat16 *dst = a.y_planes + (static_cast<size_t>(b) * V + erow) * C + cb * 128 + ehalf * 64 + hq * 32;
                    if (a.fp8) {
                        // this thread's 64 channels are exactly k-block 2 cb + ehalf of the row
                        unsigned char *row8 = reinterpret_cast<unsigned char *>(a.y_planes + a.plane_stride + (static_cast<size_t>(b) * V + erow) * C) +
                                              (cb * 2 + ehalf) * 128 + hq * 32;
                        // 32 channels: 64 bytes of fp16, 32 bytes of residuals, 32 bytes of value copies -> four 32-byte stores
                        uint4 h16[4]; uint2 r8[4], c8[4];
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            float v[8];
#pragma unroll
                            for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[0][8 * e + i]) * y_scale;
                            split8_f16e4(v, h16[e], r8[e], c8[e]);
                        }
                        st256(dst, h16[0], h16[1]);
                        st256(dst + 16, h16[2], h16[3]);
                        st256(row8, make_uint4(r8[0].x, r8[0].y, r8[1].x, r8[1].y), make_uint4(r8[2].x, r8[2].y, r8[3].x, r8[3].y));
                        st256(row8 + 64, make_uint4(c8[0].x, c8[0].y, c8[1].x, c8[1].y), make_uint4(c8[2].x, c8[2].y, c8[3].x, c8[3].y));
                    } else if (a.fp16) {
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            uint32_t w[4];
#pragma unroll
                            for (int i = 0; i < 4; ++i) {
                                const __half2 h = __floats2half2_rn(__uint_as_float(r[0][8 * q + 2 * i]) * y_scale,
                                                                    __uint_as_float(r[0][8 * q + 2 * i + 1]) * y_scale);
                                w[i] = *reinterpret_cast<const uint32_t *>(&h);
                            }
                            reinterpret_cast<uint4 *>(dst)[q] = make_uint4(w[0], w[1], w[2], w[3]);
                        }
                    } else {
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            float v[8];
#pragma unroll
                            for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[0][8 * q + i]);
                            if (a.P == 3) {
                                uint4 pl[3];
                                split8<3>(v, pl);
#pragma unroll
                                for (int p = 0; p < 3; ++p) reinterpret_cast<uint4 *>(dst + p * a.plane_stride)[q] = pl[p];
                            } else {
                                uint4 pl[2];
                                split8<2>(v, pl);
#pragma unroll
                                for (int p = 0; p < 2; ++p) reinterpret_cast<uint4 *>(dst + p * a.plane_stride)[q] = pl[p];
                            }
                        }
                    }
                }
            }
        }
    }
    if (warp == 0) AGRL_TL(3);
    gemm::tc_fence_before();
    __syncthreads();
    if (warp == 0) gemm::tmem_dealloc(tmem, 256);
}

// ------------------------------------------------------------------------------------------------
// low-rank first layer, part 2: out = (1 - gamma) X + gamma LeakyReLU(BN((G.T) . Z)) with
// Z = Q.W^T (4S rows per tracklet, from the GEMM) and G.T (V x 4S, from graph_kernel_tc).  A thread keeps its columns of
// Z in registers, the rows of G.T come as shared-memory broadcasts.
// ------------------------------------------------------------------------------------------------
constexpr int kMixLdMax = 36;                          // 4S <= 36 for V <= 64; the kernel is instantiated for 32 (S <= 8) and 36
struct MixArgs {
    const float *x, *z, *gt;           // (B, V, C), (B, 4S, C), (B, V, 4S)
    float *out;                        // (B, V, C)
    const float *scale, *shift;        // folded BatchNorm of the layer
    int V, S4, C;
    float gamma, slope;
};

// Two channels per thread -- every shared-memory broadcast of four G.T weights feeds eight FMAs -- and the residual rows
// of eight nodes loaded ahead of their use, so that the row loop is not bound by the latency of one load per 36 FMAs.
// grid (C / 512, tracklets).  (Packed fma.rn.f32x2 with the weights duplicated in shared memory was measured: 4.67 vs
// 4.40 ms per pass -- FFMA2 issues at half rate on sm_100, the extra LDS traffic is pure cost.)
constexpr int kMixRows = 8;                             // (4: same time, 14: 4.6 instead of 4.0 ms per pass, A/B on one box)
template <int kMixLd>                                  // row length of G.T in shared memory / registers: 4S padded with zeros
__global__ void __launch_bounds__(kHeadThreads, 2)
graph_mix_kernel(MixArgs a) {
    __shared__ __align__(16) float s_gt[kMaxNodes * kMixLd];
    const int b = blockIdx.y, c = (blockIdx.x * kHeadThreads + threadIdx.x) * 2;
    const int V = a.V, S4 = a.S4, C = a.C;
    const float *gt = a.gt + static_cast<size_t>(b) * V * S4;
    for (int i = threadIdx.x; i < V * kMixLd; i += kHeadThreads) {
        const int r = i / kMixLd, k = i - r * kMixLd;
        s_gt[i] = (k < S4) ? gt[r * S4 + k] : 0.f;
    }
    float2 z[kMixLd];
    const float *zc = a.z + static_cast<size_t>(b) * S4 * C + c;
#pragma unroll
    for (int k = 0; k < kMixLd; ++k)
        z[k] = (k < S4) ? __ldg(reinterpret_cast<const float2 *>(zc + static_cast<size_t>(k) * C)) : make_float2(0.f, 0.f);
    const float2 sc = __ldg(reinterpret_cast<const float2 *>(a.scale + c)), sh = __ldg(reinterpret_cast<const float2 *>(a.shift + c));
    const float keep = 1.0f - a.gamma;
    const float *xc = a.x + static_cast<size_t>(b) * V * C + c;
    float *oc = a.out + static_cast<size_t>(b) * V * C + c;
    __syncthreads();
    for (int r0 = 0; r0 < V; r0 += kMixRows) {
        float2 xin[kMixRows];
#pragma unroll
        for (int i = 0; i < kMixRows; ++i)
            xin[i] = (r0 + i < V) ? __ldg(reinterpret_cast<const float2 *>(xc + static_cast<size_t>(r0 + i) * C)) : make_float2(0.f, 0.f);
#pragma unroll
        for (int i = 0; i < kMixRows; ++i) {
            if (r0 + i < V) {
                const float4 *g4 = reinterpret_cast<const float4 *>(s_gt + (r0 + i) * kMixLd);
                float a0 = 0.f, a1 = 0.f;
#pragma unroll
                for (int k4 = 0; k4 < kMixLd / 4; ++k4) {
                    const float4 w = g4[k4];
                    a0 = fmaf(w.x, z[4 * k4 + 0].x, a0); a1 = fmaf(w.x, z[4 * k4 + 0].y, a1);
                    a0 = fmaf(w.y, z[4 * k4 + 1].x, a0); a1 = fmaf(w.y, z[4 * k4 + 1].y, a1);
                    a0 = fmaf(w.z, z[4 * k4 + 2].x, a0); a1 = fmaf(w.z, z[4 * k4 + 2].y, a1);
                    a0 = fmaf(w.w, z[4 * k4 + 3].x, a0); a1 = fmaf(w.w, z[4 * k4 + 3].y, a1);
                }
                float h0 = fmaf(a0, sc.x, sh.x), h1 = fmaf(a1, sc.y, sh.y);
                h0 = h0 >= 0.f ? h0 : h0 * a.slope;
                h1 = h1 >= 0.f ? h1 : h1 * a.slope;
                float2 o;
                o.x = fmaf(a.gamma, h0, keep * xin[i].x);
                o.y = fmaf(a.gamma, h1, keep * xin[i].y);
                *reinterpret_cast<float2 *>(oc + static_cast<size_t>(r0 + i) * C) = o;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// temporal attention + part mean + BN neck: one CTA per tracklet
// ------------------------------------------------------------------------------------------------
struct AttnArgs {
    const float *x;                    // (B, V, C) output of the last graph layer
    float *out; int64_t ld_out;        // (B, 2C): attention branch -> [:, C:]
    const float *a_scale, *a_shift;    // folded att_bottleneck
    int S, C;
    const float *row_sumsq;            // optional (B*V, slots): partial sums of squares from the last GEMM's epilogue
    int slots;
};

__global__ void __launch_bounds__(kHeadThreads)
attn_kernel(AttnArgs a) {
    __shared__ float s_norm[kMaxNodes];
    __shared__ float s_att[kMaxNodes];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int V = a.S * kParts, C = a.C, b = blockIdx.x;
    const float *x = a.x + static_cast<size_t>(b) * V * C;
    // a[s,p] = ||f[s,p,:]||_2
    if (a.row_sumsq) {                                     // the last GEMM epilogue already summed the squares per column tile
        if (tid < V) {
            const float *ps = a.row_sumsq + (static_cast<size_t>(b) * V + tid) * a.slots;
            float s = 0.f;
            for (int i = 0; i < a.slots; ++i) s += ps[i];
            s_norm[tid] = sqrtf(s);
        }
    } else {
        for (int r = warp; r < V; r += kHeadThreads / 32) {
            const float4 *row = reinterpret_cast<const float4 *>(x + static_cast<size_t>(r) * C);
            float s = 0.f;
            for (int i = lane; i < C / 4; i += 32) {
                const float4 v = __ldg(row + i);
                s = fmaf(v.x, v.x, s); s = fmaf(v.y, v.y, s); s = fmaf(v.z, v.z, s); s = fmaf(v.w, v.w, s);
            }
            s = warp_sum(s);
            if (lane == 0) s_norm[r] = sqrtf(s);
        }
    }
    __syncthreads();
    // att = a / max(sum_s |a|, 1e-12)   (F.normalize p=1 over the frame axis)
    if (tid < V) {
        const int p = tid % kParts;
        float t = 0.f;
        for (int s = 0; s < a.S; ++s) t += fabsf(s_norm[s * kParts + p]);
        s_att[tid] = __fdiv_rn(s_norm[tid], fmaxf(t, 1e-12f));
    }
    __syncthreads();
    // fused[p] = sum_s f * att ; mean over p ; BN.  gridDim.y CTAs share a tracklet's channels (small calls: more CTAs
    // than tracklets, so that the machine is filled; the per-element arithmetic does not depend on the split)
    const int per_slab = (C / 4 + gridDim.y - 1) / gridDim.y;
    const int c4_lo = blockIdx.y * per_slab, c4_hi = min(C / 4, c4_lo + per_slab);
    for (int c4 = c4_lo + tid; c4 < c4_hi; c4 += kHeadThreads) {
        float4 tot = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int p = 0; p < kParts; ++p) {
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
            for (int s = 0; s < a.S; ++s) {
                const int r = s * kParts + p;
                const float w = s_att[r];
                const float4 v = __ldg(reinterpret_cast<const float4 *>(x + static_cast<size_t>(r) * C) + c4);
                acc.x = fmaf(v.x, w, acc.x); acc.y = fmaf(v.y, w, acc.y);
                acc.z = fmaf(v.z, w, acc.z); acc.w = fmaf(v.w, w, acc.w);
            }
            tot.x += acc.x; tot.y += acc.y; tot.z += acc.z; tot.w += acc.w;
        }
        const int c = c4 * 4;
        float *o = a.out + static_cast<size_t>(b) * a.ld_out + C + c;
        const float kP = static_cast<float>(kParts);
        o[0] = fmaf(__fdiv_rn(tot.x, kP), a.a_scale[c], a.a_shift[c]);
        o[1] = fmaf(__fdiv_rn(tot.y, kP), a.a_scale[c + 1], a.a_shift[c + 1]);
        o[2] = fmaf(__fdiv_rn(tot.z, kP), a.a_scale[c + 2], a.a_shift[c + 2]);
        o[3] = fmaf(__fdiv_rn(tot.w, kP), a.a_scale[c + 3], a.a_shift[c + 3]);
    }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
struct HeadWorkspace {
    float *x[2];
    __nv_bfloat16 *y_planes;
    float *z;                          // (batch, 4S, C) low-rank first layer: Q.W^T
    float *gt;                         // (batch, V, 4S) low-rank first layer: G.T
    float *y_unscale;                  // (batch) scaled fp16 modes
    float *row_sumsq;                  // (batch*V, sumsq_slots_of) partial row norms of the last layer's output
    size_t bytes;
};

// the first layer runs low-rank (G.X.W^T = (G.T).(Q.W^T) on the 4S quarter-strip rows) unless switched off or impossible
static bool lowrank_enabled(const agrl_head_params *p, int S) {
    return !p->lowrank_off && p->num_layers > 0 && p->channels % (2 * kHeadThreads) == 0 && S * kParts <= kMaxNodes;
}

// partial row sums of squares that the last layer's GEMM epilogue leaves for the attention: one per (column tile, half)
static int sumsq_slots_of(const agrl_head_params *p) {
    const int bn = p->split == AGRL_SPLIT_BF16X3 ? 128 : 256;
    return 2 * ((p->channels + bn - 1) / bn);
}

static HeadWorkspace carve_head(const agrl_head_params *p, void *ws, int64_t batch, int32_t S) {
    Carver c(ws);
    HeadWorkspace w;
    const size_t n = static_cast<size_t>(batch) * S * kParts * p->channels;
    w.x[0] = c.take<float>(n);
    w.x[1] = c.take<float>(n);
    w.y_planes = c.take<__nv_bfloat16>(static_cast<size_t>(planes_of(p->split)) * n);
    w.y_unscale = c.take<float>(static_cast<size_t>(batch));
    // no fewer than 32 floats per row, so that the workspace size of every split at C <= 2048 stays what callers allocate
    const int sumsq_room = sumsq_slots_of(p) > 32 ? sumsq_slots_of(p) : 32;
    w.row_sumsq = c.take<float>(static_cast<size_t>(batch) * S * kParts * sumsq_room);
    const bool lowrank = lowrank_enabled(p, S);
    w.z = lowrank ? c.take<float>(static_cast<size_t>(batch) * S * 4 * p->channels) : nullptr;
    w.gt = lowrank ? c.take<float>(static_cast<size_t>(batch) * S * kParts * S * 4) : nullptr;
    w.bytes = c.total();
    return w;
}

static int check_params(const agrl_head_params *p) {
    if (!p) return AGRL_E_INVALID;
    if (p->num_layers < 0 || p->num_layers > AGRL_HEAD_MAX_LAYERS) return AGRL_E_INVALID;
    if (p->split != AGRL_SPLIT_BF16X2 && p->split != AGRL_SPLIT_BF16X3 && p->split != AGRL_SPLIT_FP16X1 &&
        p->split != AGRL_SPLIT_FP16_E4M3) return AGRL_E_INVALID;
    if (p->channels < kChunk || p->channels % kChunk != 0) return AGRL_E_UNSUPPORTED;
    if (!p->use_pose && !p->learn_graph) return AGRL_E_INVALID;            // vmgn.py:92 assert
    if (p->pool_stages != 0 && (p->pool_stages < 2 || p->pool_stages > 12)) return AGRL_E_INVALID;
    if (p->maps_dtype != AGRL_MAPS_FP32 && p->maps_dtype != AGRL_MAPS_BF16 && p->maps_dtype != AGRL_MAPS_FP16) return AGRL_E_INVALID;
    return AGRL_OK;
}

static int launch_graph(const GraphArgs &ga, int64_t batch, cudaStream_t st) {
    // + two stages of raw node tiles: 109 KiB at V = 56, two CTAs per SM
    const int smem = kTcSmem + 2 * ga.V * 256;
    AGRL_CUDA_TRY(cudaFuncSetAttribute(graph_kernel_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, kTcSmem + 2 * kMaxNodes * 256));
    CUtensorMap map_x;
    int rc = gemm::make_rows_tensor_map_f32(&map_x, ga.x, batch, ga.V, ga.C, 64);
    if (rc) return rc;
    graph_kernel_tc<<<static_cast<unsigned>(batch), kTcThreads, smem, st>>>(map_x, ga);
    AGRL_LAUNCH_CHECK(st, "graph");
    return AGRL_OK;
}

}  // namespace agrl

using namespace agrl;

#ifdef AGRL_TIMELINE
extern "C" __attribute__((visibility("default"))) int agrl_timeline_set(long long *buf) {
    return cudaMemcpyToSymbol(g_timeline, &buf, sizeof(buf)) == cudaSuccess ? 0 : -3;
}
#endif

extern "C" size_t agrl_head_prepared_bytes(const agrl_head_params *p) {
    if (check_params(p)) return 0;
    return carve_prepared(p, nullptr).bytes;
}

extern "C" int agrl_head_prepare_dev(const agrl_head_params *p, void *prepared, size_t prepared_bytes, void *stream) {
    int rc = check_params(p);
    if (rc) return rc;
    if ((rc = agrl_device_ok())) return rc;
    Prepared pr = carve_prepared(p, prepared);
    if (!prepared || prepared_bytes < pr.bytes) return AGRL_E_WORKSPACE;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int C = p->channels;
    FoldArgs fa;
    fa.channels = C; fa.eps = p->bn_eps;
    const int nvec = p->num_layers + 2;
    for (int l = 0; l < p->num_layers; ++l) {
        if (!p->linear_weight[l] || !p->bn_weight[l] || !p->bn_bias[l] || !p->bn_mean[l] || !p->bn_var[l]) return AGRL_E_INVALID;
        fa.w[l] = p->bn_weight[l]; fa.b[l] = p->bn_bias[l]; fa.mean[l] = p->bn_mean[l]; fa.var[l] = p->bn_var[l];
        gemm::SplitArgs sa{p->linear_weight[l], C, pr.w_planes[l], nullptr, C, C, C, planes_of(p->split), 0};
        if (scaled_mode(p->split)) {
            float *slot = pr.w_scale + 4 * l;
            AGRL_CUDA_TRY(cudaMemsetAsync(slot, 0, 4 * sizeof(float), st));
            absmax_kernel<<<4 * kNumSMs, 256, 0, st>>>(p->linear_weight[l], static_cast<size_t>(C) * C, slot);
            AGRL_LAUNCH_CHECK(st, "absmax");
            w_scale_kernel<<<1, 1, 0, st>>>(slot);
            AGRL_LAUNCH_CHECK(st, "w_scale");
            sa.fp16 = 1; sa.prescale = slot;
            sa.fp8 = p->split == AGRL_SPLIT_FP16_E4M3;
        }
        if ((rc = gemm::launch_split_planes(sa, st))) return rc;
    }
    const float *const *extra[2] = {p->global_bn, p->att_bn};
    for (int e = 0; e < 2; ++e) {
        const int l = p->num_layers + e;
        for (int k = 0; k < 4; ++k) if (!extra[e][k]) return AGRL_E_INVALID;
        fa.w[l] = extra[e][0]; fa.b[l] = extra[e][1]; fa.mean[l] = extra[e][2]; fa.var[l] = extra[e][3];
    }
    for (int l = 0; l < nvec; ++l) { fa.scale[l] = pr.scale[l]; fa.shift[l] = pr.shift[l]; }
    fold_bn_kernel<<<dim3((C + 255) / 256, nvec), 256, 0, st>>>(fa);
    AGRL_LAUNCH_CHECK(st, "fold_bn");
    return AGRL_OK;
}

extern "C" size_t agrl_head_workspace_bytes(const agrl_head_params *p, int64_t batch, int32_t seq_len) {
    if (check_params(p) || batch < 0 || seq_len < 1) return 0;
    return carve_head(p, nullptr, batch, seq_len).bytes;
}

namespace agrl {

// pooling of `n` tracklets starting at tracklet `b0`, on stream `st`; maps of element type T
template <class T>
static int launch_pool(const agrl_head_params *p, const Prepared &pr, const HeadWorkspace &hwk, const T *x4_1,
                       const T *x4_2, float *out, int64_t ld_out, int64_t b0, int64_t n, int S, int hw, bool tma,
                       cudaStream_t st) {
    const int C = p->channels, V = S * kParts, L = p->num_layers;
    const size_t in_off = static_cast<size_t>(b0) * S * C * hw;
    float *nodes = hwk.x[0] + static_cast<size_t>(b0) * V * C;
    float *o = out + static_cast<size_t>(b0) * ld_out;
    AGRL_LAUNCH_BEGIN(st);
    if (p->maps_nhwc) {
        PoolArgs<T> pa{x4_1 + in_off, x4_2 + in_off, nodes, o, ld_out, pr.scale[L], pr.shift[L], S, C, hw};
        const dim3 grid((C / 4 + kHeadThreads - 1) / kHeadThreads, static_cast<unsigned>(n));
        pool_nhwc_kernel<T><<<grid, kHeadThreads, 0, st>>>(pa);
        AGRL_LAUNCH_CHECK(st, "pool");
        return AGRL_OK;
    }
    if (tma) {
        const int64_t units = n * (C / kTpCh);
        PoolTmaArgs<T> ta{x4_1 + in_off, x4_2 + in_off, nodes, o, ld_out, pr.scale[L], pr.shift[L], S, C,
                          p->pool_stages ? p->pool_stages : tp_default_stages<T>(), 0, static_cast<int>(units),
                          p->pool_no_l2_hint ? 0 : 1};
        const size_t smem = pool_tma_smem(S, ta.stages, tp_stage_bytes<T>());
        AGRL_CUDA_TRY(cudaFuncSetAttribute(pool_tma_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
        int64_t grid = static_cast<int64_t>(kNumSMs) * 2;                 // persistent, two small CTAs per SM
        if (grid > units) grid = units;
        pool_tma_kernel<T><<<static_cast<unsigned>(grid), kTpThreads, smem, st>>>(ta);
        AGRL_LAUNCH_CHECK(st, "pool");
        return AGRL_OK;
    }
    PoolArgs<T> pa{x4_1 + in_off, x4_2 + in_off, nodes, o, ld_out, pr.scale[L], pr.shift[L], S, C, hw};
    const size_t pool_smem = static_cast<size_t>(S) * kParts * kPoolCh * sizeof(float);
    const dim3 pgrid(C / kPoolCh, static_cast<unsigned>(n));
    // vector loads of four elements need the maps aligned to four elements
    const uintptr_t vec_align = 4 * sizeof(T) - 1;
    const bool vec = (hw == 128) && ((reinterpret_cast<uintptr_t>(x4_1) | reinterpret_cast<uintptr_t>(x4_2)) & vec_align) == 0;
    if (vec) pool_kernel<true, T><<<pgrid, kHeadThreads, pool_smem, st>>>(pa);
    else pool_kernel<false, T><<<pgrid, kHeadThreads, pool_smem, st>>>(pa);
    AGRL_LAUNCH_CHECK(st, "pool");
    return AGRL_OK;
}

// the maps' element type chosen at run time (agrl_head_params.maps_dtype; check_params has vetted it)
static int launch_pool_any(const agrl_head_params *p, const Prepared &pr, const HeadWorkspace &hwk, const void *x4_1,
                           const void *x4_2, float *out, int64_t ld_out, int64_t b0, int64_t n, int S, int hw, bool tma,
                           cudaStream_t st) {
    switch (p->maps_dtype) {
        case AGRL_MAPS_BF16:
            return launch_pool(p, pr, hwk, static_cast<const __nv_bfloat16 *>(x4_1), static_cast<const __nv_bfloat16 *>(x4_2),
                               out, ld_out, b0, n, S, hw, tma, st);
        case AGRL_MAPS_FP16:
            return launch_pool(p, pr, hwk, static_cast<const __half *>(x4_1), static_cast<const __half *>(x4_2),
                               out, ld_out, b0, n, S, hw, tma, st);
        default:
            return launch_pool(p, pr, hwk, static_cast<const float *>(x4_1), static_cast<const float *>(x4_2),
                               out, ld_out, b0, n, S, hw, tma, st);
    }
}

// one GEMM of a graph layer in the caller's operand mode; Epi is built by `make(fp8)` for the scaled modes
template <class EpiBf16, class EpiF16, class EpiF16E4>
static int launch_layer_gemm(int split, bool pair, const CUtensorMap &map_a, const CUtensorMap &map_w, int rows, int C,
                             const EpiBf16 &e2, const EpiF16 &e1, const EpiF16E4 &e4, cudaStream_t st) {
    switch (split) {
        case AGRL_SPLIT_FP16X1: return gemm::launch_split_gemm<1, 256, false>(map_a, map_w, rows, C, C, e1, st);
        case AGRL_SPLIT_FP16_E4M3:
            return pair ? gemm::launch_pair_gemm<2, 256, false>(map_a, map_w, rows, C, C, e4, st)
                        : gemm::launch_split_gemm<2, 256, false>(map_a, map_w, rows, C, C, e4, st);
        case AGRL_SPLIT_BF16X3: return gemm::launch_split_gemm<3, 128, false>(map_a, map_w, rows, C, C, e2, st);
        default: return gemm::launch_split_gemm<2, 256, false>(map_a, map_w, rows, C, C, e2, st);
    }
}

// graph layers + attention of `n` tracklets starting at tracklet `b0` (their nodes are in hwk.x[0])
static int launch_layers(const agrl_head_params *p, const Prepared &pr, HeadWorkspace hwk, const float *adj,
                         const uint64_t *masks, float *out,
                         int64_t ld_out, float *nodes_out, int64_t b0, int64_t n, int64_t batch, int S, cudaStream_t st) {
    const int C = p->channels, V = S * kParts, L = p->num_layers, P = planes_of(p->split);
    const int64_t rows = n * V, row0 = b0 * V, all_rows = batch * V;
    float *x[2] = {hwk.x[0] + row0 * C, hwk.x[1] + row0 * C};
    __nv_bfloat16 *y = hwk.y_planes + row0 * C;
    if (nodes_out) nodes_out += row0 * C;
    if (adj) adj += b0 * V * V;
    if (masks) masks += b0 * 3;
    int rc;
    const float *attn_sumsq = nullptr;
    int attn_slots = 0;
    CUtensorMap map_y, map_w;
    if (L > 0 && (rc = gemm::make_plane_tensor_map(&map_y, y, rows, C, P, gemm::BM, all_rows))) return rc;
    const int scaled = scaled_mode(p->split), fp8 = p->split == AGRL_SPLIT_FP16_E4M3;
    const int bn = p->split == AGRL_SPLIT_BF16X3 ? 128 : 256;
    const bool pair = fp8 && !p->gemm_no_pair;              // CTA pairs (cta_group::2): each CTA loads half of the W tile
    int cur = 0;
    for (int l = 0; l < L; ++l) {
        GraphArgs ga{x[cur], adj, masks, y, all_rows * C, V, C, P, p->use_pose, p->learn_graph, scaled, hwk.y_unscale + b0};
        ga.fp8 = fp8;
        float *dst = (l == L - 1 && nodes_out) ? nodes_out : x[cur ^ 1];
        if ((rc = gemm::make_plane_tensor_map(&map_w, pr.w_planes[l], C, C, P, pair ? bn / 2 : bn, C))) return rc;
        // Low-rank first layer: only layer 0 sees nodes that are T.(quarter strips)
        if (l == 0 && hwk.z) {
            const int S4 = S * 4;
            const int64_t qrows = n * S4, q_all = batch * S4;
            __nv_bfloat16 *yq = hwk.y_planes + b0 * S4 * C;
            float *z = hwk.z + b0 * S4 * C;
            ga.y_planes = yq; ga.plane_stride = q_all * C; ga.lowrank = 1; ga.gt = hwk.gt + b0 * V * S4;
            AGRL_LAUNCH_BEGIN(st);
            if ((rc = launch_graph(ga, n, st))) return rc;
            CUtensorMap map_q;
            if ((rc = gemm::make_plane_tensor_map(&map_q, yq, qrows, C, P, gemm::BM, q_all))) return rc;
            AGRL_LAUNCH_BEGIN(st);
            gemm::EpiPlainT<false> z2{z, C, nullptr, nullptr, S4};
            gemm::EpiPlainT<true> z1{z, C, hwk.y_unscale + b0, pr.w_scale + 4 * l + 1, S4};
            gemm::EpiPlainT<true, true> z4{z, C, hwk.y_unscale + b0, pr.w_scale + 4 * l + 1, S4};
            if ((rc = launch_layer_gemm(p->split, pair, map_q, map_w, static_cast<int>(qrows), C, z2, z1, z4, st))) return rc;
            MixArgs ma{x[cur], z, ga.gt, dst, pr.scale[l], pr.shift[l], V, S4, C, p->gamma, p->leaky_slope};
            AGRL_LAUNCH_BEGIN(st);
            if (S4 <= 32) graph_mix_kernel<32><<<dim3(C / (2 * kHeadThreads), static_cast<unsigned>(n)), kHeadThreads, 0, st>>>(ma);
            else graph_mix_kernel<kMixLdMax><<<dim3(C / (2 * kHeadThreads), static_cast<unsigned>(n)), kHeadThreads, 0, st>>>(ma);
            AGRL_LAUNCH_CHECK(st, "graph_mix");
            if (dst == nodes_out) x[cur ^ 1] = nodes_out;
            cur ^= 1;
            continue;
        }
        AGRL_LAUNCH_BEGIN(st);
        if ((rc = launch_graph(ga, n, st))) return rc;
        const int sumsq_slots = sumsq_slots_of(p);
        float *sumsq = (l == L - 1 && C % bn == 0) ? hwk.row_sumsq + row0 * sumsq_slots : nullptr;
        if (sumsq) { attn_sumsq = sumsq; attn_slots = sumsq_slots; }
        gemm::EpiGraphLayer e2{x[cur], pr.scale[l], pr.shift[l], dst, C, C, p->gamma, p->leaky_slope, nullptr, nullptr, V};
        gemm::EpiGraphLayerF16 e1{x[cur], pr.scale[l], pr.shift[l], dst, C, C, p->gamma, p->leaky_slope,
                                  hwk.y_unscale + b0, pr.w_scale + 4 * l + 1, V};
        gemm::EpiGraphLayerF16E4 e4{x[cur], pr.scale[l], pr.shift[l], dst, C, C, p->gamma, p->leaky_slope,
                                    hwk.y_unscale + b0, pr.w_scale + 4 * l + 1, V};
        e2.row_sumsq = e1.row_sumsq = e4.row_sumsq = sumsq;
        e2.sumsq_slots = e1.sumsq_slots = e4.sumsq_slots = sumsq ? sumsq_slots : 0;
        AGRL_LAUNCH_BEGIN(st);
        if ((rc = launch_layer_gemm(p->split, pair, map_y, map_w, static_cast<int>(rows), C, e2, e1, e4, st))) return rc;
        if (dst == nodes_out) x[cur ^ 1] = nodes_out;
        cur ^= 1;
    }
    if (L == 0 && nodes_out)
        AGRL_CUDA_TRY(cudaMemcpyAsync(nodes_out, x[0], sizeof(float) * rows * C, cudaMemcpyDeviceToDevice, st));
    AttnArgs aa{x[cur], out + static_cast<size_t>(b0) * ld_out, ld_out, pr.scale[L + 1], pr.shift[L + 1], S, C, attn_sumsq, attn_slots};
    AGRL_LAUNCH_BEGIN(st);
    // channel slabs per tracklet: 1 iteration per thread at C = 2048 with two slabs; more when the call is small
    int slabs = 1;
    if (attn_sumsq) { slabs = n >= 600 ? 2 : (n >= 300 ? 4 : 8); while (slabs > 1 && (C / 4) % slabs != 0) slabs >>= 1; }
    attn_kernel<<<dim3(static_cast<unsigned>(n), slabs), kHeadThreads, 0, st>>>(aa);
    AGRL_LAUNCH_CHECK(st, "attn");
    return AGRL_OK;
}

}  // namespace agrl

// Pipeline: pooling, then per layer graph kernel -> GEMM (-> mixing kernel for the low-rank first layer), attention; all on
// the caller's stream, no allocation, no synchronisation, no state outside the caller's buffers (re-entrant).  The
// maps are the only HBM-heavy input; every phase runs the board at its power limit (profiles/r2/energy_probe.log: the
// pooling kernel alone draws ~960 W while it streams at the HBM peak), so co-scheduling phases cannot shorten the pass
// -- the round-1 sub-batch / partition plumbing measured exactly that and is gone.
static int head_forward_impl(const agrl_head_params *p, const void *prepared,
                             const float *x4_1, const float *x4_2, const float *adj, const uint64_t *masks,
                             float *out, int64_t ld_out, float *nodes_out,
                             int64_t batch, int32_t S, int32_t h, int32_t w,
                             void *ws, size_t ws_bytes, void *stream) {
    int rc = check_params(p);
    if (rc) return rc;
    if (!prepared || !x4_1 || !x4_2 || !out || batch < 0 || S < 1 || h < 1 || w < 1) return AGRL_E_INVALID;
    if (p->use_pose && !adj && !masks) return AGRL_E_INVALID;
    const int C = p->channels, V = S * kParts, hw = h * w;
    if (ld_out < 2 * C) return AGRL_E_INVALID;
    if (V > kMaxNodes || h % 4 != 0) return AGRL_E_UNSUPPORTED;
    if ((rc = agrl_device_ok())) return rc;
    if (batch == 0) return AGRL_OK;
    HeadWorkspace hwk = carve_head(p, ws, batch, S);
    if (!ws || ws_bytes < hwk.bytes) return AGRL_E_WORKSPACE;
    Prepared pr = carve_prepared(p, const_cast<void *>(prepared));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (!p->use_pose) { adj = nullptr; masks = nullptr; }
    if (adj) masks = nullptr;

    // channels-last pooling loads four channels at once: maps aligned to four elements (16 B at fp32, 8 B at 16 bits);
    // the bulk copies need 16-byte aligned sources whatever the element size
    const uintptr_t maps_bits = reinterpret_cast<uintptr_t>(x4_1) | reinterpret_cast<uintptr_t>(x4_2);
    const uintptr_t vec_align = (p->maps_dtype == AGRL_MAPS_FP32 ? 16u : 8u) - 1u;
    if (p->maps_nhwc && (maps_bits & vec_align) != 0) return AGRL_E_UNSUPPORTED;
    const bool tma = !p->maps_nhwc && !p->pool_register_loads && hw == 128 && C % kTpCh == 0 && (maps_bits & 15u) == 0;
    constexpr int64_t kMaxPerLaunch = 32768;           // grid.y / int index limits of the per-tracklet kernels
    for (int64_t b0 = 0; b0 < batch; b0 += kMaxPerLaunch) {
        const int64_t n = batch - b0 < kMaxPerLaunch ? batch - b0 : kMaxPerLaunch;
        if ((rc = launch_pool_any(p, pr, hwk, x4_1, x4_2, out, ld_out, b0, n, S, hw, tma, st))) return rc;
        if ((rc = launch_layers(p, pr, hwk, adj, masks, out, ld_out, nodes_out, b0, n, batch, S, st))) return rc;
    }
    return AGRL_OK;
}

extern "C" int agrl_head_forward_dev(const agrl_head_params *p, const void *prepared,
                                     const float *x4_1, const float *x4_2, const float *adj,
                                     float *out, int64_t ld_out, float *nodes_out,
                                     int64_t batch, int32_t S, int32_t h, int32_t w,
                                     void *ws, size_t ws_bytes, void *stream) {
    return head_forward_impl(p, prepared, x4_1, x4_2, adj, nullptr, out, ld_out, nodes_out, batch, S, h, w, ws, ws_bytes, stream);
}

// same head, pose graph given as three membership masks per tracklet (pose.cu) instead of the dense matrix
extern "C" int agrl_head_forward_compact_dev(const agrl_head_params *p, const void *prepared,
                                             const float *x4_1, const float *x4_2, const uint64_t *part_masks,
                                             float *out, int64_t ld_out, float *nodes_out,
                                             int64_t batch, int32_t S, int32_t h, int32_t w,
                                             void *ws, size_t ws_bytes, void *stream) {
    return head_forward_impl(p, prepared, x4_1, x4_2, nullptr, part_masks, out, ld_out, nodes_out, batch, S, h, w, ws, ws_bytes, stream);
}

// ------------------------------------------------------------------------------------------------
// clip pooling for the `dense` / `skipdense` test sampling (SURVEY.md section 8f, row 2):
// train_vidreid_xent_htri.py:461-476 folds the clips of a tracklet into the batch, runs the model,
// then reduces the per-clip features with torch.mean(features, 0) or torch.max(features, 0).
// feats (tracklets, clips, dim) -> out (tracklets, dim); one thread per output element, clips in order.
// ------------------------------------------------------------------------------------------------
namespace agrl {
__global__ void clip_pool_kernel(const float *__restrict__ feats, float *__restrict__ out, int64_t tracklets,
                                 int clips, int64_t dim, int64_t ld_feat, int64_t ld_out, int mode) {
    const int64_t n = tracklets * dim;
    for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n;
         i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const int64_t t = i / dim, c = i % dim;
        const float *p = feats + t * clips * ld_feat + c;
        float acc = p[0];
        if (mode == AGRL_CLIP_POOL_MAX) {
            // torch.max propagates NaN
            for (int k = 1; k < clips; ++k) { const float v = p[k * ld_feat]; acc = (v > acc || v != v) ? v : acc; }
        } else {
            for (int k = 1; k < clips; ++k) acc = __fadd_rn(acc, p[k * ld_feat]);
            acc = __fdiv_rn(acc, static_cast<float>(clips));
        }
        out[t * ld_out + c] = acc;
    }
}
}  // namespace agrl

extern "C" int agrl_clip_pool_dev(const float *feats, int64_t ld_feat, int64_t tracklets, int64_t clips, int64_t dim,
                                  int mode, float *out, int64_t ld_out, void *stream) {
    if (!feats || !out || tracklets < 0 || clips < 1 || dim < 1 || ld_feat < dim || ld_out < dim) return AGRL_E_INVALID;
    if (mode != AGRL_CLIP_POOL_AVG && mode != AGRL_CLIP_POOL_MAX) return AGRL_E_INVALID;
    if (clips > (1 << 20)) return AGRL_E_UNSUPPORTED;
    int rc = agrl_device_ok();
    if (rc) return rc;
    if (tracklets == 0) return AGRL_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int64_t n = tracklets * dim;
    int64_t blocks = (n + 255) / 256;
    if (blocks > 8 * kNumSMs) blocks = 8 * kNumSMs;
    clip_pool_kernel<<<static_cast<unsigned>(blocks), 256, 0, st>>>(feats, out, tracklets, static_cast<int>(clips), dim,
                                                                   ld_feat, ld_out, mode);
    AGRL_LAUNCH_CHECK(st, "clip_pool");
    return AGRL_OK;
}

