// qe.cu -- the mix step of alpha query expansion (FastReID fastreid/evaluation/query_expansion.py `aqe`).
//
// One iteration of AQE replaces every feature row by the mean of its k nearest neighbours' rows, each weighted by its
// cosine similarity to the power alpha.  The neighbour lists come from the existing path (prepared cosine operands,
// fused distance -> top-k, rank_lists_kernel); this file holds the only new device code, the weighted gather
//   out[r, :] = (sum_{j < k} powf(1 - dist[r, j], alpha) * feats[idx[r, j], :]) / k
// over rows x k x dim.  Each thread owns 4 consecutive columns (16-byte loads and stores when every row starts 16-byte
// aligned) or 1 column (any dim and row stride) of one row, so the sum over j runs in list order for every column and
// the result does not depend on the path or the launch shape.
#include "common.cuh"

namespace agrl {

constexpr int kQeThreads = 256;
constexpr int kQeChunk = kQeThreads;       // list entries staged in shared memory at a time (one per thread)
constexpr int kQeBatch = 4;                // gathers in flight per thread before their sums

struct QeMixArgs {
    const int64_t *idx;
    const float   *dist;
    int64_t        ld_list;
    int            k;
    const float   *feats;
    int64_t        ld_feat, num_feats, dim;
    float          alpha;
    float         *out;
    int64_t        ld_out;
};

template <int W> struct QeVec { float v[W]; };

template <int W>
__device__ __forceinline__ QeVec<W> qe_load(const float *p) {
    QeVec<W> r;
    if constexpr (W == 4) {
        const float4 t = __ldg(reinterpret_cast<const float4 *>(p));
        r.v[0] = t.x; r.v[1] = t.y; r.v[2] = t.z; r.v[3] = t.w;
    } else {
        r.v[0] = __ldg(p);
    }
    return r;
}

// Grid: x = row, y = tile of kQeThreads * W columns.  Every CTA of a row stages the row's list in chunks of kQeChunk
// entries (feature row, or -1 where the index is outside [0, num_feats); weight), then each thread sums its columns
// over the chunk in list order.
template <int W>
__global__ void __launch_bounds__(kQeThreads)
qe_mix_kernel(QeMixArgs a) {
    __shared__ int64_t s_row[kQeChunk];
    __shared__ float s_w[kQeChunk];
    const int64_t r = blockIdx.x;
    const int64_t c = (static_cast<int64_t>(blockIdx.y) * kQeThreads + threadIdx.x) * W;
    const bool active = c < a.dim;
    const int64_t *idx = a.idx + r * a.ld_list;
    const float *dist = a.dist + r * a.ld_list;
    const float *base = a.feats + c;
    float acc[W];
#pragma unroll
    for (int u = 0; u < W; ++u) acc[u] = 0.0f;
    for (int j0 = 0; j0 < a.k; j0 += kQeChunk) {
        const int n = min(kQeChunk, a.k - j0);
        if (static_cast<int>(threadIdx.x) < n) {
            const int64_t g = idx[j0 + threadIdx.x];
            s_row[threadIdx.x] = (g >= 0 && g < a.num_feats) ? g : -1;
            s_w[threadIdx.x] = powf(1.0f - dist[j0 + threadIdx.x], a.alpha);
        }
        __syncthreads();
        if (active) {
            for (int j = 0; j < n; j += kQeBatch) {
                QeVec<W> v[kQeBatch];
#pragma unroll
                for (int b = 0; b < kQeBatch; ++b) {
                    const int64_t g = (j + b < n) ? s_row[j + b] : -1;
                    if (g >= 0) {
                        v[b] = qe_load<W>(base + g * a.ld_feat);
                    } else {
#pragma unroll
                        for (int u = 0; u < W; ++u) v[b].v[u] = 0.0f;
                    }
                }
#pragma unroll
                for (int b = 0; b < kQeBatch; ++b) {
                    if (j + b < n && s_row[j + b] >= 0) {
                        const float w = s_w[j + b];
#pragma unroll
                        for (int u = 0; u < W; ++u) acc[u] = fmaf(w, v[b].v[u], acc[u]);
                    }
                }
            }
        }
        __syncthreads();
    }
    if (!active) return;
    const float kf = static_cast<float>(a.k);
    float *dst = a.out + r * a.ld_out + c;
    if constexpr (W == 4) {
        *reinterpret_cast<float4 *>(dst) = make_float4(acc[0] / kf, acc[1] / kf, acc[2] / kf, acc[3] / kf);
    } else {
        dst[0] = acc[0] / kf;
    }
}

}  // namespace agrl

using namespace agrl;

extern "C" int agrl_qe_mix_dev(const int64_t *idx, const float *dist, int64_t ld_list, int64_t rows, int64_t k,
                               const float *feats, int64_t ld_feat, int64_t num_feats, int64_t dim, float alpha,
                               float *out, int64_t ld_out, void *stream) {
    if (rows < 0 || num_feats < 0 || dim < 0 || k < 1) return AGRL_E_INVALID;
    if (ld_list < k || ld_feat < dim || ld_out < dim || !isfinite(alpha)) return AGRL_E_INVALID;
    if (rows > 0 && dim > 0 && (!idx || !dist || !out || (num_feats > 0 && !feats))) return AGRL_E_INVALID;
    if (rows > 0 && dim > 0 && num_feats > 0) {                // out must not overlap feats
        const char *f0 = reinterpret_cast<const char *>(feats);
        const char *f1 = reinterpret_cast<const char *>(feats + (num_feats - 1) * ld_feat + dim);
        const char *o0 = reinterpret_cast<const char *>(out);
        const char *o1 = reinterpret_cast<const char *>(out + (rows - 1) * ld_out + dim);
        if (o0 < f1 && f0 < o1) return AGRL_E_INVALID;
    }
    const bool vec = dim % 4 == 0 && ld_feat % 4 == 0 && ld_out % 4 == 0 &&
                     reinterpret_cast<uintptr_t>(feats) % 16 == 0 && reinterpret_cast<uintptr_t>(out) % 16 == 0;
    const int64_t cols = kQeThreads * (vec ? 4 : 1);
    const int64_t tiles = (dim + cols - 1) / cols;
    if (k > INT32_MAX || rows > INT32_MAX || tiles > 65535) return AGRL_E_UNSUPPORTED;
    int rc = agrl_device_ok();
    if (rc) return rc;
    if (rows == 0 || dim == 0) return AGRL_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    QeMixArgs a;
    a.idx = idx; a.dist = dist; a.ld_list = ld_list; a.k = static_cast<int>(k);
    a.feats = feats; a.ld_feat = ld_feat; a.num_feats = num_feats; a.dim = dim;
    a.alpha = alpha; a.out = out; a.ld_out = ld_out;
    const dim3 grid(static_cast<unsigned>(rows), static_cast<unsigned>(tiles));
    if (vec)
        qe_mix_kernel<4><<<grid, kQeThreads, 0, st>>>(a);
    else
        qe_mix_kernel<1><<<grid, kQeThreads, 0, st>>>(a);
    AGRL_LAUNCH_CHECK(st, "qe_mix");
    return AGRL_OK;
}
