// distance.cu -- query x gallery distance matrix (torchreid/metrics/distance.py:11-89) on tcgen05.
//
//   euclidean : out[i,j] = (|q_i|^2 + |g_j|^2) - 2 q_i.g_j      (no clamp, no sqrt; distance.py:70-72)
//   cosine    : out[i,j] = 1 - q^_i . g^_j,  x^ = x / max(|x|_2, 1e-12)   (distance.py:86-88)
//
// Pipeline: split.cu turns both operands into operand planes (planes.cuh; and norms / normalised rows) in one
// pass each, then one persistent tcgen05 GEMM (gemm_sm100.cuh) with the distance epilogue fused.
#include "gemm_sm100.cuh"
#include "planes.cuh"
#include "topk.cuh"

namespace agrl {

// One prepared operand: 16-bit planes [P][rows][K_pad], the per-row squared norms, the per-row 1 / scale (fp16 x 2).
struct Operand {
    __nv_bfloat16 *planes;
    float *sumsq, *unscale;
    size_t bytes;
};

static Operand carve_operand(void *buf, int64_t rows, int64_t dim, int split) {
    Carver c(buf);
    Operand o;
    o.planes = c.take<__nv_bfloat16>(static_cast<size_t>(planes::count(split)) * rows * gemm::pad_k(dim));
    o.sumsq = c.take<float>(rows);
    o.unscale = c.take<float>(rows);
    o.bytes = c.total();
    return o;
}

// q x (g_rows rows of the gallery planes, g_plane_rows rows apart) on the split's GEMM: one CTA per 128 x 128 tile (for
// fp16 x 2 the two-MMA k-step of gemm_sm100.cuh, kWideB; CTA pairs on 256 x 128 tiles were measured as well: 0.397
// against 0.383 ms at 1980 x 9330 x 4096 -- not kept).  make(mode) builds the epilogue of that mode.
template <class Make>
static int launch_distance_gemm(int split, const void *q_planes, int64_t num_q, const void *g_planes, int64_t g_rows,
                                int64_t g_plane_rows, int kp, Make make, cudaStream_t st) {
    return planes::with_distance_mode(split, [&](auto mode) {
        using M = decltype(mode);
        CUtensorMap map_q, map_g;
        int rc;
        if ((rc = gemm::make_plane_tensor_map(&map_q, q_planes, num_q, kp, M::kP, gemm::BM, num_q))) return rc;
        if ((rc = gemm::make_plane_tensor_map(&map_g, g_planes, g_rows, kp, M::kP, 128, g_plane_rows))) return rc;
        return gemm::launch_split_gemm<M::kP, 128, true>(map_q, map_g, static_cast<int>(num_q), static_cast<int>(g_rows), kp,
                                                         make(mode), st);
    });
}

static bool metric_ok(int metric) { return metric == AGRL_METRIC_EUCLIDEAN || metric == AGRL_METRIC_COSINE; }

}  // namespace agrl

using namespace agrl;

extern "C" size_t agrl_distance_operand_bytes(int64_t rows, int64_t dim, int split) {
    if (rows < 0 || dim < 1 || !planes::distance_ok(split)) return 0;
    return carve_operand(nullptr, rows, dim, split).bytes;
}

extern "C" int agrl_distance_prepare_operand_dev(const float *x, int64_t ld, int64_t rows, int64_t dim,
                                                 int metric, int split, void *operand, size_t operand_bytes,
                                                 void *stream) {
    if (!x || rows < 0 || dim < 1 || ld < dim || !metric_ok(metric) || !planes::distance_ok(split)) return AGRL_E_INVALID;
    if (rows > (1 << 30) || dim > (1 << 24)) return AGRL_E_UNSUPPORTED;
    int rc = agrl_device_ok();
    if (rc) return rc;
    Operand o = carve_operand(operand, rows, dim, split);
    if (!operand || operand_bytes < o.bytes) return AGRL_E_WORKSPACE;
    const int normalize = (metric == AGRL_METRIC_COSINE);
    gemm::SplitArgs sa{x, ld, o.planes, normalize ? nullptr : o.sumsq, rows, static_cast<int>(dim),
                       static_cast<int>(gemm::pad_k(dim)), split, normalize};
    sa.unscale = o.unscale;
    return gemm::launch_split_planes(sa, static_cast<cudaStream_t>(stream));
}

extern "C" int agrl_distance_prepared_dev(const void *q_operand, int64_t num_q, const void *g_operand, int64_t num_g,
                                          int64_t dim, int metric, int split, float *out, int64_t ld_out, void *stream) {
    if (!q_operand || !g_operand || !out || num_q < 0 || num_g < 0 || dim < 1 || ld_out < num_g) return AGRL_E_INVALID;
    if (!metric_ok(metric) || !planes::distance_ok(split)) return AGRL_E_INVALID;
    if (num_q > (1 << 30) || num_g > (1 << 30) || dim > (1 << 24)) return AGRL_E_UNSUPPORTED;
    int rc = agrl_device_ok();
    if (rc) return rc;
    if (num_q == 0 || num_g == 0) return AGRL_OK;
    Operand q = carve_operand(const_cast<void *>(q_operand), num_q, dim, split);
    Operand g = carve_operand(const_cast<void *>(g_operand), num_g, dim, split);
    return launch_distance_gemm(split, q.planes, num_q, g.planes, num_g, num_g, static_cast<int>(gemm::pad_k(dim)),
                                [&](auto mode) {
                                    return gemm::EpiDistanceT<decltype(mode)::kRowScaled>{q.sumsq, g.sumsq, out, ld_out, metric,
                                                                                          q.unscale, g.unscale};
                                }, static_cast<cudaStream_t>(stream));
}

extern "C" size_t agrl_distance_workspace_bytes(int64_t num_q, int64_t num_g, int64_t dim, int split) {
    if (num_q < 0 || num_g < 0 || dim < 1 || !planes::distance_ok(split)) return 0;
    return agrl_distance_operand_bytes(num_q, dim, split) + agrl_distance_operand_bytes(num_g, dim, split);
}

extern "C" int agrl_distance_dev(const float *q, int64_t ld_q, const float *g, int64_t ld_g,
                                 float *out, int64_t ld_out, int64_t num_q, int64_t num_g, int64_t dim,
                                 int metric, int split, void *ws, size_t ws_bytes, void *stream) {
    if (!q || !g || !out) return AGRL_E_INVALID;
    if (num_q < 0 || num_g < 0 || dim < 1 || ld_q < dim || ld_g < dim || ld_out < num_g) return AGRL_E_INVALID;
    if (!metric_ok(metric) || !planes::distance_ok(split)) return AGRL_E_INVALID;
    int rc = agrl_device_ok();
    if (rc) return rc;
    if (num_q == 0 || num_g == 0) return AGRL_OK;
    const size_t qb = agrl_distance_operand_bytes(num_q, dim, split), gb = agrl_distance_operand_bytes(num_g, dim, split);
    if (!ws || ws_bytes < qb + gb) return AGRL_E_WORKSPACE;
    char *qo = static_cast<char *>(ws), *go = qo + qb;
    if ((rc = agrl_distance_prepare_operand_dev(q, ld_q, num_q, dim, metric, split, qo, qb, stream))) return rc;
    if ((rc = agrl_distance_prepare_operand_dev(g, ld_g, num_g, dim, metric, split, go, gb, stream))) return rc;
    return agrl_distance_prepared_dev(qo, num_q, go, num_g, dim, metric, split, out, ld_out, stream);
}

// ------------------------------------------------------------------------------------------------
// Fused distance -> top-k (retrieval against a large gallery; SURVEY.md section 7 step 6, section 8d "ranking"):
// the (num_q x num_g) matrix is never materialised.  The gallery columns are processed in launches of growing width
// (384, then `growth` x what has been seen so far); the GEMM epilogue (EpiTopKT) appends every key below the row's
// threshold -- fixed during a launch -- to the row's candidate list, topk_compact_kernel keeps the K smallest and tightens
// the threshold.  With the columns in an order unrelated to the distances a launch adds about growth x K candidates per
// row (binomial); growth is chosen so that K + growth K + 6 sigma stays below the list capacity kTopkCap.  A list that
// would exceed it anyway (e.g. a gallery sorted by distance to the query) sets AGRL_ST_TOPK_OVERFLOW and the caller
// takes the unfused route (agrl_distance_prepared_dev + agrl_rank_mars_partial_dev) -- results never depend on the order.
// ------------------------------------------------------------------------------------------------
namespace agrl {

constexpr int kTopkCap = 1024;                // candidate slots per query row
constexpr int kTopkFirst = 384;               // columns of the first launch (threshold still open: all of them are kept)
constexpr int kTopkMaxGrowth = 8;
constexpr int kCompactThreads = 128;

struct TopkWorkspace {
    unsigned long long *tau, *cand;
    unsigned int *cnt;
    size_t bytes;
};

static TopkWorkspace carve_topk(void *ws, int64_t nq) {
    Carver c(ws);
    TopkWorkspace w;
    w.tau = c.take<unsigned long long>(nq);
    w.cnt = c.take<unsigned int>(nq);
    w.cand = c.take<unsigned long long>(static_cast<size_t>(nq) * kTopkCap);
    w.bytes = c.total();
    return w;
}

// one CTA per query: sort the occupied prefix of the candidate list, keep the K smallest, publish the threshold;
// last == 1: also write the final keys (ascending, all-ones = empty slot)
__global__ void __launch_bounds__(kCompactThreads)
topk_compact_kernel(TopkWorkspace w, int K, int last, uint64_t *keys_out, uint32_t *status) {
    __shared__ uint64_t s_keys[kTopkCap];
    const int q = blockIdx.x, tid = threadIdx.x;
    unsigned int cnt = w.cnt[q];
    if (cnt > static_cast<unsigned int>(kTopkCap)) {
        if (tid == 0) atomicOr(status, AGRL_ST_TOPK_OVERFLOW);
        cnt = kTopkCap;
    }
    unsigned long long *list = w.cand + static_cast<size_t>(q) * kTopkCap;
    int n2 = 2;
    while (n2 < static_cast<int>(cnt)) n2 <<= 1;
    for (int i = tid; i < n2; i += kCompactThreads) s_keys[i] = i < static_cast<int>(cnt) ? list[i] : kKeyMax;
    __syncthreads();
    bitonic_sort_u64<false>(s_keys, n2, tid, kCompactThreads);
    const int keep = static_cast<int>(cnt) < K ? static_cast<int>(cnt) : K;
    for (int i = tid; i < keep; i += kCompactThreads) list[i] = s_keys[i];
    if (last) for (int i = tid; i < K; i += kCompactThreads) keys_out[static_cast<size_t>(q) * K + i] = i < keep ? s_keys[i] : kKeyMax;
    if (tid == 0) {
        w.cnt[q] = keep;
        w.tau[q] = keep == K ? s_keys[K - 1] : kKeyMax;
    }
}

}  // namespace agrl

extern "C" size_t agrl_distance_topk_workspace_bytes(int64_t num_q) {
    if (num_q < 0) return 0;
    return carve_topk(nullptr, num_q).bytes;
}

extern "C" int agrl_distance_topk_dev(const void *q_operand, int64_t num_q, const void *g_operand, int64_t num_g,
                                      int64_t dim, int metric, int split, int64_t max_rank, int64_t index_offset,
                                      uint64_t *keys, uint32_t *status, void *ws, size_t ws_bytes, void *stream) {
    if (!q_operand || !g_operand || !keys || !status || num_q < 0 || num_g < 0 || dim < 1 || index_offset < 0) return AGRL_E_INVALID;
    if (!metric_ok(metric) || !planes::distance_ok(split) || max_rank < 1) return AGRL_E_INVALID;
    if (max_rank > 256 || num_q > (1 << 30) || dim > (1 << 24) || index_offset + num_g > 0xFFFFFFFFll) return AGRL_E_UNSUPPORTED;
    int rc = agrl_device_ok();
    if (rc) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    AGRL_CUDA_TRY(cudaMemsetAsync(status, 0, sizeof(uint32_t), st));
    if (num_q == 0) return AGRL_OK;
    TopkWorkspace w = carve_topk(ws, num_q);
    if (!ws || ws_bytes < w.bytes) return AGRL_E_WORKSPACE;
    const int K = static_cast<int>(max_rank), nq = static_cast<int>(num_q);
    AGRL_CUDA_TRY(cudaMemsetAsync(w.tau, 0xFF, sizeof(unsigned long long) * num_q, st));
    AGRL_CUDA_TRY(cudaMemsetAsync(w.cnt, 0, sizeof(unsigned int) * num_q, st));
    Operand q = carve_operand(const_cast<void *>(q_operand), num_q, dim, split);
    Operand g = carve_operand(const_cast<void *>(g_operand), num_g, dim, split);
    const int kp = static_cast<int>(gemm::pad_k(dim));
    int64_t c0 = 0;
    // expected candidates per row and launch: growth * K (+ the K kept ones); leave 30 % of the list for the spread
    int growth = static_cast<int>(0.7 * (kTopkCap - K) / K);
    growth = growth < 1 ? 1 : (growth > kTopkMaxGrowth ? kTopkMaxGrowth : growth);
    if (num_g == 0) {
        topk_compact_kernel<<<nq, kCompactThreads, 0, st>>>(w, K, 1, keys, status);
        AGRL_LAUNCH_CHECK(st, "topk_compact");
        return AGRL_OK;
    }
    while (c0 < num_g) {
        // the first launch may keep everything it sees (kTopkFirst <= capacity); later ones add ~growth * K per row
        int64_t width = c0 == 0 ? kTopkFirst : growth * c0;
        if (c0 + width > num_g || num_g - (c0 + width) < width / 8) width = num_g - c0;      // no tiny tail launch
        rc = launch_distance_gemm(split, q.planes, num_q, g.planes + c0 * kp, width, num_g, kp, [&](auto mode) {
            return gemm::EpiTopKT<decltype(mode)::kRowScaled>{q.sumsq, g.sumsq + c0, metric, w.tau, w.cnt, w.cand, kTopkCap,
                                                              static_cast<uint32_t>(index_offset + c0), q.unscale, g.unscale + c0};
        }, st);
        if (rc) return rc;
        c0 += width;
        topk_compact_kernel<<<nq, kCompactThreads, 0, st>>>(w, K, c0 >= num_g ? 1 : 0, keys, status);
        AGRL_LAUNCH_CHECK(st, "topk_compact");
    }
    return AGRL_OK;
}
