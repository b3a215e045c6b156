// rerank.cu -- k-reciprocal re-ranking on the GPU (SURVEY.md section 8f, row 3).
//
// Reference: torchreid/utils/re_ranking.py:30-94 (Zhong et al., CVPR 2017), the optional step between the distance
// matrix and the ranking in test() (train_vidreid_xent_htri.py:523-527).  The reference works on dense N x N numpy
// matrices (N = num_q + num_g) with python loops over rows; the work is really sparse:
//
//   normalise   D[i,j] = orig[j,i]^2 / max_k orig[k,i]^2 over the block matrix [[qq, qg],[qg^T, gg]]   (:34-40)
//   rank        first k1+1 columns of every row in (value, index) order -- the stable top-K of topk.cuh       (:42)
//   expand      per row the k-reciprocal set, grown by the candidates' half-size sets that overlap it by more
//               than 2/3, sorted unique (<= (k1+1)(k1/2+2) entries), weights exp(-D) normalised to sum 1    (:48-67)
//   average     V_qe[i] = mean of the rows of i's first k2 neighbours (a merge of k2 sorted sparse rows)    (:69-74)
//   jaccard     per query the sum over shared columns of min(V[i,c], V[j,c]) through an inverted index of
//               the gallery rows, in ascending column order, then 1 - t/(2-t) and the lambda blend         (:76-91)
//
// The kernels work on a set of *local* rows: all num_q queries, then a contiguous run of gallery rows that starts at
// global gallery index goff.  Local row l is global row glob(l) = l (l < nq) or l + goff.  The single-device entry
// uses goff = 0 (local == global); the gallery-sharded entries (agrl_rerank_shard_*) give each rank its own gallery
// rows, so that D is held as (nq + n_own) x N rows and rank / V tables are exchanged between the three phases.
//
// Index work (ranks, sets) is exact; values are float32 with the reference's operation order (numpy's pairwise
// sum for the weight normalisation, rows added in rank order for the mean, columns in ascending order for the
// Jaccard sums).  The only departure is expf vs numpy's float32 exp (<= 2 ulp), so results agree to ~1e-6, not
// bit for bit.  One CTA / warp per row; no atomics on floating-point data, so runs are reproducible.
// NaN propagates as in numpy: a NaN in column c of the block matrix makes the column maximum NaN (np.max), so D row c
// is all NaN, and the Jaccard minimum of a NaN weight is NaN (np.minimum).
#include "topk.cuh"

namespace agrl {

__device__ __forceinline__ int glob_row(int l, int nq, int goff) { return l < nq ? l : l + goff; }

struct RerankGeom {
    const float *qg, *qq, *gg;
    int64_t ld_qg, ld_qq, ld_gg;
    int nq, ng, N;
    int goff;                          // local row l >= nq is global row l + goff
    int gcol0;                         // gallery index of gg's first column (gg may hold a column slab only)
    // element (r, c) of the block matrix [[qq, qg], [qg^T, gg]], global indices
    __device__ __forceinline__ float orig(int r, int c) const {
        if (r < nq) return c < nq ? qq[static_cast<size_t>(r) * ld_qq + c] : qg[static_cast<size_t>(r) * ld_qg + (c - nq)];
        return c < nq ? qg[static_cast<size_t>(c) * ld_qg + (r - nq)] : gg[static_cast<size_t>(r - nq) * ld_gg + (c - nq - gcol0)];
    }
};

// ---- column maxima of orig^2 (non-negative floats: unsigned order == float order) ----------------------------
// columns glob(l) of orig for local rows l in [row0, row1); colmax_bits is indexed by l.  A NaN square is kept as the
// canonical NaN 0x7fffffff, which beats +inf (0x7f800000) in the unsigned maximum: NaN propagates as in np.max.
__device__ __forceinline__ unsigned int colmax_bits_of(float sq) { return sq != sq ? 0x7fffffffu : __float_as_uint(sq); }

__global__ void rr_colmax_kernel(RerankGeom g, int row0, int row1, unsigned int *colmax_bits) {
    __shared__ unsigned int part[8][33];
    const int l = row0 + blockIdx.x * 32 + threadIdx.x;
    const int r0 = blockIdx.y * 256;
    unsigned int m = 0u;
    if (l < row1) {
        const int c = glob_row(l, g.nq, g.goff);
        const int r1 = min(r0 + 256, g.N);
        for (int r = r0 + threadIdx.y; r < r1; r += 8) {
            const float v = g.orig(r, c);
            m = max(m, colmax_bits_of(__fmul_rn(v, v)));
        }
    }
    part[threadIdx.y][threadIdx.x] = m;
    __syncthreads();
    if (threadIdx.y == 0 && l < row1) {
#pragma unroll
        for (int k = 1; k < 8; ++k) m = max(m, part[k][threadIdx.x]);
        atomicMax(colmax_bits + l, m);
    }
}

// ---- D[l][j] = orig[j][glob(l)]^2 / colmax[l] for local rows l in [row0, row1): tiled transpose -------------------
__global__ void rr_normalise_kernel(RerankGeom g, int row0, int row1, const float *colmax, float *D) {
    __shared__ float tile[32][33];
    const int i0 = row0 + blockIdx.y * 32, j0 = blockIdx.x * 32;
    for (int k = threadIdx.y; k < 32; k += 8) {                 // read orig[j0+k][glob(i0+tx)]: coalesced along i
        const int j = j0 + k, i = i0 + threadIdx.x;
        float v = 0.f;
        if (j < g.N && i < row1) { v = g.orig(j, glob_row(i, g.nq, g.goff)); v = __fmul_rn(v, v); }
        tile[k][threadIdx.x] = v;
    }
    __syncthreads();
    for (int k = threadIdx.y; k < 32; k += 8) {                 // write D[i0+k][j0+tx]
        const int i = i0 + k, j = j0 + threadIdx.x;
        if (i < row1 && j < g.N) D[static_cast<size_t>(i) * g.N + j] = __fdiv_rn(tile[threadIdx.x][k], colmax[i]);
    }
}

// ---- initial ranking: first K columns of every row (local rows row0 + blockIdx.x), ties by index ------------------
__global__ void __launch_bounds__(kRankThreads)
rr_topk_kernel(const float *D, int N, int K, int buf_len, int row0, int32_t *rank) {
    extern __shared__ __align__(16) unsigned char rr_smem[];
    uint64_t *buf = reinterpret_cast<uint64_t *>(rr_smem);
    __shared__ int s_cnt;
    __shared__ unsigned long long s_thr;
    const int i = row0 + blockIdx.x, tid = threadIdx.x;
    if (tid == 0) { s_cnt = 0; s_thr = kKeyMax; }
    __syncthreads();
    const int valid = select_topk(D + static_cast<size_t>(i) * N, N, K, buf_len, buf, &s_cnt, &s_thr, tid);
    for (int n = tid; n < K; n += kRankThreads)
        rank[static_cast<size_t>(i) * K + n] = n < valid ? static_cast<int32_t>(static_cast<uint32_t>(buf[n])) : -1;
}

// numpy's pairwise float32 summation of a contiguous array (np.sum, re_ranking.py:67)
__device__ float np_pairwise_sum(const float *a, int n) {
    if (n < 8) {
        float res = 0.f;
        for (int i = 0; i < n; ++i) res = __fadd_rn(res, a[i]);
        return res;
    }
    if (n <= 128) {
        float r[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) r[k] = a[k];
        int i;
        for (i = 8; i < n - (n % 8); i += 8)
#pragma unroll
            for (int k = 0; k < 8; ++k) r[k] = __fadd_rn(r[k], a[i + k]);
        float res = __fadd_rn(__fadd_rn(__fadd_rn(r[0], r[1]), __fadd_rn(r[2], r[3])),
                              __fadd_rn(__fadd_rn(r[4], r[5]), __fadd_rn(r[6], r[7])));
        for (; i < n; ++i) res = __fadd_rn(res, a[i]);
        return res;
    }
    int n2 = n / 2;
    n2 -= n2 % 8;
    return __fadd_rn(np_pairwise_sum(a, n2), np_pairwise_sum(a + n2, n - n2));
}

// ---- k-reciprocal expansion + weights: one warp per local row ---------------------------------------------------
// rank: (N, K) with K >= k1 + 1, all global rows; entries < 0 mean "row shorter than K" (N < K).
// D, idx, val, cnt: local rows [0, rows).
struct ExpandArgs {
    const float *D;
    const int32_t *rank;
    int N, K, k1p, half;               // k1p = k1 + 1, half = round(k1 / 2) + 1 (both clipped to N)
    int cap;                           // capacity of a sparse row
    int32_t *idx; float *val; int32_t *cnt;
    int rows, nq, goff;                // local rows and their global indices (glob_row)
};

constexpr int kExpandWarps = 4;

// does row `r` hold `target` among its first `k` ranked columns?
__device__ __forceinline__ bool in_first(const int32_t *rank, int K, int r, int k, int target) {
    const int32_t *p = rank + static_cast<size_t>(r) * K;
    bool hit = false;
    for (int t = 0; t < k; ++t) hit |= (p[t] == target);
    return hit;
}

__global__ void __launch_bounds__(32 * kExpandWarps)
rr_expand_kernel(ExpandArgs a) {
    extern __shared__ __align__(16) unsigned char rr_smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int i = blockIdx.x * kExpandWarps + warp;
    // per warp: candidate list (with duplicates, <= cap), then reused for sorted keys; weights
    uint64_t *keys = reinterpret_cast<uint64_t *>(rr_smem) + static_cast<size_t>(warp) * a.cap;
    float *w = reinterpret_cast<float *>(reinterpret_cast<uint64_t *>(rr_smem) + static_cast<size_t>(kExpandWarps) * a.cap) +
               static_cast<size_t>(warp) * a.cap;
    __shared__ int32_t s_recip[kExpandWarps][32];
    if (i >= a.rows) return;
    const int gi = glob_row(i, a.nq, a.goff);
    const int32_t *my = a.rank + static_cast<size_t>(gi) * a.K;

    // k-reciprocal neighbours (:50-53), in rank order
    int f = lane < a.k1p ? my[lane] : -1;
    const bool is_recip = f >= 0 && in_first(a.rank, a.K, f, a.k1p, gi);
    const unsigned rmask = __ballot_sync(0xffffffffu, is_recip);
    const int n_recip = __popc(rmask);
    if (is_recip) s_recip[warp][__popc(rmask & ((1u << lane) - 1u))] = f;
    __syncwarp();
    int n = 0;                                                    // entries in keys[] (low 32 bits = column)
    if (lane < n_recip) keys[lane] = static_cast<uint32_t>(s_recip[warp][lane]);
    n = n_recip;
    __syncwarp();
    // candidates' half-size reciprocal sets (:55-63)
    for (int t = 0; t < n_recip; ++t) {
        const int cand = s_recip[warp][t];
        const int32_t *cr = a.rank + static_cast<size_t>(cand) * a.K;
        const int x = lane < a.half ? cr[lane] : -1;
        const bool in_cr = x >= 0 && in_first(a.rank, a.K, x, a.half, cand);
        const unsigned cmask = __ballot_sync(0xffffffffu, in_cr);
        const int len_cr = __popc(cmask);
        bool shared_with_recip = false;
        if (in_cr) for (int u = 0; u < n_recip; ++u) shared_with_recip |= (s_recip[warp][u] == x);
        const int inter = __popc(__ballot_sync(0xffffffffu, shared_with_recip));
        if (static_cast<double>(inter) > (2.0 / 3.0) * static_cast<double>(len_cr)) {      // :62, python float compare
            if (in_cr) keys[n + __popc(cmask & ((1u << lane) - 1u))] = static_cast<uint32_t>(x);
            n += len_cr;
        }
        __syncwarp();
    }
    // np.unique: sort, drop duplicates (:65)
    int n2 = 2;
    while (n2 < n) n2 <<= 1;
    for (int t = n + lane; t < n2; t += 32) keys[t] = kKeyMax;
    __syncwarp();
    bitonic_sort_u64<true>(keys, n2, lane, 32);
    int out_n = 0;
    int32_t *oidx = a.idx + static_cast<size_t>(i) * a.cap;
    for (int base = 0; base < n; base += 32) {
        const int t = base + lane;
        const bool keep = t < n && (t == 0 || keys[t] != keys[t - 1]);
        const unsigned km = __ballot_sync(0xffffffffu, keep);
        if (keep) {
            const int pos = out_n + __popc(km & ((1u << lane) - 1u));
            const int col = static_cast<int>(static_cast<uint32_t>(keys[t]));
            oidx[pos] = col;
            w[pos] = expf(-a.D[static_cast<size_t>(i) * a.N + col]);                      // :66
        }
        out_n += __popc(km);
    }
    __syncwarp();
    float total = 0.f;
    if (lane == 0) total = np_pairwise_sum(w, out_n);
    total = __shfl_sync(0xffffffffu, total, 0);
    float *oval = a.val + static_cast<size_t>(i) * a.cap;
    for (int t = lane; t < out_n; t += 32) oval[t] = __fdiv_rn(w[t], total);                  // :67
    if (lane == 0) a.cnt[i] = out_n;
}

// ---- query expansion: V_qe[i] = mean over i's first k2 neighbours' rows (:69-74) --------------------------------
struct AverageArgs {
    const int32_t *rank; int N, K, k2;
    const int32_t *idx; const float *val; const int32_t *cnt; int cap;          // input rows: all N, global
    int32_t *oidx; float *oval; int32_t *ocnt; int ocap;                        // output rows: local
    int sort_len;                                                               // power of two >= k2 * cap
    int nq, goff;                                                               // local row -> global (glob_row)
};

constexpr int kAvgThreads = 128;

__global__ void __launch_bounds__(kAvgThreads)
rr_average_kernel(AverageArgs a) {
    extern __shared__ __align__(16) unsigned char rr_smem[];
    uint64_t *keys = reinterpret_cast<uint64_t *>(rr_smem);                     // (col << 35) | (slot << 32) | value bits
    __shared__ int s_n, s_heads[kAvgThreads / 32], s_rows;
    const int i = blockIdx.x, tid = threadIdx.x;
    if (tid == 0) { s_n = 0; s_rows = 0; }
    __syncthreads();
    const int32_t *my = a.rank + static_cast<size_t>(glob_row(i, a.nq, a.goff)) * a.K;
    int rows = 0;
    for (int r = 0; r < a.k2; ++r) {
        const int nb = my[r];
        if (nb < 0) break;
        ++rows;
        const int c = a.cnt[nb];
        __shared__ int s_base;
        if (tid == 0) { s_base = s_n; s_n += c; }
        __syncthreads();
        for (int t = tid; t < c; t += kAvgThreads) {
            const uint64_t col = static_cast<uint32_t>(a.idx[static_cast<size_t>(nb) * a.cap + t]);
            keys[s_base + t] = (col << 35) | (static_cast<uint64_t>(r) << 32) |
                               __float_as_uint(a.val[static_cast<size_t>(nb) * a.cap + t]);
        }
        __syncthreads();
    }
    const int n = s_n;
    int n2 = 2;
    while (n2 < n) n2 <<= 1;
    for (int t = n + tid; t < n2; t += kAvgThreads) keys[t] = kKeyMax;
    __syncthreads();
    bitonic_sort_u64<false>(keys, n2, tid, kAvgThreads);
    // one output per distinct column: rows are added in rank order, absent rows contribute +0 (exact), then / rows
    const float denom = static_cast<float>(rows);
    int out_n = 0;
    for (int base = 0; base < n; base += kAvgThreads) {
        const int t = base + tid;
        const bool head = t < n && (t == 0 || (keys[t] >> 35) != (keys[t - 1] >> 35));
        const unsigned hm = __ballot_sync(0xffffffffu, head);
        if ((tid & 31) == 0) s_heads[tid >> 5] = __popc(hm);
        __syncthreads();
        int pos = out_n;
        for (int wv = 0; wv < (tid >> 5); ++wv) pos += s_heads[wv];
        pos += __popc(hm & ((1u << (tid & 31)) - 1u));
        if (head) {
            float acc = 0.f;
            const uint64_t col = keys[t] >> 35;
            for (int u = t; u < n && (keys[u] >> 35) == col; ++u)
                acc = __fadd_rn(acc, __uint_as_float(static_cast<uint32_t>(keys[u])));
            a.oidx[static_cast<size_t>(i) * a.ocap + pos] = static_cast<int32_t>(col);
            a.oval[static_cast<size_t>(i) * a.ocap + pos] = __fdiv_rn(acc, denom);
        }
        int total = 0;
        for (int wv = 0; wv < kAvgThreads / 32; ++wv) total += s_heads[wv];
        out_n += total;
        __syncthreads();
    }
    if (tid == 0) a.ocnt[i] = out_n;
}

// ---- inverted index over the gallery rows (:76-78): sparse rows row0 + blockIdx.x are gallery columns blockIdx.x --
struct SparseRows { const int32_t *idx; const float *val; const int32_t *cnt; int cap; };

__global__ void rr_inv_count_kernel(SparseRows v, int row0, int32_t *col_cnt) {
    const int j = row0 + blockIdx.x;
    const int c = v.cnt[j];
    for (int t = threadIdx.x; t < c; t += blockDim.x) atomicAdd(col_cnt + v.idx[static_cast<size_t>(j) * v.cap + t], 1);
}

// exclusive scan of n counts by one CTA of 1024 threads
__global__ void __launch_bounds__(1024)
rr_scan_kernel(const int32_t *cnt, int n, int32_t *off) {
    __shared__ int s_part[1024];
    const int tid = threadIdx.x;
    const int per = (n + 1023) / 1024;
    const int lo = min(tid * per, n), hi = min(lo + per, n);
    int s = 0;
    for (int t = lo; t < hi; ++t) s += cnt[t];
    s_part[tid] = s;
    __syncthreads();
    for (int d = 1; d < 1024; d <<= 1) {
        const int v = tid >= d ? s_part[tid - d] : 0;
        __syncthreads();
        s_part[tid] += v;
        __syncthreads();
    }
    int run = s_part[tid] - s;
    for (int t = lo; t < hi; ++t) { off[t] = run; run += cnt[t]; }
    if (tid == 1023) off[n] = s_part[1023];
}

__global__ void rr_inv_fill_kernel(SparseRows v, int row0, const int32_t *col_off, int32_t *col_cur,
                                   int32_t *inv_row, float *inv_val) {
    const int j = row0 + blockIdx.x;
    const int c = v.cnt[j];
    for (int t = threadIdx.x; t < c; t += blockDim.x) {
        const int col = v.idx[static_cast<size_t>(j) * v.cap + t];
        const int pos = col_off[col] + atomicAdd(col_cur + col, 1);      // order inside a column is irrelevant:
        inv_row[pos] = blockIdx.x;                                       // its entries touch distinct gallery rows
        inv_val[pos] = v.val[static_cast<size_t>(j) * v.cap + t];
    }
}

// ---- Jaccard distance + blend: one CTA per query (:80-91) ------------------------------------------------------------
// v rows 0..nq are the queries; the output block has ng columns, blended with D[i][dcol0 + j] (D row stride N)
struct JaccardArgs {
    SparseRows v;
    const int32_t *col_off, *inv_row; const float *inv_val;
    const float *D; int dcol0, ng, N;
    float keep, lam;                   // (float)(1 - lambda), (float)lambda
    float *out; int64_t ld_out;
};

__global__ void __launch_bounds__(kRankThreads)
rr_jaccard_kernel(JaccardArgs a) {
    extern __shared__ __align__(16) unsigned char rr_smem[];
    float *t_min = reinterpret_cast<float *>(rr_smem);            // [ng]
    const int i = blockIdx.x, tid = threadIdx.x;
    for (int j = tid; j < a.ng; j += kRankThreads) t_min[j] = 0.f;
    __syncthreads();
    const int n = a.v.cnt[i];
    for (int t = 0; t < n; ++t) {                                  // columns in ascending order, as the reference adds them
        const int c = a.v.idx[static_cast<size_t>(i) * a.v.cap + t];
        const float vi = a.v.val[static_cast<size_t>(i) * a.v.cap + t];
        const int lo = a.col_off[c], hi = a.col_off[c + 1];
        for (int e = lo + tid; e < hi; e += kRankThreads) {
            const int j = a.inv_row[e];
            const float vj = a.inv_val[e];                        // np.minimum: NaN if either is NaN
            t_min[j] = __fadd_rn(t_min[j], (vi != vi || vj != vj) ? __uint_as_float(0x7fffffffu) : fminf(vi, vj));
        }
        __syncthreads();
    }
    const float *Drow = a.D + static_cast<size_t>(i) * a.N + a.dcol0;
    for (int j = tid; j < a.ng; j += kRankThreads) {
        const float tm = t_min[j];
        const float jac = __fsub_rn(1.0f, __fdiv_rn(tm, __fsub_rn(2.0f, tm)));
        a.out[static_cast<size_t>(i) * a.ld_out + j] = __fadd_rn(__fmul_rn(jac, a.keep), __fmul_rn(Drow[j], a.lam));
    }
}

// ---- workspace ------------------------------------------------------------------------------------------------------
static int round_half_even_half(int k1) {          // int(np.around(k1 / 2.))
    return (k1 % 2 == 0) ? k1 / 2 : ((k1 / 2) % 2 == 0 ? k1 / 2 : k1 / 2 + 1);
}
static int pow2_at_least(int n) { int p = 2; while (p < n) p <<= 1; return p; }

struct RerankWs {
    unsigned int *colmax;
    float *D;
    int32_t *rank;
    int32_t *v1_idx; float *v1_val; int32_t *v1_cnt;
    int32_t *vq_idx; float *vq_val; int32_t *vq_cnt;
    int32_t *col_cnt, *col_off, *col_cur;
    int32_t *inv_row; float *inv_val;
    int K, cap1, capq;
    size_t bytes;
};

// rows: local rows of D (all N on one device); n_inv: gallery rows of the inverted index; own_tables: the rank table
// and the expansion rows live in the workspace (single device) rather than in caller buffers (sharded)
static RerankWs carve_rerank(void *buf, int64_t rows, int64_t N, int64_t n_inv, int k1, int k2, bool own_tables) {
    Carver c(buf);
    RerankWs w;
    const size_t R = static_cast<size_t>(rows), T = own_tables ? static_cast<size_t>(N) : 0;
    const int half = round_half_even_half(k1) + 1;
    w.K = (k1 + 1 > k2) ? k1 + 1 : k2;
    w.cap1 = pow2_at_least((k1 + 1) * (half + 1));
    w.capq = (k2 == 1) ? w.cap1 : k2 * (k1 + 1) * (half + 1);
    w.colmax = c.take<unsigned int>(R);
    w.D = c.take<float>(R * N);
    w.rank = c.take<int32_t>(T * w.K);
    w.v1_idx = c.take<int32_t>(T * w.cap1); w.v1_val = c.take<float>(T * w.cap1); w.v1_cnt = c.take<int32_t>(T);
    w.vq_idx = c.take<int32_t>(R * w.capq); w.vq_val = c.take<float>(R * w.capq); w.vq_cnt = c.take<int32_t>(R);
    w.col_cnt = c.take<int32_t>(N + 1); w.col_off = c.take<int32_t>(N + 1); w.col_cur = c.take<int32_t>(N + 1);
    w.inv_row = c.take<int32_t>(static_cast<size_t>(n_inv) * w.capq); w.inv_val = c.take<float>(static_cast<size_t>(n_inv) * w.capq);
    w.bytes = c.total();
    return w;
}

static int rerank_args_ok(int64_t nq, int64_t ng, int64_t k1, int64_t k2) {
    if (nq < 1 || ng < 1 || k1 < 1 || k2 < 1) return AGRL_E_INVALID;
    if (k1 > 30 || k2 > 8) return AGRL_E_UNSUPPORTED;                    // 31 forward neighbours fit one warp
    if (nq + ng > 46000 || ng > 50000) return AGRL_E_UNSUPPORTED;        // int32 positions in D, t_min in shared memory
    return AGRL_OK;
}

// Per-rank limits of the sharded form.  Positions into D are 64-bit; the column-maximum grid has (N + 255) / 256 rows
// (<= 65535), t_min holds n_own floats in shared memory, and the inverted index (<= n_own * k2 * 527 entries) has
// int32 offsets.
constexpr int64_t kShardMaxN = 16000000;
constexpr int64_t kShardMaxOwn = 50000;

static int shard_args_ok(int64_t nq, int64_t ng, int64_t n_own, int64_t k1, int64_t k2) {
    if (nq < 1 || ng < 1 || n_own < 0 || n_own > ng || k1 < 1 || k2 < 1) return AGRL_E_INVALID;
    if (k1 > 30 || k2 > 8) return AGRL_E_UNSUPPORTED;
    if (n_own > kShardMaxOwn || nq + ng > kShardMaxN) return AGRL_E_UNSUPPORTED;
    return AGRL_OK;
}

// ---- the three stages, shared by the single-device and the sharded entries -----------------------------------------
// D rows and the initial ranking of local rows [row0, row1); rank is indexed by local row, row stride K
static int launch_rows(const RerankGeom &g, int row0, int row1, int K, unsigned int *colmax, float *D, int32_t *rank,
                       cudaStream_t st) {
    const int n = row1 - row0, N = g.N;
    if (n == 0) return AGRL_OK;
    AGRL_CUDA_TRY(cudaMemsetAsync(colmax + row0, 0, sizeof(unsigned int) * n, st));
    rr_colmax_kernel<<<dim3((n + 31) / 32, (N + 255) / 256), dim3(32, 8), 0, st>>>(g, row0, row1, colmax);
    AGRL_LAUNCH_CHECK(st, "rr_colmax");
    rr_normalise_kernel<<<dim3((N + 31) / 32, (n + 31) / 32), dim3(32, 8), 0, st>>>(g, row0, row1,
                                                                                    reinterpret_cast<const float *>(colmax), D);
    AGRL_LAUNCH_CHECK(st, "rr_normalise");
    int buf_len = pow2_at_least(2 * K);
    if (buf_len < 2 * kMarsTile) buf_len = 2 * kMarsTile;
    rr_topk_kernel<<<n, kRankThreads, static_cast<size_t>(buf_len) * 8, st>>>(D, N, K, buf_len, row0, rank);
    AGRL_LAUNCH_CHECK(st, "rr_topk");
    return AGRL_OK;
}

// k-reciprocal rows of the local rows [0, rows) from the full rank table
static int launch_expand(const float *D, const int32_t *rank, int N, int K, int k1, int rows, int nq, int goff,
                         int cap1, int32_t *idx, float *val, int32_t *cnt, cudaStream_t st) {
    if (rows == 0) return AGRL_OK;
    const int half = round_half_even_half(k1) + 1;
    ExpandArgs ea{D, rank, N, K, k1 + 1 < N ? k1 + 1 : N, half < N ? half : N, cap1, idx, val, cnt, rows, nq, goff};
    const size_t esmem = static_cast<size_t>(kExpandWarps) * cap1 * (8 + 4);
    AGRL_CUDA_TRY(cudaFuncSetAttribute(rr_expand_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(esmem)));
    rr_expand_kernel<<<(rows + kExpandWarps - 1) / kExpandWarps, 32 * kExpandWarps, esmem, st>>>(ea);
    AGRL_LAUNCH_CHECK(st, "rr_expand");
    return AGRL_OK;
}

// query expansion of the local rows, inverted index over the n_own local gallery rows, Jaccard + blend of every query
// against them.  rank and v1 hold all N rows (global); D and the workspace's vq rows are local.
static int launch_finish(const RerankWs &w, const int32_t *rank, SparseRows v1, int N, int nq, int goff, int n_own,
                         int k2, double lambda_value, float *out, int64_t ld_out, cudaStream_t st) {
    const int rows = nq + n_own;
    SparseRows v = v1;
    int inv_row0 = nq + goff;
    if (k2 != 1) {
        const int sort_len = pow2_at_least(k2 * w.cap1);
        AverageArgs aa{rank, N, w.K, k2, v1.idx, v1.val, v1.cnt, v1.cap,
                       w.vq_idx, w.vq_val, w.vq_cnt, w.capq, sort_len, nq, goff};
        const size_t asmem = static_cast<size_t>(sort_len) * 8;
        AGRL_CUDA_TRY(cudaFuncSetAttribute(rr_average_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(asmem)));
        rr_average_kernel<<<rows, kAvgThreads, asmem, st>>>(aa);
        AGRL_LAUNCH_CHECK(st, "rr_average");
        v = SparseRows{w.vq_idx, w.vq_val, w.vq_cnt, w.capq};
        inv_row0 = nq;
    }
    if (n_own == 0) return AGRL_OK;

    AGRL_CUDA_TRY(cudaMemsetAsync(w.col_cnt, 0, sizeof(int32_t) * (N + 1), st));
    AGRL_CUDA_TRY(cudaMemsetAsync(w.col_cur, 0, sizeof(int32_t) * (N + 1), st));
    rr_inv_count_kernel<<<n_own, 128, 0, st>>>(v, inv_row0, w.col_cnt);
    AGRL_LAUNCH_CHECK(st, "rr_inv_count");
    rr_scan_kernel<<<1, 1024, 0, st>>>(w.col_cnt, N, w.col_off);
    AGRL_LAUNCH_CHECK(st, "rr_scan");
    rr_inv_fill_kernel<<<n_own, 128, 0, st>>>(v, inv_row0, w.col_off, w.col_cur, w.inv_row, w.inv_val);
    AGRL_LAUNCH_CHECK(st, "rr_inv_fill");

    JaccardArgs ja{v, w.col_off, w.inv_row, w.inv_val, w.D, nq + goff, n_own, N,
                   static_cast<float>(1.0 - lambda_value), static_cast<float>(lambda_value), out, ld_out};
    const size_t jsmem = static_cast<size_t>(n_own) * 4;
    AGRL_CUDA_TRY(cudaFuncSetAttribute(rr_jaccard_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(jsmem)));
    rr_jaccard_kernel<<<nq, kRankThreads, jsmem, st>>>(ja);
    AGRL_LAUNCH_CHECK(st, "rr_jaccard");
    return AGRL_OK;
}

}  // namespace agrl

using namespace agrl;

extern "C" size_t agrl_rerank_workspace_bytes(int64_t num_q, int64_t num_g, int64_t k1, int64_t k2) {
    if (rerank_args_ok(num_q, num_g, k1, k2)) return 0;
    return carve_rerank(nullptr, num_q + num_g, num_q + num_g, num_g, static_cast<int>(k1), static_cast<int>(k2), true).bytes;
}

extern "C" int agrl_rerank_dev(const float *q_g, int64_t ld_qg, const float *q_q, int64_t ld_qq,
                               const float *g_g, int64_t ld_gg, int64_t num_q, int64_t num_g,
                               int64_t k1, int64_t k2, double lambda_value,
                               float *out, int64_t ld_out, void *ws, size_t ws_bytes, void *stream) {
    if (!q_g || !q_q || !g_g || !out) return AGRL_E_INVALID;
    int rc = rerank_args_ok(num_q, num_g, k1, k2);
    if (rc) return rc;
    if (ld_qg < num_g || ld_qq < num_q || ld_gg < num_g || ld_out < num_g) return AGRL_E_INVALID;
    if ((rc = agrl_device_ok())) return rc;
    RerankWs w = carve_rerank(ws, num_q + num_g, num_q + num_g, num_g, static_cast<int>(k1), static_cast<int>(k2), true);
    if (!ws || ws_bytes < w.bytes) return AGRL_E_WORKSPACE;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int nq = static_cast<int>(num_q), ng = static_cast<int>(num_g), N = nq + ng;
    RerankGeom g{q_g, q_q, g_g, ld_qg, ld_qq, ld_gg, nq, ng, N, 0, 0};
    if ((rc = launch_rows(g, 0, N, w.K, w.colmax, w.D, w.rank, st))) return rc;
    if ((rc = launch_expand(w.D, w.rank, N, w.K, static_cast<int>(k1), N, nq, 0, w.cap1, w.v1_idx, w.v1_val, w.v1_cnt, st)))
        return rc;
    return launch_finish(w, w.rank, SparseRows{w.v1_idx, w.v1_val, w.v1_cnt, w.cap1}, N, nq, 0, ng, static_cast<int>(k2),
                         lambda_value, out, ld_out, st);
}

// ---- gallery-sharded re-ranking (include/agrl_b200.h; the decomposition is DESIGN.md section 8) -------------------------
extern "C" size_t agrl_rerank_shard_workspace_bytes(int64_t num_q, int64_t num_g, int64_t n_own, int64_t k1, int64_t k2) {
    if (shard_args_ok(num_q, num_g, n_own, k1, k2)) return 0;
    return carve_rerank(nullptr, num_q + n_own, num_q + num_g, n_own, static_cast<int>(k1), static_cast<int>(k2), false).bytes;
}

static int shard_common(int64_t num_q, int64_t num_g, int64_t g_off, int64_t n_own, int64_t k1, int64_t k2,
                        void *ws, size_t ws_bytes, RerankWs *w) {
    int rc = shard_args_ok(num_q, num_g, n_own, k1, k2);
    if (rc) return rc;
    if (g_off < 0 || g_off + n_own > num_g) return AGRL_E_INVALID;
    if ((rc = agrl_device_ok())) return rc;
    *w = carve_rerank(ws, num_q + n_own, num_q + num_g, n_own, static_cast<int>(k1), static_cast<int>(k2), false);
    if (!ws || ws_bytes < w->bytes) return AGRL_E_WORKSPACE;
    return AGRL_OK;
}

extern "C" int agrl_rerank_shard_rows_dev(const float *q_g, int64_t ld_qg, const float *q_q, int64_t ld_qq,
                                          const float *g_cols, int64_t ld_gc, int64_t num_q, int64_t num_g,
                                          int64_t g_off, int64_t n_own, int64_t row0, int64_t row1, int64_t k1, int64_t k2,
                                          int32_t *rank_rows, void *ws, size_t ws_bytes, void *stream) {
    if (!q_g || !q_q || !rank_rows) return AGRL_E_INVALID;
    if (row0 < 0 || row1 < row0 || row1 > num_q + n_own || ld_qg < num_g || ld_qq < num_q) return AGRL_E_INVALID;
    const int64_t gal0 = row0 > num_q ? row0 : num_q;                      // first local gallery row of the range
    if (row1 > num_q && (!g_cols || ld_gc < row1 - gal0)) return AGRL_E_INVALID;
    RerankWs w;
    int rc = shard_common(num_q, num_g, g_off, n_own, k1, k2, ws, ws_bytes, &w);
    if (rc) return rc;
    const int nq = static_cast<int>(num_q), N = static_cast<int>(num_q + num_g);
    RerankGeom g{q_g, q_q, g_cols, ld_qg, ld_qq, ld_gc, nq, static_cast<int>(num_g), N, static_cast<int>(g_off),
                 static_cast<int>(g_off + gal0 - num_q)};
    return launch_rows(g, static_cast<int>(row0), static_cast<int>(row1), w.K, w.colmax, w.D, rank_rows,
                       static_cast<cudaStream_t>(stream));
}

extern "C" int agrl_rerank_shard_expand_dev(const int32_t *rank_all, int64_t num_q, int64_t num_g, int64_t g_off,
                                            int64_t n_own, int64_t k1, int64_t k2, int32_t *v_idx, float *v_val,
                                            int32_t *v_cnt, void *ws, size_t ws_bytes, void *stream) {
    if (!rank_all || !v_idx || !v_val || !v_cnt) return AGRL_E_INVALID;
    RerankWs w;
    int rc = shard_common(num_q, num_g, g_off, n_own, k1, k2, ws, ws_bytes, &w);
    if (rc) return rc;
    const int nq = static_cast<int>(num_q), N = static_cast<int>(num_q + num_g);
    return launch_expand(w.D, rank_all, N, w.K, static_cast<int>(k1), nq + static_cast<int>(n_own), nq, static_cast<int>(g_off),
                         w.cap1, v_idx, v_val, v_cnt, static_cast<cudaStream_t>(stream));
}

extern "C" int agrl_rerank_shard_finish_dev(const int32_t *rank_all, const int32_t *v_idx_all, const float *v_val_all,
                                            const int32_t *v_cnt_all, int64_t num_q, int64_t num_g, int64_t g_off,
                                            int64_t n_own, int64_t k1, int64_t k2, double lambda_value,
                                            float *out, int64_t ld_out, void *ws, size_t ws_bytes, void *stream) {
    if (!rank_all || !v_idx_all || !v_val_all || !v_cnt_all || (n_own > 0 && (!out || ld_out < n_own))) return AGRL_E_INVALID;
    RerankWs w;
    int rc = shard_common(num_q, num_g, g_off, n_own, k1, k2, ws, ws_bytes, &w);
    if (rc) return rc;
    const int N = static_cast<int>(num_q + num_g);
    return launch_finish(w, rank_all, SparseRows{v_idx_all, v_val_all, v_cnt_all, w.cap1}, N, static_cast<int>(num_q),
                         static_cast<int>(g_off), static_cast<int>(n_own), static_cast<int>(k2), lambda_value, out, ld_out,
                         static_cast<cudaStream_t>(stream));
}
