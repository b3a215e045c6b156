// rank.cu -- CMC / mAP on the GPU, bit-exact with the reference evaluators.
//
//   market1501 metric : torchreid/metrics/rank_cylib/rank_cy.pyx:154-241 (eval_market1501_cy)
//   MARS metric       : torchreid/metrics/rank.py:160-212 (evaluate_mars, Compute_AP)
//
// Neither evaluator needs a sorted row.  With the row ordered by key (distance, gallery index):
//
//   market1501  AP and the CMC step only depend on the kept-rank of the query's POSITIVES
//               (same pid, other camera).  One CTA per query gathers the few same-pid gallery items
//               (positives + same-camera junk) into shared memory, sorts that short list, then
//               streams the row ONCE, binning every element between the list's keys (upper bound
//               by branch-free binary search, per-thread private histograms -> no atomics).  A
//               prefix sum over the bins gives each positive's full rank; subtracting the junk
//               items in front of it gives the kept rank.  HBM traffic = one read of the matrix.
//   MARS        only the first max_rank entries of the ordered row are inspected.  One CTA per
//               query keeps a candidate buffer in shared memory, filtered by a running threshold
//               (k-th smallest key seen so far), re-compacted by a bitonic sort when it fills.
//
// The sequential floating-point recurrences of the reference (float accumulation with the term in
// double for rank_cy; Python-double arithmetic and numpy's pairwise mean for evaluate_mars) are
// reproduced with explicitly rounded intrinsics, so no FMA contraction can change a bit.
#include "topk.cuh"

#include <limits.h>
#include <string.h>

namespace agrl {

constexpr int kFastBins    = 64;     // fast path: same-pid list of <= 62 items, padded to 64
constexpr int kListCap     = 2048;   // shared-histogram path: list of <= 2048 items
constexpr int kOverflowCtas = 8;     // brute-force path for longer lists

// ------------------------------------------------------------------------------------------------
// labels: int64 (ABI) -> int32 (kernels), flagging values that do not fit
// ------------------------------------------------------------------------------------------------
struct LabelArrays {
    const int64_t *src[4];
    int32_t       *dst[4];
    int64_t        n[4];
};

__global__ void narrow_labels_kernel(LabelArrays a, uint32_t *status) {
    const int which = blockIdx.y;
    const int64_t *src = a.src[which];
    int32_t *dst = a.dst[which];
    const int64_t n = a.n[which];
    bool bad = false;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
         i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t v = src[i];
        bad |= (v < INT32_MIN || v > INT32_MAX);
        dst[i] = static_cast<int32_t>(v);
    }
    if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) atomicOr(status, AGRL_ST_LABEL_RANGE);
}

// elements in front of the row's first 16-byte boundary
__device__ __forceinline__ int row_head(const float *row, int n) {
    const int head = static_cast<int>(((16u - (reinterpret_cast<uintptr_t>(row) & 15u)) & 15u) >> 2);
    return head < n ? head : n;
}

// visit every element of a row once, 16-byte vector loads over the aligned body
template <class F>
__device__ __forceinline__ void for_each_in_row(const float *__restrict__ row, int n, int tid,
                                                int nthreads, F &&f) {
    const int head = row_head(row, n);
    if (tid < head) f(row[tid], tid);
    const int nvec = (n - head) >> 2;
    const float4 *v4 = reinterpret_cast<const float4 *>(row + head);
#pragma unroll 2
    for (int v = tid; v < nvec; v += nthreads) {
        const float4 x = __ldg(v4 + v);
        const int j = head + (v << 2);
        f(x.x, j); f(x.y, j + 1); f(x.z, j + 2); f(x.w, j + 3);
    }
    const int tail0 = head + (nvec << 2);
    if (tail0 + tid < n) f(row[tail0 + tid], tail0 + tid);     // < 4 leftovers
}

// the most elements one thread visits in for_each_in_row: thread 0 takes the head element, the
// largest share of the vectors and a tail element
__device__ __forceinline__ int row_max_per_thread(const float *row, int n, int nthreads) {
    const int head = row_head(row, n);
    const int nvec = (n - head) >> 2;
    return (head > 0) + 4 * ((nvec + nthreads - 1) / nthreads) + (((n - head) & 3) != 0);
}

// visit the gallery items labelled `pid`, f(j) for each, int4 loads over the labels; kRankThreads threads
template <class F>
__device__ __forceinline__ void for_each_same_pid(const int32_t *__restrict__ g_pid, int ng, int pid, int tid, F &&f) {
    const int nvec = ng >> 2;
    const int4 *p4 = reinterpret_cast<const int4 *>(g_pid);
    for (int v = tid; v < nvec; v += kRankThreads) {
        const int4 p = __ldg(p4 + v);
        if (p.x == pid) f(4 * v);
        if (p.y == pid) f(4 * v + 1);
        if (p.z == pid) f(4 * v + 2);
        if (p.w == pid) f(4 * v + 3);
    }
    const int j = (nvec << 2) + tid;
    if (j < ng && g_pid[j] == pid) f(j);
}

__device__ __forceinline__ float div_rn(float x, float y) { return __fdiv_rn(x, y); }
__device__ __forceinline__ double div_rn(double x, double y) { return __ddiv_rn(x, y); }

// cmc[r] = (number of first hits <= r) / div for r < R, from the first-hit histogram; one warp, inclusive scan over r
// in chunks of 32
template <class T>
__device__ __forceinline__ void cmc_from_hist(const int32_t *hist, int R, T div, T *cmc, int lane) {
    int carry = 0;
    for (int base = 0; base < R; base += 32) {
        const int r = base + lane;
        int x = r < R ? hist[r] : 0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int n = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += n;
        }
        if (r < R) cmc[r] = div_rn(static_cast<T>(carry + x), div);
        carry += __shfl_sync(0xffffffffu, x, 31);
    }
}

// ------------------------------------------------------------------------------------------------
// market1501: one CTA per query
// ------------------------------------------------------------------------------------------------
// what rank_market_finish_kernel reads: sizes and the per-query results of the rank kernels
struct MarketResults {
    int            num_q, rank_len;                // rank_len = min(max_rank, num_g)
    float         *ap;                             // [num_q]
    int32_t       *first_hit;                      // [num_q] kept-rank of the best positive, INT_MAX if invalid
    int32_t       *kept;                           // [num_q] gallery size after the junk filter
    uint32_t      *flags;                          // bit0: some valid query has kept < rank_len (stale cmc tail)
};

struct MarketArgs {
    const float   *dist;
    int64_t        ld;
    const int32_t *q_pid, *q_cam, *g_pid, *g_cam;
    int            num_g;
    MarketResults  res;
    int32_t       *overflow_list;                  // queries whose same-pid list exceeds kListCap
    int32_t       *overflow_count;
};

// AP recurrence of rank_cy.pyx:219-225 over the positives in rank order: term = cum/(rank+1) in
// double, accumulator rounded to float at each step.  terms[] already holds the double quotients.
__device__ __forceinline__ float ap_from_terms(const double *terms, int npos) {
    float acc = 0.f;
    for (int i = 0; i < npos; ++i) acc = __double2float_rn(__dadd_rn(static_cast<double>(acc), terms[i]));
    return __fdiv_rn(acc, static_cast<float>(npos));
}

// Kept ranks of one query's sorted same-pid list of m items, npos of them positives, by one warp.  count(i): row
// elements sorting between item i - 1 and item i; junk(i): item i has the query's camera.  The prefix sum of the counts
// is item i's full rank, minus the junk items in front of it its kept rank.  Each positive's AP term goes to
// terms[positives in front of it]; terms may alias the list, it is written behind the read cursor.  Lane 0 stores the AP
// to *ap; returns the best positive's kept rank in every lane.
template <class Count, class Junk>
__device__ __forceinline__ int market_kept_ranks(int m, int npos, int lane, double *terms, Count count, Junk junk,
                                                 float *ap) {
    int carry_rank = 0, carry_junk = 0, carry_pos = 0;
    int first_hit = INT_MAX;
    for (int base = 0; base < m; base += 32) {
        const int i = base + lane;
        const bool in = i < m;
        const int cnt = in ? count(i) : 0;
        const bool is_junk = in && junk(i);
        const bool is_pos = in && !is_junk;
        // inclusive scan of cnt, exclusive counts of junk / positives in front of item i
        int incl = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int n = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += n;
        }
        const uint32_t jm = __ballot_sync(0xffffffffu, is_junk);
        const uint32_t pm = __ballot_sync(0xffffffffu, is_pos);
        const uint32_t below = (1u << lane) - 1u;
        const int full_rank = carry_rank + incl;                       // #{j : key_j < key_i}
        const int kept_rank = full_rank - (carry_junk + __popc(jm & below));
        const int pos_before = carry_pos + __popc(pm & below);
        __syncwarp();
        if (is_pos) {
            terms[pos_before] = __ddiv_rn(static_cast<double>(pos_before + 1),
                                          static_cast<double>(kept_rank + 1));
            if (pos_before == 0) first_hit = kept_rank;
        }
        carry_rank += __shfl_sync(0xffffffffu, incl, 31);
        carry_junk += __popc(jm);
        carry_pos += __popc(pm);
        __syncwarp();
    }
    first_hit = __reduce_min_sync(0xffffffffu, first_hit);
    if (lane == 0) *ap = ap_from_terms(terms, npos);
    return first_hit;
}

__global__ void __launch_bounds__(kRankThreads)
rank_market_kernel(MarketArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint64_t *list  = reinterpret_cast<uint64_t *>(smem_raw);                       // kListCap keys
    uint16_t *hist16 = reinterpret_cast<uint16_t *>(smem_raw + kListCap * 8);       // [kFastBins][256]
    uint32_t *hist32 = reinterpret_cast<uint32_t *>(smem_raw + kListCap * 8);       // [kListCap+1] (aliases)
    __shared__ int s_m, s_njunk, s_npos;
    __shared__ int s_cnt[kFastBins];

    const int q = blockIdx.x;
    const int tid = threadIdx.x;
    const int ng = a.num_g;
    const int pid = a.q_pid[q], cam = a.q_cam[q];
    const float *row = a.dist + static_cast<size_t>(q) * a.ld;

    if (tid == 0) { s_m = 0; s_njunk = 0; s_npos = 0; }
    __syncthreads();

    // ---- phase A: gather the gallery items of the query's identity (labels only) ------------
    for_each_same_pid(a.g_pid, ng, pid, tid, [&](int j) {
        const bool junk = (a.g_cam[j] == cam);
        atomicAdd(junk ? &s_njunk : &s_npos, 1);
        const int slot = atomicAdd(&s_m, 1);
        if (slot < kListCap) list[slot] = rank_key(row[j], static_cast<uint32_t>(j));
    });
    __syncthreads();
    const int m = s_m, njunk = s_njunk, npos = s_npos;
    const int kept = ng - njunk;
    if (npos == 0) {                       // identity absent from the gallery: query skipped (pyx:203-205)
        if (tid == 0) { a.res.ap[q] = 0.f; a.res.first_hit[q] = INT_MAX; a.res.kept[q] = kept; }
        return;
    }
    if (m > kListCap) {                    // rare: handled by rank_market_overflow_kernel
        if (tid == 0) {
            a.overflow_list[atomicAdd(a.overflow_count, 1)] = q;
            a.res.kept[q] = kept;
            if (kept < a.res.rank_len) atomicOr(a.res.flags, 1u);
        }
        return;
    }

    // ---- phase B: sort the short list --------------------------------------------------------
    // u16 private counters: no thread may bin more than 65535 elements.  The bound is the busiest
    // thread's count, not ng / kRankThreads: thread 0 can take up to 5 elements more than that.
    const bool fast = (m <= kFastBins - 2) && (row_max_per_thread(row, ng, kRankThreads) <= 65535);
    // No pad entry is needed: every binned key is < list[m - 1], so the search below counts at most
    // m - 1 <= n2 - 1 list keys.  Hence n2 <= kListCap: the list never reaches into the histogram region.
    int n2 = kFastBins;
    while (n2 < m) n2 <<= 1;
    for (int i = m + tid; i < n2; i += kRankThreads) list[i] = kKeyMax;
    if (fast) {
#pragma unroll 8
        for (int t = 0; t < kFastBins; ++t) hist16[t * kRankThreads + tid] = 0;
    } else {
        for (int i = tid; i <= kListCap; i += kRankThreads) hist32[i] = 0;
    }
    __syncthreads();
    if (fast) {
        if (tid < 32) bitonic_sort_u64<true>(list, kFastBins, tid, 32);
        __syncthreads();
    } else {
        bitonic_sort_u64<false>(list, n2, tid, kRankThreads);
    }
    const uint64_t key_max = list[m - 1];

    // ---- phase C: one pass over the row, bin each element between the list keys ---------------
    if (fast) {
        uint16_t *mine = hist16 + tid;
        for_each_in_row(row, ng, tid, kRankThreads, [&](float d, int j) {
            const uint64_t key = rank_key(d, static_cast<uint32_t>(j));
            if (key < key_max) {           // otherwise it precedes none of the list items
                int t = 0;                 // t = #{i : list[i] <= key}
#pragma unroll
                for (int s = kFastBins / 2; s > 0; s >>= 1)
                    if (list[t + s - 1] <= key) t += s;
                mine[t * kRankThreads] += 1;
            }
        });
    } else {
        for_each_in_row(row, ng, tid, kRankThreads, [&](float d, int j) {
            const uint64_t key = rank_key(d, static_cast<uint32_t>(j));
            if (key < key_max) {
                int t = 0;
                for (int s = n2 >> 1; s > 0; s >>= 1)
                    if (list[t + s - 1] <= key) t += s;
                atomicAdd(&hist32[t], 1u);
            }
        });
    }
    __syncthreads();

    // ---- phase D: bins -> ranks -> AP ----------------------------------------------------------
    if (fast) {
        const int warp = tid >> 5, lane = tid & 31;
        for (int t = warp; t < m; t += kRankThreads / 32) {
            const uint4 v = *reinterpret_cast<const uint4 *>(hist16 + t * kRankThreads + lane * 8);
            int s = (v.x & 0xffff) + (v.x >> 16) + (v.y & 0xffff) + (v.y >> 16) +
                    (v.z & 0xffff) + (v.z >> 16) + (v.w & 0xffff) + (v.w >> 16);
            s = warp_sum(s);
            if (lane == 0) s_cnt[t] = s;
        }
        __syncthreads();
    }
    if (tid >= 32) return;
    const int first_hit = market_kept_ranks(
        m, npos, tid, reinterpret_cast<double *>(list),
        [&](int i) { return fast ? s_cnt[i] : static_cast<int>(hist32[i]); },
        [&](int i) { return a.g_cam[static_cast<uint32_t>(list[i])] == cam; }, &a.res.ap[q]);
    if (tid == 0) {
        a.res.first_hit[q] = first_hit;
        a.res.kept[q] = kept;
        if (kept < a.res.rank_len) atomicOr(a.res.flags, 1u);
    }
}

// Brute-force path for identities with more than kListCap gallery items: O(m * (num_g + m)) per
// query, a handful of CTAs, global-memory slabs (keys + terms).  Same arithmetic, same results.
__global__ void __launch_bounds__(kRankThreads)
rank_market_overflow_kernel(MarketArgs a, uint64_t *slab_keys, double *slab_terms) {
    __shared__ int s_m;
    __shared__ int s_first;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int ng = a.num_g;
    uint64_t *keys = slab_keys + static_cast<size_t>(blockIdx.x) * ng;
    double *terms = slab_terms + static_cast<size_t>(blockIdx.x) * ng;
    const int count = *a.overflow_count;
    for (int o = blockIdx.x; o < count; o += gridDim.x) {
        const int q = a.overflow_list[o];
        const int pid = a.q_pid[q], cam = a.q_cam[q];
        const float *row = a.dist + static_cast<size_t>(q) * a.ld;
        if (tid == 0) { s_m = 0; s_first = INT_MAX; }
        __syncthreads();
        for (int j = tid; j < ng; j += kRankThreads)
            if (a.g_pid[j] == pid) keys[atomicAdd(&s_m, 1)] = rank_key(row[j], static_cast<uint32_t>(j));
        __syncthreads();
        const int m = s_m;
        int npos_total = 0;
        for (int i = warp; i < m; i += kRankThreads / 32) {
            const uint64_t key = keys[i];
            const uint32_t idx = static_cast<uint32_t>(key);
            const bool self_junk = (a.g_cam[idx] == cam);
            if (self_junk) continue;                                   // warp-uniform
            int full = 0, junk_before = 0, pos_before = 0;
            for (int j = lane; j < ng; j += 32) full += (rank_key(row[j], static_cast<uint32_t>(j)) < key);
            for (int j = lane; j < m; j += 32) {
                const uint64_t kj = keys[j];
                if (kj < key) {
                    if (a.g_cam[static_cast<uint32_t>(kj)] == cam) ++junk_before; else ++pos_before;
                }
            }
            full = warp_sum(full); junk_before = warp_sum(junk_before); pos_before = warp_sum(pos_before);
            if (lane == 0) {
                const int kept_rank = full - junk_before;
                terms[pos_before] = __ddiv_rn(static_cast<double>(pos_before + 1),
                                              static_cast<double>(kept_rank + 1));
                if (pos_before == 0) s_first = kept_rank;
            }
        }
        __syncthreads();
        if (tid == 0) {
            for (int i = 0; i < m; ++i)
                npos_total += (a.g_cam[static_cast<uint32_t>(keys[i])] != cam);
            a.res.ap[q] = ap_from_terms(terms, npos_total);
            a.res.first_hit[q] = s_first;
        }
        __syncthreads();
    }
}

// One CTA: averages in the reference's order (rank_cy.pyx:230-239).
__global__ void __launch_bounds__(1024)
rank_market_finish_kernel(MarketResults a, int32_t *hist /*[rank_len+1], zeroed here*/,
                          float *cmc_out, float *map_out, int64_t *num_valid_out, uint32_t *status) {
    __shared__ int s_valid;
    const int tid = threadIdx.x, nthr = blockDim.x;
    const int nq = a.num_q, R = a.rank_len;
    if (tid == 0) s_valid = 0;
    for (int r = tid; r <= R; r += nthr) hist[r] = 0;
    __syncthreads();
    int v = 0;
    for (int q = tid; q < nq; q += nthr) v += (a.first_hit[q] != INT_MAX);
    v = warp_sum(v);
    if ((tid & 31) == 0 && v) atomicAdd(&s_valid, v);
    __syncthreads();
    const int nvalid = s_valid;
    if (nvalid == 0) {
        if (tid == 0) { atomicOr(status, AGRL_ST_NO_VALID_QUERY); if (num_valid_out) *num_valid_out = 0; }
        return;
    }
    const float fvalid = static_cast<float>(nvalid);     // exact: the reference counts in float by +1.
    const bool stale = (*a.flags & 1u) != 0;
    if (!stale) {
        // every valid query has kept >= rank_len: cmc row = [r >= first_hit]
        for (int q = tid; q < nq; q += nthr) {
            const int fh = a.first_hit[q];
            if (fh != INT_MAX) atomicAdd(&hist[fh < R ? fh : R], 1);
        }
        __syncthreads();
        if (tid < 32) cmc_from_hist(hist, R, fvalid, cmc_out, tid);
    } else {
        // rank_cy never clears its `cmc` scratch (pyx:177): positions >= kept keep what the last
        // valid query that reached them left there.  Replay that per rank position, in query order.
        for (int r = tid; r < R; r += nthr) {
            int last = 0, sum = 0;
            for (int q = 0; q < nq; ++q) {
                const int fh = a.first_hit[q];
                if (fh == INT_MAX) continue;
                if (r < a.kept[q]) last = (r >= fh);
                sum += last;
            }
            cmc_out[r] = __fdiv_rn(static_cast<float>(sum), fvalid);
        }
    }
    // mAP: fp32 sum in query order (rank_cy.pyx:236-239).  The chain is sequential by definition;
    // blocks of ap are staged in shared memory by the whole CTA so the one adding thread never
    // waits on global memory.
    __shared__ float s_ap[4096];
    float acc = 0.f;
    for (int base = 0; base < nq; base += 4096) {
        __syncthreads();
        for (int i = tid; i < 4096 && base + i < nq; i += nthr) s_ap[i] = a.ap[base + i];
        __syncthreads();
        if (tid == 0) {
            const int n = nq - base < 4096 ? nq - base : 4096;
#pragma unroll 8
            for (int i = 0; i < n; ++i) acc = __fadd_rn(acc, s_ap[i]);   // invalid queries hold +0
        }
    }
    if (tid == 0) {
        *map_out = __fdiv_rn(acc, fvalid);
        if (num_valid_out) *num_valid_out = nvalid;
    }
}

// ------------------------------------------------------------------------------------------------
// market1501, gallery sharded over GPUs (SURVEY.md section 8e): the same rank-by-counting, cut at the
// two points where the shards have to talk.
//   gather   each shard lists, per query, its same-pid gallery items as keys
//            (order-preserving distance bits << 32 | global index << 1 | junk bit)      -> all-gather
//   bin      every shard sorts the gathered lists (identically) and counts, per list item, how many of
//            ITS row elements sort before it                                            -> all-reduce(sum)
//   finalize prefix sums -> kept ranks -> AP / first hit, exactly as in rank_market_kernel
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t shard_key(float d, uint32_t global_idx, uint32_t junk) {
    return (static_cast<uint64_t>(mono_key(d)) << 32) | (static_cast<uint64_t>(global_idx) << 1) | junk;
}

struct MarketShardArgs {
    const float   *dist;
    int64_t        ld;
    const int32_t *q_pid, *q_cam, *g_pid, *g_cam;
    int            num_q, num_g;
    uint32_t       index_offset;
    int            cap;                 // slots per query and shard
    uint64_t      *keys;                // gather: [num_q][cap]; bin: gathered [parts][num_q][cap]
    int32_t       *npos, *njunk;        // gather out: per query counts of this shard
    int32_t       *max_count;           // count pass: max over queries of this shard's same-pid items
    // bin
    int            parts, n2;           // n2 = power of two >= parts * cap
    int32_t       *cnt;                 // [num_q][n2] elements of this shard sorting before each sorted list item
    uint64_t      *sorted;              // [num_q][n2] the sorted list (identical on every shard)
};

// count pass (cap unknown yet) / gather pass
template <bool kCountOnly>
__global__ void __launch_bounds__(kRankThreads)
rank_market_gather_kernel(MarketShardArgs a) {
    __shared__ int s_m, s_njunk, s_npos;
    const int q = blockIdx.x, tid = threadIdx.x;
    const int ng = a.num_g;
    const int pid = a.q_pid[q], cam = a.q_cam[q];
    const float *row = a.dist + static_cast<size_t>(q) * a.ld;
    uint64_t *out = kCountOnly ? nullptr : a.keys + static_cast<size_t>(q) * a.cap;
    if (tid == 0) { s_m = 0; s_njunk = 0; s_npos = 0; }
    if (!kCountOnly) for (int i = tid; i < a.cap; i += kRankThreads) out[i] = kKeyMax;
    __syncthreads();
    for_each_same_pid(a.g_pid, ng, pid, tid, [&](int j) {
        const int slot = atomicAdd(&s_m, 1);
        if (kCountOnly) return;
        const bool junk = (a.g_cam[j] == cam);
        atomicAdd(junk ? &s_njunk : &s_npos, 1);
        if (slot < a.cap) out[slot] = shard_key(row[j], a.index_offset + static_cast<uint32_t>(j), junk ? 1u : 0u);
    });
    __syncthreads();
    if (tid == 0) {
        if (kCountOnly) atomicMax(a.max_count, s_m);
        else { a.npos[q] = s_npos; a.njunk[q] = s_njunk; }
    }
}

__global__ void __launch_bounds__(kRankThreads)
rank_market_bin_kernel(MarketShardArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint64_t *list = reinterpret_cast<uint64_t *>(smem_raw);                         // n2 keys
    uint32_t *hist = reinterpret_cast<uint32_t *>(smem_raw + static_cast<size_t>(a.n2) * 8);   // n2 + 1 bins
    const int q = blockIdx.x, tid = threadIdx.x;
    const int n2 = a.n2, total = a.parts * a.cap;
    for (int i = tid; i < n2; i += kRankThreads) {
        uint64_t k = kKeyMax;
        if (i < total) k = a.keys[(static_cast<size_t>(i / a.cap) * a.num_q + q) * a.cap + (i % a.cap)];
        list[i] = k;
    }
    for (int i = tid; i <= n2; i += kRankThreads) hist[i] = 0;
    __syncthreads();
    bitonic_sort_u64<false>(list, n2, tid, kRankThreads);
    // (keys are unique, so every shard obtains the same order)
    const uint64_t last = list[n2 - 1];
    int m = n2;                                         // number of real items: first pad position
    if (last == kKeyMax) {                              // binary search for the first pad
        int lo = 0, hi = n2 - 1;
        while (lo < hi) { const int mid = (lo + hi) >> 1; if (list[mid] == kKeyMax) hi = mid; else lo = mid + 1; }
        m = lo;
    }
    uint64_t *sorted = a.sorted + static_cast<size_t>(q) * n2;
    for (int i = tid; i < n2; i += kRankThreads) sorted[i] = list[i];
    if (m > 0) {
        const uint64_t key_max = list[m - 1] & ~1ull;
        const float *row = a.dist + static_cast<size_t>(q) * a.ld;
        for_each_in_row(row, a.num_g, tid, kRankThreads, [&](float d, int j) {
            const uint64_t key = shard_key(d, a.index_offset + static_cast<uint32_t>(j), 0u);
            if (key < key_max) {
                int t = 0;                              // t = #{i : (list[i] without junk bit) <= key}
                for (int s = n2 >> 1; s > 0; s >>= 1)
                    if ((list[t + s - 1] & ~1ull) <= key) t += s;
                atomicAdd(&hist[t], 1u);
            }
        });
    }
    __syncthreads();
    int32_t *cnt = a.cnt + static_cast<size_t>(q) * n2;
    for (int i = tid; i < n2; i += kRankThreads) cnt[i] = static_cast<int32_t>(hist[i]);
}

struct MarketFinalArgs {
    const int32_t  *cnt;                // [num_q][n2] summed over shards
    const uint64_t *sorted;             // [num_q][n2]
    const int32_t  *npos, *njunk;       // [num_q] summed over shards
    int             n2;
    int64_t         num_g_total;
    double         *terms;              // [num_q][n2] scratch
    MarketResults   res;
};

// one warp per query
__global__ void __launch_bounds__(kRankThreads)
rank_market_finalize_kernel(MarketFinalArgs a) {
    const int lane = threadIdx.x & 31;
    const int q = blockIdx.x * (kRankThreads / 32) + (threadIdx.x >> 5);
    if (q >= a.res.num_q) return;
    const int npos = a.npos[q], njunk = a.njunk[q];
    const int kept = static_cast<int>(a.num_g_total - njunk);
    if (npos == 0) {
        if (lane == 0) { a.res.ap[q] = 0.f; a.res.first_hit[q] = INT_MAX; a.res.kept[q] = kept; }
        return;
    }
    const int32_t *cnt = a.cnt + static_cast<size_t>(q) * a.n2;
    const uint64_t *sorted = a.sorted + static_cast<size_t>(q) * a.n2;
    const int first_hit = market_kept_ranks(
        npos + njunk, npos, lane, a.terms + static_cast<size_t>(q) * a.n2,
        [&](int i) { return cnt[i]; }, [&](int i) { return (sorted[i] & 1ull) != 0; }, &a.res.ap[q]);
    if (lane == 0) {
        a.res.first_hit[q] = first_hit;
        a.res.kept[q] = kept;
        if (kept < a.res.rank_len) atomicOr(a.res.flags, 1u);
    }
}

// ------------------------------------------------------------------------------------------------
// MARS metric: one CTA per query
// ------------------------------------------------------------------------------------------------
// what rank_mars_finish_kernel reads: sizes and the per-query results of the rank kernels
struct MarsResults {
    int            num_q, max_rank;
    double        *ap;                              // [num_q]
    int32_t       *first_pos;                       // [num_q] junk-compacted position of the first good hit
};

struct MarsArgs {
    const float   *dist;
    int64_t        ld;
    const int32_t *q_pid, *q_cam, *g_pid, *g_cam;
    int            num_g;
    int            buf_len;                         // power of two >= 2*max_rank and >= 2*tile
    MarsResults    res;
    uint32_t      *status;
    // gallery-sharded form (rank_mars_kernel<true>): this shard's candidates instead of the AP
    uint64_t      *part_keys;                       // [num_q][max_rank] keys with GLOBAL gallery index
    uint8_t       *part_cls;                        // [num_q][max_rank] bit0 good, bit1 junk
    int32_t       *part_ngood;                      // [num_q] good images in this shard
    uint32_t       index_offset;                    // global index of this shard's first gallery row
};

// number of good images for the query: same pid, other camera (rank.py:166); result in *s_ngood
__device__ __forceinline__ void mars_count_good(const MarsArgs &a, int pid, int cam, int tid, int *s_ngood) {
    int good = 0;
    for_each_same_pid(a.g_pid, a.num_g, pid, tid, [&](int j) { good += (a.g_cam[j] != cam); });
    good = warp_sum(good);
    if ((tid & 31) == 0 && good) atomicAdd(s_ngood, good);
}

// class byte of a ranked gallery item (rank.py:166-169): bit0 good (same pid, other camera), bit1 junk (pid -1, or
// same pid and camera)
__device__ __forceinline__ uint8_t mars_class(int gp, int gc, int pid, int cam) {
    const bool good = (gp == pid) && (gc != cam);
    const bool junk = (gp == -1) || ((gp == pid) && (gc == cam));
    return static_cast<uint8_t>((good ? 1 : 0) | (junk ? 2 : 0));
}

// Compute_AP (rank.py:180-212) in Python-float (double) arithmetic, one rounding per operation.
// cls[n]: bit0 good, bit1 junk for the n-th ranked gallery item; n_ranked of them.
__device__ __forceinline__ void mars_compute_ap(const uint8_t *cls, int n_ranked, int ngood,
                                                double *ap_out, int *first_pos_out, uint32_t *status) {
    double old_recall = 0.0, old_precision = 1.0, ap = 0.0;
    int inter = 0, j_eff = 0, good_now = 0, njunk = 0, first_pos = INT_MAX;
    bool zero_div = false;
    for (int n = 0; n < n_ranked; ++n) {
        const int c = cls[n];
        if (c & 1) {
            if (first_pos == INT_MAX) first_pos = n - njunk;         // cmc[n - njunk:] = 1
            ++good_now;
        }
        if (c & 2) { ++njunk; continue; }
        if (c & 1) ++inter;
        if (ngood == 0) { zero_div = true; break; }                  // ZeroDivisionError (rank.py:203)
        double recall = 0.0, precision = 0.0;
        if (inter > 0) {
            recall = __ddiv_rn(static_cast<double>(inter), static_cast<double>(ngood));
            precision = __ddiv_rn(static_cast<double>(inter), static_cast<double>(j_eff + 1));
        }
        const double t = __ddiv_rn(__dmul_rn(__dsub_rn(recall, old_recall),
                                             __dadd_rn(old_precision, precision)), 2.0);
        ap = __dadd_rn(ap, t);
        old_recall = recall;
        old_precision = precision;
        ++j_eff;
        if (good_now == ngood) break;
    }
    if (zero_div) atomicOr(status, AGRL_ST_ZERO_DIVISION);
    *ap_out = ap;
    *first_pos_out = first_pos;
}

// kPartial = false: whole gallery on this GPU -> AP and first hit per query.
// kPartial = true : gallery shard -> this shard's top-K candidates (global indices), their classes,
//                   and the shard's good count, for rank_mars_merge_kernel.
template <bool kPartial>
__global__ void __launch_bounds__(kRankThreads)
rank_mars_kernel(MarsArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint64_t *buf = reinterpret_cast<uint64_t *>(smem_raw);                 // buf_len keys
    uint8_t  *cls = reinterpret_cast<uint8_t *>(smem_raw + a.buf_len * 8);  // max_rank class bytes
    __shared__ int s_cnt, s_ngood;
    __shared__ unsigned long long s_thr;

    const int q = blockIdx.x, tid = threadIdx.x;
    const int K = a.res.max_rank;
    const int pid = a.q_pid[q], cam = a.q_cam[q];
    const float *row = a.dist + static_cast<size_t>(q) * a.ld;

    if (tid == 0) { s_cnt = 0; s_ngood = 0; s_thr = kKeyMax; }
    __syncthreads();
    mars_count_good(a, pid, cam, tid, &s_ngood);
    const int valid = select_topk(row, a.num_g, K, a.buf_len, buf, &s_cnt, &s_thr, tid);

    for (int n = tid; n < K; n += kRankThreads) {
        uint8_t c = 0;
        if (n < valid) {
            const uint32_t g = static_cast<uint32_t>(buf[n]);
            c = mars_class(a.g_pid[g], a.g_cam[g], pid, cam);
        }
        if (kPartial) {
            a.part_keys[static_cast<size_t>(q) * K + n] = (n < valid) ? buf[n] + a.index_offset : kKeyMax;
            a.part_cls[static_cast<size_t>(q) * K + n] = c;
        } else {
            cls[n] = c;
        }
    }
    __syncthreads();
    if (tid != 0) return;
    if (kPartial) { a.part_ngood[q] = s_ngood; return; }
    mars_compute_ap(cls, valid, s_ngood, &a.res.ap[q], &a.res.first_pos[q], a.status);
}

// Position of `key`, entry `pos` of list p, in the merge of `parts` ascending key lists (list o at lists + o * stride) whose
// real keys are unique: pos plus, for every other list, the number of its keys below `key` (a binary search over the
// list's first n entries).  Positions from n on are not needed: the count stops there, and the result is then >= n.
__device__ __forceinline__ int merged_position(const uint64_t *lists, int parts, int stride, int n, int p, int pos,
                                               uint64_t key) {
    int rank = pos;
    for (int o = 0; o < parts && rank < n; ++o) {
        if (o == p) continue;
        const uint64_t *lst = lists + o * stride;
        int lo = 0, hi = n;
        while (lo < hi) { const int mid = (lo + hi) >> 1; if (lst[mid] < key) lo = mid + 1; else hi = mid; }
        rank += lo;
    }
    return rank;
}

// Merge of the shards' candidates: one CTA per query sorts parts*K (key, class) pairs and runs
// Compute_AP on the first K.  keys/cls are laid out [part][query][K].
struct MarsMergeArgs {
    const uint64_t *keys;
    const uint8_t  *cls;
    const int32_t  *ngood;              // [num_q], already summed over the shards
    int             parts, n2;          // n2 = power of two >= parts * max_rank
    MarsResults     res;
    uint32_t       *status;
};

__global__ void __launch_bounds__(kRankThreads)
rank_mars_merge_kernel(MarsMergeArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int q = blockIdx.x, tid = threadIdx.x, K = a.res.max_rank;
    const int Kp = (K + 15) & ~15;
    uint64_t *keys = reinterpret_cast<uint64_t *>(smem_raw);                                  // n2
    uint64_t *okeys = keys + a.n2;                                                            // Kp: the merged head
    uint8_t  *cls = reinterpret_cast<uint8_t *>(smem_raw + static_cast<size_t>(a.n2 + Kp) * 8);   // n2
    uint8_t  *ocls = cls + a.n2;                                                              // Kp
    const int total = a.parts * K;
    int unsorted = 0;
    for (int i = tid; i < a.n2; i += kRankThreads) {
        if (i < total) {
            const size_t src = (static_cast<size_t>(i / K) * a.res.num_q + q) * K + (i % K);
            keys[i] = a.keys[src];
            cls[i] = a.cls[src];
            if ((i % K) != 0 && a.keys[src - 1] > keys[i]) unsorted = 1;
        } else { keys[i] = kKeyMax; cls[i] = 0; }
    }
    for (int i = tid; i < Kp; i += kRankThreads) { okeys[i] = kKeyMax; ocls[i] = 0; }
#ifdef AGRL_MERGE_SORT
    unsorted = 1;
#endif
    unsorted = __syncthreads_or(unsorted);
    const uint64_t *hk = okeys;
    const uint8_t *hc = ocls;
    if (!unsorted) {
        // every shard's list is ascending (what _partial / agrl_distance_topk_dev emit) and keys are unique: the merged
        // position of a key is its position in its own list plus, for every other list, the number of smaller keys there
        // (a binary search) -- one pass instead of the 45 barrier-separated steps of a 512-key bitonic sort
        for (int i = tid; i < total; i += kRankThreads) {
            const uint64_t key = keys[i];
            if (key == kKeyMax) continue;
            const int p = i / K;
            const int rank = merged_position(keys, a.parts, K, K, p, i - p * K, key);
            if (rank < K) { okeys[rank] = key; ocls[rank] = cls[i]; }
        }
        __syncthreads();
    } else {
        // lists in arbitrary order: bitonic sort of the keys carrying the class byte
        bitonic_sort_u64<false, true>(keys, a.n2, tid, kRankThreads, cls);
        hk = keys; hc = cls;
    }
    if (tid != 0) return;
    int valid = 0;
    while (valid < K && hk[valid] != kKeyMax) ++valid;
    mars_compute_ap(hc, valid, a.ngood[q], &a.res.ap[q], &a.res.first_pos[q], a.status);
}

// numpy's pairwise float64 summation (what np.mean runs on the ap vector, rank.py:176):
// ranges of <= 128 elements ("leaves") are summed with eight interleaved partial sums and a fixed
// tree, larger ranges split at n/2 rounded down to a multiple of 8, left + right.  The split tree
// only depends on n, so the leaves are evaluated in parallel (one thread each) and a single thread
// then replays the tree over the leaf sums -- same additions, same order, same bits.
__device__ double pairwise_leaf_f64(const double *x, int n) {
    if (n < 8) {
        double r = 0.0;
        for (int i = 0; i < n; ++i) r = __dadd_rn(r, x[i]);
        return r;
    }
    double r[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) r[k] = x[k];
    int i = 8;
    for (; i < n - (n % 8); i += 8) {
#pragma unroll
        for (int k = 0; k < 8; ++k) r[k] = __dadd_rn(r[k], x[i + k]);
    }
    double res = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])),
                           __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
    for (; i < n; ++i) res = __dadd_rn(res, x[i]);
    return res;
}

// Post-order walk of the split tree with an explicit stack (device recursion would overflow the
// default 1 KiB thread stack).  leaf(offset, length, index) gives the sum of the index-th leaf in
// visiting order; the walk combines the leaf sums into *result.  Returns the number of leaves.
template <class Leaf>
__device__ int pairwise_walk(int n, Leaf leaf, double *result) {
    constexpr int kDepth = 40;
    int off[kDepth], len[kDepth], state[kDepth];     // state: 1 waiting for left, 2 waiting for right
    double left[kDepth];
    int sp = 1, nleaf = 0;
    off[0] = 0; len[0] = n; state[0] = 0;
    double ret = 0.0;
    bool have_ret = false;
    while (sp > 0) {
        const int t = sp - 1;
        if (have_ret) {                               // a child of frame t just returned
            have_ret = false;
            if (state[t] == 1) {                      // left done -> descend right
                left[t] = ret;
                state[t] = 2;
                int n2 = len[t] / 2; n2 -= n2 % 8;
                off[sp] = off[t] + n2; len[sp] = len[t] - n2; state[sp] = 0; ++sp;
            } else {                                  // right done -> combine and return
                ret = __dadd_rn(left[t], ret);
                have_ret = true;
                --sp;
            }
        } else if (len[t] <= 128) {
            ret = leaf(off[t], len[t], nleaf);
            ++nleaf;
            have_ret = true;
            --sp;
        } else {                                      // descend left
            state[t] = 1;
            int n2 = len[t] / 2; n2 -= n2 % 8;
            off[sp] = off[t]; len[sp] = n2; state[sp] = 0; ++sp;
        }
    }
    *result = ret;
    return nleaf;
}

constexpr int kMaxLeaves = 2048;             // covers num_q up to 262 144 in one pass

__global__ void __launch_bounds__(1024)
rank_mars_finish_kernel(MarsResults a, int32_t *hist /*[max_rank+1]*/, double *cmc_out, double *map_out) {
    __shared__ int2 s_leaf[kMaxLeaves];
    __shared__ double s_sum[kMaxLeaves];
    __shared__ int s_nleaf;
    const int tid = threadIdx.x, nthr = blockDim.x;
    const int nq = a.num_q, R = a.max_rank;
    for (int r = tid; r <= R; r += nthr) hist[r] = 0;
    if (tid == 32) {                         // record the leaves
        double unused;
        s_nleaf = pairwise_walk(nq, [&](int off, int len, int l) {
            if (l < kMaxLeaves) s_leaf[l] = make_int2(off, len);
            return 0.0;
        }, &unused);
    }
    __syncthreads();
    for (int q = tid; q < nq; q += nthr) {
        const int fp = a.first_pos[q];
        atomicAdd(&hist[fp < R ? fp : R], 1);
    }
    const int nleaf = s_nleaf;
    if (nleaf <= kMaxLeaves)
        for (int l = tid; l < nleaf; l += nthr) s_sum[l] = pairwise_leaf_f64(a.ap + s_leaf[l].x, s_leaf[l].y);
    __syncthreads();
    if (tid < 32) cmc_from_hist(hist, R, static_cast<double>(nq), cmc_out, tid);
    if (tid == 32) {
        double total;
        if (nleaf <= kMaxLeaves)
            pairwise_walk(nq, [&](int, int, int l) { return s_sum[l]; }, &total);
        else                                 // very large num_q: sequential leaves (still the same tree)
            pairwise_walk(nq, [&](int off, int len, int) { return pairwise_leaf_f64(a.ap + off, len); }, &total);
        *map_out = __ddiv_rn(total, static_cast<double>(nq));
    }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
struct RankWorkspace {
    int32_t *q_pid, *q_cam, *g_pid, *g_cam;
    float   *ap_f32;
    double  *ap_f64;
    int32_t *first, *kept, *overflow_list, *hist;
    int32_t *counters;       // [0] overflow_count, [1] flags
    uint64_t *slab_keys;
    double   *slab_terms;
    size_t   bytes;
};

static RankWorkspace carve_rank(void *ws, int64_t nq, int64_t ng, int64_t max_rank) {
    Carver c(ws);
    RankWorkspace w;
    w.q_pid = c.take<int32_t>(nq);  w.q_cam = c.take<int32_t>(nq);
    w.g_pid = c.take<int32_t>(ng + 4);  w.g_cam = c.take<int32_t>(ng + 4);
    w.ap_f32 = c.take<float>(nq);
    w.ap_f64 = c.take<double>(nq);
    w.first = c.take<int32_t>(nq);  w.kept = c.take<int32_t>(nq);
    w.overflow_list = c.take<int32_t>(nq);
    w.hist = c.take<int32_t>(max_rank + 1);
    w.counters = c.take<int32_t>(4);
    w.slab_keys = c.take<uint64_t>(static_cast<size_t>(kOverflowCtas) * ng);
    w.slab_terms = c.take<double>(static_cast<size_t>(kOverflowCtas) * ng);
    w.bytes = c.total();
    return w;
}

// the four label arrays to int32 in dst_*
static int narrow_labels(const int64_t *qp, const int64_t *gp, const int64_t *qc, const int64_t *gc, int64_t nq,
                         int64_t ng, int32_t *dst_qp, int32_t *dst_gp, int32_t *dst_qc, int32_t *dst_gc,
                         uint32_t *status, cudaStream_t st) {
    LabelArrays la;
    la.src[0] = qp; la.dst[0] = dst_qp; la.n[0] = nq;
    la.src[1] = qc; la.dst[1] = dst_qc; la.n[1] = nq;
    la.src[2] = gp; la.dst[2] = dst_gp; la.n[2] = ng;
    la.src[3] = gc; la.dst[3] = dst_gc; la.n[3] = ng;
    const int64_t nmax = nq > ng ? nq : ng;
    int blocks = static_cast<int>((nmax + 255) / 256);
    if (blocks > 4 * kNumSMs) blocks = 4 * kNumSMs;
    if (blocks < 1) blocks = 1;
    AGRL_LAUNCH_BEGIN(st);
    narrow_labels_kernel<<<dim3(blocks, 4), 256, 0, st>>>(la, status);
    AGRL_LAUNCH_CHECK(st, "narrow_labels");
    return AGRL_OK;
}

static int check_rank_args(const void *d, const void *a, const void *b, const void *c, const void *e,
                           int64_t nq, int64_t ng, int64_t max_rank, int64_t ld) {
    if (!d || !a || !b || !c || !e) return AGRL_E_INVALID;
    if (nq < 0 || ng < 1 || max_rank < 1 || ld < ng) return AGRL_E_INVALID;
    if (nq > INT32_MAX / 2 || ng > INT32_MAX / 2) return AGRL_E_UNSUPPORTED;
    return AGRL_OK;
}

// the smallest power of two >= x, starting from the power of two `start`
static int pow2_at_least(int64_t x, int start) {
    int p = start;
    while (p < x) p <<= 1;
    return p;
}

// Set-up and launch of rank_mars_kernel<kPartial> for agrl_rank_mars_dev / _partial_dev, whose arguments are checked.
// `a` holds the outputs; for the whole-gallery form a.res.ap == nullptr selects the workspace's AP vector.
template <bool kPartial>
static int launch_rank_mars(MarsArgs &a, RankWorkspace &w, const float *distmat, int64_t ld,
                            const int64_t *q_pids, const int64_t *g_pids, const int64_t *q_camids,
                            const int64_t *g_camids, int64_t num_q, int64_t num_g, int64_t max_rank,
                            void *ws, size_t ws_bytes, cudaStream_t st) {
    int rc = agrl_device_ok();
    if (rc) return rc;
    w = carve_rank(ws, num_q, num_g, max_rank);
    if (!ws || ws_bytes < w.bytes) return AGRL_E_WORKSPACE;
    AGRL_CUDA_TRY(cudaMemsetAsync(a.status, 0, sizeof(uint32_t), st));
    rc = narrow_labels(q_pids, g_pids, q_camids, g_camids, num_q, num_g, w.q_pid, w.g_pid, w.q_cam, w.g_cam,
                       a.status, st);
    if (rc) return rc;
    a.dist = distmat; a.ld = ld;
    a.q_pid = w.q_pid; a.q_cam = w.q_cam; a.g_pid = w.g_pid; a.g_cam = w.g_cam;
    a.num_g = static_cast<int>(num_g);
    a.res.num_q = static_cast<int>(num_q); a.res.max_rank = static_cast<int>(max_rank);
    if (!kPartial) {
        if (!a.res.ap) a.res.ap = w.ap_f64;
        a.res.first_pos = w.first;
    }
    const int L = pow2_at_least(2 * max_rank, 2 * kMarsTile);
    a.buf_len = L;
    const size_t smem = static_cast<size_t>(L) * 8 + align_up(static_cast<size_t>(max_rank), 16);
    AGRL_CUDA_TRY(cudaFuncSetAttribute(rank_mars_kernel<kPartial>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       static_cast<int>(smem)));
    AGRL_LAUNCH_BEGIN(st);
    rank_mars_kernel<kPartial><<<static_cast<unsigned>(num_q), kRankThreads, smem, st>>>(a);
    AGRL_LAUNCH_CHECK(st, kPartial ? "rank_mars_partial" : "rank_mars");
    return AGRL_OK;
}

// labels from the workspace's narrowed copies, or none (w == nullptr) for the bin pass
static MarketShardArgs shard_args(const RankWorkspace *w, const float *distmat, int64_t ld, int64_t num_q,
                                  int64_t num_g, int64_t index_offset) {
    MarketShardArgs a;
    memset(&a, 0, sizeof(a));
    a.dist = distmat; a.ld = ld;
    if (w) { a.q_pid = w->q_pid; a.q_cam = w->q_cam; a.g_pid = w->g_pid; a.g_cam = w->g_cam; }
    a.num_q = static_cast<int>(num_q); a.num_g = static_cast<int>(num_g);
    a.index_offset = static_cast<uint32_t>(index_offset);
    return a;
}

}  // namespace agrl

using namespace agrl;

extern "C" size_t agrl_rank_workspace_bytes(int64_t num_q, int64_t num_g, int64_t max_rank) {
    if (num_q < 0 || num_g < 0 || max_rank < 0) return 0;
    return carve_rank(nullptr, num_q, num_g, max_rank).bytes;
}

extern "C" int agrl_rank_market1501_dev(const float *distmat, int64_t ld,
                                        const int64_t *q_pids, const int64_t *g_pids,
                                        const int64_t *q_camids, const int64_t *g_camids,
                                        int64_t num_q, int64_t num_g, int64_t max_rank,
                                        float *cmc, float *map, float *all_ap, int64_t *num_valid,
                                        uint32_t *status, void *ws, size_t ws_bytes, void *stream) {
    int rc = check_rank_args(distmat, q_pids, g_pids, q_camids, g_camids, num_q, num_g, max_rank, ld);
    if (rc) return rc;
    if (!cmc || !map || !status) return AGRL_E_INVALID;
    if ((rc = agrl_device_ok())) return rc;
    const int64_t rank_len = max_rank < num_g ? max_rank : num_g;
    RankWorkspace w = carve_rank(ws, num_q, num_g, rank_len);
    if (!ws || ws_bytes < w.bytes) return AGRL_E_WORKSPACE;
    cudaStream_t st = static_cast<cudaStream_t>(stream);

    AGRL_CUDA_TRY(cudaMemsetAsync(status, 0, sizeof(uint32_t), st));
    AGRL_CUDA_TRY(cudaMemsetAsync(w.counters, 0, 4 * sizeof(int32_t), st));
    if (num_q == 0) {                      // no query at all -> no valid query (pyx:227)
        const uint32_t one = AGRL_ST_NO_VALID_QUERY;
        AGRL_CUDA_TRY(cudaMemcpyAsync(status, &one, sizeof(one), cudaMemcpyHostToDevice, st));
        return AGRL_OK;
    }
    rc = narrow_labels(q_pids, g_pids, q_camids, g_camids, num_q, num_g, w.q_pid, w.g_pid, w.q_cam, w.g_cam,
                       status, st);
    if (rc) return rc;

    MarketArgs a;
    a.dist = distmat; a.ld = ld;
    a.q_pid = w.q_pid; a.q_cam = w.q_cam; a.g_pid = w.g_pid; a.g_cam = w.g_cam;
    a.num_g = static_cast<int>(num_g);
    a.res.num_q = static_cast<int>(num_q); a.res.rank_len = static_cast<int>(rank_len);
    a.res.ap = all_ap ? all_ap : w.ap_f32;
    a.res.first_hit = w.first; a.res.kept = w.kept;
    a.res.flags = reinterpret_cast<uint32_t *>(w.counters + 1);
    a.overflow_list = w.overflow_list; a.overflow_count = w.counters;

    const size_t smem = kListCap * 8 + kFastBins * kRankThreads * 2;
    static_assert(kFastBins * kRankThreads * 2 >= (kListCap + 1) * 4, "hist32 must fit in the hist16 region");
    AGRL_CUDA_TRY(cudaFuncSetAttribute(rank_market_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       static_cast<int>(smem)));
    rank_market_kernel<<<static_cast<unsigned>(num_q), kRankThreads, smem, st>>>(a);
    AGRL_LAUNCH_CHECK(st, "rank_market");
    rank_market_overflow_kernel<<<kOverflowCtas, kRankThreads, 0, st>>>(a, w.slab_keys, w.slab_terms);
    AGRL_LAUNCH_CHECK(st, "rank_market_overflow");
    rank_market_finish_kernel<<<1, 1024, 0, st>>>(a.res, w.hist, cmc, map, num_valid, status);
    AGRL_LAUNCH_CHECK(st, "rank_market_finish");
    return AGRL_OK;
}

extern "C" int agrl_rank_mars_dev(const float *distmat, int64_t ld,
                                  const int64_t *q_pids, const int64_t *g_pids,
                                  const int64_t *q_camids, const int64_t *g_camids,
                                  int64_t num_q, int64_t num_g, int64_t max_rank,
                                  double *cmc, double *map, double *all_ap, uint32_t *status,
                                  void *ws, size_t ws_bytes, void *stream) {
    int rc = check_rank_args(distmat, q_pids, g_pids, q_camids, g_camids, num_q, num_g, max_rank, ld);
    if (rc) return rc;
    if (!cmc || !map || !status || num_q < 1) return AGRL_E_INVALID;
    if (max_rank > num_g || max_rank > 8192) return AGRL_E_UNSUPPORTED;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    MarsArgs a;
    memset(&a, 0, sizeof(a));
    a.res.ap = all_ap;
    a.status = status;
    RankWorkspace w;
    rc = launch_rank_mars<false>(a, w, distmat, ld, q_pids, g_pids, q_camids, g_camids, num_q, num_g, max_rank,
                                 ws, ws_bytes, st);
    if (rc) return rc;
    rank_mars_finish_kernel<<<1, 1024, 0, st>>>(a.res, w.hist, cmc, map);
    AGRL_LAUNCH_CHECK(st, "rank_mars_finish");
    return AGRL_OK;
}

// ---- gallery-sharded MARS metric (SURVEY.md section 8e) --------------------------------------------
extern "C" int agrl_rank_mars_partial_dev(const float *distmat, int64_t ld,
                                          const int64_t *q_pids, const int64_t *g_pids,
                                          const int64_t *q_camids, const int64_t *g_camids,
                                          int64_t num_q, int64_t num_g, int64_t max_rank, int64_t index_offset,
                                          uint64_t *keys, uint8_t *cls, int32_t *ngood, uint32_t *status,
                                          void *ws, size_t ws_bytes, void *stream) {
    int rc = check_rank_args(distmat, q_pids, g_pids, q_camids, g_camids, num_q, num_g, max_rank, ld);
    if (rc) return rc;
    if (!keys || !cls || !ngood || !status || num_q < 1 || index_offset < 0) return AGRL_E_INVALID;
    if (max_rank > 8192 || index_offset + num_g > 0xFFFFFFFFll) return AGRL_E_UNSUPPORTED;
    MarsArgs a;
    memset(&a, 0, sizeof(a));
    a.status = status;
    a.part_keys = keys; a.part_cls = cls; a.part_ngood = ngood;
    a.index_offset = static_cast<uint32_t>(index_offset);
    RankWorkspace w;
    return launch_rank_mars<true>(a, w, distmat, ld, q_pids, g_pids, q_camids, g_camids, num_q, num_g, max_rank,
                                  ws, ws_bytes, static_cast<cudaStream_t>(stream));
}

extern "C" int agrl_rank_mars_merge_dev(const uint64_t *keys, const uint8_t *cls, const int32_t *ngood,
                                        int64_t parts, int64_t num_q, int64_t max_rank,
                                        double *cmc, double *map, double *all_ap, uint32_t *status,
                                        void *ws, size_t ws_bytes, void *stream) {
    if (!keys || !cls || !ngood || !cmc || !map || !status) return AGRL_E_INVALID;
    if (parts < 1 || num_q < 1 || max_rank < 1) return AGRL_E_INVALID;
    if (parts * max_rank > 16384 || num_q > INT32_MAX / 2) return AGRL_E_UNSUPPORTED;
    int rc = agrl_device_ok();
    if (rc) return rc;
    RankWorkspace w = carve_rank(ws, num_q, 0, max_rank);
    if (!ws || ws_bytes < w.bytes) return AGRL_E_WORKSPACE;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    MarsMergeArgs m;
    m.keys = keys; m.cls = cls; m.ngood = ngood;
    m.parts = static_cast<int>(parts);
    const int n2 = pow2_at_least(parts * max_rank, 2);
    m.n2 = n2;
    m.res.num_q = static_cast<int>(num_q); m.res.max_rank = static_cast<int>(max_rank);
    m.res.ap = all_ap ? all_ap : w.ap_f64;
    m.res.first_pos = w.first;
    m.status = status;
    const size_t smem = (static_cast<size_t>(n2) + ((max_rank + 15) & ~static_cast<size_t>(15))) * 9;
    AGRL_CUDA_TRY(cudaFuncSetAttribute(rank_mars_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       static_cast<int>(smem)));
    AGRL_LAUNCH_BEGIN(st);          // (profiling: do not charge the collectives queued ahead on this stream to the merge)
    rank_mars_merge_kernel<<<static_cast<unsigned>(num_q), kRankThreads, smem, st>>>(m);
    AGRL_LAUNCH_CHECK(st, "rank_mars_merge");
    rank_mars_finish_kernel<<<1, 1024, 0, st>>>(m.res, w.hist, cmc, map);
    AGRL_LAUNCH_CHECK(st, "rank_mars_finish");
    return AGRL_OK;
}

// ---- gallery-sharded market1501 metric ---------------------------------------------------------------
extern "C" int agrl_rank_market1501_count_dev(const int64_t *q_pids, const int64_t *g_pids,
                                              const int64_t *q_camids, const int64_t *g_camids,
                                              int64_t num_q, int64_t num_g, int32_t *max_count, uint32_t *status,
                                              void *ws, size_t ws_bytes, void *stream) {
    if (!q_pids || !g_pids || !q_camids || !g_camids || !max_count || !status) return AGRL_E_INVALID;
    if (num_q < 1 || num_g < 1 || num_q > INT32_MAX / 2 || num_g > INT32_MAX / 2) return AGRL_E_INVALID;
    int rc = agrl_device_ok();
    if (rc) return rc;
    RankWorkspace w = carve_rank(ws, num_q, num_g, 1);
    if (!ws || ws_bytes < w.bytes) return AGRL_E_WORKSPACE;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    AGRL_CUDA_TRY(cudaMemsetAsync(status, 0, sizeof(uint32_t), st));
    AGRL_CUDA_TRY(cudaMemsetAsync(max_count, 0, sizeof(int32_t), st));
    rc = narrow_labels(q_pids, g_pids, q_camids, g_camids, num_q, num_g, w.q_pid, w.g_pid, w.q_cam, w.g_cam,
                       status, st);
    if (rc) return rc;
    MarketShardArgs a = shard_args(&w, nullptr, 0, num_q, num_g, 0);
    a.max_count = max_count;
    AGRL_LAUNCH_BEGIN(st);
    rank_market_gather_kernel<true><<<static_cast<unsigned>(num_q), kRankThreads, 0, st>>>(a);
    AGRL_LAUNCH_CHECK(st, "rank_market_count");
    return AGRL_OK;
}

extern "C" int agrl_rank_market1501_gather_dev(const float *distmat, int64_t ld,
                                               const int64_t *q_pids, const int64_t *g_pids,
                                               const int64_t *q_camids, const int64_t *g_camids,
                                               int64_t num_q, int64_t num_g, int64_t index_offset, int64_t cap,
                                               uint64_t *keys, int32_t *npos, int32_t *njunk, uint32_t *status,
                                               void *ws, size_t ws_bytes, void *stream) {
    int rc = check_rank_args(distmat, q_pids, g_pids, q_camids, g_camids, num_q, num_g, 1, ld);
    if (rc) return rc;
    if (!keys || !npos || !njunk || !status || num_q < 1 || cap < 1 || index_offset < 0) return AGRL_E_INVALID;
    if (index_offset + num_g > 0x7FFFFFFFll) return AGRL_E_UNSUPPORTED;
    if ((rc = agrl_device_ok())) return rc;
    RankWorkspace w = carve_rank(ws, num_q, num_g, 1);
    if (!ws || ws_bytes < w.bytes) return AGRL_E_WORKSPACE;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    AGRL_CUDA_TRY(cudaMemsetAsync(status, 0, sizeof(uint32_t), st));
    rc = narrow_labels(q_pids, g_pids, q_camids, g_camids, num_q, num_g, w.q_pid, w.g_pid, w.q_cam, w.g_cam,
                       status, st);
    if (rc) return rc;
    MarketShardArgs a = shard_args(&w, distmat, ld, num_q, num_g, index_offset);
    a.cap = static_cast<int>(cap); a.keys = keys; a.npos = npos; a.njunk = njunk;
    AGRL_LAUNCH_BEGIN(st);
    rank_market_gather_kernel<false><<<static_cast<unsigned>(num_q), kRankThreads, 0, st>>>(a);
    AGRL_LAUNCH_CHECK(st, "rank_market_gather");
    return AGRL_OK;
}

extern "C" int agrl_rank_market1501_bin_dev(const float *distmat, int64_t ld, int64_t num_q, int64_t num_g,
                                            int64_t index_offset, const uint64_t *keys_all, int64_t parts, int64_t cap,
                                            int32_t *cnt, uint64_t *sorted, void *stream) {
    if (!distmat || !keys_all || !cnt || !sorted || num_q < 1 || num_g < 1 || parts < 1 || cap < 1 || ld < num_g) return AGRL_E_INVALID;
    if (parts * cap > 8192 || index_offset + num_g > 0x7FFFFFFFll) return AGRL_E_UNSUPPORTED;
    int rc = agrl_device_ok();
    if (rc) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    MarketShardArgs a = shard_args(nullptr, distmat, ld, num_q, num_g, index_offset);
    a.cap = static_cast<int>(cap); a.parts = static_cast<int>(parts); a.n2 = pow2_at_least(parts * cap, 2);
    a.keys = const_cast<uint64_t *>(keys_all); a.cnt = cnt; a.sorted = sorted;
    const size_t smem = static_cast<size_t>(a.n2) * 8 + (static_cast<size_t>(a.n2) + 1) * 4;
    AGRL_CUDA_TRY(cudaFuncSetAttribute(rank_market_bin_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    AGRL_LAUNCH_BEGIN(st);
    rank_market_bin_kernel<<<static_cast<unsigned>(num_q), kRankThreads, smem, st>>>(a);
    AGRL_LAUNCH_CHECK(st, "rank_market_bin");
    return AGRL_OK;
}

extern "C" int64_t agrl_rank_market1501_list_len(int64_t parts, int64_t cap) {
    if (parts < 1 || cap < 1 || parts * cap > 8192) return 0;
    return pow2_at_least(parts * cap, 2);
}

extern "C" int agrl_rank_market1501_finalize_dev(const int32_t *cnt_total, const uint64_t *sorted,
                                                 const int32_t *npos_total, const int32_t *njunk_total,
                                                 int64_t num_q, int64_t num_g_total, int64_t parts, int64_t cap, int64_t max_rank,
                                                 float *cmc, float *map, float *all_ap, int64_t *num_valid, uint32_t *status,
                                                 void *ws, size_t ws_bytes, void *stream) {
    if (!cnt_total || !sorted || !npos_total || !njunk_total || !cmc || !map || !status) return AGRL_E_INVALID;
    if (num_q < 1 || num_g_total < 1 || parts < 1 || cap < 1 || max_rank < 1 || parts * cap > 8192) return AGRL_E_INVALID;
    int rc = agrl_device_ok();
    if (rc) return rc;
    const int64_t rank_len = max_rank < num_g_total ? max_rank : num_g_total;
    const int n2 = pow2_at_least(parts * cap, 2);
    Carver c(ws);
    RankWorkspace w = carve_rank(ws, num_q, 0, rank_len);
    c.off = w.bytes;
    double *terms = c.take<double>(static_cast<size_t>(num_q) * n2);
    if (!ws || ws_bytes < c.total()) return AGRL_E_WORKSPACE;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    AGRL_CUDA_TRY(cudaMemsetAsync(w.counters, 0, 4 * sizeof(int32_t), st));
    MarketFinalArgs f;
    f.cnt = cnt_total; f.sorted = sorted; f.npos = npos_total; f.njunk = njunk_total;
    f.n2 = n2; f.num_g_total = num_g_total; f.terms = terms;
    f.res.num_q = static_cast<int>(num_q); f.res.rank_len = static_cast<int>(rank_len);
    f.res.ap = all_ap ? all_ap : w.ap_f32; f.res.first_hit = w.first; f.res.kept = w.kept;
    f.res.flags = reinterpret_cast<uint32_t *>(w.counters + 1);
    const int wpb = kRankThreads / 32;
    AGRL_LAUNCH_BEGIN(st);
    rank_market_finalize_kernel<<<static_cast<unsigned>((num_q + wpb - 1) / wpb), kRankThreads, 0, st>>>(f);
    AGRL_LAUNCH_CHECK(st, "rank_market_finalize");
    rank_market_finish_kernel<<<1, 1024, 0, st>>>(f.res, w.hist, cmc, map, num_valid, status);
    AGRL_LAUNCH_CHECK(st, "rank_market_finish");
    return AGRL_OK;
}

extern "C" size_t agrl_rank_market1501_finalize_workspace_bytes(int64_t num_q, int64_t parts, int64_t cap, int64_t max_rank) {
    if (num_q < 1 || parts < 1 || cap < 1 || max_rank < 1 || parts * cap > 8192) return 0;
    return carve_rank(nullptr, num_q, 0, max_rank).bytes + align_up(static_cast<size_t>(num_q) * pow2_at_least(parts * cap, 2) * 8, 256) + 256;
}

// ------------------------------------------------------------------------------------------------
// MARS metric after the fused distance -> top-k (agrl_distance_topk_dev): the candidates' class bytes and the per-query
// good-image count (rank.py:166-169) from the labels alone.  The count must not cost a pass over num_q x num_g label
// pairs (10^10 for the retrieval sweep): the queries' identities go into two small open-addressing tables -- by pid and
// by (pid, camera), slot = index of a representative query -- one pass over the gallery labels counts into them, and
// good(q) = count[pid_q] - count[pid_q, cam_q].  O(num_q + num_g).
// ------------------------------------------------------------------------------------------------
namespace agrl {

struct ClassifyWorkspace {
    int32_t *q_pid, *q_cam, *g_pid, *g_cam;
    int32_t *tab_p, *tab_pc, *cnt_p, *cnt_pc;      // [slots] each
    int slots;
    size_t bytes;
};

static ClassifyWorkspace carve_classify(void *ws, int64_t nq, int64_t ng) {
    Carver c(ws);
    ClassifyWorkspace w;
    w.q_pid = c.take<int32_t>(nq); w.q_cam = c.take<int32_t>(nq);
    w.g_pid = c.take<int32_t>(ng); w.g_cam = c.take<int32_t>(ng);
    const int slots = pow2_at_least(4 * nq, 64);
    w.slots = slots;
    w.tab_p = c.take<int32_t>(4 * static_cast<size_t>(slots));      // tab_p | tab_pc | cnt_p | cnt_pc, contiguous
    w.tab_pc = w.tab_p ? w.tab_p + slots : nullptr;
    w.cnt_p = w.tab_p ? w.tab_p + 2 * slots : nullptr;
    w.cnt_pc = w.tab_p ? w.tab_p + 3 * slots : nullptr;
    w.bytes = c.total();
    return w;
}

__device__ __forceinline__ uint32_t hash_u32(uint32_t x) {
    x ^= x >> 16; x *= 0x7feb352dU; x ^= x >> 15; x *= 0x846ca68bU; x ^= x >> 16;
    return x;
}
__device__ __forceinline__ uint32_t hash_pid_cam(int pid, int cam) {
    return hash_u32(static_cast<uint32_t>(pid) * 0x9E3779B1U + hash_u32(static_cast<uint32_t>(cam) + 0x85EBCA6BU));
}

// Linear probing in `tab` from slot `hash`: walks until the slot is empty or holds a query that match()es; returns
// that slot, or -1 at an empty slot.  kClaim: an empty slot is taken for query q (atomicCAS), which ends the walk.
template <bool kClaim, class Match>
__device__ __forceinline__ int probe(int32_t *tab, uint32_t hash, int slots, int q, Match match) {
    const uint32_t mask = static_cast<uint32_t>(slots - 1);
    for (uint32_t h = hash & mask;; h = (h + 1) & mask) {
        const int cur = kClaim ? atomicCAS(&tab[h], -1, q) : tab[h];
        if (cur == -1) return -1;
        if (match(cur)) return static_cast<int>(h);
    }
}

// slot of pid in tab_p / of (pid, cam) in tab_pc, -1 if absent; kClaim inserts query q
template <bool kClaim>
__device__ __forceinline__ int probe_pid(const ClassifyWorkspace &w, int pid, int q = -1) {
    return probe<kClaim>(w.tab_p, hash_u32(static_cast<uint32_t>(pid)), w.slots, q,
                         [&](int r) { return w.q_pid[r] == pid; });
}
template <bool kClaim>
__device__ __forceinline__ int probe_pid_cam(const ClassifyWorkspace &w, int pid, int cam, int q = -1) {
    return probe<kClaim>(w.tab_pc, hash_pid_cam(pid, cam), w.slots, q,
                         [&](int r) { return w.q_pid[r] == pid && w.q_cam[r] == cam; });
}

__global__ void classify_insert_kernel(ClassifyWorkspace w, int nq) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    const int pid = w.q_pid[q], cam = w.q_cam[q];
    probe_pid<true>(w, pid, q);
    probe_pid_cam<true>(w, pid, cam, q);
}

__global__ void classify_count_kernel(ClassifyWorkspace w, int64_t ng) {
    for (int64_t j = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; j < ng;
         j += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const int pid = w.g_pid[j], cam = w.g_cam[j];
        const int hp = probe_pid<false>(w, pid);
        if (hp >= 0) atomicAdd(&w.cnt_p[hp], 1);
        const int hpc = probe_pid_cam<false>(w, pid, cam);
        if (hpc >= 0) atomicAdd(&w.cnt_pc[hpc], 1);
    }
}

// one thread per (query, slot): class byte of the listed gallery item; thread of slot 0 also looks up the good count
__global__ void classify_keys_kernel(ClassifyWorkspace w, const uint64_t *__restrict__ keys, int nq, int K, int64_t ng,
                                     uint32_t index_offset, uint8_t *cls, int32_t *ngood) {
    const int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
    if (i >= static_cast<int64_t>(nq) * K) return;
    const int q = static_cast<int>(i / K), n = static_cast<int>(i - static_cast<int64_t>(q) * K);
    const int pid = w.q_pid[q], cam = w.q_cam[q];
    const uint64_t key = keys[i];
    uint8_t c = 0;
    if (key != kKeyMax) {
        const int64_t g = static_cast<int64_t>(static_cast<uint32_t>(key)) - index_offset;
        if (g >= 0 && g < ng) c = mars_class(w.g_pid[g], w.g_cam[g], pid, cam);
    }
    cls[i] = c;
    if (n == 0) {
        const int hp = probe_pid<false>(w, pid), hpc = probe_pid_cam<false>(w, pid, cam);
        ngood[q] = (hp >= 0 ? w.cnt_p[hp] : 0) - (hpc >= 0 ? w.cnt_pc[hpc] : 0);
    }
}

// the most gallery items that share a query's pid and camera, over the queries
__global__ void rank_junk_depth_kernel(ClassifyWorkspace w, int nq, int32_t *junk_depth) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    const int h = probe_pid_cam<false>(w, w.q_pid[q], w.q_cam[q]);
    if (h >= 0) atomicMax(junk_depth, w.cnt_pc[h]);
}

// Labels to int32, the queries' identities into the two tables, one pass over the gallery labels counting into them.
static int build_label_tables(const ClassifyWorkspace &w, const int64_t *q_pids, const int64_t *g_pids,
                              const int64_t *q_camids, const int64_t *g_camids, int64_t num_q, int64_t num_g,
                              uint32_t *status, cudaStream_t st) {
    int rc = narrow_labels(q_pids, g_pids, q_camids, g_camids, num_q, num_g, w.q_pid, w.g_pid, w.q_cam, w.g_cam,
                           status, st);
    if (rc) return rc;
    AGRL_CUDA_TRY(cudaMemsetAsync(w.tab_p, 0xFF, sizeof(int32_t) * 2 * w.slots, st));       // both tables: empty (-1)
    AGRL_CUDA_TRY(cudaMemsetAsync(w.cnt_p, 0, sizeof(int32_t) * 2 * w.slots, st));
    const int nq = static_cast<int>(num_q);
    classify_insert_kernel<<<(nq + 255) / 256, 256, 0, st>>>(w, nq);
    AGRL_LAUNCH_CHECK(st, "classify_insert");
    if (num_g > 0) {
        int cb = static_cast<int>((num_g + 255) / 256);
        if (cb > 8 * kNumSMs) cb = 8 * kNumSMs;
        classify_count_kernel<<<cb, 256, 0, st>>>(w, num_g);
        AGRL_LAUNCH_CHECK(st, "classify_count");
    }
    return AGRL_OK;
}

// ------------------------------------------------------------------------------------------------
// Ranked lists: each query's first k gallery items and their distances, from ascending key lists laid out
// [part][query][depth] (_partial, agrl_distance_topk_dev or the shards' lists after an all-gather).  One CTA per query:
//   1. every list into shared memory, without the query's junk items (same pid and camera) when asked: a stable
//      compaction, so each list stays ascending;
//   2. the rank merge of rank_mars_merge_kernel (merged_position) places the keys that land among the first k;
//   3. each key -> (global gallery index, distance), the tail padded with (-1, +inf).
// Dropping junk list by list is exact when every list holds its shard's first k + J keys, J at least the number of junk
// items any query has in that shard (agrl_rank_junk_depth_dev): an item among the first k kept ones of the whole gallery
// is among the first k kept ones of its own shard.
// ------------------------------------------------------------------------------------------------
struct ListsArgs {
    const uint64_t *keys;
    int             parts, num_q, depth, k;
    int64_t         num_g;
    const int32_t  *q_pid, *q_cam, *g_pid, *g_cam;   // q_pid == nullptr: no junk exclusion
    int64_t        *index_out;
    float          *dist_out;
    int64_t         ld_out;
};

__global__ void __launch_bounds__(kRankThreads)
rank_lists_kernel(ListsArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int D = a.depth, K = a.k;
    uint64_t *lists = reinterpret_cast<uint64_t *>(smem_raw);                 // parts * D
    uint64_t *head = lists + static_cast<size_t>(a.parts) * D;                // K: the merged head
    const int q = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const bool drop_junk = a.q_pid != nullptr;
    const int pid = drop_junk ? a.q_pid[q] : 0, cam = drop_junk ? a.q_cam[q] : 0;
    for (int p = warp; p < a.parts; p += kRankThreads / 32) {
        const uint64_t *src = a.keys + (static_cast<size_t>(p) * a.num_q + q) * D;
        uint64_t *dst = lists + static_cast<size_t>(p) * D;
        int n = 0;
        for (int base = 0; base < D; base += 32) {
            const int j = base + lane;
            const uint64_t key = j < D ? src[j] : kKeyMax;
            bool keep = key != kKeyMax;
            if (keep && drop_junk) {
                const uint32_t g = static_cast<uint32_t>(key);
                keep = !(g < a.num_g && a.g_pid[g] == pid && a.g_cam[g] == cam);
            }
            const uint32_t m = __ballot_sync(0xffffffffu, keep);
            if (keep) dst[n + __popc(m & ((1u << lane) - 1u))] = key;
            n += __popc(m);
        }
        for (int j = n + lane; j < D; j += 32) dst[j] = kKeyMax;
    }
    for (int i = tid; i < K; i += kRankThreads) head[i] = kKeyMax;
    __syncthreads();
    for (int i = tid; i < a.parts * K; i += kRankThreads) {
        const int p = i / K, pos = i - p * K;
        const uint64_t key = lists[static_cast<size_t>(p) * D + pos];
        if (key == kKeyMax) continue;
        const int rank = merged_position(lists, a.parts, D, K, p, pos, key);
        if (rank < K) head[rank] = key;
    }
    __syncthreads();
    int64_t *idx = a.index_out + static_cast<size_t>(q) * a.ld_out;
    float *dst = a.dist_out + static_cast<size_t>(q) * a.ld_out;
    for (int i = tid; i < K; i += kRankThreads) {
        const uint64_t key = head[i];
        const bool real = key != kKeyMax;
        idx[i] = real ? static_cast<int64_t>(static_cast<uint32_t>(key)) : -1;
        dst[i] = real ? mono_key_value(static_cast<uint32_t>(key >> 32)) : __uint_as_float(0x7F800000u);
    }
}

}  // namespace agrl

extern "C" size_t agrl_rank_mars_classify_workspace_bytes(int64_t num_q, int64_t num_g) {
    if (num_q < 0 || num_g < 0) return 0;
    return carve_classify(nullptr, num_q, num_g).bytes;
}

extern "C" int agrl_rank_mars_classify_dev(const uint64_t *keys, const int64_t *q_pids, const int64_t *g_pids,
                                           const int64_t *q_camids, const int64_t *g_camids,
                                           int64_t num_q, int64_t num_g, int64_t max_rank, int64_t index_offset,
                                           uint8_t *cls, int32_t *ngood, uint32_t *status,
                                           void *ws, size_t ws_bytes, void *stream) {
    if (!keys || !q_pids || !g_pids || !q_camids || !g_camids || !cls || !ngood || !status) return AGRL_E_INVALID;
    if (num_q < 1 || num_g < 0 || max_rank < 1 || index_offset < 0) return AGRL_E_INVALID;
    if (num_q > (1 << 28) || index_offset + num_g > 0xFFFFFFFFll) return AGRL_E_UNSUPPORTED;
    int rc = agrl_device_ok();
    if (rc) return rc;
    ClassifyWorkspace w = carve_classify(ws, num_q, num_g);
    if (!ws || ws_bytes < w.bytes) return AGRL_E_WORKSPACE;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    rc = build_label_tables(w, q_pids, g_pids, q_camids, g_camids, num_q, num_g, status, st);
    if (rc) return rc;
    const int64_t total = num_q * max_rank;
    classify_keys_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, st>>>(
        w, keys, static_cast<int>(num_q), static_cast<int>(max_rank), num_g, static_cast<uint32_t>(index_offset), cls,
        ngood);
    AGRL_LAUNCH_CHECK(st, "classify_keys");
    return AGRL_OK;
}

// ---- ranked lists ------------------------------------------------------------------------------------
extern "C" int agrl_rank_junk_depth_dev(const int64_t *q_pids, const int64_t *g_pids, const int64_t *q_camids,
                                        const int64_t *g_camids, int64_t num_q, int64_t num_g, int32_t *junk_depth,
                                        uint32_t *status, void *ws, size_t ws_bytes, void *stream) {
    if (!q_pids || !q_camids || !junk_depth || !status || (num_g > 0 && (!g_pids || !g_camids))) return AGRL_E_INVALID;
    if (num_q < 1 || num_g < 0) return AGRL_E_INVALID;
    if (num_q > (1 << 28) || num_g > INT32_MAX) return AGRL_E_UNSUPPORTED;
    int rc = agrl_device_ok();
    if (rc) return rc;
    ClassifyWorkspace w = carve_classify(ws, num_q, num_g);
    if (!ws || ws_bytes < w.bytes) return AGRL_E_WORKSPACE;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    AGRL_CUDA_TRY(cudaMemsetAsync(status, 0, sizeof(uint32_t), st));
    AGRL_CUDA_TRY(cudaMemsetAsync(junk_depth, 0, sizeof(int32_t), st));
    rc = build_label_tables(w, q_pids, g_pids, q_camids, g_camids, num_q, num_g, status, st);
    if (rc) return rc;
    const int nq = static_cast<int>(num_q);
    rank_junk_depth_kernel<<<(nq + 255) / 256, 256, 0, st>>>(w, nq, junk_depth);
    AGRL_LAUNCH_CHECK(st, "rank_junk_depth");
    return AGRL_OK;
}

extern "C" int agrl_rank_lists_dev(const uint64_t *keys, int64_t parts, int64_t num_q, int64_t depth, int64_t k,
                                   const int64_t *q_pids, const int64_t *g_pids, const int64_t *q_camids,
                                   const int64_t *g_camids, int64_t num_g, int exclude_junk,
                                   int64_t *index_out, float *dist_out, int64_t ld_out, uint32_t *status,
                                   void *ws, size_t ws_bytes, void *stream) {
    if (!keys || !index_out || !dist_out || !status) return AGRL_E_INVALID;
    if (parts < 1 || num_q < 1 || k < 1 || depth < k || ld_out < k) return AGRL_E_INVALID;
    if (exclude_junk && (!q_pids || !g_pids || !q_camids || !g_camids || num_g < 1)) return AGRL_E_INVALID;
    if (depth > 8192 || parts * depth > 16384 || num_q > INT32_MAX / 2) return AGRL_E_UNSUPPORTED;
    if (exclude_junk && num_g > 0xFFFFFFFFll) return AGRL_E_UNSUPPORTED;
    int rc = agrl_device_ok();
    if (rc) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    AGRL_CUDA_TRY(cudaMemsetAsync(status, 0, sizeof(uint32_t), st));
    ListsArgs a;
    memset(&a, 0, sizeof(a));
    if (exclude_junk) {
        ClassifyWorkspace w = carve_classify(ws, num_q, num_g);
        if (!ws || ws_bytes < w.bytes) return AGRL_E_WORKSPACE;
        rc = narrow_labels(q_pids, g_pids, q_camids, g_camids, num_q, num_g, w.q_pid, w.g_pid, w.q_cam, w.g_cam,
                           status, st);
        if (rc) return rc;
        a.q_pid = w.q_pid; a.q_cam = w.q_cam; a.g_pid = w.g_pid; a.g_cam = w.g_cam;
        a.num_g = num_g;
    }
    a.keys = keys;
    a.parts = static_cast<int>(parts); a.num_q = static_cast<int>(num_q);
    a.depth = static_cast<int>(depth); a.k = static_cast<int>(k);
    a.index_out = index_out; a.dist_out = dist_out; a.ld_out = ld_out;
    const size_t smem = static_cast<size_t>(parts * depth + k) * 8;
    AGRL_CUDA_TRY(cudaFuncSetAttribute(rank_lists_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       static_cast<int>(smem)));
    AGRL_LAUNCH_BEGIN(st);
    rank_lists_kernel<<<static_cast<unsigned>(num_q), kRankThreads, smem, st>>>(a);
    AGRL_LAUNCH_CHECK(st, "rank_lists");
    return AGRL_OK;
}
