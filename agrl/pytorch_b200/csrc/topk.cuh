// topk.cuh -- stable per-row top-K selection shared by the MARS evaluator (rank.cu) and the k-reciprocal
// re-ranking (rerank.cu): keys are (order-preserving distance bits << 32 | column index), so unsigned key order is
// numpy.argsort(kind='stable') order.
#pragma once
#include "common.cuh"

namespace agrl {

constexpr int kRankThreads = 256;
constexpr uint64_t kKeyMax = 0xFFFFFFFFFFFFFFFFull;

// ------------------------------------------------------------------------------------------------
// shared-memory bitonic sort of n2 (power of two) uint64 keys by `nthreads` cooperating threads;
// kPayload: payload[i] is swapped along with keys[i]
// ------------------------------------------------------------------------------------------------
template <bool kWarpOnly, bool kPayload = false>
__device__ __forceinline__ void bitonic_sort_u64(uint64_t *keys, int n2, int tid, int nthreads,
                                                 uint8_t *payload = nullptr) {
    for (int k = 2; k <= n2; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int t = tid; t < (n2 >> 1); t += nthreads) {
                const int lo = ((t & ~(j - 1)) << 1) | (t & (j - 1));
                const int hi = lo | j;
                const uint64_t a = keys[lo], b = keys[hi];
                const bool up = ((lo & k) == 0);
                if ((a > b) == up) {
                    keys[lo] = b; keys[hi] = a;
                    if (kPayload) { const uint8_t c = payload[lo]; payload[lo] = payload[hi]; payload[hi] = c; }
                }
            }
            // (CTA-wide barriers only around the steps that cross 64-element blocks, __syncwarp elsewhere: measured, no gain)
            if (kWarpOnly) __syncwarp(); else __syncthreads();
        }
    }
}

constexpr int kMarsTile = 1024;                     // elements examined between buffer checks


// Running top-K of one row: candidates below the threshold (K-th smallest key so far) go to a
// shared buffer, which is sorted and cut back to K -- tightening the threshold -- as soon as it holds more than
// max(4 K, 128) keys (or the next tile could overflow it).  The first tile is short (one element per thread) so that a
// cheap sort establishes a threshold early.  Sorts cover just the occupied power-of-two prefix and stay at 256-512 keys:
// waiting until the buffer was nearly full cost one 2048-key sort (66 steps of 4 compare-exchanges per thread) per row,
// 86 % of the MARS evaluator's samples under ncu.  On return buf[0..valid) holds the min(K, n) smallest keys in order.
__device__ __forceinline__ int select_topk(const float *__restrict__ row, int ng, int K, int L,
                                                uint64_t *buf, int *s_cnt, unsigned long long *s_thr, int tid) {
    int base = 0;
    bool first = true;
    const int room = L - kMarsTile;
    const int trigger = min(room, max(4 * K, 128));
    while (base < ng) {
        const uint64_t thr = *s_thr;
        const int tile = (first && K <= kRankThreads / 2) ? kRankThreads : kMarsTile;
        if (tile == kRankThreads) {
            const int j = base + tid;
            if (j < ng) {
                const uint64_t key = rank_key(row[j], static_cast<uint32_t>(j));
                if (key < thr) buf[atomicAdd(s_cnt, 1)] = key;
            }
        } else {
            const int j = base + tid * 4;               // thread t owns 4 consecutive elements of the tile
            float d[4];
            int n_here = 0;
            if (j + 3 < ng && ((reinterpret_cast<uintptr_t>(row + j) & 15u) == 0)) {
                const float4 x = __ldg(reinterpret_cast<const float4 *>(row + j));
                d[0] = x.x; d[1] = x.y; d[2] = x.z; d[3] = x.w; n_here = 4;
            } else {
                for (int k = 0; k < 4; ++k) if (j + k < ng) { d[k] = row[j + k]; n_here = k + 1; }
            }
            for (int k = 0; k < n_here; ++k) {
                const uint64_t key = rank_key(d[k], static_cast<uint32_t>(j + k));
                if (key < thr) buf[atomicAdd(s_cnt, 1)] = key;    // *s_cnt <= L - kMarsTile before a tile
            }
        }
        base += tile;
        __syncthreads();
        const int cnt = *s_cnt;
        __syncthreads();                   // everyone holds the same cnt before anyone appends again
        const bool last = (base >= ng);
        if (cnt > trigger || last || first) {
            int n2 = 2;
            while (n2 < cnt) n2 <<= 1;                 // cnt <= L and L is a power of two
            for (int i = cnt + tid; i < n2; i += kRankThreads) buf[i] = kKeyMax;
            __syncthreads();
            bitonic_sort_u64<false>(buf, n2, tid, kRankThreads);
            if (tid == 0) {
                const int keep = cnt < K ? cnt : K;
                *s_cnt = keep;
                if (keep == K) *s_thr = buf[K - 1];    // later keys must beat the current K-th
            }
            __syncthreads();
        }
        first = false;
    }
    return *s_cnt;
}


}  // namespace agrl
