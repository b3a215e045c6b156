// gemm_sm100.cuh -- split-bf16 GEMM on tcgen05 tensor cores (sm_100a), shared by the distance matrix
// (distance.cu) and the graph layers' X.W^T (head.cu).
//
//   D[M,N] = sum over plane pairs (pa,pb) of  A_pa[M,K] . B_pb[N,K]^T        (both operands K-major)
//
// fp32 operands are pre-split into P bf16 planes (x = x0 + x1 (+ x2), each the bf16 rounding of the
// remaining residual), laid out [P][rows][K_pad] so ONE 3-D TMA descriptor per operand serves every
// plane.  P = 3 keeps the six products whose weight is >= 2^-16 of the leading one (fp32-accurate,
// 24 operand bits); P = 2 keeps three (about 16 operand bits).  Products are exact in the tensor
// core; accumulation is fp32 in TMEM.
//
// Kernel anatomy (one persistent CTA per SM, 256 threads, warp-specialised):
//   warp 0      TMA producer: cp.async.bulk.tensor (128B swizzle) of the A and B plane tiles into a
//               ring of shared-memory stages, completion on mbarriers
//   warp 1      MMA issuer: one lane issues tcgen05.mma (cta_group::1, 128 x BN x 16, kind::f16),
//               tcgen05.commit frees the smem stage / publishes the accumulator
//   warp 2      TMEM allocator (2 stages x [main | correction] x 128 columns = all 512 columns)
//   warps 4..   epilogue: tcgen05.ld (32 lanes x 32 columns) + fused element-wise functor; either
//               4 warps transposing through padded smem so stores are full 128 B lines at any row
//               alignment (distance), or 8 warps doing 16-byte accesses straight from registers with
//               the residual tile prefetched into L2 during the mainloop (graph layer)
// The accumulator is double-buffered in TMEM, so the epilogue of tile i overlaps the MMAs of tile i+1.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>

#include "common.cuh"

namespace agrl {
namespace gemm {

constexpr int BM = 128, BK = 64;                     // CTA tile rows; BK bf16 = one 128-byte swizzle row
constexpr int UMMA_K = 16;
constexpr int kTileBytesA = BM * BK * 2;             // 16 KiB: one plane of an A tile
constexpr int kCtrlWarps = 4;                        // TMA producer, MMA issuer, TMEM allocator, spare
constexpr int kAccStages = 2;
constexpr int kTmemCols = 512;                       // all of TMEM: 2 stages x 256 columns
constexpr int kEpiPad = 33;
constexpr int kEpiBytes = 4 * 32 * kEpiPad * 4;       // transpose staging of the 4-warp (scalar-store) epilogue

// P      operand planes (2: three products, 3: six products)
// BN     tile width: 128 or 256 (UMMA 128 x BN x 16)
// kSplit keep the dominant a0.b0 sum and the correction products in separate TMEM accumulators
//        (needs 2*BN columns per stage, hence BN = 128)
// kChunkKb > 0: the accumulator is drained every kChunkKb k-blocks and summed in registers with
//        round-to-nearest fp32 adds (the tensor core truncates on accumulate; short chains keep that
//        bias below the fp32 rounding of the result).  Needs 8 epilogue warps (64 sums per thread).
// kPair  CTA pairs (cta_group::2): a 256 x BN tile per pair of SMs, each CTA loading its 128 rows of A and HALF of the B
//        tile.  Nothing for the bf16 modes (three / six products per loaded byte: MMA- or power-bound), but the modes
//        with FEWER products per byte -- the fp16 + e4m3 graph layers -- are bound by the operand fill with one CTA
//        per tile, which the halved B traffic removes (16.0 -> 12.05 ms per pass).  The fp16 x 2 distance GEMM gained
//        nothing from pairs; it is paced by its 128-wide MMAs (see kWideB).
template <int P, int BN, bool kSplit, bool kDirect = false, int kChunkKb = 0, bool kPair = false> struct Config {
    // epilogue flavour: kDirect = registers -> 16-byte global accesses, 8 warps (two per TMEM lane
    // quarter, half the columns each), no smem; otherwise 4 warps and a padded smem transpose so
    // that stores are coalesced along rows of arbitrary alignment.
    static_assert(kChunkKb == 0 || (!kDirect && BN == 128), "chunked accumulation: 128-wide tiles, smem-transposed stores");
    static constexpr int kEpiWarps = (kDirect || kChunkKb > 0) ? 8 : 4;
    static constexpr int kThreads = 32 * (kCtrlWarps + kEpiWarps);
    static_assert(BN == 128 || BN == 256, "tile width");
    static_assert(!kSplit || BN == 128, "two accumulators of 256 columns do not fit twice in TMEM");
    static constexpr int kLoadN = kPair ? BN / 2 : BN;                  // rows of the B tile this CTA loads
    static constexpr int kTileBytesB = kLoadN * BK * 2;
    static constexpr int kStageBytes = P * (kTileBytesA + kTileBytesB);
    static constexpr int kTileM = kPair ? 2 * BM : BM;                  // rows per scheduled tile
    static constexpr int kStages = (200 * 1024) / kStageBytes;          // 96 KiB stages -> 2, 64 KiB -> 3
    static constexpr int kAccCols = kSplit ? 2 * BN : BN;               // columns per accumulator stage
    static constexpr int kNumPairs = (P == 3) ? 6 : (P == 2 ? 3 : 1);
    static_assert(kStages >= 2 && kAccStages * kAccCols <= kTmemCols, "resources");
    static constexpr int kEpiSmem = kDirect ? 0 : (kEpiWarps / 4) * kEpiBytes;
    // Register cap (384 threads x 144 / 168 registers fit the 64 K file; one CTA per SM).
    static constexpr int kMaxRegs = 168;
    static constexpr int kChunk = kChunkKb;
    // dynamic smem: stages | epilogue staging | barriers ; +1024 for manual alignment
    static constexpr int kSmemBytes = kStages * kStageBytes + kEpiSmem + 256 + 1024;
    static_assert(8 * (3 * kStages + 2 * kAccStages + 1) <= 256, "barrier area");
};

// plane pairs, least significant products first
__device__ __forceinline__ void pair_of(int P, int i, int &pa, int &pb) {
    if (P == 3) {
        const int A[6] = {2, 0, 1, 1, 0, 0}, B[6] = {0, 2, 1, 0, 1, 0};
        pa = A[i]; pb = B[i];
    } else if (P == 2) {
        const int A[3] = {1, 0, 0}, B[3] = {0, 1, 0};
        pa = A[i]; pb = B[i];
    } else { pa = 0; pb = 0; }
}

// ---- PTX wrappers ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra WAIT_DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "WAIT_DONE:\n\t"
        "}" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap *map, uint32_t bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void prefetch_tensormap(const CUtensorMap *map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_mma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// 8-bit operands (kind::f8f6f4, here E4M3 x E4M3 -> fp32): K = 32 per instruction, i.e. the same 32 bytes per row and
// instruction as a 16-element bf16 / fp16 step, at twice the multiply rate.  The instruction descriptor is the one of an
// fp16 MMA (format code 0 = F16 for kind::f16, = E4M3 for kind::f8f6f4).
__device__ __forceinline__ void tc_mma_e4m3(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// ---- CTA-pair (cta_group::2) flavours: one 256 x BN tile per pair of SMs, each CTA loads its 128 rows of A and HALF of B ----
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ uint32_t mapa_shared(uint32_t addr, uint32_t rank) {      // same offset in CTA `rank`
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// TMA load whose completion is signalled on a barrier of the pair's leader CTA
__device__ __forceinline__ void tma_load_3d_pair(uint32_t dst, const CUtensorMap *map, uint32_t leader_bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(leader_bar), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish_pair() {
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// commit: arrive on the barrier at this offset in BOTH CTAs of the pair when the MMAs issued so far retire
__device__ __forceinline__ void tc_commit_pair(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(bar), "h"(static_cast<uint16_t>(3)) : "memory");
}
__device__ __forceinline__ void tc_mma_bf16_pair(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tc_mma_e4m3_pair(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// shared-memory matrix descriptor: K-major, 128-byte swizzle, 8-row groups 1024 B apart
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);      // start address, 16-byte units
    d |= static_cast<uint64_t>(1) << 16;                          // leading byte offset (unused when swizzled)
    d |= static_cast<uint64_t>(1024 >> 4) << 32;                  // stride byte offset
    d |= static_cast<uint64_t>(1) << 46;                          // descriptor version (Blackwell)
    d |= static_cast<uint64_t>(2) << 61;                          // SWIZZLE_128B
    return d;
}
// instruction descriptor: D fp32, A/B bf16 (format 1) or fp16 (format 0), both K-major, dense
constexpr uint32_t make_idesc(int m, int n, bool f16 = false) {
    return (1u << 4) | (f16 ? 0u : ((1u << 7) | (1u << 10))) | (static_cast<uint32_t>(n >> 3) << 17) |
           (static_cast<uint32_t>(m >> 4) << 24);
}

// ---- epilogue functors: value for output element (row, col) given the accumulator -------------
// kF16x2: AGRL_SPLIT_FP16X2 operands -- fp16 planes h = fp16(x s), l = fp16((x s - h) 2^11) with a power-of-two scale s
// per row: the correction accumulator (h.l + l.h) enters with 2^-11, the result is un-scaled by 2^-kq 2^-kg (exact).
template <bool kF16x2>
struct EpiDistanceT {           // distance.py:59-73 / :76-89
    static constexpr const char *kName = "gemm_distance";
    static constexpr bool kF16 = kF16x2;
    static constexpr float kCorrScale = kF16x2 ? 0.00048828125f : 1.0f;
    static constexpr bool kDirect = false;      // rows of arbitrary alignment: coalesce through smem
    static constexpr int kChunkKb = 4;          // drain the accumulator every 256 k (fp32-accurate sums).  Measured at 1980 x 9330 x 4096,
                                                // fp16 x 2: 4 -> 0.383 ms, 1.5e-6 on clustered data; 16 -> 0.347 ms, 6.0e-6; never -> 0.345 ms, 2.5e-5
    static constexpr bool kRowwise = false;
    static constexpr bool kFp8 = false;
    const float *qn, *gn;       // squared norms (euclidean); unused for cosine
    float *out;
    int64_t ld;
    int metric;
    const float *qu, *gu;       // kF16x2: 1 / s per row of either operand
    struct Col { float gn, gu; };
    __device__ __forceinline__ Col col_state(int col) const {
        Col c; c.gn = (metric == AGRL_METRIC_EUCLIDEAN) ? __ldg(gn + col) : 0.f;
        c.gu = kF16x2 ? __ldg(gu + col) : 1.0f; return c;
    }
    __device__ __forceinline__ void store(int row, int col, float acc, const Col &c) const {
        float v;
        if (kF16x2) acc = acc * __ldg(qu + row) * c.gu;
        if (metric == AGRL_METRIC_EUCLIDEAN) v = fmaf(-2.0f, acc, __fadd_rn(__ldg(qn + row), c.gn));
        else v = 1.0f - acc;
        out[static_cast<size_t>(row) * ld + col] = v;
    }
};

// Distance -> per-query top-k candidates, fused (SURVEY 7 step 6: the num_q x num_g matrix is never written).  Same
// accumulation and the same final expression as EpiDistanceT, so every distance has the bits the matrix would hold; the
// thread that owns (row, 64 columns) turns them into ranking keys (order-preserving distance bits << 32 | GLOBAL gallery
// index) and appends the ones below the row's threshold -- the K-th smallest key of the columns seen by earlier
// launches -- to the row's candidate list.  Launches cover growing column ranges; topk_compact_kernel (distance.cu) cuts
// each list back to its K smallest keys and tightens the threshold in between, so after the first few thousand columns
// only ~K ln(growth) candidates per row and launch pass the filter.
template <bool kF16x2>
struct EpiTopKT {
    static constexpr const char *kName = "gemm_distance_topk";
    static constexpr bool kF16 = kF16x2;
    static constexpr float kCorrScale = kF16x2 ? 0.00048828125f : 1.0f;
    static constexpr bool kDirect = false;
    static constexpr int kChunkKb = 4;
    static constexpr bool kRowwise = true;
    static constexpr bool kFp8 = false;
    const float *qn, *gn;               // squared norms (euclidean), gn already offset to this launch's first column
    int metric;
    const unsigned long long *tau;      // [M] threshold key per row (all-ones: accept everything)
    unsigned int *cnt;                  // [M] candidates appended so far (may run past `cap`: overflow, detected later)
    unsigned long long *cand;           // [M][cap]
    int cap;
    uint32_t idx_base;                  // global gallery index of this launch's column 0
    const float *qu, *gu;               // kF16x2: 1 / s per row of either operand (gu offset like gn)
    __device__ __forceinline__ void consume(int row, int col0, int n_cols, const float (&sum)[64]) const {
        const unsigned long long t = tau[row];
        const float q = (metric == AGRL_METRIC_EUCLIDEAN) ? __ldg(qn + row) : 0.f;
        const float uq = kF16x2 ? __ldg(qu + row) : 1.0f;
        unsigned long long *list = cand + static_cast<size_t>(row) * cap;
#pragma unroll
        for (int j = 0; j < 64; ++j) {
            const int col = col0 + j;
            if (col < n_cols) {
                float v;
                const float acc = kF16x2 ? sum[j] * uq * __ldg(gu + col) : sum[j];      // the expression EpiDistanceT::store uses
                if (metric == AGRL_METRIC_EUCLIDEAN) v = fmaf(-2.0f, acc, __fadd_rn(q, __ldg(gn + col)));
                else v = 1.0f - acc;
                const unsigned long long key = rank_key(v, idx_base + static_cast<uint32_t>(col));
                if (key < t) {
                    const unsigned int slot = atomicAdd(cnt + row, 1u);
                    if (slot < static_cast<unsigned int>(cap)) list[slot] = key;
                }
            }
        }
    }
};

// kScaled: single-plane fp16 operands (AGRL_SPLIT_FP16X1).  Both operands were multiplied by powers of two to sit
// in the middle of the fp16 range (per tracklet for Y, per layer for W); the epilogue undoes that exactly.
// kFp8 (with kScaled): AGRL_SPLIT_FP16_E4M3 -- plane 0 is the scaled fp16 operand, plane 1 holds, per 64-element k-block,
// 64 E4M3 residuals and 64 E4M3 copies of the values (planes.cuh): one fp16 product + one K-concatenated 8-bit product.
template <bool kScaled, bool kFp8_ = false>
struct EpiGraphLayerT {         // vmgn.py:169-172: gamma * LeakyReLU(BN(acc)) + (1-gamma) * x
    static constexpr const char *kName = "gemm_graph_layer";
    static constexpr bool kF16 = kScaled;
    static constexpr float kCorrScale = 1.0f;
    static constexpr bool kFp8 = kFp8_;
    static constexpr bool kDirect = true;       // C % 4 == 0 and 16-byte aligned rows: vector accesses
    static constexpr int kChunkKb = 0;          // one accumulation over all of K
    static constexpr bool kRowwise = false;
    // pull this thread's slice of the residual row into L2 before the accumulator is ready
    __device__ __forceinline__ void prefetch(int row, int col0, int ncols, bool valid) const {
        if (!valid) return;
        const float *p = x + static_cast<size_t>(row) * ldx + col0;
        for (int c = 0; c < ncols; c += 32) asm volatile("prefetch.global.L2 [%0];" ::"l"(p + c));
    }
    // residual of 32 consecutive columns of one row (independent of the accumulator: issued a round ahead)
    __device__ __forceinline__ void load_row32(int row, int col0, float4 (&xin)[8]) const {
        const float4 *xr = reinterpret_cast<const float4 *>(x + static_cast<size_t>(row) * ldx + col0);
#pragma unroll
        for (int q = 0; q < 8; ++q) xin[q] = __ldg(xr + q);
    }
    // 32 consecutive columns of one row: the math, then the stores
    __device__ __forceinline__ void store_row32(int row, int col0, int n_cols, const uint32_t (&acc)[32], const float4 (&xin)[8],
                                                float &sumsq) const {
        float4 *orow = reinterpret_cast<float4 *>(out + static_cast<size_t>(row) * ldo + col0);
        const float4 *sc = reinterpret_cast<const float4 *>(scale + col0);
        const float4 *sh = reinterpret_cast<const float4 *>(shift + col0);
        if (col0 + 32 > n_cols) return;                       // N is a multiple of 32 for this epilogue
        const float unscale = kScaled ? __ldg(row_unscale + row / nodes) * __ldg(w_unscale) : 1.0f;
        const float keep = 1.0f - gamma;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const float4 s4 = __ldg(sc + q), t4 = __ldg(sh + q);
            float4 o;
            float h;
            h = fmaf(kScaled ? __uint_as_float(acc[4 * q + 0]) * unscale : __uint_as_float(acc[4 * q + 0]), s4.x, t4.x); h = h >= 0.f ? h : h * slope; o.x = fmaf(gamma, h, keep * xin[q].x);
            h = fmaf(kScaled ? __uint_as_float(acc[4 * q + 1]) * unscale : __uint_as_float(acc[4 * q + 1]), s4.y, t4.y); h = h >= 0.f ? h : h * slope; o.y = fmaf(gamma, h, keep * xin[q].y);
            h = fmaf(kScaled ? __uint_as_float(acc[4 * q + 2]) * unscale : __uint_as_float(acc[4 * q + 2]), s4.z, t4.z); h = h >= 0.f ? h : h * slope; o.z = fmaf(gamma, h, keep * xin[q].z);
            h = fmaf(kScaled ? __uint_as_float(acc[4 * q + 3]) * unscale : __uint_as_float(acc[4 * q + 3]), s4.w, t4.w); h = h >= 0.f ? h : h * slope; o.w = fmaf(gamma, h, keep * xin[q].w);
            orow[q] = o;
            sumsq = fmaf(o.x, o.x, sumsq); sumsq = fmaf(o.y, o.y, sumsq); sumsq = fmaf(o.z, o.z, sumsq); sumsq = fmaf(o.w, o.w, sumsq);
        }
    }
    const float *x;             // layer input (M, ldx)
    const float *scale, *shift; // folded eval-mode BatchNorm1d per output channel
    float *out;
    int64_t ldx, ldo;
    float gamma, slope;
    const float *row_unscale;   // kScaled: 2^-k of each tracklet's Y rows (one float per tracklet)
    const float *w_unscale;     // kScaled: 2^-k of this layer's W (one float)
    int nodes;                  // rows per tracklet
    // optional (last layer): per row and per (column tile, half) the sum of squares of the stored outputs, so that the
    // attention kernel gets its row norms (vmgn.py:276) without a pass of its own: (M, sumsq_slots) floats
    float *row_sumsq = nullptr;
    int sumsq_slots = 0;
    __device__ __forceinline__ void store_sumsq(int row, int slot, float v) const {
        if (row_sumsq) row_sumsq[static_cast<size_t>(row) * sumsq_slots + slot] = v;
    }
    struct Col { float scale, shift; };
    __device__ __forceinline__ Col col_state(int col) const {
        Col c; c.scale = __ldg(scale + col); c.shift = __ldg(shift + col); return c;
    }
    __device__ __forceinline__ void store(int row, int col, float acc, const Col &c) const {
        if (kScaled) acc *= __ldg(row_unscale + row / nodes) * __ldg(w_unscale);
        float h = fmaf(acc, c.scale, c.shift);
        h = h >= 0.f ? h : h * slope;
        const float xin = __ldg(x + static_cast<size_t>(row) * ldx + col);
        out[static_cast<size_t>(row) * ldo + col] = fmaf(gamma, h, (1.0f - gamma) * xin);
    }
};
// Plain store of the accumulator as fp32 (first graph layer on the quarter-strip rows: Z = Q.W^T, the layer's element-wise
// part follows in graph_mix_kernel).  Same direct-epilogue interface as EpiGraphLayerT; nothing to prefetch or reload.
template <bool kScaled, bool kFp8_ = false>
struct EpiPlainT {
    static constexpr const char *kName = "gemm_graph_layer";
    static constexpr bool kF16 = kScaled;
    static constexpr float kCorrScale = 1.0f;
    static constexpr bool kFp8 = kFp8_;
    static constexpr bool kDirect = true;
    static constexpr int kChunkKb = 0;
    static constexpr bool kRowwise = false;
    float *out; int64_t ldo;
    const float *row_unscale;   // kScaled: 2^-k per tracklet
    const float *w_unscale;     // kScaled: 2^-k of the layer's W
    int rows_per_unit;          // GEMM rows per tracklet
    __device__ __forceinline__ void prefetch(int, int, int, bool) const {}
    __device__ __forceinline__ void load_row32(int, int, float4 (&)[8]) const {}
    __device__ __forceinline__ void store_row32(int row, int col0, int n_cols, const uint32_t (&acc)[32], const float4 (&)[8],
                                                float &) const {
        if (col0 + 32 > n_cols) return;
        const float unscale = kScaled ? __ldg(row_unscale + row / rows_per_unit) * __ldg(w_unscale) : 1.0f;
        float4 *orow = reinterpret_cast<float4 *>(out + static_cast<size_t>(row) * ldo + col0);
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            float4 o;
            o.x = __uint_as_float(acc[4 * q + 0]); o.y = __uint_as_float(acc[4 * q + 1]);
            o.z = __uint_as_float(acc[4 * q + 2]); o.w = __uint_as_float(acc[4 * q + 3]);
            if (kScaled) { o.x *= unscale; o.y *= unscale; o.z *= unscale; o.w *= unscale; }
            orow[q] = o;
        }
    }
    __device__ __forceinline__ void store_sumsq(int, int, float) const {}
};

// ---- the kernel --------------------------------------------------------------------------------
// kPair: the CTA pair (cluster of 2, tcgen05 cta_group::2) owns a 256 x BN tile.  Every CTA loads its own 128 rows of A
// and its half of the B tile; both CTAs' loads complete on the LEADER's full barrier (which expects the bytes of both
// stages), the leader issues the MMAs for the pair, its commits arrive on the empty / accumulator-full barriers of both
// CTAs, and both CTAs' epilogue warps release the accumulator on the leader's barrier.
template <int P, int BN, bool kSplit, class Epi, bool kPair = false>
__device__ __forceinline__ void split_gemm_body(const CUtensorMap &map_a, const CUtensorMap &map_b,
                                                int M, int N, int k_pad, const Epi &epi) {
    using Cfg = Config<P, BN, kSplit, Epi::kDirect, Epi::kChunkKb, kPair>;
    constexpr int kAccCols = Cfg::kAccCols;
    // kWideB (two planes, two accumulators, one CTA per tile): the B tile's planes lie back to back in the stage, so ONE
    // 128 x 256 MMA per k-step multiplies a0 with [b0 ; b1] into [main | corr] and a second, 128-wide one adds a1.b0 to corr:
    // 20 instead of 24 KiB of operand reads per k-step on the shared-memory port that paces these GEMMs
    constexpr bool kWideB = kSplit && P == 2 && !kPair && BN == 128;
    constexpr bool kCorrPersist = kSplit && Cfg::kChunk > 0 && !kWideB;
    extern __shared__ unsigned char smem_dyn[];
    // 128B-swizzled tiles need 1024-byte alignment
    unsigned char *smem = reinterpret_cast<unsigned char *>(
        (reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~static_cast<uintptr_t>(1023));
    float *epi_buf = reinterpret_cast<float *>(smem + Cfg::kStages * Cfg::kStageBytes);
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + Cfg::kStages * Cfg::kStageBytes + Cfg::kEpiSmem);
    // bars: full[kStages], empty[kStages], tmem_full[2], tmem_empty[2], then the TMEM base address
    const uint32_t bar_full = smem_u32(bars);
    const uint32_t bar_empty = bar_full + 8 * Cfg::kStages;
    const uint32_t bar_tfull = bar_empty + 8 * Cfg::kStages;
    const uint32_t bar_tempty = bar_tfull + 8 * kAccStages;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2 * Cfg::kStages + 2 * kAccStages);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = kPair ? cluster_ctarank() : 0u;             // 0 = the pair's leader (issues the MMAs)
    const int tile0 = kPair ? static_cast<int>(blockIdx.x >> 1) : static_cast<int>(blockIdx.x);
    const int tile_step = kPair ? static_cast<int>(gridDim.x >> 1) : static_cast<int>(gridDim.x);
    const int tiles_m = (M + Cfg::kTileM - 1) / Cfg::kTileM, tiles_n = (N + BN - 1) / BN;
    const int num_tiles = tiles_m * tiles_n;
    const int num_kb = k_pad / BK;
    const int chunk_kb = Cfg::kChunk > 0 ? Cfg::kChunk : num_kb;       // k-blocks per accumulator drain
    // Raster: the operand with FEWER tiles varies fastest, so the CTAs running at any moment share it
    // (L2-resident) while the larger operand streams through exactly once.  When even the smaller operand is too big
    // to stay in L2 (10 000 queries x 2048 x 3 planes = 123 MB), its tiles are taken in groups of kGroupM row tiles
    // (25 MB at K = 2048): the other operand streams once per group.
    constexpr int kGroupM = 16;
    const bool m_fast = tiles_m <= tiles_n;
    const int grp_m = tiles_m < kGroupM ? tiles_m : kGroupM;
    const int full_tiles = (tiles_m / grp_m) * grp_m * tiles_n;      // tiles in complete groups
    auto tile_origin = [&](int tile, int &m0, int &n0) {
        if (m_fast) {
            int base_m, gm, r;
            if (tile < full_tiles) { const int per = grp_m * tiles_n; const int g = tile / per; base_m = g * grp_m; gm = grp_m; r = tile - g * per; }
            else { base_m = (tiles_m / grp_m) * grp_m; gm = tiles_m - base_m; r = tile - full_tiles; }
            m0 = (base_m + r % gm) * Cfg::kTileM; n0 = (r / gm) * BN;
        } else { n0 = (tile % tiles_n) * BN; m0 = (tile / tiles_n) * Cfg::kTileM; }
        m0 += static_cast<int>(rank) * BM;                            // this CTA's 128 rows of the tile
    };

    if (warp == 0 && lane == 0) {
        prefetch_tensormap(&map_a);
        prefetch_tensormap(&map_b);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < Cfg::kStages; ++s) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); }
        for (int s = 0; s < kAccStages; ++s) { mbar_init(bar_tfull + 8 * s, 1); mbar_init(bar_tempty + 8 * s, Cfg::kEpiWarps * (kPair ? 2 : 1)); }
        fence_barrier_init();
    }
    if (warp == 2) {
        if (kPair) { tmem_alloc_pair(smem_u32(tmem_slot), kTmemCols); tmem_relinquish_pair(); }
        else { tmem_alloc(smem_u32(tmem_slot), kTmemCols); tmem_relinquish(); }
    }
    tc_fence_before();
    if (kPair) cluster_sync_all(); else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ================= TMA producer =================
        int stage = 0; uint32_t phase = 0;
        for (int tile = tile0; tile < num_tiles; tile += tile_step) {
            int m0, n0;
            tile_origin(tile, m0, n0);
            for (int kb = 0; kb < num_kb; ++kb) {
                mbar_wait(bar_empty + 8 * stage, phase ^ 1);
                if (lane == 0) {
                    const uint32_t sa = smem_u32(smem + stage * Cfg::kStageBytes);
                    const uint32_t sb = sa + P * kTileBytesA;
                    const uint32_t full = bar_full + 8 * stage;
                    if (kPair && rank != 0) {
                        // (the peer's bytes may land before the leader's expect_tx of the phase: the transaction count goes
                        // negative until then, the phase cannot complete before the leader's arrive)
                        const uint32_t lfull = mapa_shared(full, 0);
                        const int nb = n0 + Cfg::kLoadN;
#pragma unroll
                        for (int p = 0; p < P; ++p) tma_load_3d_pair(sa + p * kTileBytesA, &map_a, lfull, kb * BK, m0, p);
#pragma unroll
                        for (int p = 0; p < P; ++p) tma_load_3d_pair(sb + p * Cfg::kTileBytesB, &map_b, lfull, kb * BK, nb, p);
                    } else {
                        mbar_arrive_expect_tx(full, (kPair ? 2 : 1) * Cfg::kStageBytes);
#pragma unroll
                        for (int p = 0; p < P; ++p) tma_load_3d(sa + p * kTileBytesA, &map_a, full, kb * BK, m0, p);
#pragma unroll
                        for (int p = 0; p < P; ++p) tma_load_3d(sb + p * Cfg::kTileBytesB, &map_b, full, kb * BK, n0, p);
                    }
                }
                __syncwarp();
                if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1 && rank == 0) {
        // ================= MMA issuer (the pair's leader only) =================
        constexpr uint32_t idesc = make_idesc(Cfg::kTileM, BN, Epi::kF16);
        int stage = 0; uint32_t phase = 0;
        int cit = 0;                                               // accumulator-drain counter (chunks)
        int tcount = 0;                                            // tiles of this CTA so far
        for (int tile = tile0; tile < num_tiles; tile += tile_step, ++tcount) {
            for (int kb0 = 0; kb0 < num_kb; kb0 += chunk_kb, ++cit) {
                const int acc = cit & 1;
                const uint32_t acc_phase = (cit >> 1) & 1;
                const int kb_end = (kb0 + chunk_kb < num_kb) ? kb0 + chunk_kb : num_kb;
                mbar_wait(bar_tempty + 8 * acc, acc_phase ^ 1);    // epilogue has drained this accumulator
                tc_fence_after();
                // Two accumulators per stage when kSplit.  The tensor core truncates (round-toward-zero)
                // on every accumulate, at the ulp of the running sum; keeping the small correction
                // products out of the big a0.b0 sum spares it 5/6 (P=3) of those truncations, and the
                // correction sum itself is ~2^-8 smaller, so its own truncation is negligible.
                // Chunked + split (kCorrPersist): the two MAIN accumulators alternate per chunk in columns [0, 2 BN); the
                // correction sum -- 2^-8 (bf16) / 2^-11 (fp16 x 2) of the main one, its own truncation negligible -- stays
                // in TMEM for the whole tile, columns [2 BN, 4 BN) alternating per TILE, and is drained once: half the
                // TMEM reads of draining both every chunk (same kernel time: the 128-wide MMAs, not the drains, pace
                // this GEMM -- tensor pipe 62 % under ncu; a 256 x 256 pair tile with ONE accumulator and no chunked
                // drain ran 0.31 instead of 0.39 ms at MARS size but lost a digit and a half to accumulate truncation;
                // issuing the products as corr, main, corr per k-step -- consecutive MMAs on different accumulators --
                // changed nothing either).
                const uint32_t d_main = kCorrPersist ? tmem_base + acc * BN : tmem_base + acc * kAccCols;
                const uint32_t d_corr = kCorrPersist ? tmem_base + 2 * BN + (tcount & 1) * BN : (kSplit ? d_main + BN : d_main);
                for (int kb = kb0; kb < kb_end; ++kb) {
                    mbar_wait(bar_full + 8 * stage, phase);        // TMA bytes have landed
                    tc_fence_after();
                    if (lane == 0) {
                        const uint32_t sa = smem_u32(smem + stage * Cfg::kStageBytes);
                        const uint32_t sb = sa + P * kTileBytesA;
                        const int first = kb - kb0;                // 0 on the chunk's first k-block
                        if constexpr (Epi::kFp8) {
                            // fp16 product of the value planes, then ONE 8-bit product over the k-block's 128 bytes:
                            // [r_a | a8] . [b8 | r_b] = r_a.b8 + a8.r_b, the two first-order corrections of a.b
                            static_assert(P == 2 && !kSplit, "fp16 + e4m3 mode: two byte-identical planes, one accumulator");
                            if constexpr (kPair) {
                                const uint64_t pa0 = make_smem_desc(sa), pb0 = make_smem_desc(sb);
                                const uint64_t pa1 = make_smem_desc(sa + kTileBytesA), pb1 = make_smem_desc(sb + Cfg::kTileBytesB);
                                const uint32_t pd = tmem_base + acc * kAccCols;
#pragma unroll
                                for (int k = 0; k < BK / UMMA_K; ++k) tc_mma_bf16_pair(pd, pa0 + 2 * k, pb0 + 2 * k, idesc, (first | k) != 0 ? 1u : 0u);
#pragma unroll
                                for (int k = 0; k < BK / UMMA_K; ++k) tc_mma_e4m3_pair(pd, pa1 + 2 * k, pb1 + 2 * k, idesc, 1u);
                            } else {
                            const uint64_t da0 = make_smem_desc(sa), db0 = make_smem_desc(sb);
                            const uint64_t da1 = make_smem_desc(sa + kTileBytesA), db1 = make_smem_desc(sb + Cfg::kTileBytesB);
                            const uint32_t d = tmem_base + acc * kAccCols;
#pragma unroll
                            for (int k = 0; k < BK / UMMA_K; ++k) tc_mma_bf16(d, da0 + 2 * k, db0 + 2 * k, idesc, (first | k) != 0 ? 1u : 0u);
#pragma unroll
                            for (int k = 0; k < BK / UMMA_K; ++k) tc_mma_e4m3(d, da1 + 2 * k, db1 + 2 * k, idesc, 1u);
                            }
                        } else if constexpr (kWideB) {
                            constexpr uint32_t idesc_wide = make_idesc(BM, 2 * BN, Epi::kF16);
                            const uint64_t a0 = make_smem_desc(sa), a1 = make_smem_desc(sa + kTileBytesA), b0 = make_smem_desc(sb);
#pragma unroll
                            for (int k = 0; k < BK / UMMA_K; ++k) {
                                tc_mma_bf16(d_main, a0 + 2 * k, b0 + 2 * k, idesc_wide, (first | k) != 0 ? 1u : 0u);   // a0.[b0 ; b1]
                                tc_mma_bf16(d_corr, a1 + 2 * k, b0 + 2 * k, idesc, 1u);                                // + a1.b0
                            }
                        } else
#pragma unroll
                        for (int i = 0; i < Cfg::kNumPairs; ++i) {
                            int pa, pb;
                            pair_of(P, i, pa, pb);
                            const uint64_t da = make_smem_desc(sa + pa * kTileBytesA);
                            const uint64_t db = make_smem_desc(sb + pb * Cfg::kTileBytesB);
#pragma unroll
                            for (int k = 0; k < BK / UMMA_K; ++k) {
                                // advance 32 bytes (16 bf16) along K inside the 128-byte swizzle row
                                const bool main_acc = kSplit && i == Cfg::kNumPairs - 1;
                                const uint32_t d = main_acc ? d_main : d_corr;
                                const uint32_t accum = main_acc ? ((first | k) != 0 ? 1u : 0u)
                                                                : (((kCorrPersist ? kb : first) | i | k) != 0 ? 1u : 0u);
                                if (kPair) tc_mma_bf16_pair(d, da + 2 * k, db + 2 * k, idesc, accum);
                                else tc_mma_bf16(d, da + 2 * k, db + 2 * k, idesc, accum);
                            }
                        }
                        // frees the smem stage when the MMAs retire; publishes the accumulator (chunk) when complete
                        if (kPair) {
                            tc_commit_pair(bar_empty + 8 * stage);
                            if (kb == kb_end - 1) tc_commit_pair(bar_tfull + 8 * acc);
                        } else {
                            tc_commit(bar_empty + 8 * stage);
                            if (kb == kb_end - 1) tc_commit(bar_tfull + 8 * acc);
                        }
                    }
                    __syncwarp();
                    if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp >= kCtrlWarps) {
        // ================= epilogue =================
        const int ew = warp - kCtrlWarps;
        const int quarter = ew & 3;                                // == warp % 4: the TMEM lane quarter
        // "accumulator drained" goes to the barrier the MMA issuer waits on: the leader's
        auto release_acc = [&](int acc) {
            if (kPair) mbar_arrive_cluster(mapa_shared(bar_tempty + 8 * acc, 0));
            else mbar_arrive(bar_tempty + 8 * acc);
        };
        int cit = 0, tcount = 0;
        for (int tile = tile0; tile < num_tiles; tile += tile_step, ++tcount) {
            int m0, n0;
            tile_origin(tile, m0, n0);
            const int row_base = m0 + quarter * 32;
            const uint32_t tlane = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16);
            if constexpr (Epi::kDirect) {
                // thread = one output row, 16-byte accesses straight from registers; warps 4-7 of the
                // group take the upper half of the tile's columns
                const int acc = cit & 1;
                const uint32_t acc_phase = (cit >> 1) & 1;
                const uint32_t tq = tlane + acc * kAccCols;
                const int col_half = (ew >> 2) * (BN / 2);
                const int row = row_base + lane;
                const bool live = row < M && n0 + col_half + BN / 2 <= N;
                epi.prefetch(row, n0 + col_half, BN / 2, live);        // residual tile -> L2 while the MMAs run
                // the residual of round c + 1 is in flight while round c is computed and stored; round 0's loads
                // are issued before the wait for the accumulator
                float4 xa[8], xb[8];
                float sumsq = 0.f;
                if (live) epi.load_row32(row, n0 + col_half, xa);
                mbar_wait(bar_tfull + 8 * acc, acc_phase);
                tc_fence_after();
#pragma unroll
                for (int c = 0; c < BN / 2; c += 64) {
                    uint32_t r[32];
                    tmem_ld_32x32(tq + col_half + c, r);
                    if (live && c + 32 < BN / 2) epi.load_row32(row, n0 + col_half + c + 32, xb);
                    tmem_ld_wait();
                    if (live) epi.store_row32(row, n0 + col_half + c, N, r, xa, sumsq);
                    if (c + 32 < BN / 2) {
                        tmem_ld_32x32(tq + col_half + c + 32, r);
                        if (live && c + 64 < BN / 2) epi.load_row32(row, n0 + col_half + c + 64, xa);
                        tmem_ld_wait();
                        if (live) epi.store_row32(row, n0 + col_half + c + 32, N, r, xb, sumsq);
                    }
                }
                if (live) epi.store_sumsq(row, (n0 / BN) * 2 + (ew >> 2), sumsq);
                tc_fence_before();
                if (lane == 0) release_acc(acc);
                ++cit;
            } else if constexpr (Cfg::kChunk > 0) {
                // chunked accumulation: this warp owns 32 rows x 64 columns; every chunk's partial
                // (main + correction) is added into registers with round-to-nearest
                const int col_half = (ew >> 2) * (BN / 2);
                float sum[BN / 2];
#pragma unroll
                for (int j = 0; j < BN / 2; ++j) sum[j] = 0.f;
                for (int kb0 = 0; kb0 < num_kb; kb0 += chunk_kb, ++cit) {
                    const int acc = cit & 1;
                    const uint32_t acc_phase = (cit >> 1) & 1;
                    const uint32_t tq = tlane + (kCorrPersist ? acc * BN : acc * kAccCols) + col_half;
                    const bool last_chunk = kb0 + chunk_kb >= num_kb;
                    mbar_wait(bar_tfull + 8 * acc, acc_phase);
                    tc_fence_after();
#pragma unroll
                    for (int c = 0; c < BN / 2; c += 32) {
                        uint32_t r[32];
                        tmem_ld_32x32(tq + c, r);
                        if constexpr (kSplit && !kCorrPersist) {       // this chunk's correction sum sits next to the main one
                            uint32_t rc[32];
                            tmem_ld_32x32(tq + BN + c, rc);
                            tmem_ld_wait();
#pragma unroll
                            for (int j = 0; j < 32; ++j) {
                                const float part = Epi::kCorrScale == 1.0f ? __fadd_rn(__uint_as_float(r[j]), __uint_as_float(rc[j]))
                                                                           : fmaf(__uint_as_float(rc[j]), Epi::kCorrScale, __uint_as_float(r[j]));
                                sum[c + j] = __fadd_rn(sum[c + j], part);
                            }
                            continue;
                        }
                        tmem_ld_wait();
#pragma unroll
                        for (int j = 0; j < 32; ++j) sum[c + j] = __fadd_rn(sum[c + j], __uint_as_float(r[j]));
                        if (kCorrPersist && last_chunk) {              // the tile's correction sum, once
                            tmem_ld_32x32(tlane + 2 * BN + (tcount & 1) * BN + col_half + c, r);
                            tmem_ld_wait();
#pragma unroll
                            for (int j = 0; j < 32; ++j)
                                sum[c + j] = Epi::kCorrScale == 1.0f ? __fadd_rn(sum[c + j], __uint_as_float(r[j]))
                                                                     : fmaf(__uint_as_float(r[j]), Epi::kCorrScale, sum[c + j]);
                        }
                    }
                    tc_fence_before();
                    if (lane == 0) release_acc(acc);
                }
                if constexpr (Epi::kRowwise) {
                    static_assert(BN == 128, "row-wise consumers take 64 columns per thread");
                    if (row_base + lane < M) epi.consume(row_base + lane, n0 + col_half, N, sum);
                } else {
                    float *buf = epi_buf + ew * 32 * kEpiPad;
#pragma unroll
                    for (int c = 0; c < BN / 2; c += 32) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) buf[lane * kEpiPad + j] = sum[c + j];
                        __syncwarp();
                        const int col = n0 + col_half + c + lane;
                        if (col < N) {
                            const typename Epi::Col cs = epi.col_state(col);
#pragma unroll 8
                            for (int rr = 0; rr < 32; ++rr) {
                                const int row = row_base + rr;
                                if (row < M) epi.store(row, col, buf[rr * kEpiPad + lane], cs);
                            }
                        }
                        __syncwarp();
                    }
                }
            } else {
                const int acc = cit & 1;
                const uint32_t acc_phase = (cit >> 1) & 1;
                const uint32_t tq = tlane + acc * kAccCols;
                float *buf = epi_buf + quarter * 32 * kEpiPad;
                mbar_wait(bar_tfull + 8 * acc, acc_phase);
                tc_fence_after();
#pragma unroll 1
                for (int c = 0; c < BN / 32; ++c) {
                    uint32_t r[32];
                    tmem_ld_32x32(tq + c * 32, r);
                    if (kSplit) {
                        uint32_t rc[32];
                        tmem_ld_32x32(tq + BN + c * 32, rc);
                        tmem_ld_wait();
#pragma unroll
                        for (int j = 0; j < 32; ++j)
                            buf[lane * kEpiPad + j] = Epi::kCorrScale == 1.0f ? __fadd_rn(__uint_as_float(r[j]), __uint_as_float(rc[j]))
                                                                              : fmaf(__uint_as_float(rc[j]), Epi::kCorrScale, __uint_as_float(r[j]));
                    } else {
                        tmem_ld_wait();
#pragma unroll
                        for (int j = 0; j < 32; ++j) buf[lane * kEpiPad + j] = __uint_as_float(r[j]);
                    }
                    __syncwarp();
                    const int col = n0 + c * 32 + lane;
                    if (col < N) {
                        const typename Epi::Col cs = epi.col_state(col);
#pragma unroll 8
                        for (int rr = 0; rr < 32; ++rr) {
                            const int row = row_base + rr;
                            if (row < M) epi.store(row, col, buf[rr * kEpiPad + lane], cs);
                        }
                    }
                    __syncwarp();
                }
                tc_fence_before();
                if (lane == 0) release_acc(acc);
                ++cit;
            }
        }
    }

    tc_fence_before();
    if (kPair) cluster_sync_all(); else __syncthreads();
    if (warp == 2) {
        if (kPair) tmem_dealloc_pair(tmem_base, kTmemCols);
        else tmem_dealloc(tmem_base, kTmemCols);
    }
}

template <int P, int BN, bool kSplit, class Epi>
__global__ void __maxnreg__((Config<P, BN, kSplit, Epi::kDirect, Epi::kChunkKb>::kMaxRegs))
split_gemm_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                  int M, int N, int k_pad, Epi epi) {
    split_gemm_body<P, BN, kSplit, Epi>(map_a, map_b, M, N, k_pad, epi);
}

template <int P, int BN, bool kSplit, class Epi>
__global__ void __cluster_dims__(2, 1, 1) __maxnreg__((Config<P, BN, kSplit, Epi::kDirect, Epi::kChunkKb>::kMaxRegs))
pair_gemm_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                 int M, int N, int k_pad, Epi epi) {
    split_gemm_body<P, BN, kSplit, Epi, true>(map_a, map_b, M, N, k_pad, epi);
}

// ---- host side -----------------------------------------------------------------------------------
// 3-D tensor map over planes [P][rows][k_pad] of bf16: box = (BK, box_rows, 1), 128-byte swizzle.
// box_rows = BM for the A operand, the kernel's BN for the B operand.
// plane_rows = rows between consecutive planes (>= rows when the map covers a row slice of the planes).
int make_plane_tensor_map(CUtensorMap *map, const void *planes, int64_t rows, int64_t k_pad, int P, int box_rows,
                          int64_t plane_rows);

int make_rows_tensor_map_f32(CUtensorMap *map, const float *x, int64_t batch, int V, int C, int box_channels);       // split.cu

// CTA-pair flavour; map_b must have been built with box_rows = BN / 2.
template <int P, int BN, bool kSplit, class Epi>
int launch_pair_gemm(const CUtensorMap &map_a, const CUtensorMap &map_b, int M, int N, int k_pad, const Epi &epi, cudaStream_t st) {
    using Cfg = Config<P, BN, kSplit, Epi::kDirect, Epi::kChunkKb, true>;
    static_assert(!Epi::kDirect || !kSplit, "the direct epilogue reads a single accumulator");
    auto kern = pair_gemm_kernel<P, BN, kSplit, Epi>;
    AGRL_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
    // persistent grid = the number of CTA pairs that can be resident at once (a GPC with an odd SM left over hosts no
    // pair there), asked once per kernel
    static const int max_pairs = [&] {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(kNumSMs & ~1); cfg.blockDim = dim3(Cfg::kThreads); cfg.dynamicSmemBytes = Cfg::kSmemBytes;
        cudaLaunchAttribute at;
        at.id = cudaLaunchAttributeClusterDimension;
        at.val.clusterDim.x = 2; at.val.clusterDim.y = 1; at.val.clusterDim.z = 1;
        cfg.attrs = &at; cfg.numAttrs = 1;
        int n = 0;
        if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess || n < 1) { (void)cudaGetLastError(); n = kNumSMs / 2; }
        return n < kNumSMs / 2 ? n : kNumSMs / 2;
    }();
    const int tiles = ((M + Cfg::kTileM - 1) / Cfg::kTileM) * ((N + BN - 1) / BN);
    const int pairs = tiles < max_pairs ? tiles : max_pairs;
    AGRL_LAUNCH_BEGIN(st);
    kern<<<2 * pairs, Cfg::kThreads, Cfg::kSmemBytes, st>>>(map_a, map_b, M, N, k_pad, epi);
    AGRL_LAUNCH_CHECK(st, Epi::kName);
    return AGRL_OK;
}

template <int P, int BN, bool kSplit, class Epi>
int launch_split_gemm(const CUtensorMap &map_a, const CUtensorMap &map_b, int M, int N, int k_pad,
                      const Epi &epi, cudaStream_t st, int max_ctas = 0) {
    using Cfg = Config<P, BN, kSplit, Epi::kDirect, Epi::kChunkKb>;
    static_assert(!Epi::kDirect || !kSplit, "the direct epilogue reads a single accumulator");
    auto kern = split_gemm_kernel<P, BN, kSplit, Epi>;
    AGRL_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
    const int tiles = ((M + BM - 1) / BM) * ((N + BN - 1) / BN);
    // persistent grid: one CTA per SM, or per SM of the partition the caller leaves to this kernel (max_ctas > 0)
    const int width = (max_ctas > 0 && max_ctas < kNumSMs) ? max_ctas : kNumSMs;
    const int grid = tiles < width ? tiles : width;
    AGRL_LAUNCH_BEGIN(st);
    kern<<<grid, Cfg::kThreads, Cfg::kSmemBytes, st>>>(map_a, map_b, M, N, k_pad, epi);
    AGRL_LAUNCH_CHECK(st, Epi::kName);
    return AGRL_OK;
}

// fp32 rows -> operand planes of one split format (+ optional squared norms / L2 normalisation); see split.cu
struct SplitArgs {
    const float *src; int64_t ld;      // (rows, dim) fp32
    __nv_bfloat16 *planes;             // [P][rows][k_pad]
    float *sumsq;                      // optional: per-row sum of squares (of the un-normalised row)
    int64_t rows; int dim; int k_pad;
    int split;                         // AGRL_SPLIT_*: the format of the planes (planes.cuh)
    int normalize;                     // 1: split x / max(||x||, 1e-12) instead of x (cosine_distance)
    const float *prescale = nullptr;   // device, the power of two of the tensor (AGRL_SPLIT_FP16X1 / AGRL_SPLIT_FP16_E4M3)
    float *unscale = nullptr;          // AGRL_SPLIT_FP16X2: 1 / s per row
};
int launch_split_planes(const SplitArgs &a, cudaStream_t st);

static inline int64_t pad_k(int64_t dim) { return (dim + BK - 1) / BK * BK; }

}  // namespace gemm
}  // namespace agrl
