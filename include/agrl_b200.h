/*
 * agrl_b200.h -- C ABI of libagrl_b200.so: AGRL's test-time hot path on one B200 (sm_100a).
 *
 * The reference (weleen/AGRL.pytorch) is Python; its only native component is the Cython evaluator
 * torchreid/metrics/rank_cylib/rank_cy.pyx.  Each entry point below names the reference interface
 * it replaces (file:line in the reference tree).  The reference-side bindings (ctypes stubs that a
 * maintainer would drop into torchreid/) are shown in INTEGRATION.md and shipped, ready-made, as
 * the Python package agrl.pytorch_b200.
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / C++ types cross the boundary;
 *   - "dev" pointers are device memory of the CURRENT CUDA device, "host" pointers are ordinary
 *     host memory (pageable or pinned);
 *   - every *_dev entry point is asynchronous on `stream` (a cudaStream_t passed as void*), does
 *     no allocation and no synchronisation, and needs a caller-owned workspace whose size comes
 *     from the matching *_workspace_bytes(); it is re-entrant -- the library keeps NO process-global mutable
 *     state, every tuning knob is a field of the call's parameter struct -- so one host thread per GPU may
 *     call concurrently (nn.DataParallel, train_vidreid_xent_htri.py:318);
 *   - every *_host entry point copies host->device, runs the same kernels, copies the result back
 *     and synchronises before returning (this is the end-to-end path bench.py reports as `e2e`);
 *   - return value: AGRL_OK (0) or a negative AGRL_E_* code; nothing throws across the boundary.
 *     Data-dependent conditions the reference reports as Python exceptions are returned through
 *     `status` words (see each function) so the async path needs no sync to detect them.
 *   - there is NO CPU fallback: without a CUDA device of compute capability 10.x every compute
 *     entry point returns AGRL_E_NO_DEVICE.
 */
#ifndef AGRL_B200_H_
#define AGRL_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AGRL_B200_ABI_VERSION 2

#if defined(__GNUC__)
#define AGRL_API __attribute__((visibility("default")))
#else
#define AGRL_API
#endif

/* ---- return codes ------------------------------------------------------------------------- */
#define AGRL_OK               0
#define AGRL_E_INVALID       -1   /* bad argument (null pointer, negative size, unknown metric)   */
#define AGRL_E_NO_DEVICE     -2   /* no CUDA device / not compute capability 10.x                  */
#define AGRL_E_CUDA          -3   /* a CUDA runtime call failed; see agrl_last_cuda_error()        */
#define AGRL_E_WORKSPACE     -4   /* workspace missing or smaller than *_workspace_bytes()         */
#define AGRL_E_UNSUPPORTED   -5   /* shape outside what the kernels handle (documented per call)   */
#define AGRL_E_NO_VALID_QUERY  -6 /* rank_cy.pyx:227 AssertionError "all query identities do not
                                     appear in gallery" (host entry points only)                  */
#define AGRL_E_ZERO_DIVISION -7   /* rank.py:203 ZeroDivisionError: a query has no cross-camera
                                     match under the MARS metric (host entry points only)          */
#define AGRL_E_LABEL_RANGE   -8   /* a pid / camid does not fit in int32 (host entry points only)  */

/* ---- bits of the device-side `status` word written by the *_dev ranking calls -------------- */
#define AGRL_ST_NO_VALID_QUERY  1u
#define AGRL_ST_ZERO_DIVISION   2u
#define AGRL_ST_LABEL_RANGE     4u
#define AGRL_ST_TOPK_OVERFLOW   8u   /* agrl_distance_topk_dev: a candidate list ran out of slots; take the unfused route */

/* ---- distance metrics (torchreid/metrics/distance.py:46-54) -------------------------------- */
#define AGRL_METRIC_EUCLIDEAN 0   /* squared euclidean, no clamp, no sqrt (distance.py:59-73)     */
#define AGRL_METRIC_COSINE    1   /* 1 - cos, rows L2-normalised with eps 1e-12 (distance.py:76-89) */

/* ---- operand split of the tensor-core GEMMs ------------------------------------------------- */
#define AGRL_SPLIT_BF16X3     3   /* fp32 = 3 bf16 planes, 6 products: all 24 significand bits (the distance
                                     matrix's default in rounds 1-2a; re-ranking; selectable)      */
#define AGRL_SPLIT_BF16X2     2   /* 2 planes, 3 products: ~2^-17 relative per product (default for
                                     the graph layers, whose output enters with gamma = 0.1)       */

#define AGRL_SPLIT_FP16X1      1   /* graph layers only, opt-in: ONE fp16 plane per operand (11 significant
                                     bits, the precision class of TF32), operands pre-scaled by exact powers
                                     of two (per tracklet / per layer) into the fp16 range; one product
                                     instead of three.  Measured head error 1e-5 norm-relative, 3e-5
                                     max-scaled (bar 1e-4); not offered for the distance matrix            */

#define AGRL_SPLIT_FP16_E4M3   4   /* graph layers only: the scaled fp16 plane of AGRL_SPLIT_FP16X1 plus the two first-order
                                     corrections as ONE K-concatenated 8-bit product, y.w ~ fp16(y).fp16(w) + e4m3(r_y).e4m3(w)
                                     + e4m3(y).e4m3(r_w) with r = x - fp16(x): the operand bits of AGRL_SPLIT_BF16X2 (11 + 4
                                     vs 8 + 8) at two thirds of its tensor-core time (kind::f8f6f4 runs at twice the fp16 rate).
                                     Measured head error ~1e-6 (bar 1e-4), like BF16X2.  Needs the tensor-core graph kernel
                                     (<= 64 nodes per tracklet, C % 128 == 0); AGRL_E_UNSUPPORTED otherwise.                      */

#define AGRL_SPLIT_FP16X2      5   /* distance matrix only (its default): fp32 = fp16(x s) + 2^-11 fp16((x s - fp16(x s)) 2^11), s a power
                                     of two PER ROW that puts the row's largest element in [2^7, 2^8): 22 operand bits in two planes,
                                     THREE products (h.h in one accumulator, h.l + l.h in another, joined as main + 2^-11 corr)
                                     instead of the six of AGRL_SPLIT_BF16X3 -- the "3xTF32" scheme with fp16's 11-bit significand.
                                     Operand error <= 2^-22 per element (4.5e-9 of |q||g| on a 4096-long dot product, below
                                     fp32 accumulation noise); elements more than 2^22 below their row's maximum lose
                                     relative (never absolute) precision.                                                      */

AGRL_API int         agrl_abi_version(void);
AGRL_API const char *agrl_status_string(int code);
AGRL_API const char *agrl_last_cuda_error(void);           /* thread-local text of the last CUDA failure   */
/* 0 when the current device can run this library (compute capability 10.x), else AGRL_E_NO_DEVICE */
AGRL_API int         agrl_device_ok(void);
/* number of kernels this library has launched from the calling thread (bench.py `gpu_launches`)   */
AGRL_API uint64_t    agrl_launch_count(void);
/* Kernel timeline of the calling thread: between begin and end every kernel this library launches is
 * followed by a CUDA event on its stream; end synchronises and writes "name:ms;name:ms;..." (the
 * time from the previous event to this one, i.e. the kernel's duration on a busy stream). */
AGRL_API int         agrl_profile_begin(void *stream);
AGRL_API int         agrl_profile_end(char *text, size_t capacity);
/* =============================================================================================
 * (3) Ranking -- replaces rank_cy.evaluate_cy (torchreid/metrics/rank_cylib/rank_cy.pyx:24-32,
 *     eval_market1501_cy :154-241) and evaluate_mars / Compute_AP (torchreid/metrics/rank.py:160-212),
 *     both reached through evaluate_rank (rank.py:215-238).
 *
 *     Ordering: each row is ranked by (distance, gallery index) ascending, NaN last, -0 == +0,
 *     i.e. numpy.argsort(kind='stable'); the reference's default argsort leaves ties undefined.
 *     Labels are int64 in the ABI (rank_cy.pyx:26-29 casts to int64) but must fit in int32.
 * ============================================================================================= */

AGRL_API size_t agrl_rank_workspace_bytes(int64_t num_q, int64_t num_g, int64_t max_rank);

/*
 * market1501 metric, fp32 semantics of rank_cy (float accumulators, AP term in double rounded to
 * float at every step, stale `cmc` scratch tail when the kept gallery is shorter than max_rank).
 *   distmat_dev   (num_q, num_g) fp32, row stride ld_dist elements
 *   cmc_dev       out, min(max_rank, num_g) floats      all_ap_dev  out, num_q floats (may be NULL)
 *   map_dev       out, 1 float                          num_valid_dev out, 1 int64 (may be NULL)
 *   status_dev    out, 1 uint32: AGRL_ST_NO_VALID_QUERY | AGRL_ST_LABEL_RANGE (outputs then undefined)
 */
AGRL_API int agrl_rank_market1501_dev(const float *distmat_dev, int64_t ld_dist,
                             const int64_t *q_pids_dev, const int64_t *g_pids_dev,
                             const int64_t *q_camids_dev, const int64_t *g_camids_dev,
                             int64_t num_q, int64_t num_g, int64_t max_rank,
                             float *cmc_dev, float *map_dev, float *all_ap_dev,
                             int64_t *num_valid_dev, uint32_t *status_dev,
                             void *workspace_dev, size_t workspace_bytes, void *stream);

/*
 * MARS metric, float64 semantics of evaluate_mars: only the top max_rank of each row is inspected,
 * junk = pid == -1 or same pid & same camera, trapezoid AP, CMC/mAP are means over ALL queries
 * (np.mean: pairwise summation for mAP).  Needs 1 <= max_rank <= min(num_g, 8192).
 *   cmc_dev  out, max_rank doubles     map_dev out, 1 double     all_ap_dev out, num_q doubles (may be NULL)
 *   status_dev out: AGRL_ST_ZERO_DIVISION | AGRL_ST_LABEL_RANGE
 */
AGRL_API int agrl_rank_mars_dev(const float *distmat_dev, int64_t ld_dist,
                       const int64_t *q_pids_dev, const int64_t *g_pids_dev,
                       const int64_t *q_camids_dev, const int64_t *g_camids_dev,
                       int64_t num_q, int64_t num_g, int64_t max_rank,
                       double *cmc_dev, double *map_dev, double *all_ap_dev,
                       uint32_t *status_dev,
                       void *workspace_dev, size_t workspace_bytes, void *stream);

/*
 * Gallery-sharded MARS metric (one gallery shard per GPU, SURVEY.md section 8e).  Each shard calls
 * _partial on its (num_q, num_g_shard) distance block: it emits, per query, the shard's best max_rank
 * candidates as 64-bit keys (order-preserving distance bits << 32 | GLOBAL gallery index; all-ones =
 * empty slot), their class bytes (bit0 good, bit1 junk) and the shard's good-image count.  After an
 * all-gather of keys/classes ([part][query][max_rank]) and an all-reduce(sum) of the good counts,
 * _merge produces exactly what agrl_rank_mars_dev would on the concatenated gallery.
 * The status word of _partial only ever carries AGRL_ST_LABEL_RANGE; _merge ORs AGRL_ST_ZERO_DIVISION
 * into its own (which the caller zeroes).  parts * max_rank <= 16384.
 */
AGRL_API int agrl_rank_mars_partial_dev(const float *distmat_dev, int64_t ld_dist,
                               const int64_t *q_pids_dev, const int64_t *g_pids_dev,
                               const int64_t *q_camids_dev, const int64_t *g_camids_dev,
                               int64_t num_q, int64_t num_g, int64_t max_rank, int64_t index_offset,
                               uint64_t *keys_dev, uint8_t *cls_dev, int32_t *ngood_dev,
                               uint32_t *status_dev,
                               void *workspace_dev, size_t workspace_bytes, void *stream);
AGRL_API int agrl_rank_mars_merge_dev(const uint64_t *keys_dev, const uint8_t *cls_dev,
                             const int32_t *ngood_dev, int64_t parts, int64_t num_q, int64_t max_rank,
                             double *cmc_dev, double *map_dev, double *all_ap_dev,
                             uint32_t *status_dev,
                             void *workspace_dev, size_t workspace_bytes, void *stream);

/*
 * Gallery-sharded market1501 metric (SURVEY.md section 8e, last row).  Per shard:
 *   _count     max over queries of this shard's same-pid gallery items  (host: all-reduce MAX -> cap)
 *   _gather    per query the shard's same-pid items as keys (distance bits << 32 | global index << 1 |
 *              junk bit; all-ones = empty), positive / junk counts       (all-gather keys [part][query][cap],
 *                                                                        all-reduce(sum) counts)
 *   _bin       sorts the gathered list (same order on every shard) and counts, per list item, the
 *              shard's row elements sorting before it -> cnt [query][len], sorted [query][len]
 *              with len = agrl_rank_market1501_list_len(parts, cap)       (all-reduce(sum) cnt)
 *   _finalize  kept ranks -> AP / CMC / mAP, bit-identical to agrl_rank_market1501_dev on the whole gallery
 * parts * cap <= 8192; global gallery indices < 2^31.
 */
AGRL_API int agrl_rank_market1501_count_dev(const int64_t *q_pids_dev, const int64_t *g_pids_dev,
                                   const int64_t *q_camids_dev, const int64_t *g_camids_dev,
                                   int64_t num_q, int64_t num_g, int32_t *max_count_dev, uint32_t *status_dev,
                                   void *workspace_dev, size_t workspace_bytes, void *stream);
AGRL_API int agrl_rank_market1501_gather_dev(const float *distmat_dev, int64_t ld_dist,
                                    const int64_t *q_pids_dev, const int64_t *g_pids_dev,
                                    const int64_t *q_camids_dev, const int64_t *g_camids_dev,
                                    int64_t num_q, int64_t num_g, int64_t index_offset, int64_t cap,
                                    uint64_t *keys_dev, int32_t *npos_dev, int32_t *njunk_dev, uint32_t *status_dev,
                                    void *workspace_dev, size_t workspace_bytes, void *stream);
AGRL_API int64_t agrl_rank_market1501_list_len(int64_t parts, int64_t cap);
AGRL_API int agrl_rank_market1501_bin_dev(const float *distmat_dev, int64_t ld_dist, int64_t num_q, int64_t num_g,
                                 int64_t index_offset, const uint64_t *keys_all_dev, int64_t parts, int64_t cap,
                                 int32_t *cnt_dev, uint64_t *sorted_dev, void *stream);
AGRL_API size_t agrl_rank_market1501_finalize_workspace_bytes(int64_t num_q, int64_t parts, int64_t cap, int64_t max_rank);
AGRL_API int agrl_rank_market1501_finalize_dev(const int32_t *cnt_total_dev, const uint64_t *sorted_dev,
                                      const int32_t *npos_total_dev, const int32_t *njunk_total_dev,
                                      int64_t num_q, int64_t num_g_total, int64_t parts, int64_t cap, int64_t max_rank,
                                      float *cmc_dev, float *map_dev, float *all_ap_dev, int64_t *num_valid_dev,
                                      uint32_t *status_dev, void *workspace_dev, size_t workspace_bytes, void *stream);

/* Host-buffer forms (numpy in / numpy out like the reference).  cmc_host must hold max_rank
 * entries; *rank_len_out receives min(max_rank, num_g) for the market1501 metric. */
AGRL_API int agrl_rank_market1501_host(const float *distmat_host,
                              const int64_t *q_pids, const int64_t *g_pids,
                              const int64_t *q_camids, const int64_t *g_camids,
                              int64_t num_q, int64_t num_g, int64_t max_rank,
                              float *cmc_host, float *map_host, float *all_ap_host,
                              int64_t *rank_len_out, int64_t *num_valid_out);
AGRL_API int agrl_rank_mars_host(const float *distmat_host,
                        const int64_t *q_pids, const int64_t *g_pids,
                        const int64_t *q_camids, const int64_t *g_camids,
                        int64_t num_q, int64_t num_g, int64_t max_rank,
                        double *cmc_host, double *map_host, double *all_ap_host);

/* =============================================================================================
 * (2) Distance matrix -- replaces compute_distance_matrix (torchreid/metrics/distance.py:11-56):
 *     euclidean_squared_distance :59-73 and cosine_distance :76-89.
 *     out[i,j] = (|q_i|^2 + |g_j|^2) - 2 q_i.g_j     or     1 - q^_i.g^_j
 *     The contraction runs on tcgen05 tensor cores with 16-bit operand planes (`split`: AGRL_SPLIT_FP16X2,
 *     AGRL_SPLIT_BF16X3 or AGRL_SPLIT_BF16X2), fp32 accumulation in TMEM; norms and the epilogue are fp32.
 * ============================================================================================= */
AGRL_API size_t agrl_distance_workspace_bytes(int64_t num_q, int64_t num_g, int64_t dim, int split);

AGRL_API int agrl_distance_dev(const float *q_dev, int64_t ld_q, const float *g_dev, int64_t ld_g,
                      float *out_dev, int64_t ld_out,
                      int64_t num_q, int64_t num_g, int64_t dim, int metric, int split,
                      void *workspace_dev, size_t workspace_bytes, void *stream);

/* Retrieval form: an operand (e.g. the gallery) is prepared once -- bf16 planes + norms, or planes
 * of the L2-normalised rows for the cosine metric -- and reused for many query batches.
 * agrl_distance_dev(q, g) == prepare(q) + prepare(g) + agrl_distance_prepared_dev. */
AGRL_API size_t agrl_distance_operand_bytes(int64_t rows, int64_t dim, int split);
AGRL_API int agrl_distance_prepare_operand_dev(const float *x_dev, int64_t ld, int64_t rows, int64_t dim,
                                      int metric, int split, void *operand_dev, size_t operand_bytes,
                                      void *stream);
AGRL_API int agrl_distance_prepared_dev(const void *q_operand_dev, int64_t num_q,
                               const void *g_operand_dev, int64_t num_g, int64_t dim, int metric, int split,
                               float *out_dev, int64_t ld_out, void *stream);

/* Fused distance -> per-query top-k (SURVEY.md section 7 step 6; compute_distance_matrix distance.py:11-89 followed by
 * `np.argsort(score)[:max_rank]` of evaluate_mars, rank.py:171-172): the (num_q x num_g) matrix is never written.  The
 * distance of every pair has exactly the bits agrl_distance_prepared_dev would store; the GEMM epilogue turns them into
 * ranking keys (order-preserving distance bits << 32 | index_offset + gallery row, i.e. numpy's stable order) and keeps,
 * per query, the max_rank smallest.
 *   keys_dev    out (num_q, max_rank) uint64, ascending, all-ones = empty slot (num_g < max_rank)
 *   status_dev  out, 1 uint32: zeroed, then AGRL_ST_TOPK_OVERFLOW if a query's candidate list ran out of slots (a
 *               gallery ordered by distance to the query defeats the running threshold): keys are then NOT valid and
 *               the caller takes agrl_distance_prepared_dev + agrl_rank_mars_partial_dev instead.
 * Same result as agrl_rank_mars_partial_dev's keys on the materialised matrix.  max_rank <= 256.
 * agrl_rank_mars_classify_dev then gives what agrl_rank_mars_merge_dev needs besides the keys: the class bytes of the
 * listed items (bit0 good, bit1 junk, rank.py:166-169) and the per-query good-image count of this shard, from the labels
 * alone in O(num_q + num_g); it ORs AGRL_ST_LABEL_RANGE into *status_dev (which the caller, or agrl_distance_topk_dev,
 * initialised). */
AGRL_API size_t agrl_distance_topk_workspace_bytes(int64_t num_q);
AGRL_API int agrl_distance_topk_dev(const void *q_operand_dev, int64_t num_q, const void *g_operand_dev, int64_t num_g,
                           int64_t dim, int metric, int split, int64_t max_rank, int64_t index_offset,
                           uint64_t *keys_dev, uint32_t *status_dev,
                           void *workspace_dev, size_t workspace_bytes, void *stream);
AGRL_API size_t agrl_rank_mars_classify_workspace_bytes(int64_t num_q, int64_t num_g);
AGRL_API int agrl_rank_mars_classify_dev(const uint64_t *keys_dev,
                                const int64_t *q_pids_dev, const int64_t *g_pids_dev,
                                const int64_t *q_camids_dev, const int64_t *g_camids_dev,
                                int64_t num_q, int64_t num_g, int64_t max_rank, int64_t index_offset,
                                uint8_t *cls_dev, int32_t *ngood_dev, uint32_t *status_dev,
                                void *workspace_dev, size_t workspace_bytes, void *stream);

AGRL_API int agrl_distance_host(const float *q_host, const float *g_host, float *out_host,
                       int64_t num_q, int64_t num_g, int64_t dim, int metric, int split);

/* =============================================================================================
 * (1) Graph head -- replaces the eval-mode tail of GSTA.forward (torchreid/models/vmgn.py:296-321):
 *     global pooling + BN neck (:299-301), pyramid part pooling into S*P region nodes (:304-308),
 *     num_gb x GraphLayer.forward (:142-172, affinity :104-123), temporal attention (:270-278),
 *     part mean + BN neck + concat (:317-321).  The ResNet-50 backbone (featuremaps, :280-290)
 *     stays on stock cuDNN in the caller.
 *
 *     Canonical geometry only: pyramid strips of num_split = 4 ([4,2,1] -> P = 7 parts,
 *     utils/reidtools.py:13-15), feature-map height h divisible by 4, C divisible by 128,
 *     S*P <= 64 nodes per tracklet.  Anything else returns AGRL_E_UNSUPPORTED.
 * ============================================================================================= */
#define AGRL_HEAD_MAX_LAYERS 4

typedef struct agrl_head_params {
    int32_t channels;             /* C = 2048 (vmgn.py:221)                                        */
    int32_t num_layers;           /* num_gb (vmgn.py:254-260)                                      */
    int32_t use_pose;             /* GraphLayer.use_pose  (vmgn.py:155)                            */
    int32_t learn_graph;          /* GraphLayer.learn_graph (vmgn.py:159)                          */
    float   gamma;                /* 0.1 (vmgn.py:74,172)                                          */
    float   leaky_slope;          /* 0.1 (vmgn.py:95)                                              */
    float   bn_eps;               /* 1e-5                                                          */
    int32_t split;                /* AGRL_SPLIT_BF16X2, AGRL_SPLIT_BF16X3, AGRL_SPLIT_FP16X1 or AGRL_SPLIT_FP16_E4M3 */
    /* device pointers, fp32; BN vectors have C entries, linear weights are (C, C) row-major [out,in] */
    const float *linear_weight[AGRL_HEAD_MAX_LAYERS];      /* graph_layers.i.linear.weight          */
    const float *bn_weight[AGRL_HEAD_MAX_LAYERS];          /* graph_layers.i.bn.{weight,bias,...}    */
    const float *bn_bias[AGRL_HEAD_MAX_LAYERS];
    const float *bn_mean[AGRL_HEAD_MAX_LAYERS];
    const float *bn_var[AGRL_HEAD_MAX_LAYERS];
    const float *global_bn[4];    /* global_bottleneck.{weight,bias,running_mean,running_var}      */
    const float *att_bn[4];       /* att_bottleneck.{weight,bias,running_mean,running_var}         */
    int32_t maps_nhwc;            /* 0: x4_1 / x4_2 are (B*S, C, h, w) NCHW-contiguous (the reference);
                                     1: channels-last memory, (B*S, h, w, C) (torch.channels_last
                                     backbone): pooled directly, no layout conversion pass            */
    /* tuning knobs; 0 = the library's default.  Results change at most by summation order (far below the parity bars). */
    int32_t lowrank_off;          /* 1: run the FIRST layer's X.W^T on all 7S node rows.  Default: on the 4S quarter-strip
                                     rows (the pooled nodes of a frame are linear combinations of its four quarter strips:
                                     G.X.W^T = (G.T).(Q.W^T)), then a mixing kernel applies G.T and the layer's epilogue
                                     (needs C % 512 == 0; else this is ignored).  Changes the workspace size.          */
    int32_t pool_register_loads;  /* 1: the register-load pooling kernel even where the bulk-copy (TMA ring) kernel
                                     applies (16x8 maps, 16-byte aligned)                                             */
    int32_t pool_stages;          /* ring stages per pooling CTA, 2..12 (16 KiB each at fp32, 8 KiB at 16 bits);
                                     0 = 4 at fp32, 12 at 16 bits                                                     */
    int32_t pool_no_l2_hint;      /* 1: no evict-first L2 hint on the pooling bulk copies                              */
    int32_t gemm_no_pair;         /* AGRL_SPLIT_FP16_E4M3 only.  Default: the layer GEMMs run as CTA pairs (tcgen05
                                     cta_group::2, 256 x 256 tiles, each CTA loads half of the W tile: a third less L2 -> SM
                                     traffic, which is what bounds this mode; 16.0 -> 12.7 ms per 11310-tracklet pass).
                                     1: one CTA per 128 x 256 tile.  Bit-identical results either way.                   */
    int32_t maps_dtype;           /* element type of x4_1 / x4_2: AGRL_MAPS_FP32 (0, default), AGRL_MAPS_BF16 (1),
                                     AGRL_MAPS_FP16 (2) -- the maps of a backbone run under autocast, read as they are
                                     (half the bytes of fp32) and summed in fp32: the same bits as their fp32 copy gives.
                                     Prepared buffer and workspace sizes do not depend on it.                          */
} agrl_head_params;

#define AGRL_MAPS_FP32 0
#define AGRL_MAPS_BF16 1
#define AGRL_MAPS_FP16 2

/* bytes of the persistent, weight-derived buffer (bf16 planes of W, folded BN scale/shift) */
AGRL_API size_t agrl_head_prepared_bytes(const agrl_head_params *p);
/* fills `prepared_dev`; call once per weight load, asynchronous on stream */
AGRL_API int    agrl_head_prepare_dev(const agrl_head_params *p, void *prepared_dev, size_t prepared_bytes,
                             void *stream);
AGRL_API size_t agrl_head_workspace_bytes(const agrl_head_params *p, int64_t batch, int32_t seq_len);

/*
 *   x4_1_dev, x4_2_dev  (batch*seq_len, C, h, w) NCHW contiguous (layer4_1 / layer4_2 outputs), or the same
 *                       tensors in channels-last memory when p->maps_nhwc (aligned to 4 elements); the pointers are
 *                       typed float but point to elements of p->maps_dtype (fp32, bf16 or fp16)
 *   adj_dev             (batch, V, V) fp32, V = seq_len * 7 (dataset_loader.py:345-388); may be NULL
 *                       when use_pose == 0
 *   out_dev             (batch, 2*C) fp32, row stride ld_out: [BN(global mean) | BN(attention feature)]
 *   nodes_out_dev       optional (batch, V, C) fp32 copy of the node features after the last graph
 *                       layer (for tests); NULL in production
 */
AGRL_API int agrl_head_forward_dev(const agrl_head_params *p, const void *prepared_dev,
                          const float *x4_1_dev, const float *x4_2_dev, const float *adj_dev,
                          float *out_dev, int64_t ld_out, float *nodes_out_dev,
                          int64_t batch, int32_t seq_len, int32_t h, int32_t w,
                          void *workspace_dev, size_t workspace_bytes, void *stream);

/* =============================================================================================
 * SURVEY.md section 8(f) rows ("next"): the callers / data formats either side of the path.
 * ============================================================================================= */

/* ---- Pose-guided adjacency (torchreid/dataset_loader.py: generate_graph :218-343, adj_graph :345-388) ----------
 * Canonical configuration only: num_parts = 3 (head / body / leg keypoint classes, :318-320), num_split = 4 with
 * the pyramid strips [4,2,1] (7 nodes per frame), method 'same', num_scale = 1.  The reference builds the dense
 * (V, V) matrix with python sets and itertools.permutations inside the loader workers; the graph is completely
 * described by three V-bit membership masks per tracklet (bit s*7 + strip: that node holds the class), 24 bytes
 * instead of 12.5 KB.
 *
 * agrl_pose_part_masks_dev: raw detections -> masks.
 *   keypoints_dev (batch, seq_len, 18, 3) float64 [x, y, confidence] in ORIGINAL image coordinates (the pose dict
 *                 entry poses[key], :316); heights_dev (batch, seq_len) float64 = im_sizes[..][1] (:313);
 *   valid_dev     (batch, seq_len) uint8, 0 where the pose lookup fails (:337-338 leaves the frame empty); may be
 *                 NULL (all valid);  threshold: 0.1 in the reference (:219);
 *   masks_dev     out (batch, 3) uint64.
 * agrl_pose_adjacency_dev: masks -> the reference's dense fp32 matrix (batch, nodes, nodes), binary, zero diagonal.
 * agrl_head_forward_compact_dev: agrl_head_forward_dev with the masks in place of adj_dev (the dense matrix is
 *   never materialised).  Bit-identical to running agrl_head_forward_dev on the expanded matrix. */
AGRL_API int agrl_pose_part_masks_dev(const double *keypoints_dev, const double *heights_dev, const uint8_t *valid_dev,
                             int64_t batch, int32_t seq_len, int32_t num_split, double threshold,
                             uint64_t *masks_dev, void *stream);
AGRL_API int agrl_pose_adjacency_dev(const uint64_t *masks_dev, int64_t batch, int32_t nodes, float *adj_dev,
                            void *stream);
AGRL_API int agrl_head_forward_compact_dev(const agrl_head_params *p, const void *prepared_dev,
                                  const float *x4_1_dev, const float *x4_2_dev, const uint64_t *part_masks_dev,
                                  float *out_dev, int64_t ld_out, float *nodes_out_dev,
                                  int64_t batch, int32_t seq_len, int32_t h, int32_t w,
                                  void *workspace_dev, size_t workspace_bytes, void *stream);

/* ---- k-reciprocal re-ranking (torchreid/utils/re_ranking.py:30-94; test() :523-527 with --re-rank) ---------------
 * q_g (num_q, num_g), q_q (num_q, num_q), g_g (num_g, num_g) fp32 distance matrices with row strides ld_*;
 * out (num_q, num_g) fp32 = jaccard * (1 - lambda) + normalised original distance * lambda.
 * Ties of the initial ranking are broken by index (numpy.argsort(kind='stable')).  Index work is exact; values
 * follow the reference's float32 operation order except expf vs numpy's exp (<= 2 ulp) -> agreement ~1e-6.
 * Limits: k1 <= 30, k2 <= 8, num_q + num_g <= 46000 (AGRL_E_UNSUPPORTED beyond; workspace_bytes returns 0). */
AGRL_API size_t agrl_rerank_workspace_bytes(int64_t num_q, int64_t num_g, int64_t k1, int64_t k2);
AGRL_API int    agrl_rerank_dev(const float *q_g_dev, int64_t ld_qg, const float *q_q_dev, int64_t ld_qq,
                       const float *g_g_dev, int64_t ld_gg, int64_t num_q, int64_t num_g,
                       int64_t k1, int64_t k2, double lambda_value,
                       float *out_dev, int64_t ld_out, void *workspace_dev, size_t workspace_bytes, void *stream);

/* ---- gallery-sharded k-reciprocal re-ranking: the same output split over ranks ------------------------------------
 * Rank r owns the gallery rows [g_off, g_off + n_own) of the global gallery (num_g rows, N = num_q + num_g).  Its
 * n_loc = num_q + n_own *local rows* are all queries, then its gallery rows: local row l is global row l (l < num_q)
 * or l + g_off.  Three calls, with exchanges between them, give its block out[:, j] = re-ranked distance of every query
 * to gallery item g_off + j, bit-identical to agrl_rerank_dev on the whole problem given the same distance bits.
 *   rows    D rows (N fp32 each, in the workspace) and the stable top-K of the local rows [row0, row1) -> rank_rows.
 *           q_g (num_q, num_g) and q_q (num_q, num_q) whole; g_cols (num_g, row1 - max(row0, num_q)), row stride ld_gc,
 *           holds the g_g columns of the range's gallery rows: column t = distances of all gallery items to gallery item
 *           g_off + max(row0, num_q) - num_q + t (NULL when row1 <= num_q).  Call it for any partition of [0, n_loc)
 *           into ranges, e.g. the queries and then one call per column slab.
 *   expand  after every rank's rows: rank_all (N, K) = the query rows (identical on every rank) and every rank's
 *           gallery rows, in global order.  Writes this rank's k-reciprocal rows v_idx / v_val (n_loc, cap) and v_cnt
 *           (n_loc): global column indices ascending, weights summing to 1.
 *   finish  after every rank's expand: v_*_all = the query rows and every rank's gallery rows of v_*, (N, cap) and
 *           (N), in global order.  Writes out (num_q, n_own), row stride ld_out (out may be NULL when n_own == 0).
 * K = max(k1 + 1, k2) and cap = the least power of two >= (k1 + 1)(round_half_even(k1 / 2) + 2), both row strides.
 * The workspace carries the per-rank state (D rows, query expansion, inverted index) from rows to finish: pass the
 * same buffer to all three calls.  Its size is 4 n_loc N + 8 n_loc cap_q + 8 n_own cap_q + 12 (N + 1) + 8 n_loc bytes
 * (+ alignment), cap_q = cap when k2 == 1 else k2 (k1 + 1)(round_half_even(k1 / 2) + 2): the D rows dominate.
 * Limits per rank: 1 <= k1 <= 30, 1 <= k2 <= 8, 0 <= n_own <= 50000, N <= 16 000 000 (AGRL_E_UNSUPPORTED beyond;
 * the workspace query returns 0).  Positions into D are 64-bit. */
AGRL_API size_t agrl_rerank_shard_workspace_bytes(int64_t num_q, int64_t num_g, int64_t n_own, int64_t k1, int64_t k2);
AGRL_API int    agrl_rerank_shard_rows_dev(const float *q_g_dev, int64_t ld_qg, const float *q_q_dev, int64_t ld_qq,
                       const float *g_cols_dev, int64_t ld_gc, int64_t num_q, int64_t num_g, int64_t g_off, int64_t n_own,
                       int64_t row0, int64_t row1, int64_t k1, int64_t k2, int32_t *rank_rows_dev,
                       void *workspace_dev, size_t workspace_bytes, void *stream);
AGRL_API int    agrl_rerank_shard_expand_dev(const int32_t *rank_all_dev, int64_t num_q, int64_t num_g, int64_t g_off,
                       int64_t n_own, int64_t k1, int64_t k2, int32_t *v_idx_dev, float *v_val_dev, int32_t *v_cnt_dev,
                       void *workspace_dev, size_t workspace_bytes, void *stream);
AGRL_API int    agrl_rerank_shard_finish_dev(const int32_t *rank_all_dev, const int32_t *v_idx_all_dev,
                       const float *v_val_all_dev, const int32_t *v_cnt_all_dev, int64_t num_q, int64_t num_g,
                       int64_t g_off, int64_t n_own, int64_t k1, int64_t k2, double lambda_value,
                       float *out_dev, int64_t ld_out, void *workspace_dev, size_t workspace_bytes, void *stream);

/* Clip pooling of the `dense` / `skipdense` test sampling (train_vidreid_xent_htri.py:461-476):
 * feats (tracklets * clips, dim) with the clips of a tracklet consecutive -> out (tracklets, dim),
 * torch.mean(features, 0) (AVG) or torch.max(features, 0) values (MAX) over the clip axis. */
#define AGRL_CLIP_POOL_AVG 0
#define AGRL_CLIP_POOL_MAX 1
AGRL_API int agrl_clip_pool_dev(const float *feats_dev, int64_t ld_feat, int64_t tracklets, int64_t clips,
                       int64_t dim, int mode, float *out_dev, int64_t ld_out, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* AGRL_B200_H_ */
