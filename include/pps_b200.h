/*
 * pps_b200.h — C ABI of libpps_b200.so: the B200 (sm_100a) retrieval hot path of
 * shenyunhang/PPS (part-power-set pooling + distance / ranking / CMC / mAP).
 *
 * Every entry point is `extern "C"`, takes plain pointers and sizes, returns 0 or a
 * negative PPS_ERR_* code, never allocates device memory behind the caller's back
 * (scratch is passed in as `workspace` whose size the matching *_workspace_bytes()
 * call reports) and never synchronises the stream unless its name ends in `_host`.
 * `stream` is a `cudaStream_t` passed as `void*` (0 = legacy default stream).
 *
 * Reference interfaces replaced (paths relative to the reference repo root):
 *   pooling   detectron/modeling/bpm_heads.py:18-55   add_uniform_partition
 *             detectron/modeling/pps_heads.py:38-80   add_pps_part_head_
 *             detectron/modeling/pps_heads.py:83-142  add_pps_part_head (pyramid)
 *             (a Caffe2 sub-graph of Split/AveragePool/MaxPool/Mean/Max/Add; the op
 *             idiom a custom op would follow is detectron/ops/pairwise_distance_op.h:10-21)
 *   distance  detectron/datasets/reid_dataset_evaluator.py:244-272  compute_dist
 *   masks     detectron/datasets/reid_dataset_evaluator.py:327-328,427-428
 *   mAP       detectron/datasets/reid_dataset_evaluator.py:366-439  mean_ap
 *   CMC       detectron/datasets/reid_dataset_evaluator.py:283-363  cmc
 *   evaluate  detectron/datasets/reid_dataset_evaluator.py:29-125   evaluate (single query)
 *   gradient  the op idiom of detectron/ops/pairwise_distance_op.cc:14-24 (GetGradientDefs)   pps_pool_bwd
 *   multi-GPU detectron/utils/subprocess.py:39-103 + core/test_engine.py:205-213             pps_pass_*
 */
#ifndef PPS_B200_H_
#define PPS_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PPS_ABI_VERSION 10

/* ---- error codes (the Python mirror turns every non-zero code into RuntimeError,
 * like CAFFE_ENFORCE does: detectron/tests/test_zero_even_op.py:50-53) ---- */
#define PPS_OK                   0
#define PPS_ERR_INVALID_ARG     -1  /* null pointer, negative size, unknown enum   */
#define PPS_ERR_SHAPE           -2  /* sum(split) != H, n_parts out of range, ...  */
#define PPS_ERR_ALIGN           -3  /* pointer / leading dimension alignment       */
#define PPS_ERR_CUDA            -4  /* a CUDA call failed: pps_last_cuda_error()   */
#define PPS_ERR_UNSUPPORTED     -5  /* valid request this build does not implement */
#define PPS_ERR_WORKSPACE       -6  /* workspace too small                         */
#define PPS_ERR_NO_VALID_QUERY  -7  /* reid_dataset_evaluator.py:358-359           */
#define PPS_ERR_PASS_RESIZE     -9  /* pps_pass_end: a speculative size bound was too small; repeat the pass with
                                       PPS_PASS_SIZING (every rank of a sharded run gets this code) */
#define PPS_ERR_TOPK_OVERFLOW   -8  /* pps_pass_end: a top-k candidate buffer ran over; repeat the pass with
                                       PPS_PASS_NO_EPILOGUE_TOPK (every rank of a sharded run gets this code) */

int         pps_abi_version(void);
const char* pps_strerror(int code);
const char* pps_last_cuda_error(void);   /* thread-local text of the last CUDA failure */

/* ------------------------------------------------------------------------------------
 * Part 1 — part-power-set pooling          (bpm_heads.py:18-55 + pps_heads.py:38-80)
 *
 * x : [N, C, H, W] fp32, NCHW, contiguous (a conv5 map, e.g. [N,2048,24,8]).
 * split[n_parts] : rows per horizontal strip, sum == H   (bpm_heads.py:25-45).
 * mode : PPS_POOL_AVG_MAX  y[m] = max_{j in S_m} avg_j                (pps_heads.py:69-76)
 *        PPS_POOL_MAX_AVE  y[m] = mean_{j in S_m} avg_j + max_{j in S_m} max_j  (:58-68)
 *        where S_m = { j : bit j of m set } and avg_j / max_j are the global average /
 *        max pool of strip j.
 * combos : NULL -> all masks m = 1 .. 2^n_parts - 1 in ascending order (pps_heads.py:47-52);
 *          otherwise n_combos explicit masks (e.g. the 21 contiguous `pyramid_combs`,
 *          pps_heads.py:22-25) emitted in the given order.
 * y : element (n, k, c) of output k (k-th emitted combo) at y[n*y_stride_n + k*y_stride_k + c].
 *     [N, K, C] layout: y_stride_n = K*C, y_stride_k = C.  The reference's list of K blobs
 *     [N,C,1,1] is the [K, N, C] layout: y_stride_n = C, y_stride_k = N*C.
 * ---------------------------------------------------------------------------------- */
#define PPS_POOL_AVG_MAX 0
#define PPS_POOL_MAX_AVE 1
#define PPS_POOL_MAX_PARTS 10

int pps_pool_fwd(const float* x, int N, int C, int H, int W,
                 int n_parts, const int* split, int mode,
                 const int* combos, int n_combos,
                 float* y, long long y_stride_n, long long y_stride_k,
                 void* stream);

/* same pooling, written straight into the bf16 operand planes pps_embed_tc consumes: output k of image n is row
 * k*N + n of out_planes [planes][K*N][pps_kpad(C)] (the [K, N, C] layout, split like pps_split_rows splits it), so the
 * fp32 pooled intermediate and its split pass never touch HBM. */
int pps_pool_planes_fwd(const float* x, int N, int C, int H, int W,
                        int n_parts, const int* split, int mode,
                        const int* combos, int n_combos,
                        void* out_planes, int planes, void* stream);

/* Backward of pps_pool_fwd: dx[N, C, H, W] = d loss / d x given dy = d loss / d y, addressed like y
 * (element (n, k, c) at dy[n*dy_stride_n + k*dy_stride_k + c]).  The reference trains through this sub-graph (the
 * multi-scale branch exists only at train time, pps_heads.py:88-142); a custom op would register it the way
 * detectron/ops/pairwise_distance_op.cc:14-24 registers PairWiseDistanceGradient (inputs {X, dY} -> dX).  Gradients of
 * the stock operators it fuses: AveragePool spreads d avg_j / (h_j W) over strip j; MaxPool routes d max_j to the first
 * maximal element of the strip; Mean divides by |S|; Max passes dY to EVERY input equal to the maximum (Caffe2's
 * MaxGradient), Add to both.  dx is written in full (no accumulation into an existing gradient). */
int pps_pool_bwd(const float* x, const float* dy, int N, int C, int H, int W,
                 int n_parts, const int* split, int mode,
                 const int* combos, int n_combos,
                 long long dy_stride_n, long long dy_stride_k,
                 float* dx, void* stream);

/* ------------------------------------------------------------------------------------
 * Part 2a — operand preparation for the tensor-core distance.
 *
 * Splits fp32 rows into `planes` bf16 planes (x = p0 + p1 [+ p2], each plane the bf16
 * rounding of the remaining residual), K zero-padded to a multiple of 64, and computes
 * the fp32 squared norm of every row (reid_dataset_evaluator.py:266-268) accumulated in
 * fp64.  out_planes : [planes][rows][kpad] bf16 with kpad = pps_kpad(dim).
 * For PPS_DTYPE_F16 input there is no split: planes must be 1 and the rows are copied
 * (padded) as fp16.
 * planes = 2 | PPS_SPLIT_F16_SCALED (fp32 input; what PPS_PREC_F16X3 consumes): the two planes are fp16
 * roundings of the residual of the row SCALED by a power of two s (max|x| s in [2^14, 2^15)), i.e. 22
 * significant bits per element instead of the 16 of two bf16 planes, at the same cost.  out_sqnorm then has
 * 2 * rows entries: |x|^2 of every row, followed by the inverse scales 1 / s (exact powers of two); with the
 * _slab form the second half starts at out_sqnorm + total_rows.
 * ---------------------------------------------------------------------------------- */
#define PPS_DTYPE_F32 0
#define PPS_DTYPE_F16 1
#define PPS_SPLIT_F16_SCALED 0x100

int       pps_kpad(int dim);
long long pps_split_bytes(long long rows, int dim, int planes);
int pps_split_rows(const void* feats, int dtype, long long rows, int dim, long long ld,
                   int planes, void* out_planes, float* out_sqnorm, void* stream);
/* same, for rows [row0, row0+nrows) of a [total_rows, dim] array whose base is `feats`
 * (lets a host->device upload in slabs overlap the split of the slabs already there). */
int pps_split_rows_slab(const void* feats, int dtype, long long row0, long long nrows,
                        long long total_rows, int dim, long long ld, int planes,
                        void* out_planes, float* out_sqnorm, void* stream);

/* same, gathering: output row r is source row row_index[r] - index_base of `feats`
 * (the threshold pass of a multi-block gallery splits only the rows that appear in a same-id pair). */
int pps_split_rows_gather(const void* feats, int dtype, const int32_t* row_index, long long index_base,
                          long long rows, int dim, long long ld, int planes,
                          void* out_planes, float* out_sqnorm, void* stream);

/* ------------------------------------------------------------------------------------
 * Part 2b — distance matrix        (reid_dataset_evaluator.py:244-272, 'euclidean')
 *
 * dist[i*ldd + j] = sqrt(max(0, |a_i|^2 + |b_j|^2 - 2 a_i.b_j)).
 * precision selects how a.b is formed:
 *   PPS_PREC_BF16X1  one tcgen05 pass on the leading bf16 plane       (not parity grade)
 *   PPS_PREC_BF16X3  p0.p0 + p0.p1 + p1.p0, fp32 accumulate in TMEM   (default; ~3e-7 rel)
 *   PPS_PREC_BF16X6  all products down to 2^-24                       (fp32-exact grade)
 *   PPS_PREC_F16X1   operands are fp16 planes (dtype F16), one pass, exact products
 *   PPS_PREC_F16X3   fp32 rows split into two power-of-two-scaled fp16 planes (PPS_SPLIT_F16_SCALED), the three
 *                    terms of BF16X3; dot-product error ~2^-22 |a||b| / sqrt(K), below a float32 sgemm's own
 *                    rounding (measured: tools/split_precision_sim.py).  a_sqnorm / b_sqnorm hold
 *                    2 * plane_rows floats (norms, then inverse scales) and are required even with PPS_DIST_DOT
 *   PPS_PREC_FP32    CUDA-core fp32 FMA kernel on the original fp32 rows (a_f32/b_f32)
 * a_planes/b_planes come from pps_split_rows (need >= the planes the precision uses).
 * a_plane_rows / b_plane_rows: rows between consecutive planes of the buffer (0 = m1 / m2); a row
 * window [r0, r0+m) of a larger [planes][total_rows][kpad] buffer is passed as base + r0*kpad
 * elements, its sqnorm + r0, m rows and plane_rows = total_rows.
 * Default kernel: cluster of 2 CTAs, tcgen05.mma.cta_group::2, 256 x 256 tiles, every plane tile
 * loaded once per k-block and reused by all terms.
 * flags: PPS_DIST_SQUARED returns the clamped squared distance (no sqrt);
 *        PPS_DIST_DOT returns a.b only (the reference's 'cosine' branch at :259-263
 *        once rows are L2-normalised).
 * ---------------------------------------------------------------------------------- */
#define PPS_PREC_BF16X1 1
#define PPS_PREC_BF16X3 3
#define PPS_PREC_BF16X6 6
#define PPS_PREC_F16X1  16
#define PPS_PREC_F16X3  19
#define PPS_PREC_FP32   32

#define PPS_DIST_SQUARED 1
#define PPS_DIST_DOT     2
#define PPS_DIST_KERNEL_1CTA 0x100   /* use the single-CTA 128x256 kernel instead of the 2-CTA 256x256 one */
#define PPS_DIST_CLUSTER4 0x400        /* single-plane products: clusters of 4 CTAs whose two CTA pairs share the B tile by TMA
                                          multicast (bit-identical; 25 % less L2 -> SM traffic but measured slower, opt-in) */
#define PPS_DIST_SEPARATE_SMALL 0x800  /* multi-term precisions: the cross terms accumulate in a TMEM buffer of their own and are
                                          added in the epilogue - the large accumulator then sees a third of the MMA steps
                                          (the tensor core truncates ~1 ulp of the accumulator per step) */
#define PPS_DIST_SQRT_RN 0x1000        /* correctly rounded square root in the epilogue (what np.sqrt gives) instead of the
                                          hardware approximation */
#define PPS_DIST_RESERVE_SM_PAIR 0x200 /* persistent grid leaves one SM pair idle: the kernel fills the shared memory
                                          of every SM it runs on, so a concurrent NCCL / pair-list kernel on another
                                          stream could otherwise only start when it ends */

int pps_dist_tc(const void* a_planes, const float* a_sqnorm, long long m1, int a_planes_n, long long a_plane_rows,
                const void* b_planes, const float* b_sqnorm, long long m2, int b_planes_n, long long b_plane_rows,
                int dim, int precision, int flags,
                float* dist, long long ldd, void* stream);

int pps_dist_fp32(const float* a, long long lda, const float* a_sqnorm, long long m1,
                  const float* b, long long ldb, const float* b_sqnorm, long long m2,
                  int dim, int flags, float* dist, long long ldd, void* stream);

/* row squared norms only (fp64 accumulate, fp32 result) */
int pps_row_sqnorm(const void* feats, int dtype, long long rows, int dim, long long ld,
                   float* out_sqnorm, void* stream);

/* ------------------------------------------------------------------------------------
 * Part 2c — same-id pair lists (host side; reid_dataset_evaluator.py:320,327-328,421,427-428)
 *
 * For query i the gallery items with gallery_ids == query_ids[i] are its "pairs":
 * positives (camera differs -> valid match) and junk (same camera -> filtered out).
 * Everything else in the gallery is a valid non-match and needs no per-item mask.
 * Two-call pattern: pps_pairs_count() -> total E, then pps_pairs_fill().
 *   pair_off[nq+1] CSR offsets, pair_q[E] query index, pair_g[E] gallery index
 *   (ascending inside a query), pair_pos[E] 1 = positive, 0 = junk.
 * ---------------------------------------------------------------------------------- */
long long pps_pairs_count(const int64_t* query_ids, long long nq,
                          const int64_t* gallery_ids, long long ng);
int pps_pairs_fill(const int64_t* query_ids, const int64_t* query_cams, long long nq,
                   const int64_t* gallery_ids, const int64_t* gallery_cams, long long ng,
                   int32_t* pair_off, int32_t* pair_q, int32_t* pair_g, uint8_t* pair_pos);

/* The same lists built on the device (no sort: a deterministic brute-force sweep, pairs.cu).
 * All pointers are DEVICE pointers; workspace needs pps_pairs_workspace_bytes(nq, ng) bytes.
 * Single block:  pps_pairs_count_device writes pair_off[nq+1] and totals[2] = {n_pairs, max pairs of
 * one query}; the caller reads totals back (the only host round trip of the path, overlappable with
 * the distance GEMM), sizes pair_q/pair_g/pair_pos and calls pps_pairs_fill_device with the SAME
 * workspace (entries beyond `capacity` are dropped; the optional zero_* arrays are zero-filled for
 * the slots written).  The result is identical to pps_pairs_fill.
 * Sharded gallery (each rank sweeps only ITS block of ng rows starting at global row
 * gallery_offset): pps_pairs_local_count -> *local_cnt[nq] (inside the workspace) -> all-gather over
 * ranks into cnt_all[world][nq] -> pps_pairs_offsets (global pair_off, totals; this rank's first
 * slot per query stays in the workspace) -> pps_pairs_fill_local writes the block's pairs into their
 * GLOBAL slots with global gallery indices (pair_pos as bytes and/or as int32 for a SUM exchange). */
long long pps_pairs_workspace_bytes(long long nq, long long ng);
int pps_pairs_count_device(const int64_t* query_ids, long long nq, const int64_t* gallery_ids, long long ng,
                           void* workspace, int32_t* pair_off, int32_t* totals, void* stream);
int pps_pairs_fill_device(const int64_t* query_ids, const int64_t* query_cams, long long nq,
                          const int64_t* gallery_ids, const int64_t* gallery_cams, long long ng,
                          const void* workspace,
                          int32_t* pair_q, int32_t* pair_g, uint8_t* pair_pos,
                          float* zero_f32 /* optional [capacity]: pair_d */, uint32_t* zero_u32 /* optional: cnt_le */,
                          uint32_t* zero_per_query /* optional [nq]: cnt_first */,
                          long long capacity, void* stream);
int pps_pairs_local_count(const int64_t* query_ids, long long nq, const int64_t* gallery_ids, long long ng,
                          void* workspace, int32_t** local_cnt, void* stream);
int pps_pairs_offsets(const int32_t* cnt_all, int world, int rank, long long nq, long long ng_local,
                      void* workspace, int32_t* pair_off, int32_t* totals, void* stream);
int pps_pairs_fill_local(const int64_t* query_ids, const int64_t* query_cams, long long nq,
                         const int64_t* gallery_ids, const int64_t* gallery_cams, long long ng,
                         long long gallery_offset, const void* workspace,
                         int32_t* pair_q, int32_t* pair_g, uint8_t* pair_pos, int32_t* pair_pos32,
                         float* zero_f32, uint32_t* zero_u32, uint32_t* zero_per_query,
                         long long capacity, void* stream);
int pps_pairs_unpack_pos(const int32_t* pair_pos32, long long n_pairs, uint8_t* pair_pos, void* stream);

/* Candidate pre-filter for very large galleries (millions of distractor rows): keeps, in ascending order, only
 * the gallery rows whose id is the id of some query (hash set of the query ids + ordered compaction), so that the
 * pair sweeps above run on a few 10^4 rows instead of the whole gallery:
 *   pps_pairs_prefilter(...) -> cand_rows[*n_cand] (gallery rows), cand_gid / cand_gcam (their ids / cameras)
 *   pps_pairs_count_device / pps_pairs_fill_device on (cand_gid, cand_gcam, *n_cand)   [caller reads *n_cand back]
 *   pps_pairs_remap(pair_g, n_pairs, cand_rows, offset): pair_g[e] = cand_rows[pair_g[e]] + offset.
 * cand_* arrays need room for ng entries in the worst case (every row matches). */
long long pps_pairs_prefilter_workspace_bytes(long long nq, long long ng);
int pps_pairs_prefilter(const int64_t* query_ids, long long nq, const int64_t* gallery_ids,
                        const int64_t* gallery_cams, long long ng, void* workspace,
                        int32_t* cand_rows, int64_t* cand_gid, int64_t* cand_gcam, int32_t* n_cand, void* stream);
int pps_pairs_remap(int32_t* pair_g, long long n_pairs, const int32_t* cand_rows, long long offset, void* stream);

/* Compacted same-id gallery for the threshold pass of a gallery that does not fit one distance block.
 * The thresholds of the ranking are the distances of the same-id pairs only; all queries of one id share one
 * gallery list, so the rows needed are the lists of one representative query per id, restricted to the
 * gallery rows [row_lo, row_hi) this device holds:
 *   gp_rows[0 .. *n_rows)  the distinct gallery rows (global indices) that appear in a pair, grouped by id
 *   pair_col[e]            column of pair e in the product queries x gp_rows, or -1 (row outside the window)
 * The caller runs pps_split_rows_gather(gp_rows) + pps_dist_tc + pps_rank_gather(pair_g := pair_col), i.e. a
 * product with a few 10^4 rows instead of a first sweep over the whole gallery.  All pointers are device
 * pointers; gp_rows / pair_col have n_pairs entries; workspace: pps_pairs_compact_workspace_bytes(nq). */
long long pps_pairs_compact_workspace_bytes(long long nq);
int pps_pairs_compact_rows(const int64_t* query_ids, long long nq, const int32_t* pair_off,
                           const int32_t* pair_q, const int32_t* pair_g, long long n_pairs,
                           long long row_lo, long long row_hi, void* workspace,
                           int32_t* gp_rows, int32_t* pair_col, int32_t* n_rows, void* stream);

/* ------------------------------------------------------------------------------------
 * Part 2d — ranking on a materialised block of the distance matrix.
 *
 * dist : [nq, ncols] block (row stride ldd) holding gallery columns col0 .. col0+ncols-1.
 * Step 1  pps_rank_gather : pair_d[e] = dist[pair_q[e], pair_g[e]-col0] for pairs whose
 *         gallery item lies in the block (others untouched; zero pair_d first, then a
 *         sum-allreduce over gallery shards completes it).
 * Step 2  pps_rank_count  : for every positive pair e, cnt_le[e] += #{columns j of the
 *         block : dist[q,j] <= pair_d[e]}; cnt_first[q] += #{j : d == d*, j < g*} - #{j : d == d*}
 *         (a signed correction stored mod 2^32) with (d*, g*) the query's nearest positive, ties
 *         by gallery index, i.e. the order a stable argsort gives; step 3 adds cnt_le of that
 *         positive to get #{j : (dist[q,j], j) < (d*, g*)}.  No id/camera arrays are read: junk
 *         and positives are subtracted in step 3 from their own pair distances.
 *         Counters are exact integers, so summing them over gallery shards / chunks
 *         gives the unsharded result bit for bit.
 * Step 3  pps_rank_finalize : ap[q] (float64, sklearn >= 0.19 tie-grouped step-wise AP:
 *         (1/P) sum_p tp(d<=d_p)/n_valid(d<=d_p)), is_valid[q], first_rank[q] = 0-based
 *         position of the first correct match in the valid-filtered ranking (-1 if the
 *         query has no valid match), and optionally neg_before[e] = number of valid
 *         non-matches ranked before positive e (what cmc(first_match_break=False) needs).
 * ---------------------------------------------------------------------------------- */
int pps_rank_gather(const float* dist, long long ldd, long long nq, long long ncols, long long col0,
                    const int32_t* pair_q, const int32_t* pair_g, long long n_pairs,
                    float* pair_d, void* stream);

int pps_rank_count(const float* dist, long long ldd, long long nq, long long ncols, long long col0,
                   const int32_t* pair_off, const int32_t* pair_g, const uint8_t* pair_pos,
                   const float* pair_d, int max_pairs_per_query,
                   uint32_t* cnt_le, uint32_t* cnt_first, void* stream);

int pps_rank_finalize(long long nq,
                      const int32_t* pair_off, const int32_t* pair_g, const uint8_t* pair_pos,
                      const float* pair_d, const uint32_t* cnt_le, const uint32_t* cnt_first,
                      double* ap, uint8_t* is_valid, int32_t* first_rank, int32_t* neg_before,
                      void* stream);

/* ------------------------------------------------------------------------------------
 * Part 2e — per-query top-k (smallest distance first, ties by gallery index).
 *
 * Streams a block of the distance matrix once and merges it into the running state
 * topk_key[nq*k] (uint64 = float bits << 32 | global gallery index; initialise to all
 * ones with pps_topk_init).  excl_off / excl_g (optional, CSR per query, global gallery indices)
 * list items to skip; entries whose excl_keep[x] != 0 are NOT skipped (excl_keep may be NULL).
 * Passing the pair lists (pair_off, pair_g, pair_pos) skips exactly the junk and so ranks the
 * valid-filtered gallery.
 * pps_topk_unpack splits the state into distances / indices (-1 = fewer than k items).
 * ---------------------------------------------------------------------------------- */
#define PPS_TOPK_MAX 128
/* Fused form for gallery blocks whose thresholds are already known (multi-block sweeps): the ranking counters are
 * taken in the EPILOGUE of the tensor-core distance kernel, so the [m1, m2] distance block is never written.
 *   pps_rank_tab_prep   per query: the positives' distances sorted ascending (ties by gallery index) into
 *                       thr_tab (+inf padded), their pair indices into tpair_tab, cnt_tab zeroed, the nearest
 *                       positive into dstar / gstar (NaN / 0 for a query without one).  Tables hold
 *                       pps_rank_tab_elems(nq, p_cap) elements laid out [rows/128][p_cap][128]; p_cap is a multiple
 *                       of 8, <= 64, and must be >= the largest number of positives of a query (*overflow counts
 *                       the queries that break this: the caller then uses pps_rank_count on a materialised block).
 *   pps_dist_rank_tc    pps_dist_tc's arithmetic (same operands, same kernel mainloop, bit-identical distances)
 *                       with the counting epilogue: cnt_tab[q][j] += #{columns with exactly j thresholds of q
 *                       strictly below their distance}, cnt_first as in pps_rank_count.  col0 = global gallery
 *                       index of the block's first row.  flags: 0 or PPS_DIST_SQUARED.
 *   pps_rank_tab_finish cnt_le[pair of threshold j] += cnt_tab[q][0] + ... + cnt_tab[q][j]. */
long long pps_rank_tab_elems(long long nq, int p_cap);
int pps_rank_tab_prep(long long nq, const int32_t* pair_off, const int32_t* pair_g, const uint8_t* pair_pos,
                      const float* pair_d, int p_cap, float* thr_tab, int32_t* tpair_tab, uint32_t* cnt_tab,
                      float* dstar, int32_t* gstar, int32_t* overflow, void* stream);
int pps_dist_rank_tc(const void* a_planes, const float* a_sqnorm, long long m1, int a_planes_n, long long a_plane_rows,
                     const void* b_planes, const float* b_sqnorm, long long m2, int b_planes_n, long long b_plane_rows,
                     int dim, int precision, int flags, long long col0, int p_cap,
                     const float* thr_tab, uint32_t* cnt_tab, const float* dstar, const int32_t* gstar,
                     uint32_t* cnt_first, void* stream);
/* pps_dist_rank_tc + the top-k admission of pps_dist_topk_tc in the same epilogue (tk_cand == NULL: none): the form the
 * multi-block pass uses for single-plane operands, so that no block after the first is ever written or re-read. */
int pps_dist_rank_topk_tc(const void* a_planes, const float* a_sqnorm, long long m1, int a_planes_n, long long a_plane_rows,
                          const void* b_planes, const float* b_sqnorm, long long m2, int b_planes_n, long long b_plane_rows,
                          int dim, int precision, int flags, long long col0, int p_cap,
                          const float* thr_tab, uint32_t* cnt_tab, const float* dstar, const int32_t* gstar,
                          uint32_t* cnt_first, const uint32_t* tk_bound, uint32_t* tk_cnt, uint64_t* tk_cand, int tk_cap,
                          void* stream);
int pps_rank_tab_finish(long long nq, int p_cap, const int32_t* tpair_tab, const uint32_t* cnt_tab,
                        uint32_t* cnt_le, void* stream);

/* Secondary metric: AP as scikit-learn 0.18.1 computed it (trapezoidal area under the precision-recall curve) - the
 * version reid_dataset_evaluator.py:398-407 asks for; pps_rank_finalize gives the step-wise AP of scikit-learn >= 0.19.
 *   pps_rank_count_eq            cnt_eq[e] += #{columns of the block with distance EXACTLY pair_d[e]}
 *   pps_rank_finalize_trapezoid  ap[q] = sum over the distinct positive distances v of
 *                                (tp(v) - tp(<v)) / P * (tp(v) / n_le(v) + P_prev(v)) / 2,
 *                                P_prev(v) = tp(<v) / n_lt(v) if n_lt(v) > 0 else 1, n_lt = n_le - n_eq (valid items only). */
int pps_rank_count_eq(const float* dist, long long ldd, long long nq, long long ncols, const int32_t* pair_off,
                      const float* pair_d, int max_pairs_per_query, uint32_t* cnt_eq, void* stream);
int pps_rank_finalize_trapezoid(long long nq, const int32_t* pair_off, const int32_t* pair_g, const uint8_t* pair_pos,
                                const float* pair_d, const uint32_t* cnt_le, const uint32_t* cnt_eq, double* ap,
                                void* stream);

int pps_topk_init(uint64_t* topk_key, long long nq, int k, void* stream);
int pps_topk_update(const float* dist, long long ldd, long long nq, long long ncols, long long col0,
                    const int32_t* excl_off, const int32_t* excl_g, const uint8_t* excl_keep,
                    uint64_t* topk_key, int k, void* stream);
/* pps_rank_count + pps_topk_update in ONE read of the block (one CTA per query): same counters, same top-k state.
 * pair_off must hold nq + 1 valid offsets (all zero when there is no pair at all). */
int pps_rank_sweep(const float* dist, long long ldd, long long nq, long long ncols, long long col0,
                   const int32_t* pair_off, const int32_t* pair_g, const uint8_t* pair_pos, const float* pair_d,
                   int max_pairs_per_query, uint32_t* cnt_le, uint32_t* cnt_first,
                   uint64_t* topk_key, int k, int topk_filtered, void* stream);
/* Top-k admission in the EPILOGUE of the distance kernel (blocks after the first of a multi-block sweep):
 *   pps_topk_bound    tk_bound[q] = distance bits of the current k-th best of the state (all ones: unbounded),
 *                     tk_cnt[q] = 0
 *   pps_dist_topk_tc  pps_dist_tc (identical block) + per element one compare against tk_bound[row]; the few
 *                     that pass are appended to tk_cand[row][tk_cap] (tk_cnt counts them, also past tk_cap)
 *   pps_topk_merge    state + candidates -> new state (junk dropped through the pair lists), new tk_bound,
 *                     tk_cnt = 0; *overflow = 1 if some buffer ran over (repeat the pass with pps_rank_sweep).
 * The block is then only COUNTED (pps_rank_count), not swept for top-k as well. */
int pps_topk_bound(const uint64_t* topk_key, long long nq, int k, uint32_t* tk_bound, uint32_t* tk_cnt, void* stream);
int pps_dist_topk_tc(const void* a_planes, const float* a_sqnorm, long long m1, int a_planes_n, long long a_plane_rows,
                     const void* b_planes, const float* b_sqnorm, long long m2, int b_planes_n, long long b_plane_rows,
                     int dim, int precision, int flags, float* dist, long long ldd,
                     long long col0, const uint32_t* tk_bound, uint32_t* tk_cnt, uint64_t* tk_cand, int tk_cap,
                     void* stream);
int pps_topk_merge(uint64_t* topk_key, long long nq, int k, const uint64_t* tk_cand, int tk_cap,
                   uint32_t* tk_cnt, uint32_t* tk_bound,
                   const int32_t* pair_off, const int32_t* pair_g, const uint8_t* pair_pos,
                   int max_pairs_per_query, int topk_filtered, int32_t* overflow, void* stream);
int pps_topk_unpack(const uint64_t* topk_key, long long nq, int k,
                    float* out_dist, int32_t* out_index, void* stream);

/* ------------------------------------------------------------------------------------
 * Part 2f — the whole single-query evaluation from HOST buffers
 *           (reid_dataset_evaluator.py:104-122: compute_dist -> mean_ap + cmc(topk,
 *           first_match_break=True); the call bench.py times as `e2e`).
 *
 * Copies features to the device (gallery in row slabs; the split + tcgen05 distance of one
 * slab overlap the copy of the next), builds the pair lists on the device, runs gather ->
 * count -> finalize [-> top-k], copies the small results back and synchronises.
 * A pps_ctx owns the streams and grow-only device / pinned scratch, so repeated evaluations
 * allocate nothing; pps_evaluate_host is the one-shot form (create ctx, evaluate, destroy).
 * Host feature buffers should be pinned (cudaHostAlloc / torch pin_memory) for full PCIe
 * bandwidth; pageable memory works but the driver stages it.
 *   out_ap[nq] float64, out_valid[nq], out_first_rank[nq]; out_cmc[cmc_topk] float64 and
 *   *out_map follow the reference's averaging (:360-362, :437-438).
 *   out_topk_index / out_topk_dist [nq, topk] may be NULL (topk = 0).
 * Returns PPS_ERR_NO_VALID_QUERY if no query has a valid match.
 * ---------------------------------------------------------------------------------- */
typedef struct pps_ctx pps_ctx;
int pps_ctx_create(int device, pps_ctx** out);
int pps_ctx_destroy(pps_ctx* ctx);
int pps_evaluate_host_ctx(pps_ctx* ctx, const float* q_feats, long long nq,
                          const float* g_feats, long long ng, int dim,
                          const int64_t* query_ids, const int64_t* query_cams,
                          const int64_t* gallery_ids, const int64_t* gallery_cams,
                          int precision, int cmc_topk, int topk,
                          double* out_map, double* out_cmc,
                          double* out_ap, uint8_t* out_valid, int32_t* out_first_rank,
                          int32_t* out_topk_index, float* out_topk_dist);
/* the same evaluation with features (fp32, contiguous [rows, dim]) and int64 ids / cameras already
 * RESIDENT on the device; everything is enqueued on `stream`, the call returns once the small
 * results are on the host (what bench.py times as `value`). */
int pps_evaluate_device_ctx(pps_ctx* ctx, const float* d_q, long long nq,
                            const float* d_g, long long ng, int dim,
                            const int64_t* d_query_ids, const int64_t* d_query_cams,
                            const int64_t* d_gallery_ids, const int64_t* d_gallery_cams,
                            int precision, int cmc_topk, int topk, void* stream,
                            double* out_map, double* out_cmc,
                            double* out_ap, uint8_t* out_valid, int32_t* out_first_rank,
                            int32_t* out_topk_index, float* out_topk_dist);
/* The resident evaluation in steps, so that a gallery sharded over several GPUs can put its exchanges
 * in between (query ids / cameras are replicated; d_g, d_gallery_ids, d_gallery_cams are the rank's
 * block of ng_local rows starting at global row gallery_offset; world = number of blocks):
 *   pps_rank_begin        (also enqueues the operand split + the distance of the local block)
 *                         -> all-gather of *d_local_cnt [nq int32 per rank] into cnt_all[world][nq]
 *   pps_rank_thresholds   -> all-reduce(SUM, int32) of *d_exchange [*n_words = 3*n_pairs: thresholds as
 *                            float bits | global gallery index | positive flag; one non-zero contributor each]
 *   pps_rank_count_local  -> all-reduce(SUM) of *d_counters [*n_counters = nq + n_pairs uint32]
 *   pps_rank_end          finalize, results to the host (top-k here is the LOCAL block's; sharded top-k
 *                         is merged by the Python layer).
 * With world == 1 (d_cnt_all = NULL) there is nothing to exchange.  The returned device pointers belong
 * to the ctx and stay valid until the next pps_rank_begin. */
int pps_rank_begin(pps_ctx* ctx, const float* d_q, long long nq, const float* d_g, long long ng_local, int dim,
                   const int64_t* d_query_ids, const int64_t* d_query_cams,
                   const int64_t* d_gallery_ids, const int64_t* d_gallery_cams,
                   long long gallery_offset, int world, int precision, int topk, void* stream,
                   void* pair_stream /* optional: the pair-list kernels run here (and the caller's all-gather
                                        should too), overlapping the split + GEMM on `stream`; NULL = ctx policy */,
                   int32_t** d_local_cnt);
int pps_rank_thresholds(pps_ctx* ctx, const int32_t* d_cnt_all, int rank, void* stream,
                      long long* n_pairs, int32_t** d_exchange, long long* n_words);
int pps_rank_count_local(pps_ctx* ctx, void* stream, uint32_t** d_counters, long long* n_counters);
int pps_rank_end(pps_ctx* ctx, int cmc_topk, void* stream, double* out_map, double* out_cmc,
                 double* out_ap, uint8_t* out_valid, int32_t* out_first_rank,
                 int32_t* out_topk_index, float* out_topk_dist);

/* ------------------------------------------------------------------------------------
 * Part 2g — one ranking pass over a gallery of ANY size, optionally sharded over several GPUs (BASELINE configs[3] /
 *           configs[4]; replaces the reference's multi-GPU test path detectron/utils/subprocess.py:39-103 +
 *           core/test_engine.py:205-213, which shards images over processes and pickles results).
 *
 * d_q [nq, dim] and d_g [ng_local, dim] are contiguous device rows (dtype PPS_DTYPE_F32 or _F16); d_g is this
 * rank's block of the gallery starting at global row gallery_offset.  d_gid / d_gcam are the GLOBAL id / camera vectors
 * [ng_global] (replicated, like the queries): every rank builds the same pair lists from them (hash pre-filter of
 * the rows that can match + brute-force sweeps), so no pair metadata is exchanged.  The local rows are processed in
 * distance blocks of at most max_block_bytes (nq x rows x 4); with topk > 0 the first block is kept short and later
 * blocks take their top-k candidates in the distance epilogue.
 *   pps_pass_begin   -> *d_x1 [*n_x1 int32 words]: the thresholds (float bits; pairs of other shards are 0).
 *                       Sharded: all-gather it into d_gathered_x1 [world][*n_x1] (an all-gather of these 0.35 MB is 3x
 *                       faster than NCCL's all-reduce at 8 ranks; pps_pass_count sums the copies itself - exact, every pair
 *                       has one non-zero contributor).
 *   pps_pass_count   (d_gathered_x1 = NULL when world == 1) -> *d_x2 [*x2_bytes]: [top-k keys | counters | flags] of this
 *                       rank.  Sharded: all-gather it into d_gathered [world][*x2_bytes].
 *   pps_pass_end     reduces / merges the gathered buffers (own kernels), finalises, copies the results to the host
 *                    like pps_rank_end; d_gathered = NULL when world == 1.
 * Two collectives per pass, identical on every rank whatever its shard looks like (also an empty one).  The pair-list
 * kernels run on a stream of the ctx, everything else on `stream`; pps_pass_begin blocks the host only on 4-byte
 * read-backs that arrive while the first distance block is running.  Phase timing (pps_ctx_set_timing) reports the
 * SUMS over the pass: split, dist_gemm, rank_count (sweeps + merges), finalize. */
#define PPS_PASS_SIZING 2             /* flags: read the list sizes back (a "sizing" pass).  Without it a pass whose shape
                                         was sized before is SPECULATIVE: the earlier sizes serve as upper bounds, the kernels
                                         read the actual counts on the device and the host never waits mid-pass;
                                         pps_pass_end returns PPS_ERR_PASS_RESIZE when a bound was too small (different ids) */
#define PPS_PASS_NO_EPILOGUE_TOPK 1   /* flags: every block takes the one-read sweep (the fallback after TOPK_OVERFLOW) */
#define PPS_PASS_NO_FUSED_COUNT 4     /* flags: blocks after the first are written and counted by pps_rank_count even where the
                                         counting epilogue (pps_dist_rank_topk_tc) applies (A/B measurements, tests) */
#define PPS_PASS_TKCAP(n) (((n) & 0xffff) << 8)   /* flags: candidate-buffer entries per query (default / maximum 2048) */
int pps_pass_begin(pps_ctx* ctx, const void* d_q, long long nq, const void* d_g, long long ng_local, int dim, int dtype,
                   const int64_t* d_query_ids, const int64_t* d_query_cams,
                   const int64_t* d_gallery_ids, const int64_t* d_gallery_cams, long long ng_global,
                   long long gallery_offset, int world, int rank, int precision, int topk,
                   long long max_block_bytes, int flags, void* stream,
                   int32_t** d_x1, long long* n_x1);
/* Host sources of the NEXT pps_pass_begin only: its d_q / d_g arguments are then device STAGING buffers the call fills
 * from these host rows (pinned for full PCIe bandwidth) - the queries on `stream`, the gallery on a copy stream of the
 * ctx block by block, or in ~8 row slabs when the shard is one block, so that the split + distance of what has arrived
 * overlap the rest of the upload (the multi-GPU form of pps_evaluate_host_ctx).  NULL leaves a buffer as it is. */
int pps_pass_set_host_input(pps_ctx* ctx, const void* h_q, const void* h_g);
/* What the last pps_pass_begin of this context decided: which = 0 number of blocks of the local shard, 1 whether the blocks
 * after the first take the counting epilogue (pps_dist_rank_topk_tc: nothing written), 2 whether the layout is speculative,
 * 3 thresholds per query in the epilogue tables, 4 whether top-k candidates are admitted in the distance epilogue. */
long long pps_pass_stat(const pps_ctx* ctx, int which);
int pps_pass_count(pps_ctx* ctx, const void* d_gathered_x1, void* stream, void** d_x2, long long* x2_bytes);
int pps_pass_end(pps_ctx* ctx, const void* d_gathered, int cmc_topk, void* stream, double* out_map, double* out_cmc,
                 double* out_ap, uint8_t* out_valid, int32_t* out_first_rank,
                 int32_t* out_topk_index, float* out_topk_dist);

/* Phase timing of pps_evaluate_device_ctx: when enabled, CUDA events are recorded on the caller's
 * stream between the phases and pps_ctx_phase_ms returns the device time of each phase of the
 * LAST call: 0 hand-off of the pair-list kernels to the side stream (they overlap the GEMM),
 * 1 operand split, 2 distance GEMM, 3 wait for the pair lists + threshold gather,
 * 4 counting sweep, 5 finalize (+top-k), 6 result copies. */
#define PPS_N_PHASES 7
int pps_ctx_set_timing(pps_ctx* ctx, int enabled);
int pps_ctx_phase_ms(const pps_ctx* ctx, float* out_ms /* [PPS_N_PHASES] */);
int pps_evaluate_host(const float* q_feats, long long nq,
                      const float* g_feats, long long ng, int dim,
                      const int64_t* query_ids, const int64_t* query_cams,
                      const int64_t* gallery_ids, const int64_t* gallery_cams,
                      int precision, int cmc_topk, int topk, int device,
                      double* out_map, double* out_cmc,
                      double* out_ap, uint8_t* out_valid, int32_t* out_first_rank,
                      int32_t* out_topk_index, float* out_topk_dist);

/* ------------------------------------------------------------------------------------
 * Part 2h — resident gallery index: the k nearest gallery rows of unlabelled queries (person retrieval).
 *
 * The Euclidean top-k of pps_dist_tc's distances, smallest first, ties by gallery index (what rank_eval's top-k gives
 * when no gallery item shares a query's id).  Optional exclusion by tag: one int64 tag per gallery row and one exclude
 * tag per query; row r is left out of query q's result if and only if tag[r] == exclude_tag[q].  Two encodings:
 *   cross-camera search         tag = camera of the row, exclude tag = camera of the query
 *   the evaluation's junk rule  tag = (id << 32) | camera (ids in int32, cameras in [0, 2^32)): the result equals
 *                               rank_eval's top-k (same id and camera left out) bit for bit
 *
 * pps_search_topk_tc   top-k admission with the roles of pps_dist_topk_tc swapped: the gallery rows [ng] are the
 *                      256-row M operand and the queries [nq] the N operand (N = 32, 64, 128 or 256, the smallest that
 *                      holds the batch; larger batches take query tiles of 256), so that a small batch streams the
 *                      gallery once instead of occupying a few rows of every MMA.  Same operands and arithmetic as
 *                      pps_dist_tc (its distances, bit for bit).  Every distance whose bits are <= tk_bound[q] is
 *                      appended as (bits << 32 | col0 + row) to tk_cand[q][tk_cap] through tk_cnt[q] (which counts
 *                      past tk_cap; pps_topk_merge detects it) - the layout pps_topk_merge consumes.  Nothing else is
 *                      written.  flags: 0, PPS_DIST_SQUARED, PPS_DIST_SQRT_RN.
 * pps_search_topk_excl_tc   the same without the pairs whose tags are equal: g_tags[ng] (row r of this block: the tag
 *                      of row col0 + r is g_tags[r]) and q_tags[nq], both required.  The tags are compared only for
 *                      elements within the bound; an excluded element takes no slot.
 * pps_topk_update_excl pps_topk_update without the columns c with g_tags[c] == q_tags[q] (g_tags[ncols]: column c's
 *                      tag, q_tags[nq]).  n_excluded (may be null): n_excluded[q] = the number of such columns in this
 *                      call (every column's tag is read then; otherwise only those of admitted columns).
 * pps_index_*          a gallery kept on one device as split operand planes [planes][capacity][kpad] plus the norm
 *                      array (PPS_PREC_F16X3: capacity norms, then capacity inverse scales - the pps_split_rows_slab
 *                      layout).  pps_index_add appends n rows (device pointer, row stride ld elements) of the index's
 *                      dtype; the capacity doubles when exceeded.  dtype PPS_DTYPE_F16 uses PPS_PREC_F16X1; dtype
 *                      PPS_DTYPE_F32 takes PPS_PREC_F16X3 or PPS_PREC_BF16X1/3/6 (PPS_PREC_FP32: PPS_ERR_UNSUPPORTED).
 *                      pps_index_add_tagged appends rows with their tags d_tags[n] (device).  The first non-empty add
 *                      decides whether the index is tagged; a later add of the other kind is PPS_ERR_INVALID_ARG.
 * pps_index_search     d_keys[nq][k] = the k nearest rows of the queries d_q [nq, dim] (the index's dtype, row stride
 *                      ldq) as top-k keys whose gallery index is index_offset + row (a shard passes its first global
 *                      row); pps_topk_unpack turns them into distances / int32 indices (-1 / inf past the index's
 *                      size).  index_offset + size must stay below 2^31 (PPS_ERR_UNSUPPORTED otherwise).  The first
 *                      min(size, 32768) rows are a materialised block swept by pps_topk_update; the rest is covered by
 *                      pps_search_topk_tc + pps_topk_merge in chunks that grow with the rows already seen.  The call
 *                      reads back one 4-byte overflow flag (its only synchronisation); when a candidate buffer ran over
 *                      the search is repeated with materialised blocks only.  Scratch is owned by the index and only
 *                      grows.  flags: 0, or test hooks PPS_INDEX_TKCAP(n) (candidate entries per query, <= 2048) and
 *                      PPS_INDEX_PREFIX(n) (n * 256 rows in the materialised prefix, n <= 127).  On a tagged index
 *                      it ignores the tags.
 * pps_index_search_excluding   pps_index_search without the rows whose tag equals the query's d_q_tags[q] (device,
 *                      [nq], required); PPS_ERR_INVALID_ARG on a non-empty untagged index.  Fewer than k remaining rows:
 *                      padded with -1 / inf.  Same schedule with the excluding kernels; when the gallery is larger than
 *                      the prefix, the prefix sweep counts every query's excluded rows and one more 4-byte read-back
 *                      (the largest count) shrinks the chunks by the excluded share (at most 0.9).
 * pps_index_remove     deletes the local rows d_rows[n] (device int64, any order, duplicates allowed) with np.delete's
 *                      renumbering: every later row moves down by the number of removed rows before it, and the size
 *                      shrinks by the number of distinct rows removed (*n_removed, host, may be null).  The index is then
 *                      the index a fresh pps_index_create + add of the remaining rows in their order (with their tags)
 *                      gives, so every later search returns that index's answer bit for bit.  A row < 0 or >= size:
 *                      PPS_ERR_INVALID_ARG and the index is unchanged.  n = 0 does nothing.  The capacity is not reduced;
 *                      an index emptied by removal decides again at its next non-empty add whether it is tagged.  The
 *                      rows are compacted on the device: one byte per row marks the removed rows, a scan lists the
 *                      live rows after the first removed one, and these move down in pieces through an index-owned
 *                      buffer of at most 256 MiB (about 5 bytes of scratch per row besides it).  d_rows has been read
 *                      when the call returns: one 24-byte read-back is its only synchronisation, the moves stay queued
 *                      on `stream`.  flags: 0, or the test hook PPS_INDEX_PIECE(n) (at most n rows per piece).  Sharded:
 *                      removal is local (a rank removes its own rows); the next search's all-gather of the shard sizes
 *                      moves the global offsets.
 * pps_search_range_tc  the range form of pps_search_topk_tc (same kernel up to the admission and the address): every
 *                      distance whose bits are < lim[q] is appended as (bits << 32 | col0 + row) to
 *                      out[out_off[q] + slot] when slot < out_cap[q]; cnt[q] counts every hit, also past the capacity.
 *                      g_tags / q_tags: both null, or both set (the pairs whose tags are equal are no hits).  The limit
 *                      of a radius r is bits(r) + 1 for r >= 0 (-0 as 0; +inf: 0x7f800001) and 0 for a negative or NaN r:
 *                      then bits < lim <=> d <= r, distances being >= 0 and never NaN.
 * pps_index_range_search   every row within a radius of each query: row r is a result of query q when d(q, r) <=
 *                      d_radius[q] (device float32 [nq]; IEEE comparison: a negative or NaN radius selects nothing, +inf
 *                      every row), d being pps_index_search's distance, bit for bit.  d_q_tags (device [nq], may be null):
 *                      also leave out the rows whose tag equals the query's, as pps_index_search_excluding (a non-empty
 *                      untagged index: PPS_ERR_INVALID_ARG).  Output in FAISS's range_search layout: d_lims (caller memory,
 *                      device int64 [nq + 1]) and *total (host) = d_lims[nq]; query q's results are keys
 *                      [d_lims[q], d_lims[q + 1]) in (distance, index) order, the order of top-k keys, with gallery index
 *                      index_offset + row.  The keys stay in index-owned scratch: pps_index_range_keys copies them out.
 *                      One pass of pps_search_range_tc over every row writes uniform slices of C keys per query (C: 4 096
 *                      at first, then the power of two at or above the largest count of an earlier call, at most 1 GiB of
 *                      slices); a scan of the counts and one 16-byte read-back {total, largest count} follow, the call's
 *                      only synchronisation when no slice ran over.  Otherwise a second pass writes the keys straight into
 *                      the result layout.  pps_sort_key_segments' stages then compact and sort.  A result that does not
 *                      fit in memory: PPS_ERR_CUDA, the index unchanged and usable.  flags: 0, or the test hook
 *                      PPS_INDEX_TKCAP(n) (C = n).  An empty index or nq = 0: d_lims all zero.
 * pps_index_range_keys copies the last range search's *total keys to d_keys (device); valid until the next call on the
 *                      index.  pps_topk_unpack(keys, total, 1, ...) splits them into distances and int32 indices.
 * pps_sort_key_segments    sorts every segment [lims[s], lims[s + 1]) of keys ascending, in place (lims: device int64
 *                      [nseg + 1], ascending; scratch: device, lims[nseg] - lims[0] keys, may be null when that is at most
 *                      4 096).  Reads lims[0] and lims[nseg] back (16 bytes, a synchronisation).  Keys are sorted in tiles
 *                      of 4 096 in shared memory, then by ceil(log2(total / 4096)) merge passes; segments may hold from 0
 *                      keys to all of them.  Equal keys are allowed; keys that are unique in their segment (range search:
 *                      the row index is in the low bits) give one result whatever order they came in.
 * Grouped search: every row may carry one int64 group (a tracklet, an identity), and a grouped search returns the nearest
 * row of each of the k nearest groups.  Order the rows a search (plain or excluding) admits by their key; keep the first
 * row of each group; return the first k.  Every row its own group: the search's keys, bit for bit.
 * pps_index_add_grouped   pps_index_add with d_groups[n] (device int64, required) and d_tags[n] (device, may be null).
 *                      The first non-empty add decides whether the index is grouped (and whether tagged); a later add
 *                      of the other kind is PPS_ERR_INVALID_ARG.
 * pps_index_search_groups   d_keys[nq][k] = the keys of each query's k nearest groups' nearest rows, d_groups[nq][k] their
 *                      groups; past the last group ~0 / -1.  d_q_tags (may be null): leave out rows as
 *                      pps_index_search_excluding.  A non-empty ungrouped index: PPS_ERR_INVALID_ARG.  Schedule: materialised
 *                      blocks swept by pps_topk_group_update until every query holds k groups (a 4-byte read-back per
 *                      block), one counting pass of pps_search_range_tc over those rows (L = the most rows of a query at
 *                      or below its bound, a 4-byte read-back), then chunks of pps_search_topk(_excl)_tc +
 *                      pps_topk_group_merge sized cap * rows done / (2.2 max(k, L)), cap = 8 192 candidates per query;
 *                      the overflow read-back; on overflow materialised blocks only.  flags: as pps_index_search
 *                      (PPS_INDEX_TKCAP(n) up to 8 192).
 * pps_index_group_stats    the schedule of the index's last grouped search: rows swept as materialised blocks before
 *                      the chunks, chunks, and whether the materialised fallback ran (host pointers, each may be null).
 * pps_topk_group_update    grouped counterpart of pps_topk_update: dist [nq][ldd] columns c < ncols (gallery index col0 + c,
 *                      group g_groups[c]) into the grouped state topk_key / topk_group [nq][k] (initialised to ~0 / -1).
 *                      g_tags / q_tags: both null, or both set (columns with g_tags[c] == q_tags[q] are left out).
 * pps_topk_group_merge     grouped counterpart of pps_topk_merge: candidates tk_cand[q][tk_cap] of pps_search_topk_tc
 *                      (tk_cnt[q] of them) with groups g_groups[index - index_offset] into the state; new tk_bound
 *                      (the k-th key's distance bits, all ones while fewer than k groups are held), tk_cnt = 0,
 *                      *overflow = 1 if a buffer ran over.
 * pps_topk_group_merge_lists   the grouped state of `lists` states keys / groups [lists][nq][k] (disjoint row sets, e.g.
 *                      the shards of a gallery; a group may span lists) -> out_key / out_group [nq][k].
 * Calls on one index are ordered by the caller (one stream, or events between streams); every call sets the index's
 * device for its duration.  A sharded gallery: one index per rank, index_offset = the rows of the ranks before, an
 * all-gather of the [nq][k] keys and the k smallest per query (every rank's list is sorted, keys are unique).
 * ---------------------------------------------------------------------------------- */
#define PPS_INDEX_TKCAP(n)  (((n) & 0xffff) << 8)
#define PPS_INDEX_PREFIX(n) (((n) & 0x7f) << 24)
#define PPS_INDEX_PIECE(n)  (((n) & 0xffff) << 8)   /* pps_index_remove only */
int pps_search_topk_tc(const void* g_planes, const float* g_sqnorm, long long ng, int g_planes_n, long long g_plane_rows,
                       const void* q_planes, const float* q_sqnorm, long long nq, int q_planes_n, long long q_plane_rows,
                       int dim, int precision, int flags, long long col0, const uint32_t* tk_bound, uint32_t* tk_cnt,
                       uint64_t* tk_cand, int tk_cap, void* stream);
int pps_search_topk_excl_tc(const void* g_planes, const float* g_sqnorm, long long ng, int g_planes_n,
                            long long g_plane_rows, const void* q_planes, const float* q_sqnorm, long long nq,
                            int q_planes_n, long long q_plane_rows, int dim, int precision, int flags, long long col0,
                            const uint32_t* tk_bound, uint32_t* tk_cnt, uint64_t* tk_cand, int tk_cap, void* stream,
                            const int64_t* g_tags, const int64_t* q_tags);
int pps_topk_update_excl(const float* dist, long long ldd, long long nq, long long ncols, long long col0,
                         const int64_t* g_tags, const int64_t* q_tags, uint64_t* topk_key, int k,
                         uint32_t* n_excluded, void* stream);
typedef struct pps_index pps_index;
int       pps_index_create(int device, int dim, int dtype, int precision, pps_index** out);
int       pps_index_destroy(pps_index* idx);
int       pps_index_add(pps_index* idx, const void* d_rows, long long n, long long ld, void* stream);
int       pps_index_add_tagged(pps_index* idx, const void* d_rows, long long n, long long ld, const int64_t* d_tags,
                               void* stream);
long long pps_index_size(const pps_index* idx);
int       pps_index_search(pps_index* idx, const void* d_q, long long nq, long long ldq, int k,
                           long long index_offset, int flags, void* stream, uint64_t* d_keys);
int       pps_index_search_excluding(pps_index* idx, const void* d_q, long long nq, long long ldq,
                                     const int64_t* d_q_tags, int k, long long index_offset, int flags, void* stream,
                                     uint64_t* d_keys);
int       pps_index_remove(pps_index* idx, const int64_t* d_rows, long long n, int flags, void* stream,
                           long long* n_removed);
int pps_search_range_tc(const void* g_planes, const float* g_sqnorm, long long ng, int g_planes_n, long long g_plane_rows,
                        const void* q_planes, const float* q_sqnorm, long long nq, int q_planes_n, long long q_plane_rows,
                        int dim, int precision, int flags, long long col0, const uint32_t* lim, uint32_t* cnt,
                        const long long* out_off, const uint32_t* out_cap, uint64_t* out, const int64_t* g_tags,
                        const int64_t* q_tags, void* stream);
int       pps_index_range_search(pps_index* idx, const void* d_q, long long nq, long long ldq, const float* d_radius,
                                 const int64_t* d_q_tags /*nullable*/, long long index_offset, int flags, void* stream,
                                 int64_t* d_lims, long long* total);
int       pps_index_range_keys(pps_index* idx, uint64_t* d_keys, void* stream);
int       pps_sort_key_segments(uint64_t* keys, const int64_t* lims, long long nseg, uint64_t* scratch, void* stream);
int       pps_index_add_grouped(pps_index* idx, const void* d_rows, long long n, long long ld, const int64_t* d_tags,
                                const int64_t* d_groups, void* stream);
int       pps_index_search_groups(pps_index* idx, const void* d_q, long long nq, long long ldq,
                                  const int64_t* d_q_tags /*nullable*/, int k, long long index_offset, int flags, void* stream,
                                  uint64_t* d_keys, int64_t* d_groups);
int       pps_index_group_stats(const pps_index* idx, long long* prefix_rows, long long* chunks, int* fallback);
int pps_topk_group_update(const float* dist, long long ldd, long long nq, long long ncols, long long col0,
                          const int64_t* g_groups, const int64_t* g_tags, const int64_t* q_tags, uint64_t* topk_key,
                          int64_t* topk_group, int k, void* stream);
int pps_topk_group_merge(uint64_t* topk_key, int64_t* topk_group, long long nq, int k, const uint64_t* tk_cand, int tk_cap,
                         uint32_t* tk_cnt, uint32_t* tk_bound, const int64_t* g_groups, long long index_offset,
                         int32_t* overflow, void* stream);
int pps_topk_group_merge_lists(const uint64_t* keys, const int64_t* groups, int lists, long long nq, int k,
                               uint64_t* out_key, int64_t* out_group, void* stream);

/* ------------------------------------------------------------------------------------
 * Next row (SURVEY §8f.4) — the reference's training-side triplet mining ops.
 *   PairWiseDistance[Gradient]   detectron/ops/pairwise_distance_op.cu:9-22, :78-91
 *       z[p,q] = sum_d (x[p,d]-x[q,d])^2  (squared, no sqrt);  dx = 2 sum_q (x_n - x_q)(dz[n,q] + dz[q,n])
 *   BatchHard[Gradient]          detectron/ops/batch_hard_op.cc:9-59, :62-123
 *       ap[a] = max_{label==} xdist[a,:] (init 0), an[a] = min_{label!=} xdist[a,:] (init FLT_MAX);
 *       idx_p / idx_n (optional on forward) = the first index reaching them, -1 if none;
 *       backward scatters dap / dan to those indices of a zeroed [N, N] (rows with idx -1 get nothing:
 *       the reference writes out of the row there).
 *   pps_batch_hard_fused_fwd mines straight from the features, no [N, N] matrix.
 * ---------------------------------------------------------------------------------- */
int pps_pairwise_distance_fwd(const float* x, int N, int D, float* z, void* stream);
int pps_pairwise_distance_bwd(const float* x, const float* dz, int N, int D, float* dx, void* stream);
int pps_batch_hard_fwd(const float* xdist, const int32_t* labels, int N, float* ap, float* an,
                       int32_t* idx_p, int32_t* idx_n, void* stream);
int pps_batch_hard_fused_fwd(const float* x, const int32_t* labels, int N, int D, float* ap, float* an,
                             int32_t* idx_p, int32_t* idx_n, void* stream);
int pps_batch_hard_bwd(const int32_t* idx_p, const int32_t* idx_n, const float* dap, const float* dan, int N,
                       float* dx, void* stream);

/* ------------------------------------------------------------------------------------
 * Next row (SURVEY §8f.1) — the per-combination embedding between pooling and distance
 * (detectron/modeling/reid_heads.py:34-76 at test time, one branch per pooled blob):
 *   Conv1x1(C -> E, bias) -> SpatialBN(is_test: an affine map) -> ReLU, then Concat(axis=1) of the K
 *   branches (:95-101) and, with REID.NORMALIZE_FEATURE, Normalize(axis=1) (:123-127, triplet_loss.py:18).
 * pps_embed_tc: out[n, k*E + e] = max(0, alpha[k*E+e] * sum_c x[k, n, c] * w[k, e, c] + beta[k*E+e]);
 *   the caller folds the conv bias and the BN statistics into alpha / beta:
 *   alpha = bn_scale / sqrt(bn_var + eps), beta = (conv_bias - bn_mean) * alpha + bn_bias.
 *   x_planes : pps_split_rows of the pooled features laid out [K*N, C] (the [K, N, C] pooling output);
 *   w_planes : pps_split_rows of the weights laid out [K*E, C].  One grouped launch of the 2-CTA tcgen05
 *   kernel (256 x 128 tiles), same split precisions as pps_dist_tc.  E must be 128 (REID.BPM_DIM of
 *   every shipped PPS config) for now: PPS_ERR_UNSUPPORTED otherwise.
 * pps_l2_normalize_rows: x[r, :] /= max(|x[r, :]|_2, 1e-12)   (Caffe2 Normalize, kEps = 1e-12), in place
 *   when out == x.
 * ---------------------------------------------------------------------------------- */
int pps_embed_tc(const void* x_planes, int x_planes_n, long long N,
                 const void* w_planes, int w_planes_n, int E, int K, int C,
                 const float* alpha, const float* beta, int precision,
                 float* out, long long ldo, void* stream);
int pps_l2_normalize_rows(const float* x, long long rows, int dim, long long ld,
                          float* out, long long ldo, void* stream);

/* Multi-query pooling (SURVEY §8f.3; reid_dataset_evaluator.py:131-143): out[g] = np.mean(feats[row_idx[group_off[g] :
 * group_off[g+1]]], axis=0) - a float32 sum of the listed rows in order, then one division by their count. */
int pps_group_mean_rows(const float* feats, long long ld, int dim, const int32_t* group_off, const int32_t* row_idx,
                        long long n_groups, float* out, long long ldo, void* stream);

/* ------------------------------------------------------------------------------------
 * Next row (SURVEY §8f.2) — k-reciprocal re-ranking, reid_dataset_evaluator.py:442-519
 * `re_ranking(q_g_dist, q_q_dist, g_g_dist, k1=20, k2=6, lambda_value=0.3)` (evaluate() :161-207;
 * cfg.REID.RERANK defaults to True, config.py:1022).  M is the assembled [n, n] matrix
 * [[q_q, q_g], [q_g^T, g_g]] (n = nq + ng), images 0 .. nq-1 are the queries.  Steps, each one call:
 *   pps_rerank_normalize  od[i][j] = M[j][i]^2 / max_r M[r][i]^2                       (:447-454)
 *   initial_rank          = the k1 + 1 nearest columns of every row of od: pps_topk_init / pps_topk_update
 *                           (no exclusion list) / pps_topk_unpack on od                 (:456)
 *   pps_rerank_krecip     k-reciprocal set + expansion, V row = exp(-od) normalised     (:462-487)
 *                         rows as ELL: v_idx / v_val [n][pps_rerank_vcap()], v_cnt [n]
 *   pps_rerank_expand     V row <- mean of the V rows of the k2 nearest images          (:489-494)
 *                         q_idx / q_val [n][qe_cap], qe_cap >= k2 * pps_rerank_vcap()
 *   pps_rerank_invert     inverted index (by column) of the gallery rows                (:496-498)
 *   pps_rerank_jaccard    out[i][g] = (1 - t/(2 - t)) (1 - lambda) + od[i][nq + g] lambda,
 *                         t = sum_c min(V[i][c], V[nq + g][c])                          (:500-513)
 * All arithmetic is float32 in the reference's order (columns ascending, no atomics on floats).
 * ---------------------------------------------------------------------------------- */
int pps_rerank_vcap(void);
int pps_rerank_normalize(const float* m, long long ld, long long n, float* colmax, float* od, long long ldo,
                         void* stream);
int pps_rerank_krecip(const int32_t* initial_rank, int rank_cols, long long n, int k1,
                      const float* od, long long ldo, int32_t* v_idx, float* v_val, int32_t* v_cnt, void* stream);
int pps_rerank_expand(const int32_t* initial_rank, int rank_cols, long long n, int k2,
                      const int32_t* v_idx, const float* v_val, const int32_t* v_cnt,
                      int qe_cap, int32_t* q_idx, float* q_val, int32_t* q_cnt, void* stream);
int pps_rerank_invert(const int32_t* q_idx, const float* q_val, const int32_t* q_cnt, int qe_cap,
                      long long nq, long long n, int32_t* col_cnt, int32_t* col_off, int32_t* cursor,
                      int32_t* inv_row, float* inv_val, void* stream);
int pps_rerank_jaccard(const int32_t* q_idx, const float* q_val, const int32_t* q_cnt, int qe_cap,
                       const int32_t* col_off, const int32_t* inv_row, const float* inv_val,
                       long long nq, long long ng, const float* od, long long ldo, float lambda_value,
                       float* out, long long ld_out, void* stream);

/* instrumentation: number of kernels this library has launched in this process
 * (bench.py reports the delta over the timed region as `gpu_launches`). */
unsigned long long pps_kernel_launch_count(void);
#ifdef __cplusplus
}
#endif
#endif /* PPS_B200_H_ */
