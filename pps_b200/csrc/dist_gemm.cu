// Query x gallery Euclidean distance (reid_dataset_evaluator.py:244-272) on the 5th-gen
// tensor cores: the one dense contraction of the path, a . b^T, as TMA-fed tcgen05.mma tiles
// with fp32 accumulators in TMEM; the epilogue fuses |a|^2 + |b|^2 - 2ab, the clamp at 0 and
// the sqrt (reid_dataset_evaluator.py:269-271) and writes the [m1, m2] fp32 block.
//
// fp32-accurate path: both operands arrive as bf16 residual planes (split_prep.cu). The
// product is the sum of plane-pair terms (p0.p0 + p0.p1 + p1.p0 for BF16X3), all accumulated
// into the same TMEM tile, smallest terms first — i.e. one GEMM whose K loop walks
// (term, k-block) pairs.  Both operands are K-major, so A and B tiles are plain TMA boxes of
// 64 bf16 (128 B, SWIZZLE_128B) x {128, 256} rows and feed UMMA without any transpose.
//
// Kernel shape: persistent, one CTA per SM, 128 x 256 output tile, BK = 64.
//   warp 0   : TMA producer (4-stage ring, 48 KB per stage)
//   warp 1   : TMEM allocator + single-thread tcgen05.mma issuer (4 x K=16 per stage)
//   warps 2-5: epilogue, 128 threads = 128 TMEM lanes (rows); double-buffered accumulators
//              (2 x 256 TMEM columns) so the epilogue of tile t overlaps the mainloop of t+1.
#include "common.cuh"
#include "dist_tiles.cuh"

#include <cstdlib>
#include <mutex>

namespace pps {

constexpr int kBM = 128;
constexpr int kBN = 256;
constexpr int kBK = 64;                              // bf16 elements = 128 bytes = one swizzle row
constexpr int kGemmStages = 4;
constexpr int kABytes = kBM * kBK * 2;               // 16 KB
constexpr int kBBytes = kBN * kBK * 2;               // 32 KB
constexpr int kStageBytesG = kABytes + kBBytes;      // 48 KB
constexpr int kGemmThreads = 192;
// the counting epilogue runs on EIGHT epilogue warps: two per TMEM lane group, each taking one 128-column half of the tile.
// With one warp per scheduler every dependent instruction of its ~30-instruction-per-element search cost its full latency
// and the epilogue (46 k cycles per tile) stuck out from under the single-plane mainloop (35 k).
constexpr int kRankThreads = 64 + 8 * 32;
template <int EPI> constexpr int gemm2_threads() { return EPI == EPI_RANK ? kRankThreads : kGemmThreads; }
constexpr size_t kGemmSmem = 1024 /*align slack*/ + (size_t)kGemmStages * kStageBytesG + 256 /*barriers*/;

__global__ void __launch_bounds__(kGemmThreads, 1)
dist_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ GemmArgs g) {
  extern __shared__ unsigned char smem_dyn[];
  // SWIZZLE_128B tiles need 1024-byte alignment
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~uintptr_t(1023));
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + (size_t)kGemmStages * kStageBytesG);
  uint64_t* empty = full + kGemmStages;
  uint64_t* tfull = empty + kGemmStages;     // [2] accumulator ready for the epilogue
  uint64_t* tempty = tfull + 2;              // [2] accumulator drained
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long tiles = (long long)g.m_tiles * g.n_tiles;
  const int kiters = g.nterms * g.kblocks;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int s = 0; s < kGemmStages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tfull[s], 1);
      mbar_init(&tempty[s], 4);   // one arrive per epilogue warp
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, 2 * kBN);   // 512 columns: two 128x256 fp32 accumulators
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      uint32_t it = 0;
      for (long long t = blockIdx.x; t < tiles; t += gridDim.x) {
        const int m0 = (int)(t % g.m_tiles) * kBM;     // m fastest: concurrent CTAs share B tiles in L2
        const int n0 = (int)(t / g.m_tiles) * kBN;
        for (int term = 0; term < g.nterms; ++term) {
          const int pa = g.term_a[term], pb = g.term_b[term];
          for (int kb = 0; kb < g.kblocks; ++kb, ++it) {
            const uint32_t s = it % kGemmStages, ph = (it / kGemmStages) & 1u;
            mbar_wait(&empty[s], ph ^ 1u);
            mbar_expect_tx(&full[s], kStageBytesG);
            unsigned char* sa = smem + (size_t)s * kStageBytesG;
            tma_load_3d(sa, &tmA, &full[s], kb * kBK, m0, pa);
            tma_load_3d(sa + kABytes, &tmB, &full[s], kb * kBK, n0, pb);
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (one thread) =====================
    if (lane == 0) {
      uint32_t it = 0, acc_it = 0;
      for (long long t = blockIdx.x; t < tiles; t += gridDim.x, ++acc_it) {
        const uint32_t as = acc_it & 1u, aph = (acc_it >> 1) & 1u;
        mbar_wait(&tempty[as], aph ^ 1u);      // epilogue has drained this accumulator
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * kBN;
        for (int ki = 0; ki < kiters; ++ki, ++it) {
          const uint32_t s = it % kGemmStages, ph = (it / kGemmStages) & 1u;
          mbar_wait(&full[s], ph);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + (size_t)s * kStageBytesG);
          const uint64_t adesc = umma_desc_k_sw128(sa);
          const uint64_t bdesc = umma_desc_k_sw128(sa + kABytes);
#pragma unroll
          for (int k = 0; k < kBK / 16; ++k) {
            // advance 16 elements = 32 bytes along K inside the swizzle row: +2 in the >>4 address field
            tc_mma_f16(d_tmem, adesc + 2u * k, bdesc + 2u * k, g.idesc, (ki | k) ? 1u : 0u);
          }
          tc_commit(&empty[s]);                 // smem slot reusable once these MMAs retire
        }
        tc_commit(&tfull[as]);                  // accumulator complete
      }
    }
  } else {
    // ===================== epilogue (warps 2..5) =====================
    const int lane_grp = warp & 3;              // TMEM lanes 32*lane_grp .. +31 are this warp's
    const int row = lane_grp * 32 + lane;
    uint32_t acc_it = 0;
    const bool want_sq = (g.flags & PPS_DIST_SQUARED) != 0;
    const bool want_dot = (g.flags & PPS_DIST_DOT) != 0;
    const bool vec_ok = ((g.ldo & 3) == 0) && ((reinterpret_cast<uintptr_t>(g.out) & 15u) == 0);
    for (long long t = blockIdx.x; t < tiles; t += gridDim.x, ++acc_it) {
      const int m0 = (int)(t % g.m_tiles) * kBM;
      const int n0 = (int)(t / g.m_tiles) * kBN;
      const uint32_t as = acc_it & 1u, aph = (acc_it >> 1) & 1u;
      mbar_wait(&tfull[as], aph);
      tc_fence_after();
      const long long gi = (long long)m0 + row;
      const bool row_ok = gi < g.m1;
      const float an = (row_ok && !want_dot) ? __ldg(g.a_sqnorm + gi) : 0.f;
      const bool scaled = g.a_scale != nullptr;
      const float cs = (scaled && row_ok) ? -2.f * __ldg(g.a_scale + gi) : -2.f;
      float* orow = g.out + (row_ok ? gi : 0) * g.ldo;
      const uint32_t tbase = tmem_base + as * kBN + ((uint32_t)(lane_grp * 32) << 16);
#pragma unroll 1
      for (int c = 0; c < kBN; c += 32) {
        uint32_t r[32];
        tmem_ld_32x32(tbase + c, r);
        tmem_ld_wait();
        const long long gj0 = (long long)n0 + c;
        if (row_ok && gj0 < g.m2) {
          float v[32];
#pragma unroll
          for (int e = 0; e < 32; ++e) {
            const float dot = __uint_as_float(r[e]);
            const long long gj = gj0 + e;
            const float sc = (scaled && gj < g.m2) ? cs * __ldg(g.b_scale + gj) : cs;   // -2 / (s_a s_b): exact
            if (want_dot) {
              v[e] = scaled ? dot * (-0.5f * sc) : dot;
            } else {
              const float bn = gj < g.m2 ? __ldg(g.b_sqnorm + gj) : 0.f;
              // same association as the reference: (-2*ab + |a|^2) + |b|^2
              float d2 = __fadd_rn(__fadd_rn(__fmul_rn(sc, dot), an), bn);
              d2 = d2 < 0.f ? 0.f : d2;
              v[e] = want_sq ? d2 : __fsqrt_rn(d2);
            }
          }
          if (vec_ok && gj0 + 32 <= g.m2) {
#pragma unroll
            for (int e = 0; e < 32; e += 4)
              *reinterpret_cast<float4*>(orow + gj0 + e) = make_float4(v[e], v[e + 1], v[e + 2], v[e + 3]);
          } else {
#pragma unroll
            for (int e = 0; e < 32; ++e)
              if (gj0 + e < g.m2) orow[gj0 + e] = v[e];
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[as]);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 2 * kBN);
  }
}

// ------------------------------------------------------------------------------------
// 2-CTA kernel (default): a cluster of two CTAs (one SM pair) owns a 256 x 256 output tile and
// issues tcgen05.mma.cta_group::2 (M = 256: 128 rows per CTA, N = 256).  Per 64-wide k-block each
// CTA loads ONLY its 128 rows of every A plane and its 128-row half of every B plane, and all
// plane-pair terms of the split product reuse those tiles: for bf16x3 that is 4 x 16 KB per CTA
// for 12 MMAs (5.3 KB of L2->SM traffic per 128-cycle MMA slot and SM, against 12 KB for the
// 1-CTA kernel above, which sits at the chip's TMA/L2 delivery limit rather than at the tensor
// pipe).  Barriers: full[] lives in the leader (rank 0) and collects both CTAs' TMA bytes;
// empty[] / tfull[] exist in both CTAs and are signalled by multicast tcgen05.commit; tempty[]
// lives in the leader and takes the arrivals of both CTAs' epilogue warps.
// ------------------------------------------------------------------------------------
constexpr int kT2Rows = 128;
constexpr int kTile2Bytes = kT2Rows * kBK * 2;      // 16 KB: one plane of one operand for one k-block
constexpr int kRing2Bytes = 192 * 1024;
constexpr int kMaxStages2 = 6;
constexpr int kOutChunkBytes = 32 * 32 * 4;                 // one warp's 32 x 32 fp32 staging tile
constexpr int kOutStageBytes = 4 * 2 * kOutChunkBytes;      // 4 epilogue warps, double-buffered
constexpr size_t kGemm2Smem = (size_t)kRing2Bytes + kOutStageBytes + 2 * 256 * 4 /*|b|^2 or alpha/beta*/ + 256 /*barriers*/;

// CL4 = true: a cluster of FOUR CTAs = two CTA pairs that work on two vertically adjacent 256-row m tiles of the SAME n
// tile.  Each CTA still loads its own 128 A rows; the B halves are loaded ONCE per cluster - by the CTAs of pair 0, with
// TMA .multicast::cluster into the CTA of the same parity in pair 1 - so the L2 -> SM traffic of B halves.  For the
// single-plane (fp16 / bf16x1) product, whose tiles are used by one term only and which therefore sits at the chip's
// L2 -> SM delivery limit instead of at the tensor pipe, that is 25 % fewer bytes per MMA.
template <int BN, int EPI, bool CL4>
__device__ __forceinline__ void dist_tc2_body(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmO,
                                              const Gemm2Args& ga, const RankFuse& rf) {
  extern __shared__ __align__(1024) unsigned char smem[];   // SWIZZLE_128B tiles need 1024-byte alignment
  if ((smem_u32(smem) & 1023u) != 0) __trap();
  constexpr int kBTile = (BN / 2) * kBK * 2;                 // this CTA's half of a B plane tile
  const int planes = ga.planes, stages = ga.stages;
  const uint32_t stage_bytes = (uint32_t)planes * (kTile2Bytes + kBTile);
  // after the ring: EPI_DIST / EPI_AFFINE_RELU: output staging [4 warps][2][4 KB]; EPI_RANK: threshold and counter tables
  unsigned char* after_ring = smem + (EPI == EPI_RANK ? (size_t)stages * stage_bytes : (size_t)kRing2Bytes);
  unsigned char* stage_out = after_ring;
  float* thr_s = reinterpret_cast<float*>(after_ring);                               // [p_cap][128]
  uint32_t* cnt_s = reinterpret_cast<uint32_t*>(after_ring + (size_t)rf.p_cap * 512); // [p_cap + 1][128]; row p_cap takes what is not counted
  float* bn_s = reinterpret_cast<float*>(after_ring + (EPI == EPI_RANK ? (size_t)rf.p_cap * 1024 + 512 : (size_t)kOutStageBytes));
  uint64_t* full = reinterpret_cast<uint64_t*>(reinterpret_cast<unsigned char*>(bn_s) + 2 * 256 * 4);
  uint64_t* empty = full + kMaxStages2;
  uint64_t* tfull = empty + kMaxStages2;      // [2]
  uint64_t* tempty = tfull + 2;               // [2] (used in the leader)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

  const GemmArgs& g = ga.g;
  constexpr int kEpiWarps = EPI == EPI_RANK ? 8 : 4;
  constexpr int kEpiThreads = kEpiWarps * 32;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t crank = cluster_ctarank();                 // rank in the cluster (0..1, or 0..3 with CL4)
  const uint32_t rank = crank & 1u;                         // rank in the CTA pair
  const uint32_t lead = crank & ~1u;                        // cluster rank of this pair's leader
  const int pair_row0 = CL4 ? (int)(crank >> 1) * 256 : 0;  // this pair's rows inside the cluster's m tile
  constexpr int kClusterRows = CL4 ? 512 : 256;
  const long long pair = CL4 ? (blockIdx.x >> 2) : (blockIdx.x >> 1), npairs = CL4 ? (gridDim.x >> 2) : (gridDim.x >> 1);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    if (EPI != EPI_RANK && !epi_search(EPI)) tma_prefetch_desc(&tmO);
    for (int s = 0; s < kMaxStages2; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], CL4 ? 2 : 1);   // CL4: a slot also receives the other pair's B half, so both pairs' MMAs free it
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tfull[s], 1);
      mbar_init(&tempty[s], 2 * kEpiWarps);   // the epilogue warps of both CTAs
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc_2cta(tmem_slot, 512);
    tmem_relinquish_2cta();
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer (both CTAs) =====================
    if (lane == 0) {
      uint32_t it = 0;
      TileWalk<EPI> w(ga, pair, npairs);
      // EPI_RANK progress window (RankFuse::window): see dist_tiles.cuh
      const bool windowed = EPI == EPI_RANK && rf.window > 0 && w.balanced && !w.extra;
      uint32_t tile_j = 0;
      if (windowed && rank == 0 && w.n_cur >= w.n_stop) st_volatile_u32(rf.progress + pair, 0xffffffffu);   // nothing to do: never waited for
      while (w.next()) {
        if (windowed) {
          const uint32_t* peers = rf.progress + (long long)w.stream_i * w.m_tiles;
          for (;;) {
            uint32_t mn = 0xffffffffu;
            for (int m = 0; m < w.m_tiles; ++m) mn = min(mn, ld_volatile_u32(peers + m));
            if (tile_j - min(tile_j, mn) <= (uint32_t)rf.window) break;
            __nanosleep(200);
          }
        }
        const int m0 = (int)(w.grp * ga.a_group_rows) + w.m_tile * kClusterRows + pair_row0 + (int)rank * kT2Rows;
        const int n0 = (int)(w.grp * ga.b_group_rows) + w.n_tile * BN + (int)rank * (BN / 2);
        for (int kb = 0; kb < g.kblocks; ++kb, ++it) {
          const uint32_t s = it % stages, ph = (it / stages) & 1u;
          mbar_wait(&empty[s], ph ^ 1u);
          if (rank == 0) mbar_expect_tx(&full[s], 2u * stage_bytes);
          const uint32_t full0 = map_to_cta(smem_u32(&full[s]), lead);
          unsigned char* slot = smem + (size_t)s * stage_bytes;
          for (int p = 0; p < planes; ++p) tma_load_3d_2cta(slot + p * kTile2Bytes, &tmA, full0, kb * kBK, m0, p);
          if (!CL4) {
            for (int p = 0; p < planes; ++p)
              tma_load_3d_2cta(slot + planes * kTile2Bytes + p * kBTile, &tmB, full0, kb * kBK, n0, p);
          } else if (crank < 2) {
            // pair 0 loads the B halves for the whole cluster: CTA r and CTA r + 2 receive the same half, each signalling
            // the full barrier of its own pair leader (the barrier address is relative to the destination's pair)
            const uint16_t mask = (uint16_t)(0x5u << rank);
            for (int p = 0; p < planes; ++p)
              tma_load_3d_2cta_mcast(slot + planes * kTile2Bytes + p * kBTile, &tmB, full0, mask, kb * kBK, n0, p);
          }
        }
        ++tile_j;
        if (windowed && rank == 0) st_volatile_u32(rf.progress + pair, w.run_end ? 0xffffffffu : tile_j);
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA, one thread) =====================
    if (rank == 0 && lane == 0) {
      uint32_t it = 0, acc_it = 0;
      TileWalk<EPI> w(ga, pair, npairs);
      // sep_small: the leading term p0.p0 accumulates in columns [0, 256), every cross term in columns [256, 512) and
      // the epilogue adds the two.  The tensor core truncates ~1 ulp OF THE ACCUMULATOR per MMA step; the cross terms are
      // 2^-11 of the leading one, so in a buffer of their own their 2/3 of the steps cost nothing, and the large
      // accumulator sees K/16 steps instead of 3K/16.  Price: no second buffer to overlap the epilogue with the next tile.
      const bool sep = ga.sep_small != 0;
      int first_small = -1;
      for (int term = 0; term < g.nterms; ++term)
        if (first_small < 0 && (g.term_a[term] | g.term_b[term]) != 0) first_small = term;
      for (; w.next(); ++acc_it) {
        const uint32_t as = sep ? 0u : (acc_it & 1u), aph = sep ? (acc_it & 1u) : ((acc_it >> 1) & 1u);
        mbar_wait(&tempty[as], aph ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * BN;
        for (int kb = 0; kb < g.kblocks; ++kb, ++it) {
          const uint32_t s = it % stages, ph = (it / stages) & 1u;
          mbar_wait(&full[s], ph);
          tc_fence_after();
          const uint32_t slot = smem_u32(smem + (size_t)s * stage_bytes);
          for (int term = 0; term < g.nterms; ++term) {
            const uint64_t adesc = umma_desc_k_sw128(slot + g.term_a[term] * kTile2Bytes);
            const uint64_t bdesc = umma_desc_k_sw128(slot + planes * kTile2Bytes + g.term_b[term] * kBTile);
            const bool small = sep && (g.term_a[term] | g.term_b[term]) != 0;
            const uint32_t d_term = small ? tmem_base + 256u : d_tmem;
            const bool first = sep ? (kb == 0 && (small ? term == first_small : true)) : (kb == 0 && term == 0);
#pragma unroll
            for (int k = 0; k < kBK / 16; ++k)
              tc_mma_f16_2cta(d_term, adesc + 2u * k, bdesc + 2u * k, g.idesc, (first && k == 0) ? 0u : 1u);
          }
          tc_commit_2cta(&empty[s], CL4 ? 0xF : 3);   // the slots (of every CTA that holds a tile these MMAs read) are reusable
        }
        tc_commit_2cta(&tfull[as], (uint16_t)(3u << lead));   // accumulator complete in both CTAs of this pair
      }
    }
  } else {
    // ===================== epilogue (warps 2..5 of both CTAs) =====================
    // EPI_DIST / EPI_AFFINE_RELU: TMEM -> registers (thread = row) -> value -> 128B-swizzled staging tile in shared
    // memory -> one TMA store per 32 x 32 chunk (coalesced, clipped at the matrix edges by the tensor map).
    // EPI_RANK: TMEM -> registers -> distance -> lower bound among the row's thresholds -> private counter.
    const int lane_grp = warp & 3;              // the TMEM lanes a warp may read: 32 * (warp % 4) ..
    const int row = lane_grp * 32 + lane;
    const int etid = (int)threadIdx.x - 64;     // 0 .. kEpiThreads - 1 among the epilogue threads
    const int col_half = EPI == EPI_RANK ? ((warp - 2) >> 2) : 0;    // EPI_RANK: which 128 columns of the tile this warp takes
    uint32_t acc_it = 0, chunk_it = 0;
    const bool want_sq = (g.flags & PPS_DIST_SQUARED) != 0;
    const bool want_dot = (g.flags & PPS_DIST_DOT) != 0;
    const bool sqrt_rn = (g.flags & PPS_DIST_SQRT_RN) != 0;     // correctly rounded sqrt (the reference's np.sqrt) instead of MUFU
    unsigned char* my_stage = stage_out + (size_t)lane_grp * (2 * kOutChunkBytes);
    const uint32_t swz = (uint32_t)(lane & 7);
    // EPI_RANK per-row state
    const int p_cap = rf.p_cap;
    float dstar = 0.f;
    long long gstar = 0;
    uint32_t tie_corr = 0;
    float piv1 = 0.f, piv2a = 0.f, piv2b = 0.f; // thresholds probed by the first two search levels
    uint32_t rk_bound = 0u;                     // top-k admission bound of this row (EPI_RANK with candidate lists)
    const bool rk_admit = EPI == EPI_RANK && rf.tk_cand != nullptr;
    long long tab_base = 0;                     // element offset of (row group, j = 0, this row) in the global tables
    long long row_tag = 0;                      // EPI_SEARCH_EXCL: this row's tag, loaded for m tile tag_tile
    int tag_tile = -1;
    TileWalk<EPI> w(ga, pair, npairs);
    for (; w.next(); ++acc_it) {
      const int m0 = w.m_tile * kClusterRows + pair_row0 + (int)rank * kT2Rows;       // output row (within the group's rows)
      const int n0 = (int)(w.grp * ga.out_group_cols) + w.n_tile * BN;              // output column
      const int n_end = EPI == EPI_AFFINE_RELU ? (int)((w.grp + 1) * ga.out_group_cols) : (int)g.m2;   // first column not ours
      const bool sep = (EPI == EPI_DIST || EPI == EPI_DIST_TOPK) && ga.sep_small != 0;
      const uint32_t as = sep ? 0u : (acc_it & 1u), aph = sep ? (acc_it & 1u) : ((acc_it >> 1) & 1u);
      const long long gi = (long long)m0 + row;
      if (EPI == EPI_RANK && w.run_start) {
        // this row of the threshold table -> shared memory.  The two threads of a row (one per column half) write the same
        // values and each reads after its own writes; the counters are zero here: zeroed at kernel start, re-zeroed by every
        // flush, and the barrier before a flush keeps this block behind the last use of the previous run's tables
        tab_base = ((long long)(m0 >> 7) * p_cap) * 128 + row;
        for (int j = 0; j < p_cap; ++j) thr_s[j * 128 + row] = __ldg(rf.thr_tab + tab_base + (long long)j * 128);
        if (acc_it == 0)
          for (int j = col_half; j < p_cap; j += 2) cnt_s[j * 128 + row] = 0u;
        dstar = gi < g.m1 ? __ldg(rf.dstar + gi) : __int_as_float(0x7fc00000);
        gstar = gi < g.m1 ? (long long)__ldg(rf.gstar + gi) : 0;
        rk_bound = (rf.tk_cand != nullptr && gi < g.m1) ? __ldg(rf.tk_bound + gi) : 0u;
        tie_corr = 0;
        const int h1 = p_cap >> 1, h2 = (p_cap - h1) >> 1;
        piv1 = thr_s[(h1 - 1) * 128 + row];
        piv2a = thr_s[(h2 - 1) * 128 + row];
        piv2b = thr_s[(h1 + h2 - 1) * 128 + row];
      }
      // per-column operands of the tile -> shared (double-buffered by accumulator stage):
      // |b|^2 of the gallery rows, or alpha / beta of the output channels
      // (scaled operands: |b|^2 and the column scales share the two buffers, so they are single-buffered and a
      // second barrier at the end of the tile keeps a fast warp from refilling them early)
      const bool scaled = EPI != EPI_AFFINE_RELU && EPI != EPI_RANK && g.a_scale != nullptr;
      float* bn = bn_s + (scaled ? 0 : as * 256);      // (sep: as == 0 for every tile, the end-of-tile barrier below protects it)
      const float* sc_s = bn_s + 256;
      if (EPI == EPI_AFFINE_RELU) {
        const long long gj = (long long)n0 + etid;            // BN == 128 == number of epilogue threads
        bn[etid] = gj < n_end ? __ldg(g.a_sqnorm + gj) : 0.f;
        bn[etid + 128] = gj < n_end ? __ldg(g.b_sqnorm + gj) : 0.f;
      } else {
        const long long gj = (long long)n0 + etid;
        if (!want_dot) {
          bn[etid] = gj < g.m2 ? __ldg(g.b_sqnorm + gj) : 0.f;
          if (BN > kEpiThreads) bn[etid + 128] = gj + 128 < g.m2 ? __ldg(g.b_sqnorm + gj + 128) : 0.f;
        }
        if (scaled) {
          bn_s[256 + etid] = gj < g.m2 ? __ldg(g.b_scale + gj) : 0.f;
          if (BN > 128) bn_s[256 + etid + 128] = gj + 128 < g.m2 ? __ldg(g.b_scale + gj + 128) : 0.f;
        }
        if (epi_search(EPI)) {                 // the admission bound (EPI_RANGE: limit) of every query column, double-buffered
          uint32_t* bd = reinterpret_cast<uint32_t*>(stage_out) + as * 256;
          bd[etid] = gj < g.m2 ? __ldg(rf.tk_bound + gj) : 0u;
          if (BN > 128) bd[etid + 128] = gj + 128 < g.m2 ? __ldg(rf.tk_bound + gj + 128) : 0u;
        }
      }
      asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");
      const float an = (EPI != EPI_AFFINE_RELU && gi < g.m1 && !want_dot) ? __ldg(g.a_sqnorm + gi) : 0.f;
      const float cs = (scaled && gi < g.m1) ? -2.f * __ldg(g.a_scale + gi) : -2.f;    // -2 / s_a
      uint32_t tk_bound = 0u;                  // EPI_DIST_TOPK: nothing is admitted for padding rows
      if (EPI == EPI_DIST_TOPK && gi < g.m1) tk_bound = __ldg(rf.tk_bound + gi);
      mbar_wait(&tfull[as], aph);
      tc_fence_after();
      const uint32_t tbase = tmem_base + as * BN + ((uint32_t)(lane_grp * 32) << 16);
      // EPI_SEARCH: chunks of 32 query columns up to the last query of the tile
      const int c_first = EPI == EPI_RANK ? col_half * 128 : 0;
      const int c_stop = EPI == EPI_RANK ? c_first + 128 : epi_search(EPI) ? (int)min((long long)BN, (g.m2 - n0 + 31) & ~31LL) : BN;
#pragma unroll 1
      for (int c = c_first; c < c_stop; c += 32, ++chunk_it) {
        uint32_t r[32];
        tmem_ld_32x32(tbase + c, r);
        if (epi_search(EPI)) {
          // thread = gallery row, columns = queries.  pps_dist_tc's arithmetic with the roles swapped:
          // (-2ab + |q|^2) + |g|^2 with -2ab = (-2 / (s_g s_q)) dot exact, so every distance has pps_dist_tc's bits.
          tmem_ld_wait();
          const uint32_t* bd = reinterpret_cast<const uint32_t*>(stage_out) + as * 256 + c;
          const float4* qn4 = reinterpret_cast<const float4*>(bn + c);
          const bool row_ok = gi < g.m1;
          const long long valid_cols = g.m2 - n0 - c;          // query columns of this chunk that exist
          uint32_t v[32];
          bool hit = false;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float4 q4 = qn4[j];
            const float qq[4] = {q4.x, q4.y, q4.z, q4.w};
            float sc[4] = {cs, cs, cs, cs};
            if (scaled) {
              const float4 s4 = reinterpret_cast<const float4*>(sc_s + c)[j];
              sc[0] = cs * s4.x; sc[1] = cs * s4.y; sc[2] = cs * s4.z; sc[3] = cs * s4.w;
            }
            const uint4 b4 = reinterpret_cast<const uint4*>(bd)[j];
            const uint32_t bb[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float dot = __uint_as_float(r[4 * j + e]);
              float d2 = __fadd_rn(__fmaf_rn(sc[e], dot, qq[e]), an);
              d2 = clamp0_keep_nan(d2);
              v[4 * j + e] = __float_as_uint(want_sq ? d2 : (sqrt_rn ? __fsqrt_rn(d2) : sqrt_approx(d2)));
              // distances are >= 0: bits order like values.  EPI_RANGE: bb is the limit bits(radius) + 1 (0: none)
              hit |= (epi_range(EPI) ? v[4 * j + e] < bb[e] : v[4 * j + e] <= bb[e]) & (4 * j + e < valid_cols);
            }
          }
          // admission, aggregated per (warp, query): one atomic reserves the slots of every lane that passes
          if (__any_sync(0xffffffffu, hit && row_ok)) {
            const uint32_t lanes_below = (1u << lane) - 1u;
            const unsigned long long gkey = (unsigned long long)(uint32_t)(rf.col0 + gi);
            // EPI_SEARCH_EXCL, EPI_RANGE_EXCL: the row's tag is loaded on the row's first hit of the tile (the n tiles of
            // one m tile share it)
            if (epi_excl(EPI) && hit && row_ok && tag_tile != w.m_tile) {
              row_tag = __ldg(rf.g_tags + gi);
              tag_tile = w.m_tile;
            }
#pragma unroll
            for (int e = 0; e < 32; ++e) {                     // (unrolled: v[] must stay in registers)
              bool pass = row_ok && e < valid_cols && (epi_range(EPI) ? v[e] < bd[e] : v[e] <= bd[e]);
              if (epi_excl(EPI) && pass)                       // one address per warp: an L1 broadcast
                pass = row_tag != __ldg(rf.q_tags + ((long long)n0 + c + e));
              const uint32_t m = __ballot_sync(0xffffffffu, pass);
              if (m) {
                const long long col = (long long)n0 + c + e;
                const int leader = __ffs(m) - 1;
                uint32_t base = 0;
                if (lane == leader) base = atomicAdd(rf.tk_cnt + col, (uint32_t)__popc(m));
                base = __shfl_sync(0xffffffffu, base, leader);
                const uint32_t slot = base + (uint32_t)__popc(m & lanes_below);
                if (epi_range(EPI)) {                          // (the query's offset and capacity: broadcasts too)
                  if (pass && slot < __ldg(rf.out_cap + col))
                    rf.tk_cand[__ldg(rf.out_off + col) + slot] = ((unsigned long long)v[e] << 32) | gkey;
                } else if (pass && slot < (uint32_t)rf.tk_cap) {
                  rf.tk_cand[col * rf.tk_cap + slot] = ((unsigned long long)v[e] << 32) | gkey;
                }
              }
            }
          }
        } else if (EPI == EPI_RANK) {
          tmem_ld_wait();
          const int valid_cols = n_end - n0 - c;             // columns of this chunk inside the gallery block
          const long long colg = rf.col0 + n0 + c;           // global gallery index of the chunk's first column
          const float4* bn4 = reinterpret_cast<const float4*>(bn + c);
          float d[32];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float4 b4 = bn4[j];
            const float bb[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float dot = __uint_as_float(r[4 * j + e]);
              float d2 = __fadd_rn(__fmaf_rn(-2.f, dot, an), bb[e]);      // the EPI_DIST arithmetic, bit for bit
              d2 = clamp0_keep_nan(d2);
              d[4 * j + e] = want_sq ? d2 : sqrt_approx(d2);
            }
          }
          // lower bound of every element among this row's thresholds: 32 independent searches per step, the first two
          // levels against pivots held in registers.  The position is kept as the BYTE offset of (threshold lo, this row)
          // in the [threshold][row] tables, so that a probe is one LDS at (uniform base + offset) and the counter of the
          // result sits at the same offset of the counter table.  "Above t" is the unordered !(d <= t), so that a NaN
          // distance falls past every threshold (as in the reference's argsort) for the price of a plain compare.
          uint32_t off[32];
          const int half1 = p_cap >> 1, half2 = (p_cap - half1) >> 1;
          const uint32_t row_off = (uint32_t)row * 4u, h1o = (uint32_t)half1 * 512u, h2o = (uint32_t)half2 * 512u;
#pragma unroll
          for (int e = 0; e < 32; ++e) {
            const bool up = !(d[e] <= piv1);
            off[e] = row_off + (up ? h1o : 0u);
            off[e] += !(d[e] <= (up ? piv2b : piv2a)) ? h2o : 0u;
          }
          const uint32_t thr_base = smem_u32(thr_s);
          int len = p_cap - half1 - half2;
          while (len > 1) {
            const int half = len >> 1;
            const uint32_t probe = thr_base + (uint32_t)(half - 1) * 512u, step = (uint32_t)half * 512u;
#pragma unroll
            for (int e = 0; e < 32; ++e) off[e] += !(d[e] <= lds_f32(probe + off[e])) ? step : 0u;
            len -= half;
          }
          bool tie = false;
#pragma unroll
          for (int e = 0; e < 32; ++e) {
            off[e] += !(d[e] <= lds_f32(thr_base + off[e])) ? 512u : 0u;
            tie |= (d[e] == dstar);
          }
          // one fire-and-forget shared-memory add per element (no read-back, so no dependent chain).  An element beyond every
          // threshold lands in row p_cap of the counter table, which nobody reads; so do the columns past the block's end.
          const uint32_t cnt_base = smem_u32(cnt_s);
          if (valid_cols >= 32) {
#pragma unroll
            for (int e = 0; e < 32; ++e) red_shared_add_u32(cnt_base + off[e], 1u);
          } else {
            const uint32_t dump = row_off + (uint32_t)p_cap * 512u;
#pragma unroll
            for (int e = 0; e < 32; ++e) red_shared_add_u32(cnt_base + (e < valid_cols ? off[e] : dump), 1u);
          }
          if (tie) {                                         // exact ties with the nearest positive: rare
#pragma unroll                                               // (unrolled: a runtime index would push d[] to local memory)
            for (int e = 0; e < 32; ++e)
              if (e < valid_cols && d[e] == dstar) tie_corr += ((colg + e) < gstar ? 1u : 0u) - 1u;
          }
          if (rk_admit) {
            // top-k admission, as EPI_DIST_TOPK: one compare per element against the row's k-th best so far (distances
            // are >= 0: their bits order like the values); almost never true once a bound exists
            bool hit = false;
#pragma unroll
            for (int e = 0; e < 32; ++e) hit |= __float_as_uint(d[e]) <= rk_bound;
            if (hit && gi < g.m1) {
#pragma unroll
              for (int e = 0; e < 32; ++e) {
                if (__float_as_uint(d[e]) <= rk_bound && e < valid_cols) {
                  const uint32_t slot = atomicAdd(rf.tk_cnt + gi, 1u);
                  if (slot < (uint32_t)rf.tk_cap)
                    rf.tk_cand[(long long)gi * rf.tk_cap + slot] =
                        ((unsigned long long)__float_as_uint(d[e]) << 32) | (unsigned long long)(uint32_t)(colg + e);
                }
              }
            }
          }
        } else {
          unsigned char* buf = my_stage + (chunk_it & 1u) * kOutChunkBytes;
          if (sep) {                               // + the cross terms from their own accumulator
            uint32_t r2[32];
            tmem_ld_32x32(tbase + 256u + c, r2);
            tmem_ld_wait();
#pragma unroll
            for (int e = 0; e < 32; ++e) r[e] = __float_as_uint(__fadd_rn(__uint_as_float(r[e]), __uint_as_float(r2[e])));
          }
          bulk_wait_group_read<1>();               // the store that last read this buffer has drained it
          __syncwarp();
          tmem_ld_wait();
          const float4* bn4 = reinterpret_cast<const float4*>(bn + c);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            float v[4];
            const float4 b4 = bn4[j];
            const float bb[4] = {b4.x, b4.y, b4.z, b4.w};
            float cc[4] = {0.f, 0.f, 0.f, 0.f};
            if (EPI == EPI_AFFINE_RELU) {
              const float4 c4 = reinterpret_cast<const float4*>(bn + 128 + c)[j];
              cc[0] = c4.x; cc[1] = c4.y; cc[2] = c4.z; cc[3] = c4.w;
            }
            float sc[4] = {cs, cs, cs, cs};
            if (scaled) {                       // -2 / (s_a s_b): a product of powers of two, exact
              const float4 q4 = reinterpret_cast<const float4*>(sc_s + c)[j];
              sc[0] = cs * q4.x; sc[1] = cs * q4.y; sc[2] = cs * q4.z; sc[3] = cs * q4.w;
            }
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float dot = __uint_as_float(r[4 * j + e]);
              if (EPI == EPI_AFFINE_RELU) {
                v[e] = fmaxf(fmaf(dot, bb[e], cc[e]), 0.f);
              } else if (want_dot) {
                v[e] = scaled ? dot * (-0.5f * sc[e]) : dot;
              } else {
                // same association as the reference: (-2*ab + |a|^2) + |b|^2   (-2*ab is exact, so the FMA rounds once;
                // with scaled operands sc = -2 / (s_a s_b) and sc * dot is the same exact product)
                float d2 = __fadd_rn(__fmaf_rn(sc[e], dot, an), bb[e]);
                d2 = clamp0_keep_nan(d2);
                v[e] = want_sq ? d2 : (sqrt_rn ? __fsqrt_rn(d2) : sqrt_approx(d2));
              }
            }
            *reinterpret_cast<float4*>(buf + lane * 128 + (((uint32_t)j ^ swz) << 4)) = make_float4(v[0], v[1], v[2], v[3]);
            if (EPI == EPI_DIST_TOPK) {
              // distances are >= 0: their bits order like the values.  Almost never true once a bound exists.
              if ((__float_as_uint(v[0]) <= tk_bound) | (__float_as_uint(v[1]) <= tk_bound) |
                  (__float_as_uint(v[2]) <= tk_bound) | (__float_as_uint(v[3]) <= tk_bound)) {
#pragma unroll
                for (int e = 0; e < 4; ++e) {             // (unrolled: v[] must stay in registers)
                  const int col = n0 + c + 4 * j + e;
                  if (__float_as_uint(v[e]) <= tk_bound && col < n_end && gi < g.m1) {   // (an exact 0 passes even a 0 bound)
                    const uint32_t slot = atomicAdd(rf.tk_cnt + gi, 1u);
                    if (slot < (uint32_t)rf.tk_cap)
                      rf.tk_cand[(long long)gi * rf.tk_cap + slot] =
                          ((unsigned long long)__float_as_uint(v[e]) << 32) | (unsigned long long)(uint32_t)(rf.col0 + col);
                  }
                }
              }
            }
          }
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) {
            if (m0 + lane_grp * 32 < g.m1 && n0 + c < n_end) tma_store_2d(&tmO, buf, n0 + c, m0 + lane_grp * 32);
            bulk_commit_group();
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (rank == 0) mbar_arrive(&tempty[as]);
        else mbar_arrive_cluster(map_to_cta(smem_u32(&tempty[as]), lead));
      }
      if (scaled || sep) asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");   // every warp is done with bn / sc of this tile
      if (EPI == EPI_RANK && w.run_end) {
        // counters -> global table at the end of the run (a handful of CTA pairs share a row: atomics).  Both threads of a
        // row must be done with the tile first; each then flushes (and re-zeroes) every other counter.
        asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");
        for (int j = col_half; j < p_cap; j += 2) {
          const uint32_t v = cnt_s[j * 128 + row];
          if (v) {
            cnt_s[j * 128 + row] = 0u;
            if (gi < g.m1) atomicAdd(rf.cnt_tab + tab_base + (long long)j * 128, v);
          }
        }
        if (gi < g.m1 && tie_corr) atomicAdd(rf.cnt_first + gi, tie_corr);
      }
    }
    if (EPI != EPI_RANK && !epi_search(EPI)) bulk_wait_group_read<0>();
  }

  tc_fence_before();
  cluster_sync_all();      // no CTA of the pair leaves (or frees TMEM) while its peer still signals it
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_2cta(tmem_base, 512);
  }
}

template <int BN, int EPI>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(gemm2_threads<EPI>(), 1)
dist_tc2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                const __grid_constant__ CUtensorMap tmO, const __grid_constant__ Gemm2Args ga,
                const __grid_constant__ RankFuse rf) {
  dist_tc2_body<BN, EPI, false>(tmA, tmB, tmO, ga, rf);
}

template <int BN, int EPI>
__global__ void __cluster_dims__(4, 1, 1) __launch_bounds__(kGemmThreads, 1)
dist_tc4_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                const __grid_constant__ CUtensorMap tmO, const __grid_constant__ Gemm2Args ga,
                const __grid_constant__ RankFuse rf) {
  dist_tc2_body<BN, EPI, true>(tmA, tmB, tmO, ga, rf);
}

// ------------------------------------------------------------------------------------
// CUDA-core fp32 distance (PPS_PREC_FP32): exact-product FMA path on the original rows.
// 64x64 tile per CTA, 16x16 threads, 4x4 outputs per thread, K tile 16.
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) dist_fp32_kernel(const float* __restrict__ a, long long lda,
                                                        const float* __restrict__ an, long long m1,
                                                        const float* __restrict__ b, long long ldb,
                                                        const float* __restrict__ bn, long long m2, int dim, int flags,
                                                        float* __restrict__ out, long long ldo) {
  __shared__ float sa[16][64 + 4];
  __shared__ float sb[16][64 + 4];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const long long m0 = (long long)blockIdx.y * 64, n0 = (long long)blockIdx.x * 64;
  float acc[4][4] = {};
  for (int k0 = 0; k0 < dim; k0 += 16) {
    for (int i = threadIdx.x; i < 64 * 16; i += 256) {
      const int r = i >> 4, k = i & 15;
      sa[k][r] = (m0 + r < m1 && k0 + k < dim) ? a[(m0 + r) * lda + k0 + k] : 0.f;
      sb[k][r] = (n0 + r < m2 && k0 + k < dim) ? b[(n0 + r) * ldb + k0 + k] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      float av[4], bv[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { av[i] = sa[k][ty * 4 + i]; bv[i] = sb[k][tx * 4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    __syncthreads();
  }
  const bool want_sq = (flags & PPS_DIST_SQUARED) != 0, want_dot = (flags & PPS_DIST_DOT) != 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const long long gi = m0 + ty * 4 + i;
    if (gi >= m1) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const long long gj = n0 + tx * 4 + j;
      if (gj >= m2) continue;
      float v = acc[i][j];
      if (!want_dot) {
        float d2 = __fadd_rn(__fadd_rn(__fmul_rn(-2.f, v), an[gi]), bn[gj]);
        d2 = d2 < 0.f ? 0.f : d2;
        v = want_sq ? d2 : __fsqrt_rn(d2);
      }
      out[gi * ldo + gj] = v;
    }
  }
}

// ------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

// planes: [n_planes][rows][kpad] 16-bit elements, K-major
static int make_operand_map(CUtensorMap* tm, const void* planes, long long rows, long long plane_rows, int kpad,
                            int n_planes, int box_rows, bool f16) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return cuda_fail(cudaErrorUnknown, "cuTensorMapEncodeTiled entry point not found");
  cuuint64_t dims[3] = {(cuuint64_t)kpad, (cuuint64_t)rows, (cuuint64_t)n_planes};
  cuuint64_t strides[2] = {(cuuint64_t)kpad * 2, (cuuint64_t)plane_rows * (cuuint64_t)kpad * 2};
  cuuint32_t box[3] = {(cuuint32_t)kBK, (cuuint32_t)box_rows, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = fn(tm, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3,
                  const_cast<void*>(planes), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return cuda_fail(cudaErrorInvalidValue, "cuTensorMapEncodeTiled failed");
  return PPS_OK;
}

// plane-pair terms of a precision: returns the planes needed per operand, 0 if the precision is not a tensor-core one
static int setup_terms(int precision, GemmArgs& g, bool* f16) {
  *f16 = false;
  switch (precision) {
    case PPS_PREC_BF16X1:
      g.nterms = 1; g.term_a[0] = 0; g.term_b[0] = 0; return 1;
    case PPS_PREC_BF16X3: {
      const int ta[3] = {1, 0, 0}, tb[3] = {0, 1, 0};   // small terms first
      g.nterms = 3; for (int i = 0; i < 3; ++i) { g.term_a[i] = ta[i]; g.term_b[i] = tb[i]; }
      return 2;
    }
    case PPS_PREC_BF16X6: {
      const int ta[6] = {2, 0, 1, 1, 0, 0}, tb[6] = {0, 2, 1, 0, 1, 0};
      g.nterms = 6; for (int i = 0; i < 6; ++i) { g.term_a[i] = ta[i]; g.term_b[i] = tb[i]; }
      return 3;
    }
    case PPS_PREC_F16X1:
      g.nterms = 1; g.term_a[0] = 0; g.term_b[0] = 0; *f16 = true; return 1;
    case PPS_PREC_F16X3: {
      const int ta[3] = {1, 0, 0}, tb[3] = {0, 1, 0};
      g.nterms = 3; for (int i = 0; i < 3; ++i) { g.term_a[i] = ta[i]; g.term_b[i] = tb[i]; }
      *f16 = true; return 2;
    }
    default: return 0;
  }
}

}  // namespace pps

using namespace pps;

static int dist_tc_impl(const void* a_planes, const float* a_sqnorm, long long m1, int a_planes_n,
                        long long a_plane_rows, const void* b_planes, const float* b_sqnorm, long long m2,
                        int b_planes_n, long long b_plane_rows, int dim, int precision, int flags, float* dist,
                        long long ldd, void* stream, const RankFuse* topk) {
  if (m1 < 0 || m2 < 0 || dim <= 0 || ldd < m2) return PPS_ERR_INVALID_ARG;
  if (a_plane_rows == 0) a_plane_rows = m1;
  if (b_plane_rows == 0) b_plane_rows = m2;
  if (a_plane_rows < m1 || b_plane_rows < m2) return PPS_ERR_INVALID_ARG;
  if (m1 == 0 || m2 == 0) return PPS_OK;
  if (!a_planes || !b_planes || !dist) return PPS_ERR_INVALID_ARG;
  if (!(flags & PPS_DIST_DOT) && (!a_sqnorm || !b_sqnorm)) return PPS_ERR_INVALID_ARG;
  if ((reinterpret_cast<uintptr_t>(a_planes) & 15u) || (reinterpret_cast<uintptr_t>(b_planes) & 15u))
    return PPS_ERR_ALIGN;
  if (m1 > 0x7fffff00LL || m2 > 0x7fffff00LL) return PPS_ERR_UNSUPPORTED;   // TMA coordinates are int32

  GemmArgs g;
  bool f16 = false;
  const int need = setup_terms(precision, g, &f16);
  if (need == 0) return PPS_ERR_INVALID_ARG;
  const bool scaled = precision == PPS_PREC_F16X3;
  if (scaled && (!a_sqnorm || !b_sqnorm)) return PPS_ERR_INVALID_ARG;     // they carry the row scales too
  if (a_planes_n < need || b_planes_n < need) return PPS_ERR_INVALID_ARG;

  const int kpad = pps_kpad(dim);
  g.m1 = m1; g.m2 = m2;
  g.kblocks = kpad / kBK;
  const uint32_t fmt = f16 ? 0u : 1u;   // F16F32Format: F16 = 0, BF16 = 1
  g.idesc = (1u << 4) /*D = f32*/ | (fmt << 7) | (fmt << 10) | ((uint32_t)(kBN >> 3) << 17) | ((uint32_t)(kBM >> 4) << 24);
  g.a_sqnorm = a_sqnorm; g.b_sqnorm = b_sqnorm;
  g.a_scale = scaled ? a_sqnorm + a_plane_rows : nullptr;
  g.b_scale = scaled ? b_sqnorm + b_plane_rows : nullptr;
  g.out = dist; g.ldo = ldd; g.flags = flags;
  g.m_tiles = (int)((m1 + kBM - 1) / kBM);
  g.n_tiles = (int)((m2 + kBN - 1) / kBN);

  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int dev = 0;
  PPS_CUDA_TRY(cudaGetDevice(&dev));
  const int sms = sm_count();
  CUtensorMap tmA, tmB;

  const bool out_tma_ok = ((ldd & 3) == 0) && ((reinterpret_cast<uintptr_t>(dist) & 15u) == 0);
  if (!(flags & PPS_DIST_KERNEL_1CTA) && sms >= 2 && out_tma_ok) {
    // ---- 2-CTA kernel: 256 x 256 tiles, 128-row boxes for both operands ----
    Gemm2Args ga;
    ga.g = g;
    ga.g.m_tiles = (int)((m1 + 255) / 256);
    ga.g.n_tiles = (int)((m2 + 255) / 256);
    ga.g.idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(256 >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
    ga.planes = need;
    static const int env_sep = [] { const char* e = getenv("PPS_SEPARATE_SMALL"); return e ? atoi(e) : -1; }();
    static const int env_sqrt = [] { const char* e = getenv("PPS_SQRT_RN"); return e ? atoi(e) : -1; }();
    if (env_sqrt >= 0) ga.g.flags = env_sqrt ? (ga.g.flags | PPS_DIST_SQRT_RN) : (ga.g.flags & ~PPS_DIST_SQRT_RN);
    ga.sep_small = (g.nterms > 1 && (env_sep >= 0 ? env_sep != 0 : (flags & PPS_DIST_SEPARATE_SMALL) != 0)) ? 1 : 0;
    ga.stages = kRing2Bytes / (2 * need * kTile2Bytes);
    if (ga.stages > kMaxStages2) ga.stages = kMaxStages2;
    ga.groups = 1; ga.a_group_rows = 0; ga.b_group_rows = 0; ga.out_group_cols = 0;
    int rc = make_operand_map(&tmA, a_planes, m1, a_plane_rows, kpad, a_planes_n, kT2Rows, f16);
    if (rc) return rc;
    rc = make_operand_map(&tmB, b_planes, m2, b_plane_rows, kpad, b_planes_n, kT2Rows, f16);
    if (rc) return rc;
    CUtensorMap tmO;
    {
      EncodeTiledFn fn = encode_fn();
      if (!fn) return cuda_fail(cudaErrorUnknown, "cuTensorMapEncodeTiled entry point not found");
      cuuint64_t dims[2] = {(cuuint64_t)m2, (cuuint64_t)m1};
      cuuint64_t strides[1] = {(cuuint64_t)ldd * 4};
      cuuint32_t box[2] = {32, 32};
      cuuint32_t estr[2] = {1, 1};
      CUresult r = fn(&tmO, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, dist, dims, strides, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) return cuda_fail(cudaErrorInvalidValue, "cuTensorMapEncodeTiled(output) failed");
    }
    static thread_local int configured2_dev = -1;
    if (configured2_dev != dev) {
      PPS_CUDA_TRY(cudaFuncSetAttribute(dist_tc2_kernel<256, EPI_DIST>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)kGemm2Smem));
      configured2_dev = dev;
    }
    // Opt-in (PPS_DIST_CLUSTER4, or PPS_CLUSTER4=1 in the environment): clusters of four CTAs whose two pairs share the B
    // halves by TMA multicast.  Bit-identical, 25 % fewer L2 reads - and measured SLOWER on B200 (10 M x 2048 fp16: 149.7 vs
    // 141.1 ms of distance kernels per pass): the single-plane product is bound by what each SM can take in, which multicast
    // does not change, and 4-CTA clusters leave 12 of the 148 SMs idle.  Kept for the record and for other shapes.
    static const bool env_cluster4 = getenv("PPS_CLUSTER4") != nullptr;
    if (need == 1 && m1 > 256 && ((flags & PPS_DIST_CLUSTER4) || env_cluster4) && sms >= 4) {
      static thread_local int cfg4_dev = -1;
      static thread_local int max_clusters[2] = {0, 0};
      if (cfg4_dev != dev) {
        PPS_CUDA_TRY(cudaFuncSetAttribute(dist_tc4_kernel<256, EPI_DIST>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)kGemm2Smem));
        PPS_CUDA_TRY(cudaFuncSetAttribute(dist_tc4_kernel<256, EPI_DIST_TOPK>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)kGemm2Smem));
        for (int v = 0; v < 2; ++v) {
          cudaLaunchConfig_t cfg = {};
          cfg.gridDim = dim3((unsigned)(sms / 4 * 4));
          cfg.blockDim = dim3(kGemmThreads);
          cfg.dynamicSmemBytes = kGemm2Smem;
          cudaLaunchAttribute at;
          at.id = cudaLaunchAttributeClusterDimension;
          at.val.clusterDim.x = 4; at.val.clusterDim.y = 1; at.val.clusterDim.z = 1;
          cfg.attrs = &at; cfg.numAttrs = 1;
          int n = 0;
          cudaError_t e = v == 0 ? cudaOccupancyMaxActiveClusters(&n, dist_tc4_kernel<256, EPI_DIST>, &cfg)
                                 : cudaOccupancyMaxActiveClusters(&n, dist_tc4_kernel<256, EPI_DIST_TOPK>, &cfg);
          if (e != cudaSuccess) { cudaGetLastError(); n = 0; }
          max_clusters[v] = n;
        }
        cfg4_dev = dev;
      }
      const int mc = max_clusters[topk ? 1 : 0];
      if (mc > 0) {
        ga.g.m_tiles = (int)((m1 + 511) / 512);
        const long long tiles4 = (long long)ga.g.m_tiles * ga.g.n_tiles;
        long long clusters = tiles4 < mc ? tiles4 : mc;
        if ((flags & PPS_DIST_RESERVE_SM_PAIR) && clusters == mc && clusters > 4) clusters -= 1;
        if (topk) {
          dist_tc4_kernel<256, EPI_DIST_TOPK><<<(unsigned)(4 * clusters), kGemmThreads, kGemm2Smem, st>>>(tmA, tmB, tmO, ga, *topk);
          PPS_LAUNCH_CHECK("dist_tc4_kernel<topk>");
        } else {
          dist_tc4_kernel<256, EPI_DIST><<<(unsigned)(4 * clusters), kGemmThreads, kGemm2Smem, st>>>(tmA, tmB, tmO, ga, RankFuse{});
          PPS_LAUNCH_CHECK("dist_tc4_kernel");
        }
        return PPS_OK;
      }
    }
    const long long tiles2 = (long long)ga.g.m_tiles * ga.g.n_tiles;
    long long slots = sms / 2;
    if ((flags & PPS_DIST_RESERVE_SM_PAIR) && slots > 8) slots -= 1;   // leave one SM pair to concurrent small kernels
    const long long pairs = tiles2 < slots ? tiles2 : slots;
    if (topk) {
      static thread_local int configured3_dev = -1;
      if (configured3_dev != dev) {
        PPS_CUDA_TRY(cudaFuncSetAttribute(dist_tc2_kernel<256, EPI_DIST_TOPK>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)kGemm2Smem));
        configured3_dev = dev;
      }
      dist_tc2_kernel<256, EPI_DIST_TOPK><<<(unsigned)(2 * pairs), kGemmThreads, kGemm2Smem, st>>>(tmA, tmB, tmO, ga, *topk);
      PPS_LAUNCH_CHECK("dist_tc2_kernel<topk>");
      return PPS_OK;
    }
    dist_tc2_kernel<256, EPI_DIST><<<(unsigned)(2 * pairs), kGemmThreads, kGemm2Smem, st>>>(tmA, tmB, tmO, ga, RankFuse{});
    PPS_LAUNCH_CHECK("dist_tc2_kernel");
    return PPS_OK;
  }
  if (topk) return PPS_ERR_UNSUPPORTED;        // the admission epilogue exists in the 2-CTA kernel only

  int rc = make_operand_map(&tmA, a_planes, m1, a_plane_rows, kpad, a_planes_n, kBM, f16);
  if (rc) return rc;
  rc = make_operand_map(&tmB, b_planes, m2, b_plane_rows, kpad, b_planes_n, kBN, f16);
  if (rc) return rc;
  static thread_local int configured_dev = -1;
  if (configured_dev != dev) {
    PPS_CUDA_TRY(cudaFuncSetAttribute(dist_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kGemmSmem));
    configured_dev = dev;
  }
  const long long tiles = (long long)g.m_tiles * g.n_tiles;
  const int grid = (int)(tiles < sms ? tiles : sms);
  dist_tc_kernel<<<grid, kGemmThreads, kGemmSmem, st>>>(tmA, tmB, g);
  PPS_LAUNCH_CHECK("dist_tc_kernel");
  return PPS_OK;
}

extern "C" int pps_dist_tc(const void* a_planes, const float* a_sqnorm, long long m1, int a_planes_n,
                           long long a_plane_rows, const void* b_planes, const float* b_sqnorm, long long m2,
                           int b_planes_n, long long b_plane_rows, int dim, int precision, int flags, float* dist,
                           long long ldd, void* stream) {
  return dist_tc_impl(a_planes, a_sqnorm, m1, a_planes_n, a_plane_rows, b_planes, b_sqnorm, m2, b_planes_n, b_plane_rows, dim,
                      precision, flags, dist, ldd, stream, nullptr);
}

// pps_dist_tc + top-k admission in the epilogue: while the block is written, every distance is compared with its
// query's current k-th best (tk_bound) and the few that pass are appended to the query's candidate buffer; a later
// pps_topk_merge folds them into the top-k state.  The block itself is identical to pps_dist_tc's.
extern "C" int pps_dist_topk_tc(const void* a_planes, const float* a_sqnorm, long long m1, int a_planes_n,
                                long long a_plane_rows, const void* b_planes, const float* b_sqnorm, long long m2,
                                int b_planes_n, long long b_plane_rows, int dim, int precision, int flags, float* dist,
                                long long ldd, long long col0, const uint32_t* tk_bound, uint32_t* tk_cnt,
                                uint64_t* tk_cand, int tk_cap, void* stream) {
  if (!tk_bound || !tk_cnt || !tk_cand || tk_cap < 1 || col0 < 0 || col0 + m2 > 0xffffffffLL) return PPS_ERR_INVALID_ARG;
  if (flags & PPS_DIST_DOT) return PPS_ERR_INVALID_ARG;      // keys order by the bits of a non-negative distance
  RankFuse rf{};
  rf.col0 = col0;
  rf.tk_bound = tk_bound; rf.tk_cnt = tk_cnt; rf.tk_cand = reinterpret_cast<unsigned long long*>(tk_cand); rf.tk_cap = tk_cap;
  return dist_tc_impl(a_planes, a_sqnorm, m1, a_planes_n, a_plane_rows, b_planes, b_sqnorm, m2, b_planes_n, b_plane_rows, dim,
                      precision, flags, dist, ldd, stream, &rf);
}

// Top-k admission for a batch of queries against a block of gallery rows, with the roles of pps_dist_topk_tc swapped: the
// gallery is the 256-row M operand and the queries are N = BN in {32, 64, 128, 256} (the smallest that holds the batch;
// larger batches take several query tiles of 256).  A small batch then streams the gallery through the SMs once instead
// of filling a few rows of every 256-row MMA.  Nothing is written but the candidates.
// The exclusion is an instance of its own (EPI_SEARCH_EXCL), so that the untagged kernel keeps its code.
template <int BN, int EPI>
static int launch_search(const CUtensorMap& tmA, const CUtensorMap& tmB, const Gemm2Args& ga, const RankFuse& rf, int dev,
                         long long pairs, cudaStream_t st) {
  static thread_local int configured_dev = -1;
  if (configured_dev != dev) {
    PPS_CUDA_TRY(cudaFuncSetAttribute(dist_tc2_kernel<BN, EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)kGemm2Smem));
    configured_dev = dev;
  }
  dist_tc2_kernel<BN, EPI><<<(unsigned)(2 * pairs), kGemmThreads, kGemm2Smem, st>>>(tmA, tmB, tmA /*no output map*/, ga, rf);
  PPS_LAUNCH_CHECK(EPI == EPI_SEARCH        ? "dist_tc2_kernel<search>"
                   : EPI == EPI_SEARCH_EXCL ? "dist_tc2_kernel<search_excl>"
                   : EPI == EPI_RANGE       ? "dist_tc2_kernel<range>"
                                            : "dist_tc2_kernel<range_excl>");
  return PPS_OK;
}

template <int BN>
static int launch_search(const CUtensorMap& tmA, const CUtensorMap& tmB, const Gemm2Args& ga, const RankFuse& rf, int dev,
                         long long pairs, cudaStream_t st) {
  if (rf.out_off)
    return rf.q_tags ? launch_search<BN, EPI_RANGE_EXCL>(tmA, tmB, ga, rf, dev, pairs, st)
                     : launch_search<BN, EPI_RANGE>(tmA, tmB, ga, rf, dev, pairs, st);
  return rf.q_tags ? launch_search<BN, EPI_SEARCH_EXCL>(tmA, tmB, ga, rf, dev, pairs, st)
                   : launch_search<BN, EPI_SEARCH>(tmA, tmB, ga, rf, dev, pairs, st);
}

// g_tags / q_tags: both null (no exclusion) or both set (pps_search_topk_excl_tc, pps_search_range_tc with tags).
// out_off / out_cap: null (top-k candidates, tk_cand[q][tk_cap]) or both set (range search, tk_cap unused)
static int search_topk_impl(const void* g_planes, const float* g_sqnorm, long long ng, int g_planes_n, long long g_plane_rows,
                            const void* q_planes, const float* q_sqnorm, long long nq, int q_planes_n, long long q_plane_rows,
                            int dim, int precision, int flags, long long col0, const uint32_t* tk_bound, uint32_t* tk_cnt,
                            uint64_t* tk_cand, int tk_cap, const int64_t* g_tags, const int64_t* q_tags, void* stream,
                            const long long* out_off = nullptr, const uint32_t* out_cap = nullptr) {
  if (ng < 0 || nq < 0 || dim <= 0 || col0 < 0 || (!out_off && tk_cap < 1)) return PPS_ERR_INVALID_ARG;
  if (flags & ~(PPS_DIST_SQUARED | PPS_DIST_SQRT_RN)) return PPS_ERR_INVALID_ARG;   // keys order by the bits of a distance
  if (g_plane_rows == 0) g_plane_rows = ng;
  if (q_plane_rows == 0) q_plane_rows = nq;
  if (g_plane_rows < ng || q_plane_rows < nq || col0 + ng > 0xffffffffLL) return PPS_ERR_INVALID_ARG;
  if (ng == 0 || nq == 0) return PPS_OK;
  if (!g_planes || !g_sqnorm || !q_planes || !q_sqnorm || !tk_bound || !tk_cnt || !tk_cand) return PPS_ERR_INVALID_ARG;
  if ((out_off == nullptr) != (out_cap == nullptr)) return PPS_ERR_INVALID_ARG;
  if ((reinterpret_cast<uintptr_t>(g_planes) & 15u) || (reinterpret_cast<uintptr_t>(q_planes) & 15u)) return PPS_ERR_ALIGN;
  if (ng > 0x7fffff00LL || nq > 0x7fffff00LL) return PPS_ERR_UNSUPPORTED;   // TMA coordinates are int32
  GemmArgs terms;
  bool f16 = false;
  const int need = setup_terms(precision, terms, &f16);
  if (need == 0 || g_planes_n < need || q_planes_n < need) return PPS_ERR_INVALID_ARG;
  const int sms = sm_count();
  if (sms < 2) return PPS_ERR_UNSUPPORTED;
  const bool scaled = precision == PPS_PREC_F16X3;
  const int bn = nq <= 32 ? 32 : nq <= 64 ? 64 : nq <= 128 ? 128 : 256;
  const int kpad = pps_kpad(dim);
  const uint32_t fmt = f16 ? 0u : 1u;
  Gemm2Args ga;
  GemmArgs& g = ga.g;
  g.nterms = terms.nterms;
  for (int t = 0; t < terms.nterms; ++t) {     // the same (query plane, gallery plane) products in the same order
    g.term_a[t] = terms.term_b[t];
    g.term_b[t] = terms.term_a[t];
  }
  g.m1 = ng; g.m2 = nq;
  g.kblocks = kpad / kBK;
  g.idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(bn >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
  g.a_sqnorm = g_sqnorm; g.b_sqnorm = q_sqnorm;
  g.a_scale = scaled ? g_sqnorm + g_plane_rows : nullptr;
  g.b_scale = scaled ? q_sqnorm + q_plane_rows : nullptr;
  g.out = nullptr; g.ldo = 0; g.flags = flags;
  static const int env_sqrt = [] { const char* e = getenv("PPS_SQRT_RN"); return e ? atoi(e) : -1; }();   // as pps_dist_tc
  if (env_sqrt >= 0) g.flags = env_sqrt ? (g.flags | PPS_DIST_SQRT_RN) : (g.flags & ~PPS_DIST_SQRT_RN);
  g.m_tiles = (int)((ng + 255) / 256);
  g.n_tiles = (int)((nq + bn - 1) / bn);
  ga.planes = need;
  ga.sep_small = 0;
  ga.stages = kRing2Bytes / (need * (kTile2Bytes + (bn / 2) * kBK * 2));
  if (ga.stages > kMaxStages2) ga.stages = kMaxStages2;
  ga.groups = 1; ga.a_group_rows = 0; ga.b_group_rows = 0; ga.out_group_cols = 0;
  CUtensorMap tmA, tmB;
  int rc = make_operand_map(&tmA, g_planes, ng, g_plane_rows, kpad, g_planes_n, kT2Rows, f16);
  if (rc) return rc;
  rc = make_operand_map(&tmB, q_planes, nq, q_plane_rows, kpad, q_planes_n, bn / 2, f16);
  if (rc) return rc;
  RankFuse rf{};
  rf.col0 = col0;
  rf.tk_bound = tk_bound; rf.tk_cnt = tk_cnt; rf.tk_cand = reinterpret_cast<unsigned long long*>(tk_cand); rf.tk_cap = tk_cap;
  rf.g_tags = reinterpret_cast<const long long*>(g_tags); rf.q_tags = reinterpret_cast<const long long*>(q_tags);
  rf.out_off = out_off; rf.out_cap = out_cap;
  int dev = 0;
  PPS_CUDA_TRY(cudaGetDevice(&dev));
  const long long tiles = (long long)g.m_tiles * g.n_tiles;
  const long long pairs = tiles < sms / 2 ? tiles : sms / 2;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  switch (bn) {
    case 32: return launch_search<32>(tmA, tmB, ga, rf, dev, pairs, st);
    case 64: return launch_search<64>(tmA, tmB, ga, rf, dev, pairs, st);
    case 128: return launch_search<128>(tmA, tmB, ga, rf, dev, pairs, st);
    default: return launch_search<256>(tmA, tmB, ga, rf, dev, pairs, st);
  }
}

extern "C" int pps_search_topk_tc(const void* g_planes, const float* g_sqnorm, long long ng, int g_planes_n,
                                  long long g_plane_rows, const void* q_planes, const float* q_sqnorm, long long nq,
                                  int q_planes_n, long long q_plane_rows, int dim, int precision, int flags, long long col0,
                                  const uint32_t* tk_bound, uint32_t* tk_cnt, uint64_t* tk_cand, int tk_cap, void* stream) {
  return search_topk_impl(g_planes, g_sqnorm, ng, g_planes_n, g_plane_rows, q_planes, q_sqnorm, nq, q_planes_n, q_plane_rows,
                          dim, precision, flags, col0, tk_bound, tk_cnt, tk_cand, tk_cap, nullptr, nullptr, stream);
}

// pps_search_topk_tc without the pairs whose tags are equal: row r of the block is no candidate of query q when
// g_tags[r] == q_tags[q].  The tags are compared only for elements that pass the bound.
extern "C" int pps_search_topk_excl_tc(const void* g_planes, const float* g_sqnorm, long long ng, int g_planes_n,
                                       long long g_plane_rows, const void* q_planes, const float* q_sqnorm, long long nq,
                                       int q_planes_n, long long q_plane_rows, int dim, int precision, int flags,
                                       long long col0, const uint32_t* tk_bound, uint32_t* tk_cnt, uint64_t* tk_cand,
                                       int tk_cap, void* stream, const int64_t* g_tags, const int64_t* q_tags) {
  if (ng > 0 && nq > 0 && (!g_tags || !q_tags)) return PPS_ERR_INVALID_ARG;
  return search_topk_impl(g_planes, g_sqnorm, ng, g_planes_n, g_plane_rows, q_planes, q_sqnorm, nq, q_planes_n, q_plane_rows,
                          dim, precision, flags, col0, tk_bound, tk_cnt, tk_cand, tk_cap, g_tags, q_tags, stream);
}

// Range search: every element whose distance bits are below lim[q] (pps_index_range_search's limit of a radius) is
// appended to out[out_off[q] + slot] while slot < out_cap[q]; cnt[q] counts every hit, also past the capacity.  The
// same kernel as pps_search_topk_tc up to the admission and the address (instances EPI_RANGE / EPI_RANGE_EXCL).
extern "C" int pps_search_range_tc(const void* g_planes, const float* g_sqnorm, long long ng, int g_planes_n,
                                   long long g_plane_rows, const void* q_planes, const float* q_sqnorm, long long nq,
                                   int q_planes_n, long long q_plane_rows, int dim, int precision, int flags, long long col0,
                                   const uint32_t* lim, uint32_t* cnt, const long long* out_off, const uint32_t* out_cap,
                                   uint64_t* out, const int64_t* g_tags, const int64_t* q_tags, void* stream) {
  if ((g_tags == nullptr) != (q_tags == nullptr)) return PPS_ERR_INVALID_ARG;
  if (ng > 0 && nq > 0 && (!out_off || !out_cap)) return PPS_ERR_INVALID_ARG;
  return search_topk_impl(g_planes, g_sqnorm, ng, g_planes_n, g_plane_rows, q_planes, q_sqnorm, nq, q_planes_n, q_plane_rows,
                          dim, precision, flags, col0, lim, cnt, out, 0, g_tags, q_tags, stream, out_off, out_cap);
}

extern "C" int pps_dist_fp32(const float* a, long long lda, const float* a_sqnorm, long long m1, const float* b,
                             long long ldb, const float* b_sqnorm, long long m2, int dim, int flags, float* dist,
                             long long ldd, void* stream) {
  if (m1 < 0 || m2 < 0 || dim <= 0 || lda < dim || ldb < dim || ldd < m2) return PPS_ERR_INVALID_ARG;
  if (m1 == 0 || m2 == 0) return PPS_OK;
  if (!a || !b || !dist) return PPS_ERR_INVALID_ARG;
  if (!(flags & PPS_DIST_DOT) && (!a_sqnorm || !b_sqnorm)) return PPS_ERR_INVALID_ARG;
  const long long gx = (m2 + 63) / 64, gy = (m1 + 63) / 64;
  if (gy > 65535 || gx > 0x7fffffffLL) return PPS_ERR_UNSUPPORTED;
  dist_fp32_kernel<<<dim3((unsigned)gx, (unsigned)gy), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      a, lda, a_sqnorm, m1, b, ldb, b_sqnorm, m2, dim, flags, dist, ldd);
  PPS_LAUNCH_CHECK("dist_fp32_kernel");
  return PPS_OK;
}

// ------------------------------------------------------------------------------------
// Next row (SURVEY §8f.1): the per-combination embedding between pooling and distance
// (detectron/modeling/reid_heads.py:34-76 at test time): for every combination k
//   out[n, k*E + e] = max(0, alpha[k*E+e] * (sum_c pooled[k, n, c] * W[k, e, c]) + beta[k*E+e])
// i.e. Conv1x1(C -> E) + bias + SpatialBN(test: an affine map) + ReLU with the conv bias and the BN statistics
// folded into alpha / beta by the caller, written straight into the concatenated [N, K*E] feature
// (Concat(axis=1), :95-101).  K independent [N, C] x [C, E] products = one grouped launch of the 2-CTA kernel
// (256 x 128 tiles, tcgen05.mma.cta_group::2 with N = 128), same split-precision operands as the distance.
// ------------------------------------------------------------------------------------
extern "C" int pps_embed_tc(const void* x_planes /*[planes][K*N][kpad]*/, int x_planes_n, long long N,
                            const void* w_planes /*[planes][K*E][kpad]*/, int w_planes_n, int E, int K, int C,
                            const float* alpha, const float* beta, int precision, float* out /*[N, ldo >= K*E]*/,
                            long long ldo, void* stream) {
  if (N < 0 || K <= 0 || C <= 0 || E <= 0 || ldo < (long long)K * E) return PPS_ERR_INVALID_ARG;
  if (N == 0) return PPS_OK;
  if (E != 128) return PPS_ERR_UNSUPPORTED;             // cfg.REID.BPM_DIM of every shipped PPS config
  if (!x_planes || !w_planes || !alpha || !beta || !out) return PPS_ERR_INVALID_ARG;
  if ((reinterpret_cast<uintptr_t>(x_planes) & 15u) || (reinterpret_cast<uintptr_t>(w_planes) & 15u)) return PPS_ERR_ALIGN;
  if ((ldo & 3) || (reinterpret_cast<uintptr_t>(out) & 15u)) return PPS_ERR_ALIGN;
  if ((long long)K * N > 0x7fffff00LL) return PPS_ERR_UNSUPPORTED;
  Gemm2Args ga;
  GemmArgs& g = ga.g;
  int need = 1;
  switch (precision) {
    case PPS_PREC_BF16X1: g.nterms = 1; g.term_a[0] = 0; g.term_b[0] = 0; need = 1; break;
    case PPS_PREC_BF16X3: {
      const int ta[3] = {1, 0, 0}, tb[3] = {0, 1, 0};
      g.nterms = 3; for (int i = 0; i < 3; ++i) { g.term_a[i] = ta[i]; g.term_b[i] = tb[i]; }
      need = 2; break;
    }
    case PPS_PREC_BF16X6: {
      const int ta[6] = {2, 0, 1, 1, 0, 0}, tb[6] = {0, 2, 1, 0, 1, 0};
      g.nterms = 6; for (int i = 0; i < 6; ++i) { g.term_a[i] = ta[i]; g.term_b[i] = tb[i]; }
      need = 3; break;
    }
    default: return PPS_ERR_INVALID_ARG;
  }
  if (x_planes_n < need || w_planes_n < need) return PPS_ERR_INVALID_ARG;
  const int kpad = pps_kpad(C);
  g.m1 = N; g.m2 = (long long)K * E;
  g.kblocks = kpad / kBK;
  g.idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(128 >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
  g.a_sqnorm = alpha; g.b_sqnorm = beta;
  g.a_scale = nullptr; g.b_scale = nullptr;
  g.out = out; g.ldo = ldo; g.flags = 0;
  g.m_tiles = (int)((N + 255) / 256);
  g.n_tiles = 1;
  ga.planes = need;
  ga.sep_small = 0;
  ga.stages = kRing2Bytes / (need * (kTile2Bytes + 64 * kBK * 2));
  if (ga.stages > kMaxStages2) ga.stages = kMaxStages2;
  ga.groups = K; ga.a_group_rows = N; ga.b_group_rows = E; ga.out_group_cols = E;

  CUtensorMap tmA, tmB, tmO;
  int rc = make_operand_map(&tmA, x_planes, (long long)K * N, (long long)K * N, kpad, x_planes_n, kT2Rows, false);
  if (rc) return rc;
  rc = make_operand_map(&tmB, w_planes, (long long)K * E, (long long)K * E, kpad, w_planes_n, 64, false);
  if (rc) return rc;
  {
    EncodeTiledFn fn = encode_fn();
    if (!fn) return cuda_fail(cudaErrorUnknown, "cuTensorMapEncodeTiled entry point not found");
    cuuint64_t dims[2] = {(cuuint64_t)((long long)K * E), (cuuint64_t)N};
    cuuint64_t strides[1] = {(cuuint64_t)ldo * 4};
    cuuint32_t box[2] = {32, 32};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(&tmO, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, out, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return cuda_fail(cudaErrorInvalidValue, "cuTensorMapEncodeTiled(output) failed");
  }
  static thread_local int configured_dev = -1;
  int dev = 0;
  PPS_CUDA_TRY(cudaGetDevice(&dev));
  if (configured_dev != dev) {
    PPS_CUDA_TRY(cudaFuncSetAttribute(dist_tc2_kernel<128, EPI_AFFINE_RELU>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)kGemm2Smem));
    configured_dev = dev;
  }
  const int sms = sm_count();
  const long long tiles = (long long)g.m_tiles * K;
  const long long pairs = tiles < sms / 2 ? tiles : sms / 2;
  dist_tc2_kernel<128, EPI_AFFINE_RELU><<<(unsigned)(2 * pairs), kGemmThreads, kGemm2Smem,
                                          static_cast<cudaStream_t>(stream)>>>(tmA, tmB, tmO, ga, RankFuse{});
  PPS_LAUNCH_CHECK("dist_tc2_kernel<embed>");
  return PPS_OK;
}

// ------------------------------------------------------------------------------------
// Distance + ranking counters in one kernel (EPI_RANK): for gallery blocks of a multi-block sweep whose thresholds
// are already known (pps_rank_tab_prep).  The [m1, m2] distance block is never written: the epilogue turns every
// distance into one increment of cnt_tab and, for exact ties with the nearest positive, of cnt_first.
// ------------------------------------------------------------------------------------
extern "C" int pps_dist_rank_topk_tc(const void* a_planes, const float* a_sqnorm, long long m1, int a_planes_n,
                                     long long a_plane_rows, const void* b_planes, const float* b_sqnorm, long long m2,
                                     int b_planes_n, long long b_plane_rows, int dim, int precision, int flags,
                                     long long col0, int p_cap, const float* thr_tab, uint32_t* cnt_tab, const float* dstar,
                                     const int32_t* gstar, uint32_t* cnt_first, const uint32_t* tk_bound, uint32_t* tk_cnt,
                                     uint64_t* tk_cand, int tk_cap, void* stream) {
  if (m1 < 0 || m2 < 0 || dim <= 0 || col0 < 0) return PPS_ERR_INVALID_ARG;
  if (tk_cand && (!tk_bound || !tk_cnt || tk_cap <= 0)) return PPS_ERR_INVALID_ARG;
  if (p_cap < 8 || p_cap > 64 || (p_cap & 7)) return PPS_ERR_INVALID_ARG;
  if (flags & ~PPS_DIST_SQUARED) return PPS_ERR_INVALID_ARG;
  if (a_plane_rows == 0) a_plane_rows = m1;
  if (b_plane_rows == 0) b_plane_rows = m2;
  if (a_plane_rows < m1 || b_plane_rows < m2) return PPS_ERR_INVALID_ARG;
  if (m1 == 0 || m2 == 0) return PPS_OK;
  if (!a_planes || !b_planes || !a_sqnorm || !b_sqnorm || !thr_tab || !cnt_tab || !dstar || !gstar || !cnt_first)
    return PPS_ERR_INVALID_ARG;
  if ((reinterpret_cast<uintptr_t>(a_planes) & 15u) || (reinterpret_cast<uintptr_t>(b_planes) & 15u))
    return PPS_ERR_ALIGN;
  if (m1 > 0x7fffff00LL || m2 > 0x7fffff00LL) return PPS_ERR_UNSUPPORTED;
  Gemm2Args ga;
  GemmArgs& g = ga.g;
  bool f16 = false;
  if (precision == PPS_PREC_F16X3) return PPS_ERR_UNSUPPORTED;   // the counting epilogue has no row-scale path
  const int need = setup_terms(precision, g, &f16);
  if (need == 0 || a_planes_n < need || b_planes_n < need) return PPS_ERR_INVALID_ARG;
  const int sms = sm_count();
  if (sms < 2) return PPS_ERR_UNSUPPORTED;
  const int kpad = pps_kpad(dim);
  const uint32_t fmt = f16 ? 0u : 1u;
  g.m1 = m1; g.m2 = m2;
  g.kblocks = kpad / kBK;
  g.idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(256 >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
  g.a_sqnorm = a_sqnorm; g.b_sqnorm = b_sqnorm;
  g.a_scale = nullptr; g.b_scale = nullptr;
  g.out = nullptr; g.ldo = 0; g.flags = flags;
  g.m_tiles = (int)((m1 + 255) / 256);
  g.n_tiles = (int)((m2 + 255) / 256);
  ga.planes = need;
  ga.sep_small = 0;
  ga.groups = 1; ga.a_group_rows = 0; ga.b_group_rows = 0; ga.out_group_cols = 0;
  // shared memory: ring | thresholds [p_cap][128] f32 | counters [p_cap + 1][128] u32 | |b|^2 [2][256] | barriers
  const int stage_bytes = 2 * need * kTile2Bytes;
  const int tail = p_cap * 1024 + 512 + 2 * 256 * 4 + 256;
  int stages = (227 * 1024 - tail) / stage_bytes;
  if (stages > kMaxStages2) stages = kMaxStages2;
  if (stages < 2) return PPS_ERR_UNSUPPORTED;
  ga.stages = stages;
  const size_t smem = (size_t)stages * stage_bytes + tail;
  CUtensorMap tmA, tmB;
  int rc = make_operand_map(&tmA, a_planes, m1, a_plane_rows, kpad, a_planes_n, kT2Rows, f16);
  if (rc) return rc;
  rc = make_operand_map(&tmB, b_planes, m2, b_plane_rows, kpad, b_planes_n, kT2Rows, f16);
  if (rc) return rc;
  RankFuse rf;
  rf.thr_tab = thr_tab; rf.cnt_tab = cnt_tab; rf.dstar = dstar; rf.gstar = gstar; rf.cnt_first = cnt_first;
  rf.col0 = col0; rf.p_cap = p_cap;
  rf.tk_bound = tk_cand ? tk_bound : nullptr; rf.tk_cnt = tk_cand ? tk_cnt : nullptr;
  rf.tk_cand = reinterpret_cast<unsigned long long*>(tk_cand); rf.tk_cap = tk_cand ? tk_cap : 0;
  rf.progress = nullptr; rf.window = 0;
  rf.g_tags = nullptr; rf.q_tags = nullptr;
  static thread_local int configured_dev = -1;
  int dev = 0;
  PPS_CUDA_TRY(cudaGetDevice(&dev));
  if (configured_dev != dev) {
    PPS_CUDA_TRY(cudaFuncSetAttribute(dist_tc2_kernel<256, EPI_RANK>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      227 * 1024));
    configured_dev = dev;
  }
  const long long tiles = (long long)g.m_tiles * g.n_tiles;
  const long long slots = sms / 2;
  const long long pairs = tiles < slots ? tiles : slots;
  {
    // progress window of the aligned streams (PPS_STREAM_WINDOW = tiles a pair may run ahead of the slowest of its stream)
    static const int window_env = [] { const char* e = std::getenv("PPS_STREAM_WINDOW"); return e ? std::atoi(e) : 0; }();
    static thread_local uint32_t* progress_buf[64] = {};
    if (window_env > 0 && dev >= 0 && dev < 64 && pairs <= 1024) {
      if (!progress_buf[dev]) PPS_CUDA_TRY(cudaMalloc(&progress_buf[dev], 1024 * sizeof(uint32_t)));
      PPS_CUDA_TRY(cudaMemsetAsync(progress_buf[dev], 0, (size_t)pairs * sizeof(uint32_t), static_cast<cudaStream_t>(stream)));
      rf.progress = progress_buf[dev];
      rf.window = window_env;
    }
  }
  dist_tc2_kernel<256, EPI_RANK><<<(unsigned)(2 * pairs), kRankThreads, smem, static_cast<cudaStream_t>(stream)>>>(
      tmA, tmB, tmA /*no output map*/, ga, rf);
  PPS_LAUNCH_CHECK("dist_tc2_kernel<rank>");
  return PPS_OK;
}

extern "C" int pps_dist_rank_tc(const void* a_planes, const float* a_sqnorm, long long m1, int a_planes_n,
                                long long a_plane_rows, const void* b_planes, const float* b_sqnorm, long long m2,
                                int b_planes_n, long long b_plane_rows, int dim, int precision, int flags,
                                long long col0, int p_cap, const float* thr_tab, uint32_t* cnt_tab, const float* dstar,
                                const int32_t* gstar, uint32_t* cnt_first, void* stream) {
  return pps_dist_rank_topk_tc(a_planes, a_sqnorm, m1, a_planes_n, a_plane_rows, b_planes, b_sqnorm, m2, b_planes_n,
                               b_plane_rows, dim, precision, flags, col0, p_cap, thr_tab, cnt_tab, dstar, gstar, cnt_first,
                               nullptr, nullptr, nullptr, 0, stream);
}
