// Argument blocks and the persistent tile schedule of the tensor-core distance kernels (dist_gemm.cu).  In a header of its
// own so that the test-only library (test_hooks.cu) can replay the schedule on the host without the product ABI
// exporting any instrumentation.
#pragma once

#include "common.cuh"

namespace pps {

constexpr int kMaxTerms = 6;

struct GemmArgs {
  long long m1, m2;
  int kblocks;                // ceil(K / 64)
  int nterms;
  int term_a[kMaxTerms];      // plane of A used by term t
  int term_b[kMaxTerms];
  uint32_t idesc;
  const float* a_sqnorm;
  const float* b_sqnorm;
  const float* a_scale;       // PPS_PREC_F16X3: inverse power-of-two row scales of the operands (else nullptr)
  const float* b_scale;
  float* out;
  long long ldo;
  int flags;
  int m_tiles, n_tiles;
};

struct Gemm2Args {
  GemmArgs g;
  int planes;       // planes of each operand loaded per k-block (1..3)
  int sep_small;    // 1: the cross terms (every term but p0.p0) accumulate in a TMEM buffer of their own (see dist_gemm.cu)
  int stages;       // ring depth = ring bytes / stage bytes
  // grouped form (embedding head): `groups` independent products; group grp uses A rows [grp*a_group_rows, ...),
  // B rows [grp*b_group_rows, ...) and writes output columns [grp*out_group_cols, ...).  Distance: groups = 1.
  int groups;
  long long a_group_rows, b_group_rows, out_group_cols;
};

// Fused ranking epilogue (EPI_RANK): the distance tile never leaves the SM.  Per element one lower-bound search
// among the row's sorted positive distances (shared memory, [threshold][row] so that bank = row for every
// thread whatever it searches) and one increment of a thread-private 16-bit histogram counter.
struct RankFuse {
  const float* thr_tab;     // [row groups of 128][p_cap][128] ascending positive distances of each query, +inf padded
  uint32_t* cnt_tab;        // same shape: #{columns whose lower bound among the row's thresholds is j}
  const float* dstar;       // [rows] nearest positive distance (NaN: the query has no positive)
  const int32_t* gstar;     // [rows] its global gallery index
  uint32_t* cnt_first;      // [rows] += -#{d == d*} + #{d == d*, column < g*}   (mod 2^32)
  long long col0;           // global gallery index of column 0 of this block
  int p_cap;                // thresholds per row in the tables (multiple of 8, <= 64)
  // EPI_DIST_TOPK: admission of top-k candidates while the distance block is being written
  const uint32_t* tk_bound; // [rows] distance bits of the current k-th best of each query (0xffffffff: unbounded)
  uint32_t* tk_cnt;         // [rows] candidates appended so far (may run past tk_cap: the excess is dropped and detected)
  unsigned long long* tk_cand;   // [rows][tk_cap] keys (distance bits << 32 | global gallery index)
  int tk_cap;
  // EPI_RANK, balanced walk: progress window between the CTA pairs of an aligned stream (same n range, different m tiles).
  // Nothing else keeps them in step; once they drift apart by more than their share of L2 every pair fetches the B tiles
  // from DRAM again (measured: 4.6x the operands).  progress[pair] = n tiles whose loads the pair has issued (0xffffffff:
  // done); a producer starts tile j only when j <= min over its stream + window.  window = 0: off.
  uint32_t* progress;
  int window;
  // EPI_SEARCH_EXCL: row r of the block is no candidate of query q when g_tags[r] == q_tags[q]
  const long long* g_tags;  // [rows of the block]
  const long long* q_tags;  // [queries]
};

constexpr int EPI_DIST = 0;          // |a|^2 + |b|^2 - 2ab, clamp, sqrt (or squared / raw dot by flags) -> matrix
constexpr int EPI_AFFINE_RELU = 1;   // max(0, dot * alpha[col] + beta[col])   (a_sqnorm = alpha, b_sqnorm = beta)
constexpr int EPI_RANK = 2;          // distance as EPI_DIST, consumed by the counting epilogue; no matrix
constexpr int EPI_DIST_TOPK = 3;     // EPI_DIST + one compare per element against the row's top-k admission bound
constexpr int EPI_SEARCH = 4;        // A = gallery, B = queries: distance -> top-k admission per COLUMN; no matrix
constexpr int EPI_SEARCH_EXCL = 5;   // EPI_SEARCH without the (row, query) pairs whose tags are equal
__host__ __device__ constexpr bool epi_search(int epi) { return epi == EPI_SEARCH || epi == EPI_SEARCH_EXCL; }

// Tile order.  EPI_DIST / EPI_AFFINE_RELU: tile t = pair, pair + npairs, ... with the m index fastest, so that the
// CTA pairs running concurrently share B tiles in L2.  EPI_SEARCH(_EXCL): the same tiles with the n index fastest, so that a
// gallery (m) tile is read from HBM once and its other query tiles find it in L2.  EPI_RANK: a CTA pair keeps ONE m tile per run (its rows'
// thresholds and counters stay in shared memory) and walks a contiguous range of n tiles.
//   npairs >= m_tiles: k = npairs / m_tiles pairs per m tile walk n tiles [0, Na) in k aligned parts - the pairs that own
//     the other m tiles walk the same n range at the same pace, which keeps the L2 sharing of B - and the X = npairs % m_tiles
//     pairs left over share the columns [Na, n_tiles) of ALL m tiles (m-major, a few runs each); Na = n_tiles * k * m_tiles /
//     npairs makes every pair's tile count equal to within one run's rounding.  (Round 1 gave the X pairs to X of the m
//     tiles: 6 owners against 5 at 14 m tiles x 74 pairs, 5.7 % of the kernel lost to the imbalance.)
//   npairs < m_tiles: the schedule repeats per "superblock" of npairs m tiles, remainders as in round 1.
template <int EPI>
struct TileWalk {
  long long t, tiles, tiles_per_group, npairs, pair;
  int m_tiles, n_tiles;
  int sb, n_sb, n_cur, n_stop;
  // balanced EPI_RANK schedule (npairs >= m_tiles)
  bool balanced, extra;
  int stream_i;                 // aligned pairs: index of the n range this pair walks (its peers: pairs stream_i * m_tiles + m)
  int n_first, n_a, n_b;
  long long lin_cur, lin_first, lin_stop;
  // outputs
  long long grp;
  int m_tile, n_tile;
  bool run_start, run_end;

  __host__ __device__ TileWalk(const Gemm2Args& ga, long long pair_, long long npairs_) {
    pair = pair_; npairs = npairs_;
    m_tiles = ga.g.m_tiles; n_tiles = ga.g.n_tiles;
    tiles_per_group = (long long)m_tiles * n_tiles;
    tiles = tiles_per_group * ga.groups;
    t = pair - npairs;
    sb = -1; n_sb = (int)((m_tiles + npairs - 1) / npairs); n_cur = 0; n_stop = 0;
    grp = 0; m_tile = 0; n_tile = 0; run_start = run_end = false;
    balanced = false; extra = false; stream_i = 0; n_first = 0; n_a = n_tiles; n_b = 0; lin_cur = lin_first = lin_stop = 0;
    if (EPI == EPI_RANK && m_tiles > 0 && npairs >= m_tiles) {
      balanced = true;
      const long long k = npairs / m_tiles, aligned = k * m_tiles, x = npairs - aligned;
      n_a = x == 0 ? n_tiles : (int)(((long long)n_tiles * aligned + npairs - 1) / npairs);
      n_b = n_tiles - n_a;
      if (pair < aligned) {
        m_tile = (int)(pair % m_tiles);
        const long long i = pair / m_tiles;
        stream_i = (int)i;
        n_first = n_cur = (int)((long long)n_a * i / k);
        n_stop = (int)((long long)n_a * (i + 1) / k);
      } else {
        extra = true;
        const long long e = pair - aligned, total = (long long)m_tiles * n_b;
        lin_first = lin_cur = total * e / x;
        lin_stop = total * (e + 1) / x;
      }
    }
  }
  __host__ __device__ bool next() {
    if (EPI != EPI_RANK) {
      t += npairs;
      if (t >= tiles) return false;
      grp = t / tiles_per_group;
      const long long tt = t % tiles_per_group;
      if (epi_search(EPI)) {
        m_tile = (int)(tt / n_tiles);
        n_tile = (int)(tt % n_tiles);
      } else {
        m_tile = (int)(tt % m_tiles);
        n_tile = (int)(tt / m_tiles);
      }
      return true;
    }
    if (balanced) {
      if (!extra) {
        if (n_cur >= n_stop) return false;
        run_start = n_cur == n_first;
        n_tile = n_cur++;
        run_end = n_cur >= n_stop;
        return true;
      }
      if (lin_cur >= lin_stop) return false;
      m_tile = (int)(lin_cur / n_b);
      n_tile = n_a + (int)(lin_cur % n_b);
      run_start = lin_cur == lin_first || n_tile == n_a;
      ++lin_cur;
      run_end = lin_cur >= lin_stop || n_tile == n_tiles - 1;
      return true;
    }
    run_start = false;
    while (n_cur >= n_stop) {                     // next superblock with a non-empty range for this pair
      if (++sb >= n_sb) return false;
      const long long m0 = (long long)sb * npairs;
      const long long mt = (m_tiles - m0) < npairs ? (m_tiles - m0) : npairs;
      const long long ml = pair % mt, i = pair / mt;
      const long long owners = npairs / mt + (ml < npairs % mt ? 1 : 0);
      m_tile = (int)(m0 + ml);
      n_cur = (int)((long long)n_tiles * i / owners);
      n_stop = (int)((long long)n_tiles * (i + 1) / owners);
      run_start = true;
    }
    n_tile = n_cur++;
    run_end = n_cur >= n_stop;
    return true;
  }
};

}  // namespace pps
