// Ranking without a sort (replaces the two np.argsort calls and the per-query Python loops of
// mean_ap / cmc, reid_dataset_evaluator.py:319-357 and :420-434).
//
// For a query, the only gallery items whose identity matters are the ones with the same
// person id ("pairs": positives = other camera, junk = same camera, :327-328/:427-428).
// Everything the metrics need follows from integer counts against the positives' distances:
//   n_le(p)   = #{gallery j : d(q,j) <= d(q,p)}                         (this file, count kernel)
//   AP(q)     = (1/P) sum_p  #{p' : d_p' <= d_p} / (n_le(p) - #{junk j : d_j <= d_p})
//               == sklearn.metrics.average_precision_score (>= 0.19, tie-grouped step AP)
//   first(q)  = #{valid j ranked before the nearest positive}  -> CMC with first_match_break
// The count kernel is a single HBM-bound sweep of the distance block: per element one
// branch-free binary search into the (<= 63 per pass) sorted positive distances held in shared
// memory and one increment of a lane-private histogram column (bank = lane, so no atomics
// and no conflicts).  It reads no id / camera arrays.  Counters are exact integers: adding
// them across gallery chunks or shards reproduces the unsharded ranking bit for bit.
#include "common.cuh"

#include <cfloat>

namespace pps {

constexpr int kCntThreads = 128;
constexpr int kNB = 1024;           // bins of the per-query distance histogram

// monotone integer key of a float: signed-int order == float order (negative values: flip the low 31 bits)
__device__ __forceinline__ int fkey(float x) {
  const int k = __float_as_int(x);
  return k ^ ((k >> 31) & 0x7fffffff);
}

constexpr int kTopkThreads = 256;
constexpr int kCand = 2048;

__device__ __noinline__ void bitonic_sort_smem(unsigned long long* a, int n /*pow2*/, int tid, int nthreads) {
  for (int k = 2; k <= n; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = tid; i < n; i += nthreads) {
        const int ixj = i ^ j;
        if (ixj > i) {
          const unsigned long long x = a[i], y = a[ixj];
          const bool up = (i & k) == 0;
          if ((x > y) == up) { a[i] = y; a[ixj] = x; }
        }
      }
      __syncthreads();
    }
  }
}

// Keep the k smallest of the n_buf keys in a[] (unused slots hold ~0) WITHOUT sorting: a 32-step bisection on the
// high word (the distance bits) finds the smallest v with #{hi <= v} >= k, every key with hi <= v moves to the front
// (all ties at v included, in no particular order), the rest becomes ~0.  Returns the number kept (same in every
// thread) and sets *bound_out (thread 0) to the largest key that can still enter.  ~1/8 of the instructions of the
// full bitonic sort it replaces.  NPT = n_buf / nthreads keys per thread live in registers.
template <int NPT>
__device__ __noinline__ int select_k_smallest(unsigned long long* a, int k, int tid, int nthreads, int* s_part /*[2][32]*/,
                                                 int* s_cnt, unsigned long long* bound_out) {
  unsigned long long key[NPT];
#pragma unroll
  for (int j = 0; j < NPT; ++j) key[j] = a[tid + j * nthreads];
  const int lane = tid & 31, warp = tid >> 5, nwarps = nthreads >> 5;
  uint32_t lo = 0u, hi = 0xffffffffu;
  int it = 0;
  while (lo < hi) {
    const uint32_t mid = lo + ((hi - lo) >> 1);
    int c = 0;
#pragma unroll
    for (int j = 0; j < NPT; ++j) c += ((uint32_t)(key[j] >> 32) <= mid) ? 1 : 0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    int* part = s_part + (it & 1) * 32;
    if (lane == 0) part[warp] = c;
    __syncthreads();
    int tot = 0;
    for (int w = 0; w < nwarps; ++w) tot += part[w];
    if (tot >= k) hi = mid; else lo = mid + 1;
    ++it;
  }
  if (tid == 0) *s_cnt = 0;
  __syncthreads();                      // every key is in registers: the buffer can be rewritten
#pragma unroll
  for (int j = 0; j < NPT; ++j) a[tid + j * nthreads] = ~0ull;
  __syncthreads();
#pragma unroll
  for (int j = 0; j < NPT; ++j)
    if ((uint32_t)(key[j] >> 32) <= lo && key[j] != ~0ull) a[atomicAdd(s_cnt, 1)] = key[j];
  __syncthreads();
  if (tid == 0) *bound_out = ((unsigned long long)lo << 32) | 0xffffffffull;
  return *s_cnt;
}

// ------------------------------------------------------------------------------------
// step 1: gather the pair distances out of the block
// ------------------------------------------------------------------------------------
__global__ void rank_gather_kernel(const float* __restrict__ dist, long long ldd, long long ncols, long long col0,
                                   const int32_t* __restrict__ pair_q, const int32_t* __restrict__ pair_g,
                                   long long n_pairs, float* __restrict__ pair_d, const int32_t* __restrict__ n_dev) {
  if (n_dev) n_pairs = min(n_pairs, (long long)*n_dev);
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n_pairs;
       e += (long long)gridDim.x * blockDim.x) {
    const int q = pair_q[e];
    if (q < 0) continue;                 // slot of a pair that lives on another gallery shard
    const long long c = (long long)pair_g[e] - col0;
    if (c < 0 || c >= ncols) continue;
    pair_d[e] = dist[(long long)q * ldd + c];
  }
}

// ------------------------------------------------------------------------------------
// step 2: counts.  grid = (nq, splits); CTA (q, s) sweeps columns [s*seg, (s+1)*seg).
//
// n_le(t_p) for all P thresholds of a query in ONE sweep and ~8 instructions per element:
// float bits (low 31 bits flipped for negatives) are monotone integer keys.  The key range
// [key(t_min), key(t_max)] is cut into kNB equal-width bins (shift chosen per query).  Per element:
//   key < key(t_min)  -> a register counter (it lies below every threshold);
//   bin >= kNB        -> beyond every threshold, ignored;
//   else              -> one shared-memory atomicAdd on hist[bin].  Bins that contain a threshold
//                        carry a flag in bit 31 of their counter, which the atomic returns: only
//                        those elements (a few % of a row) take the exact path - a short search
//                        among the thresholds of that bin and one atomicAdd on exact[first + j],
//                        j = #thresholds of the bin below the element.
// Then n_le(t_p) = below + sum of hist over bins before bin(t_p) + sum of exact[] from the bin's
// first threshold up to p.  Integer arithmetic throughout, so partial results add up exactly over
// column splits, gallery chunks and gallery shards.  The first-match counter is not touched per
// element either: with (d*, g*) the nearest positive, first = n_le(d*) - #{d == d*} + #{d == d*,
// col < g*}; exact ties with d* (on the exact path by construction) accumulate the signed correction.
// dynamic smem: thr[maxp] sorted positive distances, tpair[maxp] their pair index, sd/sg[maxp] the
//               staged pair list, exact[maxp]
// ------------------------------------------------------------------------------------
// rare path of the top-k sweep: one column whose distance bits do not exceed the admission bound
__device__ __noinline__ void topk_admit(float d, unsigned long long gcol, unsigned long long bound, const int32_t* sj, int nj,
                                        unsigned long long* cand, int* s_n, int* app_ctr) {
  const unsigned long long ukey = ((unsigned long long)__float_as_uint(d) << 32) | (gcol & 0xffffffffull);
  if (ukey >= bound) return;
  for (int x = 0; x < nj; ++x)
    if ((unsigned long long)(long long)sj[x] == gcol) return;       // junk: same id, same camera
  cand[atomicAdd(s_n, 1)] = ukey;                                    // *s_n <= kCandC - 1024 when a half pass starts
  atomicAdd(app_ctr, 1);
}

// TOPK = true (one CTA per query, no column splits): the same sweep also keeps the query's k nearest valid gallery
// items.  A column is admitted only if its key beats the current k-th best (one compare per element), candidates
// collect in a 2048-entry shared buffer that is re-selected by bitonic sort when it fills; junk items (same id, same
// camera) are skipped through the staged pair list.  One read of the block serves counts and top-k.
constexpr int kCandC = 2048;

template <bool TOPK>
__global__ void __launch_bounds__(kCntThreads, TOPK ? 6 : 16) rank_count_kernel(const float* __restrict__ dist, long long ldd,
                                                                     long long ncols, long long col0, long long seg,
                                                                     const int32_t* __restrict__ pair_off,
                                                                     const int32_t* __restrict__ pair_g,
                                                                     const uint8_t* __restrict__ pair_pos,
                                                                     const float* __restrict__ pair_d, int maxp,
                                                                     uint32_t* __restrict__ cnt_le,
                                                                     uint32_t* __restrict__ cnt_first,
                                                                     unsigned long long* __restrict__ topk_key, int k,
                                                                     int topk_filtered) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* thr = reinterpret_cast<float*>(smem_raw);                          // [maxp]
  int32_t* tpair = reinterpret_cast<int32_t*>(thr + maxp);                  // [maxp]
  float* sd = reinterpret_cast<float*>(tpair + maxp);                       // [maxp] pair distances
  int32_t* sg = reinterpret_cast<int32_t*>(sd + maxp);                      // [maxp] gallery index, -1 = junk
  uint32_t* exact = reinterpret_cast<uint32_t*>(sg + maxp);                 // [maxp]
  int32_t* sj = reinterpret_cast<int32_t*>(exact + maxp);                   // [maxp] junk gallery indices (TOPK)
  __shared__ uint32_t hist[kNB];          // bit 31: the bin holds a threshold
  __shared__ uint32_t binfo[kNB];         // (index of the bin's first threshold << 16) | thresholds in the bin
  __shared__ uint32_t part[kCntThreads];
  __shared__ int s_np, s_nj;
  __shared__ uint32_t s_below, s_first_cnt;
  __shared__ unsigned long long cand[TOPK ? kCandC : 1];
  __shared__ int s_n;
  __shared__ int s_app[3];                // appends of half pass h in s_app[h % 3]
  __shared__ int s_sel[64];               // partial counts of select_k_smallest
  __shared__ unsigned long long s_bound;

  const int q = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31;
  const int e0 = pair_off[q], e1 = pair_off[q + 1];

  // --- positives of this query, rank-sorted by (distance, gallery index) into thr[] ---
  // stage the pair list in shared memory first (coalesced): the O(P^2) ranking must not chase global latency
  if (tid == 0) { s_np = 0; s_nj = 0; s_below = 0; s_first_cnt = 0; }
  const int npair = min(e1 - e0, maxp);       // (maxp may be a speculative bound: a longer list is cut - safely - and the
                                              // caller, who checks the real maximum afterwards, repeats the pass)
  for (int i = tid; i < npair; i += kCntThreads) {
    sd[i] = pair_d[e0 + i];
    sg[i] = pair_pos[e0 + i] ? pair_g[e0 + i] : -1;
  }
  for (int i = tid; i < kNB; i += kCntThreads) { hist[i] = 0; binfo[i] = 0; }
  unsigned long long* state = nullptr;
  if (TOPK) {
    state = topk_key + (long long)q * k;
    for (int i = tid; i < kCandC; i += kCntThreads) cand[i] = i < k ? state[i] : ~0ull;
    if (tid == 0) { s_n = k; s_bound = state[k - 1]; s_app[0] = s_app[1] = s_app[2] = 0; }
  }
  __syncthreads();
  if (TOPK && topk_filtered) {
    for (int i = tid; i < npair; i += kCntThreads)
      if (sg[i] < 0) sj[atomicAdd(&s_nj, 1)] = pair_g[e0 + i];
  }
  for (int i = tid; i < npair; i += kCntThreads) {
    const int g = sg[i];
    if (g < 0) continue;
    const float d = sd[i];
    int pos = 0;
    for (int f = 0; f < npair; ++f) {
      const int gf = sg[f];
      const float df = sd[f];
      pos += (gf >= 0) && ((df < d) || (df == d && gf < g));
    }
    thr[pos] = d;
    tpair[pos] = e0 + i;
    atomicAdd(&s_np, 1);
  }
  __syncthreads();
  const int np = s_np;
  if (!TOPK && np == 0) return;                            // query without a valid match: nothing to count
  const bool count_on = np > 0;                            // (TOPK: the sweep still runs for the nearest items)
  const float dstar = count_on ? thr[0] : 0.f;
  const long long gstar = count_on ? pair_g[tpair[0]] : 0;
  const int key_min = count_on ? fkey(thr[0]) : 0;
  const unsigned key_span = count_on ? (unsigned)fkey(thr[np - 1]) - (unsigned)key_min : 0u;
  int shift = 0;
  while ((key_span >> shift) >= (unsigned)kNB) ++shift;
  const int nj = TOPK ? s_nj : 0;

  const long long c_begin = (long long)blockIdx.y * seg;
  const long long c_end = min(ncols, c_begin + seg);
  if (c_begin >= c_end) return;

  // --- flag the bins that hold thresholds; thresholds are sorted, so a bin's thresholds are contiguous ---
  for (int p = tid; p < np; p += kCntThreads) {
    const unsigned b = ((unsigned)fkey(thr[p]) - (unsigned)key_min) >> shift;
    const bool is_first = (p == 0) || ((((unsigned)fkey(thr[p - 1]) - (unsigned)key_min) >> shift) != b);
    atomicAdd(&binfo[b], 1u + (is_first ? ((uint32_t)p << 16) : 0u));
    if (is_first) hist[b] = 0x80000000u;
    exact[p] = 0;
  }
  __syncthreads();

  const float* drow = dist + (long long)q * ldd;
  const bool vec = ((ldd & 3) == 0) && ((reinterpret_cast<uintptr_t>(dist) & 15u) == 0) && ((c_begin & 3) == 0);
  uint32_t below = 0;                                      // elements under every threshold
  uint32_t tie_corr = 0;                                   // signed: -#{d == d*} + #{d == d*, col < g*}

  unsigned long long bound = ~0ull;                        // TOPK: key of the current k-th best (sampled per half pass)
  int* app_ctr = s_app;                                    // TOPK: this half pass's append counter
  auto visit = [&](float d, long long col) {
    const int key = fkey(d);
    const bool lt = key < key_min;
    below += lt ? 1u : 0u;
    const unsigned b = ((unsigned)key - (unsigned)key_min) >> shift;
    if (count_on && !lt && b < (unsigned)kNB) {
      const uint32_t old = atomicAdd(&hist[b], 1u);
      if (old & 0x80000000u) {                             // the bin holds thresholds: exact comparison
        const uint32_t info = binfo[b];
        const int first = (int)(info >> 16), cnt = (int)(info & 0xffffu);
        int j = 0;
        while (j < cnt && thr[first + j] < d) ++j;
        if (j < cnt) atomicAdd(&exact[first + j], 1u);
        if (d == dstar) tie_corr += ((col0 + col) < gstar ? 1u : 0u) - 1u;
      }
    }
  };

  if (TOPK) {
    // passes of 2048 columns; the loads of the next pass are issued before the current one is consumed, so the stream
    // never drains at the barriers.  After every 1024 columns one barrier: it sums the threads that appended, which
    // bounds the fill of the candidate buffer (<= 8 appends per thread and half pass) identically in every thread.
    constexpr long long kStep = 4LL * kCntThreads;
    float4 v[4], vn[4];
    auto load_pass = [&](long long base, float4 (&dst)[4]) {
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const long long cu = base + u * kStep + 4LL * tid;
        if (vec && cu + 3 < c_end) dst[u] = ld_stream_f4(reinterpret_cast<const float4*>(drow + cu));
      }
    };
    load_pass(c_begin, v);
    int fill = k;                                            // entries in the candidate buffer, the same in every thread
    int hp = 0;                                              // half pass index mod 3
    for (long long base = c_begin; base < c_end; base += 4 * kStep) {
      if (base + 4 * kStep < c_end) load_pass(base + 4 * kStep, vn);
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        bound = s_bound;
        app_ctr = s_app + hp;
#pragma unroll
        for (int uu = 0; uu < 2; ++uu) {
          const int u = 2 * h + uu;
          const long long cu = base + u * kStep + 4LL * tid;
          const uint32_t bh = (uint32_t)(bound >> 32);
          if (vec && cu + 3 < c_end) {
            visit(v[u].x, cu); visit(v[u].y, cu + 1); visit(v[u].z, cu + 2); visit(v[u].w, cu + 3);
            const float dv[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
            if ((__float_as_uint(dv[0]) <= bh) | (__float_as_uint(dv[1]) <= bh) | (__float_as_uint(dv[2]) <= bh) |
                (__float_as_uint(dv[3]) <= bh)) {
#pragma unroll                                               // (a runtime index would put dv[] in local memory)
              for (int e = 0; e < 4; ++e)
                if (__float_as_uint(dv[e]) <= bh)
                  topk_admit(dv[e], (unsigned long long)(col0 + cu + e), bound, sj, nj, cand, &s_n, app_ctr);
            }
          } else {
#pragma unroll 1
            for (int e = 0; e < 4; ++e)
              if (cu + e < c_end) {
                const float d = drow[cu + e];
                visit(d, cu + e);
                if (__float_as_uint(d) <= bh)
                  topk_admit(d, (unsigned long long)(col0 + cu + e), bound, sj, nj, cand, &s_n, app_ctr);
              }
          }
        }
        __syncthreads();
        // s_app[hp] is complete and nobody writes it again before it is reset two half passes from now, so every
        // thread reads the same value without a second barrier
        fill += s_app[hp];
        const int hp_reset = hp == 0 ? 2 : hp - 1;           // the counter half pass h + 2 will use (last read: h - 1)
        if (tid == 0) s_app[hp_reset] = 0;
        hp = hp == 2 ? 0 : hp + 1;
        if (fill > kCandC - 1024) {
          fill = select_k_smallest<kCandC / kCntThreads>(cand, k, tid, kCntThreads, s_sel, &s_n, &s_bound);
          if (fill > kCandC - 1024) {                      // > 1000 exact distance ties at the k-th place: full sort
            bitonic_sort_smem(cand, kCandC, tid, kCntThreads);
            for (int i = k + tid; i < kCandC; i += kCntThreads) cand[i] = ~0ull;
            if (tid == 0) { s_n = k; s_bound = cand[k - 1]; }
            fill = k;
          }
          __syncthreads();
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = vn[u];
    }
    // final state: the k smallest, sorted.  Select first, then sort only what was kept (k plus ties).
    const int kept = select_k_smallest<kCandC / kCntThreads>(cand, k, tid, kCntThreads, s_sel, &s_n, &s_bound);
    __syncthreads();
    if (kept <= 256) bitonic_sort_smem(cand, 256, tid, kCntThreads);
    else bitonic_sort_smem(cand, kCandC, tid, kCntThreads);
    for (int i = tid; i < k; i += kCntThreads) state[i] = cand[i];
    if (!count_on) return;                                 // uniform: no positives, only the top-k was wanted
  } else if (vec) {
    const long long c4_end = c_begin + ((c_end - c_begin) & ~3LL);
    constexpr long long kStep = 4LL * kCntThreads;         // columns per pass of the CTA
    long long c = c_begin + 4LL * tid;
    // four independent 128-bit loads in flight per thread before any of them is consumed
    for (; c + 3 * kStep < c4_end; c += 4 * kStep) {
      float4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = ld_stream_f4(reinterpret_cast<const float4*>(drow + c + u * kStep));
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const long long cu = c + u * kStep;
        visit(v[u].x, cu); visit(v[u].y, cu + 1); visit(v[u].z, cu + 2); visit(v[u].w, cu + 3);
      }
    }
    for (; c < c4_end; c += kStep) {
      const float4 v = ld_stream_f4(reinterpret_cast<const float4*>(drow + c));
      visit(v.x, c); visit(v.y, c + 1); visit(v.z, c + 2); visit(v.w, c + 3);
    }
    for (c = c4_end + tid; c < c_end; c += kCntThreads) visit(drow[c], c);
  } else {
    for (long long c = c_begin + tid; c < c_end; c += kCntThreads) visit(drow[c], c);
  }

  // --- reductions: below, tie correction, exclusive prefix of the histogram ---
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    below += __shfl_xor_sync(0xffffffffu, below, o);
    tie_corr += __shfl_xor_sync(0xffffffffu, tie_corr, o);
  }
  if (lane == 0) {
    if (below) atomicAdd(&s_below, below);
    if (tie_corr) atomicAdd(&s_first_cnt, tie_corr);
  }
  __syncthreads();
  constexpr int kPer = kNB / kCntThreads;                  // 8 consecutive bins per thread
  uint32_t local[kPer], sum = 0;
#pragma unroll
  for (int k = 0; k < kPer; ++k) {
    local[k] = hist[tid * kPer + k] & 0x7fffffffu;
    sum += local[k];
  }
  part[tid] = sum;
  __syncthreads();
  if (tid < 32) {                                          // scan of the 128 per-thread sums by one warp
    uint32_t v[4], run = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) { v[k] = part[tid * 4 + k]; run += v[k]; }
    uint32_t incl = run;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    uint32_t excl = incl - run;
#pragma unroll
    for (int k = 0; k < 4; ++k) { part[tid * 4 + k] = excl; excl += v[k]; }
  }
  __syncthreads();
  {
    uint32_t run = part[tid];
#pragma unroll
    for (int k = 0; k < kPer; ++k) { hist[tid * kPer + k] = run; run += local[k]; }   // hist := exclusive prefix
  }
  __syncthreads();
  const uint32_t below_all = s_below;
  for (int p = tid; p < np; p += kCntThreads) {
    const unsigned b = ((unsigned)fkey(thr[p]) - (unsigned)key_min) >> shift;
    const int first = (int)(binfo[b] >> 16);
    uint32_t n = below_all + hist[b];
    for (int k = first; k <= p; ++k) n += exact[k];
    if (n) atomicAdd(&cnt_le[tpair[p]], n);
  }
  if (tid == 0 && s_first_cnt) atomicAdd(&cnt_first[q], s_first_cnt);
}

// ------------------------------------------------------------------------------------
// step 3: finalize (one warp per query; pair lists are short)
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) rank_finalize_kernel(long long nq, const int32_t* __restrict__ pair_off,
                                                            const int32_t* __restrict__ pair_g,
                                                            const uint8_t* __restrict__ pair_pos,
                                                            const float* __restrict__ pair_d,
                                                            const uint32_t* __restrict__ cnt_le,
                                                            const uint32_t* __restrict__ cnt_first,
                                                            double* __restrict__ ap, uint8_t* __restrict__ is_valid,
                                                            int32_t* __restrict__ first_rank,
                                                            int32_t* __restrict__ neg_before) {
  const int lane = threadIdx.x & 31;
  const long long q = (long long)blockIdx.x * 4 + (threadIdx.x >> 5);
  if (q >= nq) return;
  const int e0 = pair_off[q], e1 = pair_off[q + 1];
  double acc = 0.0;
  int np = 0;
  float dstar = FLT_MAX;
  int gstar = 0x7fffffff;
  uint32_t le_star = 0;        // cnt_le of the nearest positive (ties by gallery index)
  for (int e = e0 + lane; e < e1; e += 32) {
    if (!pair_pos[e]) continue;
    const float d = pair_d[e];
    const int g = pair_g[e];
    int c_pos = 0, c_junk = 0;
    for (int f = e0; f < e1; ++f) {
      const bool le = pair_d[f] <= d;
      if (pair_pos[f]) c_pos += le; else c_junk += le;
    }
    const int n_valid = (int)cnt_le[e] - c_junk;           // valid items with d <= d_p (includes p)
    acc += (double)c_pos / (double)n_valid;
    if (neg_before) neg_before[e] = n_valid - c_pos;
    ++np;
    if (d < dstar || (d == dstar && g < gstar)) { dstar = d; gstar = g; le_star = cnt_le[e]; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    acc += __shfl_xor_sync(0xffffffffu, acc, o);
    np += __shfl_xor_sync(0xffffffffu, np, o);
    const float od = __shfl_xor_sync(0xffffffffu, dstar, o);
    const int og = __shfl_xor_sync(0xffffffffu, gstar, o);
    const uint32_t ol = __shfl_xor_sync(0xffffffffu, le_star, o);
    if (od < dstar || (od == dstar && og < gstar)) { dstar = od; gstar = og; le_star = ol; }
  }
  // junk items ranked before the nearest positive
  int jb = 0;
  if (np > 0) {
    for (int e = e0 + lane; e < e1; e += 32) {
      if (pair_pos[e]) continue;
      const float d = pair_d[e];
      jb += (d < dstar) || (d == dstar && pair_g[e] < gstar);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) jb += __shfl_xor_sync(0xffffffffu, jb, o);
  }
  if (lane == 0) {
    ap[q] = np > 0 ? acc / (double)np : 0.0;
    is_valid[q] = np > 0 ? 1 : 0;
    // #{(d, g) < (d*, g*)} = #{d <= d*} - #{d == d*} + #{d == d*, g < g*}; cnt_first holds the last two (mod 2^32)
    first_rank[q] = np > 0 ? (int32_t)(le_star + cnt_first[q]) - jb : -1;
  }
}

// ------------------------------------------------------------------------------------
// top-k: one CTA per query keeps <= 2048 candidate keys in shared memory, admits a column
// only if its key beats the current k-th best, and re-selects by bitonic sort when full.
// key = (float bits << 32) | global gallery index: unsigned order == (distance, index) order
// for the non-negative distances this path produces.
// ------------------------------------------------------------------------------------
// TAGS (a separate instance, so that the untagged sweep keeps its registers and occupancy): column c is skipped when
// g_tags[c] == q_tags[q].  The tag is compared at admission only, unless the excluded columns are counted (n_tag_excl
// set): then every column's tag is read.
template <bool TAGS>
__global__ void __launch_bounds__(kTopkThreads) topk_update_kernel(const float* __restrict__ dist, long long ldd,
                                                                    long long ncols, long long col0,
                                                                    const int32_t* __restrict__ excl_off,
                                                                    const int32_t* __restrict__ excl_g,
                                                                    const uint8_t* __restrict__ excl_keep,
                                                                    const long long* __restrict__ g_tags,
                                                                    const long long* __restrict__ q_tags,
                                                                    uint32_t* __restrict__ n_tag_excl,
                                                                    unsigned long long* __restrict__ topk_key, int k) {
  __shared__ unsigned long long cand[kCand];
  __shared__ int s_n;
  __shared__ unsigned long long s_bound;
  __shared__ uint32_t s_excl;
  const int q = blockIdx.x, tid = threadIdx.x;
  unsigned long long* state = topk_key + (long long)q * k;
  for (int i = tid; i < kCand; i += kTopkThreads) cand[i] = i < k ? state[i] : ~0ull;
  if (tid == 0) { s_n = k; s_bound = state[k - 1]; if (TAGS) s_excl = 0u; }
  __syncthreads();
  const float* drow = dist + (long long)q * ldd;
  const int x0 = excl_off ? excl_off[q] : 0, x1 = excl_off ? excl_off[q + 1] : 0;
  const long long qtag = TAGS ? q_tags[q] : 0;
  uint32_t n_tx = 0;
  const long long tile = 4LL * kTopkThreads;
  for (long long c0 = 0; c0 < ncols; c0 += tile) {
    const unsigned long long bound = s_bound;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const long long c = c0 + (long long)u * kTopkThreads + tid;
      if (c < ncols) {
        const float d = ld_stream_f32(drow + c);
        const unsigned long long key = ((unsigned long long)__float_as_uint(d) << 32) | (unsigned long long)(uint32_t)(col0 + c);
        bool tag_out = false;
        if (TAGS && n_tag_excl) {
          tag_out = __ldg(g_tags + c) == qtag;
          n_tx += tag_out;
        }
        if (key < bound) {
          if (TAGS && !n_tag_excl) tag_out = __ldg(g_tags + c) == qtag;
          bool skip = tag_out;
          for (int x = x0; x < x1; ++x)
            skip |= ((long long)excl_g[x] == col0 + c) && !(excl_keep && excl_keep[x]);
          if (!skip) {
            const int slot = atomicAdd(&s_n, 1);
            cand[slot] = key;        // s_n <= kCand - tile at tile start, so slot < kCand
          }
        }
      }
    }
    __syncthreads();
    const int n_now = s_n;
    __syncthreads();           // every thread has sampled s_n before anyone appends again
    if (n_now > kCand - (int)tile) {
      bitonic_sort_smem(cand, kCand, tid, kTopkThreads);
      for (int i = k + tid; i < kCand; i += kTopkThreads) cand[i] = ~0ull;
      if (tid == 0) { s_n = k; s_bound = cand[k - 1]; }
      __syncthreads();
    }
  }
  bitonic_sort_smem(cand, kCand, tid, kTopkThreads);
  for (int i = tid; i < k; i += kTopkThreads) state[i] = cand[i];
  if (TAGS && n_tag_excl) {
    if (n_tx) atomicAdd(&s_excl, n_tx);
    __syncthreads();
    if (tid == 0) n_tag_excl[q] = s_excl;
  }
}

__global__ void topk_fill_kernel(unsigned long long* p, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = ~0ull;
}

__global__ void topk_unpack_kernel(const unsigned long long* __restrict__ key, long long n, float* __restrict__ od,
                                   int32_t* __restrict__ oi) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const unsigned long long kk = key[i];
  const bool none = kk == ~0ull;
  if (od) od[i] = none ? __int_as_float(0x7f800000) : __uint_as_float((uint32_t)(kk >> 32));
  if (oi) oi[i] = none ? -1 : (int32_t)(uint32_t)(kk & 0xffffffffu);
}

// ------------------------------------------------------------------------------------
// Tables for the fused ranking epilogue of the distance kernel (dist_gemm.cu, EPI_RANK).
// Row groups of 128 queries; element (group, j, r) at ((group * p_cap) + j) * 128 + r:
//   thr_tab   j-th smallest positive distance of query 128*group + r (ties by gallery index), +inf beyond the last
//   tpair_tab its pair index, -1 beyond the last
//   cnt_tab   zeroed here; the epilogue adds #{columns with exactly j thresholds below them}
// so that n_le(threshold j) = cnt_tab[0] + ... + cnt_tab[j]   (rank_tab_finish_kernel).
// One warp per query; rows up to the next multiple of 256 are padded.
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) rank_tab_prep_kernel(long long nq, long long rows_pad,
                                                            const int32_t* __restrict__ pair_off,
                                                            const int32_t* __restrict__ pair_g,
                                                            const uint8_t* __restrict__ pair_pos,
                                                            const float* __restrict__ pair_d, int p_cap,
                                                            float* __restrict__ thr_tab, int32_t* __restrict__ tpair_tab,
                                                            uint32_t* __restrict__ cnt_tab, float* __restrict__ dstar,
                                                            int32_t* __restrict__ gstar, int* __restrict__ overflow) {
  const int lane = threadIdx.x & 31;
  const long long q = (long long)blockIdx.x * 4 + (threadIdx.x >> 5);
  if (q >= rows_pad) return;
  const long long base = ((q >> 7) * p_cap) * 128 + (q & 127);
  for (int j = lane; j < p_cap; j += 32) {
    thr_tab[base + (long long)j * 128] = __int_as_float(0x7f800000);
    tpair_tab[base + (long long)j * 128] = -1;
    cnt_tab[base + (long long)j * 128] = 0u;
  }
  __syncwarp();
  if (q >= nq) return;
  const int e0 = pair_off[q], e1 = pair_off[q + 1];
  int np = 0;
  for (int e = e0 + lane; e < e1; e += 32) {
    if (!pair_pos[e]) continue;
    const float d = pair_d[e];
    const int g = pair_g[e];
    int pos = 0;
    for (int f = e0; f < e1; ++f) {
      const float df = pair_d[f];
      pos += pair_pos[f] && ((df < d) || (df == d && pair_g[f] < g));
    }
    if (pos < p_cap) {
      thr_tab[base + (long long)pos * 128] = d;
      tpair_tab[base + (long long)pos * 128] = e;
    }
    if (pos == 0) { dstar[q] = d; gstar[q] = g; }
    ++np;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) np += __shfl_xor_sync(0xffffffffu, np, o);
  if (lane == 0) {
    if (np == 0) { dstar[q] = __int_as_float(0x7fc00000); gstar[q] = 0; }
    if (np > p_cap) atomicAdd(overflow, 1);
  }
}

__global__ void __launch_bounds__(128) rank_tab_finish_kernel(long long nq, int p_cap, const int32_t* __restrict__ tpair_tab,
                                                              const uint32_t* __restrict__ cnt_tab,
                                                              uint32_t* __restrict__ cnt_le) {
  const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= nq) return;
  const long long base = ((q >> 7) * p_cap) * 128 + (q & 127);
  uint32_t run = 0;
  for (int j = 0; j < p_cap; ++j) {
    const int e = tpair_tab[base + (long long)j * 128];
    if (e < 0) break;
    run += cnt_tab[base + (long long)j * 128];
    cnt_le[e] += run;
  }
}

// ------------------------------------------------------------------------------------
// Top-k candidates admitted by the distance kernel's epilogue (dist_gemm.cu, EPI_DIST_TOPK) -> top-k state.
// One CTA per query: state (k sorted keys) + the query's candidate buffer go through the same 2048-entry shared
// buffer and bisection select as the sweep kernel; junk items (same id, same camera) are dropped here.  Writes the
// new state, the new admission bound and resets the candidate count; a buffer that overflowed raises *overflow
// (the caller then repeats the pass with the one-read sweep).
// ------------------------------------------------------------------------------------
__global__ void topk_bound_kernel(const unsigned long long* __restrict__ key, long long nq, int k,
                                  uint32_t* __restrict__ tk_bound, uint32_t* __restrict__ tk_cnt) {
  const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= nq) return;
  const unsigned long long kk = key[q * k + k - 1];
  tk_bound[q] = kk == ~0ull ? 0xffffffffu : (uint32_t)(kk >> 32);
  tk_cnt[q] = 0u;
}

__global__ void __launch_bounds__(kCntThreads) topk_merge_kernel(unsigned long long* __restrict__ topk_key, int k,
                                                                 const unsigned long long* __restrict__ tk_cand, int tk_cap,
                                                                 uint32_t* __restrict__ tk_cnt, uint32_t* __restrict__ tk_bound,
                                                                 const int32_t* __restrict__ pair_off,
                                                                 const int32_t* __restrict__ pair_g,
                                                                 const uint8_t* __restrict__ pair_pos, int filtered,
                                                                 int* __restrict__ overflow, int sj_cap) {
  extern __shared__ int32_t sj_dyn[];                    // junk gallery indices of this query
  __shared__ unsigned long long cand[kCandC];
  __shared__ int s_n, s_nj;
  __shared__ int s_sel[64];
  __shared__ unsigned long long s_bound;
  const int q = blockIdx.x, tid = threadIdx.x;
  unsigned long long* state = topk_key + (long long)q * k;
  const uint32_t raw = tk_cnt[q];
  if (raw == 0u) return;                                 // nothing was admitted for this query in the block
  if (raw > (uint32_t)tk_cap && tid == 0) atomicExch(overflow, 1);
  const int cnt = raw < (uint32_t)tk_cap ? (int)raw : tk_cap;
  for (int i = tid; i < kCandC; i += kCntThreads) cand[i] = i < k ? state[i] : ~0ull;
  if (tid == 0) { s_n = k; s_nj = 0; }
  __syncthreads();
  if (filtered && pair_off) {
    const int e0 = pair_off[q], e1 = pair_off[q + 1];
    for (int e = e0 + tid; e < e1; e += kCntThreads)
      if (!pair_pos[e]) {
        const int slot = atomicAdd(&s_nj, 1);
        if (slot < sj_cap) sj_dyn[slot] = pair_g[e];       // (sj_cap may be a speculative bound, see rank_count_kernel)
      }
  }
  __syncthreads();
  const int nj = min(s_nj, sj_cap);
  const unsigned long long* src = tk_cand + (long long)q * tk_cap;
  int fill = k;
  for (int base = 0; base < cnt;) {
    const int take = min(cnt - base, kCandC - fill);
    for (int i = tid; i < take; i += kCntThreads) {
      const unsigned long long key = src[base + i];
      const long long gcol = (long long)(key & 0xffffffffull);
      bool skip = false;
      for (int x = 0; x < nj; ++x) skip |= ((long long)sj_dyn[x] == gcol);
      if (!skip) cand[atomicAdd(&s_n, 1)] = key;
    }
    base += take;
    __syncthreads();
    fill = select_k_smallest<kCandC / kCntThreads>(cand, k, tid, kCntThreads, s_sel, &s_n, &s_bound);
    if (fill > kCandC - 1024) {                          // > 1000 exact ties at the k-th place: full sort, keep k
      bitonic_sort_smem(cand, kCandC, tid, kCntThreads);
      for (int i = k + tid; i < kCandC; i += kCntThreads) cand[i] = ~0ull;
      if (tid == 0) s_n = k;
      fill = k;
    }
    __syncthreads();
  }
  if (fill <= 256) bitonic_sort_smem(cand, 256, tid, kCntThreads);
  else bitonic_sort_smem(cand, kCandC, tid, kCntThreads);
  for (int i = tid; i < k; i += kCntThreads) state[i] = cand[i];
  if (tid == 0) {
    const unsigned long long kk = cand[k - 1];
    tk_bound[q] = kk == ~0ull ? 0xffffffffu : (uint32_t)(kk >> 32);
    tk_cnt[q] = 0u;
  }
}

// ------------------------------------------------------------------------------------
// Secondary metric: AP as scikit-learn 0.18.1 defined it (the version reid_dataset_evaluator.py:398-407 asks for):
// area under the precision-recall curve by the trapezoidal rule.  From counts, with v the distinct positive distances:
//   AP = sum_v (tp(v) - tp(<v)) / P * ( tp(v) / n_le(v) + P_prev(v) ) / 2,
//   P_prev(v) = tp(<v) / n_lt(v) if n_lt(v) > 0 else 1        (the curve's prepended (recall 0, precision 1) point)
// n_lt = n_le - n_eq needs, besides the <=-counts of the main sweep, the number of items at EXACTLY each pair's
// distance: rank_count_eq_kernel (a second, unhurried pass over the block; only run when this metric is asked for).
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) rank_count_eq_kernel(const float* __restrict__ dist, long long ldd, long long ncols,
                                                            const int32_t* __restrict__ pair_off,
                                                            const float* __restrict__ pair_d, int maxp,
                                                            uint32_t* __restrict__ cnt_eq) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* sd = reinterpret_cast<float*>(smem_raw);                  // [maxp]
  uint32_t* se = reinterpret_cast<uint32_t*>(sd + maxp);           // [maxp]
  __shared__ float s_min, s_max;
  const int q = blockIdx.x, tid = threadIdx.x;
  const int e0 = pair_off[q], np = pair_off[q + 1] - e0;
  if (np == 0) return;
  for (int i = tid; i < np; i += blockDim.x) { sd[i] = pair_d[e0 + i]; se[i] = 0u; }
  __syncthreads();
  if (tid == 0) {
    float mn = sd[0], mx = sd[0];
    for (int i = 1; i < np; ++i) { mn = fminf(mn, sd[i]); mx = fmaxf(mx, sd[i]); }
    s_min = mn; s_max = mx;
  }
  __syncthreads();
  const float mn = s_min, mx = s_max;
  const float* drow = dist + (long long)q * ldd;
  for (long long c = tid; c < ncols; c += blockDim.x) {
    const float d = drow[c];
    if (d < mn || d > mx) continue;
    for (int i = 0; i < np; ++i)
      if (sd[i] == d) atomicAdd(&se[i], 1u);
  }
  __syncthreads();
  for (int i = tid; i < np; i += blockDim.x)
    if (se[i]) atomicAdd(&cnt_eq[e0 + i], se[i]);
}

__global__ void __launch_bounds__(128) rank_finalize_trapezoid_kernel(long long nq, const int32_t* __restrict__ pair_off,
                                                                      const int32_t* __restrict__ pair_g,
                                                                      const uint8_t* __restrict__ pair_pos,
                                                                      const float* __restrict__ pair_d,
                                                                      const uint32_t* __restrict__ cnt_le,
                                                                      const uint32_t* __restrict__ cnt_eq,
                                                                      double* __restrict__ ap) {
  const int lane = threadIdx.x & 31;
  const long long q = (long long)blockIdx.x * 4 + (threadIdx.x >> 5);
  if (q >= nq) return;
  const int e0 = pair_off[q], e1 = pair_off[q + 1];
  double acc = 0.0;
  int npos = 0;
  for (int e = e0 + lane; e < e1; e += 32) {
    if (!pair_pos[e]) continue;
    ++npos;
    const float d = pair_d[e];
    int tp = 0, tp_lt = 0, junk_le = 0, junk_eq = 0;
    bool rep = true;                         // one term per distinct positive distance: its lowest pair index
    for (int f = e0; f < e1; ++f) {
      const float df = pair_d[f];
      if (pair_pos[f]) {
        tp += df <= d;
        tp_lt += df < d;
        rep &= !(df == d && f < e);
      } else {
        junk_le += df <= d;
        junk_eq += df == d;
      }
    }
    if (!rep) continue;
    const double n_le = (double)((int)cnt_le[e] - junk_le);
    const double n_lt = n_le - (double)((int)cnt_eq[e] - junk_eq);
    const double p_prev = n_lt > 0.0 ? (double)tp_lt / n_lt : 1.0;
    acc += (double)(tp - tp_lt) * ((double)tp / n_le + p_prev) * 0.5;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    acc += __shfl_xor_sync(0xffffffffu, acc, o);
    npos += __shfl_xor_sync(0xffffffffu, npos, o);
  }
  if (lane == 0) ap[q] = npos > 0 ? acc / (double)npos : 0.0;
  (void)pair_g;
}

}  // namespace pps

using namespace pps;

namespace pps {
int rank_gather_ex(const float* dist, long long ldd, long long nq, long long ncols, long long col0, const int32_t* pair_q,
                   const int32_t* pair_g, long long n_pairs, float* pair_d, void* stream, const int32_t* n_dev) {
  if (nq < 0 || ncols < 0 || n_pairs < 0 || ldd < ncols) return PPS_ERR_INVALID_ARG;
  if (n_pairs == 0 || ncols == 0 || nq == 0) return PPS_OK;
  if (!dist || !pair_q || !pair_g || !pair_d) return PPS_ERR_INVALID_ARG;
  const long long blocks = (n_pairs + 255) / 256;
  if (blocks > 0x7fffffffLL) return PPS_ERR_UNSUPPORTED;
  rank_gather_kernel<<<(unsigned)blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(dist, ldd, ncols, col0, pair_q,
                                                                                      pair_g, n_pairs, pair_d, n_dev);
  PPS_LAUNCH_CHECK("rank_gather_kernel");
  return PPS_OK;
}
}  // namespace pps

extern "C" int pps_rank_gather(const float* dist, long long ldd, long long nq, long long ncols, long long col0,
                               const int32_t* pair_q, const int32_t* pair_g, long long n_pairs, float* pair_d,
                               void* stream) {
  return rank_gather_ex(dist, ldd, nq, ncols, col0, pair_q, pair_g, n_pairs, pair_d, stream, nullptr);
}

static int rank_count_launch(const float* dist, long long ldd, long long nq, long long ncols, long long col0,
                             const int32_t* pair_off, const int32_t* pair_g, const uint8_t* pair_pos,
                             const float* pair_d, int max_pairs_per_query, uint32_t* cnt_le, uint32_t* cnt_first,
                             unsigned long long* topk_key, int k, int topk_filtered, void* stream) {
  const bool topk = topk_key != nullptr;
  const int maxp = ((max_pairs_per_query > 0 ? max_pairs_per_query : 1) + 3) & ~3;
  const size_t smem = (size_t)maxp * 24;                      // thr, tpair, staged distances / indices, exact, junk
  if (smem > 150 * 1024) return PPS_ERR_UNSUPPORTED;          // > ~6k same-id items for one query
  // column splits: enough CTAs to fill the GPU when there are few queries (not with top-k: one CTA owns a query's state)
  const int sms = sm_count();
  long long splits = 1;
  if (!topk && nq < 4LL * sms) splits = (4LL * sms + nq - 1) / nq;
  long long seg = (ncols + splits - 1) / splits;
  seg = (seg + 1023) & ~1023LL;                               // keeps 16-byte alignment of segment starts
  splits = (ncols + seg - 1) / seg;
  if (splits > 65535) return PPS_ERR_UNSUPPORTED;
  static thread_local int configured_dev = -1;
  int dev = 0;
  PPS_CUDA_TRY(cudaGetDevice(&dev));
  if (configured_dev != dev) {
    PPS_CUDA_TRY(cudaFuncSetAttribute(rank_count_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 150 * 1024));
    PPS_CUDA_TRY(cudaFuncSetAttribute(rank_count_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 150 * 1024));
    configured_dev = dev;
  }
  const dim3 grid((unsigned)nq, (unsigned)splits);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (topk)
    rank_count_kernel<true><<<grid, kCntThreads, smem, st>>>(dist, ldd, ncols, col0, seg, pair_off, pair_g, pair_pos,
                                                             pair_d, maxp, cnt_le, cnt_first, topk_key, k, topk_filtered);
  else
    rank_count_kernel<false><<<grid, kCntThreads, smem, st>>>(dist, ldd, ncols, col0, seg, pair_off, pair_g, pair_pos,
                                                              pair_d, maxp, cnt_le, cnt_first, nullptr, 0, 0);
  PPS_LAUNCH_CHECK("rank_count_kernel");
  return PPS_OK;
}

extern "C" int pps_rank_count(const float* dist, long long ldd, long long nq, long long ncols, long long col0,
                              const int32_t* pair_off, const int32_t* pair_g, const uint8_t* pair_pos,
                              const float* pair_d, int max_pairs_per_query, uint32_t* cnt_le, uint32_t* cnt_first,
                              void* stream) {
  if (nq < 0 || ncols < 0 || ldd < ncols || max_pairs_per_query < 0) return PPS_ERR_INVALID_ARG;
  if (nq == 0 || ncols == 0) return PPS_OK;
  if (!dist || !pair_off || !cnt_first) return PPS_ERR_INVALID_ARG;
  if (max_pairs_per_query == 0) return PPS_OK;               // no query has any same-id gallery item
  if (!pair_g || !pair_pos || !pair_d || !cnt_le) return PPS_ERR_INVALID_ARG;
  if (nq > 0x7fffffffLL) return PPS_ERR_UNSUPPORTED;
  return rank_count_launch(dist, ldd, nq, ncols, col0, pair_off, pair_g, pair_pos, pair_d, max_pairs_per_query, cnt_le,
                           cnt_first, nullptr, 0, 0, stream);
}

// counts + first-match counter + valid-filtered top-k in ONE read of the block
extern "C" int pps_rank_sweep(const float* dist, long long ldd, long long nq, long long ncols, long long col0,
                              const int32_t* pair_off, const int32_t* pair_g, const uint8_t* pair_pos,
                              const float* pair_d, int max_pairs_per_query, uint32_t* cnt_le, uint32_t* cnt_first,
                              uint64_t* topk_key, int k, int topk_filtered, void* stream) {
  if (nq < 0 || ncols < 0 || ldd < ncols || max_pairs_per_query < 0 || k < 1 || k > PPS_TOPK_MAX) return PPS_ERR_INVALID_ARG;
  if (nq == 0 || ncols == 0) return PPS_OK;
  if (!dist || !pair_off || !cnt_first || !topk_key) return PPS_ERR_INVALID_ARG;
  if (max_pairs_per_query > 0 && (!pair_g || !pair_pos || !pair_d || !cnt_le)) return PPS_ERR_INVALID_ARG;
  if (nq > 0x7fffffffLL || col0 + ncols > 0xffffffffLL) return PPS_ERR_UNSUPPORTED;
  return rank_count_launch(dist, ldd, nq, ncols, col0, pair_off, pair_g, pair_pos, pair_d, max_pairs_per_query, cnt_le,
                           cnt_first, reinterpret_cast<unsigned long long*>(topk_key), k, topk_filtered, stream);
}

extern "C" int pps_rank_finalize(long long nq, const int32_t* pair_off, const int32_t* pair_g, const uint8_t* pair_pos,
                                 const float* pair_d, const uint32_t* cnt_le, const uint32_t* cnt_first, double* ap,
                                 uint8_t* is_valid, int32_t* first_rank, int32_t* neg_before, void* stream) {
  if (nq < 0) return PPS_ERR_INVALID_ARG;
  if (nq == 0) return PPS_OK;
  if (!pair_off || !cnt_first || !ap || !is_valid || !first_rank) return PPS_ERR_INVALID_ARG;
  const long long blocks = (nq + 3) / 4;
  if (blocks > 0x7fffffffLL) return PPS_ERR_UNSUPPORTED;
  rank_finalize_kernel<<<(unsigned)blocks, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      nq, pair_off, pair_g, pair_pos, pair_d, cnt_le, cnt_first, ap, is_valid, first_rank, neg_before);
  PPS_LAUNCH_CHECK("rank_finalize_kernel");
  return PPS_OK;
}

extern "C" int pps_topk_init(uint64_t* topk_key, long long nq, int k, void* stream) {
  if (nq < 0 || k < 1 || k > PPS_TOPK_MAX) return PPS_ERR_INVALID_ARG;
  if (nq == 0) return PPS_OK;
  if (!topk_key) return PPS_ERR_INVALID_ARG;
  const long long n = nq * k, blocks = (n + 255) / 256;
  topk_fill_kernel<<<(unsigned)blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<unsigned long long*>(topk_key), n);
  PPS_LAUNCH_CHECK("topk_fill_kernel");
  return PPS_OK;
}

extern "C" int pps_topk_update(const float* dist, long long ldd, long long nq, long long ncols, long long col0,
                               const int32_t* excl_off, const int32_t* excl_g, const uint8_t* excl_keep,
                               uint64_t* topk_key, int k, void* stream) {
  if (nq < 0 || ncols < 0 || ldd < ncols || k < 1 || k > PPS_TOPK_MAX) return PPS_ERR_INVALID_ARG;
  if (nq == 0 || ncols == 0) return PPS_OK;
  if (!dist || !topk_key) return PPS_ERR_INVALID_ARG;
  if (excl_off && !excl_g) return PPS_ERR_INVALID_ARG;
  if (nq > 0x7fffffffLL || col0 + ncols > 0xffffffffLL) return PPS_ERR_UNSUPPORTED;
  topk_update_kernel<false><<<(unsigned)nq, kTopkThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      dist, ldd, ncols, col0, excl_off, excl_g, excl_keep, nullptr, nullptr, nullptr,
      reinterpret_cast<unsigned long long*>(topk_key), k);
  PPS_LAUNCH_CHECK("topk_update_kernel");
  return PPS_OK;
}

extern "C" int pps_topk_update_excl(const float* dist, long long ldd, long long nq, long long ncols, long long col0,
                                    const int64_t* g_tags, const int64_t* q_tags, uint64_t* topk_key, int k,
                                    uint32_t* n_excluded, void* stream) {
  if (nq < 0 || ncols < 0 || ldd < ncols || k < 1 || k > PPS_TOPK_MAX) return PPS_ERR_INVALID_ARG;
  if (nq == 0) return PPS_OK;
  if (!topk_key || !q_tags || (ncols > 0 && (!dist || !g_tags))) return PPS_ERR_INVALID_ARG;
  if (nq > 0x7fffffffLL || col0 + ncols > 0xffffffffLL) return PPS_ERR_UNSUPPORTED;
  if (ncols == 0) {
    if (n_excluded) PPS_CUDA_TRY(cudaMemsetAsync(n_excluded, 0, (size_t)nq * sizeof(uint32_t), static_cast<cudaStream_t>(stream)));
    return PPS_OK;
  }
  topk_update_kernel<true><<<(unsigned)nq, kTopkThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      dist, ldd, ncols, col0, nullptr, nullptr, nullptr, reinterpret_cast<const long long*>(g_tags),
      reinterpret_cast<const long long*>(q_tags), n_excluded, reinterpret_cast<unsigned long long*>(topk_key), k);
  PPS_LAUNCH_CHECK("topk_update_kernel<excl>");
  return PPS_OK;
}

extern "C" int pps_topk_unpack(const uint64_t* topk_key, long long nq, int k, float* out_dist, int32_t* out_index,
                               void* stream) {
  if (nq < 0 || k < 1 || k > PPS_TOPK_MAX) return PPS_ERR_INVALID_ARG;
  if (nq == 0) return PPS_OK;
  if (!topk_key) return PPS_ERR_INVALID_ARG;
  const long long n = nq * k, blocks = (n + 255) / 256;
  topk_unpack_kernel<<<(unsigned)blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const unsigned long long*>(topk_key), n, out_dist, out_index);
  PPS_LAUNCH_CHECK("topk_unpack_kernel");
  return PPS_OK;
}

// ---- tables of the fused ranking epilogue (pps_dist_rank_tc) ----
extern "C" long long pps_rank_tab_elems(long long nq, int p_cap) {
  if (nq < 0 || p_cap < 8 || p_cap > 64 || (p_cap & 7)) return PPS_ERR_INVALID_ARG;
  const long long rows_pad = (nq + 255) / 256 * 256;
  return rows_pad * p_cap;
}

extern "C" int pps_rank_tab_prep(long long nq, const int32_t* pair_off, const int32_t* pair_g, const uint8_t* pair_pos,
                                 const float* pair_d, int p_cap, float* thr_tab, int32_t* tpair_tab, uint32_t* cnt_tab,
                                 float* dstar, int32_t* gstar, int32_t* overflow, void* stream) {
  if (nq < 0 || p_cap < 8 || p_cap > 64 || (p_cap & 7)) return PPS_ERR_INVALID_ARG;
  if (nq == 0) return PPS_OK;
  if (!pair_off || !thr_tab || !tpair_tab || !cnt_tab || !dstar || !gstar || !overflow) return PPS_ERR_INVALID_ARG;
  const long long rows_pad = (nq + 255) / 256 * 256;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  PPS_CUDA_TRY(cudaMemsetAsync(overflow, 0, 4, st));
  rank_tab_prep_kernel<<<(unsigned)(rows_pad / 4), 128, 0, st>>>(nq, rows_pad, pair_off, pair_g, pair_pos, pair_d, p_cap,
                                                                thr_tab, tpair_tab, cnt_tab, dstar, gstar, overflow);
  PPS_LAUNCH_CHECK("rank_tab_prep_kernel");
  return PPS_OK;
}

extern "C" int pps_rank_tab_finish(long long nq, int p_cap, const int32_t* tpair_tab, const uint32_t* cnt_tab,
                                   uint32_t* cnt_le, void* stream) {
  if (nq < 0 || p_cap < 8 || p_cap > 64 || (p_cap & 7)) return PPS_ERR_INVALID_ARG;
  if (nq == 0) return PPS_OK;
  if (!tpair_tab || !cnt_tab || !cnt_le) return PPS_ERR_INVALID_ARG;
  rank_tab_finish_kernel<<<(unsigned)((nq + 127) / 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(nq, p_cap, tpair_tab,
                                                                                                      cnt_tab, cnt_le);
  PPS_LAUNCH_CHECK("rank_tab_finish_kernel");
  return PPS_OK;
}

// ---- top-k admission in the distance epilogue (pps_dist_topk_tc): bound initialisation and candidate merge ----
extern "C" int pps_topk_bound(const uint64_t* topk_key, long long nq, int k, uint32_t* tk_bound, uint32_t* tk_cnt,
                              void* stream) {
  if (nq < 0 || k < 1 || k > PPS_TOPK_MAX) return PPS_ERR_INVALID_ARG;
  if (nq == 0) return PPS_OK;
  if (!topk_key || !tk_bound || !tk_cnt) return PPS_ERR_INVALID_ARG;
  topk_bound_kernel<<<(unsigned)((nq + 127) / 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const unsigned long long*>(topk_key), nq, k, tk_bound, tk_cnt);
  PPS_LAUNCH_CHECK("topk_bound_kernel");
  return PPS_OK;
}

extern "C" int pps_topk_merge(uint64_t* topk_key, long long nq, int k, const uint64_t* tk_cand, int tk_cap,
                              uint32_t* tk_cnt, uint32_t* tk_bound, const int32_t* pair_off, const int32_t* pair_g,
                              const uint8_t* pair_pos, int max_pairs_per_query, int topk_filtered, int32_t* overflow,
                              void* stream) {
  if (nq < 0 || k < 1 || k > PPS_TOPK_MAX || tk_cap < 1 || max_pairs_per_query < 0) return PPS_ERR_INVALID_ARG;
  if (nq == 0) return PPS_OK;
  if (!topk_key || !tk_cand || !tk_cnt || !tk_bound || !overflow) return PPS_ERR_INVALID_ARG;
  if (nq > 0x7fffffffLL) return PPS_ERR_UNSUPPORTED;
  const bool filt = topk_filtered && max_pairs_per_query > 0;
  if (filt && (!pair_off || !pair_g || !pair_pos)) return PPS_ERR_INVALID_ARG;
  const size_t smem = (size_t)(max_pairs_per_query > 0 ? max_pairs_per_query : 1) * 4;
  if (smem > 100 * 1024) return PPS_ERR_UNSUPPORTED;
  static thread_local int configured_dev = -1;
  int dev = 0;
  PPS_CUDA_TRY(cudaGetDevice(&dev));
  if (configured_dev != dev) {
    PPS_CUDA_TRY(cudaFuncSetAttribute(topk_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    configured_dev = dev;
  }
  topk_merge_kernel<<<(unsigned)nq, kCntThreads, smem, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<unsigned long long*>(topk_key), k, reinterpret_cast<const unsigned long long*>(tk_cand), tk_cap, tk_cnt,
      tk_bound, filt ? pair_off : nullptr, pair_g, pair_pos, filt ? 1 : 0, overflow,
      max_pairs_per_query > 0 ? max_pairs_per_query : 1);
  PPS_LAUNCH_CHECK("topk_merge_kernel");
  return PPS_OK;
}

// ---- secondary metric: trapezoidal AP (scikit-learn 0.18.1) ----
extern "C" int pps_rank_count_eq(const float* dist, long long ldd, long long nq, long long ncols, const int32_t* pair_off,
                                 const float* pair_d, int max_pairs_per_query, uint32_t* cnt_eq, void* stream) {
  if (nq < 0 || ncols < 0 || ldd < ncols || max_pairs_per_query < 0) return PPS_ERR_INVALID_ARG;
  if (nq == 0 || ncols == 0 || max_pairs_per_query == 0) return PPS_OK;
  if (!dist || !pair_off || !pair_d || !cnt_eq) return PPS_ERR_INVALID_ARG;
  if (nq > 0x7fffffffLL) return PPS_ERR_UNSUPPORTED;
  const size_t smem = (size_t)max_pairs_per_query * 8;
  if (smem > 150 * 1024) return PPS_ERR_UNSUPPORTED;
  static thread_local int configured_dev = -1;
  int dev = 0;
  PPS_CUDA_TRY(cudaGetDevice(&dev));
  if (configured_dev != dev) {
    PPS_CUDA_TRY(cudaFuncSetAttribute(rank_count_eq_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 150 * 1024));
    configured_dev = dev;
  }
  rank_count_eq_kernel<<<(unsigned)nq, 256, smem, static_cast<cudaStream_t>(stream)>>>(dist, ldd, ncols, pair_off, pair_d,
                                                                                      max_pairs_per_query, cnt_eq);
  PPS_LAUNCH_CHECK("rank_count_eq_kernel");
  return PPS_OK;
}

extern "C" int pps_rank_finalize_trapezoid(long long nq, const int32_t* pair_off, const int32_t* pair_g,
                                           const uint8_t* pair_pos, const float* pair_d, const uint32_t* cnt_le,
                                           const uint32_t* cnt_eq, double* ap, void* stream) {
  if (nq < 0) return PPS_ERR_INVALID_ARG;
  if (nq == 0) return PPS_OK;
  if (!pair_off || !ap) return PPS_ERR_INVALID_ARG;
  const long long blocks = (nq + 3) / 4;
  if (blocks > 0x7fffffffLL) return PPS_ERR_UNSUPPORTED;
  rank_finalize_trapezoid_kernel<<<(unsigned)blocks, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      nq, pair_off, pair_g, pair_pos, pair_d, cnt_le, cnt_eq, ap);
  PPS_LAUNCH_CHECK("rank_finalize_trapezoid_kernel");
  return PPS_OK;
}
