// Resident gallery index (include/pps_b200.h part 2h): the gallery is split into operand planes once, when rows are added,
// and every search runs on those planes:
//   1. split the queries (scratch of the index)
//   2. prefix: the first F = min(size, 32768) rows as a materialised [nq, F] block (pps_dist_tc), swept by pps_topk_update;
//      pps_topk_bound derives the first admission bound
//   3. chunks: pps_search_topk_tc over the next R rows (the gallery is the M operand, nothing written but candidates), then
//      pps_topk_merge, which also tightens the bound.  Rows in random order admit about k * R / F_done candidates per query,
//      so R = cap * F_done / (2.2 k) (the rule of plan_blocks) keeps the buffers well under cap: chunks grow ~9x each
//      (cap 2048, k 100) and 10 M rows take 3-4 launches.
//   4. one 4-byte read-back of the overflow flag; when a buffer ran over (an adversarial row order) the search is repeated
//      with materialised blocks and pps_topk_update only.
// The keys are built in the caller's d_keys directly.
//
// Tagged rows (pps_index_add_tagged, pps_index_search_excluding): one int64 tag per row, indexed by local row.  An
// excluding search runs the same schedule with the excluding variant of every kernel, so excluded rows never become
// candidates.  A query whose excluded rows fill a fraction f of the prefix got its bound from F (1 - f) rows, and a chunk
// of rows it may all take admits up to k R / (F (1 - f)): the prefix sweep counts each query's excluded rows, one 4-byte
// read-back gives the largest count, and the chunks shrink by (1 - f^), f^ <= 0.9.
//
// Removal (pps_index_remove) compacts the rows in place, with np.delete's renumbering:
//   1. mark: one byte per row (rm_flag), set for every listed row; out-of-range rows are counted, the first removed row
//      is an atomicMin.  Block sums of the flags, one block scans them (exclusive offsets + the number removed), and one
//      12-byte read-back {out of range, removed, first} is the call's only synchronisation.
//   2. kept list: the live rows of [first, size) in order (int32), from the scanned offsets.
//   3. move, in pieces [j0, j1) of the kept list: gather rows kept[j0..j1) of every plane, their norms / inverse scales
//      and tags into the piece buffer, then cudaMemcpyAsync it to rows [first + j0, first + j1).  kept[j] >= first + j,
//      so a piece's destinations overlap only its own sources (already in the buffer) or earlier pieces' (already read).
// The moved rows are the bytes a fresh add of the remaining rows would have written (the split is per row), so every
// later search equals a fresh index's bit for bit.
//
// Range search (pps_index_range_search): radius -> per-query limit, one pps_search_range_tc over every row into uniform
// slices, a scan of the counts into lims and one 16-byte read-back {total, largest count}; a second pass straight into
// the lims layout only when a slice ran over.  The segment sort (pps_sort_key_segments) compacts the slices and sorts
// each query's keys: tiles of 4 096 keys in shared memory, then merge passes of aligned runs, all sized by the total.
#include "ctx.cuh"

namespace {

using pps::GrowBuf;
using pps::PinBuf;

constexpr long long kPrefixRows = 32768;
constexpr int kTkCap = 2048;
constexpr int kGroupTkCap = 8192;     // grouped search: candidates per query and chunk (DESIGN §4.16)
constexpr long long kMinCapacity = 1024;
constexpr long long kMaxIndex = 0x7fffffffLL;   // keys carry the gallery index in 32 bits, unpacked as int32

struct DeviceGuard {          // every call runs on the index's device and leaves the caller's current device as it was
  int prev = -1;
  cudaError_t err = cudaSuccess;
  explicit DeviceGuard(int dev) {
    err = cudaGetDevice(&prev);
    if (err == cudaSuccess && prev != dev) err = cudaSetDevice(dev);
  }
  ~DeviceGuard() {
    int cur = -1;
    if (prev >= 0 && cudaGetDevice(&cur) == cudaSuccess && cur != prev) cudaSetDevice(prev);
  }
};

}  // namespace

struct pps_index {
  int device = 0, dim = 0, kpad = 0, dtype = 0, precision = 0, planes = 0, split_planes = 0;
  long long size = 0, capacity = 0;
  void* g_planes = nullptr;     // [planes][capacity][kpad] 16-bit elements
  float* g_norm = nullptr;      // [capacity] norms (+ [capacity] inverse scales for PPS_PREC_F16X3)
  int64_t* g_tags = nullptr;    // [capacity] row tags (tagged indexes)
  int64_t* g_groups = nullptr;  // [capacity] row groups (grouped indexes)
  bool tagged = false;          // decided by the first non-empty add
  bool grouped = false;         // decided by the first non-empty add
  GrowBuf qs, qn, dist, tk_bound, tk_cnt, tk_cand, flag, n_excl;
  GrowBuf rm_flag, rm_bsum, rm_stat, rm_kept, rm_piece;    // scratch of pps_index_remove
  GrowBuf rg_lim, rg_cnt, rg_off, rg_cap, rg_slices, rg_stat, rg_keys, rg_tmp;   // scratch of pps_index_range_search
  long long rg_total = 0;       // keys of the last range search (in rg_keys)
  long long rg_slice = 4096;    // first-pass slice per query: a power of two >= the largest count seen so far
  long long last_prefix = 0, last_chunks = 0;   // schedule of the last grouped search (pps_index_group_stats)
  int last_fallback = 0;
  PinBuf flag_h;
  bool scaled() const { return precision == PPS_PREC_F16X3; }
  size_t plane_bytes(long long rows) const { return (size_t)rows * kpad * 2; }
  const void* planes_at(long long row) const { return static_cast<const unsigned char*>(g_planes) + plane_bytes(row); }
};

namespace {

// capacity -> new_cap: planes, both halves of the norm array, the tags and the groups move to their new offsets
int grow(pps_index* x, long long need, cudaStream_t st) {
  long long cap = std::max(x->capacity * 2, std::max(need, kMinCapacity));
  if (cap > kMaxIndex) cap = kMaxIndex;
  void* planes = nullptr;
  float* norm = nullptr;
  int64_t* tags = nullptr;
  int64_t* groups = nullptr;
  const size_t norm_n = (size_t)cap * (x->scaled() ? 2 : 1);
  cudaError_t e = cudaMalloc(&planes, (size_t)x->planes * x->plane_bytes(cap));
  if (e == cudaSuccess) e = cudaMalloc(&norm, norm_n * sizeof(float));
  if (e == cudaSuccess && x->tagged) e = cudaMalloc(&tags, (size_t)cap * sizeof(int64_t));
  if (e == cudaSuccess && x->grouped) e = cudaMalloc(&groups, (size_t)cap * sizeof(int64_t));
  if (e != cudaSuccess) {
    if (planes) cudaFree(planes);
    if (norm) cudaFree(norm);
    if (tags) cudaFree(tags);
    return pps::cuda_fail(e, "cudaMalloc(index)");
  }
  if (x->size > 0) {
    for (int p = 0; p < x->planes; ++p)
      PPS_CUDA_TRY(cudaMemcpyAsync(static_cast<unsigned char*>(planes) + p * x->plane_bytes(cap),
                                   static_cast<const unsigned char*>(x->g_planes) + p * x->plane_bytes(x->capacity),
                                   x->plane_bytes(x->size), cudaMemcpyDeviceToDevice, st));
    PPS_CUDA_TRY(cudaMemcpyAsync(norm, x->g_norm, (size_t)x->size * sizeof(float), cudaMemcpyDeviceToDevice, st));
    if (x->scaled())
      PPS_CUDA_TRY(cudaMemcpyAsync(norm + cap, x->g_norm + x->capacity, (size_t)x->size * sizeof(float),
                                   cudaMemcpyDeviceToDevice, st));
    if (tags)
      PPS_CUDA_TRY(cudaMemcpyAsync(tags, x->g_tags, (size_t)x->size * sizeof(int64_t), cudaMemcpyDeviceToDevice, st));
    if (groups)
      PPS_CUDA_TRY(cudaMemcpyAsync(groups, x->g_groups, (size_t)x->size * sizeof(int64_t), cudaMemcpyDeviceToDevice, st));
    PPS_CUDA_TRY(cudaStreamSynchronize(st));     // the old buffers are read until here
  }
  if (x->g_planes) cudaFree(x->g_planes);
  if (x->g_norm) cudaFree(x->g_norm);
  if (x->g_tags) cudaFree(x->g_tags);
  if (x->g_groups) cudaFree(x->g_groups);
  x->g_planes = planes;
  x->g_norm = norm;
  x->g_tags = tags;
  x->g_groups = groups;
  x->capacity = cap;
  return PPS_OK;
}

// materialised block: distances of the queries to rows [r0, r0 + rows), swept into the top-k state (q_tags: without
// the rows whose tag is the query's; n_excl: their count per query)
int block_update(pps_index* x, long long nq, long long r0, long long rows, long long ldd, long long index_offset, int k,
                 uint64_t* keys, const int64_t* q_tags, uint32_t* n_excl, cudaStream_t st) {
  PPS_TRY(pps_dist_tc(x->qs.p, x->qn.as<float>(), nq, x->planes, 0, x->planes_at(r0), x->g_norm + r0, rows, x->planes,
                      x->capacity, x->dim, x->precision, 0, x->dist.as<float>(), ldd, st));
  if (q_tags)
    return pps_topk_update_excl(x->dist.as<float>(), ldd, nq, rows, index_offset + r0, x->g_tags + r0, q_tags, keys, k, n_excl,
                                st);
  return pps_topk_update(x->dist.as<float>(), ldd, nq, rows, index_offset + r0, nullptr, nullptr, nullptr, keys, k, st);
}

__global__ void max_u32_kernel(const uint32_t* __restrict__ v, long long n, uint32_t* __restrict__ out) {
  __shared__ uint32_t s_max;
  if (threadIdx.x == 0) s_max = 0u;
  __syncthreads();
  uint32_t m = 0u;
  for (long long i = threadIdx.x; i < n; i += blockDim.x) m = max(m, v[i]);
  atomicMax(&s_max, m);
  __syncthreads();
  if (threadIdx.x == 0) *out = s_max;
}

// ---- removal (pps_index_remove) ----
constexpr int kRmThreads = 256;
constexpr int kRmTile = kRmThreads * 16;            // rows per block of the flag scan: 16 one-byte flags per thread
constexpr size_t kRmPieceBytes = 256ull << 20;      // the piece buffer of the move
constexpr unsigned long long kRmNone = ~0ull;

// exclusive prefix of v over the block (blockDim.x a multiple of 32, <= 1024) and the block's total
template <class T>
__device__ __forceinline__ T block_excl_scan(T v, T* s_warp, T* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  T x = v;
  for (int o = 1; o < 32; o <<= 1) {
    const T y = __shfl_up_sync(~0u, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) s_warp[warp] = x;
  __syncthreads();
  if (warp == 0) {
    T w = lane < nw ? s_warp[lane] : T(0);
    for (int o = 1; o < 32; o <<= 1) {
      const T y = __shfl_up_sync(~0u, w, o);
      if (lane >= o) w += y;
    }
    s_warp[lane] = w;
  }
  __syncthreads();
  *total = s_warp[nw - 1];
  const T r = (warp ? s_warp[warp - 1] : T(0)) + x - v;
  __syncthreads();                                   // s_warp is reused by the caller's next scan
  return r;
}

// flags of 16 rows (one byte each, 0 or 1) -> how many are set
__device__ __forceinline__ uint32_t flag_count(uint4 v) { return __popc(v.x) + __popc(v.y) + __popc(v.z) + __popc(v.w); }

// stat: [0] listed rows out of [0, size), [1] distinct rows removed (rm_scan_kernel), [2] first removed row (kRmNone: none)
__global__ void __launch_bounds__(kRmThreads) rm_mark_kernel(const int64_t* __restrict__ rows, long long n, long long size,
                                                             uint8_t* __restrict__ flag, unsigned long long* __restrict__ stat) {
  unsigned long long bad = 0, first = kRmNone;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const long long r = rows[i];
    if (r < 0 || r >= size) {
      ++bad;
    } else {
      flag[r] = 1;                                   // a duplicate writes the same byte again
      first = min(first, (unsigned long long)r);
    }
  }
  for (int o = 16; o; o >>= 1) {
    bad += __shfl_xor_sync(~0u, bad, o);
    first = min(first, __shfl_xor_sync(~0u, first, o));
  }
  if ((threadIdx.x & 31) == 0) {
    if (bad) atomicAdd(stat, bad);
    if (first != kRmNone) atomicMin(stat + 2, first);
  }
}

// bsum[b] = flags set among rows [b * kRmTile, (b + 1) * kRmTile)
__global__ void __launch_bounds__(kRmThreads) rm_count_kernel(const uint8_t* __restrict__ flag, uint32_t* __restrict__ bsum) {
  __shared__ uint32_t s_warp[32];
  const uint4 v = reinterpret_cast<const uint4*>(flag)[(size_t)blockIdx.x * kRmThreads + threadIdx.x];
  uint32_t total;
  block_excl_scan(flag_count(v), s_warp, &total);
  if (threadIdx.x == 0) bsum[blockIdx.x] = total;
}

// one block: bsum -> its exclusive prefix sums (rows removed before each tile), stat[1] = their total
__global__ void __launch_bounds__(1024) rm_scan_kernel(uint32_t* __restrict__ bsum, long long nblk,
                                                       unsigned long long* __restrict__ stat) {
  __shared__ uint32_t s_warp[32];
  uint32_t carry = 0;                                // < 2^31: the index holds fewer rows
  for (long long base = 0; base < nblk; base += blockDim.x) {
    const long long i = base + threadIdx.x;
    const uint32_t v = i < nblk ? bsum[i] : 0u;
    uint32_t total;
    const uint32_t e = block_excl_scan(v, s_warp, &total);
    if (i < nblk) bsum[i] = carry + e;
    carry += total;
  }
  if (threadIdx.x == 0) stat[1] = carry;
}

// kept[j] = the j-th live row of [first, size), for the tiles b0, b0 + 1, ... (boff: rm_scan_kernel's offsets).  A live
// row r has boff + (flags set before r in its tile) removed rows before it, all >= first.
__global__ void __launch_bounds__(kRmThreads) rm_fill_kernel(const uint8_t* __restrict__ flag, const uint32_t* __restrict__ boff,
                                                             long long b0, long long first, long long size,
                                                             int32_t* __restrict__ kept) {
  __shared__ uint32_t s_warp[32];
  const long long b = b0 + blockIdx.x;
  const uint4 v = reinterpret_cast<const uint4*>(flag)[(size_t)b * kRmThreads + threadIdx.x];
  uint32_t total;
  uint32_t removed = boff[b] + block_excl_scan(flag_count(v), s_warp, &total);
  const uint32_t w[4] = {v.x, v.y, v.z, v.w};
  const long long r0 = b * kRmTile + (long long)threadIdx.x * 16;
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const long long r = r0 + i;
    const uint32_t f = (w[i >> 2] >> ((i & 3) * 8)) & 1u;
    if (!f && r >= first && r < size) kept[r - first - removed] = (int32_t)r;
    removed += f;
  }
}

// one warp per piece row j < rows: source row kept[j] of every plane (vec 16-byte words per row, plane_vec words between
// planes) -> row j of the piece's planes (piece_vec words between them), and its norm / inverse scale / tag
__global__ void __launch_bounds__(kRmThreads) rm_gather_kernel(const int32_t* __restrict__ kept, long long rows, int planes,
                                                               int vec, const float4* __restrict__ src, long long plane_vec,
                                                               const float* __restrict__ norm, const float* __restrict__ scale,
                                                               const int64_t* __restrict__ tags, float4* __restrict__ piece,
                                                               long long piece_vec, float* __restrict__ p_norm,
                                                               float* __restrict__ p_scale, int64_t* __restrict__ p_tags) {
  const long long j = blockIdx.x * (long long)(kRmThreads / 32) + (threadIdx.x >> 5);
  if (j >= rows) return;
  const int lane = threadIdx.x & 31;
  const long long r = kept[j];
  for (int p = 0; p < planes; ++p) {
    const float4* s = src + p * plane_vec + r * vec;
    float* d = reinterpret_cast<float*>(piece + p * piece_vec + j * vec);
    int i = lane;
    for (; i + 96 < vec; i += 128) {                 // four 16-byte loads in flight per lane
      const float4 a = pps::ld_stream_f4(s + i), b = pps::ld_stream_f4(s + i + 32);
      const float4 c = pps::ld_stream_f4(s + i + 64), e = pps::ld_stream_f4(s + i + 96);
      pps::st_stream_f4(d + 4 * i, a);
      pps::st_stream_f4(d + 4 * (i + 32), b);
      pps::st_stream_f4(d + 4 * (i + 64), c);
      pps::st_stream_f4(d + 4 * (i + 96), e);
    }
    for (; i < vec; i += 32) pps::st_stream_f4(d + 4 * i, pps::ld_stream_f4(s + i));
  }
  if (lane == 0) {
    p_norm[j] = norm[r];
    if (scale) p_scale[j] = scale[r];
    if (tags) p_tags[j] = tags[r];
  }
}

// the groups of piece rows j < rows (kept apart from rm_gather_kernel, which moves everything else)
__global__ void __launch_bounds__(kRmThreads) rm_gather_i64_kernel(const int32_t* __restrict__ kept, long long rows,
                                                                   const int64_t* __restrict__ src, int64_t* __restrict__ dst) {
  const long long j = blockIdx.x * (long long)kRmThreads + threadIdx.x;
  if (j < rows) dst[j] = src[kept[j]];
}

// ---- range search (pps_index_range_search) and the segment sort (pps_sort_key_segments) ----
constexpr int kSortThreads = 256;
constexpr int kSortTile = 4096;                     // S: keys one CTA sorts in shared memory (16 per thread)
constexpr int kMergeTile = 2048;                    // output keys per CTA of a merge pass (< S: at most two pair blocks)
constexpr size_t kSortSmem = 2 * kSortTile * sizeof(unsigned long long);
constexpr long long kSliceBytes = 1LL << 30;        // cap of the first pass's slices, nq * C * 8 bytes

// radius -> admission limit of the range kernel: distance bits < lim  <=>  d <= r (distances are >= 0 and never NaN).
// -0 counts as 0, +inf gives 0x7f800001 (every row), a negative or NaN radius 0 (none).  Counters zeroed, slice q at q * C.
__global__ void range_prep_kernel(const float* __restrict__ radius, long long nq, long long slice, uint32_t* __restrict__ lim,
                                  uint32_t* __restrict__ cnt, long long* __restrict__ off, uint32_t* __restrict__ cap) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= nq) return;
  const float r = radius[i];
  lim[i] = r >= 0.f ? (r == 0.f ? 0u : __float_as_uint(r)) + 1u : 0u;
  cnt[i] = 0u;
  off[i] = i * slice;
  cap[i] = (uint32_t)slice;
}

// one block: lims = exclusive prefix sums of cnt (int64, [n + 1]); stat = {total, largest count}
__global__ void __launch_bounds__(1024) range_scan_kernel(const uint32_t* __restrict__ cnt, long long n, long long* __restrict__ lims,
                                                          unsigned long long* __restrict__ stat) {
  __shared__ unsigned long long s_warp[32];
  __shared__ uint32_t s_max;
  if (threadIdx.x == 0) s_max = 0u;
  unsigned long long carry = 0;
  uint32_t m = 0u;
  for (long long base = 0; base < n; base += blockDim.x) {
    const long long i = base + threadIdx.x;
    const uint32_t v = i < n ? cnt[i] : 0u;
    m = max(m, v);
    unsigned long long total;
    const unsigned long long e = block_excl_scan<unsigned long long>(v, s_warp, &total);
    if (i < n) lims[i] = (long long)(carry + e);
    carry += total;
  }
  __syncthreads();                                   // (n == 0: s_max's initialisation)
  atomicMax(&s_max, m);
  __syncthreads();
  if (threadIdx.x == 0) {
    lims[n] = (long long)carry;
    stat[0] = carry;
    stat[1] = s_max;
  }
}

// The segment sort works on CSR positions o in [0, total) of keys[base + o] (base = lims[0]).  Runs are aligned to
// multiples of their width w counted from position 0 and clipped to their segment; the tile stage leaves every aligned
// S-block of a segment sorted, and the merge pass of width w merges the two w-runs of every aligned 2w-block.  After
// ceil(log2(total / S)) passes every segment lies in one sorted run.

// segment of position o: the last s with lims[s] - base <= o  (o < lims[nseg] - base)
__device__ __forceinline__ long long seg_of(const long long* __restrict__ lims, long long nseg, long long base, long long o) {
  long long lo = 0, hi = nseg;
  while (hi - lo > 1) {
    const long long mid = (lo + hi) >> 1;
    if (__ldg(lims + mid) - base <= o) lo = mid;
    else hi = mid;
  }
  return lo;
}

// #{i < n : a[i] < x} (LE: a[i] <= x) of an ascending a.  A merge places a key of run A after the smaller keys of run B
// and a key of B after the keys of A that are not greater: equal keys keep A before B.
template <bool LE>
__device__ __forceinline__ int count_below(const unsigned long long* a, int n, unsigned long long x) {
  int lo = 0;
  while (n > 0) {
    const int h = n >> 1;
    if (LE ? a[lo + h] <= x : a[lo + h] < x) {
      lo += h + 1;
      n -= h + 1;
    } else {
      n = h;
    }
  }
  return lo;
}

// merge path of one warp: how many of the first d outputs of merge(a[0, na), b[0, nb)) come from a (A first on ties).
// 32 probes per step, so a split in runs of 2^20 keys takes 4 dependent loads instead of 20.
__device__ long long merge_split_warp(const unsigned long long* __restrict__ a, long long na,
                                      const unsigned long long* __restrict__ b, long long nb, long long d) {
  long long lo = d - nb > 0 ? d - nb : 0, hi = d < na ? d : na;
  const int lane = threadIdx.x & 31;
  while (lo < hi) {                                  // a[i] <= b[d - 1 - i] holds for i < answer, fails from there on
    const long long step = (hi - lo + 31) / 32, i = lo + lane * step;
    const bool p = i < hi && a[i] <= b[d - 1 - i];
    const long long c = __popc(__ballot_sync(~0u, p));
    if (c == 0) {
      hi = lo;
    } else {
      const long long nlo = lo + (c - 1) * step + 1;
      hi = min(hi, lo + c * step);
      lo = nlo;
    }
  }
  return lo;
}

// tile stage: CTA b sorts positions [b S, b S + S) ∩ [0, total) piece by piece of segment, in shared memory, by merging
// aligned runs of 1, 2, 4, ... keys (every piece at once: no pass per segment).  Position o's key comes from
// src[s * stride + o - (lims[s] - base)] (stride > 0: the first pass's per-query slices) or src[o]; the result goes to
// dst[o] (may be src: the tile is read before it is written).  src / dst point at position 0.
__global__ void __launch_bounds__(kSortThreads) seg_tile_sort_kernel(const unsigned long long* src, long long stride,
                                                                     unsigned long long* dst, const long long* __restrict__ lims,
                                                                     long long nseg, long long base, long long total) {
  extern __shared__ unsigned long long s_keys[];     // [2][S]
  constexpr int kPer = kSortTile / kSortThreads;
  const long long t0 = (long long)blockIdx.x * kSortTile;
  const int n = (int)min((long long)kSortTile, total - t0);
  int seg_lo[kPer], seg_hi[kPer];                    // the segment's piece of the tile, per position (positions stay put)
  unsigned long long* cur = s_keys;
  unsigned long long* nxt = s_keys + kSortTile;
#pragma unroll
  for (int j = 0; j < kPer; ++j) {
    const int i = threadIdx.x + j * kSortThreads;
    seg_lo[j] = seg_hi[j] = i;
    if (i < n) {
      const long long o = t0 + i, s = seg_of(lims, nseg, base, o);
      const long long l = __ldg(lims + s) - base, r = __ldg(lims + s + 1) - base;
      seg_lo[j] = (int)(max(l, t0) - t0);
      seg_hi[j] = (int)(min(r, t0 + n) - t0);
      cur[i] = stride > 0 ? src[s * stride + (o - l)] : src[o];
    }
  }
  __syncthreads();
  for (int w = 1; w < n; w <<= 1) {
#pragma unroll
    for (int j = 0; j < kPer; ++j) {
      const int i = threadIdx.x + j * kSortThreads;
      if (i < n) {
        const unsigned long long x = cur[i];
        const int ps = i & ~(2 * w - 1), m = ps + w;
        const int a0 = max(ps, seg_lo[j]), a1 = min(m, seg_hi[j]);          // run A of i's pair block, clipped
        const int b0 = max(m, seg_lo[j]), b1 = min(ps + 2 * w, seg_hi[j]);  // run B
        const int pos = i < m ? i + count_below<false>(cur + b0, max(b1 - b0, 0), x)
                              : a0 + (i - b0) + count_below<true>(cur + a0, max(a1 - a0, 0), x);
        nxt[pos] = x;
      }
    }
    __syncthreads();
    unsigned long long* t = cur;
    cur = nxt;
    nxt = t;
  }
#pragma unroll
  for (int j = 0; j < kPer; ++j) {
    const int i = threadIdx.x + j * kSortThreads;
    if (i < n) dst[t0 + i] = cur[i];
  }
}

// merge pass of width w >= S: CTA b writes output positions [b T, b T + T) ∩ [0, total) of dst (src, dst: position 0).
// A pair block [ps, ps + 2w) needs a merge only where a segment crosses its middle m = ps + w; the tile touches at most two pair blocks (T < 2w),
// so it holds at most two merged pieces.  Each piece: merge-path splits of its ends (one warp each), the keys of both runs
// that land in it -> shared memory, every key's rank in the other run there.  Every other position is copied.
__global__ void __launch_bounds__(kSortThreads) seg_merge_kernel(const unsigned long long* __restrict__ src,
                                                                 unsigned long long* __restrict__ dst,
                                                                 const long long* __restrict__ lims, long long nseg,
                                                                 long long base, long long total, long long w) {
  __shared__ unsigned long long s_in[kMergeTile];
  __shared__ long long s_pc[2][6];                   // piece: out begin, out end, P0 (pair start in the segment), m, ia, ib
  __shared__ int s_ok[2];
  const long long o0 = (long long)blockIdx.x * kMergeTile, o1 = min(o0 + kMergeTile, total);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const unsigned long long* in = src;
  if (warp < 2) {
    const long long ps = ((warp == 0 ? o0 : o1 - 1) / (2 * w)) * (2 * w), m = ps + w;
    bool ok = m < total && !(warp == 1 && ps == (o0 / (2 * w)) * (2 * w));
    if (ok) {
      const long long s = seg_of(lims, nseg, base, m);
      const long long l = __ldg(lims + s) - base, r = __ldg(lims + s + 1) - base;
      const long long p0 = max(ps, l), p1 = min(ps + 2 * w, r);
      const long long a = max(o0, p0), b = min(o1, p1);
      ok = l < m && a < b;                           // the segment crosses m and its pair block meets the tile
      if (ok) {
        const long long ia = merge_split_warp(in + p0, m - p0, in + m, p1 - m, a - p0);
        const long long ib = merge_split_warp(in + p0, m - p0, in + m, p1 - m, b - p0);
        if (lane == 0) {
          s_pc[warp][0] = a; s_pc[warp][1] = b; s_pc[warp][2] = p0; s_pc[warp][3] = m;
          s_pc[warp][4] = ia; s_pc[warp][5] = ib;
        }
      }
    }
    if (lane == 0) s_ok[warp] = ok;
  }
  __syncthreads();
  for (long long o = o0 + threadIdx.x; o < o1; o += kSortThreads) {
    const bool merged = (s_ok[0] && o >= s_pc[0][0] && o < s_pc[0][1]) || (s_ok[1] && o >= s_pc[1][0] && o < s_pc[1][1]);
    if (!merged) dst[o] = in[o];
  }
  for (int k = 0; k < 2; ++k) {
    if (!s_ok[k]) continue;                          // (uniform)
    const long long a = s_pc[k][0], b = s_pc[k][1], p0 = s_pc[k][2], m = s_pc[k][3], ia = s_pc[k][4], ib = s_pc[k][5];
    const int na = (int)(ib - ia), nb = (int)((b - a) - na);
    const long long jb = (a - p0) - ia;              // first key of run B in the piece
    for (int u = threadIdx.x; u < na + nb; u += kSortThreads) s_in[u] = u < na ? in[p0 + ia + u] : in[m + jb + (u - na)];
    __syncthreads();
    for (int u = threadIdx.x; u < na + nb; u += kSortThreads) {
      const unsigned long long x = s_in[u];
      const int pos = u < na ? u + count_below<false>(s_in + na, nb, x) : (u - na) + count_below<true>(s_in, na, x);
      dst[a + pos] = x;
    }
    __syncthreads();
  }
}

// sorts every segment [lims[s], lims[s + 1]) of keys ascending (base = lims[0], total = lims[nseg] - base; scratch holds
// total keys when total > S); slices / stride > 0: the keys come from the first pass's slices and the tile stage
// compacts them into keys.  Ends in keys.
int sort_segments(unsigned long long* keys, const long long* lims, long long nseg, long long base, long long total,
                  unsigned long long* scratch, const unsigned long long* slices, long long stride, cudaStream_t st) {
  if (total <= 0) return PPS_OK;
  int passes = 0;
  for (long long w = kSortTile; w < total; w <<= 1) ++passes;
  if (passes > 0 && !scratch) return PPS_ERR_INVALID_ARG;
  static thread_local int configured_dev = -1;
  int dev = 0;
  PPS_CUDA_TRY(cudaGetDevice(&dev));
  if (configured_dev != dev) {
    PPS_CUDA_TRY(cudaFuncSetAttribute(seg_tile_sort_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSortSmem));
    configured_dev = dev;
  }
  // the tile stage writes where an even number of merge passes after it ends in keys
  unsigned long long* const out = keys + base;
  unsigned long long* cur = (passes & 1) ? scratch : out;
  seg_tile_sort_kernel<<<(unsigned)((total + kSortTile - 1) / kSortTile), kSortThreads, kSortSmem, st>>>(
      slices ? slices : out, slices ? stride : 0, cur, lims, nseg, base, total);
  PPS_LAUNCH_CHECK("seg_tile_sort_kernel");
  for (long long w = kSortTile; w < total; w <<= 1) {
    unsigned long long* nxt = cur == out ? scratch : out;
    seg_merge_kernel<<<(unsigned)((total + kMergeTile - 1) / kMergeTile), kSortThreads, 0, st>>>(cur, nxt, lims, nseg, base,
                                                                                                  total, w);
    PPS_LAUNCH_CHECK("seg_merge_kernel");
    cur = nxt;
  }
  return PPS_OK;
}
}  // namespace

extern "C" int pps_index_create(int device, int dim, int dtype, int precision, pps_index** out) {
  if (!out) return PPS_ERR_INVALID_ARG;
  *out = nullptr;
  if (dim <= 0 || device < 0) return PPS_ERR_INVALID_ARG;
  if (dtype != PPS_DTYPE_F32 && dtype != PPS_DTYPE_F16) return PPS_ERR_INVALID_ARG;
  if (precision == PPS_PREC_FP32) return PPS_ERR_UNSUPPORTED;     // the search runs on the tensor cores only
  int planes = 0;
  if (dtype == PPS_DTYPE_F16) {
    precision = PPS_PREC_F16X1;
    planes = 1;
  } else {
    switch (precision) {
      case PPS_PREC_BF16X1: planes = 1; break;
      case PPS_PREC_BF16X3: planes = 2; break;
      case PPS_PREC_BF16X6: planes = 3; break;
      case PPS_PREC_F16X3: planes = 2; break;
      default: return PPS_ERR_INVALID_ARG;
    }
  }
  int n_dev = 0;
  PPS_CUDA_TRY(cudaGetDeviceCount(&n_dev));
  if (device >= n_dev) return PPS_ERR_INVALID_ARG;
  pps_index* x = new (std::nothrow) pps_index();
  if (!x) return PPS_ERR_CUDA;
  x->device = device; x->dim = dim; x->kpad = pps_kpad(dim); x->dtype = dtype; x->precision = precision; x->planes = planes;
  x->split_planes = precision == PPS_PREC_F16X3 ? (2 | PPS_SPLIT_F16_SCALED) : planes;
  *out = x;
  return PPS_OK;
}

extern "C" int pps_index_destroy(pps_index* x) {
  if (!x) return PPS_OK;
  DeviceGuard dg(x->device);
  if (x->g_planes) cudaFree(x->g_planes);
  if (x->g_norm) cudaFree(x->g_norm);
  if (x->g_tags) cudaFree(x->g_tags);
  if (x->g_groups) cudaFree(x->g_groups);
  GrowBuf* bufs[] = {&x->qs,      &x->qn,     &x->dist,    &x->tk_bound, &x->tk_cnt,    &x->tk_cand, &x->flag,
                     &x->n_excl,  &x->rm_flag, &x->rm_bsum, &x->rm_stat,  &x->rm_kept,   &x->rm_piece, &x->rg_lim,
                     &x->rg_cnt,  &x->rg_off, &x->rg_cap,  &x->rg_slices, &x->rg_stat, &x->rg_keys,  &x->rg_tmp};
  for (GrowBuf* b : bufs) b->release();
  x->flag_h.release();
  delete x;
  return PPS_OK;
}

extern "C" long long pps_index_size(const pps_index* x) { return x ? x->size : PPS_ERR_INVALID_ARG; }

namespace {

int add_rows(pps_index* x, const void* d_rows, long long n, long long ld, const int64_t* d_tags, const int64_t* d_groups,
             void* stream) {
  if (!x || n < 0 || ld < x->dim) return PPS_ERR_INVALID_ARG;
  if (n == 0) return PPS_OK;
  if (!d_rows) return PPS_ERR_INVALID_ARG;
  if (x->size > 0 && x->tagged != (d_tags != nullptr)) return PPS_ERR_INVALID_ARG;   // all rows tagged, or none
  if (x->size > 0 && x->grouped != (d_groups != nullptr)) return PPS_ERR_INVALID_ARG; // all rows grouped, or none
  if (x->size + n > kMaxIndex) return PPS_ERR_UNSUPPORTED;
  DeviceGuard dg(x->device);
  if (dg.err != cudaSuccess) return pps::cuda_fail(dg.err, "cudaSetDevice");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (x->size == 0) {
    x->tagged = d_tags != nullptr;
    x->grouped = d_groups != nullptr;
  }
  if (x->size + n > x->capacity || (x->tagged && !x->g_tags) || (x->grouped && !x->g_groups))
    PPS_TRY(grow(x, x->size + n, st));
  // pps_split_rows_slab reads row r of the source at base + r * ld: the new rows sit at rows [size, size + n) of it
  const size_t esz = x->dtype == PPS_DTYPE_F16 ? 2 : 4;
  const unsigned char* base = static_cast<const unsigned char*>(d_rows) - (size_t)x->size * (size_t)ld * esz;
  PPS_TRY(pps_split_rows_slab(base, x->dtype, x->size, n, x->capacity, x->dim, ld, x->split_planes, x->g_planes, x->g_norm, st));
  if (d_tags)
    PPS_CUDA_TRY(cudaMemcpyAsync(x->g_tags + x->size, d_tags, (size_t)n * sizeof(int64_t), cudaMemcpyDeviceToDevice, st));
  if (d_groups)
    PPS_CUDA_TRY(cudaMemcpyAsync(x->g_groups + x->size, d_groups, (size_t)n * sizeof(int64_t), cudaMemcpyDeviceToDevice, st));
  x->size += n;
  return PPS_OK;
}

// q_tags: null (every row), or the excluding search (a tagged index)
int search(pps_index* x, const void* d_q, long long nq, long long ldq, const int64_t* q_tags, int k, long long index_offset,
           int flags, void* stream, uint64_t* d_keys) {
  if (nq < 0 || k < 1 || k > PPS_TOPK_MAX || index_offset < 0) return PPS_ERR_INVALID_ARG;
  if (flags & ~(PPS_INDEX_TKCAP(0xffff) | PPS_INDEX_PREFIX(0x7f))) return PPS_ERR_INVALID_ARG;
  if (nq > 0 && (ldq < x->dim || !d_q || !d_keys)) return PPS_ERR_INVALID_ARG;
  if (index_offset + x->size > kMaxIndex || nq > kMaxIndex) return PPS_ERR_UNSUPPORTED;
  if (nq == 0) return PPS_OK;
  DeviceGuard dg(x->device);
  if (dg.err != cudaSuccess) return pps::cuda_fail(dg.err, "cudaSetDevice");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  PPS_TRY(pps_topk_init(d_keys, nq, k, st));
  const long long size = x->size;
  if (size == 0) return PPS_OK;
  int tk_cap = (flags >> 8) & 0xffff;
  if (tk_cap <= 0 || tk_cap > kTkCap) tk_cap = kTkCap;
  const long long prefix_hook = (long long)((flags >> 24) & 0x7f) * 256;
  const long long first = std::min(size, prefix_hook > 0 ? prefix_hook : kPrefixRows);
  const long long ldd = (first + 3) / 4 * 4;
  const bool chunked = first < size;

  PPS_TRY(x->qs.ensure((size_t)pps_split_bytes(nq, x->dim, x->planes)));
  PPS_TRY(x->qn.ensure((size_t)nq * 2 * sizeof(float)));
  PPS_TRY(x->dist.ensure((size_t)nq * ldd * sizeof(float)));
  if (chunked) {
    PPS_TRY(x->flag.ensure(8));         // [0] overflow flag, [1] largest excluded count of the prefix
    PPS_TRY(x->flag_h.ensure(4));
  }
  uint32_t* n_excl = nullptr;
  if (q_tags && chunked) {
    PPS_TRY(x->n_excl.ensure((size_t)nq * 4));
    n_excl = x->n_excl.as<uint32_t>();
  }
  PPS_TRY(pps_split_rows(d_q, x->dtype, nq, x->dim, ldq, x->split_planes, x->qs.p, x->qn.as<float>(), st));
  PPS_TRY(block_update(x, nq, 0, first, ldd, index_offset, k, d_keys, q_tags, n_excl, st));
  if (!chunked) return PPS_OK;

  PPS_TRY(x->tk_bound.ensure((size_t)nq * 4));
  PPS_TRY(x->tk_cnt.ensure((size_t)nq * 4));
  PPS_TRY(x->tk_cand.ensure((size_t)nq * tk_cap * 8));
  uint32_t* bound = x->tk_bound.as<uint32_t>();
  uint32_t* cnt = x->tk_cnt.as<uint32_t>();
  int32_t* flag = x->flag.as<int32_t>();
  double keep = 1.0;                    // share of the rows a query may take, as the chunk sizing assumes it
  if (n_excl) {
    max_u32_kernel<<<1, 256, 0, st>>>(n_excl, nq, reinterpret_cast<uint32_t*>(flag + 1));
    PPS_LAUNCH_CHECK("max_u32_kernel");
    PPS_CUDA_TRY(cudaMemcpyAsync(x->flag_h.p, flag + 1, 4, cudaMemcpyDeviceToHost, st));
    PPS_CUDA_TRY(cudaStreamSynchronize(st));
    keep = 1.0 - std::min(0.9, (double)*x->flag_h.as<uint32_t>() / (double)first);
  }
  PPS_CUDA_TRY(cudaMemsetAsync(flag, 0, 4, st));
  PPS_TRY(pps_topk_bound(d_keys, nq, k, bound, cnt, st));
  for (long long done = first; done < size;) {
    long long rows = (long long)((double)tk_cap * (double)done * keep / (2.2 * k)) / 256 * 256;
    rows = std::min(size - done, std::max<long long>(rows, 256));
    if (q_tags)
      PPS_TRY(pps_search_topk_excl_tc(x->planes_at(done), x->g_norm + done, rows, x->planes, x->capacity, x->qs.p,
                                      x->qn.as<float>(), nq, x->planes, 0, x->dim, x->precision, 0, index_offset + done, bound,
                                      cnt, x->tk_cand.as<uint64_t>(), tk_cap, st, x->g_tags + done, q_tags));
    else
      PPS_TRY(pps_search_topk_tc(x->planes_at(done), x->g_norm + done, rows, x->planes, x->capacity, x->qs.p,
                                 x->qn.as<float>(), nq, x->planes, 0, x->dim, x->precision, 0, index_offset + done, bound, cnt,
                                 x->tk_cand.as<uint64_t>(), tk_cap, st));
    PPS_TRY(pps_topk_merge(d_keys, nq, k, x->tk_cand.as<uint64_t>(), tk_cap, cnt, bound, nullptr, nullptr, nullptr, 0, 0, flag,
                           st));
    done += rows;
  }
  PPS_CUDA_TRY(cudaMemcpyAsync(x->flag_h.p, flag, 4, cudaMemcpyDeviceToHost, st));
  PPS_CUDA_TRY(cudaStreamSynchronize(st));
  if (*x->flag_h.as<int32_t>() == 0) return PPS_OK;
  // a candidate buffer ran over: every block materialised and swept (slower, right for any row order)
  PPS_TRY(pps_topk_init(d_keys, nq, k, st));
  for (long long r0 = 0; r0 < size; r0 += first)
    PPS_TRY(block_update(x, nq, r0, std::min(first, size - r0), ldd, index_offset, k, d_keys, q_tags, nullptr, st));
  return PPS_OK;
}

// grouped materialised block: rows [r0, r0 + rows) swept into the grouped state
int group_block_update(pps_index* x, long long nq, long long r0, long long rows, long long ldd, long long index_offset, int k,
                       uint64_t* keys, int64_t* groups, const int64_t* q_tags, cudaStream_t st) {
  PPS_TRY(pps_dist_tc(x->qs.p, x->qn.as<float>(), nq, x->planes, 0, x->planes_at(r0), x->g_norm + r0, rows, x->planes,
                      x->capacity, x->dim, x->precision, 0, x->dist.as<float>(), ldd, st));
  return pps_topk_group_update(x->dist.as<float>(), ldd, nq, rows, index_offset + r0, x->g_groups + r0,
                               q_tags ? x->g_tags + r0 : nullptr, q_tags, keys, groups, k, st);
}

// *out = the number of queries whose state holds fewer than k groups (its k-th key is ~0)
__global__ void short_count_kernel(const unsigned long long* __restrict__ keys, long long nq, int k, uint32_t* __restrict__ out) {
  __shared__ uint32_t s_n;
  if (threadIdx.x == 0) s_n = 0u;
  __syncthreads();
  uint32_t n = 0u;
  for (long long q = threadIdx.x; q < nq; q += blockDim.x) n += keys[q * k + k - 1] == ~0ull;
  atomicAdd(&s_n, n);
  __syncthreads();
  if (threadIdx.x == 0) *out = s_n;
}

// range-kernel limits that count the rows at or below each query's bound (bits <= bound <=> bits < bound + 1), with no
// room for keys: counters zeroed, capacities 0
__global__ void count_lim_kernel(const uint32_t* __restrict__ bound, long long nq, uint32_t* __restrict__ lim,
                                 uint32_t* __restrict__ cnt, long long* __restrict__ off, uint32_t* __restrict__ cap) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= nq) return;
  lim[i] = bound[i] == 0xffffffffu ? 0xffffffffu : bound[i] + 1u;
  cnt[i] = 0u;
  off[i] = 0;
  cap[i] = 0u;
}

// Grouped search (pps_index_search_groups).  The admission kernels are search's: a row above the bound of a state that
// holds k groups is either worse than its own group's row in the state or beaten by k other groups (DESIGN §4.16).
//   1. prefix: materialised blocks of F rows swept by the grouped sweep until every query holds k groups (a 4-byte
//      read-back per block: the queries still short) or the gallery ends
//   2. L = the largest number of prefix rows at or below their query's bound (one counting pass of the range kernel over
//      the prefix, one 4-byte read-back); chunks of R = cap F_done / (2.2 max(k, L)) rows, each admitted by the search
//      kernel and merged by the grouped merge
//   3. the overflow read-back; on overflow every block materialised and swept (right for any row order)
int search_groups(pps_index* x, const void* d_q, long long nq, long long ldq, const int64_t* q_tags, int k,
                  long long index_offset, int flags, void* stream, uint64_t* d_keys, int64_t* d_groups) {
  if (nq < 0 || k < 1 || k > PPS_TOPK_MAX || index_offset < 0) return PPS_ERR_INVALID_ARG;
  if (flags & ~(PPS_INDEX_TKCAP(0xffff) | PPS_INDEX_PREFIX(0x7f))) return PPS_ERR_INVALID_ARG;
  if (nq > 0 && (ldq < x->dim || !d_q || !d_keys || !d_groups)) return PPS_ERR_INVALID_ARG;
  if (index_offset + x->size > kMaxIndex || nq > kMaxIndex) return PPS_ERR_UNSUPPORTED;
  if (nq == 0) return PPS_OK;
  DeviceGuard dg(x->device);
  if (dg.err != cudaSuccess) return pps::cuda_fail(dg.err, "cudaSetDevice");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  PPS_TRY(pps_topk_init(d_keys, nq, k, st));
  PPS_CUDA_TRY(cudaMemsetAsync(d_groups, 0xff, (size_t)nq * k * sizeof(int64_t), st));   // -1
  const long long size = x->size;
  x->last_prefix = size;
  x->last_chunks = 0;
  x->last_fallback = 0;
  if (size == 0) return PPS_OK;
  int tk_cap = (flags >> 8) & 0xffff;
  if (tk_cap <= 0 || tk_cap > kGroupTkCap) tk_cap = kGroupTkCap;
  const long long prefix_hook = (long long)((flags >> 24) & 0x7f) * 256;
  const long long first = std::min(size, prefix_hook > 0 ? prefix_hook : kPrefixRows);
  const long long ldd = (first + 3) / 4 * 4;

  PPS_TRY(x->qs.ensure((size_t)pps_split_bytes(nq, x->dim, x->planes)));
  PPS_TRY(x->qn.ensure((size_t)nq * 2 * sizeof(float)));
  PPS_TRY(x->dist.ensure((size_t)nq * ldd * sizeof(float)));
  PPS_TRY(x->flag.ensure(8));           // [0] overflow flag, [1] queries short of k groups / largest count L
  PPS_TRY(x->flag_h.ensure(4));
  int32_t* flag = x->flag.as<int32_t>();
  uint32_t* stat = reinterpret_cast<uint32_t*>(flag + 1);
  PPS_TRY(pps_split_rows(d_q, x->dtype, nq, x->dim, ldq, x->split_planes, x->qs.p, x->qn.as<float>(), st));

  // 1. prefix
  long long done = 0;
  while (done < size) {
    const long long rows = std::min(first, size - done);
    PPS_TRY(group_block_update(x, nq, done, rows, ldd, index_offset, k, d_keys, d_groups, q_tags, st));
    done += rows;
    if (done == size) break;
    short_count_kernel<<<1, 256, 0, st>>>(reinterpret_cast<const unsigned long long*>(d_keys), nq, k, stat);
    PPS_LAUNCH_CHECK("short_count_kernel");
    PPS_CUDA_TRY(cudaMemcpyAsync(x->flag_h.p, stat, 4, cudaMemcpyDeviceToHost, st));
    PPS_CUDA_TRY(cudaStreamSynchronize(st));
    if (*x->flag_h.as<uint32_t>() == 0) break;
  }
  if (done == size) return PPS_OK;

  // 2. L, then the chunks
  PPS_TRY(x->tk_bound.ensure((size_t)nq * 4));
  PPS_TRY(x->tk_cnt.ensure((size_t)nq * 4));
  PPS_TRY(x->tk_cand.ensure((size_t)nq * tk_cap * 8));
  PPS_TRY(x->rg_lim.ensure((size_t)nq * 4));
  PPS_TRY(x->rg_cnt.ensure((size_t)nq * 2 * 4));
  PPS_TRY(x->rg_off.ensure((size_t)nq * 8));
  PPS_TRY(x->rg_cap.ensure((size_t)nq * 4));
  uint32_t* bound = x->tk_bound.as<uint32_t>();
  uint32_t* cnt = x->tk_cnt.as<uint32_t>();
  uint32_t* n_le = x->rg_cnt.as<uint32_t>();
  PPS_TRY(pps_topk_bound(d_keys, nq, k, bound, cnt, st));
  count_lim_kernel<<<(unsigned)((nq + 255) / 256), 256, 0, st>>>(bound, nq, x->rg_lim.as<uint32_t>(), n_le,
                                                                 x->rg_off.as<long long>(), x->rg_cap.as<uint32_t>());
  PPS_LAUNCH_CHECK("count_lim_kernel");
  PPS_TRY(pps_search_range_tc(x->planes_at(0), x->g_norm, done, x->planes, x->capacity, x->qs.p, x->qn.as<float>(), nq,
                              x->planes, 0, x->dim, x->precision, 0, index_offset, x->rg_lim.as<uint32_t>(), n_le,
                              x->rg_off.as<long long>(), x->rg_cap.as<uint32_t>(), x->tk_cand.as<uint64_t>(),
                              q_tags ? x->g_tags : nullptr, q_tags, st));
  max_u32_kernel<<<1, 256, 0, st>>>(n_le, nq, stat);
  PPS_LAUNCH_CHECK("max_u32_kernel");
  PPS_CUDA_TRY(cudaMemcpyAsync(x->flag_h.p, stat, 4, cudaMemcpyDeviceToHost, st));
  PPS_CUDA_TRY(cudaMemsetAsync(flag, 0, 4, st));
  PPS_CUDA_TRY(cudaStreamSynchronize(st));
  const double per_row = (double)std::max<uint32_t>((uint32_t)k, *x->flag_h.as<uint32_t>());
  x->last_prefix = done;
  for (; done < size;) {
    long long rows = (long long)((double)tk_cap * (double)done / (2.2 * per_row)) / 256 * 256;
    rows = std::min(size - done, std::max<long long>(rows, 256));
    if (q_tags)
      PPS_TRY(pps_search_topk_excl_tc(x->planes_at(done), x->g_norm + done, rows, x->planes, x->capacity, x->qs.p,
                                      x->qn.as<float>(), nq, x->planes, 0, x->dim, x->precision, 0, index_offset + done, bound,
                                      cnt, x->tk_cand.as<uint64_t>(), tk_cap, st, x->g_tags + done, q_tags));
    else
      PPS_TRY(pps_search_topk_tc(x->planes_at(done), x->g_norm + done, rows, x->planes, x->capacity, x->qs.p,
                                 x->qn.as<float>(), nq, x->planes, 0, x->dim, x->precision, 0, index_offset + done, bound, cnt,
                                 x->tk_cand.as<uint64_t>(), tk_cap, st));
    PPS_TRY(pps_topk_group_merge(d_keys, d_groups, nq, k, x->tk_cand.as<uint64_t>(), tk_cap, cnt, bound, x->g_groups,
                                 index_offset, flag, st));
    done += rows;
    ++x->last_chunks;
  }
  PPS_CUDA_TRY(cudaMemcpyAsync(x->flag_h.p, flag, 4, cudaMemcpyDeviceToHost, st));
  PPS_CUDA_TRY(cudaStreamSynchronize(st));
  if (*x->flag_h.as<int32_t>() == 0) return PPS_OK;
  // 3. a candidate buffer ran over: every block materialised and swept
  x->last_fallback = 1;
  PPS_TRY(pps_topk_init(d_keys, nq, k, st));
  PPS_CUDA_TRY(cudaMemsetAsync(d_groups, 0xff, (size_t)nq * k * sizeof(int64_t), st));
  for (long long r0 = 0; r0 < size; r0 += first)
    PPS_TRY(group_block_update(x, nq, r0, std::min(first, size - r0), ldd, index_offset, k, d_keys, d_groups, q_tags, st));
  return PPS_OK;
}

}  // namespace

extern "C" int pps_index_add(pps_index* x, const void* d_rows, long long n, long long ld, void* stream) {
  return add_rows(x, d_rows, n, ld, nullptr, nullptr, stream);
}

extern "C" int pps_index_add_tagged(pps_index* x, const void* d_rows, long long n, long long ld, const int64_t* d_tags,
                                    void* stream) {
  if (n > 0 && !d_tags) return PPS_ERR_INVALID_ARG;
  return add_rows(x, d_rows, n, ld, d_tags, nullptr, stream);
}

extern "C" int pps_index_add_grouped(pps_index* x, const void* d_rows, long long n, long long ld, const int64_t* d_tags,
                                     const int64_t* d_groups, void* stream) {
  if (n > 0 && !d_groups) return PPS_ERR_INVALID_ARG;
  return add_rows(x, d_rows, n, ld, d_tags, d_groups, stream);
}

extern "C" int pps_index_search(pps_index* x, const void* d_q, long long nq, long long ldq, int k, long long index_offset,
                                int flags, void* stream, uint64_t* d_keys) {
  if (!x) return PPS_ERR_INVALID_ARG;
  return search(x, d_q, nq, ldq, nullptr, k, index_offset, flags, stream, d_keys);
}

extern "C" int pps_index_search_excluding(pps_index* x, const void* d_q, long long nq, long long ldq, const int64_t* d_q_tags,
                                          int k, long long index_offset, int flags, void* stream, uint64_t* d_keys) {
  if (!x) return PPS_ERR_INVALID_ARG;
  if (nq > 0 && !d_q_tags) return PPS_ERR_INVALID_ARG;
  if (x->size > 0 && !x->tagged) return PPS_ERR_INVALID_ARG;     // nothing to compare the query tags with
  return search(x, d_q, nq, ldq, d_q_tags, k, index_offset, flags, stream, d_keys);
}

extern "C" int pps_index_search_groups(pps_index* x, const void* d_q, long long nq, long long ldq, const int64_t* d_q_tags,
                                       int k, long long index_offset, int flags, void* stream, uint64_t* d_keys,
                                       int64_t* d_groups) {
  if (!x) return PPS_ERR_INVALID_ARG;
  if (x->size > 0 && !x->grouped) return PPS_ERR_INVALID_ARG;    // no groups to collapse
  if (d_q_tags && x->size > 0 && !x->tagged) return PPS_ERR_INVALID_ARG;
  return search_groups(x, d_q, nq, ldq, d_q_tags, k, index_offset, flags, stream, d_keys, d_groups);
}

extern "C" int pps_index_group_stats(const pps_index* x, long long* prefix_rows, long long* chunks, int* fallback) {
  if (!x) return PPS_ERR_INVALID_ARG;
  if (prefix_rows) *prefix_rows = x->last_prefix;
  if (chunks) *chunks = x->last_chunks;
  if (fallback) *fallback = x->last_fallback;
  return PPS_OK;
}

extern "C" int pps_index_remove(pps_index* x, const int64_t* d_rows, long long n, int flags, void* stream,
                                long long* n_removed) {
  if (n_removed) *n_removed = 0;
  if (!x || n < 0 || (flags & ~PPS_INDEX_PIECE(0xffff))) return PPS_ERR_INVALID_ARG;
  if (n == 0) return PPS_OK;
  if (!d_rows || x->size == 0) return PPS_ERR_INVALID_ARG;      // (an empty index has no row to remove)
  DeviceGuard dg(x->device);
  if (dg.err != cudaSuccess) return pps::cuda_fail(dg.err, "cudaSetDevice");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long size = x->size;
  const long long nblk = (size + kRmTile - 1) / kRmTile;
  PPS_TRY(x->rm_flag.ensure((size_t)nblk * kRmTile));
  PPS_TRY(x->rm_bsum.ensure((size_t)nblk * 4));
  PPS_TRY(x->rm_stat.ensure(3 * 8));
  PPS_TRY(x->flag_h.ensure(3 * 8));
  uint8_t* flag = x->rm_flag.as<uint8_t>();
  uint32_t* bsum = x->rm_bsum.as<uint32_t>();
  unsigned long long* stat = x->rm_stat.as<unsigned long long>();

  // 1. mark, count, scan; one read-back
  PPS_CUDA_TRY(cudaMemsetAsync(flag, 0, (size_t)nblk * kRmTile, st));
  PPS_CUDA_TRY(cudaMemsetAsync(stat, 0, 2 * 8, st));
  PPS_CUDA_TRY(cudaMemsetAsync(stat + 2, 0xff, 8, st));
  const long long mark_blocks = std::min<long long>((n + kRmThreads - 1) / kRmThreads, (long long)pps::sm_count() * 8);
  rm_mark_kernel<<<(unsigned)mark_blocks, kRmThreads, 0, st>>>(d_rows, n, size, flag, stat);
  PPS_LAUNCH_CHECK("rm_mark_kernel");
  rm_count_kernel<<<(unsigned)nblk, kRmThreads, 0, st>>>(flag, bsum);
  PPS_LAUNCH_CHECK("rm_count_kernel");
  rm_scan_kernel<<<1, 1024, 0, st>>>(bsum, nblk, stat);
  PPS_LAUNCH_CHECK("rm_scan_kernel");
  PPS_CUDA_TRY(cudaMemcpyAsync(x->flag_h.p, stat, 3 * 8, cudaMemcpyDeviceToHost, st));
  PPS_CUDA_TRY(cudaStreamSynchronize(st));
  const unsigned long long* h = x->flag_h.as<unsigned long long>();
  if (h[0] != 0) return PPS_ERR_INVALID_ARG;                     // nothing has moved
  const long long removed = (long long)h[1], first = (long long)h[2];
  const long long moving = size - first - removed;              // the live rows after the first removed one

  if (moving > 0) {
    // 2. kept list
    PPS_TRY(x->rm_kept.ensure((size_t)moving * 4));
    int32_t* kept = x->rm_kept.as<int32_t>();
    const long long b0 = first / kRmTile;
    rm_fill_kernel<<<(unsigned)(nblk - b0), kRmThreads, 0, st>>>(flag, bsum, b0, first, size, kept);
    PPS_LAUNCH_CHECK("rm_fill_kernel");

    // 3. move in pieces: gather into the piece buffer [planes][piece][kpad] | tags | groups | norms | inverse scales,
    //    copy down
    const size_t per_row = x->plane_bytes(1) * x->planes + (x->tagged ? 8 : 0) + (x->scaled() ? 8 : 4) + (x->grouped ? 8 : 0);
    const long long hook = (flags >> 8) & 0xffff;
    const long long piece = std::min(moving, hook > 0 ? hook : std::max<long long>(1, (long long)(kRmPieceBytes / per_row)));
    PPS_TRY(x->rm_piece.ensure((size_t)piece * per_row));
    unsigned char* pb = x->rm_piece.as<unsigned char>();
    int64_t* p_tags = reinterpret_cast<int64_t*>(pb + x->planes * x->plane_bytes(piece));
    int64_t* p_groups = p_tags + (x->tagged ? piece : 0);
    float* p_norm = reinterpret_cast<float*>(p_groups + (x->grouped ? piece : 0));
    float* p_scale = p_norm + piece;
    const int vec = x->kpad * 2 / 16;
    for (long long j0 = 0; j0 < moving; j0 += piece) {
      const long long len = std::min(piece, moving - j0);
      const long long dst = first + j0;
      rm_gather_kernel<<<(unsigned)((len + kRmThreads / 32 - 1) / (kRmThreads / 32)), kRmThreads, 0, st>>>(
          kept + j0, len, x->planes, vec, static_cast<const float4*>(x->g_planes), x->capacity * vec, x->g_norm,
          x->scaled() ? x->g_norm + x->capacity : nullptr, x->tagged ? x->g_tags : nullptr, reinterpret_cast<float4*>(pb),
          piece * vec, p_norm, p_scale, p_tags);
      PPS_LAUNCH_CHECK("rm_gather_kernel");
      if (x->grouped) {
        rm_gather_i64_kernel<<<(unsigned)((len + kRmThreads - 1) / kRmThreads), kRmThreads, 0, st>>>(kept + j0, len,
                                                                                                  x->g_groups, p_groups);
        PPS_LAUNCH_CHECK("rm_gather_i64_kernel");
      }
      for (int p = 0; p < x->planes; ++p)
        PPS_CUDA_TRY(cudaMemcpyAsync(static_cast<unsigned char*>(x->g_planes) + p * x->plane_bytes(x->capacity) +
                                         x->plane_bytes(dst),
                                     pb + p * x->plane_bytes(piece), x->plane_bytes(len), cudaMemcpyDeviceToDevice, st));
      PPS_CUDA_TRY(cudaMemcpyAsync(x->g_norm + dst, p_norm, (size_t)len * 4, cudaMemcpyDeviceToDevice, st));
      if (x->scaled())
        PPS_CUDA_TRY(cudaMemcpyAsync(x->g_norm + x->capacity + dst, p_scale, (size_t)len * 4, cudaMemcpyDeviceToDevice, st));
      if (x->tagged)
        PPS_CUDA_TRY(cudaMemcpyAsync(x->g_tags + dst, p_tags, (size_t)len * 8, cudaMemcpyDeviceToDevice, st));
      if (x->grouped)
        PPS_CUDA_TRY(cudaMemcpyAsync(x->g_groups + dst, p_groups, (size_t)len * 8, cudaMemcpyDeviceToDevice, st));
    }
  }
  x->size = size - removed;
  if (n_removed) *n_removed = removed;
  return PPS_OK;
}

namespace {

// cudaMalloc's failure is also the runtime's last error: clear it, so that the index's next call does not report it again
int ensure_or_clear(GrowBuf& b, size_t bytes) {
  const int rc = b.ensure(bytes);
  if (rc != PPS_OK) cudaGetLastError();
  return rc;
}

int range_search(pps_index* x, const void* d_q, long long nq, long long ldq, const float* d_radius, const int64_t* q_tags,
                 long long index_offset, int flags, void* stream, int64_t* d_lims, long long* total) {
  if (!total) return PPS_ERR_INVALID_ARG;
  *total = 0;
  if (nq < 0 || index_offset < 0 || (flags & ~PPS_INDEX_TKCAP(0xffff))) return PPS_ERR_INVALID_ARG;
  if (!d_lims || (nq > 0 && (ldq < x->dim || !d_q || !d_radius))) return PPS_ERR_INVALID_ARG;
  if (index_offset + x->size > kMaxIndex || nq > kMaxIndex) return PPS_ERR_UNSUPPORTED;
  DeviceGuard dg(x->device);
  if (dg.err != cudaSuccess) return pps::cuda_fail(dg.err, "cudaSetDevice");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  x->rg_total = 0;
  const long long size = x->size;
  if (nq == 0 || size == 0) {
    PPS_CUDA_TRY(cudaMemsetAsync(d_lims, 0, (size_t)(nq + 1) * sizeof(int64_t), st));
    return PPS_OK;
  }
  long long* lims = reinterpret_cast<long long*>(d_lims);
  const long long hook = (flags >> 8) & 0xffff;
  const long long slice = hook > 0 ? hook : std::min(x->rg_slice, std::max(1LL, kSliceBytes / 8 / nq));
  PPS_TRY(ensure_or_clear(x->qs, (size_t)pps_split_bytes(nq, x->dim, x->planes)));
  PPS_TRY(ensure_or_clear(x->qn, (size_t)nq * 2 * sizeof(float)));
  PPS_TRY(ensure_or_clear(x->rg_lim, (size_t)nq * 4));
  PPS_TRY(ensure_or_clear(x->rg_cnt, (size_t)nq * 2 * 4));     // first-pass counts | second-pass counters
  PPS_TRY(ensure_or_clear(x->rg_off, (size_t)nq * 8));
  PPS_TRY(ensure_or_clear(x->rg_cap, (size_t)nq * 4));
  PPS_TRY(ensure_or_clear(x->rg_slices, (size_t)nq * slice * 8));
  PPS_TRY(ensure_or_clear(x->rg_stat, 2 * 8));
  PPS_TRY(x->flag_h.ensure(2 * 8));
  uint32_t* lim = x->rg_lim.as<uint32_t>();
  uint32_t* cnt = x->rg_cnt.as<uint32_t>();
  unsigned long long* stat = x->rg_stat.as<unsigned long long>();
  const int64_t* g_tags = q_tags ? x->g_tags : nullptr;

  // 1. split, limits; 2. first pass into uniform slices; 3. counts -> lims, one 16-byte read-back
  PPS_TRY(pps_split_rows(d_q, x->dtype, nq, x->dim, ldq, x->split_planes, x->qs.p, x->qn.as<float>(), st));
  range_prep_kernel<<<(unsigned)((nq + 255) / 256), 256, 0, st>>>(d_radius, nq, slice, lim, cnt, x->rg_off.as<long long>(),
                                                                  x->rg_cap.as<uint32_t>());
  PPS_LAUNCH_CHECK("range_prep_kernel");
  PPS_TRY(pps_search_range_tc(x->planes_at(0), x->g_norm, size, x->planes, x->capacity, x->qs.p, x->qn.as<float>(), nq,
                              x->planes, 0, x->dim, x->precision, 0, index_offset, lim, cnt, x->rg_off.as<long long>(),
                              x->rg_cap.as<uint32_t>(), x->rg_slices.as<uint64_t>(), g_tags, q_tags, st));
  range_scan_kernel<<<1, 1024, 0, st>>>(cnt, nq, lims, stat);
  PPS_LAUNCH_CHECK("range_scan_kernel");
  PPS_CUDA_TRY(cudaMemcpyAsync(x->flag_h.p, stat, 2 * 8, cudaMemcpyDeviceToHost, st));
  PPS_CUDA_TRY(cudaStreamSynchronize(st));
  const long long tot = (long long)x->flag_h.as<unsigned long long>()[0];
  const long long largest = (long long)x->flag_h.as<unsigned long long>()[1];
  while (x->rg_slice < largest) x->rg_slice <<= 1;
  if (tot == 0) return PPS_OK;

  // 4. the sorted keys in index-owned scratch (grow-only); a result that does not fit fails here, before anything changes
  if (tot > (1LL << 56)) return pps::cuda_fail(cudaErrorMemoryAllocation, "range search result");
  PPS_TRY(ensure_or_clear(x->rg_keys, (size_t)tot * 8));
  if (tot > kSortTile) PPS_TRY(ensure_or_clear(x->rg_tmp, (size_t)tot * 8));
  unsigned long long* keys = x->rg_keys.as<unsigned long long>();
  unsigned long long* tmp = tot > kSortTile ? x->rg_tmp.as<unsigned long long>() : nullptr;
  if (largest > slice) {
    // 5. a slice ran over: the same pass again, straight into the CSR layout (capacities = the exact counts)
    uint32_t* cnt2 = cnt + nq;
    PPS_CUDA_TRY(cudaMemsetAsync(cnt2, 0, (size_t)nq * 4, st));
    PPS_TRY(pps_search_range_tc(x->planes_at(0), x->g_norm, size, x->planes, x->capacity, x->qs.p, x->qn.as<float>(), nq,
                                x->planes, 0, x->dim, x->precision, 0, index_offset, lim, cnt2, lims, cnt,
                                reinterpret_cast<uint64_t*>(keys), g_tags, q_tags, st));
    PPS_TRY(sort_segments(keys, lims, nq, 0, tot, tmp, nullptr, 0, st));
  } else {
    PPS_TRY(sort_segments(keys, lims, nq, 0, tot, tmp, x->rg_slices.as<unsigned long long>(), slice, st));
  }
  x->rg_total = tot;
  *total = tot;
  return PPS_OK;
}

}  // namespace

extern "C" int pps_index_range_search(pps_index* x, const void* d_q, long long nq, long long ldq, const float* d_radius,
                                      const int64_t* d_q_tags, long long index_offset, int flags, void* stream,
                                      int64_t* d_lims, long long* total) {
  if (total) *total = 0;
  if (!x) return PPS_ERR_INVALID_ARG;
  if (d_q_tags && x->size > 0 && !x->tagged) return PPS_ERR_INVALID_ARG;     // nothing to compare the query tags with
  return range_search(x, d_q, nq, ldq, d_radius, d_q_tags, index_offset, flags, stream, d_lims, total);
}

extern "C" int pps_index_range_keys(pps_index* x, uint64_t* d_keys, void* stream) {
  if (!x) return PPS_ERR_INVALID_ARG;
  if (x->rg_total == 0) return PPS_OK;
  if (!d_keys) return PPS_ERR_INVALID_ARG;
  DeviceGuard dg(x->device);
  if (dg.err != cudaSuccess) return pps::cuda_fail(dg.err, "cudaSetDevice");
  PPS_CUDA_TRY(cudaMemcpyAsync(d_keys, x->rg_keys.p, (size_t)x->rg_total * 8, cudaMemcpyDeviceToDevice,
                               static_cast<cudaStream_t>(stream)));
  return PPS_OK;
}

extern "C" int pps_sort_key_segments(uint64_t* keys, const int64_t* lims, long long nseg, uint64_t* scratch, void* stream) {
  if (nseg < 0) return PPS_ERR_INVALID_ARG;
  if (nseg == 0) return PPS_OK;
  if (!keys || !lims) return PPS_ERR_INVALID_ARG;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  long long ends[2] = {0, 0};                        // lims[0], lims[nseg]: the grid depends on their difference only
  PPS_CUDA_TRY(cudaMemcpyAsync(ends, lims, 8, cudaMemcpyDeviceToHost, st));
  PPS_CUDA_TRY(cudaMemcpyAsync(ends + 1, lims + nseg, 8, cudaMemcpyDeviceToHost, st));
  PPS_CUDA_TRY(cudaStreamSynchronize(st));
  if (ends[0] < 0 || ends[1] < ends[0]) return PPS_ERR_INVALID_ARG;
  return sort_segments(reinterpret_cast<unsigned long long*>(keys), reinterpret_cast<const long long*>(lims), nseg, ends[0],
                       ends[1] - ends[0], reinterpret_cast<unsigned long long*>(scratch), nullptr, 0, st);
}
