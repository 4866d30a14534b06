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
#include "ctx.cuh"

namespace {

using pps::GrowBuf;
using pps::PinBuf;

constexpr long long kPrefixRows = 32768;
constexpr int kTkCap = 2048;
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
  bool tagged = false;          // decided by the first non-empty add
  GrowBuf qs, qn, dist, tk_bound, tk_cnt, tk_cand, flag, n_excl;
  PinBuf flag_h;
  bool scaled() const { return precision == PPS_PREC_F16X3; }
  size_t plane_bytes(long long rows) const { return (size_t)rows * kpad * 2; }
  const void* planes_at(long long row) const { return static_cast<const unsigned char*>(g_planes) + plane_bytes(row); }
};

namespace {

// capacity -> new_cap: planes, both halves of the norm array and the tags move to their new offsets
int grow(pps_index* x, long long need, cudaStream_t st) {
  long long cap = std::max(x->capacity * 2, std::max(need, kMinCapacity));
  if (cap > kMaxIndex) cap = kMaxIndex;
  void* planes = nullptr;
  float* norm = nullptr;
  int64_t* tags = nullptr;
  const size_t norm_n = (size_t)cap * (x->scaled() ? 2 : 1);
  cudaError_t e = cudaMalloc(&planes, (size_t)x->planes * x->plane_bytes(cap));
  if (e == cudaSuccess) e = cudaMalloc(&norm, norm_n * sizeof(float));
  if (e == cudaSuccess && x->tagged) e = cudaMalloc(&tags, (size_t)cap * sizeof(int64_t));
  if (e != cudaSuccess) {
    if (planes) cudaFree(planes);
    if (norm) cudaFree(norm);
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
    PPS_CUDA_TRY(cudaStreamSynchronize(st));     // the old buffers are read until here
  }
  if (x->g_planes) cudaFree(x->g_planes);
  if (x->g_norm) cudaFree(x->g_norm);
  if (x->g_tags) cudaFree(x->g_tags);
  x->g_planes = planes;
  x->g_norm = norm;
  x->g_tags = tags;
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
  GrowBuf* bufs[] = {&x->qs, &x->qn, &x->dist, &x->tk_bound, &x->tk_cnt, &x->tk_cand, &x->flag, &x->n_excl};
  for (GrowBuf* b : bufs) b->release();
  x->flag_h.release();
  delete x;
  return PPS_OK;
}

extern "C" long long pps_index_size(const pps_index* x) { return x ? x->size : PPS_ERR_INVALID_ARG; }

namespace {

int add_rows(pps_index* x, const void* d_rows, long long n, long long ld, const int64_t* d_tags, void* stream) {
  if (!x || n < 0 || ld < x->dim) return PPS_ERR_INVALID_ARG;
  if (n == 0) return PPS_OK;
  if (!d_rows) return PPS_ERR_INVALID_ARG;
  if (x->size > 0 && x->tagged != (d_tags != nullptr)) return PPS_ERR_INVALID_ARG;   // all rows tagged, or none
  if (x->size + n > kMaxIndex) return PPS_ERR_UNSUPPORTED;
  DeviceGuard dg(x->device);
  if (dg.err != cudaSuccess) return pps::cuda_fail(dg.err, "cudaSetDevice");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (x->size == 0) x->tagged = d_tags != nullptr;
  if (x->size + n > x->capacity || (x->tagged && !x->g_tags)) PPS_TRY(grow(x, x->size + n, st));
  // pps_split_rows_slab reads row r of the source at base + r * ld: the new rows sit at rows [size, size + n) of it
  const size_t esz = x->dtype == PPS_DTYPE_F16 ? 2 : 4;
  const unsigned char* base = static_cast<const unsigned char*>(d_rows) - (size_t)x->size * (size_t)ld * esz;
  PPS_TRY(pps_split_rows_slab(base, x->dtype, x->size, n, x->capacity, x->dim, ld, x->split_planes, x->g_planes, x->g_norm, st));
  if (d_tags)
    PPS_CUDA_TRY(cudaMemcpyAsync(x->g_tags + x->size, d_tags, (size_t)n * sizeof(int64_t), cudaMemcpyDeviceToDevice, st));
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

}  // namespace

extern "C" int pps_index_add(pps_index* x, const void* d_rows, long long n, long long ld, void* stream) {
  return add_rows(x, d_rows, n, ld, nullptr, stream);
}

extern "C" int pps_index_add_tagged(pps_index* x, const void* d_rows, long long n, long long ld, const int64_t* d_tags,
                                    void* stream) {
  if (n > 0 && !d_tags) return PPS_ERR_INVALID_ARG;
  return add_rows(x, d_rows, n, ld, d_tags, stream);
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
