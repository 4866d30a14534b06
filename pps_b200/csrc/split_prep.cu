// Operand preparation for the tensor-core distance: fp32 rows -> bf16 residual planes
// (x = p0 + p1 + p2, each the bf16 round-to-nearest of what is left) with K zero-padded to
// a multiple of 64, plus the row squared norms |x|^2 of compute_dist
// (reid_dataset_evaluator.py:266-268) accumulated in fp64 and rounded once to fp32.
// HBM-bound: reads 4*dim bytes per row, writes 2*kpad bytes per plane. One warp per row.
#include "common.cuh"

namespace pps {

constexpr int kSplitWarps = 8;

template <int PLANES, bool F16IN>
__global__ void __launch_bounds__(32 * kSplitWarps) split_rows_kernel(const void* __restrict__ feats, long long row_begin,
                                                                       long long row_end, long long rows, int dim,
                                                                       long long ld, int kpad,
                                                                       void* __restrict__ out_planes,
                                                                       float* __restrict__ out_sqnorm,
                                                                       const int32_t* __restrict__ row_index,
                                                                       long long index_base) {
  // output row `row` <- source row `srow` (= row unless a gather list is given)
  const int lane = threadIdx.x & 31;
  const long long row = row_begin + (long long)blockIdx.x * kSplitWarps + (threadIdx.x >> 5);
  if (row >= row_end) return;
  const long long srow = row_index ? (long long)row_index[row] - index_base : row;
  double acc = 0.0;
  const long long plane_stride = rows * (long long)kpad;   // elements
  if constexpr (F16IN) {
    const __half* src = reinterpret_cast<const __half*>(feats) + srow * ld;
    __half* dst = out_planes ? reinterpret_cast<__half*>(out_planes) + row * (long long)kpad : nullptr;
    const bool vec8 = ((dim & 7) == 0) && ((ld & 7) == 0) && ((reinterpret_cast<uintptr_t>(feats) & 15u) == 0);
    if (vec8) {
      // 128-bit loads: 8 halves per lane and step; the K padding (kpad - dim < 64 halves) is zero-filled below
      for (int k = lane * 8; k < dim; k += 256) {
        const uint4 u = *reinterpret_cast<const uint4*>(src + k);
        const __half2* h2 = reinterpret_cast<const __half2*>(&u);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float2 f = __half22float2(h2[e]);
          acc += (double)(f.x * f.x) + (double)(f.y * f.y);   // squares of fp16 values are exact in fp32
        }
        if (dst) *reinterpret_cast<uint4*>(dst + k) = u;
      }
      if (dst)
        for (int k = dim + lane; k < kpad; k += 32) dst[k] = __float2half(0.f);
    } else {
      for (int k = lane; k < kpad; k += 32) {
        const __half h = k < dim ? src[k] : __float2half(0.f);
        const float v = __half2float(h);
        acc += (double)v * (double)v;
        if (dst) dst[k] = h;
      }
    }
  } else {
    const float* src = reinterpret_cast<const float*>(feats) + srow * ld;
    __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(out_planes);
    const bool vec = ((ld & 3) == 0) && ((reinterpret_cast<uintptr_t>(feats) & 15u) == 0);
    // four 128-bit loads of the row in flight per lane before any is consumed (the rows are streamed once)
    int kfast = lane * 4;
    if (vec) {
      for (; kfast + 3 * 128 + 3 < dim; kfast += 4 * 128) {
        float4 t[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) t[u] = ld_stream_f4(reinterpret_cast<const float4*>(src + kfast + u * 128));
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int k = kfast + u * 128;
          const float v[4] = {t[u].x, t[u].y, t[u].z, t[u].w};
          __nv_bfloat16 p[3][4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            acc += (double)v[e] * (double)v[e];
            float r = v[e];
#pragma unroll
            for (int pl = 0; pl < PLANES; ++pl) {
              p[pl][e] = __float2bfloat16_rn(r);
              r -= __bfloat162float(p[pl][e]);   // exact in fp32
            }
          }
          if (dst) {
#pragma unroll
            for (int pl = 0; pl < PLANES; ++pl) {
              uint2 w;
              w.x = (uint32_t)__bfloat16_as_ushort(p[pl][0]) | ((uint32_t)__bfloat16_as_ushort(p[pl][1]) << 16);
              w.y = (uint32_t)__bfloat16_as_ushort(p[pl][2]) | ((uint32_t)__bfloat16_as_ushort(p[pl][3]) << 16);
              *reinterpret_cast<uint2*>(dst + pl * plane_stride + row * (long long)kpad + k) = w;
            }
          }
        }
      }
    }
    for (int k = kfast; k < kpad; k += 128) {
      float v[4];
      if (vec && k + 3 < dim) {
        const float4 t = ld_stream_f4(reinterpret_cast<const float4*>(src + k));
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
      } else {
#pragma unroll
        for (int e = 0; e < 4; ++e) v[e] = (k + e < dim) ? src[k + e] : 0.f;
      }
      __nv_bfloat16 p[3][4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        acc += (double)v[e] * (double)v[e];
        float r = v[e];
#pragma unroll
        for (int pl = 0; pl < PLANES; ++pl) {
          p[pl][e] = __float2bfloat16_rn(r);
          r -= __bfloat162float(p[pl][e]);   // exact in fp32
        }
      }
      if (dst) {
#pragma unroll
        for (int pl = 0; pl < PLANES; ++pl) {
          uint2 w;
          w.x = (uint32_t)__bfloat16_as_ushort(p[pl][0]) | ((uint32_t)__bfloat16_as_ushort(p[pl][1]) << 16);
          w.y = (uint32_t)__bfloat16_as_ushort(p[pl][2]) | ((uint32_t)__bfloat16_as_ushort(p[pl][3]) << 16);
          *reinterpret_cast<uint2*>(dst + pl * plane_stride + row * (long long)kpad + k) = w;
        }
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0 && out_sqnorm) out_sqnorm[row] = (float)acc;
}

// fp32 rows -> TWO fp16 residual planes of the row scaled by a power of two (PPS_SPLIT_F16_SCALED): with
// s = 2^e chosen per row so that max|x| * s lies in [2^14, 2^15), p0 = fp16(x s), p1 = fp16(x s - p0).  fp16 carries
// 11 significant bits, so p0 + p1 holds 22 bits of every element (bf16 planes: 16) at the same two-plane cost, and
// the scaling keeps p1 out of the fp16 subnormals.  The distance epilogue multiplies the accumulator by the product of
// the two inverse scales, formed as one float.  e <= 63 keeps that product a normal float (>= 2^-126), so it is exact:
// rows with max|x| < 2^-48 are scaled less than fully (max|x| s < 2^14), which costs only their smallest elements
// bits.  out_sqnorm[row] = |x|^2, out_sqnorm[rows + row] = 1 / s.
// Two streaming passes over the row (max + norm, then split); the second one hits L1 / L2.  Keeping the row in registers
// between the passes (kF16Cache4 = 16: 98 registers, 16 warps per SM) measured SLOWER: 2.9 TB/s against 4.6-5.1 TB/s
// (profiles/r02_notes.md).
template <int kF16Cache4>
__global__ void __launch_bounds__(32 * kSplitWarps) split_rows_f16s_kernel(const float* __restrict__ feats, long long row_begin,
                                                                            long long row_end, long long rows, int dim,
                                                                            long long ld, int kpad,
                                                                            __half* __restrict__ out_planes,
                                                                            float* __restrict__ out_sqnorm,
                                                                            const int32_t* __restrict__ row_index,
                                                                            long long index_base) {
  const int lane = threadIdx.x & 31;
  const long long row = row_begin + (long long)blockIdx.x * kSplitWarps + (threadIdx.x >> 5);
  if (row >= row_end) return;
  const long long srow = row_index ? (long long)row_index[row] - index_base : row;
  const float* src = feats + srow * ld;
  const bool vec = ((ld & 3) == 0) && ((reinterpret_cast<uintptr_t>(feats) & 15u) == 0);
  auto load4 = [&](int k, bool stream) -> float4 {
    if (vec && k + 3 < dim)
      return stream ? ld_stream_f4(reinterpret_cast<const float4*>(src + k)) : *reinterpret_cast<const float4*>(src + k);
    float4 t;
    t.x = k < dim ? src[k] : 0.f;
    t.y = k + 1 < dim ? src[k + 1] : 0.f;
    t.z = k + 2 < dim ? src[k + 2] : 0.f;
    t.w = k + 3 < dim ? src[k + 3] : 0.f;
    return t;
  };
  double acc = 0.0;
  float mx = 0.f;
  auto note = [&](const float4& t) {
    acc += (double)t.x * (double)t.x + (double)t.y * (double)t.y + (double)t.z * (double)t.z + (double)t.w * (double)t.w;
    mx = fmaxf(mx, fmaxf(fmaxf(fabsf(t.x), fabsf(t.y)), fmaxf(fabsf(t.z), fabsf(t.w))));
  };
  float4 cache[kF16Cache4 > 0 ? kF16Cache4 : 1];
#pragma unroll
  for (int u = 0; u < kF16Cache4; ++u) {
    const int k = lane * 4 + u * 128;
    cache[u] = k < kpad ? load4(k, true) : make_float4(0.f, 0.f, 0.f, 0.f);
    note(cache[u]);
  }
  {
    // rows (or row tails) that are not held in registers: streamed with four loads in flight, re-read by the split pass
    int k = lane * 4 + kF16Cache4 * 128;
    for (; k + 3 * 128 < kpad; k += 4 * 128) {
      float4 t[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) t[u] = load4(k + u * 128, false);
#pragma unroll
      for (int u = 0; u < 4; ++u) note(t[u]);
    }
    for (; k < kpad; k += 128) note(load4(k, false));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    acc += __shfl_xor_sync(0xffffffffu, acc, o);
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  }
  int e = 0;
  if (mx > 0.f && mx <= 3.0e38f) {          // (NaN / inf rows keep s = 1: their distances are NaN / inf either way)
    int ex;
    frexpf(mx, &ex);                        // mx = m * 2^ex, m in [0.5, 1)
    e = 15 - ex;
    e = e > 63 ? 63 : (e < -100 ? -100 : e);   // 63: 1 / (s_a s_b) >= 2^-126 (see above)
  }
  const float s = ldexpf(1.f, e), inv = ldexpf(1.f, -e);
  const long long plane_stride = rows * (long long)kpad;
  __half* dst = out_planes + row * (long long)kpad;
  auto emit = [&](int k, const float4& t) {
    // packed conversions (two floats -> half2 in one instruction; the scalar F2F path is a quarter-rate unit)
    const float2 a = make_float2(t.x * s, t.y * s), b = make_float2(t.z * s, t.w * s);
    const __half2 ha = __float22half2_rn(a), hb = __float22half2_rn(b);
    const float2 fa = __half22float2(ha), fb = __half22float2(hb);
    const __half2 la = __float22half2_rn(make_float2(a.x - fa.x, a.y - fa.y));     // the residual is exact in fp32
    const __half2 lb = __float22half2_rn(make_float2(b.x - fb.x, b.y - fb.y));
    uint2 w0, w1;
    w0.x = *reinterpret_cast<const uint32_t*>(&ha);
    w0.y = *reinterpret_cast<const uint32_t*>(&hb);
    w1.x = *reinterpret_cast<const uint32_t*>(&la);
    w1.y = *reinterpret_cast<const uint32_t*>(&lb);
    *reinterpret_cast<uint2*>(dst + k) = w0;
    *reinterpret_cast<uint2*>(dst + plane_stride + k) = w1;
  };
#pragma unroll
  for (int u = 0; u < kF16Cache4; ++u) {
    const int k = lane * 4 + u * 128;
    if (k < kpad) emit(k, cache[u]);
  }
  {
    int k = lane * 4 + kF16Cache4 * 128;
    for (; k + 3 * 128 < kpad; k += 4 * 128) {
      float4 t[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) t[u] = load4(k + u * 128, false);
#pragma unroll
      for (int u = 0; u < 4; ++u) emit(k + u * 128, t[u]);
    }
    for (; k < kpad; k += 128) emit(k, load4(k, false));
  }
  if (lane == 0 && out_sqnorm) {
    out_sqnorm[row] = (float)acc;
    out_sqnorm[rows + row] = inv;
  }
}

// Caffe2 Normalize(axis=1) of the concatenated embedding (reid_heads.py:123-127, triplet_loss.py:18):
// y = x / max(|x|_2, 1e-12).  One CTA per row; the row (<= tens of KB) is read twice, the second time from L1/L2.
__global__ void __launch_bounds__(256) l2_normalize_rows_kernel(const float* __restrict__ x, int dim, long long ld,
                                                                float* __restrict__ out, long long ldo) {
  __shared__ float part[8];
  const float* src = x + (long long)blockIdx.x * ld;
  float* dst = out + (long long)blockIdx.x * ldo;
  const bool vec = ((dim & 3) == 0) && ((ld & 3) == 0) && ((ldo & 3) == 0) &&
                   (((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(out)) & 15u) == 0);
  float acc = 0.f;
  if (vec) {
    for (int k = threadIdx.x * 4; k < dim; k += 1024) {
      const float4 t = *reinterpret_cast<const float4*>(src + k);
      acc = fmaf(t.x, t.x, acc); acc = fmaf(t.y, t.y, acc); acc = fmaf(t.z, t.z, acc); acc = fmaf(t.w, t.w, acc);
    }
  } else {
    for (int k = threadIdx.x; k < dim; k += 256) acc = fmaf(src[k], src[k], acc);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
  __syncthreads();
  float tot = 0.f;
#pragma unroll
  for (int w = 0; w < 8; ++w) tot += part[w];
  const float inv = 1.0f / fmaxf(sqrtf(tot), 1e-12f);
  if (vec) {
    for (int k = threadIdx.x * 4; k < dim; k += 1024) {
      float4 t = *reinterpret_cast<const float4*>(src + k);
      t.x *= inv; t.y *= inv; t.z *= inv; t.w *= inv;
      *reinterpret_cast<float4*>(dst + k) = t;
    }
  } else {
    for (int k = threadIdx.x; k < dim; k += 256) dst[k] = src[k] * inv;
  }
}

// Multi-query pooling (reid_dataset_evaluator.py:131-143): the features of the mark-2 images of one (id, camera) group
// are averaged, `np.mean(mq_feat[rows], axis=0)` - a float32 sum of the rows in list order, then one division by the
// count.  One CTA per group, thread = feature columns, rows added in order (bit-identical to NumPy's axis-0 reduction).
__global__ void __launch_bounds__(256) group_mean_rows_kernel(const float* __restrict__ feats, long long ld, int dim,
                                                              const int32_t* __restrict__ group_off,
                                                              const int32_t* __restrict__ row_idx, float* __restrict__ out,
                                                              long long ldo) {
  const int gidx = blockIdx.x;
  const int e0 = group_off[gidx], e1 = group_off[gidx + 1];
  const float cnt = (float)(e1 - e0);
  for (int c = threadIdx.x; c < dim; c += blockDim.x) {
    float acc = 0.f;
    for (int e = e0; e < e1; ++e) acc = __fadd_rn(acc, feats[(long long)row_idx[e] * ld + c]);
    out[(long long)gidx * ldo + c] = e1 > e0 ? __fdiv_rn(acc, cnt) : 0.f;
  }
}

}  // namespace pps

using namespace pps;

extern "C" int pps_kpad(int dim) { return dim <= 0 ? 0 : ((dim + 63) / 64) * 64; }

extern "C" long long pps_split_bytes(long long rows, int dim, int planes) {
  if (planes & PPS_SPLIT_F16_SCALED) planes = 2;
  if (rows < 0 || dim <= 0 || planes < 1 || planes > 3) return PPS_ERR_INVALID_ARG;
  return rows * (long long)pps_kpad(dim) * 2 * planes;
}

static int split_dispatch(const void* feats, int dtype, long long row0, long long nrows, long long rows, int dim,
                          long long ld, int planes, void* out_planes, float* out_sqnorm, void* stream,
                          const int32_t* row_index = nullptr, long long index_base = 0) {
  if (rows < 0 || dim <= 0 || ld < dim || row0 < 0 || nrows < 0 || row0 + nrows > rows) return PPS_ERR_INVALID_ARG;
  if (nrows == 0) return PPS_OK;
  if (!feats) return PPS_ERR_INVALID_ARG;
  if (out_planes && (reinterpret_cast<uintptr_t>(out_planes) & 15u)) return PPS_ERR_ALIGN;
  const int kpad = pps_kpad(dim);
  const long long blocks = (nrows + kSplitWarps - 1) / kSplitWarps;
  if (blocks > 0x7fffffffLL) return PPS_ERR_UNSUPPORTED;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const dim3 grid((unsigned)blocks), block(32 * kSplitWarps);
  if (dtype == PPS_DTYPE_F16) {
    if (planes != 1) return PPS_ERR_INVALID_ARG;
    split_rows_kernel<1, true><<<grid, block, 0, st>>>(feats, row0, row0 + nrows, rows, dim, ld, kpad, out_planes, out_sqnorm, row_index, index_base);
  } else if (dtype == PPS_DTYPE_F32 && (planes & PPS_SPLIT_F16_SCALED)) {
    if ((planes & ~PPS_SPLIT_F16_SCALED) != 2 || !out_planes || !out_sqnorm) return PPS_ERR_INVALID_ARG;
    split_rows_f16s_kernel<0><<<grid, block, 0, st>>>(static_cast<const float*>(feats), row0, row0 + nrows, rows, dim, ld, kpad,
                                                      static_cast<__half*>(out_planes), out_sqnorm, row_index, index_base);
  } else if (dtype == PPS_DTYPE_F32) {
    switch (planes) {
      case 1: split_rows_kernel<1, false><<<grid, block, 0, st>>>(feats, row0, row0 + nrows, rows, dim, ld, kpad, out_planes, out_sqnorm, row_index, index_base); break;
      case 2: split_rows_kernel<2, false><<<grid, block, 0, st>>>(feats, row0, row0 + nrows, rows, dim, ld, kpad, out_planes, out_sqnorm, row_index, index_base); break;
      case 3: split_rows_kernel<3, false><<<grid, block, 0, st>>>(feats, row0, row0 + nrows, rows, dim, ld, kpad, out_planes, out_sqnorm, row_index, index_base); break;
      default: return PPS_ERR_INVALID_ARG;
    }
  } else {
    return PPS_ERR_INVALID_ARG;
  }
  PPS_LAUNCH_CHECK("split_rows_kernel");
  return PPS_OK;
}

extern "C" int pps_split_rows(const void* feats, int dtype, long long rows, int dim, long long ld, int planes,
                              void* out_planes, float* out_sqnorm, void* stream) {
  if (!out_planes && rows > 0) return PPS_ERR_INVALID_ARG;
  return split_dispatch(feats, dtype, 0, rows, rows, dim, ld, planes, out_planes, out_sqnorm, stream);
}

extern "C" int pps_split_rows_slab(const void* feats, int dtype, long long row0, long long nrows, long long total_rows,
                                   int dim, long long ld, int planes, void* out_planes, float* out_sqnorm,
                                   void* stream) {
  if (!out_planes && nrows > 0) return PPS_ERR_INVALID_ARG;
  return split_dispatch(feats, dtype, row0, nrows, total_rows, dim, ld, planes, out_planes, out_sqnorm, stream);
}

extern "C" int pps_row_sqnorm(const void* feats, int dtype, long long rows, int dim, long long ld, float* out_sqnorm,
                              void* stream) {
  if (!out_sqnorm && rows > 0) return PPS_ERR_INVALID_ARG;
  return split_dispatch(feats, dtype, 0, rows, rows, dim, ld, 1, nullptr, out_sqnorm, stream);
}

extern "C" int pps_l2_normalize_rows(const float* x, long long rows, int dim, long long ld, float* out, long long ldo,
                                     void* stream) {
  if (rows < 0 || dim <= 0 || ld < dim || ldo < dim) return PPS_ERR_INVALID_ARG;
  if (rows == 0) return PPS_OK;
  if (!x || !out) return PPS_ERR_INVALID_ARG;
  if (rows > 0x7fffffffLL) return PPS_ERR_UNSUPPORTED;
  l2_normalize_rows_kernel<<<(unsigned)rows, 256, 0, static_cast<cudaStream_t>(stream)>>>(x, dim, ld, out, ldo);
  PPS_LAUNCH_CHECK("l2_normalize_rows_kernel");
  return PPS_OK;
}

extern "C" int pps_split_rows_gather(const void* feats, int dtype, const int32_t* row_index, long long index_base,
                                     long long rows, int dim, long long ld, int planes, void* out_planes,
                                     float* out_sqnorm, void* stream) {
  if ((!out_planes || !row_index) && rows > 0) return PPS_ERR_INVALID_ARG;
  return split_dispatch(feats, dtype, 0, rows, rows, dim, ld, planes, out_planes, out_sqnorm, stream, row_index,
                        index_base);
}

extern "C" int pps_group_mean_rows(const float* feats, long long ld, int dim, const int32_t* group_off,
                                   const int32_t* row_idx, long long n_groups, float* out, long long ldo, void* stream) {
  if (n_groups < 0 || dim <= 0 || ld < dim || ldo < dim) return PPS_ERR_INVALID_ARG;
  if (n_groups == 0) return PPS_OK;
  if (!feats || !group_off || !row_idx || !out) return PPS_ERR_INVALID_ARG;
  if (n_groups > 0x7fffffffLL) return PPS_ERR_UNSUPPORTED;
  group_mean_rows_kernel<<<(unsigned)n_groups, 256, 0, static_cast<cudaStream_t>(stream)>>>(feats, ld, dim, group_off, row_idx,
                                                                                          out, ldo);
  PPS_LAUNCH_CHECK("group_mean_rows_kernel");
  return PPS_OK;
}
