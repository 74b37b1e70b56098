// Scoring-side helpers: dense canonical scores, full row rankings, top-k list merge, metrics.
// (The fused tcgen05 U.V^T + top-k kernel lives in score_topk.cu.)
#include <cub/device/device_segmented_radix_sort.cuh>
#include <math.h>

#include <algorithm>

#include "common.cuh"

namespace tmf {

// canonical score: fp64 FMA chain in component order, rounded once to fp32 (SURVEY 8c item 4)
__global__ void __launch_bounds__(256) predict_dense_kernel(const float* __restrict__ U, long long n_u, const float* __restrict__ V,
                                                            long long n_i, int r, int ld, float* __restrict__ P) {
  extern __shared__ float sm[];  // [16][r] users, [16][r] items
  float* sU = sm;
  float* sV = sm + 16 * r;
  const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;
  const long long u0 = (long long)blockIdx.y * 16, i0 = (long long)blockIdx.x * 16;
  for (int t = threadIdx.x; t < 16 * r; t += 256) {
    const int row = t / r, c = t % r;
    sU[t] = (u0 + row < n_u) ? U[(u0 + row) * ld + c] : 0.f;
    sV[t] = (i0 + row < n_i) ? V[(i0 + row) * ld + c] : 0.f;
  }
  __syncthreads();
  if (u0 + ty >= n_u || i0 + tx >= n_i) return;
  double acc = 0.0;
  for (int c = 0; c < r; ++c) acc = fma((double)sU[ty * r + c], (double)sV[tx * r + c], acc);
  P[(u0 + ty) * n_i + (i0 + tx)] = (float)acc;
}

__global__ void rank_prep_kernel(const float* __restrict__ P, long long n_rows, long long n_cols, int clamp,
                                 float* __restrict__ keys, int* __restrict__ vals, int* __restrict__ offs) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long total = n_rows * n_cols;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long j = i; j <= n_rows; j += stride) offs[j] = (int)(j * n_cols);
  for (; i < total; i += stride) {
    float v = P[i];
    if (clamp) v = v > 0.f ? v : 0.f;   // tf.where(p > 0, p, 0.0), matrix_factorization.py:237
    keys[i] = v + 0.0f;                 // -0.0 -> +0.0 so equal scores share one radix key
    vals[i] = (int)(i % n_cols);
  }
}

__device__ __forceinline__ float csr_lookup(const int* __restrict__ a_idx, const float* __restrict__ a_val, int lo, int hi, int item) {
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    const int c = a_idx[mid];
    if (c == item) return a_val[mid];
    if (c < item) lo = mid + 1; else hi = mid;
  }
  return 0.f;
}

// hits = #{q : A[u, topk[u,q]] != 0} (any sign, :248,:254); relevant = #{A[u,:] > 0} (:240,:251)
__global__ void metrics_hits_kernel(const int* __restrict__ topk, long long n_users, int k, const int* __restrict__ a_ptr,
                                    const int* __restrict__ a_idx, const float* __restrict__ a_val, float* __restrict__ hits,
                                    float* __restrict__ relevant) {
  const long long u = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (u >= n_users) return;
  const int lo = a_ptr[u], hi = a_ptr[u + 1];
  int h = 0, rel = 0;
  for (int q = lane; q < k; q += 32) h += csr_lookup(a_idx, a_val, lo, hi, topk[u * k + q]) != 0.f;
  for (int e = lo + lane; e < hi; e += 32) rel += a_val[e] > 0.f;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    h += __shfl_xor_sync(0xffffffffu, h, o);
    rel += __shfl_xor_sync(0xffffffffu, rel, o);
  }
  if (lane == 0) {
    hits[u] = (float)h;
    relevant[u] = (float)rel;
  }
}

__device__ __forceinline__ float dcg_discount(int q) {  // rank q+1 -> log1p(q+1)/log(2), :342-346
  return log1pf((float)(q + 1)) / logf(2.0f);
}

__global__ void dcg_kernel(const int* __restrict__ topk, long long n_users, int k, const int* __restrict__ a_ptr,
                           const int* __restrict__ a_idx, const float* __restrict__ a_val, float* __restrict__ dcg) {
  const long long u = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (u >= n_users) return;
  const int lo = a_ptr[u], hi = a_ptr[u + 1];
  float s = 0.f;
  for (int q = 0; q < k; ++q) {
    const float a = csr_lookup(a_idx, a_val, lo, hi, topk[u * k + q]);
    s += (powf(2.0f, a) - 1.0f) / dcg_discount(q);  // :339,:348
  }
  dcg[u] = s;
}

// ideal DCG: gains 2^a - 1 of the row sorted descending -- positives, then the implicit zeros, then
// negatives (:370-384).  One warp per user; q-th pick = next element in (gain desc, position asc) order.
__global__ void idcg_kernel(long long n_users, long long n_items, int k, const int* __restrict__ a_ptr,
                            const float* __restrict__ a_val, float* __restrict__ idcg, float* __restrict__ row_nnz) {
  const long long u = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (u >= n_users) return;
  const int lo = a_ptr[u], hi = a_ptr[u + 1];
  int n_pos = 0, n_neg = 0, n_nz = 0;
  for (int e = lo + lane; e < hi; e += 32) {
    const float g = powf(2.0f, a_val[e]) - 1.0f;
    n_pos += g > 0.f;
    n_neg += g < 0.f;
    n_nz += a_val[e] != 0.f;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    n_pos += __shfl_xor_sync(0xffffffffu, n_pos, o);
    n_neg += __shfl_xor_sync(0xffffffffu, n_neg, o);
    n_nz += __shfl_xor_sync(0xffffffffu, n_nz, o);
  }
  const long long n_zero = n_items - n_pos - n_neg;
  float s = 0.f;
  float prev_g = INFINITY;
  int prev_e = -1;
  for (int q = 0; q < k; ++q) {
    bool want_pos;
    if (q < n_pos) want_pos = true;
    else if (q < n_pos + n_zero) continue;  // a zero gain contributes nothing
    else want_pos = false;
    if (q == n_pos + n_zero) { prev_g = INFINITY; prev_e = -1; }  // restart the scan for the negative tail
    // next element after (prev_g, prev_e) in (gain desc, position asc) order with the wanted sign
    float best_g = -INFINITY;
    int best_e = 0x7fffffff;
    for (int e = lo + lane; e < hi; e += 32) {
      const float g = powf(2.0f, a_val[e]) - 1.0f;
      if (want_pos ? !(g > 0.f) : !(g < 0.f)) continue;
      const bool after_prev = (g < prev_g) || (g == prev_g && e > prev_e);
      if (!after_prev) continue;
      if (g > best_g || (g == best_g && e < best_e)) { best_g = g; best_e = e; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float og = __shfl_xor_sync(0xffffffffu, best_g, o);
      const int oe = __shfl_xor_sync(0xffffffffu, best_e, o);
      if (og > best_g || (og == best_g && oe < best_e)) { best_g = og; best_e = oe; }
    }
    prev_g = best_g;
    prev_e = best_e;
    s += best_g / dcg_discount(q);
  }
  if (lane == 0) {
    idcg[u] = s;
    row_nnz[u] = (float)n_nz;
  }
}

// predict(A)'s second output without a dense A (matrix_factorization.py:197-198: gather_nd(P, where(A == 0)), row-major):
// thread (u, i) looks i up in row u of the CSR of the NON-ZERO cells; an unobserved cell lands at
// u * n_items + i - (#non-zero cells before it in row-major order) = (u * n_items - a_ptr[u]) + (i - lower_bound).
__global__ void gather_unobserved_kernel(const float* __restrict__ P, long long n_users, long long n_items, const int* __restrict__ a_ptr,
                                         const int* __restrict__ a_idx, float* __restrict__ out) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_users * n_items) return;
  const long long u = t / n_items;
  const int i = (int)(t - u * n_items);
  const int a = a_ptr[u], b = a_ptr[u + 1];
  int lo = a, hi = b;  // first stored column >= i
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (a_idx[mid] < i) lo = mid + 1; else hi = mid;
  }
  if (lo < b && a_idx[lo] == i) return;  // observed
  out[t - lo] = P[t];                    // lo = number of non-zero cells before (u, i) in row-major order
}

}  // namespace tmf

using namespace tmf;

extern "C" int tmf_gather_unobserved(const float* P, int64_t n_users, int64_t n_items, const int32_t* a_ptr, const int32_t* a_idx,
                                     float* out, tmf_stream_t stream) {
  TMF_REQUIRE(P && a_ptr && out && n_users >= 0 && n_items >= 0, "tmf_gather_unobserved: bad arguments");
  const long long total = n_users * n_items;
  if (total == 0) return TMF_OK;
  gather_unobserved_kernel<<<(unsigned)cdiv(total, 256), 256, 0, as_stream(stream)>>>(P, n_users, n_items, a_ptr, a_idx, out);
  TMF_LAUNCH_CHECK();
  return TMF_OK;
}

// ------------------------------------------------------------------ measurement aid: embedding-row gather rate
// What user_pass_kernel does to memory, and nothing else: every group of `ld / 4` lanes reads whole rows table[idx[e]] as
// float4 and folds them into registers (one fmaf per element keeps the loads alive).  Timed by bench.py on the workload's own
// index stream, it is the denominator of that kernel's roofline when the table fits the L2 (C3: 6.9 MB), where the HBM
// peak says nothing.
template <int TPR>
__global__ void __launch_bounds__(256) gather_rate_kernel(const float* __restrict__ table, int ld, const int32_t* __restrict__ idx,
                                                          long long n, float* __restrict__ out) {
  const long long grp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) / TPR;
  const long long n_grp = (long long)gridDim.x * blockDim.x / TPR;
  const int l = threadIdx.x % TPR;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  long long e = grp;
  for (; e + 3 * n_grp < n; e += 4 * n_grp) {  // four independent rows in flight per lane
    const int i0 = idx[e], i1 = idx[e + n_grp], i2 = idx[e + 2 * n_grp], i3 = idx[e + 3 * n_grp];
    const float4 a = __ldg(reinterpret_cast<const float4*>(table + (long long)i0 * ld) + l);
    const float4 b = __ldg(reinterpret_cast<const float4*>(table + (long long)i1 * ld) + l);
    const float4 c = __ldg(reinterpret_cast<const float4*>(table + (long long)i2 * ld) + l);
    const float4 d = __ldg(reinterpret_cast<const float4*>(table + (long long)i3 * ld) + l);
    acc.x += a.x + b.x + c.x + d.x; acc.y += a.y + b.y + c.y + d.y;
    acc.z += a.z + b.z + c.z + d.z; acc.w += a.w + b.w + c.w + d.w;
  }
  for (; e < n; e += n_grp) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(table + (long long)idx[e] * ld) + l);
    acc.x += a.x; acc.y += a.y; acc.z += a.z; acc.w += a.w;
  }
  out[(long long)blockIdx.x * blockDim.x + threadIdx.x] = acc.x + acc.y + acc.z + acc.w;
}

extern "C" int tmf_gather_rate(const float* table, int64_t n_rows, int32_t ld, const int32_t* idx, int64_t n, float* out,
                               int64_t out_len, tmf_stream_t stream) {
  TMF_REQUIRE(table && idx && out && n_rows > 0, "tmf_gather_rate: bad arguments");
  TMF_REQUIRE(ld == 64 || ld == 128, "tmf_gather_rate: rows of 64 or 128 floats");
  const int grid = kNumSMs * 8;
  TMF_REQUIRE(out_len >= (int64_t)grid * 256, "tmf_gather_rate: out too small (needs 148 * 8 * 256 floats)");
  if (ld == 64) gather_rate_kernel<16><<<grid, 256, 0, as_stream(stream)>>>(table, ld, idx, n, out);
  else gather_rate_kernel<32><<<grid, 256, 0, as_stream(stream)>>>(table, ld, idx, n, out);
  TMF_LAUNCH_CHECK();
  return TMF_OK;
}

extern "C" int tmf_predict_dense(const float* U, int64_t n_users, const float* V, int64_t n_items, int32_t n_comp, int32_t ld,
                                 float* P, tmf_stream_t stream) {
  TMF_REQUIRE(n_comp > 0 && n_comp <= ld && n_comp <= 1024, "tmf_predict_dense: bad n_components");
  if (n_users == 0 || n_items == 0) return TMF_OK;
  dim3 grid((unsigned)cdiv(n_items, 16), (unsigned)cdiv(n_users, 16));
  TMF_REQUIRE(grid.y <= 65535, "tmf_predict_dense: too many users for the dense path (use tmf_score_topk)");
  const size_t smem = (size_t)32 * n_comp * sizeof(float);
  if (smem > 48 * 1024) TMF_CUDA(cudaFuncSetAttribute(predict_dense_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  predict_dense_kernel<<<grid, 256, smem, as_stream(stream)>>>(U, n_users, V, n_items, n_comp, ld, P);
  TMF_LAUNCH_CHECK();
  return TMF_OK;
}

static size_t seg_sort_temp_bytes(int64_t n, int64_t n_rows) {
  size_t bytes = 0;
  cub::DeviceSegmentedRadixSort::SortPairsDescending(nullptr, bytes, (const float*)nullptr, (float*)nullptr, (const int*)nullptr,
                                                     (int*)nullptr, (int)n, (int)n_rows, (const int*)nullptr, (const int*)nullptr);
  return bytes;
}

extern "C" size_t tmf_rank_rows_ws_bytes(int64_t n_rows, int64_t n_cols) {
  const size_t n = (size_t)((n_rows * n_cols + 63) & ~63ll);
  return seg_sort_temp_bytes(n_rows * n_cols, n_rows) + 3 * n * 4 + (size_t)((n_rows + 64) & ~63ll) * 4 + 1024;
}

extern "C" int tmf_rank_rows(const float* P, int64_t n_rows, int64_t n_cols, int32_t clamp, int32_t* out_idx, void* ws,
                             size_t ws_bytes, tmf_stream_t stream) {
  const long long total = n_rows * n_cols;
  TMF_REQUIRE(total < (1ll << 31), "tmf_rank_rows: n_rows*n_cols must be < 2^31");
  TMF_REQUIRE(ws_bytes >= tmf_rank_rows_ws_bytes(n_rows, n_cols), "tmf_rank_rows: workspace too small");
  if (total == 0) return TMF_OK;
  const size_t n = (size_t)((total + 63) & ~63ll);
  float* keys = reinterpret_cast<float*>(ws);
  float* keys_out = keys + n;
  int* vals = reinterpret_cast<int*>(keys_out + n);
  int* offs = vals + n;
  void* temp = offs + ((n_rows + 64) & ~63ll);
  size_t temp_bytes = seg_sort_temp_bytes(total, n_rows);
  cudaStream_t st = as_stream(stream);
  rank_prep_kernel<<<grid_stride_blocks(cdiv(total, 256), 32), 256, 0, st>>>(P, n_rows, n_cols, clamp, keys, vals, offs);
  TMF_LAUNCH_CHECK();
  // stable LSD radix sort: equal keys keep ascending column order == tf.math.top_k tie order
  TMF_CUDA(cub::DeviceSegmentedRadixSort::SortPairsDescending(temp, temp_bytes, (const float*)keys, keys_out, (const int*)vals, out_idx,
                                                              (int)total, (int)n_rows, offs, offs + 1, 0, 32, st));
  return TMF_OK;
}

extern "C" int tmf_metrics_hits(const int32_t* topk, int64_t n_users, int32_t k, const int32_t* a_ptr, const int32_t* a_idx,
                                const float* a_val, float* hits, float* relevant, tmf_stream_t stream) {
  if (n_users == 0) return TMF_OK;
  metrics_hits_kernel<<<(unsigned)cdiv(n_users * 32, 256), 256, 0, as_stream(stream)>>>(topk, n_users, k, a_ptr, a_idx, a_val, hits, relevant);
  TMF_LAUNCH_CHECK();
  return TMF_OK;
}

extern "C" int tmf_dcg(const int32_t* topk, int64_t n_users, int32_t k, const int32_t* a_ptr, const int32_t* a_idx,
                       const float* a_val, float* dcg, tmf_stream_t stream) {
  if (n_users == 0) return TMF_OK;
  dcg_kernel<<<(unsigned)cdiv(n_users, 128), 128, 0, as_stream(stream)>>>(topk, n_users, k, a_ptr, a_idx, a_val, dcg);
  TMF_LAUNCH_CHECK();
  return TMF_OK;
}

extern "C" int tmf_idcg(int64_t n_users, int64_t n_items, int32_t k, const int32_t* a_ptr, const float* a_val, float* idcg,
                        float* row_nnz, tmf_stream_t stream) {
  if (n_users == 0) return TMF_OK;
  idcg_kernel<<<(unsigned)cdiv(n_users * 32, 256), 256, 0, as_stream(stream)>>>(n_users, n_items, k, a_ptr, a_val, idcg, row_nnz);
  TMF_LAUNCH_CHECK();
  return TMF_OK;
}
