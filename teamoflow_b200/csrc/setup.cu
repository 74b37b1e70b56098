// One-time-per-fit structure builders and initialisers: CSR row pointers, stable transposes
// (item-major views), negative sampler, Philox initialisers, error plumbing.
#include <cub/device/device_radix_sort.cuh>
#include <stdarg.h>

#include <algorithm>

#include "common.cuh"

namespace tmf {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

// ptr[j] = first position in sorted `keys` with keys[pos] >= j   (j in [0, n_keys])
__global__ void lower_bound_kernel(const int* __restrict__ keys, long long n, int n_keys, int* __restrict__ ptr) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j > n_keys) return;
  long long lo = 0, hi = n;
  while (lo < hi) {
    const long long mid = (lo + hi) >> 1;
    if (keys[mid] < j) lo = mid + 1; else hi = mid;
  }
  ptr[j] = (int)lo;
}

// COO indices [nnz, 2] (int32 or int64, tf.sparse.SparseTensor.indices layout) -> int32 rows / cols in one pass, with the two
// checks the host needs before it may use them: flags bit 0 = an id outside [0, n_rows) x [0, n_cols), bit 1 = not in
// row-major order (stored order is kept; the caller then sorts).
template <typename T>
__global__ void coo_split_kernel(const T* __restrict__ idx2, long long nnz, long long n_rows, long long n_cols, int* __restrict__ rows,
                                 int* __restrict__ cols, int* __restrict__ flags) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long stride = (long long)gridDim.x * blockDim.x;
  int f = 0;
  for (; i < nnz; i += stride) {
    const long long r = (long long)idx2[2 * i], c = (long long)idx2[2 * i + 1];
    if (r < 0 || r >= n_rows || c < 0 || c >= n_cols) f |= 1;
    if (i > 0) {
      const long long pr = (long long)idx2[2 * i - 2], pc = (long long)idx2[2 * i - 1];
      if (pr > r || (pr == r && pc > c)) f |= 2;
    }
    rows[i] = (int)r;
    cols[i] = (int)c;
  }
  if (f) atomicOr(flags, f);
}

__global__ void iota_kernel(int* __restrict__ x, long long n) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < n; i += stride) x[i] = (int)i;
}

__global__ void tlist_users_kernel(const int* __restrict__ perm, long long n, long long nnz, const int* __restrict__ coo_rows,
                                   int S, int* __restrict__ users) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < n; i += stride) {
    const long long e = perm[i];
    users[i] = e < nnz ? coo_rows[e] : (int)((e - nnz) / S);
  }
}

// ---- counter-based RNG (Philox4x32-10)
struct Philox {
  static __device__ __forceinline__ uint4 gen(uint64_t ctr, uint64_t key) {
    uint32_t c0 = (uint32_t)ctr, c1 = (uint32_t)(ctr >> 32), c2 = 0x2545F491u, c3 = 0x9E3779B9u;
    uint32_t k0 = (uint32_t)key, k1 = (uint32_t)(key >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
      const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
      const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
      const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
      c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
      k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
  }
};

__device__ __forceinline__ float u01(uint32_t x) { return (float)(x >> 8) * (1.0f / 16777216.0f); }  // [0,1)

template <int NORMAL>
__global__ void fill_kernel(float* __restrict__ w, long long n_rows, int n_cols, int ld, uint64_t seed) {
  const long long total = n_rows * n_cols;
  long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;  // quad index
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (; q * 4 < total; q += stride) {
    const uint4 r = Philox::gen((uint64_t)q, seed);
    float v[4];
    if (NORMAL) {  // Box-Muller on two uniform pairs; (0,1] for the log argument
      const float u0 = 1.0f - u01(r.x), u1 = u01(r.y), u2 = 1.0f - u01(r.z), u3 = u01(r.w);
      const float r0 = sqrtf(-2.0f * logf(u0)), r1 = sqrtf(-2.0f * logf(u2));
      float s0, c0, s1, c1;
      sincospif(2.0f * u1, &s0, &c0);
      sincospif(2.0f * u3, &s1, &c1);
      v[0] = r0 * c0; v[1] = r0 * s0; v[2] = r1 * c1; v[3] = r1 * s1;
    } else {
      v[0] = u01(r.x); v[1] = u01(r.y); v[2] = u01(r.z); v[3] = u01(r.w);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const long long e = q * 4 + i;
      if (e < total) w[(e / n_cols) * ld + (e % n_cols)] = v[i];
    }
  }
}

// keyed bijection of [0, n): 4-round Feistel on 2*hb bits + cycle walking
__device__ __forceinline__ uint32_t mix32(uint32_t x) {
  x ^= x >> 16; x *= 0x85EBCA6Bu; x ^= x >> 13; x *= 0xC2B2AE35u; x ^= x >> 16;
  return x;
}

__global__ void sample_items_kernel(int n_users, int n_items, int S, uint64_t seed, long long* __restrict__ out, int hb) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)n_users * S) return;
  const uint32_t u = (uint32_t)(i / S);
  uint32_t x = (uint32_t)(i % S);
  const uint32_t mask = (1u << hb) - 1u;
  const uint32_t ku = mix32(u * 0x9E3779B1u + (uint32_t)seed) ^ (uint32_t)(seed >> 32);
  do {
    uint32_t L = x >> hb, R = x & mask;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const uint32_t f = mix32(R ^ ku ^ (0xA511E9B3u * (r + 1))) & mask;
      const uint32_t nl = R;
      R = L ^ f;
      L = nl;
    }
    x = (L << hb) | R;
  } while (x >= (uint32_t)n_items);
  out[i] = (long long)x;
}

}  // namespace tmf

using namespace tmf;

extern "C" int tmf_abi_version(void) { return TMF_ABI_VERSION; }
extern "C" const char* tmf_last_error(void) { return g_err; }

extern "C" int tmf_rowptr_from_sorted(const int32_t* rows, int64_t nnz, int32_t n_rows, int32_t* row_ptr, tmf_stream_t stream) {
  TMF_REQUIRE(n_rows >= 0 && nnz >= 0 && nnz < (1ll << 31), "tmf_rowptr_from_sorted: bad sizes");
  lower_bound_kernel<<<(unsigned)cdiv(n_rows + 1, 256), 256, 0, as_stream(stream)>>>(rows, nnz, n_rows, row_ptr);
  TMF_LAUNCH_CHECK();
  return TMF_OK;
}

extern "C" int tmf_coo_split(const void* indices, int32_t index_bytes, int64_t nnz, int64_t n_rows, int64_t n_cols, int32_t* rows,
                             int32_t* cols, int32_t* flags, tmf_stream_t stream) {
  TMF_REQUIRE(index_bytes == 4 || index_bytes == 8, "tmf_coo_split: indices must be int32 or int64");
  TMF_REQUIRE(flags != nullptr && nnz >= 0 && nnz < (1ll << 31) && n_rows < (1ll << 31) && n_cols < (1ll << 31), "tmf_coo_split: bad sizes");
  cudaStream_t st = as_stream(stream);
  TMF_CUDA(cudaMemsetAsync(flags, 0, sizeof(int), st));
  if (nnz == 0) return TMF_OK;
  const unsigned grid = grid_stride_blocks(cdiv(nnz, 256), 16);
  if (index_bytes == 8)
    coo_split_kernel<long long><<<grid, 256, 0, st>>>(reinterpret_cast<const long long*>(indices), nnz, n_rows, n_cols, rows, cols, flags);
  else
    coo_split_kernel<int><<<grid, 256, 0, st>>>(reinterpret_cast<const int*>(indices), nnz, n_rows, n_cols, rows, cols, flags);
  TMF_LAUNCH_CHECK();
  return TMF_OK;
}

static size_t sort_temp_bytes(int64_t n) {
  size_t bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, bytes, (const int*)nullptr, (int*)nullptr, (const int*)nullptr, (int*)nullptr, (int)n);
  return bytes;
}

extern "C" size_t tmf_transpose_ws_bytes(int64_t n) {
  const size_t nn = (size_t)((n + 63) & ~63ll);
  return sort_temp_bytes(n) + 2 * nn * sizeof(int) + 1024;
}

extern "C" int tmf_transpose_build(const int32_t* keys, int64_t n, int32_t n_keys, int32_t* ptr, int32_t* perm, void* ws,
                                   size_t ws_bytes, tmf_stream_t stream) {
  TMF_REQUIRE(n >= 0 && n < (1ll << 31) && n_keys >= 0, "tmf_transpose_build: bad sizes");
  TMF_REQUIRE(ws_bytes >= tmf_transpose_ws_bytes(n), "tmf_transpose_build: workspace too small");
  cudaStream_t st = as_stream(stream);
  const size_t nn = (size_t)((n + 63) & ~63ll);
  int* keys_out = reinterpret_cast<int*>(ws);
  int* iota = keys_out + nn;
  void* temp = iota + nn;
  size_t temp_bytes = ws_bytes - 2 * nn * sizeof(int);
  if (n > 0) {
    iota_kernel<<<grid_stride_blocks(cdiv(n, 256), 16), 256, 0, st>>>(iota, n);
    int end_bit = 1;
    while (end_bit < 31 && (1ll << end_bit) < (long long)n_keys) ++end_bit;
    TMF_CUDA(cub::DeviceRadixSort::SortPairs(temp, temp_bytes, keys, keys_out, (const int*)iota, perm, (int)n, 0, end_bit, st));
  }
  lower_bound_kernel<<<(unsigned)cdiv(n_keys + 1, 256), 256, 0, st>>>(keys_out, n, n_keys, ptr);
  TMF_LAUNCH_CHECK();
  return TMF_OK;
}

extern "C" int tmf_tlist_users(const int32_t* perm, int64_t n, int64_t nnz, const int32_t* coo_rows, int32_t n_samples,
                               int32_t* users_out, tmf_stream_t stream) {
  if (n == 0) return TMF_OK;
  TMF_REQUIRE(n_samples > 0 || n <= nnz, "tmf_tlist_users: n_samples must be > 0 when the list holds samples");
  tlist_users_kernel<<<grid_stride_blocks(cdiv(n, 256), 16), 256, 0, as_stream(stream)>>>(
      perm, n, nnz, coo_rows, n_samples > 0 ? n_samples : 1, users_out);
  TMF_LAUNCH_CHECK();
  return TMF_OK;
}

extern "C" int tmf_sample_items(int32_t n_users, int32_t n_items, int32_t n_samples, uint64_t seed, int64_t* out,
                                tmf_stream_t stream) {
  TMF_REQUIRE(n_samples <= n_items, "tmf_sample_items: n_samples (%d) must be <= n_items (%d) without replacement",
              n_samples, n_items);  // numpy raises here too (utils.py:20)
  TMF_REQUIRE(n_items > 0 && n_users >= 0 && n_samples >= 0, "tmf_sample_items: bad sizes");
  const long long n = (long long)n_users * n_samples;
  if (n == 0) return TMF_OK;
  int bits = 1;
  while ((1ll << bits) < n_items) ++bits;
  const int hb = std::max(1, (bits + 1) / 2);
  sample_items_kernel<<<(unsigned)cdiv(n, 256), 256, 0, as_stream(stream)>>>(n_users, n_items, n_samples, seed,
                                                                          reinterpret_cast<long long*>(out), hb);
  TMF_LAUNCH_CHECK();
  return TMF_OK;
}

static int fill_common(int normal, float* w, int64_t n_rows, int32_t n_cols, int32_t ld, uint64_t seed, tmf_stream_t stream) {
  TMF_REQUIRE(w && n_rows >= 0 && n_cols >= 0 && n_cols <= ld, "tmf_fill: bad shape");
  const long long quads = cdiv(n_rows * n_cols, 4);
  if (quads == 0) return TMF_OK;
  const unsigned grid = grid_stride_blocks(cdiv(quads, 256), 32);
  if (normal) fill_kernel<1><<<grid, 256, 0, as_stream(stream)>>>(w, n_rows, n_cols, ld, seed);
  else fill_kernel<0><<<grid, 256, 0, as_stream(stream)>>>(w, n_rows, n_cols, ld, seed);
  TMF_LAUNCH_CHECK();
  return TMF_OK;
}

extern "C" int tmf_fill_normal(float* w, int64_t n_rows, int32_t n_cols, int32_t ld, uint64_t seed, tmf_stream_t stream) {
  return fill_common(1, w, n_rows, n_cols, ld, seed, stream);
}
extern "C" int tmf_fill_uniform(float* w, int64_t n_rows, int32_t n_cols, int32_t ld, uint64_t seed, tmf_stream_t stream) {
  return fill_common(0, w, n_rows, n_cols, ld, seed, stream);
}
