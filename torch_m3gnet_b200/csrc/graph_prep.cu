// Graph canonicalisation kernels: index narrowing, CSR construction, sortedness/symmetry checks,
// exclusive scan.  Integer work only; everything here runs once per batch and is cached by the host.
#include <stdarg.h>

#include "common.cuh"

namespace m3g {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

__global__ void narrow_kernel(const int64_t* __restrict__ in, int32_t* __restrict__ out, int64_t n) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = (int32_t)in[i];
}

__global__ void check_sorted_kernel(const int32_t* __restrict__ keys, int64_t n, int64_t n_rows,
                                    int32_t* __restrict__ flags) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int32_t k = keys[i];
  if (k < 0 || k >= n_rows) flags[1] = 0;
  if (i + 1 < n && keys[i + 1] < k) flags[0] = 0;
}

__global__ void set_flags_kernel(int32_t* flags, int n, int32_t v) {
  if (threadIdx.x < n) flags[threadIdx.x] = v;
}

// row_ptr[r] = lower_bound(keys, r)
__global__ void csr_from_sorted_kernel(const int32_t* __restrict__ keys, int64_t n, int64_t n_rows,
                                       int32_t* __restrict__ row_ptr) {
  int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r > n_rows) return;
  int64_t lo = 0, hi = n;
  while (lo < hi) {
    int64_t mid = (lo + hi) >> 1;
    if (keys[mid] < (int32_t)r) lo = mid + 1; else hi = mid;
  }
  row_ptr[r] = (int32_t)lo;
}

__global__ void zero_i32_kernel(int32_t* p, int64_t n) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = 0;
}

__global__ void histogram_kernel(const int32_t* __restrict__ keys, int64_t n, int32_t* __restrict__ count) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) atomicAdd(&count[keys[i]], 1);
}

// ---------------- exclusive scan (three phases, any n) ----------------
constexpr int SCAN_THREADS = 256;
constexpr int SCAN_ITEMS = 8;
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

__device__ __forceinline__ int32_t block_exclusive_scan(int32_t v, int32_t* total, int32_t* smem) {
  // inclusive warp scan
  int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int32_t x = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int32_t y = __shfl_up_sync(FULL, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) smem[w] = x;
  __syncthreads();
  if (w == 0) {
    int32_t s = (lane < SCAN_THREADS / 32) ? smem[lane] : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int32_t y = __shfl_up_sync(FULL, s, o);
      if (lane >= o) s += y;
    }
    smem[32 + lane] = s;  // inclusive scan of warp totals
  }
  __syncthreads();
  int32_t warp_off = (w == 0) ? 0 : smem[32 + w - 1];
  *total = smem[32 + SCAN_THREADS / 32 - 1];
  return warp_off + x - v;
}

// phase 1: per-tile local exclusive scan written to out[0..n), tile totals to work[tile]
__global__ void scan_tiles_kernel(const int32_t* __restrict__ in, int32_t* __restrict__ out, int64_t n,
                                  int32_t* __restrict__ work) {
  __shared__ int32_t smem[64];
  int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
  int32_t v[SCAN_ITEMS];
  int32_t s = 0;
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; ++k) {
    v[k] = (base + k < n) ? in[base + k] : 0;
    s += v[k];
  }
  int32_t total;
  int32_t off = block_exclusive_scan(s, &total, smem);
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; ++k) {
    if (base + k < n) out[base + k] = off;
    off += v[k];
  }
  if (threadIdx.x == 0) work[blockIdx.x] = total;
}

// phase 2: one block scans the tile totals sequentially in chunks (exclusive, in place); grand total → work[n_tiles]
__global__ void scan_totals_kernel(int32_t* __restrict__ work, int64_t n_tiles) {
  __shared__ int32_t smem[64];
  __shared__ int32_t carry_s;
  if (threadIdx.x == 0) carry_s = 0;
  __syncthreads();
  for (int64_t start = 0; start < n_tiles; start += SCAN_THREADS) {
    int64_t i = start + threadIdx.x;
    int32_t v = (i < n_tiles) ? work[i] : 0;
    int32_t total;
    int32_t off = block_exclusive_scan(v, &total, smem);
    int32_t carry = carry_s;
    if (i < n_tiles) work[i] = carry + off;
    __syncthreads();
    if (threadIdx.x == 0) carry_s = carry + total;
    __syncthreads();
  }
  if (threadIdx.x == 0) work[n_tiles] = carry_s;
}

// phase 3: add tile offsets; out[n] = grand total
__global__ void scan_add_kernel(int32_t* __restrict__ out, int64_t n, const int32_t* __restrict__ work,
                                int64_t n_tiles) {
  int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
  int32_t add = work[blockIdx.x];
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; ++k)
    if (base + k < n) out[base + k] += add;
  if (blockIdx.x == 0 && threadIdx.x == 0) out[n] = work[n_tiles];
}

static int launch_scan(const int32_t* in, int32_t* out, int64_t n, int32_t* work, cudaStream_t st) {
  int64_t n_tiles = (n + SCAN_TILE - 1) / SCAN_TILE;
  if (n_tiles < 1) n_tiles = 1;
  scan_tiles_kernel<<<(unsigned)n_tiles, SCAN_THREADS, 0, st>>>(in, out, n, work);
  scan_totals_kernel<<<1, SCAN_THREADS, 0, st>>>(work, n_tiles);
  scan_add_kernel<<<(unsigned)n_tiles, SCAN_THREADS, 0, st>>>(out, n, work, n_tiles);
  return 0;
}

// fill: position i goes to slot row_ptr[key] + atomic counter (unordered), then rows are sorted
__global__ void csr_fill_kernel(const int32_t* __restrict__ keys, int64_t n, const int32_t* __restrict__ row_ptr,
                                int32_t* __restrict__ cursor, int32_t* __restrict__ perm) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int32_t k = keys[i];
  int32_t slot = row_ptr[k] + atomicAdd(&cursor[k], 1);
  perm[slot] = (int32_t)i;
}

// in-place ascending insertion sort of every CSR row (rows are short: a neighbour shell)
__global__ void sort_rows_kernel(const int32_t* __restrict__ row_ptr, int64_t n_rows, int32_t* __restrict__ cols) {
  int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_rows) return;
  int32_t b = row_ptr[r], e = row_ptr[r + 1];
  for (int32_t i = b + 1; i < e; ++i) {
    int32_t v = cols[i];
    int32_t j = i - 1;
    while (j >= b && cols[j] > v) {
      cols[j + 1] = cols[j];
      --j;
    }
    cols[j + 1] = v;
  }
}

__global__ void gather_i32_kernel(const int32_t* __restrict__ vals, const int32_t* __restrict__ perm, int64_t n,
                                  int32_t* __restrict__ out) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = vals[perm[i]];
}

// symmetric iff for every (r, c) the pair (c, r) occurs as often as (r, c): the transpose is then the matrix itself,
// repeated entries included (a repeated triplet is summed once per occurrence, so the transpose must repeat it too).
// Rows sorted ascending: each run of c in row r is compared with the run of r in row c (two binary searches).
__global__ void csr_symmetric_kernel(const int32_t* __restrict__ row_ptr, const int32_t* __restrict__ cols,
                                     int64_t n_rows, int32_t* __restrict__ flags) {
  int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_rows) return;
  const int32_t end = row_ptr[r + 1];
  for (int32_t p = row_ptr[r]; p < end;) {
    const int32_t c = cols[p];
    if (c < 0 || c >= n_rows) { flags[0] = 0; return; }
    int32_t q = p + 1;
    while (q < end && cols[q] == c) ++q;
    int32_t lo = row_ptr[c], hi = row_ptr[c + 1];
    while (lo < hi) {  // lower bound of r in row c
      const int32_t mid = (lo + hi) >> 1;
      if (cols[mid] < (int32_t)r) lo = mid + 1; else hi = mid;
    }
    int32_t m = lo;
    hi = row_ptr[c + 1];
    while (m < hi && cols[m] == (int32_t)r) ++m;
    if (m - lo != q - p) { flags[0] = 0; return; }
    p = q;
  }
}

__global__ void rows_gather_kernel(const float* __restrict__ in, const int32_t* __restrict__ idx, int64_t n, int W,
                                   float* __restrict__ out) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * W) return;
  int64_t r = i / W;
  int c = (int)(i - r * W);
  out[i] = in[(int64_t)idx[r] * W + c];
}

// idx rows are unique per call (a ghost atom maps to exactly one owner row) → plain add, no atomics
__global__ void rows_scatter_add_kernel(const float* __restrict__ add, const int32_t* __restrict__ idx, int64_t n,
                                        int W, float* __restrict__ inout) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * W) return;
  int64_t r = i / W;
  int c = (int)(i - r * W);
  atomicAdd(&inout[(int64_t)idx[r] * W + c], add[i]);
}

// halo push over NVLink: row r of the selection goes to the absolute device address dst_addr[r] — a slot of a PEER
// GPU's landing buffer (symmetric memory, peer-mapped pointer).  The pack and the transfer are one kernel: coalesced
// 16-byte stores straight into the peer's HBM through NVSwitch, no staging buffer and no collective call.
__global__ void rows_put_kernel(const float* __restrict__ in, const int32_t* __restrict__ idx,
                                const int64_t* __restrict__ dst_addr, int64_t n, int W) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if ((W & 3) == 0) {
    const int W4 = W >> 2;
    if (i >= n * W4) return;
    const int64_t r = i / W4;
    const int c = (int)(i - r * W4);
    const int64_t row = idx ? idx[r] : r;
    reinterpret_cast<float4*>(dst_addr[r])[c] = __ldg(reinterpret_cast<const float4*>(in + row * W) + c);
  } else {
    if (i >= n * W) return;
    const int64_t r = i / W;
    const int c = (int)(i - r * W);
    const int64_t row = idx ? idx[r] : r;
    reinterpret_cast<float*>(dst_addr[r])[c] = in[row * W + c];
  }
}

}  // namespace m3g

using namespace m3g;

extern "C" {

const char* m3g_last_error(void) { return g_err; }
int m3g_abi_version(void) { return 1; }

int m3g_device_info(int* out_host) {
  M3G_REQUIRE(out_host, "m3g_device_info: null output");
  int dev = 0;
  cudaDeviceProp prop;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaGetDeviceProperties(&prop, dev) != cudaSuccess) {
    set_error("m3g_device_info: no CUDA device");
    return M3G_ERR_CUDA;
  }
  out_host[0] = prop.multiProcessorCount;
  out_host[1] = prop.major;
  out_host[2] = prop.minor;
  return M3G_OK;
}

int m3g_narrow_i64(const int64_t* in, int32_t* out, int64_t n, void* stream) {
  if (n == 0) return M3G_OK;
  M3G_REQUIRE(in && out, "m3g_narrow_i64: null pointer");
  narrow_kernel<<<blocks_for(n, 256), 256, 0, as_stream(stream)>>>(in, out, n);
  M3G_LAUNCH_CHECK("m3g_narrow_i64");
  return M3G_OK;
}

int m3g_check_sorted(const int32_t* keys, int64_t n, int64_t n_rows, int32_t* flags, void* stream) {
  M3G_REQUIRE(flags, "m3g_check_sorted: null flags");
  set_flags_kernel<<<1, 32, 0, as_stream(stream)>>>(flags, 2, 1);
  if (n > 0) {
    M3G_REQUIRE(keys, "m3g_check_sorted: null keys");
    check_sorted_kernel<<<blocks_for(n, 256), 256, 0, as_stream(stream)>>>(keys, n, n_rows, flags);
  }
  M3G_LAUNCH_CHECK("m3g_check_sorted");
  return M3G_OK;
}

int m3g_csr_from_sorted(const int32_t* keys, int64_t n, int64_t n_rows, int32_t* row_ptr, void* stream) {
  M3G_REQUIRE(row_ptr && (keys || n == 0), "m3g_csr_from_sorted: null pointer");
  csr_from_sorted_kernel<<<blocks_for(n_rows + 1, 256), 256, 0, as_stream(stream)>>>(keys, n, n_rows, row_ptr);
  M3G_LAUNCH_CHECK("m3g_csr_from_sorted");
  return M3G_OK;
}

int64_t m3g_scan_work_elems(int64_t n) { return (n + SCAN_TILE - 1) / SCAN_TILE + 2; }

int m3g_exclusive_scan_i32(const int32_t* in, int32_t* out, int64_t n, int32_t* work, void* stream) {
  M3G_REQUIRE(out && work && (in || n == 0), "m3g_exclusive_scan_i32: null pointer");
  launch_scan(in, out, n, work, as_stream(stream));
  M3G_LAUNCH_CHECK("m3g_exclusive_scan_i32");
  return M3G_OK;
}

int m3g_csr_by_key(const int32_t* keys, int64_t n, int64_t n_rows, int32_t* row_ptr, int32_t* perm, int32_t* work,
                   void* stream) {
  M3G_REQUIRE(row_ptr && work && (n == 0 || (keys && perm)), "m3g_csr_by_key: null pointer");
  cudaStream_t st = as_stream(stream);
  // work: [0, n_rows] counts / cursors; scan scratch lives after it
  int32_t* count = work;
  int32_t* scan_work = work + (n_rows + 1);
  zero_i32_kernel<<<blocks_for(n_rows + 1, 256), 256, 0, st>>>(count, n_rows + 1);
  if (n > 0) histogram_kernel<<<blocks_for(n, 256), 256, 0, st>>>(keys, n, count);
  launch_scan(count, row_ptr, n_rows, scan_work, st);
  zero_i32_kernel<<<blocks_for(n_rows + 1, 256), 256, 0, st>>>(count, n_rows + 1);
  if (n > 0) {
    csr_fill_kernel<<<blocks_for(n, 256), 256, 0, st>>>(keys, n, row_ptr, count, perm);
    sort_rows_kernel<<<blocks_for(n_rows, 128), 128, 0, st>>>(row_ptr, n_rows, perm);
  }
  M3G_LAUNCH_CHECK("m3g_csr_by_key");
  return M3G_OK;
}

int m3g_gather_i32(const int32_t* vals, const int32_t* perm, int64_t n, int32_t* out, void* stream) {
  if (n == 0) return M3G_OK;
  M3G_REQUIRE(vals && perm && out, "m3g_gather_i32: null pointer");
  gather_i32_kernel<<<blocks_for(n, 256), 256, 0, as_stream(stream)>>>(vals, perm, n, out);
  M3G_LAUNCH_CHECK("m3g_gather_i32");
  return M3G_OK;
}

int m3g_sort_rows(const int32_t* row_ptr, int64_t n_rows, int32_t* cols, void* stream) {
  if (n_rows == 0) return M3G_OK;
  M3G_REQUIRE(row_ptr && cols, "m3g_sort_rows: null pointer");
  sort_rows_kernel<<<blocks_for(n_rows, 128), 128, 0, as_stream(stream)>>>(row_ptr, n_rows, cols);
  M3G_LAUNCH_CHECK("m3g_sort_rows");
  return M3G_OK;
}

int m3g_csr_is_symmetric(const int32_t* row_ptr, const int32_t* cols, int64_t n_rows, int32_t* flags, void* stream) {
  M3G_REQUIRE(row_ptr && flags, "m3g_csr_is_symmetric: null pointer");
  set_flags_kernel<<<1, 32, 0, as_stream(stream)>>>(flags, 1, 1);
  if (n_rows > 0)
    csr_symmetric_kernel<<<blocks_for(n_rows, 128), 128, 0, as_stream(stream)>>>(row_ptr, cols, n_rows, flags);
  M3G_LAUNCH_CHECK("m3g_csr_is_symmetric");
  return M3G_OK;
}

int m3g_rows_gather(const float* in, const int32_t* idx, int64_t n, int W, float* out, void* stream) {
  if (n == 0) return M3G_OK;
  M3G_REQUIRE(in && idx && out && W > 0, "m3g_rows_gather: bad argument");
  rows_gather_kernel<<<blocks_for(n * W, 256), 256, 0, as_stream(stream)>>>(in, idx, n, W, out);
  M3G_LAUNCH_CHECK("m3g_rows_gather");
  return M3G_OK;
}

int m3g_rows_put(const float* in, const int32_t* idx, const int64_t* dst_addr, int64_t n, int W, void* stream) {
  if (n == 0) return M3G_OK;
  M3G_REQUIRE(in && dst_addr && W > 0, "m3g_rows_put: bad argument");
  const int64_t work = (W & 3) == 0 ? n * (W >> 2) : n * W;
  rows_put_kernel<<<blocks_for(work, 256), 256, 0, as_stream(stream)>>>(in, idx, dst_addr, n, W);
  M3G_LAUNCH_CHECK("m3g_rows_put");
  return M3G_OK;
}

int m3g_rows_scatter_add(const float* add, const int32_t* idx, int64_t n, int W, float* inout, void* stream) {
  if (n == 0) return M3G_OK;
  M3G_REQUIRE(add && idx && inout && W > 0, "m3g_rows_scatter_add: bad argument");
  rows_scatter_add_kernel<<<blocks_for(n * W, 256), 256, 0, as_stream(stream)>>>(add, idx, n, W, inout);
  M3G_LAUNCH_CHECK("m3g_rows_scatter_add");
  return M3G_OK;
}

}  // extern "C"
