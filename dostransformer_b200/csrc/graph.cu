// Integer graph structure: int64->int32 cast and stable counting sort to CSR.
// Bit-exact against torch.sort(stable=True) / bincount / cumsum (oracle/dost_oracle.py: csr_by_key).
// The masked build (mask != NULL) sorts only the entries with mask[i] != 0 and lists the others after rowptr[size] in
// index order; every kernel below serves both builds, the unmasked one with mask == NULL.
#include "common.cuh"

namespace dost {

__global__ void cast_i64_i32_kernel(const long long* __restrict__ src, int* __restrict__ dst, long long n) {
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < n; i += stride) dst[i] = static_cast<int>(src[i]);
}

// Keys outside [0, size) are skipped (they belong to no segment) and reported through the device error word: the
// reference raises IndexError there; writing cnt[key] unchecked would corrupt the neighbouring allocations.
__global__ void hist_kernel(const int* __restrict__ key, const unsigned char* __restrict__ mask, int* __restrict__ cnt,
                            long long n, long long size, unsigned int* __restrict__ errw) {
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < n; i += stride) {
    if (mask && !mask[i]) continue;
    const int k = key[i];
    if (static_cast<unsigned long long>(k) < static_cast<unsigned long long>(size)) atomicAdd(&cnt[k], 1);  // integer counts
    else if (errw) errw[kErrIndexRange] = 1u;
  }
}

// Single-block exclusive scan of cnt[size] -> rowptr[size+1], cursor[size]; also max(cnt).  With a mask, the masked
// entries (mask[i] == 0) then go to perm[rowptr[size]..n) in index order: a second chunked scan, of their counts.
__global__ void __launch_bounds__(1024) scan_kernel(const int* __restrict__ cnt, int* __restrict__ rowptr,
                                                    int* __restrict__ cursor, int* __restrict__ maxcount,
                                                    long long size, const unsigned char* __restrict__ mask, long long n,
                                                    int* __restrict__ perm) {
  __shared__ int part[1024];
  __shared__ int pmax[1024];
  const int t = threadIdx.x;
  const long long chunk = (size + 1023) / 1024;
  const long long beg = t * chunk, end = min(size, beg + chunk);
  int s = 0, mx = 0;
  for (long long i = beg; i < end; ++i) {
    int c = cnt[i];
    s += c;
    mx = max(mx, c);
  }
  part[t] = s;
  pmax[t] = mx;
  __syncthreads();
  // Hillis-Steele inclusive scan over the 1024 partials (ints: exact in any order)
  for (int off = 1; off < 1024; off <<= 1) {
    int v = (t >= off) ? part[t - off] : 0;
    int m = (t >= off) ? pmax[t - off] : 0;
    __syncthreads();
    part[t] += v;
    pmax[t] = max(pmax[t], m);
    __syncthreads();
  }
  int run = (t == 0) ? 0 : part[t - 1];
  for (long long i = beg; i < end; ++i) {
    rowptr[i] = run;
    cursor[i] = run;
    run += cnt[i];
  }
  if (t == 1023) {
    rowptr[size] = part[1023];
    if (maxcount) *maxcount = pmax[1023];
  }
  if (!mask) return;
  const int live = part[1023];
  __syncthreads();
  const long long mchunk = (n + 1023) / 1024;
  const long long mbeg = t * mchunk, mend = min(n, mbeg + mchunk);
  int z = 0;
  for (long long i = mbeg; i < mend; ++i) z += (mask[i] == 0);
  part[t] = z;
  __syncthreads();
  for (int off = 1; off < 1024; off <<= 1) {
    int v = (t >= off) ? part[t - off] : 0;
    __syncthreads();
    part[t] += v;
    __syncthreads();
  }
  int at = live + ((t == 0) ? 0 : part[t - 1]);
  for (long long i = mbeg; i < mend; ++i)
    if (mask[i] == 0) perm[at++] = static_cast<int>(i);
}

__global__ void fill_kernel(const int* __restrict__ key, const unsigned char* __restrict__ mask, int* __restrict__ cursor,
                            int* __restrict__ tmp, long long n, long long size) {
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < n; i += stride) {
    if (mask && !mask[i]) continue;
    const int k = key[i];
    if (static_cast<unsigned long long>(k) >= static_cast<unsigned long long>(size)) continue;
    int pos = atomicAdd(&cursor[k], 1);
    tmp[pos] = static_cast<int>(i);
  }
}

// One warp per segment: rank sort of the (unique) element ids so each segment is ascending == stable order.
__global__ void rank_sort_kernel(const int* __restrict__ rowptr, const int* __restrict__ tmp, int* __restrict__ perm,
                                 long long size) {
  const int lane = threadIdx.x & 31;
  long long seg = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (; seg < size; seg += nwarps) {
    const int beg = rowptr[seg], end = rowptr[seg + 1];
    const int d = end - beg;
    if (d <= 32) {
      int v = (lane < d) ? tmp[beg + lane] : 0x7fffffff;
      int rank = 0;
#pragma unroll 1
      for (int j = 0; j < d; ++j) {
        int o = __shfl_sync(0xffffffffu, v, j);
        rank += (o < v);
      }
      if (lane < d) perm[beg + rank] = v;
    } else {
      for (int i = lane; i < d; i += 32) {
        const int v = tmp[beg + i];
        int rank = 0;
        for (int j = 0; j < d; ++j) rank += (tmp[beg + j] < v);
        perm[beg + rank] = v;
      }
    }
  }
}

__global__ void imax_scalar_kernel(int* __restrict__ v, int floor_value) {
  if (threadIdx.x == 0 && blockIdx.x == 0 && *v < floor_value) *v = floor_value;
}

}  // namespace dost

using namespace dost;

extern "C" int dost_imax_scalar(int32_t* value, int32_t floor_value, dost_stream_t stream) {
  DOST_REQUIRE(value, "imax_scalar: null pointer");
  imax_scalar_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(value, floor_value);
  return check_launch("imax_scalar");
}

extern "C" int dost_cast_i64_i32(const int64_t* src, int32_t* dst, long long n, dost_stream_t stream) {
  if (n == 0) return DOST_OK;
  DOST_REQUIRE(src && dst && n > 0, "cast_i64_i32: bad args");
  int blocks = min(ceil_div(n, 256), kNumSMs * 8);
  cast_i64_i32_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>((const long long*)src, dst, n);
  return check_launch("cast_i64_i32");
}

extern "C" size_t dost_csr_workspace_bytes(long long n, long long size) {
  return sizeof(int) * (size_t)(2 * size + n + 8);
}

static int csr_build(const int32_t* key, const uint8_t* mask, long long n, long long size, int32_t* rowptr,
                     int32_t* perm, int32_t* maxcount, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  if (workspace_bytes < dost_csr_workspace_bytes(n, size) || !workspace) {
    set_error("csr_build: workspace too small");
    return DOST_ERR_WORKSPACE;
  }
  int* cnt = (int*)workspace;
  int* cursor = cnt + size;
  int* tmp = cursor + size;
  cudaMemsetAsync(cnt, 0, sizeof(int) * size, st);
  if (n > 0) {
    int blocks = min(ceil_div(n, 256), kNumSMs * 8);
    hist_kernel<<<blocks, 256, 0, st>>>(key, mask, cnt, n, size, device_error_words());
    count_launch();
  }
  scan_kernel<<<1, 1024, 0, st>>>(cnt, rowptr, cursor, maxcount, size, mask, n, perm);
  count_launch();
  if (n > 0) {
    int blocks = min(ceil_div(n, 256), kNumSMs * 8);
    fill_kernel<<<blocks, 256, 0, st>>>(key, mask, cursor, tmp, n, size);
    count_launch();
    int sblocks = min(ceil_div(size * 32, 256), kNumSMs * 16);
    rank_sort_kernel<<<sblocks, 256, 0, st>>>(rowptr, tmp, perm, size);
  }
  return check_launch("csr_build");
}

extern "C" int dost_csr_build(const int32_t* key, long long n, long long size, int32_t* rowptr, int32_t* perm,
                              int32_t* maxcount, void* workspace, size_t workspace_bytes, dost_stream_t stream) {
  DOST_REQUIRE(key && rowptr && perm && size > 0 && n >= 0, "csr_build: bad args");
  return csr_build(key, nullptr, n, size, rowptr, perm, maxcount, workspace, workspace_bytes, (cudaStream_t)stream);
}

extern "C" int dost_csr_build_masked(const int32_t* key, const uint8_t* mask, long long n, long long size, int32_t* rowptr,
                                     int32_t* perm, int32_t* maxcount, void* workspace, size_t workspace_bytes,
                                     dost_stream_t stream) {
  DOST_REQUIRE(rowptr && perm && size > 0 && n >= 0 && (n == 0 || (key && mask)), "csr_build_masked: bad args");
  return csr_build(key, mask, n, size, rowptr, perm, maxcount, workspace, workspace_bytes, (cudaStream_t)stream);
}
