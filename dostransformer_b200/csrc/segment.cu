// CSR segmented reductions (scatter_sum / scatter_mean / pooling / gather adjoints), row gathers and the
// phonon edge features.  HBM-bound: one warp per output row, 16-byte vector accesses, edges of a segment
// are visited in ascending edge id (the order index_add_ / torch_scatter's CPU loop uses), no atomics.
#include "common.cuh"

namespace dost {

template <typename T> struct Acc;
template <> struct Acc<float> {
  static __device__ __forceinline__ void add(float4& a, const float4& b) { a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w; }
  static __device__ __forceinline__ void scale(float4& a, float s) { a.x *= s; a.y *= s; a.z *= s; a.w *= s; }
  static __device__ __forceinline__ float4 zero() { return make_float4(0.f, 0.f, 0.f, 0.f); }
};
template <> struct Acc<double> {
  static __device__ __forceinline__ void add(double2& a, const double2& b) { a.x += b.x; a.y += b.y; }
  static __device__ __forceinline__ void scale(double2& a, double s) { a.x *= s; a.y *= s; }
  static __device__ __forceinline__ double2 zero() { return make_double2(0.0, 0.0); }
};

constexpr int kSegWarps = 8;

// NV vectors per lane: columns (lane + 32*i) * V .. +V
template <typename T, int NV>
__global__ void __launch_bounds__(kSegWarps * 32) segment_reduce_vec_kernel(
    const T* __restrict__ src, long long ld, const int* __restrict__ rowptr, const int* __restrict__ perm,
    long long nseg, int W, int mean, int accumulate, T* __restrict__ out, long long ldo) {
  constexpr int V = VecOf<T>::N;
  using Vec = typename VecOf<T>::type;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nvec = W / V;
  for (long long s = blockIdx.x * (long long)kSegWarps + warp; s < nseg; s += (long long)gridDim.x * kSegWarps) {
    const int beg = __ldg(rowptr + s), end = __ldg(rowptr + s + 1);
    Vec acc[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) acc[i] = Acc<T>::zero();
    // The row indices of (up to) 32 edges are fetched by ONE coalesced load and handed out by shuffles: the row loads of a
    // group then depend on a single index round trip instead of one per 4 rows, and RB rows are in flight per lane (8 measured slower for 256-wide rows: 128 registers, half the resident warps).
    // The sum runs over the edges in ascending CSR order (fixed order, same as before).
    constexpr int RB = NV <= 4 ? 4 : 2;
    for (int base = beg; base < end; base += 32) {
      const int n = min(32, end - base);
      int myrow = base + lane;
      if (perm && lane < n) myrow = __ldg(perm + base + lane);
      int j = 0;
      for (; j + RB <= n; j += RB) {
        Vec v[RB][NV];
#pragma unroll
        for (int k = 0; k < RB; ++k) {
          const long long r = __shfl_sync(0xffffffffu, myrow, j + k);
#pragma unroll
          for (int i = 0; i < NV; ++i) {
            const int c = lane + 32 * i;
            if (c < nvec) v[k][i] = __ldg(reinterpret_cast<const Vec*>(src + r * ld) + c);
          }
        }
#pragma unroll
        for (int k = 0; k < RB; ++k)
#pragma unroll
          for (int i = 0; i < NV; ++i)
            if (lane + 32 * i < nvec) Acc<T>::add(acc[i], v[k][i]);
      }
      for (; j < n; ++j) {
        const long long r = __shfl_sync(0xffffffffu, myrow, j);
#pragma unroll
        for (int i = 0; i < NV; ++i) {
          const int c = lane + 32 * i;
          if (c < nvec) Acc<T>::add(acc[i], __ldg(reinterpret_cast<const Vec*>(src + r * ld) + c));
        }
      }
    }
    const int cnt = end - beg;
    const T sc = (mean && cnt > 1) ? T(1) / T(cnt) : T(1);
    T* orow = out + s * ldo;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c = lane + 32 * i;
      if (c < nvec) {
        Vec v = acc[i];
        if (mean) Acc<T>::scale(v, sc);
        Vec* op = reinterpret_cast<Vec*>(orow) + c;
        if (accumulate) {
          Vec o = *op;
          Acc<T>::add(o, v);
          v = o;
        }
        *op = v;
      }
    }
  }
}

// Few segments (per-crystal reductions: the adjoint of a broadcast over the T energy tokens, crystal pooling): one BLOCK per
// segment instead of one warp - a warp walking 201 rows serially took 56-65 us at any batch size.  Warp w sums rows
// beg + w, beg + w + 8, ... in ascending order, then the 8 partial sums are added in warp order: a fixed order.
template <typename T, int NV>
__global__ void __launch_bounds__(kSegWarps * 32) segment_reduce_block_kernel(
    const T* __restrict__ src, long long ld, const int* __restrict__ rowptr, const int* __restrict__ perm,
    long long nseg, int W, int mean, int accumulate, T* __restrict__ out, long long ldo) {
  constexpr int V = VecOf<T>::N;
  using Vec = typename VecOf<T>::type;
  __shared__ Vec part[kSegWarps][NV * 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nvec = W / V;
  for (long long s = blockIdx.x; s < nseg; s += gridDim.x) {
    const int beg = __ldg(rowptr + s), end = __ldg(rowptr + s + 1);
    Vec acc[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) acc[i] = Acc<T>::zero();
    int j = beg + warp;
    for (; j + 3 * kSegWarps < end; j += 4 * kSegWarps) {     // four rows in flight per lane
      long long r[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) r[k] = perm ? (long long)__ldg(perm + j + k * kSegWarps) : (long long)(j + k * kSegWarps);
      Vec v[4][NV];
#pragma unroll
      for (int k = 0; k < 4; ++k)
#pragma unroll
        for (int i = 0; i < NV; ++i)
          if (lane + 32 * i < nvec) v[k][i] = __ldg(reinterpret_cast<const Vec*>(src + r[k] * ld) + lane + 32 * i);
#pragma unroll
      for (int k = 0; k < 4; ++k)
#pragma unroll
        for (int i = 0; i < NV; ++i)
          if (lane + 32 * i < nvec) Acc<T>::add(acc[i], v[k][i]);
    }
    for (; j < end; j += kSegWarps) {
      const long long r = perm ? (long long)__ldg(perm + j) : (long long)j;
#pragma unroll
      for (int i = 0; i < NV; ++i)
        if (lane + 32 * i < nvec) Acc<T>::add(acc[i], __ldg(reinterpret_cast<const Vec*>(src + r * ld) + lane + 32 * i));
    }
#pragma unroll
    for (int i = 0; i < NV; ++i) part[warp][lane + 32 * i] = acc[i];
    __syncthreads();
    const int cnt = end - beg;
    const T sc = (mean && cnt > 1) ? T(1) / T(cnt) : T(1);
    for (int c = threadIdx.x; c < nvec; c += kSegWarps * 32) {
      Vec v = part[0][c];
#pragma unroll
      for (int w = 1; w < kSegWarps; ++w) Acc<T>::add(v, part[w][c]);
      if (mean) Acc<T>::scale(v, sc);
      Vec* op = reinterpret_cast<Vec*>(out + s * ldo) + c;
      if (accumulate) {
        Vec o = *op;
        Acc<T>::add(o, v);
        v = o;
      }
      *op = v;
    }
    __syncthreads();
  }
}

// scalar fallback for unaligned / odd widths
template <typename T>
__global__ void __launch_bounds__(kSegWarps * 32) segment_reduce_scalar_kernel(
    const T* __restrict__ src, long long ld, const int* __restrict__ rowptr, const int* __restrict__ perm,
    long long nseg, int W, int mean, int accumulate, T* __restrict__ out, long long ldo) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (long long s = blockIdx.x * (long long)kSegWarps + warp; s < nseg; s += (long long)gridDim.x * kSegWarps) {
    const int beg = __ldg(rowptr + s), end = __ldg(rowptr + s + 1);
    const int cnt = end - beg;
    const T sc = (mean && cnt > 1) ? T(1) / T(cnt) : T(1);
    for (int c = lane; c < W; c += 32) {
      T a = T(0);
      for (int j = beg; j < end; ++j) {
        const long long r = perm ? (long long)__ldg(perm + j) : (long long)j;
        a += __ldg(src + r * ld + c);
      }
      if (mean) a *= sc;
      T* op = out + s * ldo + c;
      *op = accumulate ? (*op + a) : a;
    }
  }
}

template <typename T, int NV>
__global__ void __launch_bounds__(kSegWarps * 32) gather_rows_vec_kernel(
    const T* __restrict__ src, long long ld, const int* __restrict__ idx, const int* __restrict__ deg_rowptr,
    const T* __restrict__ add, long long ld_add, long long R, int W, T* __restrict__ out, long long ldo,
    const unsigned char* __restrict__ mask) {
  constexpr int V = VecOf<T>::N;
  using Vec = typename VecOf<T>::type;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nvec = W / V;
  for (long long r = blockIdx.x * (long long)kSegWarps + warp; r < R; r += (long long)gridDim.x * kSegWarps) {
    if (mask && !__ldg(mask + r)) {      // a masked row: written as 0, idx[r] never read
      for (int c = lane; c < W; c += 32) out[r * ldo + c] = T(0);
      continue;
    }
    const long long s = __ldg(idx + r);
    T sc = T(1);
    if (deg_rowptr) {
      const int cnt = __ldg(deg_rowptr + s + 1) - __ldg(deg_rowptr + s);
      if (cnt > 1) sc = T(1) / T(cnt);
    }
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c = lane + 32 * i;
      if (c < nvec) {
        Vec v = __ldg(reinterpret_cast<const Vec*>(src + s * ld) + c);
        if (deg_rowptr) Acc<T>::scale(v, sc);
        if (add) Acc<T>::add(v, __ldg(reinterpret_cast<const Vec*>(add + r * ld_add) + c));
        reinterpret_cast<Vec*>(out + r * ldo)[c] = v;
      }
    }
  }
}

template <typename T>
__global__ void __launch_bounds__(kSegWarps * 32) gather_rows_scalar_kernel(
    const T* __restrict__ src, long long ld, const int* __restrict__ idx, const int* __restrict__ deg_rowptr,
    const T* __restrict__ add, long long ld_add, long long R, int W, T* __restrict__ out, long long ldo,
    const unsigned char* __restrict__ mask) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (long long r = blockIdx.x * (long long)kSegWarps + warp; r < R; r += (long long)gridDim.x * kSegWarps) {
    if (mask && !__ldg(mask + r)) {
      for (int c = lane; c < W; c += 32) out[r * ldo + c] = T(0);
      continue;
    }
    const long long s = __ldg(idx + r);
    T sc = T(1);
    if (deg_rowptr) {
      const int cnt = __ldg(deg_rowptr + s + 1) - __ldg(deg_rowptr + s);
      if (cnt > 1) sc = T(1) / T(cnt);
    }
    for (int c = lane; c < W; c += 32) {
      T v = __ldg(src + s * ld + c) * sc;
      if (add) v += __ldg(add + r * ld_add + c);
      out[r * ldo + c] = v;
    }
  }
}

// smooth_cutoff(|v|/4) * [1, sqrt(3) v/|v|]; zero vector -> [cutoff(0)=1, 0, 0, 0]
template <typename T>
__global__ void phonon_edge_feat_kernel(const T* __restrict__ vec, long long E, T* __restrict__ out) {
  long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (e >= E) return;
  const T x = vec[3 * e], y = vec[3 * e + 1], z = vec[3 * e + 2];
  const T len = sqrt(x * x + y * y + z * z);
  const T inv = T(1) / max(len, T(1e-12));
  const T u = T(2) * (len / T(4) - T(1));
  T cut;
  if (u > T(0)) cut = T(0);
  else if (u < T(-1)) cut = T(1);
  else cut = (T(1) - cos(T(3.14159265358979323846) * u)) / T(2);
  const T s3 = T(1.7320508075688772935);
  out[4 * e + 0] = cut;
  out[4 * e + 1] = cut * s3 * x * inv;
  out[4 * e + 2] = cut * s3 * y * inv;
  out[4 * e + 3] = cut * s3 * z * inv;
}

// The same features computed INSIDE the first Linear of the edge encoder (DOSTransformer_phonon.py:74-77 -> GN_encoder.
// edge_encoder[0..1]): pre[e, c] = b[c] + sum_k W[c, k] feat_k(edge_vec[e]); out = PReLU(pre).  The [E, 4] feature tensor
// never exists.  One warp per edge: the 4 features are computed once per lane, lanes cover the H columns (coalesced rows).
template <typename T>
__global__ void __launch_bounds__(256) phonon_edge_encode_kernel(const T* __restrict__ vec, long long E, const T* __restrict__ W,
                                                                 const T* __restrict__ bias, const T* __restrict__ slope_p, int H,
                                                                 T* __restrict__ pre, T* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const long long e = blockIdx.x * 8LL + (threadIdx.x >> 5);
  if (e >= E) return;
  const T x = vec[3 * e], y = vec[3 * e + 1], z = vec[3 * e + 2];
  const T len = sqrt(x * x + y * y + z * z);
  const T inv = T(1) / max(len, T(1e-12));
  const T u = T(2) * (len / T(4) - T(1));
  T cut;
  if (u > T(0)) cut = T(0);
  else if (u < T(-1)) cut = T(1);
  else cut = (T(1) - cos(T(3.14159265358979323846) * u)) / T(2);
  const T s3 = T(1.7320508075688772935);
  const T f0 = cut, f1 = cut * s3 * x * inv, f2 = cut * s3 * y * inv, f3 = cut * s3 * z * inv;
  const T slope = slope_p ? slope_p[0] : T(1);
  for (int c = lane; c < H; c += 32) {
    // the accumulation order of the generic GEMM kernel (k ascending, fused multiply-adds, bias last)
    T v = fma(W[4 * c + 0], f0, T(0));
    v = fma(W[4 * c + 1], f1, v);
    v = fma(W[4 * c + 2], f2, v);
    v = fma(W[4 * c + 3], f3, v);
    if (bias) v += bias[c];
    if (pre) pre[e * H + c] = v;
    out[e * H + c] = (v > T(0)) ? v : slope * v;
  }
}

// Input gradient of the kernel above: d_vec[e] = J(e)^T g(e) with g_k = sum_c dv[e, c] W[c, k] (dv = gradient at the
// pre-activation) and J the Jacobian of feat(v) = cut(|v|) [1, sqrt(3) v / max(|v|, 1e-12)], differentiated the way torch
// autograd differentiates the reference's expression (oracle/dost_oracle.py phonon_edge_features): cut' = 0 where the
// torch.where branches replace it (u > 0 or u < -1), else (pi/4) sin(pi u); the clamp passes the norm's gradient for
// |v| >= 1e-12 (clamp_min's backward) and otherwise divides by the constant 1e-12 - the zero vector of a self-interaction
// edge therefore gets sqrt(3) * 1e12 * g[1..3], as in the reference.  One warp per edge, lanes over the H columns (dv is
// read once, coalesced); the four column sums are reduced by a fixed butterfly (bitwise reproducible).
template <typename T>
__global__ void __launch_bounds__(256) phonon_edge_encode_bwd_kernel(const T* __restrict__ vec, long long E,
                                                                     const T* __restrict__ W, const T* __restrict__ dv, int H,
                                                                     T* __restrict__ d_vec) {
  const int lane = threadIdx.x & 31;
  const long long e = blockIdx.x * 8LL + (threadIdx.x >> 5);
  if (e >= E) return;
  T g0 = T(0), g1 = T(0), g2 = T(0), g3 = T(0);
  const T* row = dv + e * H;
  for (int c = lane; c < H; c += 32) {
    const T d = row[c];
    g0 = fma(d, W[4 * c + 0], g0);
    g1 = fma(d, W[4 * c + 1], g1);
    g2 = fma(d, W[4 * c + 2], g2);
    g3 = fma(d, W[4 * c + 3], g3);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    g0 += __shfl_xor_sync(0xffffffffu, g0, o);
    g1 += __shfl_xor_sync(0xffffffffu, g1, o);
    g2 += __shfl_xor_sync(0xffffffffu, g2, o);
    g3 += __shfl_xor_sync(0xffffffffu, g3, o);
  }
  if (lane >= 3) return;
  const T v[3] = {vec[3 * e], vec[3 * e + 1], vec[3 * e + 2]};
  const T len = sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]);
  const T u = T(2) * (len / T(4) - T(1));
  const T pi = T(3.14159265358979323846);
  const T s3 = T(1.7320508075688772935);
  T cut, dcut;                        // cut(|v|) and d cut / d|v|
  if (u > T(0)) cut = T(0), dcut = T(0);
  else if (u < T(-1)) cut = T(1), dcut = T(0);
  else cut = (T(1) - cos(pi * u)) / T(2), dcut = (pi / T(4)) * sin(pi * u);
  // lane l < 3 writes component l (selects, not indexed arrays: no local memory)
  const T gl = lane == 0 ? g1 : (lane == 1 ? g2 : g3);
  const T vl = lane == 0 ? v[0] : (lane == 1 ? v[1] : v[2]);
  T r;
  if (len >= T(1e-12)) {
    const T inv = T(1) / len;
    const T gn = (g1 * v[0] + g2 * v[1] + g3 * v[2]) * inv;
    const T nl = vl * inv;
    // d cut/dv = dcut n;  d(n_i)/dv = (I - n n^T) / |v|
    r = dcut * (g0 + s3 * gn) * nl + s3 * cut * (gl - nl * gn) * inv;
  } else {
    // |v| < 2 here, so cut is the constant 1 and only the clamped direction contributes
    r = s3 * cut * gl / T(1e-12);
  }
  d_vec[3 * e + lane] = r;
}

static inline bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

template <typename T>
static int run_segment_reduce(const void* src, long long ld, const int* rowptr, const int* perm, long long nseg, int W,
                              int mean, int accumulate, void* out, long long ldo, cudaStream_t st) {
  constexpr int V = VecOf<T>::N;
  int blocks = (int)min64((nseg + kSegWarps - 1) / kSegWarps, 32LL * kNumSMs);
  const bool vec = (W % V == 0) && (ld % V == 0) && (ldo % V == 0) && al16(src) && al16(out) && W <= 32 * V * 8;
  if (vec && nseg <= 1024 && W <= 32 * V * 4) {      // few segments: a block per segment (see segment_reduce_block_kernel)
    const int nv = (W / V + 31) / 32;
    const int nb = (int)nseg;
#define DOST_SEGB(NV)                                                                                                    \
  segment_reduce_block_kernel<T, NV><<<nb, kSegWarps * 32, 0, st>>>((const T*)src, ld, rowptr, perm, nseg, W, mean, accumulate, \
                                                                    (T*)out, ldo)
    if (nv <= 1) DOST_SEGB(1);
    else if (nv <= 2) DOST_SEGB(2);
    else DOST_SEGB(4);
#undef DOST_SEGB
    return check_launch("segment_reduce");
  }
  if (vec) {
    const int nv = (W / V + 31) / 32;
#define DOST_SEG(NV)                                                                                              \
  segment_reduce_vec_kernel<T, NV><<<blocks, kSegWarps * 32, 0, st>>>((const T*)src, ld, rowptr, perm, nseg, W, mean, \
                                                                      accumulate, (T*)out, ldo)
    if (nv <= 1) DOST_SEG(1);
    else if (nv <= 2) DOST_SEG(2);
    else if (nv <= 4) DOST_SEG(4);
    else DOST_SEG(8);
#undef DOST_SEG
  } else {
    segment_reduce_scalar_kernel<T><<<blocks, kSegWarps * 32, 0, st>>>((const T*)src, ld, rowptr, perm, nseg, W, mean,
                                                                       accumulate, (T*)out, ldo);
  }
  return check_launch("segment_reduce");
}

template <typename T>
static int run_gather_rows(const void* src, long long ld, const int* idx, const int* deg_rowptr, const void* add,
                           long long ld_add, long long R, int W, void* out, long long ldo, const uint8_t* mask,
                           cudaStream_t st) {
  constexpr int V = VecOf<T>::N;
  int blocks = (int)min64((R + kSegWarps - 1) / kSegWarps, 32LL * kNumSMs);
  bool vec = (W % V == 0) && (ld % V == 0) && (ldo % V == 0) && al16(src) && al16(out) && W <= 32 * V * 8;
  if (add) vec = vec && (ld_add % V == 0) && al16(add);
  if (vec) {
    const int nv = (W / V + 31) / 32;
#define DOST_GR(NV)                                                                                              \
  gather_rows_vec_kernel<T, NV><<<blocks, kSegWarps * 32, 0, st>>>((const T*)src, ld, idx, deg_rowptr, (const T*)add, \
                                                                   ld_add, R, W, (T*)out, ldo, mask)
    if (nv <= 1) DOST_GR(1);
    else if (nv <= 2) DOST_GR(2);
    else if (nv <= 4) DOST_GR(4);
    else DOST_GR(8);
#undef DOST_GR
  } else {
    gather_rows_scalar_kernel<T><<<blocks, kSegWarps * 32, 0, st>>>((const T*)src, ld, idx, deg_rowptr, (const T*)add,
                                                                    ld_add, R, W, (T*)out, ldo, mask);
  }
  return check_launch("gather_rows");
}

}  // namespace dost

using namespace dost;

extern "C" int dost_segment_reduce(int dtype, const void* src, long long ld, const int32_t* rowptr,
                                   const int32_t* perm, long long nseg, int W, int mean, int accumulate, void* out,
                                   long long ldo, dost_stream_t stream) {
  if (nseg == 0) return DOST_OK;
  DOST_REQUIRE(src && rowptr && out && nseg > 0 && W > 0, "segment_reduce: bad args");
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == DOST_F32) return run_segment_reduce<float>(src, ld, rowptr, perm, nseg, W, mean, accumulate, out, ldo, st);
  if (dtype == DOST_F64) return run_segment_reduce<double>(src, ld, rowptr, perm, nseg, W, mean, accumulate, out, ldo, st);
  set_error("segment_reduce: unsupported dtype %d", dtype);
  return DOST_ERR_UNSUPPORTED;
}

extern "C" int dost_gather_rows(int dtype, const void* src, long long ld, const int32_t* idx,
                                const int32_t* deg_rowptr, const void* add, long long ld_add, long long R, int W,
                                void* out, long long ldo, dost_stream_t stream) {
  if (R == 0) return DOST_OK;
  DOST_REQUIRE(src && idx && out && R > 0 && W > 0, "gather_rows: bad args");
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == DOST_F32) return run_gather_rows<float>(src, ld, idx, deg_rowptr, add, ld_add, R, W, out, ldo, nullptr, st);
  if (dtype == DOST_F64) return run_gather_rows<double>(src, ld, idx, deg_rowptr, add, ld_add, R, W, out, ldo, nullptr, st);
  set_error("gather_rows: unsupported dtype %d", dtype);
  return DOST_ERR_UNSUPPORTED;
}

extern "C" int dost_gather_rows_masked(int dtype, const void* src, long long ld, const int32_t* idx,
                                       const int32_t* deg_rowptr, const uint8_t* mask, const void* add, long long ld_add,
                                       long long R, int W, void* out, long long ldo, dost_stream_t stream) {
  if (R == 0) return DOST_OK;
  DOST_REQUIRE(src && idx && mask && out && R > 0 && W > 0, "gather_rows_masked: bad args");
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == DOST_F32) return run_gather_rows<float>(src, ld, idx, deg_rowptr, add, ld_add, R, W, out, ldo, mask, st);
  if (dtype == DOST_F64) return run_gather_rows<double>(src, ld, idx, deg_rowptr, add, ld_add, R, W, out, ldo, mask, st);
  set_error("gather_rows_masked: unsupported dtype %d", dtype);
  return DOST_ERR_UNSUPPORTED;
}

extern "C" int dost_phonon_edge_feat(int dtype, const void* edge_vec, long long E, void* out, dost_stream_t stream) {
  if (E == 0) return DOST_OK;
  DOST_REQUIRE(edge_vec && out && E > 0, "phonon_edge_feat: bad args");
  cudaStream_t st = (cudaStream_t)stream;
  const int blocks = ceil_div(E, 256);
  if (dtype == DOST_F32) phonon_edge_feat_kernel<float><<<blocks, 256, 0, st>>>((const float*)edge_vec, E, (float*)out);
  else if (dtype == DOST_F64) phonon_edge_feat_kernel<double><<<blocks, 256, 0, st>>>((const double*)edge_vec, E, (double*)out);
  else {
    set_error("phonon_edge_feat: unsupported dtype %d", dtype);
    return DOST_ERR_UNSUPPORTED;
  }
  return check_launch("phonon_edge_feat");
}

extern "C" int dost_phonon_edge_encode(int dtype, const void* edge_vec, long long E, const void* weight, const void* bias,
                                       const void* prelu_slope, int H, void* pre, void* out, dost_stream_t stream) {
  if (E == 0) return DOST_OK;
  DOST_REQUIRE(edge_vec && weight && out && E > 0 && H > 0, "phonon_edge_encode: bad args");
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned blocks = (unsigned)((E + 7) / 8);
  if (dtype == DOST_F32)
    phonon_edge_encode_kernel<float><<<blocks, 256, 0, st>>>((const float*)edge_vec, E, (const float*)weight, (const float*)bias,
                                                             (const float*)prelu_slope, H, (float*)pre, (float*)out);
  else if (dtype == DOST_F64)
    phonon_edge_encode_kernel<double><<<blocks, 256, 0, st>>>((const double*)edge_vec, E, (const double*)weight, (const double*)bias,
                                                              (const double*)prelu_slope, H, (double*)pre, (double*)out);
  else {
    set_error("phonon_edge_encode: unsupported dtype %d", dtype);
    return DOST_ERR_UNSUPPORTED;
  }
  return check_launch("phonon_edge_encode");
}

extern "C" int dost_phonon_edge_encode_bwd(int dtype, const void* edge_vec, long long E, const void* weight, const void* dv,
                                           int H, void* d_edge_vec, dost_stream_t stream) {
  if (E == 0) return DOST_OK;
  DOST_REQUIRE(edge_vec && weight && dv && d_edge_vec && E > 0 && H > 0, "phonon_edge_encode_bwd: bad args");
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned blocks = (unsigned)((E + 7) / 8);
  if (dtype == DOST_F32)
    phonon_edge_encode_bwd_kernel<float><<<blocks, 256, 0, st>>>((const float*)edge_vec, E, (const float*)weight,
                                                                 (const float*)dv, H, (float*)d_edge_vec);
  else if (dtype == DOST_F64)
    phonon_edge_encode_bwd_kernel<double><<<blocks, 256, 0, st>>>((const double*)edge_vec, E, (const double*)weight,
                                                                  (const double*)dv, H, (double*)d_edge_vec);
  else {
    set_error("phonon_edge_encode_bwd: unsupported dtype %d", dtype);
    return DOST_ERR_UNSUPPORTED;
  }
  return check_launch("phonon_edge_encode_bwd");
}
