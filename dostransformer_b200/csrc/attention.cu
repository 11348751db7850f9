// Ragged energy->atom cross attention with analytic phantom keys, and the fp32 row softmax used by the
// dense energy self attention.  See include/dost.h for the reference semantics being reproduced
// (zero padding by to_dense_batch + LayerNorm => (Nmax - n_b) phantom keys equal to layer_norms[0].bias).
//
// Layout: q/out [S, T, H], kv [N, H]; sequence s reads crystal b = s % B, keys ptr[b]..ptr[b+1].
// One warp per query, lane l owns features l, l+32, ...; keys are staged in shared memory tiles; online
// softmax in fp32 (the reference forces fp32 softmax even for the float64 phonon model).
#include <math.h>
#include <cuda_bf16.h>
#include "common.cuh"

namespace dost {

// fp32, H in {128, 256, 512}: FMA-bound kernels in attention_v2.cu
bool xattn_v2_supported(int H);
int xattn_v2_fwd(const float* q, long long q_ss, const float* kv, const float* phantom, const int* ptr, const int* nmax,
                 const float* resid, long long r_ss, float* out, float* lse, int S, int B, int Tn, int H, float scale,
                 unsigned int thresh, float inv_keep, unsigned long long seed, const unsigned long long* seed_offset,
                 cudaStream_t st);
int xattn_v2_bwd(const float* dO, const float* q, long long q_ss, const float* kv, const float* phantom, const int* ptr,
                 const int* nmax, const float* out, const float* resid, long long r_ss, const float* lse, float* dq, float* dkv,
                 float* Dbuf, float* part, int S, int B, int Tn, int H, float scale, unsigned int thresh, float inv_keep,
                 unsigned long long seed, const unsigned long long* seed_offset, bool do_kv, cudaStream_t st);

constexpr int kQPW = 4;               // queries per warp
constexpr int kAttWarps = 8;
constexpr int kQPB = kQPW * kAttWarps;  // queries per block
constexpr int kKT = 32;               // keys per shared tile

template <typename T, int HV>
__device__ __forceinline__ void load_row(const T* __restrict__ p, int lane, T (&v)[HV]) {
#pragma unroll
  for (int i = 0; i < HV; ++i) v[i] = p[lane + 32 * i];
}

template <typename T, int HV>
__device__ __forceinline__ T dot_partial(const T (&a)[HV], const T (&b)[HV]) {
  T s = T(0);
#pragma unroll
  for (int i = 0; i < HV; ++i) s = fma(a[i], b[i], s);
  return s;
}

// ------------------------------------------------------------------------------------------------ forward
template <typename T, int HV>
__global__ void __launch_bounds__(kAttWarps * 32) xattn_fwd_kernel(
    const T* __restrict__ q, long long q_ss, const T* __restrict__ kv, const T* __restrict__ phantom,
    const int* __restrict__ ptr, const int* __restrict__ nmax_p, const T* __restrict__ resid, long long r_ss,
    T* __restrict__ out, float* __restrict__ lse, int S, int B, int Tn, T scale, unsigned int thresh, float inv_keep,
    unsigned long long seed, const unsigned long long* __restrict__ seed_offset) {
  constexpr int H = 32 * HV;
  seed = mask_seed(seed, seed_offset);
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* ks = reinterpret_cast<T*>(smem_raw);  // [kKT][H]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int s = blockIdx.y;
  const int b = s % B;
  const int kbeg = ptr[b], kend = ptr[b + 1];
  const int nb = kend - kbeg;
  const int nmax = *nmax_p;
  const int nph = max(nmax - nb, 0);
  const int t0 = blockIdx.x * kQPB + warp * kQPW;

  T qv[kQPW][HV], acc[kQPW][HV];
  float m[kQPW], l[kQPW];
#pragma unroll
  for (int qi = 0; qi < kQPW; ++qi) {
    const int t = min(t0 + qi, Tn - 1);
    load_row<T, HV>(q + (long long)s * q_ss + (long long)t * H, lane, qv[qi]);
#pragma unroll
    for (int i = 0; i < HV; ++i) acc[qi][i] = T(0);
    m[qi] = -INFINITY;
    l[qi] = 0.f;
  }

  for (int j0 = 0; j0 < nb; j0 += kKT) {
    const int kt = min(kKT, nb - j0);
    __syncthreads();
    for (int i = threadIdx.x; i < kt * H; i += blockDim.x) ks[i] = kv[(long long)(kbeg + j0) * H + i];
    __syncthreads();
    for (int j = 0; j < kt; ++j) {
      T kk[HV];
#pragma unroll
      for (int i = 0; i < HV; ++i) kk[i] = ks[j * H + lane + 32 * i];
      T d[kQPW];
#pragma unroll
      for (int qi = 0; qi < kQPW; ++qi) d[qi] = dot_partial<T, HV>(qv[qi], kk);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int qi = 0; qi < kQPW; ++qi) d[qi] += __shfl_xor_sync(0xffffffffu, d[qi], o);
      }
#pragma unroll
      for (int qi = 0; qi < kQPW; ++qi) {
        const float sf = static_cast<float>(d[qi] * scale);
        const float mn = fmaxf(m[qi], sf);
        const float corr = expf(m[qi] - mn);
        const float p = expf(sf - mn);
        l[qi] = l[qi] * corr + p;
        m[qi] = mn;
        float w = p;
        if (thresh) {
          const int t = t0 + qi;
          const unsigned long long idx = ((unsigned long long)s * Tn + t) * (unsigned long long)nmax + (j0 + j);
          w = keep_mask(seed, idx, thresh) ? p * inv_keep : 0.f;
        }
        const T c = static_cast<T>(corr), wt = static_cast<T>(w);
#pragma unroll
        for (int i = 0; i < HV; ++i) acc[qi][i] = fma(wt, kk[i], acc[qi][i] * c);
      }
    }
  }
  // phantom keys: nph copies of k = v = phantom
  if (nph > 0) {
    T pk[HV];
    load_row<T, HV>(phantom, lane, pk);
#pragma unroll
    for (int qi = 0; qi < kQPW; ++qi) {
      T d = warp_sum(dot_partial<T, HV>(qv[qi], pk));
      const float sf = static_cast<float>(d * scale);
      const float mn = fmaxf(m[qi], sf);
      const float corr = expf(m[qi] - mn);
      const float p = expf(sf - mn);
      l[qi] = l[qi] * corr + p * (float)nph;
      m[qi] = mn;
      float w = p * (float)nph;
      if (thresh) {
        const int t = t0 + qi;
        int kept = 0;
        for (int jj = nb + lane; jj < nmax; jj += 32) {
          const unsigned long long idx = ((unsigned long long)s * Tn + t) * (unsigned long long)nmax + jj;
          kept += keep_mask(seed, idx, thresh) ? 1 : 0;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) kept += __shfl_xor_sync(0xffffffffu, kept, o);
        w = p * inv_keep * (float)kept;
      }
      const T c = static_cast<T>(corr), wt = static_cast<T>(w);
#pragma unroll
      for (int i = 0; i < HV; ++i) acc[qi][i] = fma(wt, pk[i], acc[qi][i] * c);
    }
  }
#pragma unroll
  for (int qi = 0; qi < kQPW; ++qi) {
    const int t = t0 + qi;
    if (t < Tn) {
      const T inv = static_cast<T>(1.0f / l[qi]);
      const T* rr = resid + (long long)s * r_ss + (long long)t * H;
      T* oo = out + ((long long)s * Tn + t) * H;
#pragma unroll
      for (int i = 0; i < HV; ++i) oo[lane + 32 * i] = rr[lane + 32 * i] + acc[qi][i] * inv;
      if (lane == 0) lse[(long long)s * Tn + t] = m[qi] + logf(l[qi]);
    }
  }
}

// ------------------------------------------------------------------------------------------------ attention maps
// The probabilities of a forward recomputed from its log-sum-exp, in the reference's padded layout (attn_weights of
// multihead_attention.py:68-71 after to_dense_batch): map[s, t, j] = exp(q_t . k_j scale - lse[s, t]) for the n_b atoms,
// the same value for each of the phantom key slots n_b .. nmax - 1, 0 past nmax; with dropout mask / (1 - p) times that,
// the mask regenerated per slot (index (s T + t) nmax + j, as in the forward).  Scoring loop of xattn_fwd_kernel.
template <typename T, int HV>
__global__ void __launch_bounds__(kAttWarps * 32) xattn_probs_kernel(
    const T* __restrict__ q, long long q_ss, const T* __restrict__ kv, const T* __restrict__ phantom,
    const int* __restrict__ ptr, const int* __restrict__ nmax_p, const float* __restrict__ lse, T* __restrict__ out, int cols,
    int S, int B, int Tn, T scale, unsigned int thresh, float inv_keep, unsigned long long seed,
    const unsigned long long* __restrict__ seed_offset) {
  constexpr int H = 32 * HV;
  seed = mask_seed(seed, seed_offset);
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* ks = reinterpret_cast<T*>(smem_raw);  // [kKT][H]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int s = blockIdx.y;
  const int b = s % B;
  const int kbeg = ptr[b], kend = ptr[b + 1];
  const int nb = kend - kbeg;
  const int nmax = *nmax_p;
  const int t0 = blockIdx.x * kQPB + warp * kQPW;

  T qv[kQPW][HV];
  float ls[kQPW];
#pragma unroll
  for (int qi = 0; qi < kQPW; ++qi) {
    const int t = min(t0 + qi, Tn - 1);
    load_row<T, HV>(q + (long long)s * q_ss + (long long)t * H, lane, qv[qi]);
    ls[qi] = lse[(long long)s * Tn + t];
  }

  for (int j0 = 0; j0 < nb; j0 += kKT) {
    const int kt = min(kKT, nb - j0);
    __syncthreads();
    for (int i = threadIdx.x; i < kt * H; i += blockDim.x) ks[i] = kv[(long long)(kbeg + j0) * H + i];
    __syncthreads();
    float mine[kQPW] = {0.f, 0.f, 0.f, 0.f};     // lane j keeps key j0 + j of the tile
    for (int j = 0; j < kt; ++j) {
      T kk[HV];
#pragma unroll
      for (int i = 0; i < HV; ++i) kk[i] = ks[j * H + lane + 32 * i];
      T d[kQPW];
#pragma unroll
      for (int qi = 0; qi < kQPW; ++qi) d[qi] = dot_partial<T, HV>(qv[qi], kk);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int qi = 0; qi < kQPW; ++qi) d[qi] += __shfl_xor_sync(0xffffffffu, d[qi], o);
      }
#pragma unroll
      for (int qi = 0; qi < kQPW; ++qi) {
        float p = expf(static_cast<float>(d[qi] * scale) - ls[qi]);
        if (thresh) {
          const unsigned long long idx = ((unsigned long long)s * Tn + t0 + qi) * (unsigned long long)nmax + (j0 + j);
          p = keep_mask(seed, idx, thresh) ? p * inv_keep : 0.f;
        }
        mine[qi] = (lane == j) ? p : mine[qi];
      }
    }
#pragma unroll
    for (int qi = 0; qi < kQPW; ++qi) {
      const int t = t0 + qi;
      if (t < Tn && lane < kt && j0 + lane < cols) out[((long long)s * Tn + t) * cols + j0 + lane] = static_cast<T>(mine[qi]);
    }
  }
  // phantom slots (each the probability of ONE zero-padded key), then zeros
  T pk[HV];
  if (nmax > nb) load_row<T, HV>(phantom, lane, pk);
#pragma unroll
  for (int qi = 0; qi < kQPW; ++qi) {
    float pph = 0.f;
    if (nmax > nb) pph = expf(static_cast<float>(warp_sum(dot_partial<T, HV>(qv[qi], pk)) * scale) - ls[qi]);
    const int t = t0 + qi;
    if (t >= Tn) continue;
    T* orow = out + ((long long)s * Tn + t) * cols;
    for (int c = nb + lane; c < cols; c += 32) {
      float v = 0.f;
      if (c < nmax) {
        v = pph;
        if (thresh) v = keep_mask(seed, ((unsigned long long)s * Tn + t) * (unsigned long long)nmax + c, thresh) ? v * inv_keep : 0.f;
      }
      orow[c] = static_cast<T>(v);
    }
  }
}

// ------------------------------------------------------------------------------------------------ backward: dq
// Also writes D[s,t] = dO . (out - resid) and per-block partial sums of the phantom-key gradient.
template <typename T, int HV>
__global__ void __launch_bounds__(kAttWarps * 32) xattn_bwd_q_kernel(
    const T* __restrict__ dO, const T* __restrict__ q, long long q_ss, const T* __restrict__ kv,
    const T* __restrict__ phantom, const int* __restrict__ ptr, const int* __restrict__ nmax_p,
    const T* __restrict__ out, const T* __restrict__ resid, long long r_ss, const float* __restrict__ lse,
    T* __restrict__ dq, T* __restrict__ Dbuf, T* __restrict__ dph_part, int S, int B, int Tn, T scale,
    unsigned int thresh, float inv_keep, unsigned long long seed, const unsigned long long* __restrict__ seed_offset) {
  constexpr int H = 32 * HV;
  seed = mask_seed(seed, seed_offset);
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* ks = reinterpret_cast<T*>(smem_raw);  // [kKT][H], reused as [kAttWarps][H] for the phantom reduction
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int s = blockIdx.y;
  const int b = s % B;
  const int kbeg = ptr[b], kend = ptr[b + 1];
  const int nb = kend - kbeg;
  const int nmax = *nmax_p;
  const int nph = max(nmax - nb, 0);
  const int t0 = blockIdx.x * kQPB + warp * kQPW;

  T qv[kQPW][HV], gv[kQPW][HV], dqv[kQPW][HV];
  T Dq[kQPW];
  float ls[kQPW];
#pragma unroll
  for (int qi = 0; qi < kQPW; ++qi) {
    const int t = min(t0 + qi, Tn - 1);
    const long long row = (long long)s * Tn + t;
    load_row<T, HV>(q + (long long)s * q_ss + (long long)t * H, lane, qv[qi]);
    load_row<T, HV>(dO + row * H, lane, gv[qi]);
    T o[HV], r[HV];
    load_row<T, HV>(out + row * H, lane, o);
    load_row<T, HV>(resid + (long long)s * r_ss + (long long)t * H, lane, r);
    T d = T(0);
#pragma unroll
    for (int i = 0; i < HV; ++i) {
      d = fma(gv[qi][i], o[i] - r[i], d);
      dqv[qi][i] = T(0);
    }
    Dq[qi] = warp_sum(d);
    ls[qi] = lse[row];
  }

  for (int j0 = 0; j0 < nb; j0 += kKT) {
    const int kt = min(kKT, nb - j0);
    __syncthreads();
    for (int i = threadIdx.x; i < kt * H; i += blockDim.x) ks[i] = kv[(long long)(kbeg + j0) * H + i];
    __syncthreads();
    for (int j = 0; j < kt; ++j) {
      T kk[HV];
#pragma unroll
      for (int i = 0; i < HV; ++i) kk[i] = ks[j * H + lane + 32 * i];
      T d1[kQPW], d2[kQPW];
#pragma unroll
      for (int qi = 0; qi < kQPW; ++qi) {
        d1[qi] = dot_partial<T, HV>(qv[qi], kk);
        d2[qi] = dot_partial<T, HV>(gv[qi], kk);
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int qi = 0; qi < kQPW; ++qi) {
          d1[qi] += __shfl_xor_sync(0xffffffffu, d1[qi], o);
          d2[qi] += __shfl_xor_sync(0xffffffffu, d2[qi], o);
        }
      }
#pragma unroll
      for (int qi = 0; qi < kQPW; ++qi) {
        const float p = expf(static_cast<float>(d1[qi] * scale) - ls[qi]);
        T dP = d2[qi];
        if (thresh) {
          const int t = t0 + qi;
          const unsigned long long idx = ((unsigned long long)s * Tn + t) * (unsigned long long)nmax + (j0 + j);
          dP = keep_mask(seed, idx, thresh) ? dP * static_cast<T>(inv_keep) : T(0);
        }
        const T dS = static_cast<T>(p) * (dP - Dq[qi]) * scale;
#pragma unroll
        for (int i = 0; i < HV; ++i) dqv[qi][i] = fma(dS, kk[i], dqv[qi][i]);
      }
    }
  }

  T dph[HV];
#pragma unroll
  for (int i = 0; i < HV; ++i) dph[i] = T(0);
  if (nph > 0) {
    T pk[HV];
    load_row<T, HV>(phantom, lane, pk);
#pragma unroll
    for (int qi = 0; qi < kQPW; ++qi) {
      const int t = t0 + qi;
      const T d1 = warp_sum(dot_partial<T, HV>(qv[qi], pk));
      const T d2 = warp_sum(dot_partial<T, HV>(gv[qi], pk));
      const float p = expf(static_cast<float>(d1 * scale) - ls[qi]);
      T wkeep = T(nph);  // sum over phantom copies of mask/(1-p)
      if (thresh) {
        int kept = 0;
        for (int jj = nb + lane; jj < nmax; jj += 32) {
          const unsigned long long idx = ((unsigned long long)s * Tn + t) * (unsigned long long)nmax + jj;
          kept += keep_mask(seed, idx, thresh) ? 1 : 0;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) kept += __shfl_xor_sync(0xffffffffu, kept, o);
        wkeep = T(kept) * static_cast<T>(inv_keep);
      }
      const T pT = static_cast<T>(p);
      // sum over copies of dS = p * (wkeep * (dO.beta) - nph * D)
      const T dSsum = pT * (wkeep * d2 - T(nph) * Dq[qi]) * scale;
      if (t < Tn) {
#pragma unroll
        for (int i = 0; i < HV; ++i) {
          dqv[qi][i] = fma(dSsum, pk[i], dqv[qi][i]);
          dph[i] += pT * wkeep * gv[qi][i] + dSsum * qv[qi][i];
        }
      }
    }
  }
#pragma unroll
  for (int qi = 0; qi < kQPW; ++qi) {
    const int t = t0 + qi;
    if (t < Tn) {
      const long long row = (long long)s * Tn + t;
#pragma unroll
      for (int i = 0; i < HV; ++i) dq[row * H + lane + 32 * i] = dqv[qi][i];
      if (lane == 0) Dbuf[row] = Dq[qi];
    }
  }
  // block partial of the phantom gradient, warps combined in a fixed order
  __syncthreads();
#pragma unroll
  for (int i = 0; i < HV; ++i) ks[warp * H + lane + 32 * i] = dph[i];
  __syncthreads();
  const long long blk = (long long)blockIdx.y * gridDim.x + blockIdx.x;
  for (int h = threadIdx.x; h < H; h += blockDim.x) {
    T sacc = T(0);
#pragma unroll
    for (int w = 0; w < kAttWarps; ++w) sacc += ks[w * H + h];
    dph_part[blk * H + h] = sacc;
  }
}

// ------------------------------------------------------------------------------------------------ backward: dkv
// One block per 8 consecutive nodes; loops over every query of every sequence attending to those nodes.
constexpr int kNT = 8;  // nodes per block

template <typename T, int HV>
__global__ void __launch_bounds__(kAttWarps * 32) xattn_bwd_kv_kernel(
    const T* __restrict__ dO, const T* __restrict__ q, long long q_ss, const T* __restrict__ kv,
    const int* __restrict__ ptr, const int* __restrict__ node_crystal, const int* __restrict__ nmax_p,
    const float* __restrict__ lse, const T* __restrict__ Dbuf, T* __restrict__ dkv, int S, int B, int Tn, long long N,
    T scale, unsigned int thresh, float inv_keep, unsigned long long seed, const unsigned long long* __restrict__ seed_offset) {
  constexpr int H = 32 * HV;
  seed = mask_seed(seed, seed_offset);
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* ks = reinterpret_cast<T*>(smem_raw);  // [kNT][H] keys, then [kAttWarps][H] reduction scratch
  T* red = ks + kNT * H;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long j0 = (long long)blockIdx.x * kNT;
  const int nt = (int)min64(kNT, N - j0);
  const int nmax = *nmax_p;
  for (int i = threadIdx.x; i < nt * H; i += blockDim.x) ks[i] = kv[j0 * H + i];
  __syncthreads();

  T acc[kNT][HV];
#pragma unroll
  for (int jj = 0; jj < kNT; ++jj)
#pragma unroll
    for (int i = 0; i < HV; ++i) acc[jj][i] = T(0);

  const int bfirst = node_crystal[j0], blast = node_crystal[j0 + nt - 1];
  const int nrep = S / B;
  for (int b = bfirst; b <= blast; ++b) {
    const int cbeg = ptr[b];
    const int lo = (int)(max64(cbeg, j0) - j0), hi = (int)(min64(ptr[b + 1], j0 + nt) - j0);
    if (hi <= lo) continue;
    for (int rep = 0; rep < nrep; ++rep) {
      const int s = b + rep * B;
      for (int t = warp; t < Tn; t += kAttWarps) {
        const long long row = (long long)s * Tn + t;
        T qv[HV], gv[HV];
        load_row<T, HV>(q + (long long)s * q_ss + (long long)t * H, lane, qv);
        load_row<T, HV>(dO + row * H, lane, gv);
        const float ls = lse[row];
        const T Dv = Dbuf[row];
#pragma unroll
        for (int jj = 0; jj < kNT; ++jj) {
          if (jj >= lo && jj < hi) {
            T kk[HV];
#pragma unroll
            for (int i = 0; i < HV; ++i) kk[i] = ks[jj * H + lane + 32 * i];
            T d1 = dot_partial<T, HV>(qv, kk), d2 = dot_partial<T, HV>(gv, kk);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
              d1 += __shfl_xor_sync(0xffffffffu, d1, o);
              d2 += __shfl_xor_sync(0xffffffffu, d2, o);
            }
            const T p = static_cast<T>(expf(static_cast<float>(d1 * scale) - ls));
            T w = T(1);
            if (thresh) {
              const unsigned long long idx =
                  ((unsigned long long)s * Tn + t) * (unsigned long long)nmax + (unsigned long long)(j0 + jj - cbeg);
              w = keep_mask(seed, idx, thresh) ? static_cast<T>(inv_keep) : T(0);
            }
            const T dS = p * (w * d2 - Dv) * scale;
            const T pw = p * w;
#pragma unroll
            for (int i = 0; i < HV; ++i) acc[jj][i] = fma(dS, qv[i], fma(pw, gv[i], acc[jj][i]));
          }
        }
      }
    }
  }
  // combine warps (fixed order), one node at a time
#pragma unroll
  for (int jj = 0; jj < kNT; ++jj) {
    __syncthreads();
#pragma unroll
    for (int i = 0; i < HV; ++i) red[warp * H + lane + 32 * i] = acc[jj][i];
    __syncthreads();
    if (jj < nt) {
      for (int h = threadIdx.x; h < H; h += blockDim.x) {
        T sacc = T(0);
#pragma unroll
        for (int w = 0; w < kAttWarps; ++w) sacc += red[w * H + h];
        dkv[(j0 + jj) * H + h] = sacc;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ row softmax
template <typename T, int NPL>
__global__ void __launch_bounds__(256) softmax_fwd_kernel(const T* __restrict__ sc, T* __restrict__ p,
                                                          T* __restrict__ pd, long long rows, int cols, long long ld, T scale,
                                                          unsigned int thresh, float inv_keep,
                                                          unsigned long long seed, const unsigned long long* __restrict__ seed_offset,
                                                          __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo,
                                                          long long ldp) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  seed = mask_seed(seed, seed_offset);
  for (long long r = blockIdx.x * 8LL + warp; r < rows; r += (long long)gridDim.x * 8) {
    const T* sr = sc + r * ld;
    float v[NPL];
    float mx = -INFINITY;
#pragma unroll
    for (int i = 0; i < NPL; ++i) {
      const int c = lane + 32 * i;
      v[i] = (c < cols) ? static_cast<float>(sr[c] * scale) : -INFINITY;
      mx = fmaxf(mx, v[i]);
    }
    mx = warp_max(mx);
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < NPL; ++i) {
      const int c = lane + 32 * i;
      v[i] = (c < cols) ? expf(v[i] - mx) : 0.f;
      sum += v[i];
    }
    sum = warp_sum(sum);
    const float inv = 1.0f / sum;
#pragma unroll
    for (int i = 0; i < NPL; ++i) {
      const int c = lane + 32 * i;
      if (c < cols) {
        const float pr = v[i] * inv;
        p[r * ld + c] = static_cast<T>(pr);
        float w = pr;
        if (pd != p) {
          if (thresh) w = keep_mask(seed, (unsigned long long)r * cols + c, thresh) ? pr * inv_keep : 0.f;
          pd[r * ld + c] = static_cast<T>(w);
        }
        if (hi) {      // the (dropped-out) probabilities as GEMM operand planes
          const __nv_bfloat16 h = __float2bfloat16_rn(w);
          hi[r * ldp + c] = h;
          if (lo) lo[r * ldp + c] = __float2bfloat16_rn(w - __bfloat162float(h));
        }
      }
    }
  }
}

template <typename T, int NPL>
__global__ void __launch_bounds__(256) softmax_bwd_kernel(const T* __restrict__ p, const T* __restrict__ dpd,
                                                          T* __restrict__ ds, long long rows, int cols, long long ld, T scale,
                                                          unsigned int thresh, float inv_keep,
                                                          unsigned long long seed, const unsigned long long* __restrict__ seed_offset,
                                                          __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo,
                                                          long long ldp) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  seed = mask_seed(seed, seed_offset);
  for (long long r = blockIdx.x * 8LL + warp; r < rows; r += (long long)gridDim.x * 8) {
    T pv[NPL], dp[NPL];
    T dot = T(0);
#pragma unroll
    for (int i = 0; i < NPL; ++i) {
      const int c = lane + 32 * i;
      if (c < cols) {
        pv[i] = p[r * ld + c];
        T g = dpd[r * ld + c];
        if (thresh) g = keep_mask(seed, (unsigned long long)r * cols + c, thresh) ? g * static_cast<T>(inv_keep) : T(0);
        dp[i] = g;
        dot = fma(g, pv[i], dot);
      } else {
        pv[i] = T(0);
        dp[i] = T(0);
      }
    }
    dot = warp_sum(dot);
#pragma unroll
    for (int i = 0; i < NPL; ++i) {
      const int c = lane + 32 * i;
      if (c < cols) {
        const T o = scale * pv[i] * (dp[i] - dot);
        if (ds) ds[r * ld + c] = o;
        if (hi) {
          const float of = static_cast<float>(o);
          const __nv_bfloat16 h = __float2bfloat16_rn(of);
          hi[r * ldp + c] = h;
          if (lo) lo[r * ldp + c] = __float2bfloat16_rn(of - __bfloat162float(h));
        }
      }
    }
  }
}

template <typename T>
static int run_xattn_fwd(const void* q, long long q_ss, const void* kv, const void* phantom, const int* ptr,
                         const int* nmax, const void* resid, long long r_ss, void* out, float* lse, int S, int B,
                         int Tn, int H, double scale, double drop_p, unsigned long long seed,
                         const unsigned long long* seed_offset, cudaStream_t st) {
  const unsigned int thresh = drop_p > 0 ? drop_threshold(drop_p) : 0u;
  const float inv_keep = drop_p > 0 ? (float)(1.0 / (1.0 - drop_p)) : 1.f;
  if (sizeof(T) == 4 && xattn_v2_supported(H))
    return xattn_v2_fwd((const float*)q, q_ss, (const float*)kv, (const float*)phantom, ptr, nmax, (const float*)resid, r_ss,
                        (float*)out, lse, S, B, Tn, H, (float)scale, thresh, inv_keep, seed, seed_offset, st);
  dim3 grid(ceil_div(Tn, kQPB), S);
  const size_t smem = sizeof(T) * (size_t)kKT * H;
#define DOST_XF(HV)                                                                                                  \
  case HV:                                                                                                           \
    if (smem > 48 * 1024)                                                                                            \
      cudaFuncSetAttribute(xattn_fwd_kernel<T, HV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);         \
    xattn_fwd_kernel<T, HV><<<grid, kAttWarps * 32, smem, st>>>((const T*)q, q_ss, (const T*)kv, (const T*)phantom, ptr, \
                                                                nmax, (const T*)resid, r_ss, (T*)out, lse, S, B, Tn,  \
                                                                (T)scale, thresh, inv_keep, seed, seed_offset);      \
    break;
  switch (H / 32) {
    DOST_XF(1) DOST_XF(2) DOST_XF(4) DOST_XF(8) DOST_XF(16)
    default:
      set_error("xattn_fwd: hidden %d unsupported (32,64,128,256,512)", H);
      return DOST_ERR_UNSUPPORTED;
  }
#undef DOST_XF
  return check_launch("xattn_fwd");
}

template <typename T>
static int run_xattn_probs(const void* q, long long q_ss, const void* kv, const void* phantom, const int* ptr, const int* nmax,
                           const float* lse, void* out, int cols, int S, int B, int Tn, int H, double scale, double drop_p,
                           unsigned long long seed, const unsigned long long* seed_offset, cudaStream_t st) {
  const unsigned int thresh = drop_p > 0 ? drop_threshold(drop_p) : 0u;
  const float inv_keep = drop_p > 0 ? (float)(1.0 / (1.0 - drop_p)) : 1.f;
  dim3 grid(ceil_div(Tn, kQPB), S);
  const size_t smem = sizeof(T) * (size_t)kKT * H;
#define DOST_XP(HV)                                                                                                    \
  case HV:                                                                                                             \
    if (smem > 48 * 1024)                                                                                              \
      cudaFuncSetAttribute(xattn_probs_kernel<T, HV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);         \
    xattn_probs_kernel<T, HV><<<grid, kAttWarps * 32, smem, st>>>((const T*)q, q_ss, (const T*)kv, (const T*)phantom, ptr, \
                                                                  nmax, lse, (T*)out, cols, S, B, Tn, (T)scale, thresh, \
                                                                  inv_keep, seed, seed_offset);                        \
    break;
  switch (H / 32) {
    DOST_XP(1) DOST_XP(2) DOST_XP(4) DOST_XP(8) DOST_XP(16)
    default:
      set_error("xattn_probs: hidden %d unsupported (32,64,128,256,512)", H);
      return DOST_ERR_UNSUPPORTED;
  }
#undef DOST_XP
  return check_launch("xattn_probs");
}

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

template <typename T>
static int run_xattn_bwd(const void* dO, const void* q, long long q_ss, const void* kv, const void* phantom,
                         const int* ptr, const int* node_crystal, const int* nmax, const void* out, const void* resid,
                         long long r_ss, const float* lse, void* dq, void* dkv, void* dphantom, int S, int B, int Tn,
                         int H, long long N, double scale, double drop_p, unsigned long long seed,
                         const unsigned long long* seed_offset, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  const unsigned int thresh = drop_p > 0 ? drop_threshold(drop_p) : 0u;
  const float inv_keep = drop_p > 0 ? (float)(1.0 / (1.0 - drop_p)) : 1.f;
  dim3 grid(ceil_div(Tn, kQPB), S);
  const long long nblk = (long long)grid.x * grid.y;
  const int dt = sizeof(T) == 8 ? DOST_F64 : DOST_F32;
  const size_t o_D = 0;
  const size_t o_part = align_up(o_D + sizeof(T) * (size_t)S * Tn, 256);
  const size_t o_cs = align_up(o_part + sizeof(T) * (size_t)nblk * H, 256);
  const size_t cs_bytes = dost_colsum_workspace_bytes(dt, nblk, H);
  if (!workspace || workspace_bytes < o_cs + cs_bytes) {
    set_error("xattn_bwd: workspace too small (%zu < %zu)", workspace_bytes, o_cs + cs_bytes);
    return DOST_ERR_WORKSPACE;
  }
  T* Dbuf = (T*)((char*)workspace + o_D);
  T* part = (T*)((char*)workspace + o_part);
  void* csws = (char*)workspace + o_cs;
  const bool v2 = sizeof(T) == 4 && xattn_v2_supported(H);
  if (v2) {   // dq, D and the phantom partials from the FMA-bound kernel; dkv keeps the node-block kernel below
    int rc2 = xattn_v2_bwd((const float*)dO, (const float*)q, q_ss, (const float*)kv, (const float*)phantom, ptr, nmax,
                           (const float*)out, (const float*)resid, r_ss, lse, (float*)dq, (float*)dkv, (float*)Dbuf, (float*)part, S,
                           B, Tn, H, (float)scale, thresh, inv_keep, seed, seed_offset, false, st);
    if (rc2 != DOST_OK) return rc2;
  }
  const size_t smem_q = sizeof(T) * (size_t)kKT * H;
  const size_t smem_kv = sizeof(T) * (size_t)(kNT + kAttWarps) * H;
  const int kvblocks = ceil_div(N, kNT);
#define DOST_XB(HV)                                                                                                   \
  case HV:                                                                                                            \
    if (smem_q > 48 * 1024)                                                                                           \
      cudaFuncSetAttribute(xattn_bwd_q_kernel<T, HV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_q);      \
    if (smem_kv > 48 * 1024)                                                                                          \
      cudaFuncSetAttribute(xattn_bwd_kv_kernel<T, HV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_kv);    \
    if (!v2) {                                                                                                        \
      xattn_bwd_q_kernel<T, HV><<<grid, kAttWarps * 32, smem_q, st>>>(                                                \
          (const T*)dO, (const T*)q, q_ss, (const T*)kv, (const T*)phantom, ptr, nmax, (const T*)out, (const T*)resid, \
          r_ss, lse, (T*)dq, Dbuf, part, S, B, Tn, (T)scale, thresh, inv_keep, seed, seed_offset);                    \
      count_launch();                                                                                                 \
    }                                                                                                                 \
    xattn_bwd_kv_kernel<T, HV><<<kvblocks, kAttWarps * 32, smem_kv, st>>>(                                            \
        (const T*)dO, (const T*)q, q_ss, (const T*)kv, ptr, node_crystal, nmax, lse, Dbuf, (T*)dkv, S, B, Tn, N,      \
        (T)scale, thresh, inv_keep, seed, seed_offset);                                                               \
    break;
  switch (H / 32) {
    DOST_XB(1) DOST_XB(2) DOST_XB(4) DOST_XB(8) DOST_XB(16)
    default:
      set_error("xattn_bwd: hidden %d unsupported (32,64,128,256,512)", H);
      return DOST_ERR_UNSUPPORTED;
  }
#undef DOST_XB
  int rc = check_launch("xattn_bwd");
  if (rc != DOST_OK) return rc;
  return dost_colsum(dt, part, H, nblk, H, dphantom, csws, cs_bytes, (dost_stream_t)st);
}

template <typename T>
static int run_softmax(bool fwd, const void* a, void* b, void* c, long long rows, int cols, long long ld, double scale,
                       double drop_p, unsigned long long seed, const unsigned long long* seed_offset, cudaStream_t st,
                       void* hi = nullptr, void* lo = nullptr, long long ldp = 0) {
  const unsigned int thresh = drop_p > 0 ? drop_threshold(drop_p) : 0u;
  const float inv_keep = drop_p > 0 ? (float)(1.0 / (1.0 - drop_p)) : 1.f;
  int npl = (cols + 31) / 32, pw = 1;
  while (pw < npl) pw <<= 1;
  const int blocks = (int)min64((rows + 7) / 8, 32LL * kNumSMs);
#define DOST_SM(NPL)                                                                                              \
  case NPL:                                                                                                       \
    if (fwd)                                                                                                      \
      softmax_fwd_kernel<T, NPL><<<blocks, 256, 0, st>>>((const T*)a, (T*)b, (T*)c, rows, cols, ld, (T)scale, thresh, \
                                                         inv_keep, seed, seed_offset, (__nv_bfloat16*)hi,         \
                                                         (__nv_bfloat16*)lo, ldp);                                \
    else                                                                                                          \
      softmax_bwd_kernel<T, NPL><<<blocks, 256, 0, st>>>((const T*)a, (const T*)b, (T*)c, rows, cols, ld, (T)scale,   \
                                                         thresh, inv_keep, seed, seed_offset, (__nv_bfloat16*)hi, \
                                                         (__nv_bfloat16*)lo, ldp);                                \
    break;
  switch (pw) {
    DOST_SM(1) DOST_SM(2) DOST_SM(4) DOST_SM(8) DOST_SM(16) DOST_SM(32)
    default:
      set_error("softmax: %d columns unsupported (max 1024)", cols);
      return DOST_ERR_UNSUPPORTED;
  }
#undef DOST_SM
  return check_launch(fwd ? "softmax_fwd" : "softmax_bwd");
}

}  // namespace dost

using namespace dost;

extern "C" int dost_xattn_fwd_dseed(int dtype, const void* q, long long q_sstride, const void* kv, const void* phantom,
                                    const int32_t* ptr, const int32_t* nmax, const void* resid, long long resid_sstride,
                                    void* out, float* lse, int S, int B, int T, int H, double scale, double drop_p,
                                    unsigned long long seed, const unsigned long long* seed_offset, dost_stream_t stream) {
  DOST_REQUIRE(q && kv && phantom && ptr && nmax && resid && out && lse, "xattn_fwd: null pointer");
  DOST_REQUIRE(S > 0 && B > 0 && S % B == 0 && T > 0 && H % 32 == 0, "xattn_fwd: bad shape S=%d B=%d T=%d H=%d", S, B, T, H);
  DOST_REQUIRE(drop_p >= 0.0 && drop_p < 1.0, "xattn_fwd: dropout must be in [0,1)");
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == DOST_F32)
    return run_xattn_fwd<float>(q, q_sstride, kv, phantom, ptr, nmax, resid, resid_sstride, out, lse, S, B, T, H, scale, drop_p, seed,
                                seed_offset, st);
  if (dtype == DOST_F64)
    return run_xattn_fwd<double>(q, q_sstride, kv, phantom, ptr, nmax, resid, resid_sstride, out, lse, S, B, T, H, scale, drop_p, seed,
                                 seed_offset, st);
  set_error("xattn_fwd: unsupported dtype %d", dtype);
  return DOST_ERR_UNSUPPORTED;
}

extern "C" int dost_xattn_fwd(int dtype, const void* q, long long q_sstride, const void* kv, const void* phantom,
                              const int32_t* ptr, const int32_t* nmax, const void* resid, long long resid_sstride,
                              void* out, float* lse, int S, int B, int T, int H, double scale, double drop_p,
                              unsigned long long seed, dost_stream_t stream) {
  return dost_xattn_fwd_dseed(dtype, q, q_sstride, kv, phantom, ptr, nmax, resid, resid_sstride, out, lse, S, B, T, H, scale, drop_p,
                              seed, nullptr, stream);
}

extern "C" int dost_xattn_probs(int dtype, const void* q, long long q_sstride, const void* kv, const void* phantom,
                                const int32_t* ptr, const int32_t* nmax, const float* lse, void* out, int cols, int S, int B, int T,
                                int H, double scale, double drop_p, unsigned long long mask_seed,
                                const unsigned long long* seed_offset, dost_stream_t stream) {
  DOST_REQUIRE(q && kv && phantom && ptr && nmax && lse && out, "xattn_probs: null pointer");
  DOST_REQUIRE(S > 0 && B > 0 && S % B == 0 && T > 0 && H % 32 == 0 && cols > 0, "xattn_probs: bad shape S=%d B=%d T=%d H=%d cols=%d",
               S, B, T, H, cols);
  DOST_REQUIRE(drop_p >= 0.0 && drop_p < 1.0, "xattn_probs: dropout must be in [0,1)");
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == DOST_F32)
    return run_xattn_probs<float>(q, q_sstride, kv, phantom, ptr, nmax, lse, out, cols, S, B, T, H, scale, drop_p, mask_seed, seed_offset,
                                  st);
  if (dtype == DOST_F64)
    return run_xattn_probs<double>(q, q_sstride, kv, phantom, ptr, nmax, lse, out, cols, S, B, T, H, scale, drop_p, mask_seed, seed_offset,
                                   st);
  set_error("xattn_probs: unsupported dtype %d", dtype);
  return DOST_ERR_UNSUPPORTED;
}

extern "C" size_t dost_xattn_bwd_workspace_bytes(int dtype, int S, int T, int H) {
  const size_t es = dtype == DOST_F64 ? 8 : 4;
  const long long nblk = (long long)ceil_div(T, kQPB) * S;
  size_t o_part = align_up(es * (size_t)S * T, 256);
  size_t o_cs = align_up(o_part + es * (size_t)nblk * H, 256);
  return o_cs + dost_colsum_workspace_bytes(dtype, nblk, H);
}

extern "C" int dost_xattn_bwd_dseed(int dtype, const void* d_out, const void* q, long long q_sstride, const void* kv,
                                    const void* phantom, const int32_t* ptr, const int32_t* node_crystal,
                                    const int32_t* nmax, const void* out, const void* resid, long long resid_sstride,
                                    const float* lse, void* dq, void* dkv, void* dphantom, int S, int B, int T, int H,
                                    long long N, double scale, double drop_p, unsigned long long seed,
                                    const unsigned long long* seed_offset, void* workspace, size_t workspace_bytes,
                                    dost_stream_t stream) {
  DOST_REQUIRE(d_out && q && kv && phantom && ptr && node_crystal && nmax && out && resid && lse && dq && dkv && dphantom,
               "xattn_bwd: null pointer");
  DOST_REQUIRE(S > 0 && B > 0 && S % B == 0 && T > 0 && H % 32 == 0 && N > 0, "xattn_bwd: bad shape");
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == DOST_F32)
    return run_xattn_bwd<float>(d_out, q, q_sstride, kv, phantom, ptr, node_crystal, nmax, out, resid, resid_sstride, lse,
                                dq, dkv, dphantom, S, B, T, H, N, scale, drop_p, seed, seed_offset, workspace, workspace_bytes, st);
  if (dtype == DOST_F64)
    return run_xattn_bwd<double>(d_out, q, q_sstride, kv, phantom, ptr, node_crystal, nmax, out, resid, resid_sstride, lse,
                                 dq, dkv, dphantom, S, B, T, H, N, scale, drop_p, seed, seed_offset, workspace, workspace_bytes, st);
  set_error("xattn_bwd: unsupported dtype %d", dtype);
  return DOST_ERR_UNSUPPORTED;
}

extern "C" int dost_xattn_bwd(int dtype, const void* d_out, const void* q, long long q_sstride, const void* kv,
                              const void* phantom, const int32_t* ptr, const int32_t* node_crystal,
                              const int32_t* nmax, const void* out, const void* resid, long long resid_sstride,
                              const float* lse, void* dq, void* dkv, void* dphantom, int S, int B, int T, int H,
                              long long N, double scale, double drop_p, unsigned long long seed, void* workspace,
                              size_t workspace_bytes, dost_stream_t stream) {
  return dost_xattn_bwd_dseed(dtype, d_out, q, q_sstride, kv, phantom, ptr, node_crystal, nmax, out, resid, resid_sstride, lse, dq,
                              dkv, dphantom, S, B, T, H, N, scale, drop_p, seed, nullptr, workspace, workspace_bytes, stream);
}

extern "C" int dost_softmax_fwd_dseed(int dtype, const void* s, void* p, void* pd, long long rows, int cols, long long ld,
                                      double scale, double drop_p, unsigned long long seed, const unsigned long long* seed_offset,
                                      dost_stream_t stream) {
  DOST_REQUIRE(s && p && rows > 0 && cols > 0 && ld >= cols, "softmax_fwd: bad args");
  if (!pd) pd = p;
  DOST_REQUIRE(!(drop_p > 0 && pd == p), "softmax_fwd: dropout needs a separate pd buffer");
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == DOST_F32) return run_softmax<float>(true, s, p, pd, rows, cols, ld, scale, drop_p, seed, seed_offset, st);
  if (dtype == DOST_F64) return run_softmax<double>(true, s, p, pd, rows, cols, ld, scale, drop_p, seed, seed_offset, st);
  set_error("softmax_fwd: unsupported dtype %d", dtype);
  return DOST_ERR_UNSUPPORTED;
}

extern "C" int dost_softmax_fwd(int dtype, const void* s, void* p, void* pd, long long rows, int cols, long long ld, double scale,
                                double drop_p, unsigned long long seed, dost_stream_t stream) {
  return dost_softmax_fwd_dseed(dtype, s, p, pd, rows, cols, ld, scale, drop_p, seed, nullptr, stream);
}

extern "C" int dost_softmax_bwd_dseed(int dtype, const void* p, const void* dpd, void* ds, long long rows, int cols, long long ld,
                                      double scale, double drop_p, unsigned long long seed, const unsigned long long* seed_offset,
                                      dost_stream_t stream) {
  DOST_REQUIRE(p && dpd && ds && rows > 0 && cols > 0 && ld >= cols, "softmax_bwd: bad args");
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == DOST_F32) return run_softmax<float>(false, p, (void*)dpd, ds, rows, cols, ld, scale, drop_p, seed, seed_offset, st);
  if (dtype == DOST_F64) return run_softmax<double>(false, p, (void*)dpd, ds, rows, cols, ld, scale, drop_p, seed, seed_offset, st);
  set_error("softmax_bwd: unsupported dtype %d", dtype);
  return DOST_ERR_UNSUPPORTED;
}

extern "C" int dost_softmax_bwd(int dtype, const void* p, const void* dpd, void* ds, long long rows, int cols, long long ld,
                                double scale, double drop_p, unsigned long long seed, dost_stream_t stream) {
  return dost_softmax_bwd_dseed(dtype, p, dpd, ds, rows, cols, ld, scale, drop_p, seed, nullptr, stream);
}

/* fp32 softmax whose (dropped-out) probabilities / score gradients are also written as bf16 hi/lo operand planes
 * (rows ldp elements apart) for the batched tensor-core GEMMs that consume them. */
extern "C" int dost_softmax_fwd_planes_dseed(const float* s, float* p, float* pd, long long rows, int cols, long long ld,
                                             double scale, double drop_p, unsigned long long seed,
                                             const unsigned long long* seed_offset, void* hi, void* lo, long long ldp,
                                             dost_stream_t stream) {
  DOST_REQUIRE(s && p && hi && rows > 0 && cols > 0 && ld >= cols && ldp >= cols, "softmax_fwd_planes: bad args");
  if (!pd) pd = p;
  DOST_REQUIRE(!(drop_p > 0 && pd == p), "softmax_fwd_planes: dropout needs a separate pd buffer");
  return run_softmax<float>(true, s, p, pd, rows, cols, ld, scale, drop_p, seed, seed_offset, (cudaStream_t)stream, hi, lo, ldp);
}

extern "C" int dost_softmax_fwd_planes(const float* s, float* p, float* pd, long long rows, int cols, long long ld, double scale,
                                       double drop_p, unsigned long long seed, void* hi, void* lo, long long ldp,
                                       dost_stream_t stream) {
  return dost_softmax_fwd_planes_dseed(s, p, pd, rows, cols, ld, scale, drop_p, seed, nullptr, hi, lo, ldp, stream);
}

extern "C" int dost_softmax_bwd_planes_dseed(const float* p, const float* dpd, float* ds, long long rows, int cols, long long ld,
                                             double scale, double drop_p, unsigned long long seed,
                                             const unsigned long long* seed_offset, void* hi, void* lo, long long ldp,
                                             dost_stream_t stream) {
  DOST_REQUIRE(p && dpd && hi && rows > 0 && cols > 0 && ld >= cols && ldp >= cols, "softmax_bwd_planes: bad args");
  return run_softmax<float>(false, p, (void*)dpd, ds, rows, cols, ld, scale, drop_p, seed, seed_offset, (cudaStream_t)stream, hi, lo,
                            ldp);
}

extern "C" int dost_softmax_bwd_planes(const float* p, const float* dpd, float* ds, long long rows, int cols, long long ld,
                                       double scale, double drop_p, unsigned long long seed, void* hi, void* lo, long long ldp,
                                       dost_stream_t stream) {
  return dost_softmax_bwd_planes_dseed(p, dpd, ds, rows, cols, ld, scale, drop_p, seed, nullptr, hi, lo, ldp, stream);
}
