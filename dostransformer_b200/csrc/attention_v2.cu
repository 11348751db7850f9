// Ragged energy->atom cross attention, fp32, H = 128 * NF (the hidden sizes the tensor-core path uses).
//
// Same semantics as attention.cu (analytic phantom keys, fp32 softmax, counter-based dropout, deterministic backward)
// restructured so that almost every issued instruction is an FMA: a block owns 32 queries of one sequence, the keys of
// its crystal are staged in shared memory 32 at a time, and the two contractions use different lane mappings
//   scores  s[t, j] = q_t . k_j : lane <-> key j; q rows are broadcast 16-byte shared loads, key rows are read with a
//                                 260-float pitch (conflict-free LDS.128); no shuffles inside the dot products
//   values  o[t, :] += p[t, j] k_j : lane <-> 4 NF features; p is broadcast from shared memory
// instead of one warp-shuffle reduction per (query, key) pair.  The forward is bound by the FMA pipe / HBM
// (q, resid read and out written once), not by shuffle and exp latency.
#include <math.h>
#include "common.cuh"

namespace dost {
namespace xa2 {

constexpr int kWarps = 8, kQW = 4, kQB = kWarps * kQW, kKT = 32;

__device__ __forceinline__ float dot4(const float4& a, const float4& b, float acc) {
  acc = fmaf(a.x, b.x, acc);
  acc = fmaf(a.y, b.y, acc);
  acc = fmaf(a.z, b.z, acc);
  acc = fmaf(a.w, b.w, acc);
  return acc;
}
__device__ __forceinline__ void axpy4(float a, const float4& x, float4& y) {
  y.x = fmaf(a, x.x, y.x);
  y.y = fmaf(a, x.y, y.y);
  y.z = fmaf(a, x.z, y.z);
  y.w = fmaf(a, x.w, y.w);
}
__device__ __forceinline__ float comp(const float4& v, int i) { return i == 0 ? v.x : (i == 1 ? v.y : (i == 2 ? v.z : v.w)); }

// rows [row0, row0 + 32) of a [*, H] matrix -> smem tile with `pitch` floats per row; rows >= nrows are clamped
// (clamp = true: repeat the last valid row) or zero-filled.
template <int H>
__device__ __forceinline__ void load_tile(float* dst, int pitch, const float* __restrict__ src, long long row0, int nrows,
                                          bool clamp) {
  constexpr int C4 = H / 4;
  for (int idx = threadIdx.x; idx < 32 * C4; idx += blockDim.x) {
    const int r = idx / C4, c = idx - r * C4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r < nrows || clamp) v = __ldg(reinterpret_cast<const float4*>(src + (row0 + min(r, nrows - 1)) * H) + c);
    *reinterpret_cast<float4*>(dst + r * pitch + 4 * c) = v;
  }
}

// ------------------------------------------------------------------------------------------------ forward
template <int NF>
__global__ void __launch_bounds__(kWarps * 32) fwd_kernel(const float* __restrict__ q, long long q_ss, const float* __restrict__ kv,
                                                          const float* __restrict__ phantom, const int* __restrict__ ptr,
                                                          const int* __restrict__ nmax_p, const float* __restrict__ resid,
                                                          long long r_ss, float* __restrict__ out, float* __restrict__ lse, int S,
                                                          int B, int Tn, float scale, unsigned int thresh, float inv_keep,
                                                          unsigned long long seed,
                                                          const unsigned long long* __restrict__ seed_offset) {
  constexpr int H = 128 * NF, KP = H + 4;
  seed = mask_seed(seed, seed_offset);
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* Qs = reinterpret_cast<float*>(smem_raw);   // [32][H]
  float* Ks = Qs + 32 * H;                           // [32][KP]
  float* Ps = Ks + 32 * KP;                          // [kWarps][32][4]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int s = blockIdx.y, b = s % B;
  const int kbeg = ptr[b], nb = ptr[b + 1] - kbeg;
  const int nmax = *nmax_p;
  const int nph = max(nmax - nb, 0);
  const int t0 = blockIdx.x * kQB;
  load_tile<H>(Qs, H, q + (long long)s * q_ss, t0, Tn - t0, true);
  __syncthreads();

  float4 acc[kQW][NF];
  float m[kQW], l[kQW];
#pragma unroll
  for (int qi = 0; qi < kQW; ++qi) {
#pragma unroll
    for (int i = 0; i < NF; ++i) acc[qi][i] = make_float4(0.f, 0.f, 0.f, 0.f);
    m[qi] = -INFINITY;
    l[qi] = 0.f;
  }
  const float* qrow = Qs + (warp * kQW) * H;
  float* pw = Ps + warp * 32 * 4;

  for (int j0 = 0; j0 < nb; j0 += kKT) {
    const int kt = min(kKT, nb - j0);
    __syncthreads();
    load_tile<H>(Ks, KP, kv, kbeg + j0, kt, false);
    __syncthreads();
    // ---- scores: lane <-> key
    float d[kQW] = {0.f, 0.f, 0.f, 0.f};
    const float* krow = Ks + lane * KP;
#pragma unroll 4
    for (int h4 = 0; h4 < H / 4; ++h4) {
      const float4 k4 = *reinterpret_cast<const float4*>(krow + 4 * h4);
#pragma unroll
      for (int qi = 0; qi < kQW; ++qi) d[qi] = dot4(*reinterpret_cast<const float4*>(qrow + qi * H + 4 * h4), k4, d[qi]);
    }
    float4 w4;
    float* wv = &w4.x;
#pragma unroll
    for (int qi = 0; qi < kQW; ++qi) {
      const float sc = (lane < kt) ? d[qi] * scale : -INFINITY;
      const float mn = fmaxf(m[qi], warp_max(sc));
      const float corr = expf(m[qi] - mn);
      const float p = (lane < kt) ? expf(sc - mn) : 0.f;
      l[qi] = l[qi] * corr + warp_sum(p);
      m[qi] = mn;
      float w = p;
      if (thresh) {
        const int t = t0 + warp * kQW + qi;
        const unsigned long long idx = ((unsigned long long)s * Tn + t) * (unsigned long long)nmax + (j0 + lane);
        w = keep_mask(seed, idx, thresh) ? p * inv_keep : 0.f;
      }
      wv[qi] = w;
#pragma unroll
      for (int i = 0; i < NF; ++i) {
        acc[qi][i].x *= corr; acc[qi][i].y *= corr; acc[qi][i].z *= corr; acc[qi][i].w *= corr;
      }
    }
    *reinterpret_cast<float4*>(pw + lane * 4) = w4;
    __syncwarp();
    // ---- values: lane <-> features
    for (int j = 0; j < kt; ++j) {
      const float4 p4 = *reinterpret_cast<const float4*>(pw + j * 4);
#pragma unroll
      for (int i = 0; i < NF; ++i) {
        const float4 kf = *reinterpret_cast<const float4*>(Ks + j * KP + lane * 4 + 128 * i);
#pragma unroll
        for (int qi = 0; qi < kQW; ++qi) axpy4(comp(p4, qi), kf, acc[qi][i]);
      }
    }
    __syncwarp();
  }
  // ---- phantom keys: nph copies of k = v = phantom
  if (nph > 0) {
    float4 pk[NF];
#pragma unroll
    for (int i = 0; i < NF; ++i) pk[i] = __ldg(reinterpret_cast<const float4*>(phantom) + lane + 32 * i);
#pragma unroll
    for (int qi = 0; qi < kQW; ++qi) {
      float dpart = 0.f;
#pragma unroll
      for (int i = 0; i < NF; ++i) dpart = dot4(*reinterpret_cast<const float4*>(qrow + qi * H + lane * 4 + 128 * i), pk[i], dpart);
      const float sc = warp_sum(dpart) * scale;
      const float mn = fmaxf(m[qi], sc);
      const float corr = expf(m[qi] - mn);
      const float p = expf(sc - mn);
      l[qi] = l[qi] * corr + p * (float)nph;
      m[qi] = mn;
      float w = p * (float)nph;
      if (thresh) {
        const int t = t0 + warp * kQW + qi;
        int kept = 0;
        for (int jj = nb + lane; jj < nmax; jj += 32) {
          const unsigned long long idx = ((unsigned long long)s * Tn + t) * (unsigned long long)nmax + jj;
          kept += keep_mask(seed, idx, thresh) ? 1 : 0;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) kept += __shfl_xor_sync(0xffffffffu, kept, o);
        w = p * inv_keep * (float)kept;
      }
#pragma unroll
      for (int i = 0; i < NF; ++i) {
        acc[qi][i].x = fmaf(w, pk[i].x, acc[qi][i].x * corr);
        acc[qi][i].y = fmaf(w, pk[i].y, acc[qi][i].y * corr);
        acc[qi][i].z = fmaf(w, pk[i].z, acc[qi][i].z * corr);
        acc[qi][i].w = fmaf(w, pk[i].w, acc[qi][i].w * corr);
      }
    }
  }
#pragma unroll
  for (int qi = 0; qi < kQW; ++qi) {
    const int t = t0 + warp * kQW + qi;
    if (t < Tn) {
      const float inv = 1.0f / l[qi];
      const float4* rr = reinterpret_cast<const float4*>(resid + (long long)s * r_ss + (long long)t * H);
      float4* oo = reinterpret_cast<float4*>(out + ((long long)s * Tn + t) * H);
#pragma unroll
      for (int i = 0; i < NF; ++i) {
        const float4 r4 = __ldg(rr + lane + 32 * i);
        oo[lane + 32 * i] = make_float4(fmaf(acc[qi][i].x, inv, r4.x), fmaf(acc[qi][i].y, inv, r4.y),
                                        fmaf(acc[qi][i].z, inv, r4.z), fmaf(acc[qi][i].w, inv, r4.w));
      }
      if (lane == 0) lse[(long long)s * Tn + t] = m[qi] + logf(l[qi]);
    }
  }
}

// ------------------------------------------------------------------------------------------------ backward: dq
// Also writes D[s,t] = dO . (out - resid) and per-block partial sums of the phantom-key gradient.
template <int NF>
__global__ void __launch_bounds__(kWarps * 32) bwd_q_kernel(const float* __restrict__ dO, const float* __restrict__ q, long long q_ss,
                                                            const float* __restrict__ kv, const float* __restrict__ phantom,
                                                            const int* __restrict__ ptr, const int* __restrict__ nmax_p,
                                                            const float* __restrict__ out, const float* __restrict__ resid,
                                                            long long r_ss, const float* __restrict__ lse, float* __restrict__ dq,
                                                            float* __restrict__ Dbuf, float* __restrict__ dph_part, int S, int B, int Tn,
                                                            float scale, unsigned int thresh, float inv_keep,
                                                            unsigned long long seed,
                                                            const unsigned long long* __restrict__ seed_offset) {
  constexpr int H = 128 * NF, KP = H + 4;
  seed = mask_seed(seed, seed_offset);
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* Qs = reinterpret_cast<float*>(smem_raw);   // [32][H]
  float* Gs = Qs + 32 * H;                           // [32][H]   dO
  float* Ks = Gs + 32 * H;                           // [32][KP]  (reused as [kWarps][H] for the phantom reduction)
  float* Ps = Ks + 32 * KP;                          // [kWarps][32][4]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int s = blockIdx.y, b = s % B;
  const int kbeg = ptr[b], nb = ptr[b + 1] - kbeg;
  const int nmax = *nmax_p;
  const int nph = max(nmax - nb, 0);
  const int t0 = blockIdx.x * kQB;
  load_tile<H>(Qs, H, q + (long long)s * q_ss, t0, Tn - t0, true);
  load_tile<H>(Gs, H, dO + (long long)s * Tn * H, t0, Tn - t0, true);
  __syncthreads();
  const float* qrow = Qs + (warp * kQW) * H;
  const float* grow = Gs + (warp * kQW) * H;
  float* pw = Ps + warp * 32 * 4;

  float4 dqa[kQW][NF];
  float Dq[kQW], ls[kQW];
#pragma unroll
  for (int qi = 0; qi < kQW; ++qi) {
    const int t = min(t0 + warp * kQW + qi, Tn - 1);
    const long long row = (long long)s * Tn + t;
    const float4* oo = reinterpret_cast<const float4*>(out + row * H);
    const float4* rr = reinterpret_cast<const float4*>(resid + (long long)s * r_ss + (long long)t * H);
    float dpart = 0.f;
#pragma unroll
    for (int i = 0; i < NF; ++i) {
      const float4 o4 = __ldg(oo + lane + 32 * i), r4 = __ldg(rr + lane + 32 * i);
      const float4 g4 = *reinterpret_cast<const float4*>(grow + qi * H + lane * 4 + 128 * i);
      dpart = dot4(g4, make_float4(o4.x - r4.x, o4.y - r4.y, o4.z - r4.z, o4.w - r4.w), dpart);
      dqa[qi][i] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    Dq[qi] = warp_sum(dpart);
    ls[qi] = __ldg(lse + row);
  }

  for (int j0 = 0; j0 < nb; j0 += kKT) {
    const int kt = min(kKT, nb - j0);
    __syncthreads();
    load_tile<H>(Ks, KP, kv, kbeg + j0, kt, false);
    __syncthreads();
    float d1[kQW] = {0.f, 0.f, 0.f, 0.f}, d2[kQW] = {0.f, 0.f, 0.f, 0.f};
    const float* krow = Ks + lane * KP;
#pragma unroll 2
    for (int h4 = 0; h4 < H / 4; ++h4) {
      const float4 k4 = *reinterpret_cast<const float4*>(krow + 4 * h4);
#pragma unroll
      for (int qi = 0; qi < kQW; ++qi) {
        d1[qi] = dot4(*reinterpret_cast<const float4*>(qrow + qi * H + 4 * h4), k4, d1[qi]);
        d2[qi] = dot4(*reinterpret_cast<const float4*>(grow + qi * H + 4 * h4), k4, d2[qi]);
      }
    }
    float4 s4;
    float* sv = &s4.x;
#pragma unroll
    for (int qi = 0; qi < kQW; ++qi) {
      const float p = (lane < kt) ? expf(d1[qi] * scale - ls[qi]) : 0.f;
      float dP = d2[qi];
      if (thresh) {
        const int t = t0 + warp * kQW + qi;
        const unsigned long long idx = ((unsigned long long)s * Tn + t) * (unsigned long long)nmax + (j0 + lane);
        dP = keep_mask(seed, idx, thresh) ? dP * inv_keep : 0.f;
      }
      sv[qi] = p * (dP - Dq[qi]) * scale;
    }
    *reinterpret_cast<float4*>(pw + lane * 4) = s4;
    __syncwarp();
    for (int j = 0; j < kt; ++j) {
      const float4 p4 = *reinterpret_cast<const float4*>(pw + j * 4);
#pragma unroll
      for (int i = 0; i < NF; ++i) {
        const float4 kf = *reinterpret_cast<const float4*>(Ks + j * KP + lane * 4 + 128 * i);
#pragma unroll
        for (int qi = 0; qi < kQW; ++qi) axpy4(comp(p4, qi), kf, dqa[qi][i]);
      }
    }
    __syncwarp();
  }

  float4 dph[NF];
#pragma unroll
  for (int i = 0; i < NF; ++i) dph[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  if (nph > 0) {
    float4 pk[NF];
#pragma unroll
    for (int i = 0; i < NF; ++i) pk[i] = __ldg(reinterpret_cast<const float4*>(phantom) + lane + 32 * i);
#pragma unroll
    for (int qi = 0; qi < kQW; ++qi) {
      const int t = t0 + warp * kQW + qi;
      float a1 = 0.f, a2 = 0.f;
      float4 q4[NF], g4[NF];
#pragma unroll
      for (int i = 0; i < NF; ++i) {
        q4[i] = *reinterpret_cast<const float4*>(qrow + qi * H + lane * 4 + 128 * i);
        g4[i] = *reinterpret_cast<const float4*>(grow + qi * H + lane * 4 + 128 * i);
        a1 = dot4(q4[i], pk[i], a1);
        a2 = dot4(g4[i], pk[i], a2);
      }
      const float d1 = warp_sum(a1), d2 = warp_sum(a2);
      const float p = expf(d1 * scale - ls[qi]);
      float wkeep = (float)nph;  // sum over phantom copies of mask / (1 - p_drop)
      if (thresh) {
        int kept = 0;
        for (int jj = nb + lane; jj < nmax; jj += 32) {
          const unsigned long long idx = ((unsigned long long)s * Tn + t) * (unsigned long long)nmax + jj;
          kept += keep_mask(seed, idx, thresh) ? 1 : 0;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) kept += __shfl_xor_sync(0xffffffffu, kept, o);
        wkeep = (float)kept * inv_keep;
      }
      const float dSsum = p * (wkeep * d2 - (float)nph * Dq[qi]) * scale;   // summed over the copies
      if (t < Tn) {
        const float pwk = p * wkeep;
#pragma unroll
        for (int i = 0; i < NF; ++i) {
          axpy4(dSsum, pk[i], dqa[qi][i]);
          axpy4(pwk, g4[i], dph[i]);
          axpy4(dSsum, q4[i], dph[i]);
        }
      }
    }
  }
#pragma unroll
  for (int qi = 0; qi < kQW; ++qi) {
    const int t = t0 + warp * kQW + qi;
    if (t < Tn) {
      const long long row = (long long)s * Tn + t;
      float4* dd = reinterpret_cast<float4*>(dq + row * H);
#pragma unroll
      for (int i = 0; i < NF; ++i) dd[lane + 32 * i] = dqa[qi][i];
      if (lane == 0) Dbuf[row] = Dq[qi];
    }
  }
  // block partial of the phantom gradient, warps combined in a fixed order
  __syncthreads();
#pragma unroll
  for (int i = 0; i < NF; ++i) *reinterpret_cast<float4*>(Ks + warp * H + lane * 4 + 128 * i) = dph[i];
  __syncthreads();
  const long long blk = (long long)blockIdx.y * gridDim.x + blockIdx.x;
  for (int h = threadIdx.x; h < H; h += blockDim.x) {
    float sacc = 0.f;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) sacc += Ks[w * H + h];
    dph_part[blk * H + h] = sacc;
  }
}

// ------------------------------------------------------------------------------------------------ backward: dkv
// One block per (crystal, tile of 32 of its atoms); loops over the queries of every sequence attending to that crystal.
//   phase 1: warp <-> 4 queries, lane <-> key : p, dS = p (w dO.k - D) scale, pw = p w      -> shared [32 t][32 j]
//   phase 2: warp <-> 4 keys,   lane <-> features: dk_j += sum_t dS[t, j] q_t + pw[t, j] dO_t
template <int NF>
__global__ void __launch_bounds__(kWarps * 32) bwd_kv_kernel(const float* __restrict__ dO, const float* __restrict__ q, long long q_ss,
                                                             const float* __restrict__ kv, const int* __restrict__ ptr,
                                                             const int* __restrict__ nmax_p, const float* __restrict__ lse,
                                                             const float* __restrict__ Dbuf, float* __restrict__ dkv, int S, int B, int Tn,
                                                             float scale, unsigned int thresh, float inv_keep,
                                                             unsigned long long seed,
                                                             const unsigned long long* __restrict__ seed_offset) {
  constexpr int H = 128 * NF, KP = H + 4;
  seed = mask_seed(seed, seed_offset);
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* Qs = reinterpret_cast<float*>(smem_raw);   // [32][H]
  float* Gs = Qs + 32 * H;                           // [32][H]
  float* Ks = Gs + 32 * H;                           // [32][KP]
  float* Ds = Ks + 32 * KP;                          // [32 t][32 j]  dS
  float* Ws = Ds + 32 * 32;                          // [32 t][32 j]  p * w
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int b = blockIdx.x;
  const int kbeg = ptr[b], nb = ptr[b + 1] - kbeg;
  const int nmax = *nmax_p;
  const int nrep = S / B;
  for (int j0 = blockIdx.y * kKT; j0 < nb; j0 += gridDim.y * kKT) {
    const int kt = min(kKT, nb - j0);
    __syncthreads();
    load_tile<H>(Ks, KP, kv, kbeg + j0, kt, false);
    float4 acc[4][NF];
#pragma unroll
    for (int kk = 0; kk < 4; ++kk)
#pragma unroll
      for (int i = 0; i < NF; ++i) acc[kk][i] = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int rep = 0; rep < nrep; ++rep) {
      const int s = b + rep * B;
      for (int tt0 = 0; tt0 < Tn; tt0 += 32) {
        __syncthreads();
        load_tile<H>(Qs, H, q + (long long)s * q_ss, tt0, Tn - tt0, true);
        load_tile<H>(Gs, H, dO + (long long)s * Tn * H, tt0, Tn - tt0, true);
        __syncthreads();
        // ---- phase 1
        {
          const float* qrow = Qs + (warp * kQW) * H;
          const float* grow = Gs + (warp * kQW) * H;
          const float* krow = Ks + lane * KP;
          float d1[kQW] = {0.f, 0.f, 0.f, 0.f}, d2[kQW] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 2
          for (int h4 = 0; h4 < H / 4; ++h4) {
            const float4 k4 = *reinterpret_cast<const float4*>(krow + 4 * h4);
#pragma unroll
            for (int qi = 0; qi < kQW; ++qi) {
              d1[qi] = dot4(*reinterpret_cast<const float4*>(qrow + qi * H + 4 * h4), k4, d1[qi]);
              d2[qi] = dot4(*reinterpret_cast<const float4*>(grow + qi * H + 4 * h4), k4, d2[qi]);
            }
          }
#pragma unroll
          for (int qi = 0; qi < kQW; ++qi) {
            const int tl = warp * kQW + qi, t = tt0 + tl;
            float dS = 0.f, pwv = 0.f;
            if (t < Tn && lane < kt) {
              const long long row = (long long)s * Tn + t;
              const float p = expf(d1[qi] * scale - __ldg(lse + row));
              float w = 1.f;
              if (thresh) {
                const unsigned long long idx = ((unsigned long long)s * Tn + t) * (unsigned long long)nmax + (j0 + lane);
                w = keep_mask(seed, idx, thresh) ? inv_keep : 0.f;
              }
              dS = p * (w * d2[qi] - __ldg(Dbuf + row)) * scale;
              pwv = p * w;
            }
            Ds[tl * 32 + lane] = dS;
            Ws[tl * 32 + lane] = pwv;
          }
        }
        __syncthreads();
        // ---- phase 2
        for (int tl = 0; tl < 32; ++tl) {
          const float4 s4 = *reinterpret_cast<const float4*>(Ds + tl * 32 + warp * 4);
          const float4 w4 = *reinterpret_cast<const float4*>(Ws + tl * 32 + warp * 4);
#pragma unroll
          for (int i = 0; i < NF; ++i) {
            const float4 qf = *reinterpret_cast<const float4*>(Qs + tl * H + lane * 4 + 128 * i);
            const float4 gf = *reinterpret_cast<const float4*>(Gs + tl * H + lane * 4 + 128 * i);
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
              axpy4(comp(s4, kk), qf, acc[kk][i]);
              axpy4(comp(w4, kk), gf, acc[kk][i]);
            }
          }
        }
      }
    }
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      const int j = warp * 4 + kk;
      if (j < kt) {
        float4* dd = reinterpret_cast<float4*>(dkv + (long long)(kbeg + j0 + j) * H);
#pragma unroll
        for (int i = 0; i < NF; ++i) dd[lane + 32 * i] = acc[kk][i];
      }
    }
  }
}

template <int NF>
static int launch_fwd(const float* q, long long q_ss, const float* kv, const float* phantom, const int* ptr, const int* nmax,
                      const float* resid, long long r_ss, float* out, float* lse, int S, int B, int Tn, float scale,
                      unsigned int thresh, float inv_keep, unsigned long long seed, const unsigned long long* seed_offset,
                      cudaStream_t st) {
  constexpr int H = 128 * NF;
  const size_t smem = sizeof(float) * (32 * H + 32 * (H + 4) + kWarps * 32 * 4);
  static PerDevice cfg_once;
  if (bool* cfg_flag = cfg_once.pending()) {
    cudaFuncSetAttribute(fwd_kernel<NF>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    *cfg_flag = true;
  }
  dim3 grid(ceil_div(Tn, kQB), S);
  fwd_kernel<NF><<<grid, kWarps * 32, smem, st>>>(q, q_ss, kv, phantom, ptr, nmax, resid, r_ss, out, lse, S, B, Tn, scale, thresh,
                                                  inv_keep, seed, seed_offset);
  return check_launch("xattn_fwd");
}

template <int NF>
static int launch_bwd(const float* dO, const float* q, long long q_ss, const float* kv, const float* phantom, const int* ptr,
                      const int* nmax, const float* out, const float* resid, long long r_ss, const float* lse, float* dq,
                      float* dkv, float* Dbuf, float* part, int S, int B, int Tn, float scale, unsigned int thresh,
                      float inv_keep, unsigned long long seed, const unsigned long long* seed_offset, bool do_kv,
                      cudaStream_t st) {
  constexpr int H = 128 * NF;
  const size_t smem_q = sizeof(float) * (2 * 32 * H + 32 * (H + 4) + kWarps * 32 * 4);
  const size_t smem_kv = sizeof(float) * (2 * 32 * H + 32 * (H + 4) + 2 * 32 * 32);
  static PerDevice cfg_once;
  if (bool* cfg_flag = cfg_once.pending()) {
    cudaFuncSetAttribute(bwd_q_kernel<NF>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_q);
    cudaFuncSetAttribute(bwd_kv_kernel<NF>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_kv);
    *cfg_flag = true;
  }
  dim3 grid(ceil_div(Tn, kQB), S);
  bwd_q_kernel<NF><<<grid, kWarps * 32, smem_q, st>>>(dO, q, q_ss, kv, phantom, ptr, nmax, out, resid, r_ss, lse, dq, Dbuf, part, S, B,
                                                      Tn, scale, thresh, inv_keep, seed, seed_offset);
  int rc = check_launch("xattn_bwd_q");
  if (rc != DOST_OK || !do_kv) return rc;
  dim3 gkv(B, 4);
  bwd_kv_kernel<NF><<<gkv, kWarps * 32, smem_kv, st>>>(dO, q, q_ss, kv, ptr, nmax, lse, Dbuf, dkv, S, B, Tn, scale, thresh, inv_keep,
                                                       seed, seed_offset);
  return check_launch("xattn_bwd_kv");
}

}  // namespace xa2

bool xattn_v2_supported(int H) { return H == 128 || H == 256 || H == 512; }

int xattn_v2_fwd(const float* q, long long q_ss, const float* kv, const float* phantom, const int* ptr, const int* nmax,
                 const float* resid, long long r_ss, float* out, float* lse, int S, int B, int Tn, int H, float scale,
                 unsigned int thresh, float inv_keep, unsigned long long seed, const unsigned long long* seed_offset,
                 cudaStream_t st) {
  switch (H) {
    case 128: return xa2::launch_fwd<1>(q, q_ss, kv, phantom, ptr, nmax, resid, r_ss, out, lse, S, B, Tn, scale, thresh, inv_keep, seed, seed_offset, st);
    case 256: return xa2::launch_fwd<2>(q, q_ss, kv, phantom, ptr, nmax, resid, r_ss, out, lse, S, B, Tn, scale, thresh, inv_keep, seed, seed_offset, st);
    default: return xa2::launch_fwd<4>(q, q_ss, kv, phantom, ptr, nmax, resid, r_ss, out, lse, S, B, Tn, scale, thresh, inv_keep, seed, seed_offset, st);
  }
}

int xattn_v2_bwd(const float* dO, const float* q, long long q_ss, const float* kv, const float* phantom, const int* ptr,
                 const int* nmax, const float* out, const float* resid, long long r_ss, const float* lse, float* dq, float* dkv,
                 float* Dbuf, float* part, int S, int B, int Tn, int H, float scale, unsigned int thresh, float inv_keep,
                 unsigned long long seed, const unsigned long long* seed_offset, bool do_kv, cudaStream_t st) {
  switch (H) {
    case 128: return xa2::launch_bwd<1>(dO, q, q_ss, kv, phantom, ptr, nmax, out, resid, r_ss, lse, dq, dkv, Dbuf, part, S, B, Tn, scale, thresh, inv_keep, seed, seed_offset, do_kv, st);
    case 256: return xa2::launch_bwd<2>(dO, q, q_ss, kv, phantom, ptr, nmax, out, resid, r_ss, lse, dq, dkv, Dbuf, part, S, B, Tn, scale, thresh, inv_keep, seed, seed_offset, do_kv, st);
    default: return xa2::launch_bwd<4>(dO, q, q_ss, kv, phantom, ptr, nmax, out, resid, r_ss, lse, dq, dkv, Dbuf, part, S, B, Tn, scale, thresh, inv_keep, seed, seed_offset, do_kv, st);
  }
}

}  // namespace dost
