// Helper kernels of the tensor-core formulation of the ragged energy->atom cross attention.
//
// The two contractions of every attention call (scores = q k^T and out = p k, and their four adjoints) run as ragged
// batched GEMMs on the TMA-fed tcgen05 kernel (gemm_bf.cu: one problem per sequence, per-problem row offsets into ONE
// key plane).  What remains here is O(S T npad) element-wise work:
//   kv_ext_build : LayerNorm'd atoms [N, H] -> bf16 hi/lo planes [N + B, H] with one extra row per crystal holding the
//                  phantom key (that layer's layer_norms[0].bias = what LayerNorm maps a zero-padded row to), so the
//                  (Nmax - n_b) phantom keys of the reference's zero padding become ONE extra GEMM column / row whose
//                  probability carries the multiplicity
//   softmax_fwd  : fp32 softmax over the n_b real columns + the phantom column (weight Nmax - n_b), probabilities written
//                  as operand planes (phantom column = total phantom probability), log-sum-exp saved
//   softmax_bwd  : dS = p (dP - sum p dP) scale, phantom column = the sum over its copies, written as planes
//   kv_ext_split : gradient of the extended key plane -> gradient of the atoms and of the phantom key
//   maps_from_planes : probability planes -> fp32 attention maps in the reference's padded layout (attention_maps recording)
#include <math.h>
#include <cuda_bf16.h>
#include "common.cuh"

namespace dost {
namespace xtc {

__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}

// one warp per output row of the extended plane; H % 128 == 0
__global__ void __launch_bounds__(256) kv_ext_build_kernel(const float* __restrict__ y, const float* __restrict__ beta,
                                                           const int* __restrict__ batch, const int* __restrict__ ptr, long long N,
                                                           int B, int H, __nv_bfloat16* __restrict__ hi,
                                                           __nv_bfloat16* __restrict__ lo, long long ldp) {
  const int lane = threadIdx.x & 31;
  const long long r = blockIdx.x * 8LL + (threadIdx.x >> 5);
  if (r >= N + B) return;
  const float* src;
  long long dst;
  if (r < N) {
    src = y + r * H;
    dst = r + __ldg(batch + r);
  } else {
    const int b = (int)(r - N);
    src = beta;
    dst = (long long)__ldg(ptr + b + 1) + b;      // the row after the crystal's last atom
  }
  for (int c = lane * 4; c < H; c += 128) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(src + c));
    uint2 h, l;
    h.x = pack_bf16(v.x, v.y);
    h.y = pack_bf16(v.z, v.w);
    l.x = pack_bf16(v.x - __uint_as_float(h.x << 16), v.y - __uint_as_float(h.x & 0xFFFF0000u));
    l.y = pack_bf16(v.z - __uint_as_float(h.y << 16), v.w - __uint_as_float(h.y & 0xFFFF0000u));
    *reinterpret_cast<uint2*>(hi + dst * ldp + c) = h;
    if (lo) *reinterpret_cast<uint2*>(lo + dst * ldp + c) = l;
  }
}

__global__ void __launch_bounds__(256) kv_ext_split_kernel(const float* __restrict__ dext, const int* __restrict__ batch,
                                                           const int* __restrict__ ptr, long long N, int B, int H,
                                                           float* __restrict__ dkv, float* __restrict__ dbeta_rows) {
  const int lane = threadIdx.x & 31;
  const long long r = blockIdx.x * 8LL + (threadIdx.x >> 5);
  if (r >= N + B) return;
  long long src;
  float* dst;
  if (r < N) {
    src = r + __ldg(batch + r);
    dst = dkv + r * H;
  } else {
    const int b = (int)(r - N);
    src = (long long)__ldg(ptr + b + 1) + b;
    dst = dbeta_rows + (long long)b * H;
  }
  for (int c = lane * 4; c < H; c += 128)
    *reinterpret_cast<float4*>(dst + c) = __ldg(reinterpret_cast<const float4*>(dext + src * H + c));
}

// Key gradients computed per SEQUENCE into a padded buffer dpad [reps * B][npad][H] (plain batched GEMMs with TMA / reduction
// stores instead of ragged accumulating ones) -> gradient of the atoms (sum over the `reps` sequences of a crystal, fixed
// order) and of the phantom key (row n_b of every block).  One warp per output row; H % 128 == 0.
__global__ void __launch_bounds__(256) kv_pad_split_kernel(const float* __restrict__ dpad, int npad, int reps,
                                                           const int* __restrict__ batch, const int* __restrict__ ptr, long long N,
                                                           int B, int H, float* __restrict__ dkv, float* __restrict__ dbeta_rows) {
  const int lane = threadIdx.x & 31;
  const long long r = blockIdx.x * 8LL + (threadIdx.x >> 5);
  if (r >= N + B) return;
  int b, j;
  float* dst;
  if (r < N) {
    b = __ldg(batch + r);
    j = (int)(r - __ldg(ptr + b));
    dst = dkv + r * H;
  } else {
    b = (int)(r - N);
    j = __ldg(ptr + b + 1) - __ldg(ptr + b);      // the phantom row follows the crystal's atoms
    dst = dbeta_rows + (long long)b * H;
  }
  const bool inside = j < npad;                   // (a crystal larger than the padding length was reported by the forward)
  for (int c = lane * 4; c < H; c += 128) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int rep = 0; rep < reps && inside; ++rep) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(dpad + (((long long)rep * B + b) * npad + j) * H + c));
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    *reinterpret_cast<float4*>(dst + c) = acc;
  }
}

// Number of the nph = nmax - nb phantom copies of row r that survive dropout (warp-cooperative; the copies occupy the key
// slots nb .. nmax-1 of the padded row, the mask index convention of attention_v2.cu: idx = r * nmax + key slot).
__device__ __forceinline__ int phantom_kept(unsigned long long seed, long long r, int nb, int nmax, unsigned int thresh, int lane) {
  int kept = 0;
  for (int jj = nb + lane; jj < nmax; jj += 32)
    kept += keep_mask(seed, (unsigned long long)r * (unsigned long long)nmax + jj, thresh) ? 1 : 0;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) kept += __shfl_xor_sync(0xffffffffu, kept, o);
  return kept;
}

// one warp per (sequence, query) row; NPL = ceil(npad / 32) columns per lane.  Dropout (thresh != 0): the planes receive
// the dropped-out probabilities mask / (1 - p) * P (multiheaded_attention.py:71); the phantom column carries
// (surviving copies) / (1 - p) * P_phantom.
template <int NPL>
__global__ void __launch_bounds__(256) softmax_fwd_kernel(const float* __restrict__ sc, const int* __restrict__ ptr,
                                                          const int* __restrict__ nmax_p, long long rows, int B, int Tn, int npad,
                                                          float scale, __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo,
                                                          long long ldp, float* __restrict__ lse, unsigned int* __restrict__ errw,
                                                          unsigned int thresh, float inv_keep, unsigned long long seed,
                                                          const unsigned long long* __restrict__ seed_offset) {
  const int lane = threadIdx.x & 31;
  const int nmax = *nmax_p;
  seed = mask_seed(seed, seed_offset);
  for (long long r = blockIdx.x * 8LL + (threadIdx.x >> 5); r < rows; r += (long long)gridDim.x * 8) {
    const int b = (int)((r / Tn) % B);
    int nb = __ldg(ptr + b + 1) - __ldg(ptr + b);
    if (nb + 1 > npad) {      // the host's padding length undercuts this crystal: reported, never read past the row
      if (errw && lane == 0) errw[kErrNmaxTooSmall] = 1u;
      nb = npad - 1;
    }
    const int nph = max(nmax - nb, 0);
    const int ncol = nb + (nph > 0 ? 1 : 0);     // columns that take part: the real keys, then the phantom column
    float v[NPL];
    float mx = -INFINITY;
#pragma unroll
    for (int i = 0; i < NPL; ++i) {
      const int c = lane + 32 * i;
      v[i] = (c < ncol) ? sc[r * npad + c] * scale : -INFINITY;
      mx = fmaxf(mx, v[i]);
    }
    mx = warp_max(mx);
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < NPL; ++i) {
      const int c = lane + 32 * i;
      float e = (c < ncol) ? expf(v[i] - mx) : 0.f;
      sum += (c == nb) ? e * (float)nph : e;      // the phantom column stands for nph identical keys
      v[i] = e;
    }
    sum = warp_sum(sum);
    const float inv = 1.0f / sum;
    float wph = (float)nph;                        // weight of the phantom column: surviving copies / (1 - p)
    if (thresh && nph > 0) wph = (float)phantom_kept(seed, r, nb, nmax, thresh, lane) * inv_keep;
#pragma unroll
    for (int i = 0; i < NPL; ++i) {
      const int c = lane + 32 * i;
      if (c < ldp) {
        float p = v[i] * inv;                     // zero for masked columns
        if (c == nb) p *= wph;
        else if (thresh && c < nb) p = keep_mask(seed, (unsigned long long)r * (unsigned long long)nmax + c, thresh) ? p * inv_keep : 0.f;
        const __nv_bfloat16 h = __float2bfloat16_rn(p);
        hi[r * ldp + c] = h;
        if (lo) lo[r * ldp + c] = __float2bfloat16_rn(p - __bfloat162float(h));
      }
    }
    if (lane == 0) lse[r] = mx + logf(sum);
  }
}

template <int NPL>
__global__ void __launch_bounds__(256) softmax_bwd_kernel(const float* __restrict__ sc, const float* __restrict__ lse,
                                                          const float* __restrict__ dP, const int* __restrict__ ptr,
                                                          const int* __restrict__ nmax_p, long long rows, int B, int Tn, int npad,
                                                          float scale, __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo,
                                                          long long ldp, unsigned int thresh, float inv_keep, unsigned long long seed,
                                                          const unsigned long long* __restrict__ seed_offset) {
  const int lane = threadIdx.x & 31;
  const int nmax = *nmax_p;
  seed = mask_seed(seed, seed_offset);
  for (long long r = blockIdx.x * 8LL + (threadIdx.x >> 5); r < rows; r += (long long)gridDim.x * 8) {
    const int b = (int)((r / Tn) % B);
    const int nb = min(__ldg(ptr + b + 1) - __ldg(ptr + b), npad - 1);
    const int nph = max(nmax - nb, 0);
    const int ncol = nb + (nph > 0 ? 1 : 0);
    const float ls = __ldg(lse + r);
    float wph = (float)nph;                        // sum over the phantom copies of mask / (1 - p)
    if (thresh && nph > 0) wph = (float)phantom_kept(seed, r, nb, nmax, thresh, lane) * inv_keep;
    // p: probability of ONE key (one phantom copy); g: gradient wrt its dropped-out probability, already weighted by the
    // mask (real keys) or by the surviving copies (phantom column)
    float p[NPL], g[NPL];
    float dot = 0.f;
#pragma unroll
    for (int i = 0; i < NPL; ++i) {
      const int c = lane + 32 * i;
      p[i] = 0.f;
      g[i] = 0.f;
      if (c < ncol) {
        p[i] = expf(sc[r * npad + c] * scale - ls);
        float gv = dP[r * npad + c];
        if (c == nb) gv *= wph;
        else if (thresh) gv = keep_mask(seed, (unsigned long long)r * (unsigned long long)nmax + c, thresh) ? gv * inv_keep : 0.f;
        g[i] = gv;
        dot = fmaf(p[i], gv, dot);
      }
    }
    dot = warp_sum(dot);
#pragma unroll
    for (int i = 0; i < NPL; ++i) {
      const int c = lane + 32 * i;
      if (c < ldp) {
        // d(score) summed over the copies a column stands for: real key p (g - dot); phantom p (wph g_raw - nph dot)
        const float o = scale * p[i] * (g[i] - ((c == nb) ? (float)nph : 1.f) * dot);
        const __nv_bfloat16 h = __float2bfloat16_rn(o);
        hi[r * ldp + c] = h;
        if (lo) lo[r * ldp + c] = __float2bfloat16_rn(o - __bfloat162float(h));
      }
    }
  }
}

// Attention maps (the reference's attn_weights, multihead_attention.py:68-71) from the probability planes a forward wrote:
// map[r, c] = hi + lo (hi alone without lo), i.e. exactly the P that the P K product consumed.  One warp per row, lane l owns
// columns 8 l .. 8 l + 7 of every 256-column pass (16-byte plane loads).
//   dense  (ptr == NULL): plane column c -> map column c < cols
//   ragged (ptr != NULL): row r belongs to crystal b = (r / Tn) % B; its n_b atom columns are copied, the phantom column n_b
//                         (total probability of the nmax - n_b zero-padded keys) is expanded into the key slots
//                         n_b .. nmax - 1 of the map - total / (nmax - n_b) each, or with dropout total / kept for the
//                         slots whose mask bit (index r * nmax + slot, as in the forward) survived and 0 for the others;
//                         columns past nmax are 0.
__global__ void __launch_bounds__(256) maps_from_planes_kernel(const __nv_bfloat16* __restrict__ hi, const __nv_bfloat16* __restrict__ lo,
                                                               long long ldp, long long rows, int cols, int Tn, int B,
                                                               const int* __restrict__ ptr, const int* __restrict__ nmax_p,
                                                               float* __restrict__ out, unsigned int thresh, unsigned long long seed,
                                                               const unsigned long long* __restrict__ seed_offset) {
  const int lane = threadIdx.x & 31;
  seed = mask_seed(seed, seed_offset);
  const int nmax = ptr ? *nmax_p : 0;
  const bool vec = (cols & 3) == 0;
  for (long long r = blockIdx.x * 8LL + (threadIdx.x >> 5); r < rows; r += (long long)gridDim.x * 8) {
    int nb = cols, nph = 0;
    float slot = 0.f;                              // value of one surviving phantom slot
    if (ptr) {
      const int b = (int)((r / Tn) % B);
      nb = min(__ldg(ptr + b + 1) - __ldg(ptr + b), (int)ldp - 1);
      nph = max(nmax - nb, 0);
      if (nph > 0) {
        float total = __bfloat162float(hi[r * ldp + nb]);
        if (lo) total += __bfloat162float(lo[r * ldp + nb]);
        const int kept = thresh ? phantom_kept(seed, r, nb, nmax, thresh, lane) : nph;
        slot = kept > 0 ? total / (float)kept : 0.f;
      }
    }
    const int pend = min(nb + nph, cols);          // last map column that carries probability (exclusive)
    float* orow = out + r * cols;
    for (int c0 = lane * 8; c0 < cols; c0 += 256) {
      float v[8];
      if (c0 < nb && c0 < ldp) {
        const uint4 h = __ldg(reinterpret_cast<const uint4*>(hi + r * ldp + c0));
        uint4 l = make_uint4(0u, 0u, 0u, 0u);
        if (lo) l = __ldg(reinterpret_cast<const uint4*>(lo + r * ldp + c0));
        const uint32_t hw[4] = {h.x, h.y, h.z, h.w}, lw[4] = {l.x, l.y, l.z, l.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          v[2 * k] = __uint_as_float(hw[k] << 16) + __uint_as_float(lw[k] << 16);
          v[2 * k + 1] = __uint_as_float(hw[k] & 0xFFFF0000u) + __uint_as_float(lw[k] & 0xFFFF0000u);
        }
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int c = c0 + j;
        if (c >= nb) {
          float s = 0.f;
          if (c < pend) s = (!thresh || keep_mask(seed, (unsigned long long)r * (unsigned long long)nmax + c, thresh)) ? slot : 0.f;
          v[j] = s;
        }
      }
      if (vec && c0 + 8 <= cols) {
        *reinterpret_cast<float4*>(orow + c0) = make_float4(v[0], v[1], v[2], v[3]);
        *reinterpret_cast<float4*>(orow + c0 + 4) = make_float4(v[4], v[5], v[6], v[7]);
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j)
          if (c0 + j < cols) orow[c0 + j] = v[j];
      }
    }
  }
}

}  // namespace xtc
}  // namespace dost

using namespace dost;

extern "C" int dost_attn_maps_from_planes(const void* p_hi, const void* p_lo, long long ld_p, long long rows, int cols, int T, int B,
                                          const int32_t* ptr, const int32_t* nmax, float* out, double drop_p,
                                          unsigned long long mask_seed, const unsigned long long* seed_offset,
                                          dost_stream_t stream) {
  DOST_REQUIRE(p_hi && out && rows > 0 && cols > 0 && ld_p > 0 && ld_p % 8 == 0 && ((uintptr_t)p_hi & 15) == 0 &&
                   ((uintptr_t)p_lo & 15) == 0 && ((uintptr_t)out & 15) == 0,
               "attn_maps_from_planes: bad args (ld_p %% 8 == 0, 16-byte aligned planes and map)");
  DOST_REQUIRE(ptr ? (nmax && T > 0 && B > 0) : cols <= ld_p, "attn_maps_from_planes: ragged maps need ptr, nmax, T and B; dense "
               "maps at most ld_p columns");
  DOST_REQUIRE(drop_p >= 0.0 && drop_p < 1.0, "attn_maps_from_planes: drop_p must be in [0, 1)");
  const unsigned int thresh = drop_p > 0.0 ? drop_threshold(drop_p) : 0u;
  const int blocks = (int)min64((rows + 7) / 8, 32LL * kNumSMs);
  xtc::maps_from_planes_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)p_hi, (const __nv_bfloat16*)p_lo, ld_p,
                                                                         rows, cols, T, B, ptr, nmax, out, thresh, mask_seed,
                                                                         seed_offset);
  return check_launch("attn_maps_from_planes");
}

extern "C" int dost_xattn_kv_ext_build(const float* y, const float* beta, const int32_t* batch, const int32_t* ptr, long long N, int B,
                                       int H, void* hi, void* lo, long long ldp, dost_stream_t stream) {
  DOST_REQUIRE(y && beta && batch && ptr && hi && N > 0 && B > 0 && H % 128 == 0 && ldp >= H && ldp % 8 == 0, "kv_ext_build: bad args");
  const long long rows = N + B;
  xtc::kv_ext_build_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, (cudaStream_t)stream>>>(y, beta, batch, ptr, N, B, H, (__nv_bfloat16*)hi,
                                                                                       (__nv_bfloat16*)lo, ldp);
  return check_launch("xattn_kv_ext_build");
}

extern "C" int dost_xattn_kv_ext_split(const float* dext, const int32_t* batch, const int32_t* ptr, long long N, int B, int H,
                                       float* dkv, float* dbeta_rows, dost_stream_t stream) {
  DOST_REQUIRE(dext && batch && ptr && dkv && dbeta_rows && N > 0 && B > 0 && H % 128 == 0, "kv_ext_split: bad args");
  const long long rows = N + B;
  xtc::kv_ext_split_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, (cudaStream_t)stream>>>(dext, batch, ptr, N, B, H, dkv, dbeta_rows);
  return check_launch("xattn_kv_ext_split");
}

extern "C" int dost_xattn_kv_pad_split(const float* dpad, int npad, int reps, const int32_t* batch, const int32_t* ptr, long long N, int B,
                                       int H, float* dkv, float* dbeta_rows, dost_stream_t stream) {
  DOST_REQUIRE(dpad && batch && ptr && dkv && dbeta_rows && N > 0 && B > 0 && H % 128 == 0 && npad > 0 && reps >= 1, "kv_pad_split: bad args");
  const long long rows = N + B;
  xtc::kv_pad_split_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, (cudaStream_t)stream>>>(dpad, npad, reps, batch, ptr, N, B, H, dkv, dbeta_rows);
  return check_launch("xattn_kv_pad_split");
}

#define DOST_XTC_DISPATCH(KERNEL, ...)                                        \
  switch (npl) {                                                              \
    case 1: xtc::KERNEL<1><<<blocks, 256, 0, st>>>(__VA_ARGS__); break;       \
    case 2: xtc::KERNEL<2><<<blocks, 256, 0, st>>>(__VA_ARGS__); break;       \
    case 4: xtc::KERNEL<4><<<blocks, 256, 0, st>>>(__VA_ARGS__); break;       \
    case 8: xtc::KERNEL<8><<<blocks, 256, 0, st>>>(__VA_ARGS__); break;       \
    case 16: xtc::KERNEL<16><<<blocks, 256, 0, st>>>(__VA_ARGS__); break;     \
    default: xtc::KERNEL<32><<<blocks, 256, 0, st>>>(__VA_ARGS__); break;     \
  }

static inline int npl_for(long long ldp) {
  int npl = (int)((ldp + 31) / 32), p = 1;
  while (p < npl) p <<= 1;
  return p;
}

extern "C" int dost_xattn_softmax_fwd_dseed(const float* scores, const int32_t* ptr, const int32_t* nmax, long long rows, int B,
                                            int T, int npad, double scale, void* hi, void* lo, long long ldp, float* lse,
                                            double drop_p, unsigned long long seed, const unsigned long long* seed_offset,
                                            dost_stream_t stream) {
  DOST_REQUIRE(scores && ptr && nmax && hi && lse && rows > 0 && npad > 0 && ldp >= npad && ldp <= 1024, "xattn_softmax_fwd: bad args");
  cudaStream_t st = (cudaStream_t)stream;
  const int npl = npl_for(ldp);
  const int blocks = (int)min64((rows + 7) / 8, 32LL * kNumSMs);
  DOST_REQUIRE(drop_p >= 0.0 && drop_p < 1.0, "xattn_softmax_fwd: drop_p must be in [0, 1)");
  const unsigned int thresh = drop_p > 0.0 ? drop_threshold(drop_p) : 0u;
  const float inv_keep = (float)(1.0 / (1.0 - drop_p));
  DOST_XTC_DISPATCH(softmax_fwd_kernel, scores, ptr, nmax, rows, B, T, npad, (float)scale, (__nv_bfloat16*)hi, (__nv_bfloat16*)lo, ldp, lse,
                    device_error_words(), thresh, inv_keep, seed, seed_offset)
  return check_launch("xattn_softmax_fwd");
}

extern "C" int dost_xattn_softmax_fwd(const float* scores, const int32_t* ptr, const int32_t* nmax, long long rows, int B, int T,
                                      int npad, double scale, void* hi, void* lo, long long ldp, float* lse, double drop_p,
                                      unsigned long long seed, dost_stream_t stream) {
  return dost_xattn_softmax_fwd_dseed(scores, ptr, nmax, rows, B, T, npad, scale, hi, lo, ldp, lse, drop_p, seed, nullptr, stream);
}

extern "C" int dost_xattn_softmax_bwd_dseed(const float* scores, const float* lse, const float* dP, const int32_t* ptr,
                                            const int32_t* nmax, long long rows, int B, int T, int npad, double scale, void* hi,
                                            void* lo, long long ldp, double drop_p, unsigned long long seed,
                                            const unsigned long long* seed_offset, dost_stream_t stream) {
  DOST_REQUIRE(scores && lse && dP && ptr && nmax && hi && rows > 0 && npad > 0 && ldp >= npad && ldp <= 1024, "xattn_softmax_bwd: bad args");
  cudaStream_t st = (cudaStream_t)stream;
  const int npl = npl_for(ldp);
  const int blocks = (int)min64((rows + 7) / 8, 32LL * kNumSMs);
  DOST_REQUIRE(drop_p >= 0.0 && drop_p < 1.0, "xattn_softmax_bwd: drop_p must be in [0, 1)");
  const unsigned int thresh = drop_p > 0.0 ? drop_threshold(drop_p) : 0u;
  const float inv_keep = (float)(1.0 / (1.0 - drop_p));
  DOST_XTC_DISPATCH(softmax_bwd_kernel, scores, lse, dP, ptr, nmax, rows, B, T, npad, (float)scale, (__nv_bfloat16*)hi, (__nv_bfloat16*)lo,
                    ldp, thresh, inv_keep, seed, seed_offset)
  return check_launch("xattn_softmax_bwd");
}

extern "C" int dost_xattn_softmax_bwd(const float* scores, const float* lse, const float* dP, const int32_t* ptr, const int32_t* nmax,
                                      long long rows, int B, int T, int npad, double scale, void* hi, void* lo, long long ldp,
                                      double drop_p, unsigned long long seed, dost_stream_t stream) {
  return dost_xattn_softmax_bwd_dseed(scores, lse, dP, ptr, nmax, rows, B, T, npad, scale, hi, lo, ldp, drop_p, seed, nullptr, stream);
}
