// Fused single-head attention forward on the tensor cores (sm_100a):  out = resid + softmax_fp32(q k^T * scale) k
// for S sequences of Lq queries against their own key set (keys ARE the values: layers/multihead_attention.py:68-72 has
// no projections), in ONE kernel: no score matrix in HBM.
//
//   dense  : sequence s owns keys k[s*Lk .. s*Lk+Lk)                       (energy self-attention, DOSTransformer.py:85-91)
//   ragged : sequence s owns rows k_rowoff[s] .. +k_count[s] of ONE extended key plane whose last row per crystal is the
//            phantom key; that column stands for nmax - n_b identical zero-padded keys (to_dense_batch + LayerNorm,
//            DOSTransformer.py:61-63): its exp() is weighted by the multiplicity
//
// One persistent CTA per SM; a work item is (sequence, 128-query tile).  Operands are the bf16 hi/lo planes every other
// tensor-core kernel of this library uses (bf16x3: lo*hi + hi*lo + hi*hi per product).
//   warp 0      TMA producer.  Phase A (S = Q K^T): Q and the key set stream together in 64-column slices through two
//               96 KB stages - Q[128, 64] and K[NB keys, 64], NB in {32, 64, 128, 256} covering the sequence's keys - so
//               every MMA has N = NB (a 32-key-wide MMA re-reads the 4 KB A tile for 1 KB of B: shared-memory bound at a
//               fifth of the tensor rate; measured 13 of 24 us per item).  Phase B (O = P K): the keys again, in 32-key chunks
//               {64 columns, 32 keys} as the MN-major B operand, through two 32 KB stages.
//   warp 1      MMA issuer (one lane): S[128, NB] into TMEM columns 0..255; after the softmax O[128, H] += P[:, chunk] K_c
//               into TMEM columns 256..; issues the TMA stores that save P (training)
//   warps 2-9   softmax + epilogue, thread = query row (TMEM lane), two warps per lane quarter splitting the columns:
//               pass 1 row max; pass 2 e = exp2((s - max) * scale * log2 e) (phantom column x multiplicity), written back to
//               TMEM, row sum; pass 3 p = e / sum -> bf16 hi/lo into shared memory in the UMMA K-major SWIZZLE_128B layout
//               (over the phase-A stages, dead by then) = the A operand of P K and, unchanged, the source of the TMA store
//               that saves P for the backward pass.  Epilogue: O -> swizzled staging tile -> row-contiguous reads, +
//               residual, coalesced fp32 stores (thread-per-row global accesses touch 32 lines per instruction: measured
//               15 us per item), overlapping phase A of the next item.
// TMEM: 256 columns of scores + H columns of output (<= 512).  Shared memory: 192 KB of stages / P tile + 32 KB staging.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cstdlib>
#include "common.cuh"
#include "tc_ptx.cuh"

namespace dost {
namespace fa {

constexpr int BM = 128;                 // queries per tile
constexpr int KC = 32;                  // keys per phase-B chunk
constexpr int kSoftWarps = 8;
constexpr int kThreads = (2 + kSoftWarps) * 32;
constexpr int kMaxKeys = 256;           // score columns that fit TMEM next to the output
constexpr int QP_PLANE = BM * 256 * 2;  // 64 KB: one plane of P (<= 256 keys)
// phase A stage: Q slice [128, 64] hi | lo (16 KB each), K slice [<= 256, 64] hi | lo (32 KB each)
constexpr int A_STAGE = 98304, A_QLO = 16384, A_KHI = 32768, A_KLO = 65536;
// phase B: P tile at 0 (hi) / 64 KB (lo), key chunks [32, H] hi | lo (16 KB each) in two stages after it
constexpr int OFF_VS = 2 * QP_PLANE, V_PLANE = KC * 256 * 2, V_STAGE = 2 * V_PLANE;
constexpr int OFF_STG = 2 * A_STAGE;                      // epilogue staging: one 32 x 32 fp32 tile per softmax warp
constexpr int OFF_XCH = OFF_STG + kSoftWarps * 4096;     // float [2][2][128]: row max / row sum exchange between the halves
constexpr int OFF_BAR = OFF_XCH + 2 * 2 * BM * 4;
constexpr int kSmemBytes = OFF_BAR + 256;
static_assert(OFF_VS + 2 * V_STAGE <= OFF_STG, "phase B must fit the phase A stages");

struct Maps {
  CUtensorMap q_hi, q_lo;
  CUtensorMap ka_hi[4], ka_lo[4];      // phase A key slices: box {64 columns, 32 << i keys}
  CUtensorMap k_hi, k_lo;              // phase B key chunks: box {64 columns, 32 keys}
  CUtensorMap p_hi, p_lo;
};

struct Params {
  int S, Lq, Lk, H, QT, total_tiles, kpad;
  const int* k_rowoff;
  const int* k_count;
  const int* nmax;
  float scale_log2e;
  const float* residual;
  long long res_seq_stride;
  float* out;
  int store_p;
  unsigned int* errw;
  // attention dropout (multihead_attention.py:71): counter-based keep mask of the library (common.cuh), index =
  // row * mask_ld + key slot with mask_ld = Lk (dense) or the padding length Nmax (ragged: the phantom copies occupy the slots
  // n_b .. Nmax-1 and survive individually); thresh == 0: off
  unsigned int thresh;
  float inv_keep;
  unsigned long long seed;
  const unsigned long long* seed_offset;   // optional device word added to seed (dost.h), read before the work-item loop
  float* lse;                    // optional [S * Lq]: log-sum-exp of the scaled scores (the dropout backward recomputes P)
};

using namespace ptx;      // tcgen05 / TMA / mbarrier wrappers (tc_ptx.cuh)

__device__ __forceinline__ void soft_bar() { asm volatile("bar.sync 1, %0;" ::"r"(kSoftWarps * 32) : "memory"); }
// K-major operands: lbo = 0; the MN-major key chunks of phase B are 32-row TMA boxes: lbo = 4096
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo) { return make_smem_desc(saddr, lbo); }
__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// Phase timeline of CTA 0 (development aid, compiled in with -DDOST_ATTN_TIMELINE): globaltimer stamps per work item.
#ifdef DOST_ATTN_TIMELINE
__device__ unsigned long long g_timeline[64 * 16];
__device__ __forceinline__ void stamp(int local, int slot) {
  if (blockIdx.x == 0 && local < 64) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    g_timeline[local * 16 + slot] = t;
  }
}
#define FA_STAMP(local, slot) stamp(local, slot)
#else
#define FA_STAMP(local, slot)
#endif

struct Item {
  int s, m0, krow, zb, nk, nch, ncol, nb, nph, nbi;    // nbi: phase A box index, NB = 32 << nbi keys
};
__device__ __forceinline__ Item item_of(const Params& p, int tile) {
  Item it;
  it.s = tile / p.QT;
  it.m0 = (tile - it.s * p.QT) * BM;
  if (p.k_rowoff) {
    it.krow = __ldg(p.k_rowoff + it.s);
    it.zb = 0;
    int cnt = __ldg(p.k_count + it.s);          // real keys + the phantom row
    if (cnt > p.kpad) {                         // the host's padding length undercuts this crystal: reported, clamped
      if (p.errw) p.errw[kErrNmaxTooSmall] = 1u;
      cnt = p.kpad;
    }
    it.nb = cnt - 1;
    it.nph = p.nmax ? max(__ldg(p.nmax) - it.nb, 0) : 0;
    it.ncol = it.nb + (it.nph > 0 ? 1 : 0);
    it.nk = cnt;
  } else {
    it.krow = 0;
    it.zb = it.s;
    it.nk = p.Lk;
    it.nb = -1;
    it.nph = 0;
    it.ncol = p.Lk;
  }
  it.nch = (it.nk + KC - 1) / KC;
  it.nbi = it.nk <= 32 ? 0 : (it.nk <= 64 ? 1 : (it.nk <= 128 ? 2 : 3));
  return it;
}

template <int NSPLIT>
__global__ void __launch_bounds__(kThreads, 1) attn_fwd_kernel(const __grid_constant__ Maps maps, const Params p) {
  constexpr bool SPLIT = NSPLIT == 3;
  extern __shared__ __align__(1024) unsigned char smem[];
  const uint32_t sbase = smem_u32(smem);
  if ((sbase & 1023u) != 0u) __trap();             // the swizzled tiles need a 1024-byte aligned window
  float* xch = reinterpret_cast<float*>(smem + OFF_XCH);
  unsigned long long* bars = reinterpret_cast<unsigned long long*>(smem + OFF_BAR);
  uint32_t* tmem_base_s = reinterpret_cast<uint32_t*>(smem + OFF_BAR + 128);
  const uint32_t s_full = smem_u32(&bars[0]), p_full = smem_u32(&bars[1]), o_full = smem_u32(&bars[2]);
  const uint32_t o_empty = smem_u32(&bars[3]), x_free = smem_u32(&bars[4]);
  const uint32_t afull0 = smem_u32(&bars[5]), aempty0 = smem_u32(&bars[7]);
  const uint32_t vfull0 = smem_u32(&bars[9]), vempty0 = smem_u32(&bars[11]);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int H = p.H, HB = H / 64;

  if (threadIdx.x == 0) {
    mbar_init(s_full, 1);
    mbar_init(p_full, kSoftWarps);
    mbar_init(o_full, 1);
    mbar_init(o_empty, kSoftWarps);
    mbar_init(x_free, 2);                          // PV MMAs retired (tcgen05.commit) + the P stores have read the tile
    for (int s = 0; s < 2; ++s) {
      mbar_init(afull0 + 8 * s, 1);
      mbar_init(aempty0 + 8 * s, 1);
      mbar_init(vfull0 + 8 * s, 1);
      mbar_init(vempty0 + 8 * s, 1);
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_base_s)), "r"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_base_s;
  const uint32_t tmem_S = tmem_base, tmem_O = tmem_base + kMaxKeys;
  const uint32_t sQP = sbase, sVS = sbase + OFF_VS;

  if (warp == 0) {
    // ============================================================== TMA producer
    if (lane == 0) {
      int ast = 0, vst = 0;
      uint32_t aphase = 0, vphase = 0;
      int local = 0;
      for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++local) {
        const Item it = item_of(p, tile);
        if (local > 0) mbar_wait(x_free, (local - 1) & 1);           // the previous item's P tile and key chunks are dead
        FA_STAMP(local, 0);
        const int NB = 32 << it.nbi;
        // ---- phase A: Q[:, 64 hb .. +64) and K[0 .. NB, 64 hb .. +64)
        for (int hb = 0; hb < HB; ++hb) {
          mbar_wait(aempty0 + 8 * ast, aphase ^ 1);
          const uint32_t bar = afull0 + 8 * ast;
          mbar_expect_tx(bar, (SPLIT ? 2 : 1) * (BM + NB) * 128);
          const uint32_t dst = sbase + ast * A_STAGE;
          tma_load_3d(dst, &maps.q_hi, hb * 64, it.m0, it.s, bar);
          tma_load_3d(dst + A_KHI, &maps.ka_hi[it.nbi], hb * 64, it.krow, it.zb, bar);
          if (SPLIT) {
            tma_load_3d(dst + A_QLO, &maps.q_lo, hb * 64, it.m0, it.s, bar);
            tma_load_3d(dst + A_KLO, &maps.ka_lo[it.nbi], hb * 64, it.krow, it.zb, bar);
          }
          if (++ast == 2) {
            ast = 0;
            aphase ^= 1;
          }
        }
        // ---- phase B: the key chunks land on the phase A stages: all of its MMAs must have retired
        mbar_wait(s_full, local & 1);
        for (int c = 0; c < it.nch; ++c) {
          mbar_wait(vempty0 + 8 * vst, vphase ^ 1);
          const uint32_t bar = vfull0 + 8 * vst;
          mbar_expect_tx(bar, (SPLIT ? 2 : 1) * KC * H * 2);
          const uint32_t dst = sVS + vst * V_STAGE;
          for (int hb = 0; hb < HB; ++hb) {
            tma_load_3d(dst + hb * 4096, &maps.k_hi, hb * 64, it.krow + c * KC, it.zb, bar);
            if (SPLIT) tma_load_3d(dst + V_PLANE + hb * 4096, &maps.k_lo, hb * 64, it.krow + c * KC, it.zb, bar);
          }
          if (++vst == 2) {
            vst = 0;
            vphase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ============================================================== MMA issuer
    const uint32_t idesc_pv = make_idesc(BM, H, false, true);
    int ast = 0, vst = 0;
    uint32_t aphase = 0, vphase = 0;
    int local = 0;
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++local) {
      const Item it = item_of(p, tile);
      const uint32_t idesc_qk = make_idesc(BM, 32 << it.nbi, false, false);
      // ---- S[128, NB] = Q K^T, one 64-column slice of both operands per stage
      for (int hb = 0; hb < HB; ++hb) {
        mbar_wait(afull0 + 8 * ast, aphase);
        tc_fence_after();
        if (lane == 0) {
          if (hb == 0) FA_STAMP(local, 1);
          const uint32_t sA = sbase + ast * A_STAGE;
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) {
            const uint64_t dAhi = make_desc(sA + ks * 32, 0), dBhi = make_desc(sA + A_KHI + ks * 32, 0);
            const uint32_t first = (hb > 0 || ks > 0) ? 1u : 0u;
            if (SPLIT) {
              const uint64_t dAlo = make_desc(sA + A_QLO + ks * 32, 0), dBlo = make_desc(sA + A_KLO + ks * 32, 0);
              umma_f16(tmem_S, dAlo, dBhi, idesc_qk, first);
              umma_f16(tmem_S, dAhi, dBlo, idesc_qk, 1u);
              umma_f16(tmem_S, dAhi, dBhi, idesc_qk, 1u);
            } else {
              umma_f16(tmem_S, dAhi, dBhi, idesc_qk, first);
            }
          }
          umma_commit(aempty0 + 8 * ast);
          if (hb == HB - 1) umma_commit(s_full);
        }
        __syncwarp();
        if (++ast == 2) {
          ast = 0;
          aphase ^= 1;
        }
      }
      // ---- P is in shared memory (written over the phase A stages by the softmax warps)
      if (lane == 0) FA_STAMP(local, 2);
      mbar_wait(p_full, local & 1);
      tc_fence_after();
      if (lane == 0) FA_STAMP(local, 3);
      if (lane == 0 && p.store_p) {                // save P for the backward pass: the tile already has the TMA layout
        for (int jb = 0; jb < (p.kpad + 63) / 64; ++jb) {
          tma_store_3d(&maps.p_hi, sQP + jb * 16384, jb * 64, it.m0, it.s);
          if (SPLIT) tma_store_3d(&maps.p_lo, sQP + QP_PLANE + jb * 16384, jb * 64, it.m0, it.s);
        }
        bulk_commit();
      }
      if (local > 0) {                             // the epilogue of the previous item has drained O
        mbar_wait(o_empty, (local - 1) & 1);
        tc_fence_after();
      }
      // ---- O += P[:, chunk] K_c
      for (int c = 0; c < it.nch; ++c) {
        mbar_wait(vfull0 + 8 * vst, vphase);
        tc_fence_after();
        if (lane == 0) {
          const uint32_t sB = sVS + vst * V_STAGE;
#pragma unroll
          for (int k2 = 0; k2 < KC / 16; ++k2) {
            const int k16 = c * (KC / 16) + k2;    // 16-key step inside the P tile
            const uint32_t a_off = (k16 >> 2) * 16384 + (k16 & 3) * 32, b_off = k2 * 2048;
            const uint64_t dAhi = make_desc(sQP + a_off, 0), dBhi = make_desc(sB + b_off, 4096);
            const uint32_t first = (c > 0 || k2 > 0) ? 1u : 0u;
            if (SPLIT) {
              const uint64_t dAlo = make_desc(sQP + QP_PLANE + a_off, 0), dBlo = make_desc(sB + V_PLANE + b_off, 4096);
              umma_f16(tmem_O, dAlo, dBhi, idesc_pv, first);
              umma_f16(tmem_O, dAhi, dBlo, idesc_pv, 1u);
              umma_f16(tmem_O, dAhi, dBhi, idesc_pv, 1u);
            } else {
              umma_f16(tmem_O, dAhi, dBhi, idesc_pv, first);
            }
          }
          umma_commit(vempty0 + 8 * vst);
          if (c == it.nch - 1) {
            FA_STAMP(local, 4);
            umma_commit(o_full);
            umma_commit(x_free);
            if (p.store_p) bulk_wait_read0();      // the P stores have read the tile too
            mbar_arrive(x_free);
          }
        }
        __syncwarp();
        if (++vst == 2) {
          vst = 0;
          vphase ^= 1;
        }
      }
    }
    if (lane == 0 && p.store_p) bulk_wait0();
  } else {
    // ============================================================== softmax + epilogue (8 warps, thread = query row)
    const int quarter = warp & 3, half = (warp - 2) >> 2;
    const int row = quarter * 32 + lane;
    const uint32_t lane_addr = static_cast<uint32_t>(quarter * 32) << 16;
    float* xmax = xch;                 // [2][128]
    float* xsum = xch + 2 * BM;        // [2][128]
    const float sl2 = p.scale_log2e;
    const unsigned long long seed = mask_seed(p.seed, p.seed_offset);
    int local = 0;
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++local) {
      const Item it = item_of(p, tile);
      const int hsplit = (it.nch + 1) / 2;
      const int cbeg = half ? hsplit : 0, cend = half ? it.nch : hsplit;
      mbar_wait(s_full, local & 1);
      tc_fence_after();
      if (threadIdx.x == 64) FA_STAMP(local, 5);
      uint32_t r[32];
      // ---- pass 1: row maximum of the scaled scores over the columns that take part
      float mx = -INFINITY;
      for (int c = cbeg; c < cend; ++c) {
        tmem_ld32(tmem_S + lane_addr + c * KC, r);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const float v = __uint_as_float(r[j]) * sl2;
          mx = (c * KC + j < it.ncol) ? fmaxf(mx, v) : mx;
        }
      }
      xmax[half * BM + row] = mx;
      soft_bar();
      if (threadIdx.x == 64) FA_STAMP(local, 6);
      mx = fmaxf(xmax[row], xmax[BM + row]);
      // ---- pass 2: e = exp2(s - max) (the phantom column stands for nph identical keys), kept in TMEM; row sum
      float sum = 0.f;
      const float wph = static_cast<float>(it.nph);
      for (int c = cbeg; c < cend; ++c) {
        tmem_ld32(tmem_S + lane_addr + c * KC, r);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const int col = c * KC + j;
          float e = (col < it.ncol) ? ex2(fmaf(__uint_as_float(r[j]), sl2, -mx)) : 0.f;
          e = (col == it.nb) ? e * wph : e;
          sum += e;
          r[j] = __float_as_uint(e);
        }
        tmem_st32(tmem_S + lane_addr + c * KC, r);
      }
      tmem_st_wait();
      xsum[half * BM + row] = sum;
      soft_bar();
      if (threadIdx.x == 64) FA_STAMP(local, 7);
      const float inv = 1.0f / (xsum[row] + xsum[BM + row]);
      // ---- pass 3: p = e / sum as bf16 hi/lo, K-major SWIZZLE_128B tile [128 rows][64-key blocks] over the dead Q tile
      const uint32_t prow = sQP + row * 128;
      const uint32_t swz = row & 7;
      // dropout: this row's mask indices start at rglob * mask_ld; the phantom column keeps (surviving copies) / nph of its mass
      const unsigned int thresh = p.thresh;
      const long long rglob = (long long)it.s * p.Lq + it.m0 + row;
      const int mask_ld = p.k_rowoff ? (p.nmax ? __ldg(p.nmax) : p.kpad) : p.Lk;
      const unsigned long long mbase = (unsigned long long)rglob * (unsigned long long)mask_ld;
      float ph_scale = 1.f;
      if (thresh && it.nph > 0 && it.nb >= cbeg * KC && it.nb < cend * KC) {
        int kept = 0;
        for (int jj = it.nb; jj < it.nb + it.nph; ++jj) kept += keep_mask(seed, mbase + jj, thresh) ? 1 : 0;
        ph_scale = (float)kept * p.inv_keep / (float)it.nph;
      }
      if (p.lse && half == 0 && it.m0 + row < p.Lq) p.lse[rglob] = mx * 0.6931471805599453f + logf(xsum[row] + xsum[BM + row]);
      for (int c = cbeg; c < cend; ++c) {
        tmem_ld32(tmem_S + lane_addr + c * KC, r);
        tmem_ld_wait();
        const uint32_t pb = prow + (c >> 1) * 16384;
        if (thresh) {
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const int col = c * KC + j;
            float e = __uint_as_float(r[j]);
            if (col == it.nb) e *= ph_scale;
            else e = keep_mask(seed, mbase + col, thresh) ? e * p.inv_keep : 0.f;
            r[j] = __float_as_uint(e);
          }
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          uint32_t hi[4], lo[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float a = __uint_as_float(r[8 * i + 2 * q]) * inv, b = __uint_as_float(r[8 * i + 2 * q + 1]) * inv;
            hi[q] = pack_bf16(a, b);
            lo[q] = pack_bf16(a - __uint_as_float(hi[q] << 16), b - __uint_as_float(hi[q] & 0xFFFF0000u));
          }
          const uint32_t off = (((c & 1) * 4 + i) ^ swz) << 4;
          sts128(pb + off, hi[0], hi[1], hi[2], hi[3]);
          if (SPLIT) sts128(pb + QP_PLANE + off, lo[0], lo[1], lo[2], lo[3]);
        }
      }
      if (p.store_p) {       // key chunks this sequence does not have: the saved planes read as zero there
        const int call = (p.kpad + 63) / 64 * 2;
        for (int c = it.nch + half; c < call; c += 2) {
          const uint32_t pb = prow + (c >> 1) * 16384;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const uint32_t off = (((c & 1) * 4 + i) ^ swz) << 4;
            sts128(pb + off, 0u, 0u, 0u, 0u);
            if (SPLIT) sts128(pb + QP_PLANE + off, 0u, 0u, 0u, 0u);
          }
        }
      }
      fence_async_smem();          // generic-proxy writes of P -> visible to the tensor core / TMA (async proxy)
      tc_fence_before();           // this thread's tcgen05.ld / st of S are ordered before the next item's MMAs into S
      __syncwarp();
      if (lane == 0) mbar_arrive(p_full);
      if (threadIdx.x == 64) FA_STAMP(local, 8);
      // ---- epilogue: O + residual -> out (this warp: its 32 rows, one half of the H columns)
      mbar_wait(o_full, local & 1);
      tc_fence_after();
      if (threadIdx.x == 64) FA_STAMP(local, 9);
      // this warp: its 32 rows x one half of the H columns, 32 columns at a time through its staging tile (lane = row in,
      // 4 rows x 128 contiguous bytes per instruction out)
      const int hw = H / 2;
      const int rsub = lane >> 3, cj = lane & 7;
      const uint32_t stg = sbase + OFF_STG + (warp - 2) * 4096;
      const int grow0 = it.m0 + quarter * 32 + rsub;
      float* obase = p.out + ((long long)it.s * p.Lq + grow0) * H + half * hw + cj * 4;
      const float* rbase = p.residual ? p.residual + (long long)it.s * p.res_seq_stride + (long long)grow0 * H + half * hw + cj * 4 : nullptr;
      for (int c0 = 0; c0 < hw; c0 += 32) {
        tmem_ld32(tmem_O + lane_addr + half * hw + c0, r);
        float4 res[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {                 // residual rows requested before the accumulator round trip
          res[i] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (rbase && grow0 + 4 * i < p.Lq) res[i] = __ldg(reinterpret_cast<const float4*>(rbase + (long long)(4 * i) * H + c0));
        }
        tmem_ld_wait();
        if (c0 + 32 >= hw) {       // last read of O: the MMA warp may overwrite it
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(o_empty);
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) sts128(stg + lane * 128 + ((j ^ (lane & 7)) << 4), r[4 * j], r[4 * j + 1], r[4 * j + 2], r[4 * j + 3]);
        __syncwarp();
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int rl = rsub + 4 * i;
          float4 v = lds128(stg + rl * 128 + ((cj ^ (rl & 7)) << 4));
          v.x += res[i].x; v.y += res[i].y; v.z += res[i].z; v.w += res[i].w;
          if (grow0 + 4 * i < p.Lq) *reinterpret_cast<float4*>(obase + (long long)(4 * i) * H + c0) = v;
        }
        __syncwarp();              // the staging tile may be overwritten by the next chunk
      }
      if (threadIdx.x == 64) FA_STAMP(local, 10);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

// dS = scale * P (dP - sum_c P dP) per row, P read back from its saved bf16 hi/lo planes (hi + lo carries the probability to
// 2^-17; masked / padded columns hold exact zeros, and a phantom column holds the TOTAL probability of its copies, for which
// the same formula gives the gradient summed over the copies).  Output: operand planes of dS.  One warp per row.
// (16-byte accesses: lane l owns columns 8 l .. 8 l + 7 of a pass of 256 columns)
__global__ void __launch_bounds__(256) ds_from_planes_kernel(const __nv_bfloat16* __restrict__ p_hi, const __nv_bfloat16* __restrict__ p_lo,
                                                             long long ld_pp, const float* __restrict__ dP, long long ld_dp,
                                                             long long rows, int cols, float scale, __nv_bfloat16* __restrict__ hi,
                                                             __nv_bfloat16* __restrict__ lo, long long ldp) {
  const int lane = threadIdx.x & 31;
  const int c0 = lane * 8;
  for (long long r = blockIdx.x * 8LL + (threadIdx.x >> 5); r < rows; r += (long long)gridDim.x * 8) {
    float pv[8], g[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) pv[j] = g[j] = 0.f;
    if (c0 < cols) {
      const uint4 h = __ldg(reinterpret_cast<const uint4*>(p_hi + r * ld_pp + c0));
      uint4 l = make_uint4(0u, 0u, 0u, 0u);
      if (p_lo) l = __ldg(reinterpret_cast<const uint4*>(p_lo + r * ld_pp + c0));
      const uint32_t hw[4] = {h.x, h.y, h.z, h.w}, lw[4] = {l.x, l.y, l.z, l.w};
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        pv[2 * q] = __uint_as_float(hw[q] << 16) + __uint_as_float(lw[q] << 16);
        pv[2 * q + 1] = __uint_as_float(hw[q] & 0xFFFF0000u) + __uint_as_float(lw[q] & 0xFFFF0000u);
      }
      const float* gp = dP + r * ld_dp + c0;
      const float4 g0 = __ldg(reinterpret_cast<const float4*>(gp));
      float4 g1 = make_float4(0.f, 0.f, 0.f, 0.f);
      if (c0 + 4 < ld_dp) g1 = __ldg(reinterpret_cast<const float4*>(gp) + 1);
      g[0] = g0.x; g[1] = g0.y; g[2] = g0.z; g[3] = g0.w; g[4] = g1.x; g[5] = g1.y; g[6] = g1.z; g[7] = g1.w;
    }
    float dot = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      g[j] = (c0 + j < cols && pv[j] != 0.f) ? g[j] : 0.f;      // (a masked column's dP is whatever the padded GEMM produced)
      pv[j] = (c0 + j < cols) ? pv[j] : 0.f;
      dot = fmaf(pv[j], g[j], dot);
    }
    dot = warp_sum(dot);
    if (c0 < ldp) {
      uint4 oh, ol;
      uint32_t* ohp = &oh.x;
      uint32_t* olp = &ol.x;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float a = scale * pv[2 * q] * (g[2 * q] - dot), b = scale * pv[2 * q + 1] * (g[2 * q + 1] - dot);
        ohp[q] = pack_bf16(a, b);
        olp[q] = pack_bf16(a - __uint_as_float(ohp[q] << 16), b - __uint_as_float(ohp[q] & 0xFFFF0000u));
      }
      *reinterpret_cast<uint4*>(hi + r * ldp + c0) = oh;
      if (lo) *reinterpret_cast<uint4*>(lo + r * ldp + c0) = ol;
    }
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = [] {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess)
      ptr = nullptr;
    return reinterpret_cast<EncodeTiledFn>(ptr);
  }();
  return fn;
}

// bf16 [batch][rows][inner contiguous], row pitch ld, batch pitch bstride (elements); box {64, box_rows, 1}, SWIZZLE_128B
static int make_map(CUtensorMap* m, const void* base, long long inner, long long rows, long long ld, int box_rows, long long batch,
                    long long bstride) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) {
    set_error("attn_fused: cuTensorMapEncodeTiled is not available");
    return DOST_ERR_UNSUPPORTED;
  }
  if (batch <= 1 || bstride <= 0) {
    batch = 1;
    bstride = rows * ld;
  }
  cuuint64_t dims[3] = {(cuuint64_t)inner, (cuuint64_t)rows, (cuuint64_t)batch};
  cuuint64_t strides[2] = {(cuuint64_t)ld * 2, (cuuint64_t)bstride * 2};
  cuuint32_t box[3] = {64u, (cuuint32_t)box_rows, 1u};
  cuuint32_t estr[3] = {1u, 1u, 1u};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("attn_fused: cuTensorMapEncodeTiled failed (%d) base=%p inner=%lld rows=%lld ld=%lld box_rows=%d", (int)r, base, inner, rows,
              ld, box_rows);
    return DOST_ERR_ARG;
  }
  return DOST_OK;
}

template <int NSPLIT>
static int launch(const Maps& maps, const Params& p, cudaStream_t st) {
  auto kern = attn_fwd_kernel<NSPLIT>;
  static PerDevice cfg_once;
  if (bool* flag = cfg_once.pending()) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
    if (e != cudaSuccess) {
      set_error("attn_fused: cudaFuncSetAttribute failed: %s", cudaGetErrorString(e));
      return DOST_ERR_LAUNCH;
    }
    *flag = true;
  }
  const int sms = sm_count();
  const int grid = p.total_tiles < sms ? p.total_tiles : sms;
  kern<<<grid, kThreads, kSmemBytes, st>>>(maps, p);
  return check_launch("attn_fused_fwd");
}

}  // namespace fa
}  // namespace dost

using namespace dost;

extern "C" int dost_attn_fused_supported(int Lq, int H, int max_keys) {
  return (Lq >= 1 && H >= 64 && H <= 256 && H % 64 == 0 && max_keys >= 1 && max_keys <= fa::kMaxKeys) ? 1 : 0;
}

extern "C" int dost_attn_fused_fwd_dseed(const void* q_hi, const void* q_lo, long long ld_q, const void* k_hi, const void* k_lo,
                                         long long ld_k, long long k_rows, int S, int Lq, int Lk, int H, const int32_t* k_rowoff,
                                         const int32_t* k_count, const int32_t* nmax, int max_keys, double scale,
                                         const float* residual, long long res_seq_stride, float* out, void* p_hi, void* p_lo,
                                         long long ld_p, int precision, double drop_p,
                                         unsigned long long seed, const unsigned long long* seed_offset, float* lse,
                                         dost_stream_t stream) {
  DOST_REQUIRE(q_hi && k_hi && out && S > 0 && Lq > 0, "attn_fused_fwd: null pointer / empty problem");
  DOST_REQUIRE(precision == DOST_PREC_BF16X3 || precision == DOST_PREC_BF16, "attn_fused_fwd: precision must be bf16x3 or bf16");
  const bool split3 = precision == DOST_PREC_BF16X3;
  DOST_REQUIRE(!split3 || (q_lo && k_lo), "attn_fused_fwd: bf16x3 needs the lo planes");
  DOST_REQUIRE(H >= 64 && H <= 256 && H % 64 == 0, "attn_fused_fwd: H must be 64, 128, 192 or 256 (got %d)", H);
  DOST_REQUIRE(ld_q >= H && ld_q % 8 == 0 && ld_k >= H && ld_k % 8 == 0, "attn_fused_fwd: plane pitches must be >= H and multiples of 8");
  const bool ragged = k_rowoff != nullptr;
  DOST_REQUIRE(!ragged || (k_count && k_rows > 0), "attn_fused_fwd: ragged keys need k_count and the number of stored rows");
  DOST_REQUIRE(ragged || Lk > 0, "attn_fused_fwd: dense keys need Lk");
  if (!ragged) max_keys = Lk;
  DOST_REQUIRE(max_keys >= 1 && max_keys <= fa::kMaxKeys, "attn_fused_fwd: at most %d keys per sequence (got %d)", fa::kMaxKeys, max_keys);
  DOST_REQUIRE(((uintptr_t)q_hi & 15) == 0 && ((uintptr_t)q_lo & 15) == 0 && ((uintptr_t)k_hi & 15) == 0 && ((uintptr_t)k_lo & 15) == 0 &&
                   ((uintptr_t)out & 15) == 0 && ((uintptr_t)residual & 15) == 0 && res_seq_stride % 4 == 0,
               "attn_fused_fwd: 16-byte alignment");
  fa::Maps maps;
  fa::Params p;
  p.S = S; p.Lq = Lq; p.Lk = Lk; p.H = H;
  p.QT = (Lq + fa::BM - 1) / fa::BM;
  const long long total = (long long)S * p.QT;
  DOST_REQUIRE(total <= 0x7fffffffLL, "attn_fused_fwd: too many tiles");
  p.total_tiles = (int)total;
  p.kpad = (max_keys + fa::KC - 1) / fa::KC * fa::KC;
  p.k_rowoff = k_rowoff; p.k_count = k_count; p.nmax = ragged ? nmax : nullptr;
  p.scale_log2e = (float)(scale * 1.4426950408889634);
  p.residual = residual; p.res_seq_stride = res_seq_stride;
  p.out = out;
  p.store_p = p_hi ? 1 : 0;
  p.errw = device_error_words();
  DOST_REQUIRE(drop_p >= 0.0 && drop_p < 1.0, "attn_fused_fwd: drop_p must be in [0, 1)");
  DOST_REQUIRE(!(drop_p > 0.0 && ragged && !nmax), "attn_fused_fwd: ragged dropout needs the device padding length");
  p.thresh = drop_p > 0.0 ? drop_threshold(drop_p) : 0u;
  p.inv_keep = (float)(1.0 / (1.0 - drop_p));
  p.seed = seed;
  p.seed_offset = seed_offset;
  p.lse = lse;
  int rc = fa::make_map(&maps.q_hi, q_hi, H, Lq, ld_q, fa::BM, S, (long long)Lq * ld_q);
  if (rc == DOST_OK && split3) rc = fa::make_map(&maps.q_lo, q_lo, H, Lq, ld_q, fa::BM, S, (long long)Lq * ld_q);
  auto kmap = [&](CUtensorMap* m, const void* base, int box_rows) {
    return ragged ? fa::make_map(m, base, H, k_rows, ld_k, box_rows, 1, 0) : fa::make_map(m, base, H, Lk, ld_k, box_rows, S, (long long)Lk * ld_k);
  };
  if (rc == DOST_OK) rc = kmap(&maps.k_hi, k_hi, fa::KC);
  if (rc == DOST_OK && split3) rc = kmap(&maps.k_lo, k_lo, fa::KC);
  // phase A boxes: {64 columns, 32 / 64 / 128 / 256 keys}; a work item takes the smallest one that covers its keys
  const int nbi_max = max_keys <= 32 ? 0 : (max_keys <= 64 ? 1 : (max_keys <= 128 ? 2 : 3));
  for (int i = 0; i < 4 && rc == DOST_OK; ++i) {
    if (i <= nbi_max) {
      rc = kmap(&maps.ka_hi[i], k_hi, 32 << i);
      if (rc == DOST_OK && split3) rc = kmap(&maps.ka_lo[i], k_lo, 32 << i);
    } else {
      maps.ka_hi[i] = maps.ka_hi[0];
      if (split3) maps.ka_lo[i] = maps.ka_lo[0];
    }
  }
  if (rc != DOST_OK) return rc;
  if (!split3) {
    maps.q_lo = maps.q_hi;
    maps.k_lo = maps.k_hi;
    for (int i = 0; i < 4; ++i) maps.ka_lo[i] = maps.ka_hi[i];
  }
  maps.p_hi = maps.q_hi;
  maps.p_lo = maps.q_hi;
  if (p.store_p) {
    DOST_REQUIRE(!split3 || p_lo, "attn_fused_fwd: bf16x3 needs p_lo");
    const int pcov = (p.kpad + 63) / 64 * 64;      // columns the kernel writes (whole 64-key blocks of the P tile)
    DOST_REQUIRE(ld_p % 8 == 0 && ld_p >= max_keys && ld_p <= pcov && ((uintptr_t)p_hi & 15) == 0 && ((uintptr_t)p_lo & 15) == 0,
                 "attn_fused_fwd: probability planes need max_keys <= ld_p <= %d, ld_p %% 8 == 0 (got %lld)", pcov, ld_p);
    rc = fa::make_map(&maps.p_hi, p_hi, ld_p, Lq, ld_p, fa::BM, S, (long long)Lq * ld_p);
    if (rc == DOST_OK && split3) rc = fa::make_map(&maps.p_lo, p_lo, ld_p, Lq, ld_p, fa::BM, S, (long long)Lq * ld_p);
    if (rc != DOST_OK) return rc;
    if (!split3) maps.p_lo = maps.p_hi;
  }
  cudaStream_t st = (cudaStream_t)stream;
  return split3 ? fa::launch<3>(maps, p, st) : fa::launch<1>(maps, p, st);
}

extern "C" int dost_attn_fused_fwd(const void* q_hi, const void* q_lo, long long ld_q, const void* k_hi, const void* k_lo, long long ld_k,
                                   long long k_rows, int S, int Lq, int Lk, int H, const int32_t* k_rowoff, const int32_t* k_count,
                                   const int32_t* nmax, int max_keys, double scale, const float* residual, long long res_seq_stride,
                                   float* out, void* p_hi, void* p_lo, long long ld_p, int precision, double drop_p,
                                   unsigned long long seed, float* lse, dost_stream_t stream) {
  return dost_attn_fused_fwd_dseed(q_hi, q_lo, ld_q, k_hi, k_lo, ld_k, k_rows, S, Lq, Lk, H, k_rowoff, k_count, nmax, max_keys, scale,
                                   residual, res_seq_stride, out, p_hi, p_lo, ld_p, precision, drop_p, seed, nullptr, lse, stream);
}

extern "C" int dost_softmax_bwd_from_planes(const void* p_hi, const void* p_lo, long long ld_pp, const float* dP, long long ld_dp,
                                            long long rows, int cols, double scale, void* hi, void* lo, long long ldp,
                                            dost_stream_t stream) {
  DOST_REQUIRE(p_hi && dP && hi && rows > 0 && cols > 0 && ld_pp >= cols && ld_dp >= cols && ldp >= cols, "softmax_bwd_from_planes: bad args");
  DOST_REQUIRE(ldp <= 256 && ld_pp % 8 == 0 && ldp % 8 == 0 && ld_dp % 4 == 0 && ((uintptr_t)p_hi & 15) == 0 && ((uintptr_t)p_lo & 15) == 0 &&
                   ((uintptr_t)dP & 15) == 0 && ((uintptr_t)hi & 15) == 0 && ((uintptr_t)lo & 15) == 0,
               "softmax_bwd_from_planes: at most 256 columns, pitches %% 8 (planes) / %% 4 (dP), 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  const int blocks = (int)min64((rows + 7) / 8, 32LL * kNumSMs);
  fa::ds_from_planes_kernel<<<blocks, 256, 0, st>>>((const __nv_bfloat16*)p_hi, (const __nv_bfloat16*)p_lo, ld_pp, dP, ld_dp, rows, cols,
                                                    (float)scale, (__nv_bfloat16*)hi, (__nv_bfloat16*)lo, ldp);
  return check_launch("softmax_bwd_from_planes");
}

#ifdef DOST_ATTN_TIMELINE
extern "C" int dost_attn_fused_timeline(unsigned long long* host, int n) {
  return cudaMemcpyFromSymbol(host, dost::fa::g_timeline, sizeof(unsigned long long) * (n < 64 * 16 ? n : 64 * 16)) == cudaSuccess ? 0 : 1;
}
#endif
