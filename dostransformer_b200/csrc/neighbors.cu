// Periodic neighbour lists and the eDOS bond features on the device (SURVEY.md section 8f rank 4).
//
// Replaces the offline CPU graph construction of the reference:
//   * phonon: ase.neighbor_list("ijS", cutoff=r_max, self_interaction=True) and the edge vectors
//     pos[dst] - pos[src] + shift @ lattice (utils.py:267-273);
//   * eDOS:   pymatgen Structure.get_all_neighbors(radius=8) sorted by distance, first 12 kept, short lists padded with
//     index 0 / distance radius + 1, Gaussian distance expansion exp(-(d - mu)^2 / 0.2^2), mu = 0, 0.2, ..., 8.0
//     (data/mat2graph.py:162-179, 185, 212-243).
// ASE and pymatgen are not part of the reference tree (and are unpinned), so the ORDER of the list is this library's own
// canonical one, stated here and followed by oracle/neighbors_oracle.py: edges sorted by (centre atom i, neighbour atom j,
// shift Sx, Sy, Sz); k-nearest selection is stable with respect to that order.
//
// Arithmetic contract (fp64, every operation individually rounded - no FMA contraction - so that the CPU oracle reproduces
// the bits):  s_c = (Sx*L[0][c] + Sy*L[1][c]) + Sz*L[2][c];  v_c = (pos[j][c] - pos[i][c]) + s_c;
// d = sqrt((v_0*v_0 + v_1*v_1) + v_2*v_2);  an image is a neighbour iff d < cutoff, the pair (i, i, S = 0) only with
// self_interaction.  The image ranges searched per pair are a superset derived from the fractional offset and the lattice
// plane spacings, so they do not influence the result.
//
// One warp per centre atom; candidates (j, S) are visited in canonical order 32 at a time and compacted with a ballot, so
// the list comes out sorted without a sort.  Two passes (count, exclusive scan by the caller, fill).
#include "common.cuh"

namespace dost {
namespace {

struct Cell {
  double L[9];      // rows = lattice vectors
  double Li[9];     // inverse (columns give fractional coordinates: f = v * Li)
  double inv_h[3];  // 1 / spacing of the lattice planes normal to direction k
};

__device__ __forceinline__ void make_cell(const double* __restrict__ lat, Cell& c) {
#pragma unroll
  for (int k = 0; k < 9; ++k) c.L[k] = lat[k];
  const double* a = c.L;
  const double* b = c.L + 3;
  const double* cc = c.L + 6;
  const double bxc[3] = {b[1] * cc[2] - b[2] * cc[1], b[2] * cc[0] - b[0] * cc[2], b[0] * cc[1] - b[1] * cc[0]};
  const double cxa[3] = {cc[1] * a[2] - cc[2] * a[1], cc[2] * a[0] - cc[0] * a[2], cc[0] * a[1] - cc[1] * a[0]};
  const double axb[3] = {a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]};
  const double vol = a[0] * bxc[0] + a[1] * bxc[1] + a[2] * bxc[2];
  const double iv = 1.0 / vol;
  // inverse of the row-vector matrix: columns are (b x c, c x a, a x b) / vol
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    c.Li[r * 3 + 0] = bxc[r] * iv;
    c.Li[r * 3 + 1] = cxa[r] * iv;
    c.Li[r * 3 + 2] = axb[r] * iv;
  }
  c.inv_h[0] = sqrt(bxc[0] * bxc[0] + bxc[1] * bxc[1] + bxc[2] * bxc[2]) * fabs(iv);
  c.inv_h[1] = sqrt(cxa[0] * cxa[0] + cxa[1] * cxa[1] + cxa[2] * cxa[2]) * fabs(iv);
  c.inv_h[2] = sqrt(axb[0] * axb[0] + axb[1] * axb[1] + axb[2] * axb[2]) * fabs(iv);
}

// The contract arithmetic: every operation rounded on its own.
__device__ __forceinline__ double image_dist(const double* __restrict__ L, const double dp[3], int sx, int sy, int sz,
                                             double v[3]) {
  const double fx = (double)sx, fy = (double)sy, fz = (double)sz;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const double s = __dadd_rn(__dadd_rn(__dmul_rn(fx, L[c]), __dmul_rn(fy, L[3 + c])), __dmul_rn(fz, L[6 + c]));
    v[c] = __dadd_rn(dp[c], s);
  }
  const double d2 = __dadd_rn(__dadd_rn(__dmul_rn(v[0], v[0]), __dmul_rn(v[1], v[1])), __dmul_rn(v[2], v[2]));
  return __dsqrt_rn(d2);
}

// FILL = false: count[i];  FILL = true: write the edges of atom i at edge_ptr[i]..
template <bool FILL>
__global__ void __launch_bounds__(128) neighbor_kernel(const double* __restrict__ lattice, const double* __restrict__ pos,
                                                       const long long* __restrict__ node_ptr,
                                                       const long long* __restrict__ crystal_of, long long N, double cutoff,
                                                       int self_interaction, long long* __restrict__ count,
                                                       const long long* __restrict__ edge_ptr,
                                                       long long* __restrict__ edge_src, long long* __restrict__ edge_dst,
                                                       long long* __restrict__ edge_shift, double* __restrict__ edge_vec,
                                                       double* __restrict__ edge_len, int local_ids) {
  const int lane = threadIdx.x & 31;
  const long long i = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (i >= N) return;
  const long long c = crystal_of[i];
  const long long n0 = node_ptr[c], n1 = node_ptr[c + 1];
  Cell cell;
  make_cell(lattice + 9 * c, cell);
  const double pi[3] = {pos[3 * i], pos[3 * i + 1], pos[3 * i + 2]};
  long long total = 0;
  long long base = FILL ? edge_ptr[i] : 0;
  for (long long j = n0; j < n1; ++j) {
    double dp[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) dp[k] = __dsub_rn(pos[3 * j + k], pi[k]);
    // fractional offset of the pair and the image range that can come within the cutoff (superset, with slack)
    int lo[3], cnt[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const double f = dp[0] * cell.Li[0 * 3 + k] + dp[1] * cell.Li[1 * 3 + k] + dp[2] * cell.Li[2 * 3 + k];
      const double w = cutoff * cell.inv_h[k] + 1e-6;
      lo[k] = (int)floor(-f - w);
      const int hi = (int)ceil(-f + w);
      cnt[k] = hi - lo[k] + 1;
    }
    const int ncand = cnt[0] * cnt[1] * cnt[2];
    for (int q0 = 0; q0 < ncand; q0 += 32) {
      const int q = q0 + lane;
      bool ok = false;
      int sx = 0, sy = 0, sz = 0;
      double v[3] = {0.0, 0.0, 0.0}, d = 0.0;
      if (q < ncand) {
        sz = lo[2] + q % cnt[2];
        const int r = q / cnt[2];
        sy = lo[1] + r % cnt[1];
        sx = lo[0] + r / cnt[1];
        d = image_dist(cell.L, dp, sx, sy, sz, v);
        ok = d < cutoff && (self_interaction || j != i || sx != 0 || sy != 0 || sz != 0);
      }
      const unsigned m = __ballot_sync(0xffffffffu, ok);
      if (FILL && ok) {
        const long long e = base + total + __popc(m & ((1u << lane) - 1u));
        edge_src[e] = local_ids ? i - n0 : i;
        edge_dst[e] = local_ids ? j - n0 : j;
        if (edge_shift) {
          edge_shift[3 * e] = sx;
          edge_shift[3 * e + 1] = sy;
          edge_shift[3 * e + 2] = sz;
        }
        if (edge_vec) {
          edge_vec[3 * e] = v[0];
          edge_vec[3 * e + 1] = v[1];
          edge_vec[3 * e + 2] = v[2];
        }
        if (edge_len) edge_len[e] = d;
      }
      total += __popc(m);
    }
  }
  if (!FILL && lane == 0) count[i] = total;
}

// k smallest distances of every atom's (sorted-by-(j,S)) list, ties resolved by list position; one warp per atom.
// out_idx [N,k] = neighbour atom (as stored in edge_dst), out_dist [N,k]; short lists padded with (pad_idx, pad_dist).
__global__ void __launch_bounds__(128) knn_select_kernel(const long long* __restrict__ edge_ptr,
                                                         const long long* __restrict__ edge_dst,
                                                         const double* __restrict__ edge_len, long long N, int k,
                                                         long long pad_idx, double pad_dist, long long* __restrict__ out_idx,
                                                         double* __restrict__ out_dist, long long* __restrict__ out_edge) {
  const int lane = threadIdx.x & 31;
  const long long i = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (i >= N) return;
  const long long e0 = edge_ptr[i], e1 = edge_ptr[i + 1];
  double last_d = -1.0;
  long long last_e = -1;      // the previous pick: the next one is the smallest (d, e) strictly after it
  for (int r = 0; r < k; ++r) {
    double bd = 0.0;
    long long be = -1;
    for (long long e = e0 + lane; e < e1; e += 32) {
      const double d = edge_len[e];
      const bool after = d > last_d || (d == last_d && e > last_e);
      if (after && (be < 0 || d < bd)) {      // within a lane e ascends, so the first minimum wins ties
        bd = d;
        be = e;
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double od = __shfl_xor_sync(0xffffffffu, bd, o);
      const long long oe = __shfl_xor_sync(0xffffffffu, be, o);
      if (oe >= 0 && (be < 0 || od < bd || (od == bd && oe < be))) {
        bd = od;
        be = oe;
      }
    }
    if (lane == 0) {
      out_idx[i * k + r] = be >= 0 ? edge_dst[be] : pad_idx;
      out_dist[i * k + r] = be >= 0 ? bd : pad_dist;
      if (out_edge) out_edge[i * k + r] = be;
    }
    if (be < 0) {            // list exhausted: pad the rest
      if (lane == 0)
        for (int r2 = r + 1; r2 < k; ++r2) {
          out_idx[i * k + r2] = pad_idx;
          out_dist[i * k + r2] = pad_dist;
          if (out_edge) out_edge[i * k + r2] = -1;
        }
      break;
    }
    last_d = bd;
    last_e = be;
  }
}

// GaussianDistance.expand (mat2graph.py:162-179): out[e, f] = float(exp(-(d_e - mu_f)^2 / var^2)), mu_f = dmin + f * step.
__global__ void gaussian_expand_kernel(const double* __restrict__ dist, long long n, double dmin, double step, int nfilt,
                                       double var2, float* __restrict__ out) {
  const long long total = n * nfilt;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const long long e = t / nfilt;
    const int f = (int)(t - e * nfilt);
    const double mu = __dadd_rn(dmin, __dmul_rn((double)f, step));
    const double u = __dsub_rn(dist[e], mu);
    const double q = __ddiv_rn(-__dmul_rn(u, u), var2);
    out[t] = (float)exp(q);
  }
}

// Its distance gradient: d_dist[e] = sum_f d_out[e, f] phi_f (-2 (d_e - mu_f) / var^2), phi_f recomputed in fp64 with mu_f
// formed as above (the fp32 cast of the forward differentiates as the identity, like torch's .float()).  One warp per
// distance, lanes over the filters, a fixed butterfly for the sum (bitwise reproducible).
__global__ void __launch_bounds__(256) gaussian_expand_bwd_kernel(const float* __restrict__ d_out, const double* __restrict__ dist,
                                                                  long long n, double dmin, double step, int nfilt, double var2,
                                                                  double* __restrict__ d_dist) {
  const int lane = threadIdx.x & 31;
  const long long e = blockIdx.x * 8LL + (threadIdx.x >> 5);
  if (e >= n) return;
  const double d = dist[e];
  double acc = 0.0;
  for (int f = lane; f < nfilt; f += 32) {
    const double mu = __dadd_rn(dmin, __dmul_rn((double)f, step));
    const double u = __dsub_rn(d, mu);
    const double phi = exp(__ddiv_rn(-__dmul_rn(u, u), var2));
    acc += (double)d_out[e * nfilt + f] * phi * (-2.0 * u / var2);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) d_dist[e] = acc;
}

// The geometry of a fixed list: v = (pos[dst] - pos[src]) + s and |v| through image_dist, the operations neighbor_kernel
// performs, so at the geometry the list was built at the results are its bits.  dst < 0 marks a padded slot: len = pad, v = 0.
__global__ void edge_geometry_kernel(const double* __restrict__ lattice, const double* __restrict__ pos,
                                     const long long* __restrict__ crystal_of, const long long* __restrict__ src,
                                     const long long* __restrict__ dst, const long long* __restrict__ shift, long long n,
                                     double pad, double* __restrict__ edge_vec, double* __restrict__ edge_len) {
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
    const long long j = dst[e];
    double v[3] = {0.0, 0.0, 0.0}, d = pad;
    if (j >= 0) {
      const long long i = src[e];
      double dp[3];
#pragma unroll
      for (int k = 0; k < 3; ++k) dp[k] = __dsub_rn(pos[3 * j + k], pos[3 * i + k]);
      d = image_dist(lattice + 9 * crystal_of[i], dp, (int)shift[3 * e], (int)shift[3 * e + 1], (int)shift[3 * e + 2], v);
    }
    if (edge_vec) {
      edge_vec[3 * e] = v[0];
      edge_vec[3 * e + 1] = v[1];
      edge_vec[3 * e + 2] = v[2];
    }
    if (edge_len) edge_len[e] = d;
  }
}

// Membership of a candidate list at the current geometry: mask[e] = (len[e] < cutoff), the comparison neighbor_kernel
// applies to the same image_dist bits (written by edge_geometry_kernel), so the live entries are exactly the list a fresh
// search at cutoff finds whenever the candidates contain it.  A NaN length is not within.
__global__ void edge_within_kernel(const double* __restrict__ edge_len, long long n, double cutoff,
                                   unsigned char* __restrict__ mask) {
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x)
    mask[e] = edge_len[e] < cutoff ? 1 : 0;
}

// g_e = d_vec_e + d_len_e v_e / |v_e| (v / |v| := 0 at |v| = 0), 0 on identity edges (i, i, 0) and padded slots; with the
// lattice columns g[e, 3 + 3a + b] = S_a g_b.  The operations of the torch expression in neighbors._edge_grad, one by one.
__global__ void edge_geometry_bwd_kernel(const double* __restrict__ d_vec, const double* __restrict__ d_len,
                                         const double* __restrict__ edge_vec, const double* __restrict__ edge_len,
                                         const long long* __restrict__ src, const long long* __restrict__ dst,
                                         const long long* __restrict__ shift, long long n, int with_lattice,
                                         double* __restrict__ g) {
  const int ld = with_lattice ? 12 : 3;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
    const long long j = dst[e];
    const long long s[3] = {shift[3 * e], shift[3 * e + 1], shift[3 * e + 2]};
    const bool drop = j < 0 || (j == src[e] && s[0] == 0 && s[1] == 0 && s[2] == 0);
    double gv[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      double t = d_vec ? d_vec[3 * e + c] : 0.0;
      if (d_len) {
        const double l = edge_len[e];
        const double u = l > 0.0 ? __ddiv_rn(edge_vec[3 * e + c], l) : 0.0;
        t = __dadd_rn(t, __dmul_rn(d_len[e], u));
      }
      gv[c] = drop ? 0.0 : t;
      g[e * ld + c] = gv[c];
    }
    if (with_lattice) {
#pragma unroll
      for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int b = 0; b < 3; ++b) g[e * ld + 3 + 3 * a + b] = __dmul_rn((double)s[a], gv[b]);
    }
  }
}

// The re-pick of a skin topology: atom i's candidates (every image within cutoff + skin at the build geometry, canonical
// order, rows cand_ptr[i]..cand_ptr[i+1]) get their distance at the current geometry through image_dist (written to
// cand_len, and the vector to cand_vec when given), then the k nearest with d < cutoff are selected exactly as
// knn_select_kernel selects from a list: smallest (d, candidate id) first.  Filtering the candidates at d < cutoff leaves
// the list a fresh search at this geometry finds, in the same order and with the same bits, whenever the candidates
// contain every pair within the cutoff (dost_topology_check tells when they may not).  One warp per atom.
__global__ void __launch_bounds__(128) knn_reselect_kernel(
    const double* __restrict__ lattice, const double* __restrict__ pos, const long long* __restrict__ node_ptr,
    const long long* __restrict__ crystal_of, const int* __restrict__ cand_ptr, const long long* __restrict__ cand_dst,
    const long long* __restrict__ cand_shift, long long N, int k, double cutoff, double pad_dist,
    double* __restrict__ cand_len, double* __restrict__ cand_vec, long long* __restrict__ out_pick,
    double* __restrict__ out_dist, long long* __restrict__ out_nbr, long long* __restrict__ out_shift,
    long long* __restrict__ out_edge_index) {
  const int lane = threadIdx.x & 31;
  const long long i = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (i >= N) return;
  const long long c = crystal_of[i];
  const double* L = lattice + 9 * c;
  const long long e0 = cand_ptr[i], e1 = cand_ptr[i + 1];
  for (long long e = e0 + lane; e < e1; e += 32) {
    const long long j = cand_dst[e];
    double dp[3], v[3];
#pragma unroll
    for (int q = 0; q < 3; ++q) dp[q] = __dsub_rn(pos[3 * j + q], pos[3 * i + q]);
    cand_len[e] = image_dist(L, dp, (int)cand_shift[3 * e], (int)cand_shift[3 * e + 1], (int)cand_shift[3 * e + 2], v);
    if (cand_vec) {
      cand_vec[3 * e] = v[0];
      cand_vec[3 * e + 1] = v[1];
      cand_vec[3 * e + 2] = v[2];
    }
  }
  __syncwarp();             // the distances of the whole segment are visible to every lane
  double last_d = -1.0;
  long long last_e = -1;
  bool done = false;
  for (int r = 0; r < k; ++r) {
    double bd = 0.0;
    long long be = -1;
    if (!done) {
      for (long long e = e0 + lane; e < e1; e += 32) {
        const double d = cand_len[e];
        if (!(d < cutoff)) continue;
        const bool after = d > last_d || (d == last_d && e > last_e);
        if (after && (be < 0 || d < bd)) {
          bd = d;
          be = e;
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const double od = __shfl_xor_sync(0xffffffffu, bd, o);
        const long long oe = __shfl_xor_sync(0xffffffffu, be, o);
        if (oe >= 0 && (be < 0 || od < bd || (od == bd && oe < be))) {
          bd = od;
          be = oe;
        }
      }
    }
    if (lane == 0) {
      const long long s = i * k + r;
      out_pick[s] = be;
      out_dist[s] = be >= 0 ? bd : pad_dist;
      const long long j = be >= 0 ? cand_dst[be] : -1;
      if (out_nbr) out_nbr[s] = j;
      if (out_shift)
#pragma unroll
        for (int q = 0; q < 3; ++q) out_shift[3 * s + q] = be >= 0 ? cand_shift[3 * be + q] : 0;
      if (out_edge_index) {      // the model's node ids: one prompt node per preceding crystal; padded slots -> atom 0
        out_edge_index[s] = i + c;
        out_edge_index[N * k + s] = (j >= 0 ? j : node_ptr[c]) + c;
      }
    }
    done = be < 0;          // list exhausted: the remaining slots are padded
    last_d = bd;
    last_e = be;
  }
}

// Completeness of a skin list, and (phonon) whether a held edge set is still the list at the current geometry.  Sets
// *flag = 1 (never clears it) when the result of the topology may differ from a fresh search.
//
// Per crystal, build cell L0 and positions p0, current cell L and positions p (unwrapped), fractional coordinates
// f = p L^-1, f0 = p0 L0^-1 (rows are vectors throughout).  A pair (i, j, S) has v = (f_j - f_i + S) L = u L now and
// v0 = (f0_j - f0_i + S) L0 = u0 L0 at the build.  With u - u0 = (f_j - f0_j) - (f_i - f0_i) and
// delta = max_i |(f_i - f0_i) L|:  |u0 L| <= |v| + 2 delta.  With eps = ||L0^-1 (L - L0)||_F (>= the spectral norm):
// u0 L = v0 + v0 L0^-1 (L - L0), so |u0 L| >= |v0| (1 - eps).  Hence, for eps < 1, every pair with |v| < r now had
// |v0| < (r + 2 delta) / (1 - eps) at the build, and the candidates (every image with |v0| < r + skin) contain every pair
// within r as long as (r + 2 delta) / (1 - eps) <= r + skin.  The flag is set when eps >= 1 or
// (r + 2 delta) / (1 - eps) * (1 + kSkinSlack) >= r + skin: the relative slack covers the rounding of eps, delta and the
// distances themselves (all fp64, errors ~1e-15 relative) with a wide margin; a NaN anywhere sets the flag.
//
// Phonon: cand_held[e] says whether candidate e is one of the held edges (d < cutoff at the build); the flag is also set
// when its status at the current geometry (image_dist, d < cutoff) differs.  Warps 0..C-1 test one crystal each (lanes
// over its atoms); every thread then walks the candidates grid-stride.
constexpr double kSkinSlack = 1e-9;

__global__ void __launch_bounds__(256) topology_check_kernel(
    const double* __restrict__ lattice, const double* __restrict__ pos, const double* __restrict__ lattice0,
    const double* __restrict__ pos0, const long long* __restrict__ node_ptr, long long C, double cutoff, double skin,
    const long long* __restrict__ crystal_of, const long long* __restrict__ cand_src,
    const long long* __restrict__ cand_dst, const long long* __restrict__ cand_shift,
    const unsigned char* __restrict__ cand_held, long long n_cand, int* __restrict__ flag) {
  const int lane = threadIdx.x & 31;
  const long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (w < C) {
    Cell cur, ref;
    make_cell(lattice + 9 * w, cur);
    make_cell(lattice0 + 9 * w, ref);
    double delta = 0.0;
    for (long long a = node_ptr[w] + lane; a < node_ptr[w + 1]; a += 32) {
      double df[3], m = 0.0;
#pragma unroll
      for (int q = 0; q < 3; ++q) {
        const double f = pos[3 * a] * cur.Li[q] + pos[3 * a + 1] * cur.Li[3 + q] + pos[3 * a + 2] * cur.Li[6 + q];
        const double f0 = pos0[3 * a] * ref.Li[q] + pos0[3 * a + 1] * ref.Li[3 + q] + pos0[3 * a + 2] * ref.Li[6 + q];
        df[q] = f - f0;
      }
#pragma unroll
      for (int q = 0; q < 3; ++q) {
        const double x = df[0] * cur.L[q] + df[1] * cur.L[3 + q] + df[2] * cur.L[6 + q];
        m += x * x;
      }
      m = sqrt(m);
      delta = (m > delta || m != m) ? m : delta;           // a NaN propagates
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double od = __shfl_xor_sync(0xffffffffu, delta, o);
      delta = (od > delta || od != od) ? od : delta;
    }
    if (lane == 0) {
      double eps2 = 0.0;       // ||L0^-1 (L - L0)||_F^2; L0^-1[a][m] = ref.Li[3a + m]
#pragma unroll
      for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int b = 0; b < 3; ++b) {
          double x = 0.0;
#pragma unroll
          for (int m = 0; m < 3; ++m) x += ref.Li[3 * a + m] * (cur.L[3 * m + b] - ref.L[3 * m + b]);
          eps2 += x * x;
        }
      const double eps = sqrt(eps2);
      const bool complete = eps < 1.0 && (cutoff + 2.0 * delta) / (1.0 - eps) * (1.0 + kSkinSlack) < cutoff + skin;
      if (!complete) *flag = 1;
    }
  }
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n_cand; e += (long long)gridDim.x * blockDim.x) {
    const long long i = cand_src[e], j = cand_dst[e];
    double dp[3], v[3];
#pragma unroll
    for (int q = 0; q < 3; ++q) dp[q] = __dsub_rn(pos[3 * j + q], pos[3 * i + q]);
    const double d = image_dist(lattice + 9 * crystal_of[i], dp, (int)cand_shift[3 * e], (int)cand_shift[3 * e + 1],
                                (int)cand_shift[3 * e + 2], v);
    if ((d < cutoff) != (cand_held[e] != 0)) *flag = 1;
  }
}

}  // namespace
}  // namespace dost

using namespace dost;

extern "C" int dost_neighbor_count(const double* lattice, const double* pos, const int64_t* node_ptr,
                                   const int64_t* crystal_of, long long N, double cutoff, int self_interaction,
                                   int64_t* count, dost_stream_t stream) {
  if (N == 0) return DOST_OK;
  DOST_REQUIRE(lattice && pos && node_ptr && crystal_of && count && N > 0 && cutoff > 0, "neighbor_count: bad args");
  neighbor_kernel<false><<<ceil_div(N, 4), 128, 0, (cudaStream_t)stream>>>(
      lattice, pos, (const long long*)node_ptr, (const long long*)crystal_of, N, cutoff, self_interaction,
      (long long*)count, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 0);
  return check_launch("neighbor_count");
}

extern "C" int dost_neighbor_fill(const double* lattice, const double* pos, const int64_t* node_ptr,
                                  const int64_t* crystal_of, long long N, double cutoff, int self_interaction,
                                  const int64_t* edge_ptr, int local_ids, int64_t* edge_src, int64_t* edge_dst,
                                  int64_t* edge_shift, double* edge_vec, double* edge_len, dost_stream_t stream) {
  if (N == 0) return DOST_OK;
  DOST_REQUIRE(lattice && pos && node_ptr && crystal_of && edge_ptr && edge_src && edge_dst && N > 0 && cutoff > 0,
               "neighbor_fill: bad args");
  neighbor_kernel<true><<<ceil_div(N, 4), 128, 0, (cudaStream_t)stream>>>(
      lattice, pos, (const long long*)node_ptr, (const long long*)crystal_of, N, cutoff, self_interaction, nullptr,
      (const long long*)edge_ptr, (long long*)edge_src, (long long*)edge_dst, (long long*)edge_shift, edge_vec, edge_len,
      local_ids);
  return check_launch("neighbor_fill");
}

extern "C" int dost_knn_select(const int64_t* edge_ptr, const int64_t* edge_dst, const double* edge_len, long long N, int k,
                               long long pad_idx, double pad_dist, int64_t* out_idx, double* out_dist, int64_t* out_edge,
                               dost_stream_t stream) {
  if (N == 0 || k == 0) return DOST_OK;
  DOST_REQUIRE(edge_ptr && edge_dst && edge_len && out_idx && out_dist && N > 0 && k > 0, "knn_select: bad args");
  knn_select_kernel<<<ceil_div(N, 4), 128, 0, (cudaStream_t)stream>>>(
      (const long long*)edge_ptr, (const long long*)edge_dst, edge_len, N, k, pad_idx, pad_dist, (long long*)out_idx,
      out_dist, (long long*)out_edge);
  return check_launch("knn_select");
}

extern "C" int dost_gaussian_expand(const double* dist, long long n, double dmin, double step, int nfilt, double var,
                                    float* out, dost_stream_t stream) {
  if (n == 0 || nfilt == 0) return DOST_OK;
  DOST_REQUIRE(dist && out && n > 0 && nfilt > 0 && step > 0 && var > 0, "gaussian_expand: bad args");
  const long long total = n * nfilt;
  const int blocks = (int)min64(ceil_div(total, 256), (long long)kNumSMs * 16);
  gaussian_expand_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(dist, n, dmin, step, nfilt, var * var, out);
  return check_launch("gaussian_expand");
}

extern "C" int dost_gaussian_expand_bwd(const float* d_out, const double* dist, long long n, double dmin, double step,
                                        int nfilt, double var, double* d_dist, dost_stream_t stream) {
  if (n == 0) return DOST_OK;
  DOST_REQUIRE(d_out && dist && d_dist && n > 0 && nfilt > 0 && step > 0 && var > 0, "gaussian_expand_bwd: bad args");
  gaussian_expand_bwd_kernel<<<(unsigned)((n + 7) / 8), 256, 0, (cudaStream_t)stream>>>(d_out, dist, n, dmin, step, nfilt,
                                                                                         var * var, d_dist);
  return check_launch("gaussian_expand_bwd");
}

extern "C" int dost_edge_geometry(const double* lattice, const double* pos, const int64_t* crystal_of, const int64_t* src,
                                  const int64_t* dst, const int64_t* shift, long long n, double pad, double* edge_vec,
                                  double* edge_len, dost_stream_t stream) {
  if (n == 0) return DOST_OK;
  DOST_REQUIRE(lattice && pos && crystal_of && src && dst && shift && (edge_vec || edge_len) && n > 0,
               "edge_geometry: bad args");
  const int blocks = (int)min64(ceil_div(n, 256), (long long)kNumSMs * 16);
  edge_geometry_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(
      lattice, pos, (const long long*)crystal_of, (const long long*)src, (const long long*)dst, (const long long*)shift, n,
      pad, edge_vec, edge_len);
  return check_launch("edge_geometry");
}

extern "C" int dost_edge_geometry_bwd(const double* d_vec, const double* d_len, const double* edge_vec,
                                      const double* edge_len, const int64_t* src, const int64_t* dst, const int64_t* shift,
                                      long long n, int with_lattice, double* g, dost_stream_t stream) {
  if (n == 0) return DOST_OK;
  DOST_REQUIRE(src && dst && shift && g && n > 0 && (!d_len || (edge_vec && edge_len)), "edge_geometry_bwd: bad args");
  const int blocks = (int)min64(ceil_div(n, 256), (long long)kNumSMs * 16);
  edge_geometry_bwd_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(
      d_vec, d_len, edge_vec, edge_len, (const long long*)src, (const long long*)dst, (const long long*)shift, n,
      with_lattice, g);
  return check_launch("edge_geometry_bwd");
}

extern "C" int dost_edge_within(const double* edge_len, long long n, double cutoff, uint8_t* mask, dost_stream_t stream) {
  if (n == 0) return DOST_OK;
  DOST_REQUIRE(edge_len && mask && n > 0 && cutoff > 0, "edge_within: bad args");
  const int blocks = (int)min64(ceil_div(n, 256), (long long)kNumSMs * 16);
  edge_within_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(edge_len, n, cutoff, mask);
  return check_launch("edge_within");
}

extern "C" int dost_knn_reselect(const double* lattice, const double* pos, const int64_t* node_ptr,
                                 const int64_t* crystal_of, const int32_t* cand_ptr, const int64_t* cand_dst,
                                 const int64_t* cand_shift, long long N, int k, double cutoff, double pad_dist,
                                 double* cand_len, double* cand_vec, int64_t* out_pick, double* out_dist, int64_t* out_nbr,
                                 int64_t* out_shift, int64_t* out_edge_index, dost_stream_t stream) {
  if (N == 0 || k == 0) return DOST_OK;
  DOST_REQUIRE(lattice && pos && node_ptr && crystal_of && cand_ptr && cand_dst && cand_shift && cand_len && out_pick &&
                   out_dist && N > 0 && k > 0 && cutoff > 0,
               "knn_reselect: bad args");
  knn_reselect_kernel<<<ceil_div(N, 4), 128, 0, (cudaStream_t)stream>>>(
      lattice, pos, (const long long*)node_ptr, (const long long*)crystal_of, cand_ptr, (const long long*)cand_dst,
      (const long long*)cand_shift, N, k, cutoff, pad_dist, cand_len, cand_vec, (long long*)out_pick, out_dist,
      (long long*)out_nbr, (long long*)out_shift, (long long*)out_edge_index);
  return check_launch("knn_reselect");
}

extern "C" int dost_topology_check(const double* lattice, const double* pos, const double* lattice0, const double* pos0,
                                   const int64_t* node_ptr, long long C, double cutoff, double skin,
                                   const int64_t* crystal_of, const int64_t* cand_src, const int64_t* cand_dst,
                                   const int64_t* cand_shift, const uint8_t* cand_held, long long n_cand, int32_t* flag,
                                   dost_stream_t stream) {
  if (C == 0) return DOST_OK;
  DOST_REQUIRE(lattice && pos && lattice0 && pos0 && node_ptr && flag && C > 0 && cutoff > 0 && skin >= 0 && n_cand >= 0 &&
                   (n_cand == 0 || (crystal_of && cand_src && cand_dst && cand_shift && cand_held)),
               "topology_check: bad args");
  const long long per_crystal = ceil_div(C, 8), per_cand = min64(ceil_div(n_cand, 256), (long long)kNumSMs * 16);
  const int blocks = (int)(per_crystal > per_cand ? per_crystal : per_cand);
  topology_check_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(
      lattice, pos, lattice0, pos0, (const long long*)node_ptr, C, cutoff, skin, (const long long*)crystal_of,
      (const long long*)cand_src, (const long long*)cand_dst, (const long long*)cand_shift, cand_held, n_cand, flag);
  return check_launch("topology_check");
}
