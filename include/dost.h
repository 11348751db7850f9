/*
 * dost.h -- C ABI of libdost_b200.so: the sm_100a kernels behind the DOSTransformer hot path.
 *
 * The reference (HeewoongNoh/DOSTransformer) is pure Python: it has no FFI of its own.  Every device
 * op on its hot path is a library call into ATen/cuBLAS or one of three un-vendored packages
 * (SURVEY.md section 2.2, rows k1-k22).  This header is therefore the native surface the replacement
 * *creates*: each entry point names the reference call site(s) (file:line under /root/reference) it
 * takes over.  The host side (python, dostransformer_b200/) binds these with ctypes; INTEGRATION.md
 * shows the stub.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes only; no torch / pybind types.
 *   - every device buffer (inputs, outputs, workspace) is caller-owned; the library never allocates,
 *     frees or synchronises.  Work is ordered only by the `stream` argument (a cudaStream_t).
 *   - return value: 0 = ok, negative = DOST_ERR_*; dost_last_error() gives a thread-local message.
 *   - dtype: DOST_F32 (eDOS, reference default) or DOST_F64 (phonon: main_phDOS.py:15-16 sets float64).
 *   - index arrays are int32 (dost_cast_i64_i32 converts the int64 PyG tensors once per batch).
 *   - stateless and re-entrant; one host thread per GPU in data-parallel runs.
 *   - attention dropout seeds: every entry point that takes `unsigned long long seed` has a sibling
 *     dost_<name>_dseed whose argument list inserts `const unsigned long long* seed_offset` right after
 *     `seed`.  seed_offset is NULL or a device pointer to one word; the kernels then mask with
 *     seed + *seed_offset, reading the word when they run, not when they are enqueued.  A captured CUDA
 *     graph replays its launch arguments unchanged, so a host that rewrites the word on the stream before
 *     each replay draws a new dropout mask per replay.  NULL (and the plain entry point) is seed alone.
 */
#ifndef DOST_H_
#define DOST_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DOST_ABI_VERSION 15

enum { DOST_F32 = 0, DOST_F64 = 1 };
enum { DOST_OK = 0, DOST_ERR_ARG = -1, DOST_ERR_LAUNCH = -2, DOST_ERR_WORKSPACE = -3, DOST_ERR_UNSUPPORTED = -4 };
enum { DOST_ACT_NONE = 0, DOST_ACT_RELU = 1, DOST_ACT_LEAKY = 2, DOST_ACT_PRELU = 3 };
enum { DOST_PREC_FMA = 0, DOST_PREC_BF16X3 = 1 /* error-compensated, fp32 parity */, DOST_PREC_BF16 = 2 };
enum { DOST_KC = 0 /* reduction index contiguous */, DOST_MC = 1 /* row/col index contiguous */ };

typedef void* dost_stream_t; /* cudaStream_t */

int dost_abi_version(void);
const char* dost_last_error(void);
/* Number of kernels this library has launched in this process (bench.py's gpu_launches). */
long long dost_launch_count(void);
void dost_reset_launch_count(void);

/* Device-side input checks.  Kernels that meet invalid input they can skip (an index outside its table, a padding
 * length shorter than a crystal) skip it and raise a bit in one word of mapped host memory, so the host can poll it
 * WITHOUT a device synchronisation (a bit is visible once the kernel that raised it has completed).  The reference
 * raises IndexError at the same places (x[row] DOSTransformer.py:139-140, scatter index :187, promt_token[g.system]
 * :79).  dost_device_errors_init() allocates the word (call once per process before any CUDA-graph capture; returns
 * 0 or DOST_ERR_LAUNCH); dost_device_errors(clear) returns the bit mask and optionally clears it. */
enum { DOST_DEVERR_INDEX_RANGE = 1, DOST_DEVERR_NMAX_TOO_SMALL = 2 };
int dost_device_errors_init(void);
unsigned int dost_device_errors(int clear);

/* ---------------------------------------------------------------------------------------------
 * Integer graph structure (bit-exact work).  Replaces the index handling implied by
 * torch_scatter.scatter_sum/mean (DOSTransformer.py:187, DOSTransformer_phonon.py:209),
 * to_dense_batch (DOSTransformer.py:61) and len(batch.unique()) (DOSTransformer.py:118).
 * ------------------------------------------------------------------------------------------- */
int dost_cast_i64_i32(const int64_t* src, int32_t* dst, long long n, dost_stream_t stream);

/* Stable counting sort of element ids 0..n-1 by key[i] in [0,size):  rowptr[size+1], perm[n] with
 * perm == argsort(key, stable).  maxcount (optional, 1 int) receives max segment length.
 * workspace: dost_csr_workspace_bytes(n, size). */
size_t dost_csr_workspace_bytes(long long n, long long size);
int dost_csr_build(const int32_t* key, long long n, long long size, int32_t* rowptr, int32_t* perm,
                   int32_t* maxcount, void* workspace, size_t workspace_bytes, dost_stream_t stream);

/* *value = max(*value, floor_value) on the device (one int): the data-parallel padding length Nmax = max(this rank's
 * measured maximum, the sharder's global value) without a device->host read (to_dense_batch's max(), SURVEY 8e). */
int dost_imax_scalar(int32_t* value, int32_t floor_value, dost_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * GEMM family (fp32/fp64 FMA pipe, or tcgen05 tensor cores for fp32 data).  C[m,n] = epilogue( sum_k A(m,k) * B(n,k) ).
 * Replaces nn.Linear / torch.bmm / torch.cat / x[row] / .repeat on the path:
 * DOSTransformer.py:103-105,116-120 (encoders), :139-143,174-175 (gather+cat+edge_mlp), :188-190
 * (node_mlp_2), :65-69,79-83 (repeat+cat+fc/fc_prompt), :75,89 (out_layer), :158-159 (decoder);
 * layers/transformer.py:143-145 (fc1/fc2); layers/multihead_attention.py:68,72 (bmm) and the
 * autograd backward of each (main_eDOS.py:126).
 * ------------------------------------------------------------------------------------------- */
typedef struct {
  const void* base;   /* device pointer */
  long long ld;       /* leading dimension in elements */
  const int32_t* idx; /* optional row map: row(r) = idx[r / div]; NULL: row(r) = r / div */
  int div;            /* >= 1; T for per-crystal broadcast rows */
  int width;          /* columns this segment contributes to the reduction dim (KC, A side) */
} dost_seg_t;

typedef struct {
  int dtype;
  int M, N, K;
  int batch;                 /* >= 1: independent problems, strides below (no row maps when > 1) */
  /* A operand: mode KC: A(m,k) = seg_s.base[row_s(m) * ld_s + (k - kstart_s)], up to 3 segments
   * concatenated along k (segment widths must be multiples of 16 when nseg > 1).
   * mode MC: A(m,k) = seg0.base[k * ld + m] (single segment, no map). */
  int a_mode, a_nseg;
  dost_seg_t a[3];
  long long a_bstride;
  /* B operand: KC: B(n,k) = base[n*ld + k];  MC: B(n,k) = base[row(k)*ld + n] (row map on k allowed). */
  int b_mode;
  dost_seg_t b;
  long long b_bstride;
  /* epilogue: v = acc + bias[n]; out_pre = v; v = act(v); v *= dact(saved); v += residual; out (+)= v */
  const void* bias;
  int act;
  double act_slope;          /* LEAKY slope */
  const void* prelu_slope;   /* PRELU: device pointer to the single learnable slope */
  void* out_pre; long long ld_pre;
  const void* dact_saved; long long ld_dact; int dact_kind; double dact_slope; /* multiply by act'(saved) */
  const void* residual; long long ld_res;
  void* out; long long ldc; long long c_bstride;
  int accumulate;            /* out += v instead of out = v */
  int split_k;               /* >= 1; > 1 needs workspace of split_k*M*N elements, reduced in fixed order */
  int precision;             /* DOST_PREC_*: FMA pipe, or tcgen05 tensor cores with bf16x3 / bf16 operands (F32 only;
                                problems too small for a 128 x N tile stay on the FMA pipe) */
} dost_gemm_t;

size_t dost_gemm_workspace_bytes(const dost_gemm_t* g);
int dost_gemm(const dost_gemm_t* g, void* workspace, size_t workspace_bytes, dost_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * TMA-fed tcgen05 GEMM over bf16 operand planes: the tensor-core path of the Linear / MLP stacks
 * (same reference call sites as dost_gemm: nn.Linear in DOSTransformer.py:103-105,171,182,
 * layers/transformer.py:143-145 and their backward).  An operand is stored as two bf16 matrices,
 * hi = bf16(x) and lo = bf16(x - hi); precision DOST_PREC_BF16X3 accumulates hi*hi + hi*lo + lo*hi in
 * fp32 (fp32 parity), DOST_PREC_BF16 uses hi only (lo may be NULL).  Planes are written by
 * dost_split_planes, by the LayerNorm kernels and by this GEMM's own epilogue (out_hi / out_lo).
 *   KC: plane[r * ld + k]  (A: r = m, B: r = n)        MC: plane[k * ld + r]
 * epilogue: v = acc + bias[n] + rowbias[(m / rowbias_div) * ld_rowbias + n]; out_pre = v; v = act(v);
 *           v *= (dact_hi[m, n] > 0 ? 1 : dact_slope); v += residual; out (+)= v; out_hi/out_lo = split(v)
 * ------------------------------------------------------------------------------------------- */
typedef struct {
  const void* hi;    /* bf16 plane */
  const void* lo;    /* bf16 residual plane or NULL */
  long long ld;      /* leading dimension in elements, multiple of 8 */
  long long rows;    /* rows stored (B, KC: if 0 < rows < N the missing rows read as zero; 0 means N) */
  int width;         /* valid columns (A, KC: the k-range this segment contributes) */
} dost_planes_t;

typedef struct {
  int M, N, K;               /* N % 4 == 0 */
  int a_mode, a_nseg;        /* KC: up to 3 segments concatenated along k (widths % 64 == 0 when nseg > 1) */
  dost_planes_t a[3];
  int b_mode;
  dost_planes_t b;
  const float* bias;
  const float* rowbias; long long ld_rowbias; int rowbias_div;
  int act; float act_slope; const float* prelu_slope;
  float* out_pre; long long ld_pre;
  const void* dact_hi; long long ld_dact; float dact_slope;
  const float* residual; long long ld_res;
  float* out; long long ldc; int accumulate;      /* out may be NULL when only planes are wanted */
  void* out_hi; void* out_lo; long long ld_op;
  int split_k;               /* > 1: deterministic split-K (plain fp32 stores only) */
  int precision;             /* DOST_PREC_BF16X3 or DOST_PREC_BF16 */
  /* batch > 1: independent problems (torch.bmm of the energy self attention, multihead_attention.py:68,72); element
   * strides between consecutive problems of the A / B planes, of out and of residual.  Exclusive with split_k. */
  int batch;
  long long a_bstride, b_bstride, c_bstride, res_bstride;
  /* ragged batches (variable-length atom sets of the crystals; energy->atom cross attention, DOSTransformer.py:61-63):
   * b_rowoff[z]: B is ONE plane of b.rows rows and problem z uses rows b_rowoff[z] .. (rows past the problem's own are
   * whatever follows in the plane: the caller masks them).  c_rowoff[z], c_rowlim[z]: rows m < c_rowlim[z] of problem z
   * are written at row c_rowoff[z] + m of out.  All device int32 arrays of `batch` entries, or NULL. */
  const int32_t* b_rowoff;
  const int32_t* c_rowoff;
  const int32_t* c_rowlim;
  /* optional: colsum[n] = sum_m (stored value)[m, n] in a fixed order, computed by the epilogue that stores it (the bias
   * gradient when the stored value is the gradient of a Linear's output); workspace ceil(M/32)*N floats; no split_k/batch */
  float* colsum;
  /* optional 1-bit activation gates, [N / 32][ld_gate] 32-bit words (word-major, ld_gate >= M: the 32 rows of a warp are 32
   * consecutive words), bit j of word (w, m) <-> element (m, 32 w + j); N % 32 == 0; plain single problems on the TMA-store
   * epilogue only, else DOST_ERR_UNSUPPORTED.  out_gate: written by the epilogue, bit = (value after bias / row bias, before
   * the activation) > 0.  dact_gate: read instead of dact_hi: v *= bit ? 1 : dact_slope.  (ReLU of layers/transformer.py:143:
   * the backward then reads 1 bit instead of 16 per hidden activation.) */
  uint32_t* out_gate;
  const uint32_t* dact_gate;
  long long ld_gate;
} dost_gemm_bf16_t;

size_t dost_gemm_bf16_workspace_bytes(const dost_gemm_bf16_t* g);
int dost_gemm_bf16(const dost_gemm_bf16_t* g, void* workspace, size_t workspace_bytes, dost_stream_t stream);
/* The same conversion for `ntensors` matrices in one launch per 24 (host arrays of per-tensor pointers / sizes; the
 * descriptors travel in the kernel parameters).  Refreshes the operand planes of all Linear weights once per step
 * (nn.Linear.weight in DOSTransformer.py:103-105,171,182, layers/transformer.py:114-115); lo[i] may be NULL. */
int dost_split_planes_multi(int ntensors, const float* const* x, const long long* ld, const long long* rows, const int* cols,
                            void* const* hi, void* const* lo, const long long* ldp, dost_stream_t stream);
/* fp32 [rows, cols] (ld) -> bf16 planes [rows, ldp] (ldp % 8 == 0, columns >= cols zero-filled); lo may be NULL. */
int dost_split_planes(const float* x, long long ld, long long rows, int cols, void* hi, void* lo, long long ldp,
                      dost_stream_t stream);
/* Same, plus colsum[c] = sum_r x[r, c] in a fixed order (bias gradient of the Linear whose output gradient x is). */
size_t dost_split_planes_colsum_workspace_bytes(long long rows, int cols, long long ldp);
int dost_split_planes_colsum(const float* x, long long ld, long long rows, int cols, void* hi, void* lo, long long ldp,
                             float* colsum, void* workspace, size_t workspace_bytes, dost_stream_t stream);

/* fp32 row kernels of the tensor-core path (W in {128, 256, 512, 1024}): LayerNorm(+PReLU) whose output is written
 * directly as operand planes (and/or fp32), its backward (dx as fp32 and/or planes, optional residual gradient dres
 * added to dx, column sums of dx = bias gradient of the Linear feeding the LayerNorm), and column sums over planes.
 * Same reference call sites as dost_ln_fwd / dost_ln_bwd / dost_colsum. */
/* optional gather-add prologue (split-weight message passing, DOSTransformer.py:139-143,174):
 * x[r] += ga[ia[r] * ldg + :W] + gb[ib[r] * ldg + :W], written back to x before normalising. */
int dost_ln_fwd_planes(float* x, long long ldx, const float* ga, const int32_t* ia, const float* gb, const int32_t* ib,
                       long long ldg, const float* gamma, const float* beta, const float* prelu_slope, float* y,
                       void* hi, void* lo, long long ldp, float* stats, long long M, int W, dost_stream_t stream);
size_t dost_ln_bwd_planes_workspace_bytes(long long M, int W);
int dost_ln_bwd_planes(const float* dy, long long ld_dy, const float* x, long long ldx, const float* stats,
                       const float* gamma, const float* beta, const float* prelu_slope, const float* dres,
                       long long ld_dres, float* dx, void* dx_hi, void* dx_lo, long long ldp, float* dgamma,
                       float* dbeta, float* dslope, float* dxsum, long long M, int W, void* workspace,
                       size_t workspace_bytes, dost_stream_t stream);
/* Linear(H -> 1) (out_layer, DOSTransformer.py:42,75,89) as streaming kernels, K in {128, 256, 512}:
 * out[m] = x[m, :] . w + bias;  backward: dx[m, :] = dout[m] w (dx may be NULL), dwb[0..K) = sum_m dout[m] x[m, :], dwb[K] = sum_m dout[m]. */
int dost_rowdot_fwd(const float* x, long long ldx, const float* w, const float* bias, float* out, long long M, int K,
                    dost_stream_t stream);
size_t dost_rowdot_bwd_workspace_bytes(long long M, int K);
int dost_rowdot_bwd(const float* dout, const float* x, long long ldx, const float* w, float* dx, float* dwb, long long M, int K,
                    void* workspace, size_t workspace_bytes, dost_stream_t stream);
size_t dost_colsum_planes_workspace_bytes(long long M, int W);
int dost_colsum_planes(const void* hi, const void* lo, long long ld, long long M, int W, float* out, void* workspace,
                       size_t workspace_bytes, dost_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Row kernels: LayerNorm (eps = 1e-5, affine) optionally followed by PReLU -- nn.LayerNorm + nn.PReLU
 * in edge_mlp / node_mlp_2 (DOSTransformer.py:171,182) and layers/transformer.py:132-134,142,168-170.
 * stats[M,2] = (mean, rstd).  Backward writes dx and per-block partial sums (workspace) that
 * dost_colsum-style fixed-order reduction turns into dgamma/dbeta/dslope (deterministic).
 * ------------------------------------------------------------------------------------------- */
int dost_ln_fwd(int dtype, const void* x, long long ldx, const void* gamma, const void* beta, const void* prelu_slope,
                void* y, void* stats, long long M, int W, dost_stream_t stream);
size_t dost_ln_bwd_workspace_bytes(int dtype, long long M, int W);
int dost_ln_bwd(int dtype, const void* dy, long long ld_dy, const void* x, long long ldx, const void* stats,
                const void* gamma, const void* beta, const void* prelu_slope, void* dx, void* dgamma, void* dbeta,
                void* dslope, long long M, int W, void* workspace, size_t workspace_bytes, dost_stream_t stream);

/* out[w] = sum_m x[m*ld + w] in a fixed order (bias gradients, broadcast-row gradients). */
size_t dost_colsum_workspace_bytes(int dtype, long long M, long long W);
int dost_colsum(int dtype, const void* x, long long ld, long long M, long long W, void* out, void* workspace,
                size_t workspace_bytes, dost_stream_t stream);

/* PReLU backward for Linear->PReLU->Linear encoders (DOSTransformer.py:103-105): dz = da * (z>0 ? 1 : a),
 * dslope = sum da * z * [z<=0] (fixed order). */
size_t dost_prelu_bwd_workspace_bytes(int dtype, long long n);
int dost_prelu_bwd(int dtype, const void* da, const void* z, const void* slope, void* dz, void* dslope, long long n,
                   void* workspace, size_t workspace_bytes, dost_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Segmented reductions and gathers: scatter_sum / scatter_mean (DOSTransformer.py:158,187;
 * DOSTransformer_phonon.py:180,209; utils.py:91) as CSR reductions, and the adjoint of x[row], x[col]
 * (DOSTransformer.py:143).  out[s, :W] (+)= scale_s * sum_{j in [rowptr[s], rowptr[s+1])} src[perm[j]*ld + :W]
 * with scale_s = 1 (sum) or 1/max(count,1) (mean); perm == NULL means identity (contiguous segments).
 * ------------------------------------------------------------------------------------------- */
int dost_segment_reduce(int dtype, const void* src, long long ld, const int32_t* rowptr, const int32_t* perm,
                        long long nseg, int W, int mean, int accumulate, void* out, long long ldo,
                        dost_stream_t stream);
/* out[r, :W] = src[idx[r]*ld + :W] * (deg_rowptr ? 1/max(deg(idx[r]),1) : 1) + (add ? add[r*ld_add + :W] : 0) */
int dost_gather_rows(int dtype, const void* src, long long ld, const int32_t* idx, const int32_t* deg_rowptr,
                     const void* add, long long ld_add, long long R, int W, void* out, long long ldo,
                     dost_stream_t stream);

/* Phonon edge features: smooth_cutoff(|v|/4) * [1, sqrt(3) v/|v|] (DOSTransformer_phonon.py:75-77). */
int dost_phonon_edge_feat(int dtype, const void* edge_vec, long long E, void* out, dost_stream_t stream);
/* the same features computed inside the first Linear of the edge encoder (GN_encoder.edge_encoder[0..1],
 * DOSTransformer_phonon.py:74-77): pre[e, :] = weight [H, 4] . feat(edge_vec[e]) + bias, out = PReLU(pre); the [E, 4] feature
 * tensor is never written.  pre may be NULL (inference). */
int dost_phonon_edge_encode(int dtype, const void* edge_vec, long long E, const void* weight, const void* bias,
                            const void* prelu_slope, int H, void* pre, void* out, dost_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Ragged energy->atom cross attention with analytic phantom keys: to_dense_batch zero padding +
 * LayerNorm + projection-free single-head attention (DOSTransformer.py:61-63,73,87;
 * layers/transformer.py:132-138; layers/multihead_attention.py:68-72).  q [S,T,H] (already LN'd;
 * q_sstride = 0 broadcasts one [T,H] block), kv [N,H] (already LN'd), phantom [H] = that layer's
 * layer_norms[0].bias (what LN maps a zero-padded row to), ptr [B+1] crystal offsets, sequence s
 * attends to crystal s % B and sees (*nmax - n_b) phantom keys.  out = resid + softmax(q k^T scale) k.
 * lse [S,T] float.  Dropout (training, p>0) acts on probabilities with a counter-based mask.
 * ------------------------------------------------------------------------------------------- */
int dost_xattn_fwd(int dtype, const void* q, long long q_sstride, const void* kv, const void* phantom,
                   const int32_t* ptr, const int32_t* nmax, const void* resid, long long resid_sstride, void* out,
                   float* lse, int S, int B, int T, int H, double scale, double drop_p, unsigned long long seed,
                   dost_stream_t stream);
size_t dost_xattn_bwd_workspace_bytes(int dtype, int S, int T, int H);
/* dq [S,T,H], dkv [N,H] (overwritten), dphantom [H]; attn_out = out - resid is recomputed from o_attn. */
int dost_xattn_bwd(int dtype, const void* d_out, const void* q, long long q_sstride, const void* kv,
                   const void* phantom, const int32_t* ptr, const int32_t* node_crystal, const int32_t* nmax,
                   const void* out, const void* resid, long long resid_sstride, const float* lse, void* dq,
                   void* dkv, void* dphantom, int S, int B, int T, int H, long long N, double scale, double drop_p,
                   unsigned long long seed, void* workspace, size_t workspace_bytes, dost_stream_t stream);
int dost_xattn_fwd_dseed(int dtype, const void* q, long long q_sstride, const void* kv, const void* phantom,
                         const int32_t* ptr, const int32_t* nmax, const void* resid, long long resid_sstride, void* out,
                         float* lse, int S, int B, int T, int H, double scale, double drop_p, unsigned long long seed,
                         const unsigned long long* seed_offset, dost_stream_t stream);
int dost_xattn_bwd_dseed(int dtype, const void* d_out, const void* q, long long q_sstride, const void* kv,
                         const void* phantom, const int32_t* ptr, const int32_t* node_crystal, const int32_t* nmax,
                         const void* out, const void* resid, long long resid_sstride, const float* lse, void* dq,
                         void* dkv, void* dphantom, int S, int B, int T, int H, long long N, double scale, double drop_p,
                         unsigned long long seed, const unsigned long long* seed_offset, void* workspace,
                         size_t workspace_bytes, dost_stream_t stream);
/* Attention map of a dost_xattn_fwd call (the reference's attn_weights, multihead_attention.py:68-71, batch-first, keys
 * zero-padded by to_dense_batch): out [S, T, cols] in dtype, recomputed from that call's lse.  Column j < n_b is atom j of the
 * crystal, columns n_b .. *nmax - 1 each hold the probability of ONE phantom key, columns past *nmax are 0.  drop_p,
 * mask_seed, seed_offset: those of the forward (mask / (1 - p) applied per key slot, the same bits). */
int dost_xattn_probs(int dtype, const void* q, long long q_sstride, const void* kv, const void* phantom, const int32_t* ptr,
                     const int32_t* nmax, const float* lse, void* out, int cols, int S, int B, int T, int H, double scale,
                     double drop_p, unsigned long long mask_seed, const unsigned long long* seed_offset, dost_stream_t stream);

/* Tensor-core formulation of the same attention (fp32, no dropout, one sequence per crystal): the contractions are ragged
 * batched dost_gemm_bf16 problems over an extended key plane [N + B, H] that holds one phantom-key row per crystal after its
 * atoms (dost_xattn_kv_ext_build); the fp32 softmax over the n_b real columns and the phantom column (weight *nmax - n_b)
 * writes the probabilities / score gradients as operand planes [rows, ldp] (columns past the crystal's own are zero).
 * scores, dP: [S*T, npad] fp32; lse [S*T]; dext [N + B, H] -> dkv [N, H] and the B phantom-key rows. */
int dost_xattn_kv_ext_build(const float* y, const float* beta, const int32_t* batch, const int32_t* ptr, long long N, int B,
                            int H, void* hi, void* lo, long long ldp, dost_stream_t stream);
int dost_xattn_kv_ext_split(const float* dext, const int32_t* batch, const int32_t* ptr, long long N, int B, int H, float* dkv,
                            float* dbeta_rows, dost_stream_t stream);
/* the same adjoint from key gradients computed per sequence into a padded buffer dpad [reps*B][npad][H] (sequence s = rep*B + b
 * attends to crystal b): dkv[r] = sum_rep dpad[rep*B + b][r - ptr[b]], dbeta_rows[b] = sum_rep dpad[rep*B + b][n_b] */
int dost_xattn_kv_pad_split(const float* dpad, int npad, int reps, const int32_t* batch, const int32_t* ptr, long long N, int B, int H,
                            float* dkv, float* dbeta_rows, dost_stream_t stream);
/* drop_p > 0: attention dropout (multihead_attention.py:71) with the counter-based mask of dost_xattn_fwd (index =
 * row * Nmax + key slot; the Nmax - n_b phantom copies occupy the slots n_b .. Nmax-1 and survive individually): the planes
 * hold mask / (1 - p) * P, the phantom column (surviving copies) / (1 - p) * P_phantom; the backward regenerates the mask. */
int dost_xattn_softmax_fwd(const float* scores, const int32_t* ptr, const int32_t* nmax, long long rows, int B, int T, int npad,
                           double scale, void* hi, void* lo, long long ldp, float* lse, double drop_p, unsigned long long seed,
                           dost_stream_t stream);
int dost_xattn_softmax_bwd(const float* scores, const float* lse, const float* dP, const int32_t* ptr, const int32_t* nmax,
                           long long rows, int B, int T, int npad, double scale, void* hi, void* lo, long long ldp,
                           double drop_p, unsigned long long seed, dost_stream_t stream);
int dost_xattn_softmax_fwd_dseed(const float* scores, const int32_t* ptr, const int32_t* nmax, long long rows, int B, int T,
                                 int npad, double scale, void* hi, void* lo, long long ldp, float* lse, double drop_p,
                                 unsigned long long seed, const unsigned long long* seed_offset, dost_stream_t stream);
int dost_xattn_softmax_bwd_dseed(const float* scores, const float* lse, const float* dP, const int32_t* ptr, const int32_t* nmax,
                                 long long rows, int B, int T, int npad, double scale, void* hi, void* lo, long long ldp,
                                 double drop_p, unsigned long long seed, const unsigned long long* seed_offset,
                                 dost_stream_t stream);

/* Row softmax for the dense T x T self attention (layers/multihead_attention.py:68-70): p = softmax_fp32(s*scale);
 * pd = dropout(p); rows are ld elements apart (ld >= cols).  Backward: ds = scale * p * (dp - sum(dp*p)) with dp = mask/(1-p) * dpd. */
int dost_softmax_fwd(int dtype, const void* s, void* p, void* pd, long long rows, int cols, long long ld, double scale,
                     double drop_p, unsigned long long seed, dost_stream_t stream);
int dost_softmax_bwd(int dtype, const void* p, const void* dpd, void* ds, long long rows, int cols, long long ld, double scale,
                     double drop_p, unsigned long long seed, dost_stream_t stream);
int dost_softmax_fwd_dseed(int dtype, const void* s, void* p, void* pd, long long rows, int cols, long long ld, double scale,
                           double drop_p, unsigned long long seed, const unsigned long long* seed_offset, dost_stream_t stream);
int dost_softmax_bwd_dseed(int dtype, const void* p, const void* dpd, void* ds, long long rows, int cols, long long ld,
                           double scale, double drop_p, unsigned long long seed, const unsigned long long* seed_offset,
                           dost_stream_t stream);

/* Same, with the (dropped-out) probabilities / the score gradients also written as bf16 hi/lo operand planes (ds may be
 * NULL when only the planes are wanted). */
int dost_softmax_fwd_planes(const float* s, float* p, float* pd, long long rows, int cols, long long ld, double scale,
                            double drop_p, unsigned long long seed, void* hi, void* lo, long long ldp, dost_stream_t stream);
int dost_softmax_bwd_planes(const float* p, const float* dpd, float* ds, long long rows, int cols, long long ld, double scale,
                            double drop_p, unsigned long long seed, void* hi, void* lo, long long ldp, dost_stream_t stream);
int dost_softmax_fwd_planes_dseed(const float* s, float* p, float* pd, long long rows, int cols, long long ld, double scale,
                                  double drop_p, unsigned long long seed, const unsigned long long* seed_offset, void* hi,
                                  void* lo, long long ldp, dost_stream_t stream);
int dost_softmax_bwd_planes_dseed(const float* p, const float* dpd, float* ds, long long rows, int cols, long long ld,
                                  double scale, double drop_p, unsigned long long seed, const unsigned long long* seed_offset,
                                  void* hi, void* lo, long long ldp, dost_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Fused single-head attention forward on the tensor cores (layers/multihead_attention.py:68-72 with
 * the residual of layers/transformer.py:133-134): out = residual + softmax_fp32(q k^T * scale) k in ONE
 * kernel (TMA -> tcgen05.mma -> TMEM -> fp32 softmax -> tcgen05.mma), no score matrix in HBM.  Keys are
 * the values (the reference attention has no projections).  Operands are bf16 hi/lo planes.
 *   dense  (k_rowoff == NULL): sequence s uses rows s*Lk .. s*Lk+Lk-1 of k (the T x T energy
 *          self attention, DOSTransformer.py:85-91)
 *   ragged (k_rowoff != NULL): sequence s uses rows k_rowoff[s] .. +k_count[s]-1 of ONE extended key
 *          plane of k_rows rows whose last row per crystal is the phantom key (dost_xattn_kv_ext_build);
 *          that column stands for nmax - (k_count[s] - 1) zero-padded keys (to_dense_batch + LayerNorm,
 *          DOSTransformer.py:61-63).  max_keys >= every k_count[s] (host-side padding length + 1).
 * At most 256 keys per sequence, H in {64, 128, 192, 256}.  drop_p > 0: attention dropout with the
 * library's counter-based mask (index = row * Lk + key, or row * Nmax + key slot for ragged keys, the
 * phantom copies surviving individually: the mask of dost_softmax_fwd / dost_xattn_softmax_fwd); the planes
 * then hold the DROPPED-OUT probabilities and lse (optional, [S*Lq]) the log-sum-exp of the scaled scores,
 * from which the backward recomputes P.  residual: [S, Lq, H] (res_seq_stride = Lq*H) or shared [Lq, H] (0) or NULL.
 * p_hi / p_lo (optional, [S*Lq, ld_p]): the probabilities as operand planes for the backward pass
 * (phantom column = total probability of its copies; columns past a sequence's keys are zero).
 * dost_softmax_bwd_from_planes: dS = scale * P (dP - sum P dP) per row from those planes -> planes.
 * ------------------------------------------------------------------------------------------- */
int dost_attn_fused_supported(int Lq, int H, int max_keys);
int dost_attn_fused_fwd(const void* q_hi, const void* q_lo, long long ld_q, const void* k_hi, const void* k_lo, long long ld_k,
                        long long k_rows, int S, int Lq, int Lk, int H, const int32_t* k_rowoff, const int32_t* k_count,
                        const int32_t* nmax, int max_keys, double scale, const float* residual, long long res_seq_stride,
                        float* out, void* p_hi, void* p_lo, long long ld_p, int precision, double drop_p,
                        unsigned long long seed, float* lse, dost_stream_t stream);
int dost_attn_fused_fwd_dseed(const void* q_hi, const void* q_lo, long long ld_q, const void* k_hi, const void* k_lo,
                              long long ld_k, long long k_rows, int S, int Lq, int Lk, int H, const int32_t* k_rowoff,
                              const int32_t* k_count, const int32_t* nmax, int max_keys, double scale, const float* residual,
                              long long res_seq_stride, float* out, void* p_hi, void* p_lo, long long ld_p, int precision,
                              double drop_p, unsigned long long seed, const unsigned long long* seed_offset, float* lse,
                              dost_stream_t stream);
int dost_softmax_bwd_from_planes(const void* p_hi, const void* p_lo, long long ld_pp, const float* dP, long long ld_dp,
                                 long long rows, int cols, double scale, void* hi, void* lo, long long ldp, dost_stream_t stream);
/* Attention maps from the probability planes [rows, ld_p] written by dost_attn_fused_fwd, dost_softmax_fwd_planes or
 * dost_xattn_softmax_fwd: out [rows, cols] fp32 = hi + lo (hi alone when p_lo is NULL), the P the P k product consumed.
 *   ptr == NULL: dense, plane column c -> column c < cols (cols <= ld_p)
 *   ptr != NULL: ragged rows (row r attends to crystal (r / T) % B): the n_b atom columns, then the phantom column expanded
 *                into the key slots n_b .. *nmax - 1 (total / (*nmax - n_b) each; with drop_p > 0 total / kept for the slots
 *                whose mask bit, index r * *nmax + slot with mask_seed + *seed_offset, survived, 0 for the others), 0 past *nmax. */
int dost_attn_maps_from_planes(const void* p_hi, const void* p_lo, long long ld_p, long long rows, int cols, int T, int B,
                               const int32_t* ptr, const int32_t* nmax, float* out, double drop_p, unsigned long long mask_seed,
                               const unsigned long long* seed_offset, dost_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * DOS loss.  mode 0 (eDOS, main_eDOS.py:111-123): y = max(y,0); per-crystal RMSE; mean over crystals;
 * loss = rmse_global + beta * rmse_system.  mode 1 (phonon, main_phDOS.py:109-114): sqrt of batch-wide MSE.
 * saved [4*B]: [0,2B) per-crystal rmse (mode 0) / [0,2) batch rmse (mode 1) for the backward; [2B,4B) scratch.
 * ------------------------------------------------------------------------------------------- */
int dost_loss_fwd(int dtype, int mode, const void* pred_g, const void* pred_s, const void* y, double beta, int B,
                  int T, void* loss, void* saved, dost_stream_t stream);
int dost_loss_bwd(int dtype, int mode, const void* pred_g, const void* pred_s, const void* y, double beta, int B,
                  int T, const void* saved, const void* grad_loss, void* d_pred_g, void* d_pred_s,
                  dost_stream_t stream);

/* Evaluation metrics of utils.test / utils.test_phonon (utils.py:61-143), on the device: per crystal (the reference
 * evaluates with batch_size 1); clamp_pred != 0 (eDOS, utils.py:75-76) clamps BOTH targets and predictions at 0,
 * clamp_pred == 0 (phonon, utils.py:127-131) clamps neither.  per_crystal [B,4] = (mse, rmse, mae,
 * r2 = 1 - SSE / sum (y - mean y)^2, two-pass; a constant target scores 1 if SSE == 0 else 0 like sklearn's r2_score);
 * mean [4] (optional) = their means over crystals. */
int dost_eval_metrics(int dtype, const void* pred, const void* y, int clamp_pred, int B, int T, void* per_crystal, void* mean,
                      dost_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Fused multi-tensor AdamW, fp32 (torch.optim.AdamW(lr, weight_decay=1e-2), main_eDOS.py:93,127 / main_phDOS.py:90):
 * the step right after the hot path (SURVEY.md 8f rank 1).  Host arrays of `ntensors` device pointers / element counts;
 * `step` is the 1-based step count used for the bias corrections.  Tensors without a gradient are simply not listed
 * (torch skips grad-is-None parameters, which keeps the reference's dead parameters at their initial values).
 * ------------------------------------------------------------------------------------------- */
int dost_adamw_step(int ntensors, void* const* params, const void* const* grads, void* const* exp_avg,
                    void* const* exp_avg_sq, const long long* numel, double lr, double beta1, double beta2, double eps,
                    double weight_decay, long long step, dost_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * On-device batch assembly from a packed crystal store (SURVEY.md 8f rank 3).  Replaces the CPU collate of
 * torch_geometric.loader.DataLoader / Batch.from_data_list as the launchers use it (main_eDOS.py:54-56,
 * main_phDOS.py:52-54): node and edge tensors of the selected crystals concatenated in batch order, edge_index
 * shifted by each crystal's node offset, batch = repeat_interleave(arange(B), n_b), per-crystal fields stacked.
 * Store layout: crystal c owns rows node_ptr_all[c]..node_ptr_all[c+1] of every node table and rows
 * edge_ptr_all[c]..edge_ptr_all[c+1] of every edge table; edge_index_all [2,E_all] holds crystal-LOCAL node ids.
 * All index arrays are int64 on the device.  Bit-exact (copies and integer adds only).
 * ------------------------------------------------------------------------------------------- */
/* node_ptr_out[B+1], edge_ptr_out[B+1] (edge tables optional, both or neither) = exclusive scans of the selected
 * crystals' node / edge counts; nmax_out (optional, 1 int64) = largest node count = to_dense_batch's padding length
 * (DOSTransformer.py:61); *bad_flag is set to 1 when an id is outside [0,C) (that crystal then counts as empty). */
int dost_collate_ptr(const int64_t* ids, long long B, const int64_t* node_ptr_all, const int64_t* edge_ptr_all,
                     long long C, int64_t* node_ptr_out, int64_t* edge_ptr_out, int64_t* nmax_out, int32_t* bad_flag,
                     dost_stream_t stream);
/* Segmented row copy of one table, rows of row_bytes (multiple of 4).  Ragged table: src_ptr_all = the store's
 * node_ptr_all or edge_ptr_all and out_ptr = the matching scan from dost_collate_ptr; per-crystal table (glob, system,
 * targets): both NULL, row ids[b] -> row b, rows_out == B. */
int dost_collate_rows(const void* src, const int64_t* src_ptr_all, const int64_t* ids, const int64_t* out_ptr,
                      long long B, long long rows_out, long long row_bytes, void* dst, dost_stream_t stream);
/* edge_index_out [2,E_out] = local ids + node_ptr_out[b]; batch_out [N_out] = b.  Either output may be NULL. */
int dost_collate_index(const int64_t* edge_index_all, long long E_all, const int64_t* node_ptr_all,
                       const int64_t* edge_ptr_all, const int64_t* ids, const int64_t* node_ptr_out,
                       const int64_t* edge_ptr_out, long long B, long long N_out, long long E_out,
                       int64_t* edge_index_out, int64_t* batch_out, dost_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Periodic neighbour lists and eDOS bond features on the device (SURVEY.md 8f rank 4).  Replaces the reference's offline
 * CPU graph construction: ase.neighbor_list("ijS", cutoff, self_interaction=True) + edge vectors (utils.py:267-273) and
 * pymatgen get_all_neighbors(8.0) -> 12 nearest -> Gaussian expansion (data/mat2graph.py:162-179,185,212-243).
 * lattice [C,9] fp64 (rows = lattice vectors), pos [N,3] fp64 Cartesian, node_ptr [C+1], crystal_of [N] (= batch), int64.
 * Canonical edge order: (centre i, neighbour j, shift Sx, Sy, Sz) ascending.  Arithmetic contract (each op rounded, no
 * FMA): s = (Sx*L0 + Sy*L1) + Sz*L2; v = (pos[j] - pos[i]) + s; d = sqrt((vx*vx + vy*vy) + vz*vz); neighbour iff d < cutoff;
 * the zero-shift self pair only with self_interaction.  Two passes: count [N], exclusive scan by the caller, fill.
 * ------------------------------------------------------------------------------------------- */
int dost_neighbor_count(const double* lattice, const double* pos, const int64_t* node_ptr, const int64_t* crystal_of,
                        long long N, double cutoff, int self_interaction, int64_t* count, dost_stream_t stream);
/* edge_ptr [N+1] = exclusive scan of count.  edge_src/edge_dst [E] (crystal-local ids if local_ids, else row ids of pos),
 * optional edge_shift [E,3] int64, edge_vec [E,3], edge_len [E]. */
int dost_neighbor_fill(const double* lattice, const double* pos, const int64_t* node_ptr, const int64_t* crystal_of,
                       long long N, double cutoff, int self_interaction, const int64_t* edge_ptr, int local_ids,
                       int64_t* edge_src, int64_t* edge_dst, int64_t* edge_shift, double* edge_vec, double* edge_len,
                       dost_stream_t stream);
/* The k nearest entries of every atom's list (stable: ties keep list order): out_idx [N,k] = edge_dst of the pick,
 * out_dist [N,k], optional out_edge [N,k] = its edge id; short lists are padded with (pad_idx, pad_dist, -1)
 * (mat2graph.py:223-229 pads with index 0 and distance radius + 1). */
int dost_knn_select(const int64_t* edge_ptr, const int64_t* edge_dst, const double* edge_len, long long N, int k,
                    long long pad_idx, double pad_dist, int64_t* out_idx, double* out_dist, int64_t* out_edge,
                    dost_stream_t stream);
/* GaussianDistance.expand (mat2graph.py:162-179): out [n,nfilt] fp32 = exp(-(d - mu_f)^2 / var^2), mu_f = dmin + f*step, in
 * fp64 then rounded to fp32 like torch.Tensor(numpy_array) does. */
int dost_gaussian_expand(const double* dist, long long n, double dmin, double step, int nfilt, double var, float* out,
                         dost_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* DOST_H_ */
