/*
 * csmpn_b200 -- C ABI of the B200-native CSMPN hot path (libcsmpn_b200.so, sm_100a).
 *
 * The reference (congliuUvA/Clifford-Group-Equivariant-Simplicial-Message-Passing-Networks) is pure
 * Python; its seam for this path is the class API of csmpn/algebra/cliffordalgebra.py and
 * csmpn/models/cegnn_utils.py.  Every entry point below replaces the body of one reference method
 * (cited per function as file:line, relative to the reference root) and is what a ctypes binding of
 * that method would call; INTEGRATION.md shows the binding.
 *
 * Conventions
 *  - All float tensors are fp32, contiguous, laid out [rows, channels, B] with the B = 2^dim blades
 *    innermost in grade-major ("short-lex") blade order (metric.py:18-29).
 *  - All pointers except `metric` / `*_host` and the params structs themselves are DEVICE pointers that the
 *    caller owns; nothing returned is allocated by the library.  Work is enqueued on `stream`
 *    (a cudaStream_t passed as void*); the call returns without synchronising.
 *  - `metric` is a HOST array of `dim` floats (the diagonal metric handed to CliffordAlgebra(metric),
 *    cliffordalgebra.py:11-25).  dim in 1..5.
 *  - Return value: 0 on success, a negative csmpn_status otherwise.  No exceptions cross the ABI.
 *  - Re-entrant; no global state besides immutable function attributes set on first use.
 */
#ifndef CSMPN_B200_H_
#define CSMPN_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* csmpn_stream_t; /* cudaStream_t */

enum csmpn_status {
  CSMPN_OK = 0,
  CSMPN_ERR_BAD_DIM = -1,       /* dim outside 1..5 */
  CSMPN_ERR_BAD_ARG = -2,       /* null pointer / negative size / inconsistent sizes */
  CSMPN_ERR_UNSUPPORTED = -3,   /* configuration not built (e.g. fused path with a degenerate metric) */
  CSMPN_ERR_CUDA = -4,          /* a CUDA runtime call failed; see csmpn_last_cuda_error() */
  CSMPN_ERR_WORKSPACE = -5      /* workspace too small */
};

int csmpn_version(void);
const char* csmpn_status_string(int status);
const char* csmpn_last_cuda_error(void);
/* number of SMs of the current device (grid sizing is a multiple of this) */
int csmpn_sm_count(void);
/* number of CUDA kernels this library has launched in this process (monotonic; not thread-safe accounting) */
int64_t csmpn_launch_count(void);

/* ---- algebra tables (host side; metric.py:18-120, cliffordalgebra.py:27-42,238-252) ------------------
 * out_idx[B*B]  : blade index j of e_i e_k            coef[B*B] : c[i, j(i,k), k]
 * grades[B]     : grade of each blade                 paths[G*G*G] : 1 where (g_i, g_j, g_k) occurs
 * All outputs are HOST arrays; any may be NULL. */
int csmpn_algebra_tables(int dim, const float* metric, int32_t* out_idx, float* coef, int32_t* grades,
                         uint8_t* paths);

/* ---- geometric product  (CliffordAlgebra.geometric_product, cliffordalgebra.py:44-54) ----------------
 * out[r, j] = sum_{i,k} a[r,i] c[i,j,k] b[r,k]      a, b, out: [n_mv, B]
 * a_stride_zero / b_stride_zero: 1 broadcasts a single multivector over all rows (einsum "...").   */
int csmpn_gp_fwd(int dim, const float* metric, const float* a, const float* b, float* out, int64_t n_mv,
                 int a_bcast, int b_bcast, csmpn_stream_t stream);
/* grad_a, grad_b: [n_mv, B] (per-row gradients even for a broadcast operand; the caller reduces). */
int csmpn_gp_bwd(int dim, const float* metric, const float* a, const float* b, const float* grad_out,
                 float* grad_a, float* grad_b, int64_t n_mv, int a_bcast, int b_bcast, csmpn_stream_t stream);

/* ---- per-grade quadratic forms  (CliffordAlgebra.qs / norms, cliffordalgebra.py:143-168) -------------
 * q[r, g] = sum_{i in grade g} qsign_i x[r,i]^2 ;  mode 0: q, mode 1: norm = (q^2 + 1e-16)^(1/4)  */
int csmpn_grade_forms_fwd(int dim, const float* metric, const float* x, float* out, int64_t n_mv, int mode,
                          csmpn_stream_t stream);
int csmpn_grade_forms_bwd(int dim, const float* metric, const float* x, const float* grad_out, float* grad_x,
                          int64_t n_mv, int mode, csmpn_stream_t stream);

/* ---- MVLinear  (cegnn_utils.py:287-338) ---------------------------------------------------------------
 * y[r,n,i] = sum_m x[r,m,i] W[n,m,g(i)] (+ bias[n] on blade 0)
 * weight: [Cout, Cin, G] if subspaces else [Cout, Cin]; bias: [Cout] or NULL.                          */
int csmpn_mvlinear_fwd(int dim, const float* x, const float* weight, const float* bias, float* y, int64_t rows,
                       int c_in, int c_out, int subspaces, csmpn_stream_t stream);
/* grad_x = grad_y . W  (same contraction with the roles of n and m swapped) */
int csmpn_mvlinear_bwd_input(int dim, const float* grad_y, const float* weight, float* grad_x, int64_t rows,
                             int c_in, int c_out, int subspaces, csmpn_stream_t stream);
/* grad_w[n,m,g] = sum_{r, i in g} grad_y[r,n,i] x[r,m,i] ; grad_bias[n] = sum_r grad_y[r,n,0] (NULL to skip).
 * Deterministic two-pass reduction; workspace (device) must hold csmpn_mvlinear_bwd_weight_workspace() bytes. */
int64_t csmpn_mvlinear_bwd_weight_workspace(int dim, int64_t rows, int c_in, int c_out);
int csmpn_mvlinear_bwd_weight(int dim, const float* x, const float* grad_y, float* grad_w, float* grad_bias,
                              int64_t rows, int c_in, int c_out, int subspaces, void* workspace,
                              int64_t workspace_bytes, csmpn_stream_t stream);

/* ---- MVSiLU (invariant="mag2")  (cegnn_utils.py:53-83) -----------------------------------------------
 * y_i = sigmoid(a[n,g(i)] * inv_g + b[n,g(i)]) x_i ; inv_0 = x_0, inv_g = q_g(x).   a, b: [C, G]        */
int csmpn_mvsilu_fwd(int dim, const float* metric, const float* x, const float* a, const float* b, float* y,
                     int64_t rows, int channels, csmpn_stream_t stream);
/* grad_a, grad_b: [C, G] (overwritten).  workspace: csmpn_param_grad_workspace(channels * G * 2) bytes. */
int csmpn_mvsilu_bwd(int dim, const float* metric, const float* x, const float* a, const float* b,
                     const float* grad_y, float* grad_x, float* grad_a, float* grad_b, int64_t rows, int channels,
                     void* workspace, int64_t workspace_bytes, csmpn_stream_t stream);

/* ---- NormalizationLayer  (cegnn_utils.py:34-51) -------------------------------------------------------
 * y_i = x_i / (sigmoid(a[n,g]) (norm_g(x) - 1) + 1 + 1e-6)      a: [C, G]                              */
int csmpn_mvnorm_fwd(int dim, const float* metric, const float* x, const float* a, float* y, int64_t rows,
                     int channels, csmpn_stream_t stream);
int csmpn_mvnorm_bwd(int dim, const float* metric, const float* x, const float* a, const float* grad_y,
                     float* grad_x, float* grad_a, int64_t rows, int channels, void* workspace,
                     int64_t workspace_bytes, csmpn_stream_t stream);

/* ---- MVLayerNorm  (cegnn_utils.py:86-96) --------------------------------------------------------------
 * y = a[n] x / (mean_n (Q(x[r,n])^2 + 1e-16)^(1/4) + 1e-6),  Q = sum_i qsign_i x_i^2     a: [C]        */
int csmpn_mvlayernorm_fwd(int dim, const float* metric, const float* x, const float* a, float* y, int64_t rows,
                          int channels, csmpn_stream_t stream);
int csmpn_mvlayernorm_bwd(int dim, const float* metric, const float* x, const float* a, const float* grad_y,
                          float* grad_x, float* grad_a, int64_t rows, int channels, void* workspace,
                          int64_t workspace_bytes, csmpn_stream_t stream);

/* ---- weighted geometric product of SteerableGeometricProductLayer  (cegnn_utils.py:126-155) ----------
 * z[r,n,j] = sum_{i,k} x[r,n,i] c[i,j,k] w[n, path(g_i,g_j,g_k)] r[r,n,k]
 * out = (left + z) * scale   when `left` != NULL (include_first_order: scale = 1/sqrt 2), else z * scale.
 * w: [C, P] with P = number of non-zero grade paths in row-major (g_i, g_j, g_k) order.                */
int csmpn_wgp_fwd(int dim, const float* metric, const float* x, const float* r, const float* w, const float* left,
                  float scale, float* out, int64_t rows, int channels, csmpn_stream_t stream);
/* grad_x, grad_r: [rows, C, B]; grad_w: [C, P]; grad_left = scale * grad_out is left to the caller.     */
int csmpn_wgp_bwd(int dim, const float* metric, const float* x, const float* r, const float* w,
                  const float* grad_out, float scale, float* grad_x, float* grad_r, float* grad_w, int64_t rows,
                  int channels, void* workspace, int64_t workspace_bytes, csmpn_stream_t stream);

/* bytes of workspace needed by the *_bwd calls above that reduce `n_params` parameter gradients over rows */
int64_t csmpn_param_grad_workspace(int64_t n_params);

/* ---- graph plumbing for EGCL / PyG MessagePassing.propagate  (cegnn_utils.py:277-284) ----------------
 * csr_build: stable counting sort of the E adjacency pairs by key (receiver = edge_index[1], or sender).
 *   keys      [E] int64 (row of edge_index)      n_nodes: number of simplices
 *   rowptr    [n_nodes + 1] int32 (out)          perm [E] int32 (out): perm[p] = original pair id of the
 *   p-th pair in key-sorted order; pairs with equal key keep their original relative order.
 *   workspace: csmpn_csr_workspace(E, n_nodes) bytes.                                                   */
int64_t csmpn_csr_workspace(int64_t n_pairs, int64_t n_nodes);
int csmpn_csr_build(const int64_t* keys, int64_t n_pairs, int64_t n_nodes, int32_t* rowptr, int32_t* perm,
                    void* workspace, int64_t workspace_bytes, csmpn_stream_t stream);
/* out[p, :] = h[dst[p], :] - h[src[p], :]  for width floats per row (C*B); src/dst int64 [E].          */
int csmpn_gather_diff(const float* h, const int64_t* src, const int64_t* dst, float* out, int64_t n_pairs,
                      int64_t width, csmpn_stream_t stream);
/* Deterministic segment reduce (aggr "sum" | "mean", PyG scatter semantics: mean divides by
 * max(count,1), empty receivers get 0):   out[n,:] = sum_{p in rowptr[n]..rowptr[n+1]} msg[perm[p], :]
 * scaled by 1/max(deg,1) when mean != 0.   msg rows are in ORIGINAL pair order.                       */
int csmpn_segment_reduce(const float* msg, const int32_t* rowptr, const int32_t* perm, float* out,
                         int64_t n_nodes, int64_t width, int mean, csmpn_stream_t stream);
/* Adjoint of gather_diff, deterministic:  grad_h[n,:] (+)= sum_{p: dst[p]=n} g[p,:] - sum_{p: src[p]=n} g[p,:]
 * using the two CSR orderings (by receiver and by sender).  accumulate != 0 adds to grad_h.           */
int csmpn_scatter_diff(const float* g, const int32_t* rowptr_dst, const int32_t* perm_dst,
                       const int32_t* rowptr_src, const int32_t* perm_src, float* grad_h, int64_t n_nodes,
                       int64_t width, int accumulate, csmpn_stream_t stream);
/* Adjoint of segment_reduce: grad_msg[p,:] = grad_out[dst[p],:] * (mean ? 1/max(deg[dst[p]],1) : 1).   */
int csmpn_segment_expand(const float* grad_out, const int64_t* dst, const int32_t* rowptr, float* grad_msg,
                         int64_t n_pairs, int64_t width, int mean, csmpn_stream_t stream);

/* ---- fused CEMLP block  (one [MVLinear, MVSiLU, SteerableGeometricProductLayer, MVLayerNorm] block of CEMLP,
 *      cegnn_utils.py:180-207; with the gather of EGCL.message :254-262 or the concat of EGCL.update :264-275
 *      folded into its prologue and the residual of :272-273 into its epilogue) --------------------------------
 * Non-degenerate diagonal metrics (`metric`: every entry nonzero, e.g. Cl(p,q) or a rescaled Euclidean metric), dim
 * in {2,3,5} on engine 0 and {2,3} on engine 1.  Rows are processed in tiles held in shared memory; the three per-grade
 * channel GEMMs, the gates, norms and the weighted geometric product of a block never leave the SM.
 *
 * Input row r (c_in = c0 + c1 + c2 channels):
 *   mode 0 (concat):  [ p0[r, 0:c0] | p1[r, 0:c1] | p2[r, 0:c2] ]                (p1 / p2 may be NULL with c = 0)
 *   mode 1 (gather):  [ p0[dst[r], 0:c0] - p0[src[r], 0:c0] | p1[eid[r], 0:c1] ]  rows = adjacency pairs in
 *                     receiver-sorted order; src/dst/eid are int32 [rows] (eid = original pair id)
 *   mode 2 (vertex-table gather, engine 1): the (d+1)!-permutation rows of embed_simplicial_complex, see vt_k / vt_fp
 * Forward output y[r, 0:c] (+ res[r] when res != NULL).  When save_* are non-NULL the forward also stores the three
 * [rows, c, B] intermediates the backward needs (pre-SiLU y1, pre-normalisation right input xr, pre-LayerNorm o).  */
typedef struct csmpn_block_desc {
  int32_t mode, c0, c1, c2, c;          /* c = block width (hidden/out features) */
  int32_t has_b1;                       /* MVLinear bias present */
  int64_t rows;
  const float *p0, *p1, *p2;
  const int32_t *src, *dst, *eid;
  /* parameters, reference state_dict names in brackets (layer prefix "layers.k.") */
  const float* w1;  /* [c, c_in, G]  0.weight */
  const float* b1;  /* [c]           0.bias */
  const float* sa;  /* [c, G]        1.a */
  const float* sb;  /* [c, G]        1.b */
  const float* wr;  /* [c, c, G]     2.linear_right.weight */
  const float* na;  /* [c, G]        2.normalization.a */
  const float* wl;  /* [c, c, G]     2.linear_left.weight */
  const float* bl;  /* [c]           2.linear_left.bias */
  const float* wp;  /* [c, P]        2.weight */
  const float* la;  /* [c]           3.a */
  /* forward outputs */
  float* y;         /* [rows, c, B] */
  const float* res; /* [rows, c, B] or NULL */
  float *save_y1, *save_xr, *save_o;    /* [rows, c, B] each, or all NULL (inference) */
  /* ---- engine 1: tcgen05 tensor-core kernels (csrc/tc_block_*.cu), Cl(2,0) / Cl(3,0), see csmpn_block_tc_supported.
   * Intermediates use the blade-plane tile layout "BPT": [ceil(rows/128)][B][cp/4][128][4] fp32 with the channel count
   * padded to cp = a multiple of 16 (csmpn_bpt_floats); padded rows and channels hold zeros.  With engine 1 the three
   * save_* tensors are BPT [c], save_y2 (BPT [c], MVSiLU output) is REQUIRED (it is also the scratch between the two
   * forward kernels), save_x0 (BPT [c_in], fully written by the forward) keeps the assembled input row of a block
   * whose input is not already BPT, for the weight-gradient GEMM of the backward. */
  int32_t engine;                       /* 0 = FP32 SIMT kernels (csrc/block_fused.cu), 1 = tensor-core kernels */
  int32_t in_bpt;                       /* engine 1, mode 0, c1 = c2 = 0: p0 is a BPT [c0] tensor */
  int32_t out_bpt;                      /* engine 1: y is written as a BPT [c] tensor (res must be NULL) */
  int32_t stage_mask;                   /* engine 1 diagnostics: 0 = every kernel of the call; otherwise bit k selects kernel k
                                           (fwd: 0 f1, 1 f2; bwd: 0 b1, 1 gemm dy2, 2 b3, 3 gemm grad_x, 4 dW wl/wr, 5 dW w1,
                                           6 final reduce) -- bench.py times one kernel at a time with it */
  float *save_y2, *save_x0;
  int32_t pair_attr;                    /* mode 1: the c1 extra channels of a pair are  table[src] | table[dst]  with
                                           table = p1 [n_nodes, c1/2, B] (per-simplex attributes, e.g. the simplex-type
                                           embedding of md17_cssmpnn.py:122-133) instead of a materialised [E, c1, B]
                                           edge_attr read through eid; its gradient: csmpn_scatter_pair_sorted */
  int32_t vt_k, vt_fp;                  /* mode 2 (engine 1): "permute-embed" gather of embed_simplicial_complex
                                           (md17_cssmpnn.py:85-120): row r is one vertex ORDER of a simplex, src[r * vt_k + j]
                                           = row of its j-th vertex in the per-vertex feature table p0 [V, c0 / vt_k, B];
                                           input channel (t * vt_k + j) * vt_fp + f of the row = table channel t * vt_fp + f of
                                           vertex j (feature type t, vt_fp channels per type) -- the reference's
                                           cat(pos[verts], vel[verts], ...) layout, never materialised */
  void* fwd_ws;                         /* engine 1, wide blocks (csmpn_block_fwd_workspace > 0): device scratch of the
                                           forward for the pre-split weight images streamed with the K chunks */
  int64_t fwd_ws_bytes;
  int32_t tf32;                         /* engine 1: 0 = error-compensated fp32 products (x = hi + lo, three TF32 MMAs per
                                           product; the default), 1 = single-pass TF32: every GEMM operand rounded to
                                           nearest TF32 once, one MMA per product (what PyTorch does for fp32 matmuls under
                                           torch.backends.cuda.matmul.fp32_precision = "tf32"); smaller streamed weight
                                           images (csmpn_block_fwd_workspace / csmpn_block_bwd_workspace).  Engine 0
                                           ignores it; any other value is CSMPN_ERR_BAD_ARG.  The backward of a block must
                                           be called with the value of its forward. */
  const float* metric;                  /* HOST array of `dim` floats read at launch (as the `metric` argument of the unit
                                           entry points), or NULL; NULL or all ones = Euclidean.  A zero entry (degenerate
                                           metric) is CSMPN_ERR_UNSUPPORTED: compose such blocks from the unit kernels.
                                           The metric folds into the elementwise stages only (quadratic forms of MVSiLU,
                                           the normalisation and MVLayerNorm, and the weighted geometric product); a CUDA
                                           graph keeps the metric of its capture. */
} csmpn_block_desc;

/* gradients produced by csmpn_block_bwd (all overwritten; parameter gradients reduced deterministically) */
typedef struct csmpn_block_grads {
  const float* grad_y;   /* [rows, c, B] (the residual branch, if any, is the caller's: grad_res = grad_y) */
  float* grad_x;         /* [rows, c_in, B] gradient of the assembled input row (mode 1: w.r.t. the difference and the
                            gathered extra channels, in sorted-row order; scatter with csmpn_scatter_rows) */
  float *g_w1, *g_b1, *g_sa, *g_sb, *g_wr, *g_na, *g_wl, *g_bl, *g_wp, *g_la;
  /* engine 1 only: grad_y is a BPT [c] tensor / grad_x is written as a BPT [c_in] tensor (grad_x may be NULL) */
  int32_t gy_bpt, gx_bpt;
  /* engine 1 only, reference-layout grad_y: row r of the block reads grad_y row gy_rows[r] (NULL: row r) at a row pitch of
   * gy_row_stride floats (0: c * B).  This is the adjoint of the aggregation folded into the block: the cotangent of the
   * messages of receiver i is the cotangent of its aggregate (cegnn_utils.py:262-275 through PyG's scatter), so the
   * [pairs, c, B] expansion of the [simplices, c, B] gradient is never written. */
  const int32_t* gy_rows;
  int64_t gy_row_stride;
} csmpn_block_grads;

int csmpn_block_fwd(int dim, const csmpn_block_desc* desc, csmpn_stream_t stream);
/* device bytes csmpn_block_fwd needs in desc->fwd_ws (0 for every block whose weights stay resident in shared memory;
 * -1 if engine 1 does not handle the shape) */
int64_t csmpn_block_fwd_workspace(int dim, const csmpn_block_desc* desc);
/* 1 if the tensor-core engine handles a block of this shape (c_in input channels, width c) in algebra dimension dim */
int csmpn_block_tc_supported(int dim, int c_in, int c);
/* how engine 1 runs such a block: bit 0 = supported; bit 1 / bit 2 = the first / second forward kernel streams its weights
 * with the K chunks (wide blocks: Cl(3,0) with c >= 64, ...) instead of keeping them resident in shared memory; bit 3 =
 * the backward runs the wide plan (streamed GEMM weights, slab-wise weight-gradient launches, separate MVSiLU adjoint) */
int csmpn_block_tc_plan(int dim, int c_in, int c);
/* output channels per pass of such a block on engine 1: bits 0-9 the first forward kernel (ns1), bits 10-19 the second
 * (ns2; both equal the padded width Cp = 16 * ceil(c / 16) when the weights stay resident), bits 20-29 the streamed
 * backward GEMMs of the wide plan (np; 0 for the resident backward); 0 if engine 1 does not handle the shape */
int csmpn_block_tc_passes(int dim, int c_in, int c);
/* > 0 (the rows per shared-memory tile) if engine 0 keeps the block's weights resident in shared memory (forward and
 * backward), 0 if it would stage them per GEMM; with fewer than 4 rows per tile or staged weights the unit kernels
 * (csmpn_mvlinear_*, csmpn_mvsilu_*, csmpn_wgp_*, ...) composed by the host are the faster path for that shape */
int csmpn_block_simt_resident(int dim, int c_in, int c);
/* number of floats of a BPT tensor with `rows` rows and `channels` channels (padded to a multiple of 16) */
int64_t csmpn_bpt_floats(int dim, int64_t rows, int channels);
/* workspace for csmpn_block_bwd (device bytes; zero-initialised by the call itself) */
int64_t csmpn_block_bwd_workspace(int dim, const csmpn_block_desc* desc);
int csmpn_block_bwd(int dim, const csmpn_block_desc* desc, const csmpn_block_grads* grads, void* workspace,
                    int64_t workspace_bytes, csmpn_stream_t stream);

/* Sorted-order helpers for the fused EGCL path.
 * csr_sorted_indices: src_sorted[p] = (int32) src[perm[p]], dst_sorted[p] = (int32) dst[perm[p]].            */
int csmpn_csr_sorted_indices(const int64_t* src, const int64_t* dst, const int32_t* perm, int32_t* src_sorted,
                             int32_t* dst_sorted, int64_t n_pairs, csmpn_stream_t stream);
/* rank[perm[p]] = p : position of every original pair in the sorted order (inverse permutation) */
int csmpn_csr_rank(const int32_t* perm, int32_t* rank, int64_t n_pairs, csmpn_stream_t stream);
/* Both CSRs of a batch (by receiver and by sender), the receiver-sorted int32 views (src_sorted / dst_sorted, may both be
 * NULL) and the inverse permutation rank[pair] = position in receiver order (may be NULL) in SIX launches: every kernel
 * handles both key arrays and the scan is one CTA per array.  Same results as csmpn_csr_build x 2 +
 * csmpn_csr_sorted_indices + csmpn_csr_rank (16 launches).  workspace: csmpn_csr_workspace(E, n_nodes) x 2 bytes.
 * CSMPN_ERR_UNSUPPORTED when n_nodes > 65 536 (the one-CTA scan): use the calls above.
 * Out-of-range simplex ids are skipped, as in csmpn_csr_build (PyG would raise; validate with CSMPN_CHECK_INDICES=1). */
int csmpn_csr_build_pair(const int64_t* src, const int64_t* dst, int64_t n_pairs, int64_t n_nodes, int32_t* rowptr_dst,
                         int32_t* perm_dst, int32_t* rowptr_src, int32_t* perm_src, int32_t* src_sorted, int32_t* dst_sorted,
                         int32_t* rank, void* workspace, int64_t workspace_bytes, csmpn_stream_t stream);
/* segment reduce over CONTIGUOUS rows (messages already in receiver-sorted order):
 *   out[n,:] = sum_{p in [rowptr[n], rowptr[n+1])} msg[p,:]   (/ max(deg,1) when mean)                        */
int csmpn_segment_reduce_sorted(const float* msg, const int32_t* rowptr, float* out, int64_t n_nodes, int64_t width,
                                int mean, csmpn_stream_t stream);
/* its adjoint: grad_msg[p,:] = grad_out[dst_sorted[p],:] * (mean ? 1/max(deg,1) : 1)                           */
int csmpn_segment_expand_sorted(const float* grad_out, const int32_t* dst_sorted, const int32_t* rowptr,
                                float* grad_msg, int64_t n_pairs, int64_t width, int mean, csmpn_stream_t stream);
/* adjoint of the gather prologue, deterministic.  g: [E, ld] rows in receiver-sorted order; the first `width`
 * floats of each row are the gradient of (h[dst] - h[src]):
 *   grad_h[n,:] (+)= sum_{p in rowptr_dst[n]..} g[p, 0:width] - sum_{q in rowptr_src[n]..} g[rank[perm_src[q]], 0:width]
 * rank[e] = position of pair e in receiver-sorted order (inverse of perm_dst).                                 */
int csmpn_scatter_diff_sorted(const float* g, int64_t ld, const int32_t* rowptr_dst, const int32_t* rowptr_src,
                              const int32_t* perm_src, const int32_t* rank, float* grad_h, int64_t n_nodes,
                              int64_t width, int accumulate, csmpn_stream_t stream);
/* Gradient of a per-simplex table that entered every pair as  table[src] | table[dst]  (csmpn_block_desc.pair_attr):
 * out[n, :] = sum_{dst(p) = n} g[p, col_dst : col_dst + width] + sum_{src(p) = n} g[p, col_src : col_src + width]
 * over receiver-sorted pair rows of g (leading dimension ld floats); fixed summation order.  Replaces the autograd of
 * `torch.cat((node_attr[ei[0]], node_attr[ei[1]]), 1)` (md17_cssmpnn.py:131). */
int csmpn_scatter_pair_sorted(const float* g, int64_t ld, int64_t col_src, int64_t col_dst, const int32_t* rowptr_dst,
                              const int32_t* rowptr_src, const int32_t* perm_src, const int32_t* rank, float* out,
                              int64_t n_nodes, int64_t width, csmpn_stream_t stream);
/* out[r, 0:width] = a[r, 0:width] + b[r, 0:width] + c[r, 0:width], each operand with its own leading dimension (floats):
 * the three gradient contributions of the layer input h of EGCL.forward (cegnn_utils.py:254-284: gather source of the
 * messages, first source of the update, residual) summed in ONE pass instead of two autograd adds and a slice copy.
 * All pointers 16-byte aligned, width and leading dimensions multiples of 4. */
int csmpn_add3_rows(const float* a, int64_t lda, const float* b, int64_t ldb, const float* c, int64_t ldc, float* out,
                    int64_t n_rows, int64_t width, csmpn_stream_t stream);
/* out[eid[p], 0:width] = g[p, col0 : col0 + width]   (un-permute the gathered extra channels' gradient)        */
int csmpn_scatter_rows(const float* g, int64_t ld, int64_t col0, const int32_t* eid, float* out, int64_t n_rows,
                       int64_t width, csmpn_stream_t stream);

/* ---- simplicial lifting on the GPU ------------------------------------------------------------------------------
 * Replaces, for a whole batch of complexes in one launch, the reference's per-sample CPU pipeline
 *   rips_lift (utils.py:106-136) | simplicial_lift (utils.py:151-207) | simplicial_lift_hulls (utils.py:210-248)
 *   -> generate_indices / generate_features / generate_adjacencies[_single] (utils.py:37-103, 285-388)
 *   -> SimplicialTransform.add_missing_adj / get_edge / x_ind / node_types (simplicial_data.py:105-175, 218-222)
 *   and ManualTransform (simplicial_data.py:254-302) for the fixed CMU-motion complex,
 * followed by the PyG collation of the batch (node offsets added to edge_index, SimplicialComplexData.__cat_dim__,
 * simplicial_data.py:14-25).  Outputs are bit-exact to the reference, order included.  At most 32 vertices per
 * complex; complexes of dimension <= 2.
 *
 *   mode RIPS    points [n_vertices_total, point_dim] fp32; edge iff Euclidean distance (double) <= max_edge_length;
 *                clique complex up to max_dim; adjacency of generate_adjacencies_single (extra 0_0 pairs)
 *   mode CLIQUE  pairs [2, n_pairs] int64 LOCAL vertex ids of an (un)directed graph, pptr [n_complexes+1]; clique
 *                complex up to triangles; adjacency of generate_adjacencies (no extra pairs)
 *   mode FACETS  facets [n_facets_total, facet_size] int64 local vertex ids (Qhull simplices), fptr [n_complexes+1];
 *                every <= max_dim face of every facet; adjacency of generate_adjacencies_single
 *   mode MOTION  pairs = the skeleton 0-0 pairs of every complex (31 vertices each); 12 edges, 4 triangles and the
 *                96 literal pairs of ManualTransform are appended
 * vptr [n_complexes+1]: first vertex of each complex (vertex counts).  All pointers are device pointers.           */
enum csmpn_lift_mode {
  CSMPN_LIFT_RIPS = 0, CSMPN_LIFT_CLIQUE = 1, CSMPN_LIFT_FACETS = 2, CSMPN_LIFT_MOTION = 3,
  CSMPN_LIFT_KNN = 4 /* CLIQUE whose graph is knn_graph(points, knn_k) (csmpn/data/md17.py:64, nba.py:48), built in-kernel */
};

typedef struct csmpn_lift_desc {
  int32_t mode, n_complexes, max_dim, point_dim, facet_size;
  int32_t max_vertices;  /* largest vertex count of a complex in the batch (0: at most 32).  <= 32: one 32-bit adjacency mask
                            per vertex, four complexes per CTA; 33..64: 64-bit masks, one complex per CTA; more: unsupported */
  double max_edge_length;
  int64_t n_pairs;
  const int32_t* vptr;
  const float* points;
  const int64_t* pairs;
  const int32_t* pptr;
  const int64_t* facets;
  const int32_t* fptr;
  /* CLIQUE / KNN: the filters of simplicial_lift (utils.py:181-200) over `points` [sum n, point_dim]: a graph edge enters
   * the complex iff its length <= edge_th or it is a face of a kept triangle; a 3-clique is kept iff its area
   * (triangle_area, utils.py:139-148) <= tri_th.  use_filters = 0: every edge and every 3-clique (the shipped 1e4). */
  int32_t knn_k, use_filters;
  float edge_th, tri_th;
} csmpn_lift_desc;

/* Pass 1: counts [n_complexes, 2] = (edges, triangles) of every complex; node_ptr / pair_ptr [n_complexes+1] =
 * exclusive prefix sums of simplices / adjacency pairs (last entry = batch totals, which the caller reads back to
 * size the outputs); *status (device int32) is set non-zero if a complex has more vertices than max_vertices allows (32 or 64).               */
int csmpn_lift_count(const csmpn_lift_desc* desc, int32_t* counts, int64_t* node_ptr, int64_t* pair_ptr, int32_t* status,
                     csmpn_stream_t stream);
/* Pass 2: edge_index [2, n_pairs_total] int64 (global ids), x_ind [N, 3] fp32 (local vertex ids, CPython frozenset
 * order, zero padded), node_types [N] int64 (simplex dimension), batch [N] int64 (complex id).                     */
int csmpn_lift_fill(const csmpn_lift_desc* desc, const int64_t* node_ptr, const int64_t* pair_ptr, int64_t n_pairs_total,
                    int64_t* edge_index, float* x_ind, int64_t* node_types, int64_t* batch, csmpn_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* CSMPN_B200_H_ */
