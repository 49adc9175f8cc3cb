/* stc_b200.h -- C ABI of libstc_b200.so: the B200 (sm_100a) implementation of STC-GNN's
 * per-timestep spatio-temporal-categorical graph-convolution GRU cell.
 *
 * What it replaces (reference = underdoc-wang/STC-GNN, framework/STC_GNN.py):
 *   STC_Cell.forward                STC_GNN.py:65-79   -> stc_cell_fwd
 *   BDG_Dif.forward (x2 per cell)   STC_GNN.py:31-47   -> inside stc_cell_fwd
 *   BDG_Dif.cheby_poly              STC_GNN.py:24-29   -> inside (feature-side recurrence for Gs,
 *                                                         matrix-space for the small Gc)
 *   autograd of the above           Model_Trainer.py:81 (loss.backward()) -> stc_cell_bwd
 *
 * Conventions
 *   - plain C types only; every pointer is a DEVICE pointer unless it says "host".
 *   - all tensors are fp32, row-major, feature axis fastest:  X[b][n][c][l].
 *   - the library never allocates or frees device memory.  The forward pass writes what backward
 *     needs into `saved` (size from stc_cell_saved_bytes; keep it untouched until stc_cell_bwd has
 *     run -- it is the autograd node's "saved tensors"); backward additionally takes `scratch`
 *     (size from stc_cell_bwd_scratch_bytes) which may be reused by any later call.
 *   - launches go to `stream` (a cudaStream_t passed as void*); no host synchronisation inside.
 *   - return value: 0 on success, a negative StcStatus otherwise; stc_last_error() gives the text
 *     (thread-local).  Nothing throws across the boundary.  There is no CPU fallback.
 */
#ifndef STC_B200_H_
#define STC_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define STC_ABI_VERSION 7

typedef enum {
  STC_OK = 0,
  STC_ERR_BAD_ARG = -1,      /* null pointer, non-positive size, bad enum */
  STC_ERR_UNSUPPORTED = -2,  /* shape outside what the kernels tile (message says which) */
  STC_ERR_WORKSPACE = -3,    /* saved/scratch buffer smaller than the *_bytes() query says */
  STC_ERR_CUDA = -4,         /* a CUDA runtime call or launch failed */
  STC_ERR_ARCH = -5          /* device is not compute capability 10.x */
} StcStatus;

enum { STC_ACT_NONE = 0, STC_ACT_RELU = 1 };          /* BDG_Dif(activation=...), STC_GNN.py:13,46 */
enum { STC_SUPPORT_DENSE = 0, STC_SUPPORT_CSR = 1 };

/* Static shape of one cell call.  Mirrors STC_Cell.__init__ (STC_GNN.py:52-58) plus the batch. */
typedef struct {
  int32_t B;        /* batch                                  */
  int32_t N;        /* num_nodes  (regions)                   */
  int32_t C;        /* num_categories (incident types)        */
  int32_t Din;      /* input_dim of Xt                        */
  int32_t h;        /* hidden_dim                             */
  int32_t Ks;       /* number of spatial Chebyshev terms  (orders 0..Ks-1) */
  int32_t Kc;       /* number of categorical Chebyshev terms               */
  int32_t act;      /* STC_ACT_*                              */
  int32_t has_bias; /* use_bias                               */
} StcDims;

/* Spatial support Gs [N,N].  The forward pass contracts over Gs's FIRST index
 * ('bncl,nm->bmcl', STC_GNN.py:37), i.e. applies Gs^T; backward applies Gs.
 *   dense: vals = Gs row-major [N][N]  (vals[n*N+m] = Gs[n,m]); the other fields are ignored.
 *   CSR  : (rowptr, col, vals) is Gs in CSR (row n lists the m with Gs[n,m] != 0, used by backward),
 *          (t_rowptr, t_col, t_vals) is Gs^T in CSR (row m lists the n, used by forward).
 *          Column indices are int32; nnz < 2^31.
 *          The edge values may be learned: stc_cell_bwd then returns their gradient in Gs-CSR order (the order of
 *          `vals`, [nnz]) through its dGs argument; the sparsity pattern itself is fixed.  An edge stored with the
 *          value 0 is still an edge and gets a gradient. */
typedef struct {
  int32_t kind;
  int64_t nnz;
  const float* vals;
  const int32_t* rowptr;
  const int32_t* col;
  const float* t_vals;
  const int32_t* t_rowptr;
  const int32_t* t_col;
} StcSupport;

int stc_abi_version(void);
const char* stc_last_error(void);

/* Bytes of the `saved` buffer of one cell call (forward intermediates; also the forward's scratch). */
size_t stc_cell_saved_bytes(const StcDims* d);
/* Bytes of the `scratch` buffer stc_cell_bwd needs. */
size_t stc_cell_bwd_scratch_bytes(const StcDims* d);

/* H' = STC_Cell(Gs, Gc, Xt, H)                                             STC_GNN.py:65-79
 *   gc        [C][C]
 *   xt        [B][N][C][Din], inner [N][C][Din] slab contiguous, batch stride xt_batch_stride ELEMENTS
 *             (the encoder hands in a [:,t] view: STC_GNN.py:111)
 *   h_prev    [B][N][C][h] contiguous
 *   Wg        [(Din+h)*Ks*Kc][2h]  rows ordered (n, c, l)  (STC_GNN.py:17,35-41);  bg [2h] or NULL
 *   Wc        [(Din+h)*Ks*Kc][h];                                                   bc [h]  or NULL
 *   h_out     [B][N][C][h] contiguous, must not alias an input                                   */
int stc_cell_fwd(const StcDims* d, const StcSupport* gs, const float* gc,
                 const float* xt, int64_t xt_batch_stride, const float* h_prev,
                 const float* Wg, const float* bg, const float* Wc, const float* bc,
                 float* h_out, void* saved, size_t saved_bytes, void* stream);

/* ---- the cell split at its spatial-support stages (row-partitioned graphs, stc_gnn_b200/halo.py) ----
 * A rank that owns a block of nodes cannot run the spatial hops inside stc_cell_fwd: each hop needs the
 * boundary-node features of its neighbours (an NCCL halo exchange).  The caller therefore
 *   1. fills the spatial terms of Xt and H (regions STC_SAVED_YX, STC_SAVED_YH of `saved`, Ks-1 terms each,
 *      [B][N][C][Din or h] contiguous) with stc_support_apply + its exchange,
 *   2. calls stage STC_STAGE_GATES  (node-local: Gc terms, gates conv, writes u, r and r*H = term 0 of STC_SAVED_YR),
 *   3. fills terms 1..Ks-1 of STC_SAVED_YR the same way,
 *   4. calls stage STC_STAGE_CANDI  (node-local: candidate conv, tanh, GRU blend -> h_out).
 * d->N is the number of LOCAL nodes.  stc_cell_saved_layout writes the offset (in floats) of every region of
 * `saved` into offsets[STC_SAVED_REGIONS]. */
enum { STC_STAGE_GATES = 0, STC_STAGE_CANDI = 1 };
enum { STC_SAVED_U = 0, STC_SAVED_R, STC_SAVED_C, STC_SAVED_YR, STC_SAVED_YX, STC_SAVED_YH, STC_SAVED_Q,
       STC_SAVED_PG, STC_SAVED_PC, STC_SAVED_REGIONS };
int stc_cell_saved_layout(const StcDims* d, int64_t* offsets_floats, int32_t n_offsets);
int stc_cell_fwd_stage(const StcDims* d, int32_t stage, const float* gc,
                       const float* xt, int64_t xt_batch_stride, const float* h_prev,
                       const float* Wg, const float* bg, const float* Wc, const float* bc,
                       float* h_out, void* saved, size_t saved_bytes, void* stream);

/* Gradients of stc_cell_fwd given d_h_out.  `saved` is the buffer the matching forward call filled.
 *   d_xt      [B][N][C][Din] contiguous, or NULL when Xt needs no gradient
 *   d_h_prev  [B][N][C][h]
 *   dWg,dbg,dWc,dbc  same shapes as the parameters (dbg/dbc NULL when has_bias == 0)
 *   dGs       dense support: [N][N];  CSR support: [nnz], the gradient w.r.t. the edge values `vals` (Gs-CSR
 *             order), computed inside the adjoint hops (stc_support_apply_edge_grad);  NULL: no support gradient
 *   dGc       [C][C] or NULL
 *   accumulate_params != 0: parameter/support gradients are ADDED to the buffers' contents
 *   (lets a time loop accumulate dW over steps); == 0: they are overwritten.
 *   d_xt / d_h_prev are always overwritten.                                                     */
int stc_cell_bwd(const StcDims* d, const StcSupport* gs, const float* gc,
                 const float* xt, int64_t xt_batch_stride, const float* h_prev,
                 const float* Wg, const float* Wc, const float* d_h_out,
                 float* d_xt, float* d_h_prev,
                 float* dWg, float* dbg, float* dWc, float* dbc, float* dGs, float* dGc,
                 int32_t accumulate_params, const void* saved, size_t saved_bytes,
                 void* scratch, size_t scratch_bytes, void* stream);

/* ---- spatial terms computed once for two readers (SURVEY 8f row f1; stc_gnn_b200/stack.py) ----
 * The encoder's first layer produces the Xt-side terms of ALL timesteps with one batched stc_support_apply
 * (STC_GNN.py:107-118: Xt does not depend on the recurrence), and every hidden state of the recurrent stack is read by
 * two cells, one as Xt and one as H, whose terms Y_k = T_k(Gs^T) Y_0 are the same bytes.  Per side (Xt, H):
 *   y?_terms      [Ks-1][B][N][C][Din or h] contiguous = Y_1 .. Y_{Ks-1} of that side's input (NULL: computed inside, as
 *                 stc_cell_fwd / stc_cell_bwd do); the forward then launches no hop for that side, and the backward
 *                 reads the same terms (they must be unchanged).
 *   dy?_terms_out [Ks-1][B][N][C][Din or h] (with y?_terms): stc_cell_bwd_x writes the adjoints of the supplied terms
 *                 there and does NOT fold them: no adjoint hop and no dGs contribution is launched for that side, and
 *                 d_xt / d_h_prev holds the term-0 part only.  The caller folds them: the _XSideTerms path with
 *                 stc_support_outer / stc_support_apply (stc_support_apply_edge_grad for learned CSR values), the cell
 *                 that produced shared terms through its own dy?_fold.  NULL: the adjoints are dropped (an input whose
 *                 terms are known and needs no gradient, e.g. a zero initial state).
 *   dy?_fold      [Ks-1][B][N][C][Din or h] (without y?_terms): adjoints of this call's OWN terms of that side, from
 *                 another reader of them.  They are added to the adjoints the convolutions produce (in the dx
 *                 epilogue) before that side's adjoint chain runs, so one hop and one dGs product serve both readers.
 * The stc_cell_saved_layout regions Yx / Yh of a call that computed them hold that side's terms. */
int stc_cell_fwd_x(const StcDims* d, const StcSupport* gs, const float* gc,
                   const float* xt, int64_t xt_batch_stride, const float* h_prev,
                   const float* Wg, const float* bg, const float* Wc, const float* bc,
                   float* h_out, void* saved, size_t saved_bytes, const float* yx_terms, const float* yh_terms,
                   void* stream);
int stc_cell_bwd_x(const StcDims* d, const StcSupport* gs, const float* gc,
                   const float* xt, int64_t xt_batch_stride, const float* h_prev,
                   const float* Wg, const float* Wc, const float* d_h_out,
                   float* d_xt, float* d_h_prev,
                   float* dWg, float* dbg, float* dWc, float* dbc, float* dGs, float* dGc,
                   int32_t accumulate_params, const void* saved, size_t saved_bytes,
                   void* scratch, size_t scratch_bytes, const float* yx_terms, float* dyx_terms_out,
                   const float* dyx_fold, const float* yh_terms, float* dyh_terms_out, const float* dyh_fold,
                   void* stream);
/* dGs[n][m] += coef * sum_{b,j} A[b][n][j] * Bm[b][m][j]  -- the gradient of the mode product Y = Gs^T X w.r.t. a dense
 * Gs [N][N] with A = X ([B][N][width], batch stride in elements) and Bm = dL/dY ([B][N][width] contiguous). */
int stc_support_outer(int32_t N, int32_t B, int32_t width, const float* a, int64_t a_batch_stride, const float* b,
                      float coef, float* dGs, void* stream);
/* The same gradient for a CSR support, sampled at its edges and fused into the adjoint hop (CSR only):
 *   y = alpha * Gs x + beta * z                                    (exactly what stc_support_apply, transpose = 0, writes)
 *   dvals[e] += coef * sum_{b,j} a[b][row(e)][j] * x[b][col(e)][j] (e walks Gs's CSR: rowptr / col / vals order)
 * x, z, y as in stc_support_apply; a [B][N][width] with its own batch stride (elements); dvals [nnz] is only added
 * to.  It is what stc_cell_bwd runs for every adjoint hop when it is handed dGs for a CSR support. */
int stc_support_apply_edge_grad(const StcSupport* gs, int32_t N, int32_t B, int32_t width,
                                const float* x, int64_t x_batch_stride, const float* z, int64_t z_batch_stride,
                                float* y, float alpha, float beta, const float* a, int64_t a_batch_stride, float coef,
                                float* dvals, void* stream);
/* The same fused hop restricted to the rows n listed in rows[n_rows] (int32, device), like stc_support_apply_rows:
 * only those rows of y are written (the others are not touched), only the edges of those rows get a gradient, and a
 * is read at those rows only.  The row-partitioned path (stc_gnn_b200/halo.py) runs it on the interior rows while the
 * halo exchange is in flight, then on the boundary rows, when the partitioned support's edge values are learned. */
int stc_support_apply_rows_edge_grad(const StcSupport* gs, int32_t N, int32_t B, int32_t width,
                                     const float* x, int64_t x_batch_stride, const float* z, int64_t z_batch_stride,
                                     float* y, float alpha, float beta, const float* a, int64_t a_batch_stride,
                                     float coef, float* dvals, const int32_t* rows, int32_t n_rows, void* stream);

/* ---- graph generator on a fixed CSR pattern (the sparse form of MGP_Gen's spatial half, STC_GNN.py:227-233) ----
 * gs is a CSR support whose rowptr / col give the pattern; its vals (and the Gs^T fields) are ignored.
 * u, v [N][width] row-major (node-major: width = B*T*hg, the generator's tanh(alpha X Wu), tanh(alpha X Wv)).
 * stc_pair_scores_csr:  scores[e] = <u[n], v[m]> - <v[n], u[m]>  for every stored edge e = (n, m), in Gs-CSR order
 *                       (M[n,m] - M[m,n] of the dense generator at the stored edges; a self-loop scores exactly 0).
 * stc_edge_softmax_fwd: p[e] = exp(relu(scores[e]) - max) / sum over the stored edges e' of row n of
 *                       exp(relu(scores[e']) - max); entries off the pattern take no part; an empty row writes nothing.
 * stc_edge_softmax_bwd: dscores[e] = [scores[e] > 0] * p[e] * (dp[e] - sum_{e' in row n} p[e'] dp[e']).
 * All three are deterministic (no atomics: a second call gives bitwise the same output).  The gradient of the scores
 * needs no export: with D = the pattern carrying dscores, du = (D - D^T) v and dv = (D^T - D) u, two
 * stc_support_apply hops each (transpose = 0 walks D, transpose = 1 walks D^T). */
int stc_pair_scores_csr(const StcSupport* gs, int32_t N, int64_t width, const float* u, const float* v,
                        float* scores, void* stream);
/* stc_pair_scores_csr restricted to the rows n listed in rows[n_rows] (int32, device): only the scores of those rows'
 * edges are written (every other entry of `scores` is not touched), each bitwise what stc_pair_scores_csr writes for
 * it.  u and v rows are ld >= width floats apart (u[n] = u + n * ld), so U and V may be the two halves of one
 * [N][2 * width] buffer.  Rejects ld < width; n_rows == 0 launches nothing.  The row-partitioned generator
 * (stc_gnn_b200/sparse_mgp.py) scores the rows of its local operator whose neighbours are all local while the halo
 * exchange of [U | V] is in flight, then the others. */
int stc_pair_scores_csr_rows(const StcSupport* gs, int32_t N, int64_t width, int64_t ld, const float* u, const float* v,
                             float* scores, const int32_t* rows, int32_t n_rows, void* stream);
int stc_edge_softmax_fwd(const StcSupport* gs, int32_t N, const float* scores, float* p, void* stream);
int stc_edge_softmax_bwd(const StcSupport* gs, int32_t N, const float* scores, const float* p, const float* dp,
                         float* dscores, void* stream);

/* Top-k pair scores of the graph generator over ALL candidate columns (no pattern):
 *   S[n][m] = <u[n], v[m]> - <v[n], u[m]>  (3xTF32, S[n][n] = 0 exactly), u, v [N][width] row-major, width % 4 == 0,
 *   u, v and ws 16-byte aligned.
 *   cols[n][0..k)  the k columns of row n with the largest S (ties: smaller column), ascending;  scores [N][k] the
 *   matching S values (may be NULL).  A NaN score (NaN or inf in u / v) ranks, and is reported, as -inf; cols always
 *   holds k distinct columns in [0, N).  1 <= k <= min(N, 32); k > 32 returns STC_ERR_UNSUPPORTED.  Deterministic: the
 *   output is bitwise the same on every call.  Nothing of size N^2 is formed: each row's best columns are kept on chip
 *   while the column tiles stream.  ws: at least stc_pair_topk_workspace_bytes(N, width, k) bytes of scratch (0 for
 *   arguments stc_pair_topk would reject).  The size depends on the SM count of the current device: query it with the
 *   device current on which stc_pair_topk will run.  The sparse generator (stc_gnn_b200/sparse_mgp.py topk_pattern) builds its
 *   k-regular pattern from cols. */
size_t stc_pair_topk_workspace_bytes(int32_t N, int64_t width, int32_t k);
int stc_pair_topk(int32_t N, int64_t width, const float* u, const float* v, int32_t k,
                  int32_t* cols, float* scores, void* ws, size_t ws_bytes, void* stream);

/* stc_pair_topk for the query rows [row0, row0 + n_rows) only, scored against all N columns: cols / scores are
 * [n_rows][k] (global column ids), row i holding row row0 + i of the full selection, bitwise (the K-chain order and the
 * column tiling do not depend on the rows selected; the segment merge is a total order on (score, column)).  u, v are
 * the full [N][width] operands.  0 <= row0, row0 + n_rows <= N; row0 need not be a multiple of 128.  n_rows == 0
 * launches nothing and reads no other argument.  The segment count comes from the number of 128-row blocks, so a block
 * of N / 8 rows still fills the device.  ws: at least stc_pair_topk_rows_workspace_bytes(N, width, n_rows, k) bytes
 * (sized for n_rows; 0 for n_rows == 0 and for arguments stc_pair_topk_rows would reject), queried on the device it
 * runs on.  Every argument check returns before a launch.  The row-partitioned generator (stc_gnn_b200/sparse_mgp.py)
 * selects each rank's own rows with it. */
size_t stc_pair_topk_rows_workspace_bytes(int32_t N, int64_t width, int32_t n_rows, int32_t k);
int stc_pair_topk_rows(int32_t N, int64_t width, const float* u, const float* v, int32_t row0, int32_t n_rows,
                       int32_t k, int32_t* cols, float* scores, void* ws, size_t ws_bytes, void* stream);

/* ---- the backward split the same way (gradients through a row-partitioned graph) ----
 * Order: stage STC_STAGE_CANDI first, then STC_STAGE_GATES (the reverse of the forward).
 *   1. STC_STAGE_CANDI: clears the parameter and Gc gradients unless accumulate_params, runs the candidate-conv adjoint.  Leaves
 *      d(r*H spatial terms) in region STC_SCRATCH_DYR of `scratch` (Ks terms, [B][N][C][h] each), the x-part adjoint
 *      of term 0 in d_xt and of terms 1..Ks-1 in region STC_SCRATCH_DYX.
 *   2. the caller folds terms Ks-1..1 of STC_SCRATCH_DYR into term 0 with the adjoint hops
 *      (ybar[k-1] += (k >= 2 ? 2 : 1) Gs ybar[k], ybar[k-2] -= ybar[k]; stc_support_apply with transpose = 0 + its exchange),
 *   3. STC_STAGE_GATES: GRU adjoint + gates-conv adjoint (reads term 0 of STC_SCRATCH_DYR as d(r*H)); adds its x-part
 *      adjoints to d_xt / STC_SCRATCH_DYX, writes the h-part adjoints to d_h_prev / STC_SCRATCH_DYH (Ks-1 terms),
 *      finishes dGc,
 *   4. the caller folds STC_SCRATCH_DYX into d_xt and STC_SCRATCH_DYH into d_h_prev the same way.
 * Rows whose d_h_out and STC_SCRATCH_DYR term-0 entries are zero contribute nothing to any parameter gradient (that
 * is how the halo rows of an extended node set are kept out of dW).  The stages take no dGs: when the support's edge
 * values are learned, the caller forms their gradient inside its adjoint hops (steps 2 and 4) with
 * stc_support_apply_edge_grad / stc_support_apply_rows_edge_grad, A = the matching forward terms of `saved`.      */
enum { STC_SCRATCH_DYR = 0, STC_SCRATCH_DYX, STC_SCRATCH_DYH, STC_SCRATCH_REGIONS };
int stc_cell_bwd_scratch_layout(const StcDims* d, int64_t* offsets_floats, int32_t n_offsets);
int stc_cell_bwd_stage(const StcDims* d, int32_t stage, const float* gc,
                       const float* xt, int64_t xt_batch_stride, const float* h_prev,
                       const float* Wg, const float* Wc, const float* d_h_out,
                       float* d_xt, float* d_h_prev,
                       float* dWg, float* dbg, float* dWc, float* dbc, float* dGc,
                       int32_t accumulate_params, const void* saved, size_t saved_bytes,
                       void* scratch, size_t scratch_bytes, void* stream);

/* Y[b,m,:] = alpha * sum_n A(m,n) X[b,n,:] + beta * Z[b,m,:]  with A = Gs^T (transpose != 0, the
 * forward mode product of STC_GNN.py:37) or A = Gs.  X,Z,Y: [B][N][width]; X and Z may carry a batch
 * stride (elements), Y is contiguous; Z may be NULL when beta == 0; Y may alias Z.  Exposed because it
 * is the support kernel the roofline is quoted on, and the building block of the halo-partitioned path. */
int stc_support_apply(const StcSupport* gs, int32_t N, int32_t B, int32_t width, int32_t transpose,
                      const float* x, int64_t x_batch_stride, const float* z, int64_t z_batch_stride,
                      float* y, float alpha, float beta, void* stream);

/* The same product restricted to the output nodes listed in rows[n_rows] (int32, device): the other rows of Y are
 * not touched.  CSR supports only.  The row-partitioned path (stc_gnn_b200/halo.py, SURVEY 8e) computes the rows whose
 * neighbours are all local while the halo exchange of the hop is in flight, then the boundary rows. */
int stc_support_apply_rows(const StcSupport* gs, int32_t N, int32_t B, int32_t width, int32_t transpose,
                           const float* x, int64_t x_batch_stride, const float* z, int64_t z_batch_stride,
                           float* y, float alpha, float beta, const int32_t* rows, int32_t n_rows, void* stream);

/* Halo rows of a row-partitioned hop.  x_ext is an extended tensor [B][nloc + nhalo][width] (batch stride in
 * elements).  pack: send[j][b][:] = x_ext[b][idx[j]][:] for the n_rows local boundary nodes idx (int32, device;
 * grouped by destination rank, so `send` is the input of one all-to-all with row counts as split sizes);
 * unpack: x_ext[b][row0 + j][:] = recv[j][b][:] (row0 = nloc: the halo rows, ordered by owner rank). */
int stc_halo_pack(const float* x_ext, int64_t x_batch_stride, int32_t width, int32_t B, const int32_t* idx,
                  int32_t n_rows, float* send, void* stream);
int stc_halo_unpack(const float* recv, int32_t width, int32_t B, int32_t row0, int32_t n_rows, float* x_ext,
                    int64_t x_batch_stride, void* stream);

/* Building block self-test / microbenchmark: D[M][N] = A[M][K] * B[K][N], row-major fp32, evaluated as a
 * 3xTF32 tcgen05 product with TMEM accumulation (the same code path as the gate contraction).  N <= 256. */
int stc_tf32x3_gemm(const float* a, const float* b, float* d, int32_t M, int32_t N, int32_t K, void* stream);

/* Independent kernels of one stc_cell_fwd / stc_cell_bwd call (dW beside the adjoint hops, the dGs outer products, the
 * Xt-side hops beside the H-side hops) may be forked onto internal side streams and are joined back with events
 * before the call returns; by default only for problems too small to fill the device.  mode: -1 = by problem size
 * (default; the STC_CONCURRENCY environment variable sets the initial value), 0 = always one stream, 1 = always fork. */
int stc_concurrency_set(int32_t mode);

/* Number of kernel launches the last stc_cell_fwd / stc_cell_bwd on this thread issued
 * (bench.py reports gpu_launches from these). */
int stc_last_launch_count(void);

/* Optional per-kernel instrumentation for bench.py's roofline line (off by default; when on, every kernel
 * launch is bracketed by CUDA events on its own stream).  stc_timing_collect synchronises the recorded
 * events, ADDS per-kind device milliseconds / launch counts / algorithmic bytes (the compulsory HBM traffic
 * of each launch, formulas next to each launcher) into the caller's arrays of length n_kinds (host
 * pointers), clears the record and returns the number of kinds the library knows. */
int stc_timing_enable(int32_t on);
int stc_timing_collect(double* ms_by_kind, int64_t* launches_by_kind, double* alg_bytes_by_kind, int32_t n_kinds);
const char* stc_kernel_kind_name(int32_t kind);

/* Diagnostic: while dev_buf (int64 [n_slots], device memory, caller-owned) is registered, CTA 0 of the tcgen05
 * gate-convolution kernels stamps clock64() at its phase boundaries for its first n_slots/32 tiles
 * (16 stamps per tile; the gates convolution uses the first half of the buffer, the candidate convolution the
 * second; tools/trace_conv.py prints the deltas).  Pass NULL to switch it off (the default). */
int stc_debug_trace_set(void* dev_buf, int64_t n_slots);

#ifdef __cplusplus
}
#endif
#endif /* STC_B200_H_ */
