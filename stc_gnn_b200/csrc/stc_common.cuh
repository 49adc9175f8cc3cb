// Internal helpers shared by the libstc_b200 translation units (not part of the C ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>

#include "../../include/stc_b200.h"

namespace stc {

// ---- error plumbing (thread-local message + launch counter) -------------------------------------
void set_error(const char* fmt, ...);
void count_launch(int n = 1);
void reset_launch_count();

#define STC_CUDA_OK(expr)                                                                   \
  do {                                                                                      \
    cudaError_t _e = (expr);                                                                \
    if (_e != cudaSuccess) {                                                                \
      stc::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return STC_ERR_CUDA;                                                                  \
    }                                                                                       \
  } while (0)

#define STC_LAUNCH_OK(name)                                                                 \
  do {                                                                                      \
    cudaError_t _e = cudaGetLastError();                                                    \
    if (_e != cudaSuccess) {                                                                \
      stc::set_error("launch of %s failed: %s (%s:%d)", name, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return STC_ERR_CUDA;                                                                  \
    }                                                                                       \
    stc::count_launch();                                                                    \
  } while (0)

#define STC_TRY(expr)            \
  do {                           \
    int _s = (expr);             \
    if (_s != STC_OK) return _s; \
  } while (0)

// ---- optional per-kernel timing (stc_timing_* in the ABI) ---------------------------------------
enum KernelKind {
  KK_SUPPORT_DENSE = 0, KK_SUPPORT_CSR, KK_SUPPORT_OUTER, KK_CHEBY_SMALL, KK_CONV_FWD, KK_CONV_BWD_DX,
  KK_CONV_BWD_DW, KK_TC_CONV_FWD, KK_TC_CONV_BWD_DX, KK_TC_CONV_BWD_DW, KK_TC_SUPPORT, KK_TC_GEMM_TEST, KK_TC_OUTER, KK_TC_SUPPORT_BIG,
  KK_SUPPORT_CSR_GRAD, KK_PAIR_SCORES_CSR, KK_EDGE_SOFTMAX, KK_PAIR_TOPK, KK_COUNT
};
struct ScopedKernelTimer {  // declare right before a launch; the destructor records the stop event
  ScopedKernelTimer(int kind, cudaStream_t st, double alg_bytes);
  ~ScopedKernelTimer();
  cudaEvent_t e0, e1;   // owned by the timer until the destructor hands the pair to the record (nullptr = not timing)
  int kind;
  double bytes;
  cudaStream_t st;
};

static inline size_t round_up(size_t x, size_t m) { return (x + m - 1) / m * m; }
static inline int ceil_div(long long a, long long b) { return (int)((a + b - 1) / b); }

// exact division of a 32-bit unsigned by a launch-invariant divisor: multiply-high + one correction step
// (M = floor((2^(32+s) - 1) / d), s = floor(log2 d): the estimate is q or q - 1 for every n < 2^32)
struct FastDiv {
  uint32_t d, M, s;
};
static inline FastDiv make_fastdiv(uint32_t d) {
  FastDiv f;
  f.d = d ? d : 1;
  f.s = 0;
  while ((2u << f.s) <= f.d && f.s < 31) ++f.s;
  f.M = (uint32_t)(((((uint64_t)1) << (32 + f.s)) - 1) / f.d);
  return f;
}
#ifdef __CUDACC__
__device__ __forceinline__ uint32_t fast_div(uint32_t n, const FastDiv f) {
  if (f.d == 1) return n;
  uint32_t q = __umulhi(n, f.M) >> f.s;
  if (n - q * f.d >= f.d) ++q;
  return q;
}
#endif

int device_sm_count();   // cached, current device
int check_arch();        // STC_OK when the current device is compute capability 10.x

// ---- workspace layout of one cell call (offsets in floats) -------------------------------------
struct WsLayout {
  size_t R;  // B*N*C rows
  // `saved` buffer (written by forward, read by backward)
  size_t u, r, c, Yr, Yx, Yh, Q, Pg, Pc, Wimg_g, Wimg_c, saved_total;
  // backward `scratch` buffer
  size_t dpre, dYx0, dYx, dYh, dYr, dQ, Wimg_dx, scratch_total;
};
WsLayout make_layout(const StcDims& d);

// ---- launchers implemented in the kernel TUs -----------------------------------------------------
int launch_support_apply(const StcSupport& gs, int N, int B, int width, bool transpose, const float* x,
                         int64_t x_bs, const float* z, int64_t z_bs, float* y, float alpha, float beta,
                         float* axpy_out, float axpy_coef, cudaStream_t st, const int32_t* row_list = nullptr,
                         int n_list = 0);
// halo rows of the row-partitioned path: pack (gather x_ext[b][idx[j]] -> buf[j][b]) or unpack (buf -> rows row0 + j)
int launch_halo_rows(bool pack, float* x_ext, long long x_bs, int W, int B, const int32_t* idx, int row0, int n_rows,
                     float* buf, cudaStream_t st);

// tcgen05 versions (stc_support_tc.cu): STC_OK and *handled when they took the launch
int try_launch_support_tc(const float* G, int N, int B, int width, bool transpose, const float* x, int64_t x_bs,
                          const float* z, int64_t z_bs, float* y, float alpha, float beta, cudaStream_t st,
                          bool* handled);
// dense N > 128 (stc_support_tc_big.cu)
int try_launch_support_tc_big(const float* G, int N, int B, int width, bool transpose, const float* x, int64_t x_bs,
                              const float* z, int64_t z_bs, float* y, float alpha, float beta, cudaStream_t st,
                              bool* handled);
int try_launch_outer_tc(int N, int B, int width, const float* a, int64_t a_bs, const float* bmat, float coef, float* dG,
                        cudaStream_t st, bool* handled);

// adjoint hop y = alpha * Gs x + beta * z (+ the Chebyshev axpy) of a CSR support with the edge-value gradient fused in:
// dvals[e = (n,m)] += coef * sum_{b,j} a[b,n,j] * x[b,m,j]  (dvals in the order of gs.rowptr / gs.col / gs.vals).
// row_list != nullptr: only the n_list rows n it names are computed, and only their edges get a gradient.
int launch_support_csr_edge_grad(const StcSupport& gs, int N, int B, int width, const float* x, int64_t x_bs,
                                 const float* z, int64_t z_bs, float* y, float alpha, float beta, float* axpy_out,
                                 float axpy_coef, const float* a, int64_t a_bs, float coef, float* dvals,
                                 cudaStream_t st, const int32_t* row_list = nullptr, int n_list = 0);

int launch_support_outer(int N, int B, int width, const float* a, int64_t a_bs, const float* bmat, float coef,
                         float* dG, cudaStream_t st);

// graph generator on a fixed CSR pattern (stc_pair_graph.cu): scores S[e = (n,m)] = <U_n,V_m> - <V_n,U_m> and the
// softmax of relu(S) over each row's stored edges (bwd: dS from S, P, dP into `out`)
int launch_pair_scores_csr(const int32_t* rowptr, const int32_t* col, long long nnz, int N, long long width,
                           const float* u, const float* v, float* scores, cudaStream_t st);
// the same restricted to the rows listed in rows[n_rows] (the others are not written); u, v rows are ld >= width apart
int launch_pair_scores_csr_rows(const int32_t* rowptr, const int32_t* col, long long nnz, int N, long long width,
                                long long ld, const float* u, const float* v, float* scores, const int32_t* rows,
                                int n_rows, cudaStream_t st);
int launch_edge_softmax(bool bwd, const int32_t* rowptr, long long nnz, int N, const float* s, const float* p,
                        const float* dp, float* out, cudaStream_t st);
// top-k pair scores over all columns (stc_pair_topk.cu); arguments checked by the caller (1 <= k <= min(N, 32),
// width % 4 == 0, u / v 16-byte aligned, ws of pair_topk_ws_bytes)
size_t pair_topk_ws_bytes(int N, int k);
int launch_pair_topk(int N, int width, const float* u, const float* v, int k, int32_t* cols, float* scores, void* ws,
                     cudaStream_t st);

int launch_cheby_small(const float* G, int C, int K, float* Q, cudaStream_t st);
int launch_cheby_small_bwd(const float* G, const float* Q, float* dQ, int C, int K, float* dG, cudaStream_t st);

struct ConvArgs {
  // shape
  int B, N, C, Din, h, Ks, Kc, Hout, act, phase;  // phase 0 = gates conv, 1 = candidate conv
  // feature sources: x-part (k = 0 from x0, k >= 1 from yx[k-1]) and h-part (h0 / yh[k-1])
  const float* x0;
  long long x0_bs;
  const float* yx;
  const float* h0;
  const float* yh;
  const float* W;     // [(Ks*Kc*L)][Hout]
  const float* bias;  // [Hout] or null
  const float* Q;     // [Kc][C][C]
  // forward epilogue
  const float* Hprev;
  float* u;
  float* r;
  float* rH;
  float* c;
  float* Hnew;
  float* Psave;        // [R][(Kc-1)*Hout]: pre-mix partial outputs P_c, c >= 1 (tcgen05 path, for dGc)
  float* Wimg;         // wide-hidden-state forward (stc_conv_tc_big.cu): scratch for the split, pre-swizzled weights
  // backward inputs / outputs
  const float* dHn;
  const float* drH;    // gates phase: adjoint of r*H
  float* dpre;         // [R][dpre_ld] scratch written by dx, read by dw: columns [0,Hout) = pre-activation gradient;
                       // on the tcgen05 path dpre_ld = Kc*Hout and block c >= 1 holds its T_c(Gc)-unmixed copy
  int dpre_ld;
  float* dbias;        // atomically accumulated, or null
  float* dYx0;         // k = 0 x-part adjoint destination
  float* dYx;          // k >= 1
  int accum_x;         // add into dYx* instead of overwrite (gates phase after candidate phase)
  float* dYh0;         // k = 0 h-part adjoint destination (d_h_prev for gates, d(rH) for candidate)
  float* dYh;          // k >= 1
  // adjoints another cell folds into this one's terms k >= 1 (the cell that hopped a shared hidden state once for both
  // of its readers, stack.py): the x-part starts from dYx_add (candidate phase, accum_x == 0), the h-part written by the
  // gates phase adds dYh_add; null = nothing to fold
  const float* dYx_add;   // [Ks-1][R][Din]
  const float* dYh_add;   // [Ks-1][R][h]
  float* dQ;          // [Kc][C][C] atomically accumulated, or null
  float* dW;           // atomically accumulated
  // tuning switches (STC_OPT environment bit mask, default all on) and the optional phase trace (stc_debug_trace_set)
  int opt;
  long long* trace;    // [trace_tiles][TRACE_SLOTS] clock64 stamps of CTA 0's first tiles, or null
  int trace_tiles;
};
enum { OPT_L2_PREFETCH = 1, OPT_GENERIC_EPILOGUE = 4 /* diagnostic: force the general epilogues */,
       OPT_SMEM_A = 8 /* diagnostic: convolutions with the A operand staged in shared memory */,
       OPT_WIDE_DX_FFMA = 32 /* diagnostic: wide-state backward dx on the general path */ };
constexpr int TRACE_SLOTS = 16;
int conv_opt_flags();                                  // cached STC_OPT (default: OPT_L2_PREFETCH)
void conv_trace_target(long long** buf, int* tiles);   // what stc_debug_trace_set registered (null when off)
int launch_tf32x3_gemm(const float* A, const float* Bm, float* D, int M, int N, int K, cudaStream_t st);
int launch_conv_fwd(const ConvArgs& a, cudaStream_t st);
// wide hidden states (h >= 32, Kc = 2): streamed-weight tcgen05 forward (stc_conv_tc_big.cu)
bool conv_big_shape_ok(int C, int Din, int h, int Ks, int Kc, int Hout);
size_t conv_big_img_floats(int C, int Din, int h, int Ks, int Kc, int Hout);   // 0 when the shape is not eligible
int try_launch_conv_fwd_big(const ConvArgs& a, cudaStream_t st, bool* handled);
size_t conv_big_dx_img_floats(int C, int Din, int h, int Ks, int Kc, int Hout);
int try_launch_conv_bwd_dx_big(const ConvArgs& a, cudaStream_t st, bool* handled);
bool conv_big_bwd_shape_ok(int C, int Din, int h, int Ks, int Kc, int Hout);   // wide-state dx + dW kernels tile this shape
int try_launch_conv_bwd_dw_big(const ConvArgs& a, cudaStream_t st, bool* handled);
bool conv_tc_eligible(const ConvArgs& a);  // shape-only test shared by forward and backward
bool conv_tc_dw_shape_ok(const ConvArgs& a);  // additionally: the tensor-core dW kernel tiles this shape
int launch_conv_bwd_dx(const ConvArgs& a, cudaStream_t st);
int launch_conv_bwd_dw(const ConvArgs& a, cudaStream_t st);

}  // namespace stc
