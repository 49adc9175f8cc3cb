// Spatial / categorical support kernels of the general path.
//
//  support_dense_kernel  Y = alpha * A X + beta * Z with A = Gs^T (forward, 'bncl,nm->bmcl',
//                        /root/reference/framework/STC_GNN.py:37) or A = Gs (adjoint, used by backward).
//  support_csr_kernel    same operator for a CSR support (one warp per (batch, node) row slab).  GRAD = true: the
//                        adjoint hop with the gradient of the edge values fused in (learnable CSR supports),
//                        dvals[e = (n,m)] += coef * sum_{b,j} A[b,n,j] * X[b,m,j]; Y is computed exactly as without it.
//                        PS = true: per-sample values (vals [B][nnz]); sample b is hopped with vals + b * nnz and,
//                        with GRAD, its edge gradient goes to dvals + b * nnz (no sum over the batch).
//  support_outer_kernel  dGs[n',m] += coef * sum_{b,j} A[b,n',j] * Bm[b,m,j]  (gradient of the spatial
//                        mode product w.r.t. the support; reference gets it from autograd of :37).
//  cheby_small_*         matrix-space Chebyshev terms of the small C x C categorical support and their
//                        adjoint (STC_GNN.py:24-29 applied to Gc).
#include "stc_common.cuh"

#include <algorithm>

namespace stc {

// ------------------------------------------------------------------------------------------------
// dense support: batched [N x N] x [N x width] with the batch folded into the column index
// ------------------------------------------------------------------------------------------------
constexpr int SD_BM = 64, SD_BQ = 64, SD_BK = 16, SD_THREADS = 256;

template <bool TRANS>
__global__ void __launch_bounds__(SD_THREADS)
support_dense_kernel(const float* __restrict__ G, int N, const float* __restrict__ X, long long x_bs,
                     const float* Z, long long z_bs, float* Y, int W, long long total_q, float alpha,
                     float beta, float* axpy_out, float axpy_coef) {
  __shared__ __align__(16) float As[SD_BK][SD_BM + 4];
  __shared__ __align__(16) float Xs[SD_BK][SD_BQ + 4];
  const int tid = threadIdx.x;
  const int tx = tid % 16, ty = tid / 16;
  const long long q0 = (long long)blockIdx.x * SD_BQ;
  const int m0 = blockIdx.y * SD_BM;

  // this thread always loads the same tile column: precompute its global column offset
  const int lq = tid % SD_BQ;
  const long long myq = q0 + lq;
  const bool q_ok = myq < total_q;
  long long xoff = 0;
  if (q_ok) {
    long long b = myq / W;
    int j = (int)(myq - b * W);
    xoff = b * x_bs + j;
  }
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  for (int k0 = 0; k0 < N; k0 += SD_BK) {
    // A tile -> As[kk][mm] = A(m0+mm, k0+kk)
    if (TRANS) {
      const int mm = tid % SD_BM;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        int kk = tid / SD_BM + i * 4;
        int n = k0 + kk, m = m0 + mm;
        As[kk][mm] = (n < N && m < N) ? G[(long long)n * N + m] : 0.f;
      }
    } else {
      const int kk = tid % SD_BK;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        int mm = tid / SD_BK + i * 16;
        int n = k0 + kk, m = m0 + mm;
        As[kk][mm] = (n < N && m < N) ? G[(long long)m * N + n] : 0.f;
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      int kk = tid / SD_BQ + i * 4;
      int n = k0 + kk;
      Xs[kk][lq] = (q_ok && n < N) ? X[xoff + (long long)n * W] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < SD_BK; ++kk) {
      float4 a = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
      float4 x = *reinterpret_cast<const float4*>(&Xs[kk][tx * 4]);
      float av[4] = {a.x, a.y, a.z, a.w}, xv[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], xv[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    long long q = q0 + tx * 4 + j;
    if (q >= total_q) continue;
    long long b = q / W;
    int col = (int)(q - b * W);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      int m = m0 + ty * 4 + i;
      if (m >= N) continue;
      long long yi = (b * N + m) * (long long)W + col;
      float v = alpha * acc[i][j];
      if (beta != 0.f) v = fmaf(beta, Z[b * z_bs + (long long)m * W + col], v);
      Y[yi] = v;
      if (axpy_out) axpy_out[yi] = fmaf(axpy_coef, X[b * x_bs + (long long)m * W + col], axpy_out[yi]);
    }
  }
}

// out[b][i] += coef * x[b * x_bs + i]  (16 bytes per thread and step; the Chebyshev adjoint's  ybar[k-2] -= ybar[k])
__global__ void __launch_bounds__(256)
axpy_rows_kernel(float* __restrict__ out, const float* __restrict__ x, long long x_bs, float coef, long long per_b4,
                 long long total4) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total4; i += (long long)gridDim.x * blockDim.x) {
    const long long b = i / per_b4, r = i - b * per_b4;
    const float4 xv = *reinterpret_cast<const float4*>(x + b * x_bs + 4 * r);
    float4 o = reinterpret_cast<float4*>(out)[i];
    o.x = fmaf(coef, xv.x, o.x); o.y = fmaf(coef, xv.y, o.y); o.z = fmaf(coef, xv.z, o.z); o.w = fmaf(coef, xv.w, o.w);
    reinterpret_cast<float4*>(out)[i] = o;
  }
}

int launch_axpy_rows(float* out, const float* x, int64_t x_bs, float coef, int N, int B, int width, cudaStream_t st) {
  const long long per_b4 = (long long)N * width / 4, total4 = per_b4 * B;
  const int blocks = (int)std::min<long long>((total4 + 255) / 256, (long long)device_sm_count() * 16);
  axpy_rows_kernel<<<blocks, 256, 0, st>>>(out, x, x_bs, coef, per_b4, total4);
  STC_LAUNCH_OK("axpy_rows_kernel");
  return STC_OK;
}

// ------------------------------------------------------------------------------------------------
// CSR support: one warp per (b, m) output row slab; lanes sweep the contiguous `width` axis
// ------------------------------------------------------------------------------------------------
// Edge-value gradient fused into the hop (GRAD): the warp keeps its own row's slab chunk A[b,n,j0..] in registers; every
// gathered neighbour slab X[b,m,:] is dotted with it, warp-reduced and added to dvals[e] with one atomic per
// (b, column chunk, edge).  That costs one extra read of the row's own slab instead of a second gather of the
// neighbours (a separate sampled dense x dense product).  The hop's accumulators are untouched by it.
struct CsrEdgeGrad {
  const float* a;   // [B][N][W], batch stride a_bs (elements)
  long long a_bs;
  float coef;
  float* dvals;     // [nnz] ([B][nnz] per-sample), in the order of the walked CSR (rowptr / col)
};

template <int VEC, bool GRAD, bool PS = false>
__global__ void __launch_bounds__(256)
support_csr_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                   const float* __restrict__ vals, int N, long long rows_total, const float* __restrict__ X,
                   long long x_bs, const float* Z, long long z_bs, float* Y, int W, float alpha, float beta,
                   float* axpy_out, float axpy_coef, const int32_t* __restrict__ row_list, int n_list,
                   CsrEdgeGrad eg, long long v_bs) {
  // row_list != nullptr: only the n_list output nodes it names are computed (rows_total = B * n_list); the other
  // rows of Y are not touched (the row-partitioned path computes interior rows while the halo exchange is in flight);
  // with GRAD only the edges of the listed rows get a gradient, and A is read at the listed rows only
  constexpr int U = 4;  // independent accumulators per lane per pass
  const int lane = threadIdx.x & 31;
  const long long warp0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long row = warp0; row < rows_total; row += nwarps) {
    const int per_b = row_list ? n_list : N;
    const long long b = row / per_b;
    const int mi = (int)(row - b * per_b);
    const int m = row_list ? row_list[mi] : mi;
    const int e0 = rowptr[m], e1 = rowptr[m + 1];
    const float* xb = X + b * x_bs;
    const float* vb = PS ? vals + b * v_bs : vals;   // (v_bs = nnz: the values and their gradient of sample b)
    float* dvb = (GRAD && PS) ? eg.dvals + b * v_bs : eg.dvals;
    for (int j0 = 0; j0 < W; j0 += 32 * VEC * U) {
      float acc[U][VEC];
#pragma unroll
      for (int u = 0; u < U; ++u)
#pragma unroll
        for (int v = 0; v < VEC; ++v) acc[u][v] = 0.f;
      float ar[GRAD ? U : 1][VEC];   // this row's own slab chunk (GRAD only)
      if (GRAD) {
        const float* arow = eg.a + b * eg.a_bs + (long long)m * W;
#pragma unroll
        for (int u = 0; u < (GRAD ? U : 1); ++u) {
          int j = j0 + (u * 32 + lane) * VEC;
#pragma unroll
          for (int v = 0; v < VEC; ++v) ar[u][v] = 0.f;
          if (j < W) {
            if (VEC == 4) {
              float4 t = *reinterpret_cast<const float4*>(arow + j);
              ar[u][0] = t.x; ar[u][1 % VEC] = t.y; ar[u][2 % VEC] = t.z; ar[u][3 % VEC] = t.w;
            } else {
              ar[u][0] = arow[j];
            }
          }
        }
      }
      for (int e = e0; e < e1; ++e) {
        const float g = vb[e];
        const float* xr = xb + (long long)col[e] * W;
        float dot = 0.f;
#pragma unroll
        for (int u = 0; u < U; ++u) {
          int j = j0 + (u * 32 + lane) * VEC;
          if (j < W) {
            if (VEC == 4) {
              float4 x = *reinterpret_cast<const float4*>(xr + j);
              acc[u][0] = fmaf(g, x.x, acc[u][0]);
              acc[u][1 % VEC] = fmaf(g, x.y, acc[u][1 % VEC]);
              acc[u][2 % VEC] = fmaf(g, x.z, acc[u][2 % VEC]);
              acc[u][3 % VEC] = fmaf(g, x.w, acc[u][3 % VEC]);
              if (GRAD) {
                const int ug = GRAD ? u : 0;
                dot = fmaf(ar[ug][0], x.x, dot);
                dot = fmaf(ar[ug][1 % VEC], x.y, dot);
                dot = fmaf(ar[ug][2 % VEC], x.z, dot);
                dot = fmaf(ar[ug][3 % VEC], x.w, dot);
              }
            } else {
              const float x = xr[j];
              acc[u][0] = fmaf(g, x, acc[u][0]);
              if (GRAD) dot = fmaf(ar[GRAD ? u : 0][0], x, dot);
            }
          }
        }
        if (GRAD) {
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
          if (lane == 0) atomicAdd(dvb + e, eg.coef * dot);
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        int j = j0 + (u * 32 + lane) * VEC;
        if (j >= W) continue;
        long long yi = (b * N + m) * (long long)W + j;
        float out[VEC];
#pragma unroll
        for (int v = 0; v < VEC; ++v) out[v] = alpha * acc[u][v];
        if (beta != 0.f) {
          const float* zr = Z + b * z_bs + (long long)m * W + j;
#pragma unroll
          for (int v = 0; v < VEC; ++v) out[v] = fmaf(beta, zr[v], out[v]);
        }
        if (VEC == 4) {
          *reinterpret_cast<float4*>(Y + yi) = make_float4(out[0], out[1 % VEC], out[2 % VEC], out[3 % VEC]);
        } else {
          Y[yi] = out[0];
        }
        if (axpy_out) {
          const float* xc = xb + (long long)m * W + j;
#pragma unroll
          for (int v = 0; v < VEC; ++v) axpy_out[yi + v] = fmaf(axpy_coef, xc[v], axpy_out[yi + v]);
        }
      }
    }
  }
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// Deterministic form of the edge-value gradient: one warp owns a row n and ALL of its edges' sums, over every sample and
// feature in a fixed order (lane-strided partial sums, then a shuffle tree), so every dvals[e] has exactly one writer:
//   dvals[e = (n, m)] += coef * sum_{b,j} a[b,n,j] * x[b,m,j]
// PS: per-sample values; one warp per (b, n) and one writer per (b, e) of dvals [B][nnz] (no row list), each sample's
// sums in the order the B = 1 call takes them:  dvals[b][e] += coef * sum_j a[b,n,j] * x[b,m,j]
template <bool PS = false>
__global__ void __launch_bounds__(256)
csr_edge_grad_det_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                         const int32_t* __restrict__ row_list, int n_rows, int B, int W, const float* __restrict__ X,
                         long long x_bs, const float* __restrict__ A, long long a_bs, float coef, float* dvals,
                         long long v_bs) {
  const int lane = threadIdx.x & 31;
  const long long warp0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long r = warp0; r < (PS ? (long long)B * n_rows : n_rows); r += nwarps) {
    const int bs = PS ? (int)(r / n_rows) : 0;
    const int n = PS ? (int)(r - (long long)bs * n_rows) : (row_list ? row_list[r] : (int)r);
    float* dv = PS ? dvals + bs * v_bs : dvals;
    for (int e = rowptr[n]; e < rowptr[n + 1]; ++e) {
      const long long m = col[e];
      float dot = 0.f;
      for (int b = PS ? bs : 0; b < (PS ? bs + 1 : B); ++b) {
        const float* ar = A + b * a_bs + (long long)n * W;
        const float* xr = X + b * x_bs + m * W;
        for (int j = lane; j < W; j += 32) dot = fmaf(ar[j], xr[j], dot);
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
      if (lane == 0) dv[e] += coef * dot;
    }
  }
}

// one CSR hop (rp, ci, va walk the rows of the operator applied); eg.dvals != nullptr selects the edge-gradient variant;
// v_bs: the batch stride of va (and of eg.dvals) in floats, 0 for values shared by every sample, nnz for per-sample ones
static int launch_csr(const int32_t* rp, const int32_t* ci, const float* va, long long nnz, int N, int B, int width,
                      const float* x, int64_t x_bs, const float* z, int64_t z_bs, float* y, float alpha, float beta,
                      float* axpy_out, float axpy_coef, const int32_t* row_list, int n_list, const CsrEdgeGrad& eg,
                      cudaStream_t st, long long v_bs = 0) {
  const bool grad = eg.dvals != nullptr;
  long long rows_total = (long long)B * (row_list ? n_list : N);
  bool vec = (width % 4 == 0) && (x_bs % 4 == 0) && (z == nullptr || z_bs % 4 == 0) && aligned16(x) &&
             aligned16(y) && (z == nullptr || aligned16(z)) && (axpy_out == nullptr || aligned16(axpy_out)) &&
             (!grad || (eg.a_bs % 4 == 0 && aligned16(eg.a)));
  int warps_per_block = 8;
  long long want = (rows_total + warps_per_block - 1) / warps_per_block;
  int grid = (int)(want < (long long)device_sm_count() * 16 ? want : (long long)device_sm_count() * 16);
  if (grid < 1) grid = 1;
  // compulsory traffic of the hop; the edge-gradient variant also reads the row's own slab of A and updates dvals
  // (per-sample values: B value vectors and B gradient vectors, one pattern)
  const double vals_bytes = 4.0 * nnz * (v_bs ? B : 1);
  const double hop = 4.0 * rows_total * width * (2 + (beta != 0.f ? 1 : 0) + (axpy_out ? 2 : 0)) + 4.0 * nnz +
                     vals_bytes + 4.0 * (N + 1);
  ScopedKernelTimer _t(grad ? KK_SUPPORT_CSR_GRAD : KK_SUPPORT_CSR, st, grad ? hop + 4.0 * rows_total * width + vals_bytes : hop);
  const dim3 blk(warps_per_block * 32);
#define STC_CSR_LAUNCH(V, G, P)                                                                                         \
  support_csr_kernel<V, G, P><<<grid, blk, 0, st>>>(rp, ci, va, N, rows_total, x, x_bs, z, z_bs, y, width, alpha, beta, \
                                                    axpy_out, axpy_coef, row_list, n_list, eg, v_bs)
  if (v_bs) {
    if (grad) {
      if (vec) STC_CSR_LAUNCH(4, true, true);
      else STC_CSR_LAUNCH(1, true, true);
    } else {
      if (vec) STC_CSR_LAUNCH(4, false, true);
      else STC_CSR_LAUNCH(1, false, true);
    }
    STC_LAUNCH_OK("support_csr_kernel<per-sample>");
  } else if (grad) {
    if (vec) STC_CSR_LAUNCH(4, true, false);
    else STC_CSR_LAUNCH(1, true, false);
    STC_LAUNCH_OK("support_csr_kernel<grad>");
  } else {
    if (vec) STC_CSR_LAUNCH(4, false, false);
    else STC_CSR_LAUNCH(1, false, false);
    STC_LAUNCH_OK("support_csr_kernel");
  }
#undef STC_CSR_LAUNCH
  return STC_OK;
}

int launch_support_apply(const StcSupport& gs, int N, int B, int width, bool transpose, const float* x,
                         int64_t x_bs, const float* z, int64_t z_bs, float* y, float alpha, float beta,
                         float* axpy_out, float axpy_coef, cudaStream_t st, const int32_t* row_list, int n_list) {
  if (B <= 0 || N <= 0 || width <= 0) return STC_OK;
  if (row_list) {
    if (gs.kind == STC_SUPPORT_CSR_PER_SAMPLE) {
      set_error("support_apply: a row list is not supported for a per-sample CSR support (STC_SUPPORT_CSR_PER_SAMPLE); "
                "the row-partitioned path shares one set of edge values over the batch");
      return STC_ERR_UNSUPPORTED;
    }
    if (n_list <= 0) return STC_OK;
    if (gs.kind != STC_SUPPORT_CSR) {
      set_error("support_apply: a row list is only supported for a CSR support");
      return STC_ERR_UNSUPPORTED;
    }
  }
  if (beta != 0.f && z == nullptr) {
    set_error("support_apply: beta != 0 needs z");
    return STC_ERR_BAD_ARG;
  }
  if (gs.kind == STC_SUPPORT_DENSE) {
    if (!gs.vals) {
      set_error("dense support without vals");
      return STC_ERR_BAD_ARG;
    }
    // the tensor-core kernels do not carry the fused "axpy_out += axpy_coef * x" of the Chebyshev adjoint (terms k >= 2):
    // that update is elementwise and reads x before anything overwrites it, so it runs first as its own pass
    const bool axpy_split = axpy_out != nullptr && width % 4 == 0 && x_bs % 4 == 0 && axpy_out != y && x != y &&
                            (reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(axpy_out) & 15) == 0;
    if (axpy_out == nullptr || axpy_split) {
      bool handled = false;
      if (axpy_split) STC_TRY(launch_axpy_rows(axpy_out, x, x_bs, axpy_coef, N, B, width, st));
      STC_TRY(try_launch_support_tc(gs.vals, N, B, width, transpose, x, x_bs, z, z_bs, y, alpha, beta, st, &handled));
      if (handled) return STC_OK;
      STC_TRY(try_launch_support_tc_big(gs.vals, N, B, width, transpose, x, x_bs, z, z_bs, y, alpha, beta, st, &handled));
      if (handled) return STC_OK;
      if (axpy_split) {   // neither tensor-core kernel took the product: the FFMA kernel runs it without its fused update
        axpy_out = nullptr;
      }
    }
    long long total_q = (long long)B * width;
    dim3 grid(ceil_div(total_q, SD_BQ), ceil_div(N, SD_BM));
    // compulsory traffic: read X, write Y, (+ read Z) (+ read/modify/write of the axpy target), + the support
    ScopedKernelTimer _t(KK_SUPPORT_DENSE, st,
                         4.0 * B * N * width * (2 + (beta != 0.f ? 1 : 0) + (axpy_out ? 2 : 0)) + 4.0 * N * N);
    if (grid.y > 65535) {
      set_error("dense support with N=%d is not tiled (use CSR)", N);
      return STC_ERR_UNSUPPORTED;
    }
    if (transpose)
      support_dense_kernel<true><<<grid, SD_THREADS, 0, st>>>(gs.vals, N, x, x_bs, z, z_bs, y, width, total_q,
                                                              alpha, beta, axpy_out, axpy_coef);
    else
      support_dense_kernel<false><<<grid, SD_THREADS, 0, st>>>(gs.vals, N, x, x_bs, z, z_bs, y, width, total_q,
                                                               alpha, beta, axpy_out, axpy_coef);
    STC_LAUNCH_OK("support_dense_kernel");
    return STC_OK;
  }
  if (gs.kind != STC_SUPPORT_CSR && gs.kind != STC_SUPPORT_CSR_PER_SAMPLE) {
    set_error("unknown support kind %d", gs.kind);
    return STC_ERR_BAD_ARG;
  }
  const int32_t* rp = transpose ? gs.t_rowptr : gs.rowptr;
  const int32_t* ci = transpose ? gs.t_col : gs.col;
  const float* va = transpose ? gs.t_vals : gs.vals;
  if (!rp || !ci || !va) {
    set_error("CSR support needs both Gs and Gs^T (rowptr/col/vals and t_rowptr/t_col/t_vals)");
    return STC_ERR_BAD_ARG;
  }
  return launch_csr(rp, ci, va, gs.nnz, N, B, width, x, x_bs, z, z_bs, y, alpha, beta, axpy_out, axpy_coef, row_list,
                    n_list, CsrEdgeGrad{nullptr, 0, 0.f, nullptr}, st, csr_vals_stride(gs));
}

int launch_support_csr_edge_grad(const StcSupport& gs, int N, int B, int width, const float* x, int64_t x_bs,
                                 const float* z, int64_t z_bs, float* y, float alpha, float beta, float* axpy_out,
                                 float axpy_coef, const float* a, int64_t a_bs, float coef, float* dvals,
                                 cudaStream_t st, const int32_t* row_list, int n_list) {
  if (B <= 0 || N <= 0 || width <= 0) return STC_OK;
  if (row_list && gs.kind == STC_SUPPORT_CSR_PER_SAMPLE) {
    set_error("support edge gradient: a row list is not supported for a per-sample CSR support "
              "(STC_SUPPORT_CSR_PER_SAMPLE)");
    return STC_ERR_UNSUPPORTED;
  }
  if (row_list && n_list <= 0) return STC_OK;
  if ((gs.kind != STC_SUPPORT_CSR && gs.kind != STC_SUPPORT_CSR_PER_SAMPLE) || !gs.rowptr || !gs.col || !gs.vals) {
    set_error("support edge gradient: needs a CSR support with rowptr/col/vals");
    return STC_ERR_BAD_ARG;
  }
  const long long v_bs = csr_vals_stride(gs);
  if (!a || !dvals) {
    set_error("support edge gradient: NULL a or dvals");
    return STC_ERR_BAD_ARG;
  }
  if (beta != 0.f && z == nullptr) {
    set_error("support_apply: beta != 0 needs z");
    return STC_ERR_BAD_ARG;
  }
  if (det_mode()) {   // the plain hop (y bitwise that of stc_support_apply), then the one-writer edge gradient
    STC_TRY(launch_csr(gs.rowptr, gs.col, gs.vals, gs.nnz, N, B, width, x, x_bs, z, z_bs, y, alpha, beta, axpy_out,
                       axpy_coef, row_list, n_list, CsrEdgeGrad{nullptr, 0, 0.f, nullptr}, st, v_bs));
    const int rows = row_list ? n_list : N;
    const long long warps = v_bs ? (long long)B * rows : rows;
    long long blocks = (warps + 7) / 8;
    if (blocks > (long long)device_sm_count() * 16) blocks = (long long)device_sm_count() * 16;
    ScopedKernelTimer _t(KK_SUPPORT_CSR_GRAD, st,
                         4.0 * (double)B * width * (rows + gs.nnz) + 4.0 * gs.nnz + 4.0 * gs.nnz * (v_bs ? B : 1));
    if (v_bs)
      csr_edge_grad_det_kernel<true><<<(int)blocks, 256, 0, st>>>(gs.rowptr, gs.col, nullptr, rows, B, width, x, x_bs, a,
                                                                  a_bs, coef, dvals, v_bs);
    else
      csr_edge_grad_det_kernel<false><<<(int)blocks, 256, 0, st>>>(gs.rowptr, gs.col, row_list, rows, B, width, x, x_bs, a,
                                                                   a_bs, coef, dvals, 0);
    STC_LAUNCH_OK("csr_edge_grad_det_kernel");
    return STC_OK;
  }
  return launch_csr(gs.rowptr, gs.col, gs.vals, gs.nnz, N, B, width, x, x_bs, z, z_bs, y, alpha, beta, axpy_out,
                    axpy_coef, row_list, n_list, CsrEdgeGrad{a, (long long)a_bs, coef, dvals}, st, v_bs);
}

// ------------------------------------------------------------------------------------------------
// halo rows of the row-partitioned path (stc_gnn_b200/halo.py): gather boundary-node slabs into the packed send buffer
// of the all-to-all ([row j][b][W], rows grouped by destination rank) and scatter received slabs into the halo rows.
// One warp per (j, b) slab; lanes sweep the contiguous width axis.
// ------------------------------------------------------------------------------------------------
template <int VEC, bool PACK>
__global__ void __launch_bounds__(256)
halo_rows_kernel(float* __restrict__ x_ext, long long x_bs, int W, int B, const int32_t* __restrict__ idx, int row0,
                 int n_rows, float* __restrict__ buf) {
  const int lane = threadIdx.x & 31;
  const long long warp0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  const long long total = (long long)n_rows * B;
  for (long long s = warp0; s < total; s += nwarps) {
    const int j = (int)(s / B), b = (int)(s - (long long)j * B);
    const int node = idx ? idx[j] : row0 + j;
    float* xr = x_ext + b * x_bs + (long long)node * W;
    float* br = buf + ((long long)j * B + b) * W;
    for (int w = lane * VEC; w < W; w += 32 * VEC) {
      if (VEC == 4) {
        if (PACK) *reinterpret_cast<float4*>(br + w) = *reinterpret_cast<const float4*>(xr + w);
        else *reinterpret_cast<float4*>(xr + w) = *reinterpret_cast<const float4*>(br + w);
      } else {
        if (PACK) br[w] = xr[w];
        else xr[w] = br[w];
      }
    }
  }
}

int launch_halo_rows(bool pack, float* x_ext, long long x_bs, int W, int B, const int32_t* idx, int row0, int n_rows,
                     float* buf, cudaStream_t st) {
  if (n_rows <= 0 || B <= 0 || W <= 0) return STC_OK;
  const bool vec = (W % 4 == 0) && (x_bs % 4 == 0) && aligned16(x_ext) && aligned16(buf);
  const long long slabs = (long long)n_rows * B;
  long long want = (slabs + 7) / 8;
  int grid = (int)(want < (long long)device_sm_count() * 8 ? want : (long long)device_sm_count() * 8);
  if (grid < 1) grid = 1;
  if (vec) {
    if (pack) halo_rows_kernel<4, true><<<grid, 256, 0, st>>>(x_ext, x_bs, W, B, idx, row0, n_rows, buf);
    else halo_rows_kernel<4, false><<<grid, 256, 0, st>>>(x_ext, x_bs, W, B, idx, row0, n_rows, buf);
  } else {
    if (pack) halo_rows_kernel<1, true><<<grid, 256, 0, st>>>(x_ext, x_bs, W, B, idx, row0, n_rows, buf);
    else halo_rows_kernel<1, false><<<grid, 256, 0, st>>>(x_ext, x_bs, W, B, idx, row0, n_rows, buf);
  }
  STC_LAUNCH_OK("halo_rows_kernel");
  return STC_OK;
}

// ------------------------------------------------------------------------------------------------
// dGs[n',m] += coef * sum_{b,j} A[b,n',j] * Bm[b,m,j]   (split over the batch, atomics at the end)
// ------------------------------------------------------------------------------------------------
constexpr int SO_T = 64, SO_BK = 16, SO_THREADS = 256;

// DET: batch slice z writes its partial into slot z of dG (N * N floats each) with plain stores
template <bool DET>
__global__ void __launch_bounds__(SO_THREADS)
support_outer_kernel(int N, int B, int W, const float* __restrict__ A, long long a_bs,
                     const float* __restrict__ Bm, float coef, float* dG, int b_per_cta) {
  __shared__ __align__(16) float As[SO_BK][SO_T + 4];
  __shared__ __align__(16) float Bs[SO_BK][SO_T + 4];
  const int tid = threadIdx.x, tx = tid % 16, ty = tid / 16;
  const int n0 = blockIdx.y * SO_T, m0 = blockIdx.x * SO_T;
  const int b_lo = blockIdx.z * b_per_cta;
  const int b_hi = min(B, b_lo + b_per_cta);
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  const int kk = tid % SO_BK;
  for (int b = b_lo; b < b_hi; ++b) {
    const float* Ab = A + (long long)b * a_bs;
    const float* Bb = Bm + (long long)b * N * W;
    for (int j0 = 0; j0 < W; j0 += SO_BK) {
      const int j = j0 + kk;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        int rr = tid / SO_BK + i * 16;
        As[kk][rr] = (j < W && n0 + rr < N) ? Ab[(long long)(n0 + rr) * W + j] : 0.f;
        Bs[kk][rr] = (j < W && m0 + rr < N) ? Bb[(long long)(m0 + rr) * W + j] : 0.f;
      }
      __syncthreads();
#pragma unroll
      for (int k = 0; k < SO_BK; ++k) {
        float4 a = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
        float4 c = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
        float av[4] = {a.x, a.y, a.z, a.w}, cv[4] = {c.x, c.y, c.z, c.w};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int jj = 0; jj < 4; ++jj) acc[i][jj] = fmaf(av[i], cv[jj], acc[i][jj]);
      }
      __syncthreads();
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int n = n0 + ty * 4 + i;
    if (n >= N) continue;
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) {
      int m = m0 + tx * 4 + jj;
      if (m >= N) continue;
      if constexpr (DET) dG[((long long)blockIdx.z * N + n) * N + m] = coef * acc[i][jj];
      else atomicAdd(&dG[(long long)n * N + m], coef * acc[i][jj]);
    }
  }
}

// batch slices of the FFMA form: as many as fill the device twice over
static int outer_ffma_zsplit(int N, int B) {
  const int tiles = ceil_div(N, SO_T);
  int zsplit = device_sm_count() * 2 / (tiles * tiles);
  if (zsplit < 1) zsplit = 1;
  if (zsplit > B) zsplit = B;
  return ceil_div(B, ceil_div(B, zsplit));
}

long long support_outer_det_floats(int N, int B, int width) {
  if (B <= 0 || N <= 0 || width <= 0) return 0;
  // the larger of the two forms' slot counts (operand alignment decides which one runs); one slice needs none
  const int tc = outer_tc_det_slots(N, B, width), ffma = outer_ffma_zsplit(N, B);
  const int slots = tc > ffma ? tc : ffma;
  return slots > 1 ? (long long)slots * N * N : 0;
}

int launch_support_outer(int N, int B, int width, const float* a, int64_t a_bs, const float* bmat, float coef,
                         float* dG, cudaStream_t st, float* det_ws) {
  if (B <= 0 || N <= 0 || width <= 0) return STC_OK;
  if (det_mode() && det_ws == nullptr && support_outer_det_floats(N, B, width) > 0) {
    set_error("support outer product: the deterministic form needs its slot workspace");
    return STC_ERR_WORKSPACE;
  }
  {
    bool handled = false;
    STC_TRY(try_launch_outer_tc(N, B, width, a, a_bs, bmat, coef, dG, st, &handled, det_ws));
    if (handled) return STC_OK;
  }
  int tiles = ceil_div(N, SO_T);
  if (tiles > 65535) {
    set_error("dGs for N=%d is not tiled", N);
    return STC_ERR_UNSUPPORTED;
  }
  const int zsplit = outer_ffma_zsplit(N, B);
  const int b_per = ceil_div(B, zsplit);
  dim3 grid(tiles, tiles, zsplit);
  const bool det = det_mode() && zsplit > 1;   // one slice: every element has a single writer already
  {
    ScopedKernelTimer _t(KK_SUPPORT_OUTER, st, 4.0 * B * N * width * 2 + 4.0 * N * N);
    if (det)
      support_outer_kernel<true><<<grid, SO_THREADS, 0, st>>>(N, B, width, a, a_bs, bmat, coef, det_ws, b_per);
    else
      support_outer_kernel<false><<<grid, SO_THREADS, 0, st>>>(N, B, width, a, a_bs, bmat, coef, dG, b_per);
    STC_LAUNCH_OK("support_outer_kernel");
  }
  if (det) return launch_det_reduce(dG, det_ws, zsplit, (long long)N * N, (long long)N * N, st);
  return STC_OK;
}

// ------------------------------------------------------------------------------------------------
// deterministic mode: the fixed-order sum of per-CTA partial slots, added once into the destination.  One thread per
// element walks the slots in ascending order (consecutive threads read consecutive floats of each slot).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
det_reduce_kernel(float* __restrict__ dst, const float* __restrict__ slots, int n_slots, long long n, long long stride) {
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n; i += (long long)gridDim.x * 256) {
    // (unrolled so that eight slots' loads are in flight at once; the additions keep ascending slot order)
    float s = 0.f;
#pragma unroll 8
    for (int k = 0; k < n_slots; ++k) s += __ldg(slots + (long long)k * stride + i);
    dst[i] += s;
  }
}

int launch_det_reduce(float* dst, const float* slots, int n_slots, long long n, long long slot_stride, cudaStream_t st) {
  if (n <= 0 || n_slots <= 0) return STC_OK;
  long long blocks = (n + 255) / 256;
  if (blocks > (long long)device_sm_count() * 8) blocks = (long long)device_sm_count() * 8;
  ScopedKernelTimer _t(KK_DET_REDUCE, st, 4.0 * n * (n_slots + 2));
  det_reduce_kernel<<<(int)blocks, 256, 0, st>>>(dst, slots, n_slots, n, slot_stride);
  STC_LAUNCH_OK("det_reduce_kernel");
  return STC_OK;
}

// ------------------------------------------------------------------------------------------------
// small C x C Chebyshev terms (one CTA; C is at most a few hundred)
// ------------------------------------------------------------------------------------------------
__global__ void cheby_small_kernel(const float* __restrict__ G, int C, int K, float* Q) {
  const int CC = C * C;
  for (int i = threadIdx.x; i < CC; i += blockDim.x) {
    Q[i] = (i / C == i % C) ? 1.f : 0.f;
    if (K > 1) Q[CC + i] = G[i];
  }
  __syncthreads();
  for (int k = 2; k < K; ++k) {
    const float* T1 = Q + (size_t)(k - 1) * CC;
    const float* T2 = Q + (size_t)(k - 2) * CC;
    float* T = Q + (size_t)k * CC;
    for (int i = threadIdx.x; i < CC; i += blockDim.x) {
      int a = i / C, b = i % C;
      float s = 0.f;
      for (int j = 0; j < C; ++j) s = fmaf(G[a * C + j], T1[j * C + b], s);
      T[i] = 2.f * s - T2[i];
    }
    __syncthreads();
  }
}

// adjoint: dG (+)= sum over the chain; dQ is consumed (modified in place)
__global__ void cheby_small_bwd_kernel(const float* __restrict__ G, const float* __restrict__ Q, float* dQ, int C,
                                       int K, float* dG) {
  const int CC = C * C;
  for (int k = K - 1; k >= 2; --k) {
    const float* dT = dQ + (size_t)k * CC;
    const float* T1 = Q + (size_t)(k - 1) * CC;
    float* dT1 = dQ + (size_t)(k - 1) * CC;
    float* dT2 = dQ + (size_t)(k - 2) * CC;
    for (int i = threadIdx.x; i < CC; i += blockDim.x) {
      int a = i / C, b = i % C;
      float s = 0.f, t = 0.f;
      for (int j = 0; j < C; ++j) {
        s = fmaf(dT[a * C + j], T1[b * C + j], s);   // dT * T1^T
        t = fmaf(G[j * C + a], dT[j * C + b], t);    // G^T * dT
      }
      dG[i] += 2.f * s;
      dT1[i] += 2.f * t;
      dT2[i] -= dT[i];
    }
    __syncthreads();
  }
  if (K > 1)
    for (int i = threadIdx.x; i < CC; i += blockDim.x) dG[i] += dQ[CC + i];
}

int launch_cheby_small(const float* G, int C, int K, float* Q, cudaStream_t st) {
  ScopedKernelTimer _t(KK_CHEBY_SMALL, st, 4.0 * C * C * (K + 1));
  cheby_small_kernel<<<1, 256, 0, st>>>(G, C, K, Q);
  STC_LAUNCH_OK("cheby_small_kernel");
  return STC_OK;
}

int launch_cheby_small_bwd(const float* G, const float* Q, float* dQ, int C, int K, float* dG, cudaStream_t st) {
  ScopedKernelTimer _t(KK_CHEBY_SMALL, st, 4.0 * C * C * (2 * K + 2));
  cheby_small_bwd_kernel<<<1, 256, 0, st>>>(G, Q, dQ, C, K, dG);
  STC_LAUNCH_OK("cheby_small_bwd_kernel");
  return STC_OK;
}

}  // namespace stc
