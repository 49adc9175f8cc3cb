// Graph generator on a fixed CSR pattern: the sparse form of MGP_Gen's spatial half (STC_GNN.py:227-233).
//
//  pair_scores_csr_kernel  S[e] = <U_n, V_m> - <V_n, U_m> for every stored edge e = (n, m) of the pattern, where U, V
//                          are node-major [N][width] (width = B*T*hg): M[n,m] - M[m,n] of the dense generator evaluated
//                          at the stored edges only.
//  edge_softmax_kernel     P[e] = softmax over the stored edges of row n of relu(S) (forward), and its adjoint
//                          dS[e] = [S[e] > 0] * P[e] * (dP[e] - sum_row P * dP) (backward).
//
// Both are deterministic: no atomics, every output is reduced in a fixed order and written once by one lane.  The
// backward of the scores is two plain CSR hops each for dU and dV (stc_support_apply), done by the caller.
#include "stc_common.cuh"

namespace stc {

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

static int csr_warp_grid(long long rows, int warps_per_block) {
  const long long want = (rows + warps_per_block - 1) / warps_per_block;
  const long long cap = (long long)device_sm_count() * 16;
  return (int)(want < 1 ? 1 : (want < cap ? want : cap));
}

// ------------------------------------------------------------------------------------------------
// scores: one warp per row n; lanes sweep the width.  The row's edges are taken in groups of PS_E: for every column chunk
// (32 * VEC * PS_U floats) the warp loads its own chunk of U_n, V_n once into registers and dots it with the chunk of
// every neighbour in the group, so the own row is read once per group, not once per edge.  Each lane keeps two
// accumulators per edge across all chunks (chunk order), subtracts them once, and the warp reduces the difference with
// an xor-shuffle tree.  For a self-loop the two per-lane sums are the same products in the same order, so the score is
// exactly 0, as the diagonal of the dense M - M^T is.
// ------------------------------------------------------------------------------------------------
constexpr int PS_U = 4;   // float(4)s per lane and operand in one column chunk
constexpr int PS_E = 4;   // edges of one group (8 spills at VEC = 4; the grid and kNN patterns store 8-10 edges a row)

//
// ROWS: only the n_rows rows listed in `rows` are scored (the other entries of `scores` are not touched), and U / V
// have the row stride ld >= W, so that U and V can share one extended buffer [U | V] (the row-partitioned generator,
// stc_gnn_b200/sparse_mgp.py).  A listed row's arithmetic is the plain kernel's, so its scores are bitwise the same.
// blockIdx.y is the sample of a batched launch (the per-sample generator): U, V of sample s start s * s_bs floats in,
// its scores s * nnz floats in; the arithmetic of each sample is that of the plain kernel on that sample alone.
template <int VEC, bool ROWS>
__global__ void __launch_bounds__(256)
pair_scores_csr_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, int N, long long W,
                       const float* __restrict__ U, const float* __restrict__ V, float* __restrict__ scores,
                       long long ld, const int32_t* __restrict__ rows, int n_rows, long long s_bs, long long nnz) {
  constexpr long long CHUNK = 32LL * VEC * PS_U;
  const long long LD = ROWS ? ld : W;
  U += blockIdx.y * s_bs;
  V += blockIdx.y * s_bs;
  scores += blockIdx.y * nnz;
  const int lane = threadIdx.x & 31;
  const long long warp0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long i = warp0; i < (ROWS ? n_rows : N); i += nwarps) {
    const long long n = ROWS ? rows[i] : i;
    const int e0 = rowptr[n], e1 = rowptr[n + 1];
    const float* un = U + n * LD;
    const float* vn = V + n * LD;
    for (int g0 = e0; g0 < e1; g0 += PS_E) {
      const int cnt = min(PS_E, e1 - g0);
      int nb[PS_E];
#pragma unroll
      for (int k = 0; k < PS_E; ++k) nb[k] = col[g0 + (k < cnt ? k : 0)];
      float uv[PS_E], vu[PS_E];   // <U_n, V_m> and <V_n, U_m>, this lane's share
#pragma unroll
      for (int k = 0; k < PS_E; ++k) uv[k] = vu[k] = 0.f;
      for (long long j0 = 0; j0 < W; j0 += CHUNK) {
        float ur[PS_U][VEC], vr[PS_U][VEC];
#pragma unroll
        for (int u = 0; u < PS_U; ++u) {
          const long long j = j0 + (long long)(u * 32 + lane) * VEC;
#pragma unroll
          for (int v = 0; v < VEC; ++v) ur[u][v] = vr[u][v] = 0.f;
          if (j < W) {
            if (VEC == 4) {
              const float4 a = *reinterpret_cast<const float4*>(un + j), b = *reinterpret_cast<const float4*>(vn + j);
              ur[u][0] = a.x; ur[u][1 % VEC] = a.y; ur[u][2 % VEC] = a.z; ur[u][3 % VEC] = a.w;
              vr[u][0] = b.x; vr[u][1 % VEC] = b.y; vr[u][2 % VEC] = b.z; vr[u][3 % VEC] = b.w;
            } else {
              ur[u][0] = un[j];
              vr[u][0] = vn[j];
            }
          }
        }
#pragma unroll
        for (int k = 0; k < PS_E; ++k) {
          if (k >= cnt) break;
          const float* um = U + nb[k] * LD;
          const float* vm = V + nb[k] * LD;
#pragma unroll
          for (int u = 0; u < PS_U; ++u) {
            const long long j = j0 + (long long)(u * 32 + lane) * VEC;
            if (j < W) {
              if (VEC == 4) {
                const float4 a = *reinterpret_cast<const float4*>(vm + j), b = *reinterpret_cast<const float4*>(um + j);
                uv[k] = fmaf(ur[u][0], a.x, uv[k]); vu[k] = fmaf(vr[u][0], b.x, vu[k]);
                uv[k] = fmaf(ur[u][1 % VEC], a.y, uv[k]); vu[k] = fmaf(vr[u][1 % VEC], b.y, vu[k]);
                uv[k] = fmaf(ur[u][2 % VEC], a.z, uv[k]); vu[k] = fmaf(vr[u][2 % VEC], b.z, vu[k]);
                uv[k] = fmaf(ur[u][3 % VEC], a.w, uv[k]); vu[k] = fmaf(vr[u][3 % VEC], b.w, vu[k]);
              } else {
                uv[k] = fmaf(ur[u][0], vm[j], uv[k]);
                vu[k] = fmaf(vr[u][0], um[j], vu[k]);
              }
            }
          }
        }
      }
#pragma unroll
      for (int k = 0; k < PS_E; ++k) {
        if (k >= cnt) break;
        float s = uv[k] - vu[k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) scores[g0 + k] = s;
      }
    }
  }
}

int launch_pair_scores_csr(const int32_t* rowptr, const int32_t* col, long long nnz, int N, long long width,
                           const float* u, const float* v, float* scores, cudaStream_t st) {
  const bool vec = (width % 4 == 0) && aligned16(u) && aligned16(v);
  const int grid = csr_warp_grid(N, 8);
  // own rows 4*2*N*W and the output 4*nnz are compulsory HBM traffic; the pattern 8*nnz + 4(N+1) too.  The gathered
  // neighbour rows 4*2*W*nnz are counted as well, although for a local pattern (grid, Morton-ordered kNN) most of them
  // are L2 hits of rows other warps have just read.
  ScopedKernelTimer _t(KK_PAIR_SCORES_CSR, st,
                       4.0 * 2 * N * width + 4.0 * 2 * width * nnz + 8.0 * nnz + 4.0 * (N + 1) + 4.0 * nnz);
  if (vec) pair_scores_csr_kernel<4, false><<<grid, 256, 0, st>>>(rowptr, col, N, width, u, v, scores, width, nullptr, 0, 0, 0);
  else pair_scores_csr_kernel<1, false><<<grid, 256, 0, st>>>(rowptr, col, N, width, u, v, scores, width, nullptr, 0, 0, 0);
  STC_LAUNCH_OK("pair_scores_csr_kernel");
  return STC_OK;
}

int launch_pair_scores_csr_batched(const int32_t* rowptr, const int32_t* col, long long nnz, int N, int B,
                                   long long width, const float* u, const float* v, float* scores, cudaStream_t st) {
  if (B <= 0) return STC_OK;
  // each sample's rows start N * width floats after the previous sample's, so the vector form is taken exactly when the
  // unbatched call on sample 0 takes it and every sample then starts 16-byte aligned
  const bool vec = (width % 4 == 0) && aligned16(u) && aligned16(v);
  const dim3 grid(csr_warp_grid(N, 8), B);
  const long long s_bs = (long long)N * width;
  // the unbatched count, per sample (the pattern itself is read once)
  ScopedKernelTimer _t(KK_PAIR_SCORES_CSR, st,
                       (double)B * (4.0 * 2 * N * width + 4.0 * 2 * width * nnz + 4.0 * nnz) + 8.0 * nnz + 4.0 * (N + 1));
  if (vec) pair_scores_csr_kernel<4, false><<<grid, 256, 0, st>>>(rowptr, col, N, width, u, v, scores, width, nullptr, 0, s_bs, nnz);
  else pair_scores_csr_kernel<1, false><<<grid, 256, 0, st>>>(rowptr, col, N, width, u, v, scores, width, nullptr, 0, s_bs, nnz);
  STC_LAUNCH_OK("pair_scores_csr_kernel<batched>");
  return STC_OK;
}

int launch_pair_scores_csr_rows(const int32_t* rowptr, const int32_t* col, long long nnz, int N, long long width,
                                long long ld, const float* u, const float* v, float* scores, const int32_t* rows,
                                int n_rows, cudaStream_t st) {
  if (n_rows <= 0) return STC_OK;
  const bool vec = (width % 4 == 0) && (ld % 4 == 0) && aligned16(u) && aligned16(v);
  const int grid = csr_warp_grid(n_rows, 8);
  // the plain kernel's count for the listed rows; their edge count is not known on the host, so it is taken at the
  // pattern's mean degree (nnz / N edges a row), plus the row list itself
  const double er = (double)nnz * n_rows / N;
  ScopedKernelTimer _t(KK_PAIR_SCORES_CSR, st,
                       4.0 * 2 * n_rows * width + 4.0 * 2 * width * er + 4.0 * er + 8.0 * n_rows + 4.0 * er + 4.0 * n_rows);
  if (vec) pair_scores_csr_kernel<4, true><<<grid, 256, 0, st>>>(rowptr, col, N, width, u, v, scores, ld, rows, n_rows, 0, 0);
  else pair_scores_csr_kernel<1, true><<<grid, 256, 0, st>>>(rowptr, col, N, width, u, v, scores, ld, rows, n_rows, 0, 0);
  STC_LAUNCH_OK("pair_scores_csr_kernel<rows>");
  return STC_OK;
}

// ------------------------------------------------------------------------------------------------
// softmax over the stored edges of each row: one warp per row, lanes stride over the row's edges, row sums through an
// xor-shuffle tree (fixed order).  An empty row writes nothing.  The rows are the B * N rows of [B][nnz] buffers (row
// b * N + n is row n of sample b, whose entries start b * nnz in); B = 1 is the unbatched softmax.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float s) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  return s;
}

template <bool BWD>
__global__ void __launch_bounds__(256)
edge_softmax_kernel(const int32_t* __restrict__ rowptr, int N, long long rows, long long nnz, const float* __restrict__ S,
                    const float* __restrict__ P, const float* __restrict__ dP, float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const long long warp0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long r = warp0; r < rows; r += nwarps) {
    const long long b = r / N, n = r - b * N;
    const long long e0 = rowptr[n] + b * nnz, e1 = rowptr[n + 1] + b * nnz;
    if (e0 >= e1) continue;
    if (BWD) {   // dS = [S > 0] * P * (dP - sum_row P dP)
      float dot = 0.f;
      for (long long e = e0 + lane; e < e1; e += 32) dot = fmaf(P[e], dP[e], dot);
      dot = warp_sum(dot);
      for (long long e = e0 + lane; e < e1; e += 32) out[e] = S[e] > 0.f ? P[e] * (dP[e] - dot) : 0.f;
    } else {     // P = exp(relu(S) - max) / sum, the max subtracted as torch.softmax does
      float mx = 0.f;   // relu(S) >= 0
      for (long long e = e0 + lane; e < e1; e += 32) mx = fmaxf(mx, S[e]);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
      float sum = 0.f;
      for (long long e = e0 + lane; e < e1; e += 32) sum += expf(fmaxf(S[e], 0.f) - mx);
      const float inv = 1.f / warp_sum(sum);
      for (long long e = e0 + lane; e < e1; e += 32) out[e] = expf(fmaxf(S[e], 0.f) - mx) * inv;
    }
  }
}

int launch_edge_softmax(bool bwd, const int32_t* rowptr, long long nnz, int N, const float* s, const float* p,
                        const float* dp, float* out, cudaStream_t st, int B) {
  if (B <= 0) return STC_OK;
  const long long rows = (long long)B * N;
  const int grid = csr_warp_grid(rows, 8);
  // compulsory: the pattern's rowptr, then S in / P out (forward) or S, P, dP in / dS out (backward), per sample
  ScopedKernelTimer _t(KK_EDGE_SOFTMAX, st, 4.0 * (N + 1) + (bwd ? 16.0 : 8.0) * nnz * B);
  if (bwd) edge_softmax_kernel<true><<<grid, 256, 0, st>>>(rowptr, N, rows, nnz, s, p, dp, out);
  else edge_softmax_kernel<false><<<grid, 256, 0, st>>>(rowptr, N, rows, nnz, s, nullptr, nullptr, out);
  STC_LAUNCH_OK("edge_softmax_kernel");
  return STC_OK;
}

}  // namespace stc
