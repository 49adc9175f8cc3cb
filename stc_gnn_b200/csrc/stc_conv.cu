// General-path convolution kernels: categorical mix + weight contraction + GRU epilogue, and their
// adjoints.  One CTA owns a tile of whole nodes (all C categories of each), so the C x C categorical
// mode product ('bmcl,cd->bmdl', /root/reference/framework/STC_GNN.py:38) is tile-local and the
// concatenated feature tensor of STC_GNN.py:41 never exists in HBM: each (n, c) feature block is built
// in shared memory from the spatial Chebyshev terms and consumed at once by the weight contraction
// (STC_GNN.py:42) whose epilogue applies bias / activation (:44-46) and the GRU non-linearities
// (STC_GNN.py:71-78).
#include "stc_conv_common.cuh"

namespace stc {

// acc[i][a][b] += sum_k A[(rg*4+a)*lda + k] * Bm[k*ldb + cg*4 + b]   for items it = tid + i*blockDim
template <int NI>
__device__ __forceinline__ void tile_gemm(float (&acc)[NI][4][4], const float* __restrict__ A, int lda,
                                          const float* __restrict__ Bm, int ldb, int K, int RG, int CG) {
  const int items = RG * CG;
#pragma unroll
  for (int i = 0; i < NI; ++i) {
    const int it = threadIdx.x + i * CV_THREADS;
    if (it >= items) break;
    const int rg = it / CG, cg = it - rg * CG;
    const float* ap = A + rg * 4 * lda;
    const float* bp = Bm + cg * 4;
#pragma unroll 4
    for (int k = 0; k < K; ++k) {
      float a0 = ap[k], a1 = ap[lda + k], a2 = ap[2 * lda + k], a3 = ap[3 * lda + k];
      float4 b = *reinterpret_cast<const float4*>(bp + k * ldb);
      acc[i][0][0] = fmaf(a0, b.x, acc[i][0][0]); acc[i][0][1] = fmaf(a0, b.y, acc[i][0][1]);
      acc[i][0][2] = fmaf(a0, b.z, acc[i][0][2]); acc[i][0][3] = fmaf(a0, b.w, acc[i][0][3]);
      acc[i][1][0] = fmaf(a1, b.x, acc[i][1][0]); acc[i][1][1] = fmaf(a1, b.y, acc[i][1][1]);
      acc[i][1][2] = fmaf(a1, b.z, acc[i][1][2]); acc[i][1][3] = fmaf(a1, b.w, acc[i][1][3]);
      acc[i][2][0] = fmaf(a2, b.x, acc[i][2][0]); acc[i][2][1] = fmaf(a2, b.y, acc[i][2][1]);
      acc[i][2][2] = fmaf(a2, b.z, acc[i][2][2]); acc[i][2][3] = fmaf(a2, b.w, acc[i][2][3]);
      acc[i][3][0] = fmaf(a3, b.x, acc[i][3][0]); acc[i][3][1] = fmaf(a3, b.y, acc[i][3][1]);
      acc[i][3][2] = fmaf(a3, b.z, acc[i][3][2]); acc[i][3][3] = fmaf(a3, b.w, acc[i][3][3]);
    }
  }
}


// =================================================================================================
// forward: out = sum_{k,c} F_{k,c} W_{k,c} + b ; gates: u,r = sigmoid, rH = r*H ; candi: c = tanh, H' blend
// =================================================================================================
// forward epilogue: bias, activation and the GRU non-linearities of the accumulator items this thread owns
template <int NI, bool SAVE>
__device__ __forceinline__ void conv_fwd_epilogue(const ConvArgs& a, const float (&acc)[NI][4][4], long long row0,
                                                  int rows_valid, int items, int CG) {
  const int Hout = a.Hout, h = a.h;
#pragma unroll
  for (int i = 0; i < NI; ++i) {
    const int it = threadIdx.x + i * CV_THREADS;
    if (it >= items) break;
    const int rg = it / CG, cg = it - rg * CG;
#pragma unroll
    for (int x = 0; x < 4; ++x) {
      const int row = rg * 4 + x;
      if (row >= rows_valid) continue;
      const long long gr = row0 + row;
#pragma unroll
      for (int y = 0; y < 4; ++y) {
        const int col = cg * 4 + y;
        if (col >= Hout) continue;
        float pre = acc[i][x][y] + (a.bias ? a.bias[col] : 0.f);
        if (a.act == STC_ACT_RELU) pre = fmaxf(pre, 0.f);
        if (a.phase == 0) {
          float s = sigmoidf_acc(pre);
          if (col < h) {
            a.u[gr * h + col] = s;
          } else {
            const long long o = gr * h + (col - h);
            if (SAVE) a.r[o] = s;
            a.rH[o] = s * a.Hprev[o];
          }
        } else {
          const long long o = gr * h + col;
          float cc = tanhf(pre);
          float uu = a.u[o], hp = a.Hprev[o];
          if (SAVE) a.c[o] = cc;
          a.Hnew[o] = fmaf(uu, cc - hp, hp);  // (1-u)*H + u*c
        }
      }
    }
  }
}

template <int NI>
__global__ void __launch_bounds__(CV_THREADS)
conv_fwd_kernel(const ConvArgs a, const ConvTile t) {
  extern __shared__ __align__(16) float smem[];
  const int C = a.C, L = t.L, LP = t.LP, Hout = a.Hout, HoutP = t.HoutP, h = a.h;
  float* Fin = smem;
  float* Fmx = Fin + (size_t)t.rowsP * LP;
  float* Ws = Fmx + (a.Kc > 1 ? (size_t)t.rowsP * LP : 0);
  Ws = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(Ws) + 15) & ~uintptr_t(15));
  float* Qs = Ws + (size_t)L * HoutP;  // [(Kc-1)][C][C]

  const long long total_nodes = (long long)a.B * a.N;
  const long long g0 = (long long)blockIdx.x * t.npt;
  const int nodes_valid = (int)min((long long)t.npt, total_nodes - g0);
  const int rows_valid = nodes_valid * C;
  const FeatSrc fs = feat_src(a);
  const int RG = t.rowsP / 4, CG = HoutP / 4;

  for (int i = threadIdx.x; i < (a.Kc - 1) * C * C; i += blockDim.x) Qs[i] = a.Q[C * C + i];

  float acc[NI][4][4];
#pragma unroll
  for (int i = 0; i < NI; ++i)
#pragma unroll
    for (int x = 0; x < 4; ++x)
#pragma unroll
      for (int y = 0; y < 4; ++y) acc[i][x][y] = 0.f;

  for (int k = 0; k < a.Ks; ++k) {
    __syncthreads();  // previous users of Fin are done
    load_feat_tile(fs, k, g0, nodes_valid, t.rowsP, Fin, LP);
    for (int c = 0; c < a.Kc; ++c) {
      __syncthreads();  // Fin loaded / previous Ws,Fmx consumers done
      const float* Wblk = a.W + (size_t)(k * a.Kc + c) * L * Hout;
      for (int idx = threadIdx.x; idx < L * HoutP; idx += blockDim.x) {
        int l = idx / HoutP, j = idx - l * HoutP;
        Ws[idx] = (j < Hout) ? Wblk[l * Hout + j] : 0.f;
      }
      const float* src = Fin;
      if (c > 0) {
        mix_tile(Fin, Fmx, Qs + (size_t)(c - 1) * C * C, rows_valid, C, L, LP);
        src = Fmx;
      }
      __syncthreads();
      tile_gemm<NI>(acc, src, LP, Ws, HoutP, L, RG, CG);
    }
  }

  // SAVE = false (a forward-only call, r / c null): only the backward reads r and c.  The test is taken once, outside
  // the unrolled epilogue, so that the training form keeps its code.
  if ((a.phase == 0 ? a.r : a.c) != nullptr)
    conv_fwd_epilogue<NI, true>(a, acc, g0 * C, rows_valid, RG * CG, CG);
  else
    conv_fwd_epilogue<NI, false>(a, acc, g0 * C, rows_valid, RG * CG, CG);
}

static size_t conv_fwd_smem(const ConvArgs& a, const ConvTile& t) {
  size_t f = (size_t)t.rowsP * t.LP * (a.Kc > 1 ? 2 : 1) + 4 + (size_t)t.L * t.HoutP +
             (size_t)(a.Kc > 1 ? (a.Kc - 1) : 0) * a.C * a.C;
  return f * sizeof(float);
}

static int pick_rows_fwd(const ConvArgs& a, ConvTile* out, size_t* smem_out, int* ni_out) {
  const int CG = ((a.Hout + 3) & ~3) / 4;
  int target = 4 * CV_THREADS * 2 / CG;  // two 4x4 items per thread
  if (target > 256) target = 256;
  if (target < 4) target = 4;
  for (;;) {
    ConvTile t = make_tile(a, target);
    size_t smem = conv_fwd_smem(a, t);
    int items = (t.rowsP / 4) * CG;
    int ni = ceil_div(items, CV_THREADS);
    if (smem <= 200 * 1024 && ni <= CV_MAX_NI) {
      *out = t; *smem_out = smem; *ni_out = ni;
      return STC_OK;
    }
    if (t.npt == 1) {
      set_error("conv tile does not fit: C=%d Din=%d h=%d Hout=%d needs %zu B smem, %d items/thread", a.C, a.Din,
                a.h, a.Hout, smem, ni);
      return STC_ERR_UNSUPPORTED;
    }
    target = (t.npt / 2) * a.C;
    if (target < a.C) target = a.C;
  }
}


int launch_conv_fwd(const ConvArgs& a, cudaStream_t st) {
  bool handled = false;
  STC_TRY(try_launch_conv_fwd_tc(a, st, &handled));
  if (handled) return STC_OK;
  STC_TRY(try_launch_conv_fwd_big(a, st, &handled));
  if (handled) return STC_OK;
  ConvTile t; size_t smem; int ni;
  STC_TRY(pick_rows_fwd(a, &t, &smem, &ni));
  long long total_nodes = (long long)a.B * a.N;
  int grid = ceil_div(total_nodes, t.npt);
  // compulsory traffic per row: the Ks spatial terms of [x|h] once, then the state traffic (conv_fwd_state_floats).
  // Plus the weights.
  const double R = (double)total_nodes * a.C;
  ScopedKernelTimer _t(KK_CONV_FWD, st, 4.0 * R * (a.Ks * t.L + conv_fwd_state_floats(a)) + 4.0 * a.Ks * a.Kc * t.L * a.Hout);
  switch (ni) {
    case 1: STC_TRY(set_smem(conv_fwd_kernel<1>, smem)); conv_fwd_kernel<1><<<grid, CV_THREADS, smem, st>>>(a, t); break;
    case 2: STC_TRY(set_smem(conv_fwd_kernel<2>, smem)); conv_fwd_kernel<2><<<grid, CV_THREADS, smem, st>>>(a, t); break;
    default: STC_TRY(set_smem(conv_fwd_kernel<4>, smem)); conv_fwd_kernel<4><<<grid, CV_THREADS, smem, st>>>(a, t); break;
  }
  STC_LAUNCH_OK("conv_fwd_kernel");
  return STC_OK;
}

// =================================================================================================
// backward, part 1: pre-activation gradient, bias gradient, feature adjoints dY_k, categorical dQ
// =================================================================================================
#define STC_DX_KERNEL_NAME conv_bwd_dx_kernel
#define STC_DX_DET 0
#include "stc_conv_bwd_dx.cuh"
#undef STC_DX_KERNEL_NAME
#undef STC_DX_DET
#define STC_DX_KERNEL_NAME gen_det_bwd_dx_kernel
#define STC_DX_DET 1
#include "stc_conv_bwd_dx.cuh"
#undef STC_DX_KERNEL_NAME
#undef STC_DX_DET

static size_t conv_dx_smem(const ConvArgs& a, const ConvTile& t, int DP) {
  const bool mixed = a.Kc > 1;
  const bool want_dQ = mixed && a.dQ != nullptr;
  size_t f = (size_t)t.rowsP * DP + (size_t)a.Hout * t.LP4 + (size_t)t.rowsP * t.LP * (1 + (mixed ? 1 : 0) + (want_dQ ? 1 : 0)) +
             (size_t)(mixed ? (a.Kc - 1) : 0) * a.C * a.C;
  return f * sizeof(float);
}

int det_reduce_dx(const ConvArgs& a, int grid, cudaStream_t st) {
  const long long npairs = a.Kc > 1 ? (long long)(a.Kc - 1) * a.C * a.C : 0, stride = a.Hout + npairs;
  if (a.dbias) STC_TRY(launch_det_reduce(a.dbias, a.det_ws, grid, a.Hout, stride, st));
  if (a.dQ && npairs) STC_TRY(launch_det_reduce(a.dQ + (size_t)a.C * a.C, a.det_ws + a.Hout, grid, npairs, stride, st));
  return STC_OK;
}

// tile of the general dx kernel (the largest that fits shared memory and the per-thread item budget)
static int conv_dx_general_tile(const ConvArgs& a, ConvTile* tp, size_t* smemp, int* nip, int* DPp) {
  const int L = a.Din + a.h;
  const int CGL = ((L + 3) & ~3) / 4;
  const int HoutP = (a.Hout + 3) & ~3;
  const int DP = HoutP | 1;
  int target = 4 * CV_THREADS * 2 / CGL;
  if (target > 128) target = 128;
  if (target < 4) target = 4;
  ConvTile t; size_t smem; int ni;
  for (;;) {
    t = make_tile(a, target);
    smem = conv_dx_smem(a, t, DP);
    ni = ceil_div((t.rowsP / 4) * CGL, CV_THREADS);
    if (smem <= 200 * 1024 && ni <= CV_MAX_NI) break;
    if (t.npt == 1) {
      set_error("conv backward tile does not fit: C=%d Din=%d h=%d Hout=%d needs %zu B smem, %d items/thread", a.C,
                a.Din, a.h, a.Hout, smem, ni);
      return STC_ERR_UNSUPPORTED;
    }
    target = (t.npt / 2) * a.C;
    if (target < a.C) target = a.C;
  }
  *tp = t; *smemp = smem; *nip = ni; *DPp = DP;
  return STC_OK;
}

size_t conv_dx_general_det_floats(const ConvArgs& a0) {
  ConvArgs a = a0;
  a.dQ = reinterpret_cast<float*>(16);   // sized with the dT_c(Gc) pass (the smaller tile, the larger grid)
  ConvTile t; size_t smem; int ni, DP;
  if (a.B <= 0 || conv_dx_general_tile(a, &t, &smem, &ni, &DP) != STC_OK) return 0;
  const long long grid = ceil_div((long long)a.B * a.N, t.npt);
  return (size_t)grid * (a.Hout + (size_t)a.Ks * (a.Kc - 1) * a.C * a.C);
}

int launch_conv_bwd_dx(const ConvArgs& a, cudaStream_t st) {
  {
    bool handled = false;
    STC_TRY(try_launch_conv_bwd_dx_tc(a, st, &handled));
    if (handled) return STC_OK;
    STC_TRY(try_launch_conv_bwd_dx_big(a, st, &handled));
    if (handled) return STC_OK;
  }
  const int L = a.Din + a.h;
  ConvTile t; size_t smem; int ni, DP;
  STC_TRY(conv_dx_general_tile(a, &t, &smem, &ni, &DP));
  long long total_nodes = (long long)a.B * a.N;
  int grid = ceil_div(total_nodes, t.npt);
  const bool det = a.det_ws != nullptr;
  // compulsory traffic per row: candidate reads dH',u,c (3h), gates reads dH',u,c,H,r,d(rH) (6h) and writes
  // the direct dH terms (h); both write dpre (Hout) and the Ks adjoint terms (Ks*L; the gates pass re-reads
  // the x-part it accumulates into); the spatial terms are re-read only when dGc is wanted.
  const double R = (double)total_nodes * a.C;
  {
    ScopedKernelTimer _t(KK_CONV_BWD_DX, st,
                         4.0 * R * ((a.phase == 0 ? 7 * a.h + a.Ks * a.Din : 3 * a.h) + a.Hout + a.Ks * L +
                                    ((a.dQ && a.Kc > 1) ? a.Ks * L : 0)) + 4.0 * a.Ks * a.Kc * L * a.Hout);
#define STC_DX_LAUNCH(K, N) \
  do { STC_TRY(set_smem(K<N>, smem)); K<N><<<grid, CV_THREADS, smem, st>>>(a, t, DP); } while (0)
    switch (ni) {
      case 1: if (det) STC_DX_LAUNCH(gen_det_bwd_dx_kernel, 1); else STC_DX_LAUNCH(conv_bwd_dx_kernel, 1); break;
      case 2: if (det) STC_DX_LAUNCH(gen_det_bwd_dx_kernel, 2); else STC_DX_LAUNCH(conv_bwd_dx_kernel, 2); break;
      default: if (det) STC_DX_LAUNCH(gen_det_bwd_dx_kernel, 4); else STC_DX_LAUNCH(conv_bwd_dx_kernel, 4); break;
    }
#undef STC_DX_LAUNCH
    STC_LAUNCH_OK("conv_bwd_dx_kernel");
  }
  if (!det) return STC_OK;
  // slots [grid][Hout | Ks x (Kc-1) x C x C]: the bias over the CTAs, then dT_c(Gc) over the CTAs of each term k in turn
  const long long npairs = (long long)(a.Kc - 1) * a.C * a.C, stride = a.Hout + a.Ks * npairs;
  if (a.dbias) STC_TRY(launch_det_reduce(a.dbias, a.det_ws, grid, a.Hout, stride, st));
  if (a.dQ && npairs)
    for (int k = 0; k < a.Ks; ++k)
      STC_TRY(launch_det_reduce(a.dQ + (size_t)a.C * a.C, a.det_ws + a.Hout + k * npairs, grid, npairs, stride, st));
  return STC_OK;
}

// =================================================================================================
// backward, part 2: dW_{k,c}[l][j] += sum_rows F_{k,c}[row][l] * dpre[row][j]
//   grid = (row chunks, Ks*Kc blocks, 64-column slabs of Hout); per-CTA register accumulation over its
//   chunk of tiles, one atomicAdd per element per CTA at the end.
// =================================================================================================
constexpr int DW_SLAB = 64;

// DET (deterministic mode): row group g of row chunk blockIdx.x stores its partial into slot blockIdx.x * Gmax + g of
// a.det_ws (Ks*Kc*L*Hout floats each; Gmax = the row-group count of the narrowest column slab; slot parts no group
// writes were zeroed before the launch) instead of adding it with atomics.
template <int NI, bool DET>
__device__ __forceinline__ void conv_bwd_dw_body(const ConvArgs& a, const ConvTile& t, const int tiles_per_cta) {
  extern __shared__ __align__(16) float smem[];
  const int C = a.C, L = t.L, LP4 = t.LP4, Hout = a.Hout;
  const int blk = blockIdx.y, k = blk / a.Kc, c = blk - k * a.Kc;
  const int col0 = blockIdx.z * DW_SLAB;
  const int ncol = min(DW_SLAB, Hout - col0);
  const int SP = (ncol + 3) & ~3;
  float* Fin = smem;                                     // [rowsP][LP4]
  float* Fmx = Fin + (size_t)t.rowsP * LP4;              // [rowsP][LP4] (c > 0)
  float* Dsm = Fmx + (c > 0 ? (size_t)t.rowsP * LP4 : 0);  // [rowsP][SP]
  float* Qs = Dsm + (size_t)t.rowsP * DW_SLAB;           // [C][C]
  const FeatSrc fs = feat_src(a);
  const long long total_nodes = (long long)a.B * a.N;
  const long long ntiles = (total_nodes + t.npt - 1) / t.npt;

  if (c > 0)
    for (int i = threadIdx.x; i < C * C; i += blockDim.x) Qs[i] = a.Q[(size_t)c * C * C + i];

  const int LG = LP4 / 4, CG = SP / 4, IT = LG * CG;
  // thread -> (row group g of G, item); when IT >= 256 every thread owns NI items and G = 1
  int G = 1, g = 0, item0 = threadIdx.x;
  bool active = true;
  if (IT < CV_THREADS) {
    G = CV_THREADS / IT;
    g = threadIdx.x / IT;
    item0 = threadIdx.x - g * IT;
    active = g < G;
  }
  float acc[NI][4][4];
#pragma unroll
  for (int i = 0; i < NI; ++i)
#pragma unroll
    for (int x = 0; x < 4; ++x)
#pragma unroll
      for (int y = 0; y < 4; ++y) acc[i][x][y] = 0.f;

  // zero the padding columns of the feature tiles once (they are read as float4)
  for (int idx = threadIdx.x; idx < t.rowsP * LP4 * (c > 0 ? 2 : 1); idx += blockDim.x) Fin[idx] = 0.f;

  const long long tile_lo = (long long)blockIdx.x * tiles_per_cta;
  const long long tile_hi = min(ntiles, tile_lo + tiles_per_cta);
  for (long long tile = tile_lo; tile < tile_hi; ++tile) {
    const long long g0 = tile * t.npt;
    const int nodes_valid = (int)min((long long)t.npt, total_nodes - g0);
    const int rows_valid = nodes_valid * C;
    const long long row0 = g0 * C;
    __syncthreads();
    load_feat_tile(fs, k, g0, nodes_valid, rows_valid, Fin, LP4);
    for (int idx = threadIdx.x; idx < rows_valid * SP; idx += blockDim.x) {
      int row = idx / SP, j = idx - row * SP;
      Dsm[row * SP + j] = (j < ncol) ? a.dpre[(row0 + row) * a.dpre_ld + col0 + j] : 0.f;
    }
    __syncthreads();
    const float* F = Fin;
    if (c > 0) {
      mix_tile(Fin, Fmx, Qs, rows_valid, C, L, LP4);
      F = Fmx;
      __syncthreads();
    }
    if (active) {
#pragma unroll
      for (int i = 0; i < NI; ++i) {
        const int it = item0 + i * CV_THREADS;
        if (it >= IT) break;
        const int lg = it / CG, cg = it - lg * CG;
        for (int row = g; row < rows_valid; row += G) {
          float4 f = *reinterpret_cast<const float4*>(F + row * LP4 + lg * 4);
          float4 d = *reinterpret_cast<const float4*>(Dsm + row * SP + cg * 4);
          acc[i][0][0] = fmaf(f.x, d.x, acc[i][0][0]); acc[i][0][1] = fmaf(f.x, d.y, acc[i][0][1]);
          acc[i][0][2] = fmaf(f.x, d.z, acc[i][0][2]); acc[i][0][3] = fmaf(f.x, d.w, acc[i][0][3]);
          acc[i][1][0] = fmaf(f.y, d.x, acc[i][1][0]); acc[i][1][1] = fmaf(f.y, d.y, acc[i][1][1]);
          acc[i][1][2] = fmaf(f.y, d.z, acc[i][1][2]); acc[i][1][3] = fmaf(f.y, d.w, acc[i][1][3]);
          acc[i][2][0] = fmaf(f.z, d.x, acc[i][2][0]); acc[i][2][1] = fmaf(f.z, d.y, acc[i][2][1]);
          acc[i][2][2] = fmaf(f.z, d.z, acc[i][2][2]); acc[i][2][3] = fmaf(f.z, d.w, acc[i][2][3]);
          acc[i][3][0] = fmaf(f.w, d.x, acc[i][3][0]); acc[i][3][1] = fmaf(f.w, d.y, acc[i][3][1]);
          acc[i][3][2] = fmaf(f.w, d.z, acc[i][3][2]); acc[i][3][3] = fmaf(f.w, d.w, acc[i][3][3]);
        }
      }
    }
  }
  if (active) {
    float* dWblk = a.dW + (size_t)blk * L * Hout;
    if constexpr (DET) {
      const int ncl = Hout - ((int)gridDim.z - 1) * DW_SLAB, ITl = LG * (((ncl + 3) & ~3) / 4);
      const int Gmax = max(G, ITl < CV_THREADS ? CV_THREADS / ITl : 1);
      dWblk = a.det_ws + ((size_t)blockIdx.x * Gmax + g) * a.Ks * a.Kc * L * Hout + (size_t)blk * L * Hout;
    }
#pragma unroll
    for (int i = 0; i < NI; ++i) {
      const int it = item0 + i * CV_THREADS;
      if (it >= IT) break;
      const int lg = it / CG, cg = it - lg * CG;
#pragma unroll
      for (int x = 0; x < 4; ++x) {
        const int l = lg * 4 + x;
        if (l >= L) continue;
#pragma unroll
        for (int y = 0; y < 4; ++y) {
          const int j = cg * 4 + y;
          if (j >= ncol) continue;
          if constexpr (DET) dWblk[(size_t)l * Hout + col0 + j] = acc[i][x][y];
          else atomicAdd(&dWblk[(size_t)l * Hout + col0 + j], acc[i][x][y]);
        }
      }
    }
  }
}

template <int NI>
__global__ void __launch_bounds__(CV_THREADS)
conv_bwd_dw_kernel(const ConvArgs a, const ConvTile t, const int tiles_per_cta) { conv_bwd_dw_body<NI, false>(a, t, tiles_per_cta); }
// the deterministic-mode instantiation, under a name of its own (the convolution variant list names the default kernels)
template <int NI>
__global__ void __launch_bounds__(CV_THREADS)
gen_det_bwd_dw_kernel(const ConvArgs a, const ConvTile t, const int tiles_per_cta) { conv_bwd_dw_body<NI, true>(a, t, tiles_per_cta); }

// grid and tile of the general dW kernel; *slots = the deterministic form's slot count (row chunks x row groups of the
// narrowest column slab)
struct DwGeneralPlan {
  ConvTile t;
  size_t smem;
  int ni, chunks, tiles_per_cta, slabs, slots;
};
static int conv_dw_general_plan(const ConvArgs& a, DwGeneralPlan* pl) {
  const int L = a.Din + a.h;
  const int LP4 = (L + 3) & ~3;
  int slabs = ceil_div(a.Hout, DW_SLAB);
  int ncol_max = a.Hout < DW_SLAB ? a.Hout : DW_SLAB;
  int IT = (LP4 / 4) * (((ncol_max + 3) & ~3) / 4);
  int ni = IT >= CV_THREADS ? ceil_div(IT, CV_THREADS) : 1;
  if (ni > CV_MAX_NI) {
    set_error("dW tile does not fit: Din+h=%d is larger than %d", L, CV_MAX_NI * CV_THREADS * 16 / DW_SLAB);
    return STC_ERR_UNSUPPORTED;
  }
  int target = 64;
  ConvTile t; size_t smem;
  for (;;) {
    t = make_tile(a, target);
    smem = ((size_t)t.rowsP * t.LP4 * 2 + (size_t)t.rowsP * DW_SLAB + (size_t)a.C * a.C) * sizeof(float);
    if (smem <= 200 * 1024) break;
    if (t.npt == 1) {
      set_error("dW tile does not fit in shared memory: C=%d Din+h=%d needs %zu B", a.C, L, smem);
      return STC_ERR_UNSUPPORTED;
    }
    target = (t.npt / 2) * a.C;
    if (target < a.C) target = a.C;
  }
  long long total_nodes = (long long)a.B * a.N;
  long long ntiles = (total_nodes + t.npt - 1) / t.npt;
  int P = a.Ks * a.Kc;
  long long want_chunks = (long long)device_sm_count() * 4 / (P * slabs);
  if (want_chunks < 1) want_chunks = 1;
  if (want_chunks > ntiles) want_chunks = ntiles;
  pl->t = t;
  pl->smem = smem;
  pl->ni = ni;
  pl->tiles_per_cta = ceil_div(ntiles, want_chunks);
  pl->chunks = ceil_div(ntiles, pl->tiles_per_cta);
  pl->slabs = slabs;
  const int ncl = a.Hout - (slabs - 1) * DW_SLAB, ITl = (LP4 / 4) * (((ncl + 3) & ~3) / 4);
  const int ITf = (LP4 / 4) * (((ncol_max + 3) & ~3) / 4);
  const int Gl = ITl < CV_THREADS ? CV_THREADS / ITl : 1, Gf = ITf < CV_THREADS ? CV_THREADS / ITf : 1;
  pl->slots = pl->chunks * (Gl > Gf ? Gl : Gf);
  return STC_OK;
}

size_t conv_dw_general_det_floats(const ConvArgs& a) {
  DwGeneralPlan pl;
  if (a.B <= 0 || conv_dw_general_plan(a, &pl) != STC_OK) return 0;
  return (size_t)pl.slots * a.Ks * a.Kc * (a.Din + a.h) * a.Hout;
}

int launch_conv_bwd_dw(const ConvArgs& a, cudaStream_t st) {
  {
    bool handled = false;
    STC_TRY(try_launch_conv_bwd_dw_tc(a, st, &handled));
    if (handled) return STC_OK;
    STC_TRY(try_launch_conv_bwd_dw_big(a, st, &handled));
    if (handled) return STC_OK;
  }
  const int L = a.Din + a.h;
  DwGeneralPlan pl;
  STC_TRY(conv_dw_general_plan(a, &pl));
  const ConvTile& t = pl.t;
  const size_t smem = pl.smem;
  const int tiles_per_cta = pl.tiles_per_cta, P = a.Ks * a.Kc;
  long long total_nodes = (long long)a.B * a.N;
  dim3 grid(pl.chunks, P, pl.slabs);
  const bool det = a.det_ws != nullptr;
  const size_t slot = (size_t)P * L * a.Hout;
  // (deterministic mode: a slot part that no row group of a narrower-than-widest slab writes must read as zero)
  if (det) STC_CUDA_OK(cudaMemsetAsync(a.det_ws, 0, sizeof(float) * pl.slots * slot, st));
  {
    // compulsory traffic per row: the Ks spatial terms once and dpre once; plus the dW block written
    ScopedKernelTimer _t(KK_CONV_BWD_DW, st,
                         4.0 * (double)total_nodes * a.C * (a.Ks * L + a.Hout) + 4.0 * P * L * a.Hout);
#define STC_DW_LAUNCH(K, N) \
  do { STC_TRY(set_smem(K<N>, smem)); K<N><<<grid, CV_THREADS, smem, st>>>(a, t, tiles_per_cta); } while (0)
    switch (pl.ni) {
      case 1: if (det) STC_DW_LAUNCH(gen_det_bwd_dw_kernel, 1); else STC_DW_LAUNCH(conv_bwd_dw_kernel, 1); break;
      case 2: if (det) STC_DW_LAUNCH(gen_det_bwd_dw_kernel, 2); else STC_DW_LAUNCH(conv_bwd_dw_kernel, 2); break;
      default: if (det) STC_DW_LAUNCH(gen_det_bwd_dw_kernel, 4); else STC_DW_LAUNCH(conv_bwd_dw_kernel, 4); break;
    }
#undef STC_DW_LAUNCH
    STC_LAUNCH_OK("conv_bwd_dw_kernel");
  }
  if (!det) return STC_OK;
  return launch_det_reduce(a.dW, a.det_ws, pl.slots, (long long)slot, (long long)slot, st);
}

}  // namespace stc
