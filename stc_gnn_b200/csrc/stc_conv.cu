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

  // epilogue
  const long long row0 = g0 * C;
  const int items = RG * CG;
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
            a.r[o] = s;
            a.rH[o] = s * a.Hprev[o];
          }
        } else {
          const long long o = gr * h + col;
          float cc = tanhf(pre);
          float uu = a.u[o], hp = a.Hprev[o];
          a.c[o] = cc;
          a.Hnew[o] = fmaf(uu, cc - hp, hp);  // (1-u)*H + u*c
        }
      }
    }
  }
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
  // compulsory traffic per row: the Ks spatial terms of [x|h] once, then gates: write u, r, r*H;
  // candidate: read u, H, write c, H'.  Plus the weights.
  const double R = (double)total_nodes * a.C;
  ScopedKernelTimer _t(KK_CONV_FWD, st,
                       4.0 * R * (a.Ks * t.L + (a.phase == 0 ? 3 * a.h : 4 * a.h)) + 4.0 * a.Ks * a.Kc * t.L * a.Hout);
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
template <int NI>
__global__ void __launch_bounds__(CV_THREADS)
conv_bwd_dx_kernel(const ConvArgs a, const ConvTile t, const int DP) {
  extern __shared__ __align__(16) float smem[];
  const int C = a.C, L = t.L, LP = t.LP, LP4 = t.LP4, Hout = a.Hout, h = a.h, Din = a.Din;
  const bool mixed = a.Kc > 1;
  const bool want_dQ = mixed && a.dQ != nullptr;
  float* Ds = smem;                                   // [rowsP][DP]      pre-activation gradient
  float* WsT = Ds + (size_t)t.rowsP * DP;             // [Hout][LP4]      W_{k,c}^T
  float* DY = WsT + (size_t)Hout * LP4;               // [rowsP][LP]      adjoint of spatial term k
  float* DF = DY + (size_t)t.rowsP * LP;              // [rowsP][LP]      dF_{k,c}, c > 0
  float* Fin = DF + (mixed ? (size_t)t.rowsP * LP : 0);  // [rowsP][LP]   Y_k (only for dQ)
  float* Qs = Fin + (want_dQ ? (size_t)t.rowsP * LP : 0);

  const long long total_nodes = (long long)a.B * a.N;
  const long long g0 = (long long)blockIdx.x * t.npt;
  const int nodes_valid = (int)min((long long)t.npt, total_nodes - g0);
  const int rows_valid = nodes_valid * C;
  const long long row0 = g0 * C;
  const long long R = total_nodes * C;
  const FeatSrc fs = feat_src(a);
  const int RG = t.rowsP / 4, CGL = LP4 / 4;

  for (int i = threadIdx.x; i < (a.Kc - 1) * C * C; i += blockDim.x) Qs[i] = a.Q[C * C + i];

  // ---- step 1: elementwise GRU adjoint -> Ds, dpre (global), direct dH terms ----
  for (int idx = threadIdx.x; idx < t.rowsP * h; idx += blockDim.x) {
    const int row = idx / h, j = idx - row * h;
    const long long o = (row0 + row) * h + j;
    if (row < rows_valid) {
      const float dhn = a.dHn[o], uu = a.u[o], cc = a.c[o];
      if (a.phase == 1) {
        float g = dhn * uu * (1.f - cc * cc);
        if (a.act == STC_ACT_RELU && !(cc > 0.f)) g = 0.f;
        Ds[row * DP + j] = g;
        a.dpre[(row0 + row) * a.dpre_ld + j] = g;
      } else {
        const float hp = a.Hprev[o], rr = a.r[o], drh = a.drH[o];
        float gu = dhn * (cc - hp) * uu * (1.f - uu);
        float gr = drh * hp * rr * (1.f - rr);
        if (a.act == STC_ACT_RELU) {
          if (!(uu > 0.5f)) gu = 0.f;
          if (!(rr > 0.5f)) gr = 0.f;
        }
        Ds[row * DP + j] = gu;
        Ds[row * DP + h + j] = gr;
        a.dpre[(row0 + row) * a.dpre_ld + j] = gu;
        a.dpre[(row0 + row) * a.dpre_ld + h + j] = gr;
        a.dYh0[o] = dhn * (1.f - uu) + drh * rr;   // direct terms of dH; the conv adjoint is added below
      }
    } else {
      Ds[row * DP + j] = 0.f;
      if (a.phase == 0) Ds[row * DP + h + j] = 0.f;
    }
  }
  __syncthreads();
  if (a.dbias) {
    for (int j = threadIdx.x; j < Hout; j += blockDim.x) {
      float s = 0.f;
      for (int row = 0; row < rows_valid; ++row) s += Ds[row * DP + j];
      atomicAdd(&a.dbias[j], s);
    }
  }

  // ---- step 2: per spatial term k, dY_k = sum_c unmix_c( Ds W_{k,c}^T ) ----
  for (int k = 0; k < a.Ks; ++k) {
    __syncthreads();
    for (int idx = threadIdx.x; idx < t.rowsP * LP; idx += blockDim.x) DY[idx] = 0.f;
    if (want_dQ) load_feat_tile(fs, k, g0, nodes_valid, t.rowsP, Fin, LP);
    for (int c = 0; c < a.Kc; ++c) {
      __syncthreads();
      const float* Wblk = a.W + (size_t)(k * a.Kc + c) * L * Hout;
      for (int idx = threadIdx.x; idx < Hout * LP4; idx += blockDim.x) {
        int j = idx / LP4, l = idx - j * LP4;
        WsT[idx] = (l < L) ? Wblk[l * Hout + j] : 0.f;
      }
      __syncthreads();
      float acc[NI][4][4];
#pragma unroll
      for (int i = 0; i < NI; ++i)
#pragma unroll
        for (int x = 0; x < 4; ++x)
#pragma unroll
          for (int y = 0; y < 4; ++y) acc[i][x][y] = 0.f;
      tile_gemm<NI>(acc, Ds, DP, WsT, LP4, Hout, RG, CGL);
      float* dst = (c == 0) ? DY : DF;
      const int items = RG * CGL;
#pragma unroll
      for (int i = 0; i < NI; ++i) {
        const int it = threadIdx.x + i * CV_THREADS;
        if (it >= items) break;
        const int rg = it / CGL, lg = it - rg * CGL;
#pragma unroll
        for (int x = 0; x < 4; ++x)
#pragma unroll
          for (int y = 0; y < 4; ++y) {
            const int l = lg * 4 + y;
            if (l < L) {
              float* p = dst + (rg * 4 + x) * LP + l;
              if (c == 0) *p += acc[i][x][y]; else *p = acc[i][x][y];
            }
          }
      }
      if (c > 0) {
        __syncthreads();
        const float* Qc = Qs + (size_t)(c - 1) * C * C;
        unmix_add_tile(DF, DY, Qc, rows_valid, C, L, LP);
        if (want_dQ) {
          // dQ_c[c'][d] += sum_{node,l} Y_k[(node,c')][l] * dF[(node,d)][l]
          for (int pr = threadIdx.x; pr < C * C; pr += blockDim.x) {
            const int cp = pr / C, d = pr - cp * C;
            float s = 0.f;
            for (int node = 0; node < nodes_valid; ++node) {
              const float* y = Fin + (node * C + cp) * LP;
              const float* f = DF + (node * C + d) * LP;
              for (int l = 0; l < L; ++l) s = fmaf(y[l], f[l], s);
            }
            atomicAdd(&a.dQ[(size_t)c * C * C + pr], s);
          }
        }
      }
    }
    __syncthreads();
    // write DY: x-part then h-part
    {
      float* dx = (k == 0) ? a.dYx0 : a.dYx + (size_t)(k - 1) * R * Din;
      if (dx) {
        dx += row0 * Din;
        // prior contents: the other convolution's x-part (accum_x), else a folded adjoint of the term (k >= 1)
        const float* xprior = a.accum_x ? dx
                              : (k >= 1 && a.dYx_add) ? a.dYx_add + (size_t)(k - 1) * R * Din + row0 * Din : nullptr;
        for (int idx = threadIdx.x; idx < rows_valid * Din; idx += blockDim.x) {
          int row = idx / Din, l = idx - row * Din;
          float v = DY[row * LP + l];
          dx[idx] = xprior ? xprior[idx] + v : v;
        }
      }
      float* dh = (k == 0) ? a.dYh0 : a.dYh + (size_t)(k - 1) * R * h;
      dh += row0 * h;
      const float* hprior = (k == 0 && a.phase == 0) ? dh   // direct terms of dH
                            : (k >= 1 && a.dYh_add) ? a.dYh_add + (size_t)(k - 1) * R * h + row0 * h : nullptr;
      for (int idx = threadIdx.x; idx < rows_valid * h; idx += blockDim.x) {
        int row = idx / h, l = idx - row * h;
        float v = DY[row * LP + Din + l];
        dh[idx] = hprior ? hprior[idx] + v : v;
      }
    }
  }
}

static size_t conv_dx_smem(const ConvArgs& a, const ConvTile& t, int DP) {
  const bool mixed = a.Kc > 1;
  const bool want_dQ = mixed && a.dQ != nullptr;
  size_t f = (size_t)t.rowsP * DP + (size_t)a.Hout * t.LP4 + (size_t)t.rowsP * t.LP * (1 + (mixed ? 1 : 0) + (want_dQ ? 1 : 0)) +
             (size_t)(mixed ? (a.Kc - 1) : 0) * a.C * a.C;
  return f * sizeof(float);
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
  long long total_nodes = (long long)a.B * a.N;
  int grid = ceil_div(total_nodes, t.npt);
  // compulsory traffic per row: candidate reads dH',u,c (3h), gates reads dH',u,c,H,r,d(rH) (6h) and writes
  // the direct dH terms (h); both write dpre (Hout) and the Ks adjoint terms (Ks*L; the gates pass re-reads
  // the x-part it accumulates into); the spatial terms are re-read only when dGc is wanted.
  const double R = (double)total_nodes * a.C;
  ScopedKernelTimer _t(KK_CONV_BWD_DX, st,
                       4.0 * R * ((a.phase == 0 ? 7 * a.h + a.Ks * a.Din : 3 * a.h) + a.Hout + a.Ks * L +
                                  ((a.dQ && a.Kc > 1) ? a.Ks * L : 0)) + 4.0 * a.Ks * a.Kc * L * a.Hout);
  switch (ni) {
    case 1: STC_TRY(set_smem(conv_bwd_dx_kernel<1>, smem)); conv_bwd_dx_kernel<1><<<grid, CV_THREADS, smem, st>>>(a, t, DP); break;
    case 2: STC_TRY(set_smem(conv_bwd_dx_kernel<2>, smem)); conv_bwd_dx_kernel<2><<<grid, CV_THREADS, smem, st>>>(a, t, DP); break;
    default: STC_TRY(set_smem(conv_bwd_dx_kernel<4>, smem)); conv_bwd_dx_kernel<4><<<grid, CV_THREADS, smem, st>>>(a, t, DP); break;
  }
  STC_LAUNCH_OK("conv_bwd_dx_kernel");
  return STC_OK;
}

// =================================================================================================
// backward, part 2: dW_{k,c}[l][j] += sum_rows F_{k,c}[row][l] * dpre[row][j]
//   grid = (row chunks, Ks*Kc blocks, 64-column slabs of Hout); per-CTA register accumulation over its
//   chunk of tiles, one atomicAdd per element per CTA at the end.
// =================================================================================================
constexpr int DW_SLAB = 64;

template <int NI>
__global__ void __launch_bounds__(CV_THREADS)
conv_bwd_dw_kernel(const ConvArgs a, const ConvTile t, const int tiles_per_cta) {
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
          if (j < ncol) atomicAdd(&dWblk[(size_t)l * Hout + col0 + j], acc[i][x][y]);
        }
      }
    }
  }
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
  int tiles_per_cta = ceil_div(ntiles, want_chunks);
  int chunks = ceil_div(ntiles, tiles_per_cta);
  dim3 grid(chunks, P, slabs);
  // compulsory traffic per row: the Ks spatial terms once and dpre once; plus the dW block written
  ScopedKernelTimer _t(KK_CONV_BWD_DW, st,
                       4.0 * (double)total_nodes * a.C * (a.Ks * L + a.Hout) + 4.0 * P * L * a.Hout);
  switch (ni) {
    case 1: STC_TRY(set_smem(conv_bwd_dw_kernel<1>, smem)); conv_bwd_dw_kernel<1><<<grid, CV_THREADS, smem, st>>>(a, t, tiles_per_cta); break;
    case 2: STC_TRY(set_smem(conv_bwd_dw_kernel<2>, smem)); conv_bwd_dw_kernel<2><<<grid, CV_THREADS, smem, st>>>(a, t, tiles_per_cta); break;
    default: STC_TRY(set_smem(conv_bwd_dw_kernel<4>, smem)); conv_bwd_dw_kernel<4><<<grid, CV_THREADS, smem, st>>>(a, t, tiles_per_cta); break;
  }
  STC_LAUNCH_OK("conv_bwd_dw_kernel");
  return STC_OK;
}

}  // namespace stc
