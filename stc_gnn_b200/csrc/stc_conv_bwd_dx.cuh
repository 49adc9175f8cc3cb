// Body of the general (FFMA) convolution input-adjoint kernel, included twice by stc_conv.cu:
//   STC_DX_DET 0: conv_bwd_dx_kernel, the bias and dT_c(Gc) sums of each CTA are added with atomics;
//   STC_DX_DET 1: gen_det_bwd_dx_kernel (deterministic mode), the CTA stores them into its slot of a.det_ws
//                 ([Hout | Ks x (Kc-1) x C x C] floats), summed in slot order afterwards (launch_det_reduce).
// Two preprocessor passes rather than a template flag: the default kernel is then exactly its earlier code (a template
// body changed its register allocation), and the deterministic one carries a name outside the convolution variant list.
// (no include guard: included once per form)

template <int NI>
__global__ void __launch_bounds__(CV_THREADS)
STC_DX_KERNEL_NAME(const ConvArgs a, const ConvTile t, const int DP) {
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
#if STC_DX_DET
      a.det_ws[(size_t)blockIdx.x * (Hout + a.Ks * (a.Kc - 1) * C * C) + j] = s;
#else
      atomicAdd(&a.dbias[j], s);
#endif
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
#if STC_DX_DET
            a.det_ws[(size_t)blockIdx.x * (Hout + a.Ks * (a.Kc - 1) * C * C) + Hout + ((size_t)k * (a.Kc - 1) + c - 1) * C * C +
                     pr] = s;
#else
            atomicAdd(&a.dQ[(size_t)c * C * C + pr], s);
#endif
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
