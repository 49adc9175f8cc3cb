// tcgen05 / TMEM version of the gate / candidate weight contraction with the categorical mix and the GRU
// epilogue fused (forward).  Replaces conv_fwd_kernel (stc_conv.cu) whenever the shape is eligible; the
// arithmetic is the reference's 'bmdk,kh->bmdh' (/root/reference/framework/STC_GNN.py:42) evaluated as a
// 3xTF32 tensor-core product (see stc_tc.cuh), bias/activation (:44-46) and sigmoid / tanh / blend
// (STC_GNN.py:71-78) applied on the accumulator as it is read back from TMEM.
//
// One persistent CTA per SM slot.  Per 128-row tile (whole nodes x all categories):
//   for each spatial Chebyshev term k:  stage [rows][L] fp32 <- HBM (x-part | h-part)
//     for each categorical term c and each 32-wide K atom j:
//        CUDA cores build the A atom (mix with T_c(Gc) on the fly, split hi/lo, 128B-swizzled K-major)
//        into one of two buffers; one thread issues 3 x ksteps tcgen05.mma against the resident W atoms;
//        tcgen05.commit -> mbarrier releases the buffer two atoms later.
//   epilogue: TMEM -> registers (tcgen05.ld 32x32b), bias, activation, sigmoid/tanh, GRU blend, stores.
#include "stc_conv_common.cuh"
#include "stc_tc.cuh"

#include <stdlib.h>

namespace stc {

using namespace tc;

// Formulation.  With P_c = sum_k Y_k W_{k,c}  (Y_k the k-th spatial term of [Xt | H], rows = (node, category)),
//     out[(node,d)] = P_0[(node,d)] + sum_{c>=1} sum_{c'} T_c(Gc)[c',d] * P_c[(node,c')]
// i.e. the categorical mode product is applied to the GEMM *output* (Hout wide) instead of to the features
// (K wide): the A operand is the raw staged tile, the GEMM is [rows x Ks*KBL] x [Ks*KBL x Kc*Hout], and the
// C x C mix runs in the epilogue on values read back from TMEM.  Same arithmetic as STC_GNN.py:35-45 with the
// two linear maps commuted.
//
// K layout of one spatial term: [ h-part (h floats) | x-part (Din floats, zero-padded to Dp) ] so that 16-byte
// chunks never straddle the two source tensors; the rows of W are permuted to match in the resident B atoms.
struct TcFwdPlan {
  int npt;        // nodes per tile (rows = npt*C <= 128)
  int Dp;         // Din rounded up to 8
  int KBL;        // h + Dp
  int KB;         // 32-wide atoms per spatial term
  int Ntot;       // Kc * Hout (GEMM N)
  int Npad;       // Ntot rounded up to 16
  int nacc;       // atoms along K = Ks*KB
  int nmain;      // main accumulators = ceil(nacc / TC_APM); the cross-term accumulator follows them
  int tmem_cols;  // power of two
  int ntiles;
  int x_bulk;     // x-part can be staged with bulk copies (16-byte aligned rows)
  int PS;         // row stride (floats) of the epilogue exchange buffer
  uint32_t off_a, off_b, off_sh, off_sx, off_se, off_q, off_bias, off_bar, smem_bytes;
};

// thread 0: stage every spatial term of tile `tile` with bulk copies that complete on `bar`
__device__ __forceinline__ void tc_issue_tile_loads(const ConvArgs& a, const TcFwdPlan& p, int tile, float* stage_h,
                                                    float* stage_x, uint64_t* bar) {
  const long long total_nodes = (long long)a.B * a.N;
  const long long g0 = (long long)tile * p.npt;
  const int nv = (int)min((long long)p.npt, total_nodes - g0);
  const long long R = total_nodes * a.C;
  const int CH = a.C * a.h, CD = a.C * a.Din;
  uint32_t bytes = (uint32_t)(a.Ks * nv * CH * 4);
  if (p.x_bulk) bytes += (uint32_t)(a.Ks * nv * CD * 4);
  mbar_arrive_expect_tx(bar, bytes);
  for (int k = 0; k < a.Ks; ++k) {
    const float* hsrc = (k == 0 ? a.h0 : a.yh + (long long)(k - 1) * R * a.h) + g0 * CH;
    bulk_g2s(stage_h + (size_t)k * 128 * a.h, hsrc, (uint32_t)(nv * CH * 4), bar);
    if (!p.x_bulk) continue;
    float* dst = stage_x + (size_t)k * 128 * a.Din;
    if (k > 0) {
      bulk_g2s(dst, a.yx + (long long)(k - 1) * R * a.Din + g0 * CD, (uint32_t)(nv * CD * 4), bar);
    } else {  // Xt carries a batch stride: one copy per sample segment
      long long g = g0;
      int left = nv;
      while (left > 0) {
        const long long b = g / a.N;
        const int m = (int)(g - b * a.N);
        const int seg = min(left, a.N - m);
        bulk_g2s(dst, a.x0 + b * a.x0_bs + (long long)m * CD, (uint32_t)(seg * CD * 4), bar);
        dst += seg * CD;
        g += seg;
        left -= seg;
      }
    }
  }
}

// one lane: pull tile `tile`'s spatial terms and epilogue operands towards L2 (same ranges as tc_issue_tile_loads)
__device__ __forceinline__ void tc_prefetch_tile(const ConvArgs& a, const TcFwdPlan& p, int tile) {
  const long long total_nodes = (long long)a.B * a.N;
  const long long g0 = (long long)tile * p.npt;
  const int nv = (int)min((long long)p.npt, total_nodes - g0);
  const long long R = total_nodes * a.C;
  const int CH = a.C * a.h, CD = a.C * a.Din;
  const uint32_t hb = (uint32_t)(nv * CH * 4), xb = (uint32_t)(nv * CD * 4);
  for (int k = 0; k < a.Ks; ++k) {
    l2_prefetch((k == 0 ? a.h0 : a.yh + (long long)(k - 1) * R * a.h) + g0 * CH, hb);
    if (!p.x_bulk) continue;
    if (k > 0) {
      l2_prefetch(a.yx + (long long)(k - 1) * R * a.Din + g0 * CD, xb);
    } else {
      long long g = g0;
      int left = nv;
      while (left > 0) {
        const long long b = g / a.N;
        const int m = (int)(g - b * a.N);
        const int seg = min(left, a.N - m);
        l2_prefetch(a.x0 + b * a.x0_bs + (long long)m * CD, (uint32_t)(seg * CD * 4));
        g += seg;
        left -= seg;
      }
    }
  }
  if (a.Hprev != a.h0) l2_prefetch(a.Hprev + g0 * CH, hb);
  if (a.phase != 0) l2_prefetch(a.u + g0 * CH, hb);
}

constexpr int TC_APM = 3;  // atoms (4 K-steps each) chained into one main accumulator: 12 K-steps, inside the <= 13
                           // the accumulate-truncation measurements allow (profiles/r1_tc_precision.txt)

// sum of the partial accumulators of 8 columns starting at column c0 (cross terms first, fp32 RN adds)
__device__ __forceinline__ void tc_read_acc8(uint32_t tl, const TcFwdPlan& p, int c0, float (&v)[8]) {
  if (p.nmain == 1) {   // both accumulators in flight, one wait
    uint32_t t0[8], t1[8];
    tmem_ld8_async(tl + (uint32_t)(p.Npad + c0), t1);
    tmem_ld8_async(tl + (uint32_t)c0, t0);
    tmem_ld_wait();
    tmem_ld_pin8(t0); tmem_ld_pin8(t1);
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(t1[i]) + __uint_as_float(t0[i]);
    return;
  }
  float t[8];
  tmem_ld8(tl + (uint32_t)(p.nmain * p.Npad + c0), v);
  for (int m = 0; m < p.nmain; ++m) {
    tmem_ld8(tl + (uint32_t)(m * p.Npad + c0), t);
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] += t[i];
  }
}

// Epilogue of the common shape (Kc = 2, one main accumulator, Hout = 16 * NG): each thread owns accumulator row
// `erow` and NG groups of 8 output columns, group g at column 16 g + 8 half -- for the gates convolution (NG = 2)
// every thread produces 8 channels of u and the same 8 channels of r and r*H, so all eight warps carry the same load.
// All TMEM loads of a stage are in flight before one wait; one exchange of the P_1 tile through shared memory (one
// block-wide barrier) feeds the C x C categorical mix.
template <int NG>
__device__ __forceinline__ void tc_fwd_epilogue_fast(const ConvArgs& a, const TcFwdPlan& p, uint32_t tl, float* Pm,
                                                     const float* Qs, const float* bias_s, const float* stage_e,
                                                     int erow, int enode, int ecat, int half, bool valid,
                                                     long long gr) {
  const int h = a.h, C = a.C, Hout = a.Hout;
  const int cb = half * 8;
  uint32_t sm1[NG][8], mn1[NG][8];
#pragma unroll
  for (int g = 0; g < NG; ++g) {                                          // P_1: cross terms, then main
    tmem_ld8_async(tl + (uint32_t)(p.Npad + Hout + 16 * g + cb), sm1[g]);
    tmem_ld8_async(tl + (uint32_t)(Hout + 16 * g + cb), mn1[g]);
  }
  tmem_ld_wait();
#pragma unroll
  for (int g = 0; g < NG; ++g) {
    tmem_ld_pin8(sm1[g]); tmem_ld_pin8(mn1[g]);
    float t[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) t[i] = __uint_as_float(sm1[g][i]) + __uint_as_float(mn1[g][i]);
    float* pm = Pm + erow * p.PS + 16 * g + cb;
    *reinterpret_cast<float4*>(pm) = make_float4(t[0], t[1], t[2], t[3]);
    *reinterpret_cast<float4*>(pm + 4) = make_float4(t[4], t[5], t[6], t[7]);
    if (a.Psave && valid) {   // backward forms dGc from these partials (no recomputation of the GEMM)
      float* ps = a.Psave + gr * (long long)Hout + 16 * g + cb;
      *reinterpret_cast<float4*>(ps) = make_float4(t[0], t[1], t[2], t[3]);
      *reinterpret_cast<float4*>(ps + 4) = make_float4(t[4], t[5], t[6], t[7]);
    }
  }
  uint32_t sm0[NG][8], mn0[NG][8];
#pragma unroll
  for (int g = 0; g < NG; ++g) {                                          // P_0 travels under the barrier
    tmem_ld8_async(tl + (uint32_t)(p.Npad + 16 * g + cb), sm0[g]);
    tmem_ld8_async(tl + (uint32_t)(16 * g + cb), mn0[g]);
  }
  __syncthreads();
  tmem_ld_wait();
  float v[NG][8];
#pragma unroll
  for (int g = 0; g < NG; ++g) {
    tmem_ld_pin8(sm0[g]); tmem_ld_pin8(mn0[g]);
#pragma unroll
    for (int i = 0; i < 8; ++i) v[g][i] = __uint_as_float(sm0[g][i]) + __uint_as_float(mn0[g][i]);
  }
  {
    const float* pp = Pm + (enode * C) * p.PS + cb;
#pragma unroll 5
    for (int cp = 0; cp < C; ++cp) {
      const float w = Qs[cp * C + ecat];
#pragma unroll
      for (int g = 0; g < NG; ++g) {
        const float4 x0 = *reinterpret_cast<const float4*>(pp + cp * p.PS + 16 * g);
        const float4 x1 = *reinterpret_cast<const float4*>(pp + cp * p.PS + 16 * g + 4);
        v[g][0] = fmaf(w, x0.x, v[g][0]); v[g][1] = fmaf(w, x0.y, v[g][1]);
        v[g][2] = fmaf(w, x0.z, v[g][2]); v[g][3] = fmaf(w, x0.w, v[g][3]);
        v[g][4] = fmaf(w, x1.x, v[g][4]); v[g][5] = fmaf(w, x1.y, v[g][5]);
        v[g][6] = fmaf(w, x1.z, v[g][6]); v[g][7] = fmaf(w, x1.w, v[g][7]);
      }
    }
  }
  if (!valid) return;
#pragma unroll
  for (int g = 0; g < NG; ++g) {
    const float4 b0 = *reinterpret_cast<const float4*>(bias_s + 16 * g + cb);
    const float4 b1 = *reinterpret_cast<const float4*>(bias_s + 16 * g + cb + 4);
    v[g][0] += b0.x; v[g][1] += b0.y; v[g][2] += b0.z; v[g][3] += b0.w;
    v[g][4] += b1.x; v[g][5] += b1.y; v[g][6] += b1.z; v[g][7] += b1.w;
    if (a.act == STC_ACT_RELU) {
#pragma unroll
      for (int i = 0; i < 8; ++i) v[g][i] = fmaxf(v[g][i], 0.f);
    }
  }
  if (a.phase == 0) {   // Hout = 2h: column 16 g + cb + i is u channel (same index) while it is < h, r channel (index - h) after
#pragma unroll
    for (int g = 0; g < NG; ++g) {
#pragma unroll
      for (int i = 0; i < 8; ++i) v[g][i] = sigmoidf_fast(v[g][i]);
      const int col = 16 * g + cb;
      if (col < h) {
        float* dst = a.u + gr * h + col;
        *reinterpret_cast<float4*>(dst) = make_float4(v[g][0], v[g][1], v[g][2], v[g][3]);
        *reinterpret_cast<float4*>(dst + 4) = make_float4(v[g][4], v[g][5], v[g][6], v[g][7]);
      } else {
        const int ch = col - h;
        const float4 h0 = *reinterpret_cast<const float4*>(stage_e + erow * h + ch);
        const float4 h1 = *reinterpret_cast<const float4*>(stage_e + erow * h + ch + 4);
        if (a.r) {   // null in a forward-only call: only the backward reads r
          float* dr = a.r + gr * h + ch;
          *reinterpret_cast<float4*>(dr) = make_float4(v[g][0], v[g][1], v[g][2], v[g][3]);
          *reinterpret_cast<float4*>(dr + 4) = make_float4(v[g][4], v[g][5], v[g][6], v[g][7]);
        }
        float* drh = a.rH + gr * h + ch;
        *reinterpret_cast<float4*>(drh) = make_float4(v[g][0] * h0.x, v[g][1] * h0.y, v[g][2] * h0.z, v[g][3] * h0.w);
        *reinterpret_cast<float4*>(drh + 4) = make_float4(v[g][4] * h1.x, v[g][5] * h1.y, v[g][6] * h1.z, v[g][7] * h1.w);
      }
    }
  } else {              // Hout = h: c = tanh, H' = H + u (c - H)
#pragma unroll
    for (int g = 0; g < NG; ++g) {
      const int col = 16 * g + cb;
      const long long o = gr * h + col;
      float cc[8], hn[8];
      const float4 u0 = *reinterpret_cast<const float4*>(stage_e + 128 * h + erow * h + col);
      const float4 u1 = *reinterpret_cast<const float4*>(stage_e + 128 * h + erow * h + col + 4);
      const float4 p0 = *reinterpret_cast<const float4*>(stage_e + erow * h + col);
      const float4 p1 = *reinterpret_cast<const float4*>(stage_e + erow * h + col + 4);
      const float uu[8] = {u0.x, u0.y, u0.z, u0.w, u1.x, u1.y, u1.z, u1.w};
      const float hp[8] = {p0.x, p0.y, p0.z, p0.w, p1.x, p1.y, p1.z, p1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        cc[i] = tanhf_fast(v[g][i]);
        hn[i] = fmaf(uu[i], cc[i] - hp[i], hp[i]);
      }
      if (a.c) {   // null in a forward-only call: only the backward reads c
        *reinterpret_cast<float4*>(a.c + o) = make_float4(cc[0], cc[1], cc[2], cc[3]);
        *reinterpret_cast<float4*>(a.c + o + 4) = make_float4(cc[4], cc[5], cc[6], cc[7]);
      }
      *reinterpret_cast<float4*>(a.Hnew + o) = make_float4(hn[0], hn[1], hn[2], hn[3]);
      *reinterpret_cast<float4*>(a.Hnew + o + 4) = make_float4(hn[4], hn[5], hn[6], hn[7]);
    }
  }
}

// NG = 0: general epilogue (any Kc, any Hout % 16 == 0); NG = 1 / 2: tc_fwd_epilogue_fast
template <int NG>
__global__ void __launch_bounds__(CV_THREADS, 2)
tc_conv_fwd_kernel(const ConvArgs a, const TcFwdPlan p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((smem_u32(smem) & 1023u) != 0u) __trap();  // swizzled atoms need a 1024-byte aligned base
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int C = a.C, L = a.Din + a.h, h = a.h, Din = a.Din, Hout = a.Hout;
  const uint32_t atomA = 128 * ATOM_ROW_BYTES;            // 16 KB
  const uint32_t atomB = (uint32_t)p.Npad * ATOM_ROW_BYTES;
  uint8_t* A_hi = smem + p.off_a;
  uint8_t* A_lo = A_hi + atomA;
  float* Pm = reinterpret_cast<float*>(A_hi);             // epilogue exchange buffer aliases the A atoms
  uint8_t* B_hi = smem + p.off_b;                          // [Ks*KB][atomB]
  uint8_t* B_lo = B_hi + (size_t)p.nacc * atomB;
  float* stage_h = reinterpret_cast<float*>(smem + p.off_sh);   // [Ks][128][h]
  float* stage_x = reinterpret_cast<float*>(smem + p.off_sx);   // [Ks][128][Din]
  float* Qs = reinterpret_cast<float*>(smem + p.off_q);         // [(Kc-1)][C][C]
  float* bias_s = reinterpret_cast<float*>(smem + p.off_bias);  // [Hout] (zeros without a bias)
  float* stage_e = reinterpret_cast<float*>(smem + p.off_se);   // [2][128][h]: H tile, u tile (epilogue operands)
  uint64_t* mma_bar = reinterpret_cast<uint64_t*>(smem + p.off_bar);
  uint64_t* load_bar = mma_bar + 1;
  uint64_t* epi_bar = mma_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(mma_bar + 3);

  // ---- one-time setup ----
  if (tid == 0) {
    mbar_init(mma_bar, 1);
    mbar_init(load_bar, 1);
    mbar_init(epi_bar, 1);
    mbar_fence_init();
  }
  if (warp == 0) tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols);
  for (int i = tid; i < (a.Kc - 1) * C * C; i += CV_THREADS) Qs[i] = a.Q[C * C + i];
  for (int i = tid; i < Hout; i += CV_THREADS) bias_s[i] = a.bias ? a.bias[i] : 0.f;
  for (int i = tid; i < a.Ks * 128 * h; i += CV_THREADS) stage_h[i] = 0.f;
  for (int i = tid; i < a.Ks * 128 * Din; i += CV_THREADS) stage_x[i] = 0.f;
  // resident B atoms: Bt[(c,o)][kb] = W[((k*Kc + c)*L + l(kb))*Hout + o]
  for (int k = 0; k < a.Ks; ++k)
    for (int j = 0; j < p.KB; ++j) {
      uint8_t* bh = B_hi + (size_t)(k * p.KB + j) * atomB;
      uint8_t* bl = B_lo + (size_t)(k * p.KB + j) * atomB;
      for (int it = tid; it < p.Npad * 8; it += CV_THREADS) {
        const int n = it >> 3, qq = it & 7;
        const int c = n / Hout, o = n - c * Hout;
        float v[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int kb = j * ATOM_K + qq * 4 + i;
          const int l = kb < h ? Din + kb : (kb - h < Din ? kb - h : -1);
          v[i] = (n < p.Ntot && l >= 0) ? a.W[((size_t)(k * a.Kc + c) * L + l) * Hout + o] : 0.f;
        }
        store_split4(bh, bl, atom_chunk_offset(n, qq), make_float4(v[0], v[1], v[2], v[3]));
      }
    }
  fence_async_smem();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const int warp_u = uniform_warp_index();
  const uint32_t tmem_base = uniform_u32(*tmem_slot);
  const uint32_t idesc = make_idesc_tf32(128, p.Npad);
  const uint32_t d_small = tmem_base + (uint32_t)(p.nmain * p.Npad);
  const long long total_nodes = (long long)a.B * a.N;
  const long long R = total_nodes * C;
  // operand descriptors are launch constants: only the 16-byte-granular address field moves (K-step: +32 B, atom: +atomB)
  const uint64_t dA_hi = make_smem_desc_sw128(smem_u32(A_hi)), dA_lo = make_smem_desc_sw128(smem_u32(A_lo));
  const uint64_t dB_hi = make_smem_desc_sw128(smem_u32(B_hi)), dB_lo = make_smem_desc_sw128(smem_u32(B_lo));

  // build mapping: this thread always writes chunk column q of rows r0 + 32 i
  const int q = tid & 7, r0 = tid >> 3;
  uint32_t aoff[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) aoff[i] = atom_chunk_offset(r0 + 32 * i, q);
  // epilogue mapping: this thread owns accumulator row erow (and, general path, every second 8-column chunk)
  const int lane_base = (warp & 3) * 32, half = warp >> 2;
  const int erow = lane_base + lane;
  const int enode = erow / C, ecat = erow - enode * C;
  const uint32_t tl = tmem_base + ((uint32_t)lane_base << 16);

  uint32_t mma_phase = 0, load_phase = 0, epi_phase = 0;
  bool mma_pending = false;
  const bool tracing = a.trace != nullptr && blockIdx.x == 0 && tid == 0;
  int trace_it = 0;
  // one elected lane of warp 1 owns every bulk copy and prefetch; one elected lane of warp 0 only issues MMAs
  if (warp_u == 1 && elect_one_sync() && (int)blockIdx.x < p.ntiles) tc_issue_tile_loads(a, p, blockIdx.x, stage_h, stage_x, load_bar);

  for (int tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x) {
    const long long g0 = (long long)tile * p.npt;
    const int nodes_valid = (int)min((long long)p.npt, total_nodes - g0);
    const int rows_valid = nodes_valid * C;
    STC_TRACE(0);
    if (warp_u == 1 && elect_one_sync()) {  // the epilogue's own operands (H, and u for the candidate) travel under the builds and the MMAs
      const uint32_t eb = (uint32_t)(rows_valid * h * 4);
      mbar_arrive_expect_tx(epi_bar, a.phase == 0 ? eb : 2 * eb);
      bulk_g2s(stage_e, a.Hprev + g0 * C * h, eb, epi_bar);
      if (a.phase != 0) bulk_g2s(stage_e + 128 * h, a.u + g0 * C * h, eb, epi_bar);
      if ((a.opt & OPT_L2_PREFETCH) && tile + (int)gridDim.x < p.ntiles) tc_prefetch_tile(a, p, tile + gridDim.x);
    }
    mbar_wait(load_bar, load_phase);
    load_phase ^= 1u;
    if (!p.x_bulk) {  // unaligned x-part (e.g. Din = 1): plain loads, it is tiny
      for (int k = 0; k < a.Ks; ++k) {
        float* dst = stage_x + (size_t)k * 128 * Din;
        const int per_node = C * Din;
        for (int idx = tid; idx < nodes_valid * per_node; idx += CV_THREADS) {
          const int node = idx / per_node, rem = idx - node * per_node;
          const long long g = g0 + node;
          const float* src;
          if (k == 0) {
            const long long b = g / a.N;
            src = a.x0 + b * a.x0_bs + (g - b * a.N) * per_node;
          } else {
            src = a.yx + (long long)(k - 1) * R * Din + g * per_node;
          }
          dst[idx] = src[rem];
        }
      }
      __syncthreads();
    }
    STC_TRACE(1);
    bool acc_small = false;
    int ai = 0;
    for (int k = 0; k < a.Ks; ++k) {
      const float* sh = stage_h + (size_t)k * 128 * h;
      const float* sx = stage_x + (size_t)k * 128 * Din;
      for (int j = 0; j < p.KB; ++j, ++ai) {
        // the atom's values are read and split while the previous atom's MMAs may still be reading the single A buffer
        const int kb = j * ATOM_K + q * 4;
        const bool from_h = kb < h;
        float4 vv[4];
        if (from_h || (p.x_bulk && kb - h < Din)) {   // whole 16-byte chunks of the h-part or of an aligned x-part: one path
          const float* bp = from_h ? sh + kb : sx + (kb - h);
          const int st = from_h ? h : Din;
#pragma unroll
          for (int i = 0; i < 4; ++i) vv[i] = *reinterpret_cast<const float4*>(bp + (r0 + 32 * i) * st);
        } else {
          const int xi = kb - h;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            float e[4] = {0.f, 0.f, 0.f, 0.f};
            const float* sp = sx + (r0 + 32 * i) * Din + xi;
#pragma unroll
            for (int t = 0; t < 4; ++t)
              if (xi + t < Din) e[t] = sp[t];
            vv[i] = make_float4(e[0], e[1], e[2], e[3]);
          }
        }
        float4 vh[4], vl[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          split_tf32(vv[i].x, vh[i].x, vl[i].x); split_tf32(vv[i].y, vh[i].y, vl[i].y);
          split_tf32(vv[i].z, vh[i].z, vl[i].z); split_tf32(vv[i].w, vh[i].w, vl[i].w);
        }
        if (mma_pending) {
          mbar_wait(mma_bar, mma_phase);
          mma_phase ^= 1u;
          mma_pending = false;
          if (ai == p.nacc - 1) STC_TRACE(3);
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          *reinterpret_cast<float4*>(A_hi + aoff[i]) = vh[i];
          *reinterpret_cast<float4*>(A_lo + aoff[i]) = vl[i];
        }
        if (ai == 0) STC_TRACE(12);
        fence_async_smem();
        if (ai == 0) STC_TRACE(13);
        __syncthreads();
        if (ai == 0) STC_TRACE(2);
        // the stage is dead after the last build of this tile: fetch the next tile under the MMAs + epilogue
        if (warp_u == 1 && ai == p.nacc - 1 && tile + (int)gridDim.x < p.ntiles && elect_one_sync())
          tc_issue_tile_loads(a, p, tile + gridDim.x, stage_h, stage_x, load_bar);
        if (warp_u == 0 && elect_one_sync()) {   // one lane of converged warp 0: descriptors stay in uniform registers
          fence_after_sync();
          const int kleft = p.KBL - j * ATOM_K;
          const int ksteps = kleft >= ATOM_K ? 4 : (kleft + 7) / 8;
          const uint64_t bo = (uint64_t)(((uint32_t)ai * atomB) >> 4);
          const uint32_t d_main = tmem_base + (uint32_t)((ai / TC_APM) * p.Npad);
          uint32_t acc_main = (ai % TC_APM) != 0 ? 1u : 0u;
#pragma unroll 4
          for (int ks = 0; ks < ksteps; ++ks) {   // small cross terms into their own accumulator, then the main product
            const uint64_t ko = (uint64_t)(ks * 2);
            mma_tf32(d_small, dA_lo + ko, dB_hi + bo + ko, idesc, acc_small ? 1u : 0u);
            mma_tf32(d_small, dA_hi + ko, dB_lo + bo + ko, idesc, 1u);
            mma_tf32(d_main, dA_hi + ko, dB_hi + bo + ko, idesc, acc_main);
            acc_main = 1u;
            acc_small = true;
          }
          if (ai == 0) STC_TRACE(8);
          if (ai == p.nacc - 1) STC_TRACE(10);
          mma_commit(mma_bar);
          if (ai == 0) STC_TRACE(9);
          if (ai == p.nacc - 1) STC_TRACE(11);
        }
        acc_small = true;
        mma_pending = true;
      }
    }
    // ---- epilogue ----
    STC_TRACE(4);
    mbar_wait(mma_bar, mma_phase);   // a commit covers every MMA issued before it; the A atoms are free too
    mma_phase ^= 1u;
    mma_pending = false;
    fence_after_sync();
    STC_TRACE(5);
    mbar_wait(epi_bar, epi_phase);
    epi_phase ^= 1u;
    STC_TRACE(6);
    const bool valid = erow < rows_valid;
    const long long gr = g0 * C + erow;
    if constexpr (NG != 0) {
      tc_fwd_epilogue_fast<NG>(a, p, tl, Pm, Qs, bias_s, stage_e, erow, enode, ecat, half, valid, gr);
    } else {
      for (int c0 = half * 8; c0 < Hout; c0 += 16) {
        float v[8];
        tc_read_acc8(tl, p, c0, v);                                   // P_0
        for (int c = 1; c < a.Kc; ++c) {                              // + T_c(Gc)^T-mix of P_c over the node's categories
          float t[8];
          tc_read_acc8(tl, p, c * Hout + c0, t);
          __syncthreads();                                            // previous users of Pm are done
          *reinterpret_cast<float4*>(Pm + erow * p.PS + c0) = make_float4(t[0], t[1], t[2], t[3]);
          *reinterpret_cast<float4*>(Pm + erow * p.PS + c0 + 4) = make_float4(t[4], t[5], t[6], t[7]);
          if (a.Psave && valid) {  // backward forms dGc from these partials (no recomputation of the GEMM)
            float4* ps = reinterpret_cast<float4*>(a.Psave + gr * (long long)((a.Kc - 1) * Hout) + (c - 1) * Hout + c0);
            ps[0] = make_float4(t[0], t[1], t[2], t[3]);
            ps[1] = make_float4(t[4], t[5], t[6], t[7]);
          }
          __syncthreads();
          const float* Qc = Qs + (size_t)(c - 1) * C * C;
          const float* pp = Pm + (enode * C) * p.PS + c0;
          for (int cp = 0; cp < C; ++cp) {
            const float w = Qc[cp * C + ecat];
            const float4 x0 = *reinterpret_cast<const float4*>(pp + cp * p.PS);
            const float4 x1 = *reinterpret_cast<const float4*>(pp + cp * p.PS + 4);
            v[0] = fmaf(w, x0.x, v[0]); v[1] = fmaf(w, x0.y, v[1]); v[2] = fmaf(w, x0.z, v[2]); v[3] = fmaf(w, x0.w, v[3]);
            v[4] = fmaf(w, x1.x, v[4]); v[5] = fmaf(w, x1.y, v[5]); v[6] = fmaf(w, x1.z, v[6]); v[7] = fmaf(w, x1.w, v[7]);
          }
        }
        if (!valid) continue;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          float pre = v[i] + bias_s[c0 + i];
          if (a.act == STC_ACT_RELU) pre = fmaxf(pre, 0.f);
          v[i] = pre;
        }
        if (a.phase == 0) {
#pragma unroll
          for (int i = 0; i < 8; ++i) v[i] = sigmoidf_fast(v[i]);
          if (c0 < h) {
            float4* dst = reinterpret_cast<float4*>(a.u + gr * h + c0);
            dst[0] = make_float4(v[0], v[1], v[2], v[3]);
            dst[1] = make_float4(v[4], v[5], v[6], v[7]);
          } else {
            const long long o = gr * h + (c0 - h);
            const float4 h0 = *reinterpret_cast<const float4*>(stage_e + erow * h + (c0 - h));
            const float4 h1 = *reinterpret_cast<const float4*>(stage_e + erow * h + (c0 - h) + 4);
            if (a.r) {
              float4* dr = reinterpret_cast<float4*>(a.r + o);
              dr[0] = make_float4(v[0], v[1], v[2], v[3]);
              dr[1] = make_float4(v[4], v[5], v[6], v[7]);
            }
            float4* drh = reinterpret_cast<float4*>(a.rH + o);
            drh[0] = make_float4(v[0] * h0.x, v[1] * h0.y, v[2] * h0.z, v[3] * h0.w);
            drh[1] = make_float4(v[4] * h1.x, v[5] * h1.y, v[6] * h1.z, v[7] * h1.w);
          }
        } else {
          const long long o = gr * h + c0;
          float uu[8], hp[8], cc[8], hn[8];
          *reinterpret_cast<float4*>(uu) = *reinterpret_cast<const float4*>(stage_e + 128 * h + erow * h + c0);
          *reinterpret_cast<float4*>(uu + 4) = *reinterpret_cast<const float4*>(stage_e + 128 * h + erow * h + c0 + 4);
          *reinterpret_cast<float4*>(hp) = *reinterpret_cast<const float4*>(stage_e + erow * h + c0);
          *reinterpret_cast<float4*>(hp + 4) = *reinterpret_cast<const float4*>(stage_e + erow * h + c0 + 4);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            cc[i] = tanhf_fast(v[i]);
            hn[i] = fmaf(uu[i], cc[i] - hp[i], hp[i]);
          }
          if (a.c) {
            float4* dc = reinterpret_cast<float4*>(a.c + o);
            dc[0] = make_float4(cc[0], cc[1], cc[2], cc[3]);
            dc[1] = make_float4(cc[4], cc[5], cc[6], cc[7]);
          }
          float4* dh = reinterpret_cast<float4*>(a.Hnew + o);
          dh[0] = make_float4(hn[0], hn[1], hn[2], hn[3]);
          dh[1] = make_float4(hn[4], hn[5], hn[6], hn[7]);
        }
      }
    }
    STC_TRACE(7);
    ++trace_it;
    fence_before_sync();  // TMEM reads are ordered before the next tile's first (overwriting) MMA,
    fence_async_smem();   // the epilogue's reads of its staged operands precede the next tile's bulk copies into them,
    __syncthreads();      // and the exchange buffer is free before the next tile's A build
  }
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
}

// =================================================================================================
// A-in-TMEM forward kernel for the common shape (Ks = 2, Kc = 2, h = 16, Din <= 16; SF: N=100, C=5).
//
// Measured on the kernel above (profiles/r1k_phase_trace.txt): the tensor core's own operand fetch dominates the
// shared-memory traffic of a tile (every K-step re-reads A_hi twice and A_lo once: 12 KB for 2 KB of B), the single
// A buffer forces an MMA round trip in the middle of the tile, and each A build costs a proxy fence + block barrier.
// Here the data rows never touch shared memory: thread (row, half) loads the 32 K-values of spatial term k = half
// of its own row straight from global memory, splits them and writes hi / lo into TENSOR MEMORY columns of its
// accumulator lane (tcgen05.st); the MMAs take A from TMEM (tcgen05.mma with a TMEM A operand) and only the resident
// weight atoms from shared memory.  One block barrier per tile before the (24) MMAs, no mid-tile wait, no staging
// buffers.  TMEM columns: [0, Npad) main accumulator, [Npad, 2 Npad) cross terms, then A_hi (64) and A_lo (64).
template <int NG>
__device__ __forceinline__ void tc_fwd_epilogue_regs(const ConvArgs& a, const TcFwdPlan& p, uint32_t tl, float* Pm,
                                                     const float* Qs, const float* bias_s, const float4 (&hp)[2],
                                                     const float4 (&uu)[2], int erow, int enode, int ecat, int half,
                                                     bool valid, long long gr) {
  const int h = a.h, C = a.C, Hout = a.Hout;
  const int cb = half * 8;
  uint32_t sm1[NG][8], mn1[NG][8];
#pragma unroll
  for (int g = 0; g < NG; ++g) {                                          // P_1: cross terms, then main
    tmem_ld8_async(tl + (uint32_t)(p.Npad + Hout + 16 * g + cb), sm1[g]);
    tmem_ld8_async(tl + (uint32_t)(Hout + 16 * g + cb), mn1[g]);
  }
  tmem_ld_wait();
#pragma unroll
  for (int g = 0; g < NG; ++g) {
    tmem_ld_pin8(sm1[g]); tmem_ld_pin8(mn1[g]);
    float t[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) t[i] = __uint_as_float(sm1[g][i]) + __uint_as_float(mn1[g][i]);
    float* pm = Pm + erow * p.PS + 16 * g + cb;
    *reinterpret_cast<float4*>(pm) = make_float4(t[0], t[1], t[2], t[3]);
    *reinterpret_cast<float4*>(pm + 4) = make_float4(t[4], t[5], t[6], t[7]);
    if (a.Psave && valid) {   // backward forms dGc from these partials (no recomputation of the GEMM)
      float* ps = a.Psave + gr * (long long)Hout + 16 * g + cb;
      *reinterpret_cast<float4*>(ps) = make_float4(t[0], t[1], t[2], t[3]);
      *reinterpret_cast<float4*>(ps + 4) = make_float4(t[4], t[5], t[6], t[7]);
    }
  }
  uint32_t sm0[NG][8], mn0[NG][8];
#pragma unroll
  for (int g = 0; g < NG; ++g) {                                          // P_0 travels under the barrier
    tmem_ld8_async(tl + (uint32_t)(p.Npad + 16 * g + cb), sm0[g]);
    tmem_ld8_async(tl + (uint32_t)(16 * g + cb), mn0[g]);
  }
  __syncthreads();
  tmem_ld_wait();
  float v[NG][8];
#pragma unroll
  for (int g = 0; g < NG; ++g) {
    tmem_ld_pin8(sm0[g]); tmem_ld_pin8(mn0[g]);
#pragma unroll
    for (int i = 0; i < 8; ++i) v[g][i] = __uint_as_float(sm0[g][i]) + __uint_as_float(mn0[g][i]);
  }
  {
    const float* pp = Pm + (enode * C) * p.PS + cb;
#pragma unroll 5
    for (int cp = 0; cp < C; ++cp) {
      const float w = Qs[cp * C + ecat];
#pragma unroll
      for (int g = 0; g < NG; ++g) {
        const float4 x0 = *reinterpret_cast<const float4*>(pp + cp * p.PS + 16 * g);
        const float4 x1 = *reinterpret_cast<const float4*>(pp + cp * p.PS + 16 * g + 4);
        v[g][0] = fmaf(w, x0.x, v[g][0]); v[g][1] = fmaf(w, x0.y, v[g][1]);
        v[g][2] = fmaf(w, x0.z, v[g][2]); v[g][3] = fmaf(w, x0.w, v[g][3]);
        v[g][4] = fmaf(w, x1.x, v[g][4]); v[g][5] = fmaf(w, x1.y, v[g][5]);
        v[g][6] = fmaf(w, x1.z, v[g][6]); v[g][7] = fmaf(w, x1.w, v[g][7]);
      }
    }
  }
  if (!valid) return;
#pragma unroll
  for (int g = 0; g < NG; ++g) {
    const float4 b0 = *reinterpret_cast<const float4*>(bias_s + 16 * g + cb);
    const float4 b1 = *reinterpret_cast<const float4*>(bias_s + 16 * g + cb + 4);
    v[g][0] += b0.x; v[g][1] += b0.y; v[g][2] += b0.z; v[g][3] += b0.w;
    v[g][4] += b1.x; v[g][5] += b1.y; v[g][6] += b1.z; v[g][7] += b1.w;
    if (a.act == STC_ACT_RELU) {
#pragma unroll
      for (int i = 0; i < 8; ++i) v[g][i] = fmaxf(v[g][i], 0.f);
    }
  }
  const float hpv[8] = {hp[0].x, hp[0].y, hp[0].z, hp[0].w, hp[1].x, hp[1].y, hp[1].z, hp[1].w};
  if (a.phase == 0) {   // h = 16, Hout = 32: group 0 = u channels cb.., group 1 = r channels cb..
#pragma unroll
    for (int g = 0; g < NG; ++g) {
#pragma unroll
      for (int i = 0; i < 8; ++i) v[g][i] = sigmoidf_fast(v[g][i]);
      const int col = 16 * g + cb;
      if (col < h) {
        float* dst = a.u + gr * h + col;
        *reinterpret_cast<float4*>(dst) = make_float4(v[g][0], v[g][1], v[g][2], v[g][3]);
        *reinterpret_cast<float4*>(dst + 4) = make_float4(v[g][4], v[g][5], v[g][6], v[g][7]);
      } else {
        const int ch = col - h;   // == cb
        if (a.r) {
          float* dr = a.r + gr * h + ch;
          *reinterpret_cast<float4*>(dr) = make_float4(v[g][0], v[g][1], v[g][2], v[g][3]);
          *reinterpret_cast<float4*>(dr + 4) = make_float4(v[g][4], v[g][5], v[g][6], v[g][7]);
        }
        float* drh = a.rH + gr * h + ch;
        *reinterpret_cast<float4*>(drh) = make_float4(v[g][0] * hpv[0], v[g][1] * hpv[1], v[g][2] * hpv[2], v[g][3] * hpv[3]);
        *reinterpret_cast<float4*>(drh + 4) = make_float4(v[g][4] * hpv[4], v[g][5] * hpv[5], v[g][6] * hpv[6], v[g][7] * hpv[7]);
      }
    }
  } else {              // Hout = h = 16: one group, channels cb..: c = tanh, H' = H + u (c - H)
    const float uuv[8] = {uu[0].x, uu[0].y, uu[0].z, uu[0].w, uu[1].x, uu[1].y, uu[1].z, uu[1].w};
    const long long o = gr * h + cb;
    float cc[8], hn[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      cc[i] = tanhf_fast(v[0][i]);
      hn[i] = fmaf(uuv[i], cc[i] - hpv[i], hpv[i]);
    }
    if (a.c) {
      *reinterpret_cast<float4*>(a.c + o) = make_float4(cc[0], cc[1], cc[2], cc[3]);
      *reinterpret_cast<float4*>(a.c + o + 4) = make_float4(cc[4], cc[5], cc[6], cc[7]);
    }
    *reinterpret_cast<float4*>(a.Hnew + o) = make_float4(hn[0], hn[1], hn[2], hn[3]);
    *reinterpret_cast<float4*>(a.Hnew + o + 4) = make_float4(hn[4], hn[5], hn[6], hn[7]);
  }
}

template <int NG>
__global__ void __launch_bounds__(CV_THREADS, 2)
tc_conv_fwd_at_kernel(const ConvArgs a, const TcFwdPlan p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((smem_u32(smem) & 1023u) != 0u) __trap();
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int C = a.C, L = a.Din + a.h, Din = a.Din, Hout = a.Hout;
  constexpr int h = 16;
  const uint32_t atomB = (uint32_t)p.Npad * ATOM_ROW_BYTES;
  float* Pm = reinterpret_cast<float*>(smem + p.off_a);          // [128][PS] exchange buffer of the categorical mix
  // resident weight atoms, per spatial term [hi (Npad rows) | lo (Npad rows)]: one descriptor over both is the
  // N = 2 Npad operand [W_hi ; W_lo], so A_hi x [W_hi ; W_lo] fills the main AND the cross-term accumulator in one MMA
  uint8_t* B_hi = smem + p.off_b;
  uint8_t* B_lo = B_hi + atomB;
  float* Qs = reinterpret_cast<float*>(smem + p.off_q);
  float* bias_s = reinterpret_cast<float*>(smem + p.off_bias);
  uint64_t* mma_bar = reinterpret_cast<uint64_t*>(smem + p.off_bar);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(mma_bar + 1);

  if (tid == 0) {
    mbar_init(mma_bar, 1);
    mbar_fence_init();
  }
  if (warp == 0) tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols);
  for (int i = tid; i < C * C; i += CV_THREADS) Qs[i] = a.Q[C * C + i];
  for (int i = tid; i < Hout; i += CV_THREADS) bias_s[i] = a.bias ? a.bias[i] : 0.f;
  for (int k = 0; k < 2; ++k) {   // Bt[(c,o)][kb] = W[((k*Kc + c)*L + l(kb))*Hout + o], K order [h-part | x-part | zero pad]
    uint8_t* bh = B_hi + (size_t)k * 2 * atomB;
    uint8_t* bl = B_lo + (size_t)k * 2 * atomB;
    for (int it = tid; it < p.Npad * 8; it += CV_THREADS) {
      const int n = it >> 3, qq = it & 7;
      const int c = n / Hout, o = n - c * Hout;
      float v[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int kb = qq * 4 + i;
        const int l = kb < h ? Din + kb : (kb - h < Din ? kb - h : -1);
        v[i] = (n < p.Ntot && l >= 0) ? a.W[((size_t)(k * 2 + c) * L + l) * Hout + o] : 0.f;
      }
      store_split4(bh, bl, atom_chunk_offset(n, qq), make_float4(v[0], v[1], v[2], v[3]));
    }
  }
  fence_async_smem();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const int warp_u = uniform_warp_index();
  const uint32_t tmem_base = uniform_u32(*tmem_slot);
  const uint32_t idesc = make_idesc_tf32(128, p.Npad), idesc2 = make_idesc_tf32(128, 2 * p.Npad);
  const uint32_t d_main = tmem_base, d_small = tmem_base + (uint32_t)p.Npad;
  const uint32_t colA = (uint32_t)(2 * p.Npad);              // A_hi columns [colA, colA+64), A_lo [colA+64, colA+128)
  const uint64_t dB_hi = make_smem_desc_sw128(smem_u32(B_hi));
  const int ksteps = p.KBL >> 3;                             // 3 (Din <= 8) or 4 K-steps per spatial term
  const long long total_nodes = (long long)a.B * a.N;
  const long long R = total_nodes * C;

  const int sp = warp & 3, half = warp >> 2;
  const int erow = sp * 32 + lane;                           // accumulator lane = tile row
  const int enode = erow / C, ecat = erow - enode * C;
  const uint32_t tl = tmem_base + ((uint32_t)(sp * 32) << 16);
  const uint32_t tA = tl + colA + (uint32_t)(half * 32);     // this thread writes term k = half of its row
  const bool xvec = p.x_bulk != 0;
  uint32_t mma_phase = 0;
  const bool tracing = a.trace != nullptr && blockIdx.x == 0 && tid == 0;
  int trace_it = 0;
  // (a cp.async prefetch of the rows one tile ahead was measured: the load phase shrinks but the tile time does not --
  //  the two resident CTAs already cover each other's load latency)
  for (int tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x) {
    const long long g0 = (long long)tile * p.npt;
    const int nodes_valid = (int)min((long long)p.npt, total_nodes - g0);
    const int rows_valid = nodes_valid * C;
    const bool valid = erow < rows_valid;
    const long long gr = g0 * C + erow;
    STC_TRACE(0);
    if ((a.opt & OPT_L2_PREFETCH) && warp_u == 1 && tile + (int)gridDim.x < p.ntiles && elect_one_sync())
      tc_prefetch_tile(a, p, tile + gridDim.x);
    // ---- my row's K-values of spatial term k = half: [h-part (16) | x-part (Din) | zeros] ----
    float4 xv[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) xv[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (valid) {
      const float* hs = (half == 0 ? a.h0 : a.yh) + gr * h;
#pragma unroll
      for (int i = 0; i < 4; ++i) xv[i] = *reinterpret_cast<const float4*>(hs + 4 * i);
      const float* xs;
      if (half == 0) {
        const long long g = g0 + enode;
        const long long b = g / a.N;
        xs = a.x0 + b * a.x0_bs + ((g - b * a.N) * C + ecat) * Din;
      } else {
        xs = a.yx + gr * Din;
      }
      if (xvec) {
#pragma unroll
        for (int i = 0; i < 4; ++i)
          if (4 * i < Din) xv[4 + i] = *reinterpret_cast<const float4*>(xs + 4 * i);
      } else {
        float e[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) e[i] = i < Din ? xs[i] : 0.f;
#pragma unroll
        for (int i = 0; i < 4; ++i) xv[4 + i] = make_float4(e[4 * i], e[4 * i + 1], e[4 * i + 2], e[4 * i + 3]);
      }
    }
    STC_TRACE(1);
#pragma unroll
    for (int i = 0; i < 4; ++i) {   // 8 columns at a time: hi into A_hi, lo into A_lo
      float hi[8], lo[8];
      split_tf32(xv[2 * i].x, hi[0], lo[0]); split_tf32(xv[2 * i].y, hi[1], lo[1]);
      split_tf32(xv[2 * i].z, hi[2], lo[2]); split_tf32(xv[2 * i].w, hi[3], lo[3]);
      split_tf32(xv[2 * i + 1].x, hi[4], lo[4]); split_tf32(xv[2 * i + 1].y, hi[5], lo[5]);
      split_tf32(xv[2 * i + 1].z, hi[6], lo[6]); split_tf32(xv[2 * i + 1].w, hi[7], lo[7]);
      tmem_st8(tA + (uint32_t)(8 * i), hi);
      tmem_st8(tA + 64u + (uint32_t)(8 * i), lo);
    }
    tmem_st_wait();
    STC_TRACE(12);
    fence_before_sync();
    STC_TRACE(13);
    __syncthreads();
    STC_TRACE(2);
    STC_TRACE(3);
    if (warp_u == 0 && elect_one_sync()) {
      fence_after_sync();
      uint32_t acc = 0u;
#pragma unroll
      for (int ai = 0; ai < 2; ++ai) {
        const uint64_t bo = (uint64_t)(((uint32_t)ai * 2u * atomB) >> 4);
        for (int ks = 0; ks < ksteps; ++ks) {
          const uint64_t ko = (uint64_t)(ks * 2);
          const uint32_t ah = tmem_base + colA + (uint32_t)(ai * 32 + ks * 8), al = ah + 64u;
          mma_tf32_atmem(d_main, ah, dB_hi + bo + ko, idesc2, acc);    // [main | cross] (+)= A_hi x [W_hi ; W_lo]
          mma_tf32_atmem(d_small, al, dB_hi + bo + ko, idesc, 1u);     // cross += A_lo x W_hi
          acc = 1u;
        }
      }
      STC_TRACE(8);
      STC_TRACE(10);
      mma_commit(mma_bar);
      STC_TRACE(9);
      STC_TRACE(11);
    }
    // ---- the epilogue's own operands travel under the MMAs: H (and u for the candidate), 8 channels of my row ----
    float4 hp[2], uu[2];
    hp[0] = hp[1] = uu[0] = uu[1] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (valid) {
      const float* hsrc = a.Hprev + gr * h + half * 8;
      hp[0] = *reinterpret_cast<const float4*>(hsrc);
      hp[1] = *reinterpret_cast<const float4*>(hsrc + 4);
      if (a.phase != 0) {
        const float* usrc = a.u + gr * h + half * 8;
        uu[0] = *reinterpret_cast<const float4*>(usrc);
        uu[1] = *reinterpret_cast<const float4*>(usrc + 4);
      }
    }
    STC_TRACE(4);
    mbar_wait(mma_bar, mma_phase);
    mma_phase ^= 1u;
    fence_after_sync();
    STC_TRACE(5);
    STC_TRACE(6);
    tc_fwd_epilogue_regs<NG>(a, p, tl, Pm, Qs, bias_s, hp, uu, erow, enode, ecat, half, valid, gr);
    STC_TRACE(7);
    ++trace_it;
    fence_before_sync();   // TMEM reads precede the next tile's TMEM stores and MMAs; Pm is free for the next exchange
    __syncthreads();
  }
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
}

static bool tc_disabled() {
  static int cached = -1;
  if (cached < 0) {
    const char* e = getenv("STC_DISABLE_TC");
    cached = (e && e[0] && e[0] != '0') ? 1 : 0;
  }
  return cached == 1;
}

static bool aligned16p(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// Shape-only eligibility of the tcgen05 path; forward and backward must agree (backward reads what forward saved).
bool conv_tc_eligible(const ConvArgs& a) {
  if (tc_disabled()) return false;
  if (a.h % 8 != 0 || a.Hout % 16 != 0 || a.C > 128) return false;
  const int Dp = (a.Din + 7) & ~7, KBL = a.h + Dp, KB = (KBL + ATOM_K - 1) / ATOM_K;
  // forward: N = Kc*Hout, accumulators = Ks*KB mains + 1
  const int Nf = (a.Kc * a.Hout + 15) & ~15;
  if (Nf > 256 || (a.Ks * KB + 1) * Nf > 512) return false;
  if ((size_t)128 * (a.Hout + 4) * sizeof(float) > 2 * 128 * ATOM_ROW_BYTES) return false;
  const size_t fwd_smem = 2 * 128 * ATOM_ROW_BYTES + 2 * (size_t)a.Ks * KB * Nf * ATOM_ROW_BYTES +
                          (size_t)a.Ks * 128 * (a.h + a.Din) * sizeof(float) + (size_t)2 * 128 * a.h * sizeof(float) +
                          (size_t)a.Kc * a.C * a.C * sizeof(float) + 64;
  if (fwd_smem > 200 * 1024) return false;
  // backward dx: N = Ks*KBL, K = Kc*Hout
  const int Nb = (a.Ks * KBL + 15) & ~15, KA = (a.Kc * a.Hout + ATOM_K - 1) / ATOM_K;
  if (Nb > 256 || (KA + 1) * Nb > 512) return false;
  const size_t dx_smem = 2 * 128 * ATOM_ROW_BYTES + 2 * (size_t)KA * Nb * ATOM_ROW_BYTES +
                         (size_t)128 * (a.Hout + 4 + a.h + (a.Kc - 1) * a.Hout) * sizeof(float) +
                         (size_t)2 * a.Kc * a.C * a.C * sizeof(float) + 256;
  if (dx_smem > 200 * 1024) return false;
  return true;
}

int try_launch_conv_fwd_tc(const ConvArgs& a, cudaStream_t st, bool* handled) {
  *handled = false;
  if (!conv_tc_eligible(a)) return STC_OK;
  const int L = a.Din + a.h, P = a.Ks * a.Kc;
  if (!aligned16p(a.u) || !aligned16p(a.Hprev) || !aligned16p(a.r) || !aligned16p(a.rH) || !aligned16p(a.c) ||
      !aligned16p(a.Hnew) || !aligned16p(a.h0) || !aligned16p(a.yh) || !aligned16p(a.Psave)) {
    set_error("tcgen05 path needs 16-byte aligned state / workspace tensors");
    return STC_ERR_BAD_ARG;
  }
  // an eligible shape must run here: backward (dpre layout, Psave) is planned from conv_tc_eligible alone, so a silent
  // decline would make the tensor-core backward read a Psave the FFMA forward never wrote
  auto declined = [&](const char* why) {
    set_error("tcgen05 forward declined an eligible shape (%s): N=%d C=%d Din=%d h=%d Ks=%d Kc=%d Hout=%d", why, a.N, a.C,
              a.Din, a.h, a.Ks, a.Kc, a.Hout);
    return STC_ERR_UNSUPPORTED;
  };
  TcFwdPlan p;
  p.npt = 128 / a.C;
  p.Dp = (a.Din + 7) & ~7;
  p.KBL = a.h + p.Dp;
  p.KB = (p.KBL + ATOM_K - 1) / ATOM_K;
  p.Ntot = a.Kc * a.Hout;
  p.Npad = (p.Ntot + 15) & ~15;
  if (p.Npad > 256) return declined("N tile");
  p.nacc = a.Ks * p.KB;
  p.nmain = (p.nacc + TC_APM - 1) / TC_APM;
  p.tmem_cols = 32;
  while (p.tmem_cols < (p.nmain + 1) * p.Npad) p.tmem_cols *= 2;
  if (p.tmem_cols > 512) return declined("tensor memory columns");
  p.PS = a.Hout + 4;
  if ((size_t)128 * p.PS * sizeof(float) > 2 * 128 * ATOM_ROW_BYTES) return declined("exchange buffer");  // aliases A
  p.x_bulk = (a.Din % 4 == 0) && (a.x0_bs % 4 == 0) && aligned16p(a.x0) && aligned16p(a.yx);
  const long long total_nodes = (long long)a.B * a.N;
  p.ntiles = ceil_div(total_nodes, p.npt);
  const size_t atomB = (size_t)p.Npad * ATOM_ROW_BYTES;
  size_t o = 0;
  p.off_a = (uint32_t)o; o += 2 * 128 * ATOM_ROW_BYTES;                 // A hi + lo (one atom)
  p.off_b = (uint32_t)o; o += 2 * (size_t)p.nacc * atomB;               // resident W atoms hi/lo
  p.off_sh = (uint32_t)o; o += (size_t)a.Ks * 128 * a.h * sizeof(float);
  p.off_sx = (uint32_t)o; o += round_up((size_t)a.Ks * 128 * a.Din * sizeof(float), 16);
  p.off_se = (uint32_t)o; o += (size_t)2 * 128 * a.h * sizeof(float);
  p.off_q = (uint32_t)o; o += (size_t)(a.Kc > 1 ? a.Kc - 1 : 0) * a.C * a.C * sizeof(float);
  o = round_up(o, 16);
  p.off_bias = (uint32_t)o; o += (size_t)a.Hout * sizeof(float);
  o = round_up(o, 16);
  p.off_bar = (uint32_t)o; o += 48;
  p.smem_bytes = (uint32_t)o;
  const bool smem_over = p.smem_bytes > 200 * 1024;   // checked after the A-in-TMEM layout below (it needs less)
  // batched epilogue: Kc = 2, one main accumulator, one or two 8-column groups per thread (Hout = 16 or 32)
  int ng = 0;
  if (a.Kc == 2 && p.nmain == 1 && (a.Hout == 16 || a.Hout == 32) && !(a.opt & OPT_GENERIC_EPILOGUE)) ng = a.Hout / 16;
  auto kern = ng == 2 ? tc_conv_fwd_kernel<2> : (ng == 1 ? tc_conv_fwd_kernel<1> : tc_conv_fwd_kernel<0>);
  // A-in-TMEM variant: additionally Ks = 2, h = 16, one atom per spatial term (Din <= 16)
  const bool at = ng != 0 && a.Ks == 2 && a.h == 16 && p.KB == 1 && !(a.opt & OPT_SMEM_A);
  if (at) {
    kern = ng == 2 ? tc_conv_fwd_at_kernel<2> : tc_conv_fwd_at_kernel<1>;
    size_t q = 0;
    p.off_a = (uint32_t)q; q += round_up((size_t)128 * p.PS * sizeof(float), 1024);   // exchange buffer
    p.off_b = (uint32_t)q; q += 2 * (size_t)2 * atomB;                               // resident W atoms hi/lo
    p.off_q = (uint32_t)q; q += round_up((size_t)a.C * a.C * sizeof(float), 16);
    p.off_bias = (uint32_t)q; q += round_up((size_t)a.Hout * sizeof(float), 16);
    p.off_bar = (uint32_t)q; q += 32;
    p.smem_bytes = (uint32_t)q;
    p.tmem_cols = 256;   // 2 Npad accumulator columns + 128 A columns
  }
  if (!at && smem_over) return declined("shared memory");
  STC_TRY(set_smem(kern, p.smem_bytes));
  int ctas_per_sm = (int)((228 * 1024) / (p.smem_bytes + 1024));
  if (ctas_per_sm < 1) ctas_per_sm = 1;
  if (ctas_per_sm > 2) ctas_per_sm = 2;
  if (ctas_per_sm * p.tmem_cols > 512) ctas_per_sm = 512 / p.tmem_cols;
  int grid = device_sm_count() * ctas_per_sm;
  if (grid > p.ntiles) grid = p.ntiles;
  const double R = (double)total_nodes * a.C;
  ScopedKernelTimer _t(KK_TC_CONV_FWD, st, 4.0 * R * (a.Ks * L + conv_fwd_state_floats(a)) + 4.0 * P * L * a.Hout);
  kern<<<grid, CV_THREADS, p.smem_bytes, st>>>(a, p);
  STC_LAUNCH_OK("tc_conv_fwd_kernel");
  *handled = true;
  return STC_OK;
}

// =================================================================================================
// self-test / microbenchmark of the building block:  D[M][N] = A[M][K] * Bm[K][N]  (3xTF32)
//   mode bit 0: truncating split instead of round-to-nearest (experiment)
//   nmain: number of main (hi*hi) accumulators used round-robin over K atoms; small != 0: the cross terms
//   get their own accumulator.  All accumulators are summed in fp32 round-to-nearest in the epilogue.
// =================================================================================================
__global__ void __launch_bounds__(CV_THREADS, 1)
tf32x3_gemm_kernel(const float* __restrict__ A, const float* __restrict__ Bm, float* __restrict__ D, int M, int N,
                   int K, int Npad, int tmem_cols, int mode, int nmain, int small) {
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((smem_u32(smem) & 1023u) != 0u) __trap();
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t atomA = 128 * ATOM_ROW_BYTES, atomB = (uint32_t)Npad * ATOM_ROW_BYTES;
  uint8_t* A_hi = smem;
  uint8_t* A_lo = A_hi + atomA;
  uint8_t* B_hi = A_lo + atomA;
  uint8_t* B_lo = B_hi + atomB;
  uint64_t* bar = reinterpret_cast<uint64_t*>(B_lo + atomB);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + 1);
  if (tid == 0) {
    mbar_init(bar, 1);
    mbar_fence_init();
  }
  if (warp == 0) tmem_alloc(tmem_slot, (uint32_t)tmem_cols);
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t idesc = make_idesc_tf32(128, Npad);
  const int m0 = blockIdx.x * 128;
  uint32_t phase = 0;
  bool acc_main[16], acc_small = false;
  for (int i = 0; i < 16; ++i) acc_main[i] = false;
  const int natoms = (K + ATOM_K - 1) / ATOM_K;
  for (int j = 0; j < natoms; ++j) {
    if (j > 0) {
      mbar_wait(bar, phase);
      phase ^= 1u;
    }
    for (int it = tid; it < 128 * 8; it += CV_THREADS) {
      const int row = it >> 3, q = it & 7;
      float v[4], hi[4], lo[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int k = j * ATOM_K + q * 4 + i;
        v[i] = (m0 + row < M && k < K) ? A[(size_t)(m0 + row) * K + k] : 0.f;
        if (mode & 1) split_tf32_trunc(v[i], hi[i], lo[i]); else split_tf32(v[i], hi[i], lo[i]);
      }
      const uint32_t off = atom_chunk_offset(row, q);
      *reinterpret_cast<float4*>(A_hi + off) = make_float4(hi[0], hi[1], hi[2], hi[3]);
      *reinterpret_cast<float4*>(A_lo + off) = make_float4(lo[0], lo[1], lo[2], lo[3]);
    }
    for (int it = tid; it < Npad * 8; it += CV_THREADS) {
      const int n = it >> 3, q = it & 7;
      float v[4], hi[4], lo[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int k = j * ATOM_K + q * 4 + i;
        v[i] = (n < N && k < K) ? Bm[(size_t)k * N + n] : 0.f;
        if (mode & 1) split_tf32_trunc(v[i], hi[i], lo[i]); else split_tf32(v[i], hi[i], lo[i]);
      }
      const uint32_t off = atom_chunk_offset(n, q);
      *reinterpret_cast<float4*>(B_hi + off) = make_float4(hi[0], hi[1], hi[2], hi[3]);
      *reinterpret_cast<float4*>(B_lo + off) = make_float4(lo[0], lo[1], lo[2], lo[3]);
    }
    fence_async_smem();
    __syncthreads();
    if (tid == 0) {
      fence_after_sync();
      const int kleft = K - j * ATOM_K;
      const int ksteps = kleft >= ATOM_K ? 4 : (kleft + 7) / 8;
      const int mi = j % nmain;
      const uint32_t d_main = tmem_base + (uint32_t)(mi * Npad);
      if (small) {
        const uint32_t d_small = tmem_base + (uint32_t)(nmain * Npad);
        mma_atom_3x_split(d_main, d_small, smem_u32(A_hi), smem_u32(A_lo), smem_u32(B_hi), smem_u32(B_lo), ksteps, idesc,
                          acc_main[mi], acc_small);
      } else {
        mma_atom_3x(d_main, smem_u32(A_hi), smem_u32(A_lo), smem_u32(B_hi), smem_u32(B_lo), ksteps, idesc, acc_main[mi]);
      }
      mma_commit(bar);
    }
  }
  mbar_wait(bar, phase);
  fence_after_sync();
  {
    const int lane_base = (warp & 3) * 32, half = warp >> 2;
    const int row = m0 + lane_base + lane;
    const int nchunks = Npad / 8;
    const int nbuf = (natoms < nmain ? natoms : nmain);
    for (int ch = half; ch < nchunks; ch += 2) {
      float acc[8], v[8];
      if (small) {
        tmem_ld8(tmem_base + ((uint32_t)lane_base << 16) + (uint32_t)(nmain * Npad + ch * 8), acc);
      } else {
        for (int i = 0; i < 8; ++i) acc[i] = 0.f;
      }
      for (int b = 0; b < nbuf; ++b) {
        tmem_ld8(tmem_base + ((uint32_t)lane_base << 16) + (uint32_t)(b * Npad + ch * 8), v);
        for (int i = 0; i < 8; ++i) acc[i] += v[i];
      }
      if (row < M)
        for (int i = 0; i < 8; ++i)
          if (ch * 8 + i < N) D[(size_t)row * N + ch * 8 + i] = acc[i];
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, (uint32_t)tmem_cols);
}

// MN-major variant of the self-test (STC_TC_TEST_MODE bit 1): the same product with both operand tiles stored
// [K rows][M or N contiguous] -- the layout the dW kernel uses to contract over tile rows without transposing.
//   variant 0: SWIZZLE_128B_BASE32B, LBO = column-block pitch, SBO = 4-row group pitch (production layout)
//   variant 1: the same with LBO / SBO exchanged (diagnostic)
//   variant 2: no swizzle ("interleave"): 8 x 16-byte core matrices, SBO = pitch between 4-element M/N blocks,
//              LBO = pitch between 8-row K groups (diagnostic fallback)
struct MnLayout {
  int variant;
  uint32_t colblk;   // bytes of one 32-wide column block (variants 0/1)
  uint32_t kgroup;   // bytes between 8-row K groups (variant 2)
  __device__ __forceinline__ uint32_t off(int k, int ch) const {  // ch = 16-byte chunk index along M/N
    if (variant == 2) return (uint32_t)(k >> 3) * kgroup + (uint32_t)ch * 128u + (uint32_t)(k & 7) * 16u;
    return (uint32_t)(ch >> 3) * colblk + mn32_chunk_offset(k, ch & 7);
  }
  __device__ __forceinline__ uint64_t desc(uint32_t base, int ks) const {  // K-step ks (8 rows)
    if (variant == 2) {
      uint64_t d = 0;
      d |= (uint64_t)(((base + ks * kgroup) >> 4) & 0x3FFF);
      d |= (uint64_t)((kgroup >> 4) & 0x3FFF) << 16;   // LBO
      d |= (uint64_t)((128u >> 4) & 0x3FFF) << 32;     // SBO
      d |= (uint64_t)1 << 46;
      return d;
    }
    const uint32_t a = base + ks * 2 * MN32_GROUP_BYTES;
    return variant == 0 ? make_smem_desc_mn32(a, colblk, MN32_GROUP_BYTES) : make_smem_desc_mn32(a, MN32_GROUP_BYTES, colblk);
  }
};

__global__ void __launch_bounds__(CV_THREADS, 1)
tf32x3_gemm_mn_kernel(const float* __restrict__ A, const float* __restrict__ Bm, float* __restrict__ D, int M, int N,
                      int K, int Npad, int tmem_cols, int variant) {
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((smem_u32(smem) & 1023u) != 0u) __trap();
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int ncolB = (Npad + 31) / 32;                  // 32-wide column blocks of B
  const uint32_t colblk = 32 * ATOM_ROW_BYTES;         // [32 K-rows][128 B] = 4 KB
  const MnLayout la{variant, colblk, 32u * 128u};      // A: 128 M = 32 chunks per K row
  const MnLayout lb{variant, colblk, (uint32_t)(ncolB * 8) * 128u};
  uint8_t* A_hi = smem;                                // 4 column blocks (M = 128)
  uint8_t* A_lo = A_hi + 4 * colblk;
  uint8_t* B_hi = A_lo + 4 * colblk;
  uint8_t* B_lo = B_hi + ncolB * colblk;
  uint64_t* bar = reinterpret_cast<uint64_t*>(B_lo + ncolB * colblk);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + 1);
  if (tid == 0) {
    mbar_init(bar, 1);
    mbar_fence_init();
  }
  if (warp == 0) tmem_alloc(tmem_slot, (uint32_t)tmem_cols);
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t idesc = make_idesc_tf32_mn(128, Npad);
  const int m0 = blockIdx.x * 128;
  uint32_t phase = 0;
  const int nchunksK = (K + 31) / 32;
  bool acc_main = false, acc_small = false;
  for (int j = 0; j < nchunksK; ++j) {
    if (j > 0) {
      mbar_wait(bar, phase);
      phase ^= 1u;
    }
    for (int it = tid; it < 32 * 32; it += CV_THREADS) {    // 32 k-rows x 32 chunks (128 m / 4)
      const int k = it >> 5, ch = it & 31;
      float v[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int m = ch * 4 + i, kk = j * 32 + k;
        v[i] = (m0 + m < M && kk < K) ? A[(size_t)(m0 + m) * K + kk] : 0.f;
      }
      store_split4(A_hi, A_lo, la.off(k, ch), make_float4(v[0], v[1], v[2], v[3]));
    }
    for (int it = tid; it < 32 * ncolB * 8; it += CV_THREADS) {
      const int k = it / (ncolB * 8), ch = it - k * (ncolB * 8);
      float v[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int n = ch * 4 + i, kk = j * 32 + k;
        v[i] = (n < N && kk < K) ? Bm[(size_t)kk * N + n] : 0.f;
      }
      store_split4(B_hi, B_lo, lb.off(k, ch), make_float4(v[0], v[1], v[2], v[3]));
    }
    fence_async_smem();
    __syncthreads();
    if (tid == 0) {
      fence_after_sync();
      const int kleft = K - j * 32;
      const int ksteps = kleft >= 32 ? 4 : (kleft + 7) / 8;
      for (int ks = 0; ks < ksteps; ++ks) {
        const uint64_t ah = la.desc(smem_u32(A_hi), ks), al = la.desc(smem_u32(A_lo), ks);
        const uint64_t bh = lb.desc(smem_u32(B_hi), ks), bl = lb.desc(smem_u32(B_lo), ks);
        mma_tf32(tmem_base + (uint32_t)Npad, al, bh, idesc, acc_small ? 1u : 0u);
        mma_tf32(tmem_base + (uint32_t)Npad, ah, bl, idesc, 1u);
        mma_tf32(tmem_base, ah, bh, idesc, acc_main ? 1u : 0u);
        acc_main = acc_small = true;
      }
      mma_commit(bar);
    }
  }
  mbar_wait(bar, phase);
  fence_after_sync();
  {
    const int lane_base = (warp & 3) * 32, half = warp >> 2;
    const int row = m0 + lane_base + lane;
    for (int ch = half; ch < Npad / 8; ch += 2) {
      float v[8], t[8];
      tmem_ld8(tmem_base + ((uint32_t)lane_base << 16) + (uint32_t)(Npad + ch * 8), v);
      tmem_ld8(tmem_base + ((uint32_t)lane_base << 16) + (uint32_t)(ch * 8), t);
      if (row < M)
        for (int i = 0; i < 8; ++i)
          if (ch * 8 + i < N) D[(size_t)row * N + ch * 8 + i] = v[i] + t[i];
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, (uint32_t)tmem_cols);
}

int launch_tf32x3_gemm(const float* A, const float* Bm, float* D, int M, int N, int K, cudaStream_t st) {
  if (M <= 0 || N <= 0 || K <= 0 || N > 256) {
    set_error("tf32x3 gemm self-test: need M,K > 0 and 0 < N <= 256");
    return STC_ERR_BAD_ARG;
  }
  // experiment knobs (defaults = what the production kernels use)
  int mode = 0, nmain = 1, small = 0;
  if (const char* e = getenv("STC_TC_TEST_MODE")) mode = atoi(e);
  if (const char* e = getenv("STC_TC_TEST_NMAIN")) nmain = atoi(e);
  if (const char* e = getenv("STC_TC_TEST_SMALL")) small = atoi(e);
  const int Npad = (N + 15) & ~15;
  if (mode & 2) {
    int cols = 32;
    while (cols < 2 * Npad) cols *= 2;
    const size_t smem_mn = (size_t)(8 + 2 * ((Npad + 31) / 32)) * 32 * ATOM_ROW_BYTES + 64;
    STC_TRY(set_smem(tf32x3_gemm_mn_kernel, smem_mn));
    ScopedKernelTimer _t(KK_TC_GEMM_TEST, st, 4.0 * ((double)M * K + (double)K * N + (double)M * N));
    int variant = 0;
    if (const char* e = getenv("STC_TC_MN_VARIANT")) variant = atoi(e);
    tf32x3_gemm_mn_kernel<<<ceil_div(M, 128), CV_THREADS, smem_mn, st>>>(A, Bm, D, M, N, K, Npad, cols, variant);
    STC_LAUNCH_OK("tf32x3_gemm_mn_kernel");
    return STC_OK;
  }
  if (nmain < 1) nmain = 1;
  if (nmain > 15) nmain = 15;
  while ((nmain + (small ? 1 : 0)) * Npad > 512 && nmain > 1) --nmain;
  int tmem_cols = 32;
  while (tmem_cols < (nmain + (small ? 1 : 0)) * Npad) tmem_cols *= 2;
  const size_t smem = 2 * 128 * ATOM_ROW_BYTES + 2 * (size_t)Npad * ATOM_ROW_BYTES + 64;
  STC_TRY(set_smem(tf32x3_gemm_kernel, smem));
  ScopedKernelTimer _t(KK_TC_GEMM_TEST, st, 4.0 * ((double)M * K + (double)K * N + (double)M * N));
  tf32x3_gemm_kernel<<<ceil_div(M, 128), CV_THREADS, smem, st>>>(A, Bm, D, M, N, K, Npad, tmem_cols, mode, nmain, small);
  STC_LAUNCH_OK("tf32x3_gemm_kernel");
  return STC_OK;
}

}  // namespace stc
