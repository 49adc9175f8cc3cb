// tcgen05 / TMEM weight-gradient kernel of the gate / candidate convolution.
//
// Reference semantics: autograd of 'bmdk,kh->bmdh' (/root/reference/framework/STC_GNN.py:42) w.r.t. W, i.e.
//     dW_{k,c}[l][o] = sum_rows F_{k,c}[row][l] * dpre[row][o],   F_{k,c} = mix_c(Y_k)        (STC_GNN.py:35-41)
// With the categorical mix moved onto the gradient side (the same identity tc_conv_bwd_dx_kernel uses),
//     dW_{k,c} = Y_k^T * DD_c,      DD_0 = dpre,  DD_c[(node,c')] = sum_d T_c(Gc)[c',d] dpre[(node,d)]
// this is ONE GEMM contracting over rows:  [Ks*KBL x rows] x [rows x Kc*Hout].  The dx kernel leaves DD in HBM
// ([R][Kc*Hout]); here both operands are read straight from HBM with 16-byte loads, split hi/lo (3xTF32) and
// stored MN-major (rows = K index, SWIZZLE_128B_BASE32B) so no transpose is needed.  One 64-row tile = 8 K-steps
// is accumulated in TMEM (short chains: the tensor core truncates on accumulate, profiles/r1_tc_precision.txt),
// then added in fp32 round-to-nearest to per-thread register accumulators; one atomicAdd per element per CTA at
// the end.
#include "stc_conv_common.cuh"
#include "stc_tc.cuh"

#include <stdlib.h>

namespace stc {

using namespace tc;

constexpr int DW_TR = 64;  // rows per tile (K extent of one accumulation chain)

struct TcDwPlan {
  int Dp, KBL;
  int M1, Mpad;   // Ks*KBL, rounded up to 64 / 128 (GEMM M)
  int N1, Npad;   // Kc*Hout, rounded up to 16 (GEMM N)
  int mblk, nblk; // 32-wide column blocks of the two operands
  int tmem_cols;
  long long ntiles;
  int x_vec;      // x-part rows can be read with float4 loads
  int idx32;      // every row index fits 32 bits: divisions by C and N use the multiply-high form
  FastDiv divC, divN;
  uint32_t off_a, off_b, off_bar, smem_bytes;
};

// NCH: 8-column accumulator chunks per thread.  DET: CTA blockIdx.x stores its partial dW into slot blockIdx.x of
// a.det_ws (Ks*Kc*L*Hout floats each; every CTA writes its whole slot) instead of reducing into a.dW.
template <int NCH, bool DET>
__device__ __forceinline__ void tc_conv_bwd_dw_body(const ConvArgs& a, const TcDwPlan& p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((smem_u32(smem) & 1023u) != 0u) __trap();
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int C = a.C, h = a.h, Din = a.Din, Hout = a.Hout, L = a.Din + a.h;
  const uint32_t imgA = (uint32_t)p.mblk * DW_TR * ATOM_ROW_BYTES;   // one hi or lo image
  const uint32_t imgB = (uint32_t)p.nblk * DW_TR * ATOM_ROW_BYTES;
  uint8_t* A_hi = smem + p.off_a;
  uint8_t* A_lo = A_hi + imgA;
  uint8_t* B_hi = smem + p.off_b;
  uint8_t* B_lo = B_hi + imgB;
  uint64_t* mma_bar = reinterpret_cast<uint64_t*>(smem + p.off_bar);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(mma_bar + 1);

  if (tid == 0) {
    mbar_init(mma_bar, 1);
    mbar_fence_init();
  }
  if (warp == 0) tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols);
  // zero both images once: padding columns are never written again
  for (uint32_t i = tid * 16u; i < 2 * imgA + 2 * imgB; i += CV_THREADS * 16u)
    *reinterpret_cast<float4*>(smem + p.off_a + i) = make_float4(0.f, 0.f, 0.f, 0.f);
  fence_async_smem();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t idesc = make_idesc_tf32_mn(p.Mpad, p.Npad);
  const uint32_t d_main = tmem_base, d_small = tmem_base + (uint32_t)p.Npad;
  const long long total_nodes = (long long)a.B * a.N;
  const long long R = total_nodes * C;

  // ---- per-thread chunk mapping.  Every thread owns ONE 16-byte chunk column of each operand and walks the tile
  // rows with a fixed step, so the source pointer / kind are tile- and slot-invariant:
  //   A: 16 chunk columns (Mpad = 64), rows ar0 + 16 i, i < 4;   B: bcols = 4|8|16 chunk columns, rows br0 + bstep i
  constexpr int NA = 4, NB = 4;
  const int am0 = (tid & 15) << 2, ar0 = tid >> 4;
  const float* asrc = nullptr;   // row 0 of the source tensor (+ column), nullptr = zero padding
  int astride = 0, akind = 0, anvalid = 0, axi = 0;   // kind 0 = float4, 1 = scalar, 2 = Xt (batch-strided view)
  if (am0 < p.M1) {
    const int k = am0 / p.KBL, kb = am0 - k * p.KBL;
    if (kb < h) {
      asrc = (k == 0 ? a.h0 : a.yh + (long long)(k - 1) * R * h) + kb;
      astride = h;
    } else if (kb - h < Din) {
      axi = kb - h;
      anvalid = min(4, Din - axi);
      astride = Din;
      if (k == 0) {
        asrc = a.x0;
        akind = 2;
      } else {
        asrc = a.yx + (long long)(k - 1) * R * Din + axi;
        akind = p.x_vec ? 0 : 1;
      }
    }
  }
  const uint32_t asoff = (uint32_t)(am0 >> 5) * (DW_TR * ATOM_ROW_BYTES) + mn32_chunk_offset(ar0, (am0 & 31) >> 2);
  const int bcols = p.Npad > 32 ? 16 : (p.Npad > 16 ? 8 : 4);
  const int bstep = CV_THREADS / bcols, nbs = DW_TR / bstep;   // nbs <= NB
  const int bn0 = (tid % bcols) << 2, br0 = tid / bcols;
  const float* bsrc = bn0 < p.N1 ? a.dpre + bn0 : nullptr;
  const uint32_t bsoff = (uint32_t)(bn0 >> 5) * (DW_TR * ATOM_ROW_BYTES) + mn32_chunk_offset(br0, (bn0 & 31) >> 2);

  auto fetch_a = [&](int row, long long row0, int rows_valid) -> float4 {
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (asrc == nullptr || row >= rows_valid) return v;
    const long long gr = row0 + row;
    if (akind == 0) return __ldg(reinterpret_cast<const float4*>(asrc + gr * astride));
    const float* s;
    if (akind == 2) {  // Xt[b][n][cat][xi..]: the batch axis carries a stride (STC_GNN.py:111 hands in a view)
      if (p.idx32) {
        const uint32_t g = fast_div((uint32_t)gr, p.divC), b = fast_div(g, p.divN);
        // (g - b N) C + cat = gr - b N C
        s = asrc + (long long)b * a.x0_bs + (long long)((uint32_t)gr - b * (uint32_t)(a.N * C)) * Din + axi;
      } else {
        const long long g = gr / C;
        const int cat = (int)(gr - g * C);
        const long long b = g / a.N;
        s = asrc + b * a.x0_bs + ((g - b * a.N) * C + cat) * (long long)Din + axi;
      }
      if (p.x_vec) return __ldg(reinterpret_cast<const float4*>(s));
    } else {
      s = asrc + gr * astride;
    }
    v.x = __ldg(s);
    if (anvalid > 1) v.y = __ldg(s + 1);
    if (anvalid > 2) v.z = __ldg(s + 2);
    if (anvalid > 3) v.w = __ldg(s + 3);
    return v;
  };
  auto fetch_b = [&](int row, long long row0, int rows_valid) -> float4 {
    if (bsrc == nullptr || row >= rows_valid) return make_float4(0.f, 0.f, 0.f, 0.f);
    return __ldg(reinterpret_cast<const float4*>(bsrc + (row0 + row) * p.N1));
  };

  // accumulator ownership: M = 64 uses lanes 0..15 of each 32-lane TMEM sub-partition (row = 16*sp + lane),
  // M = 128 uses all of them (row = 32*sp + lane); the two warps sharing a sub-partition split the columns.
  const int sp = warp & 3, half = warp >> 2;
  const bool m64 = p.Mpad == 64;
  const bool own = m64 ? lane < 16 : true;
  const int mrow = m64 ? sp * 16 + lane : sp * 32 + lane;
  const uint32_t tl = tmem_base + ((uint32_t)(sp * 32) << 16);
  const int ncols_half = p.Npad >> 1;        // Npad % 16 == 0
  const int col0 = half * ncols_half;
  float acc[NCH][8];
#pragma unroll
  for (int i = 0; i < NCH; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

  uint32_t phase = 0;
  float4 ra[NA], rb[NB];
  long long tile = blockIdx.x;
  if (tile < p.ntiles) {
    const long long row0 = tile * DW_TR;
    const int rv = (int)min((long long)DW_TR, R - row0);
#pragma unroll
    for (int i = 0; i < NA; ++i) ra[i] = fetch_a(ar0 + 16 * i, row0, rv);
#pragma unroll
    for (int i = 0; i < NB; ++i)
      if (i < nbs) rb[i] = fetch_b(br0 + bstep * i, row0, rv);
  }
  for (; tile < p.ntiles; tile += gridDim.x) {
    // the images are free: the previous tile's MMAs were waited for before its accumulators were read
#pragma unroll
    for (int i = 0; i < NA; ++i) store_split4(A_hi, A_lo, asoff + (uint32_t)(16 * i) * ATOM_ROW_BYTES, ra[i]);
#pragma unroll
    for (int i = 0; i < NB; ++i)
      if (i < nbs) store_split4(B_hi, B_lo, bsoff + (uint32_t)(bstep * i) * ATOM_ROW_BYTES, rb[i]);
    fence_async_smem();
    __syncthreads();
    if (uniform_warp_index() == 0 && elect_one_sync()) {   // uniform issue path, see stc_tc.cuh
      fence_after_sync();
      const uint32_t lboA = DW_TR * ATOM_ROW_BYTES, lboB = DW_TR * ATOM_ROW_BYTES;
#pragma unroll 1
      for (int ks = 0; ks < DW_TR / 8; ++ks) {
        const uint32_t o = ks * 2 * MN32_GROUP_BYTES;
        const uint64_t ah = make_smem_desc_mn32(smem_u32(A_hi) + o, lboA, MN32_GROUP_BYTES);
        const uint64_t al = make_smem_desc_mn32(smem_u32(A_lo) + o, lboA, MN32_GROUP_BYTES);
        const uint64_t bh = make_smem_desc_mn32(smem_u32(B_hi) + o, lboB, MN32_GROUP_BYTES);
        const uint64_t bl = make_smem_desc_mn32(smem_u32(B_lo) + o, lboB, MN32_GROUP_BYTES);
        mma_tf32(d_small, al, bh, idesc, ks > 0 ? 1u : 0u);
        mma_tf32(d_small, ah, bl, idesc, 1u);
        mma_tf32(d_main, ah, bh, idesc, ks > 0 ? 1u : 0u);
      }
      mma_commit(mma_bar);
    }
    // next tile's operands travel while the tensor core works
    {
      const long long nt = tile + gridDim.x;
      if (nt < p.ntiles) {
        const long long row0 = nt * DW_TR;
        const int rv = (int)min((long long)DW_TR, R - row0);
#pragma unroll
        for (int i = 0; i < NA; ++i) ra[i] = fetch_a(ar0 + 16 * i, row0, rv);
#pragma unroll
        for (int i = 0; i < NB; ++i)
          if (i < nbs) rb[i] = fetch_b(br0 + bstep * i, row0, rv);
      }
    }
    mbar_wait(mma_bar, phase);
    phase ^= 1u;
    fence_after_sync();
#pragma unroll
    for (int i = 0; i < NCH; ++i) {
      if (i * 8 < ncols_half) {
        float v[8], t[8];
        tmem_ld8(tl + (uint32_t)(p.Npad + col0 + i * 8), v);
        tmem_ld8(tl + (uint32_t)(col0 + i * 8), t);
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] += v[j] + t[j];
      }
    }
    fence_before_sync();   // the reads above are ordered before the MMAs issued after the next __syncthreads
  }

  // ---- one (vector) atomic per owned element group ----
  float* const dWo = DET ? a.det_ws + (size_t)blockIdx.x * a.Ks * a.Kc * L * Hout : a.dW;
  const bool dw_v4 = (Hout & 3) == 0 && (col0 & 3) == 0 && (reinterpret_cast<uintptr_t>(dWo) & 15) == 0;
  if (own && mrow < p.M1) {
    const int k = mrow / p.KBL, kb = mrow - k * p.KBL;
    const int l = kb < h ? Din + kb : (kb - h < Din ? kb - h : -1);
    if (l >= 0) {
#pragma unroll
      for (int i = 0; i < NCH; ++i) {
        if (i * 8 >= ncols_half) break;
#pragma unroll
        for (int j = 0; j < 8; j += 4) {
          const int n = col0 + i * 8 + j;
          const int c = n / Hout, o = n - c * Hout;
          float* dst = &dWo[((size_t)(k * a.Kc + c) * L + l) * Hout + o];
          if (dw_v4 && n + 3 < p.N1) {
            grad_out_v4<DET>(dst, acc[i][j], acc[i][j + 1], acc[i][j + 2], acc[i][j + 3]);
          } else {
#pragma unroll
            for (int e = 0; e < 4; ++e)
              if (n + e < p.N1) {
                const int ce = (n + e) / Hout, oe = (n + e) - ce * Hout;
                grad_out<DET>(&dWo[((size_t)(k * a.Kc + ce) * L + l) * Hout + oe], acc[i][j + e]);
              }
          }
        }
      }
    }
  }
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
}

template <int NCH>
__global__ void __launch_bounds__(CV_THREADS, 2)
tc_conv_bwd_dw_kernel(const ConvArgs a, const TcDwPlan p) { tc_conv_bwd_dw_body<NCH, false>(a, p); }
// the deterministic-mode instantiation, under a name of its own (the convolution variant list names the default
// kernels)
template <int NCH>
__global__ void __launch_bounds__(CV_THREADS, 2)
tc_det_bwd_dw_kernel(const ConvArgs a, const TcDwPlan p) { tc_conv_bwd_dw_body<NCH, true>(a, p); }

// =================================================================================================
// Pipelined variant (taken whenever every row piece is 16-byte aligned): the same product, but the operand tiles
// travel HBM -> shared memory as 1-D bulk copies issued by a dedicated producer warp several tiles ahead
// (DWP_STAGES x up to 32 KB in flight per SM), so the consumer warps never wait on a global load: they read the raw
// tile from shared memory, split it hi/lo into one of TWO MN-major image buffers, and the tensor core works on tile t
// while tile t+1 is being split and tile t-1's accumulators are drained (two TMEM accumulator pairs).
// =================================================================================================
constexpr int DWP_CONS_WARPS = 8, DWP_THREADS = 32 * (DWP_CONS_WARPS + 2), DWP_MAX_STAGES = 4;   // + TMA warp + MMA warp

struct TcDwPipePlan {
  int Dp, KBL, M1, N1, Npad, mblk, nblk, stages, tmem_cols;
  long long ntiles;
  uint32_t stage_floats, off_xk, off_d;       // raw stage layout (floats): H_k at k*64*h, X_k at off_xk + k*64*Din, dpre at off_d
  uint32_t off_raw, off_img, img_bytes, off_bar, smem_bytes;
};

template <int NCH, bool DET>   // DET: as tc_conv_bwd_dw_body
__device__ __forceinline__ void tc_conv_bwd_dw_pipe_body(const ConvArgs& a, const TcDwPipePlan& p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((smem_u32(smem) & 1023u) != 0u) __trap();
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int C = a.C, h = a.h, Din = a.Din, Hout = a.Hout, L = a.Din + a.h;
  const uint32_t imgA = (uint32_t)p.mblk * DW_TR * ATOM_ROW_BYTES, imgB = (uint32_t)p.nblk * DW_TR * ATOM_ROW_BYTES;
  float* raw = reinterpret_cast<float*>(smem + p.off_raw);
  uint8_t* img = smem + p.off_img;                       // [2][A_hi | A_lo | B_hi | B_lo]
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + p.off_bar);   // [stages] bytes landed
  uint64_t* empty = full + DWP_MAX_STAGES;                          // [stages] consumer warps done reading
  uint64_t* mma_bar = empty + DWP_MAX_STAGES;                       // [2] MMAs of an image buffer complete
  uint64_t* img_full = mma_bar + 2;                                 // [2] every consumer warp has written its part
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(img_full + 2);
  const long long total_nodes = (long long)a.B * a.N;
  const long long R = total_nodes * C;

  if (tid == 0) {
    for (int i = 0; i < DWP_MAX_STAGES; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], DWP_CONS_WARPS);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&mma_bar[i], 1);
      mbar_init(&img_full[i], DWP_CONS_WARPS);
    }
    mbar_fence_init();
  }
  if (warp == 0) tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols);
  for (uint32_t i = tid * 16u; i < 2 * p.img_bytes; i += DWP_THREADS * 16u)   // padding columns stay zero for good
    *reinterpret_cast<float4*>(img + i) = make_float4(0.f, 0.f, 0.f, 0.f);
  fence_async_smem();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const int warp_u = uniform_warp_index();
  const uint32_t tmem_base = uniform_u32(*tmem_slot);
  const int my_tiles = (int)((p.ntiles - blockIdx.x + gridDim.x - 1) / gridDim.x);

  if (warp_u == DWP_CONS_WARPS) {
    // =========================== producer: one thread issues every bulk copy ===========================
    if (elect_one_sync()) {
      for (int it = 0; it < my_tiles; ++it) {
        const long long tile = blockIdx.x + (long long)it * gridDim.x;
        const int st = it % p.stages;
        mbar_wait(&empty[st], ((uint32_t)(it / p.stages) & 1u) ^ 1u);
        const long long row0 = tile * DW_TR;
        const int rv = (int)min((long long)DW_TR, R - row0);
        float* dst = raw + (size_t)st * p.stage_floats;
        mbar_arrive_expect_tx(&full[st], (uint32_t)(rv * (a.Ks * L + p.N1) * 4));
        for (int k = 0; k < a.Ks; ++k) {
          const float* hsrc = (k == 0 ? a.h0 : a.yh + (long long)(k - 1) * R * h) + row0 * h;
          bulk_g2s(dst + (size_t)k * DW_TR * h, hsrc, (uint32_t)(rv * h * 4), &full[st]);
          float* xd = dst + p.off_xk + (size_t)k * DW_TR * Din;
          if (k > 0) {
            bulk_g2s(xd, a.yx + (long long)(k - 1) * R * Din + row0 * Din, (uint32_t)(rv * Din * 4), &full[st]);
          } else {   // Xt carries a batch stride (STC_GNN.py:111 hands in a view): one copy per sample segment
            long long r = row0;
            int left = rv;
            const long long rows_per_sample = (long long)a.N * C;
            while (left > 0) {
              const long long b = r / rows_per_sample;
              const long long within = r - b * rows_per_sample;
              const int seg = (int)min((long long)left, rows_per_sample - within);
              bulk_g2s(xd, a.x0 + b * a.x0_bs + within * Din, (uint32_t)(seg * Din * 4), &full[st]);
              xd += (size_t)seg * Din;
              r += seg;
              left -= seg;
            }
          }
        }
        bulk_g2s(dst + p.off_d, a.dpre + row0 * p.N1, (uint32_t)(rv * p.N1 * 4), &full[st]);
      }
    }
  } else if (warp_u == DWP_CONS_WARPS + 1) {
    // =========================== MMA issuer: a warp of its own, so no worker ever waits behind the issue queue =====
    if (elect_one_sync()) {   // one lane of the converged warp: descriptors stay in uniform registers (stc_tc.cuh)
      const uint32_t idesc = make_idesc_tf32_mn(64, p.Npad);
      const uint32_t lbo = DW_TR * ATOM_ROW_BYTES;
      for (int it = 0; it < my_tiles; ++it) {
        mbar_wait(&img_full[it & 1], (uint32_t)(it >> 1) & 1u);   // images written, accumulator pair drained
        fence_after_sync();
        const uint32_t base = smem_u32(img + (size_t)(it & 1) * p.img_bytes);
        const uint32_t d_main = tmem_base + (uint32_t)((it & 1) * 2 * p.Npad), d_small = d_main + (uint32_t)p.Npad;
#pragma unroll 1
        for (int ks = 0; ks < DW_TR / 8; ++ks) {
          const uint32_t o = ks * 2 * MN32_GROUP_BYTES;
          const uint64_t ah = make_smem_desc_mn32(base + o, lbo, MN32_GROUP_BYTES);
          const uint64_t al = make_smem_desc_mn32(base + imgA + o, lbo, MN32_GROUP_BYTES);
          const uint64_t bh = make_smem_desc_mn32(base + 2 * imgA + o, lbo, MN32_GROUP_BYTES);
          const uint64_t bl = make_smem_desc_mn32(base + 2 * imgA + imgB + o, lbo, MN32_GROUP_BYTES);
          mma_tf32(d_small, al, bh, idesc, ks > 0 ? 1u : 0u);
          mma_tf32(d_small, ah, bl, idesc, 1u);
          mma_tf32(d_main, ah, bh, idesc, ks > 0 ? 1u : 0u);
        }
        mma_commit(&mma_bar[it & 1]);
      }
    }
  } else {
    // =========================== consumers ===========================
    // chunk mapping (as in the kernel above): A has 16 chunk columns (Mpad = 64), rows ar0 + 16 i; B bcols chunk columns
    constexpr int NA = 4, NB = 4;
    const int am0 = (tid & 15) << 2, ar0 = tid >> 4;
    int asrc_off = -1, astride = 0, anvalid = 4;   // offset of (row 0, this chunk) inside a raw stage; -1 = zero padding
    if (am0 < p.M1) {
      const int k = am0 / p.KBL, kb = am0 - k * p.KBL;
      if (kb < h) {
        asrc_off = k * DW_TR * h + kb;
        astride = h;
      } else if (kb - h < Din) {
        asrc_off = (int)p.off_xk + k * DW_TR * Din + (kb - h);
        astride = Din;
        anvalid = min(4, Din - (kb - h));
      }
    }
    const bool avec = anvalid == 4 && (astride % 4) == 0;
    const uint32_t asoff = (uint32_t)(am0 >> 5) * (DW_TR * ATOM_ROW_BYTES) + mn32_chunk_offset(ar0, (am0 & 31) >> 2);
    const int bcols = p.Npad > 32 ? 16 : (p.Npad > 16 ? 8 : 4);
    const int bstep = (32 * DWP_CONS_WARPS) / bcols, nbs = DW_TR / bstep;   // nbs <= NB
    const int bn0 = (tid % bcols) << 2, br0 = tid / bcols;
    const bool blive = bn0 < p.N1;
    const uint32_t bsoff = (uint32_t)(bn0 >> 5) * (DW_TR * ATOM_ROW_BYTES) + mn32_chunk_offset(br0, (bn0 & 31) >> 2);

    auto split_tile = [&](int it) {   // raw stage of local tile `it` -> image buffer it & 1
      const long long tile = blockIdx.x + (long long)it * gridDim.x;
      const int rv = (int)min((long long)DW_TR, R - tile * DW_TR);
      const int st = it % p.stages;
      mbar_wait(&full[st], (uint32_t)(it / p.stages) & 1u);
      const float* src = raw + (size_t)st * p.stage_floats;
      uint8_t* A_hi = img + (size_t)(it & 1) * p.img_bytes;
      uint8_t* A_lo = A_hi + imgA;
      uint8_t* B_hi = A_lo + imgA;
      uint8_t* B_lo = B_hi + imgB;
#pragma unroll
      for (int i = 0; i < NA; ++i) {
        const int row = ar0 + 16 * i;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (asrc_off >= 0 && row < rv) {
          const float* s = src + asrc_off + row * astride;
          if (avec) {
            v = *reinterpret_cast<const float4*>(s);
          } else {
            v.x = s[0];
            if (anvalid > 1) v.y = s[1];
            if (anvalid > 2) v.z = s[2];
            if (anvalid > 3) v.w = s[3];
          }
        }
        store_split4(A_hi, A_lo, asoff + (uint32_t)(16 * i) * ATOM_ROW_BYTES, v);
      }
#pragma unroll
      for (int i = 0; i < NB; ++i)
        if (i < nbs) {
          const int row = br0 + bstep * i;
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (blive && row < rv) v = *reinterpret_cast<const float4*>(src + p.off_d + row * p.N1 + bn0);
          store_split4(B_hi, B_lo, bsoff + (uint32_t)(bstep * i) * ATOM_ROW_BYTES, v);
        }
      fence_async_smem();                        // image stores visible to the tensor core's (async) proxy
      fence_before_sync();                       // ... and this warp's earlier TMEM reads ordered before the hand-over
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(&empty[st]);                 // this warp no longer reads the raw stage
        mbar_arrive(&img_full[it & 1]);          // its share of the image is in place
      }
    };
    // accumulator ownership (M = 64): lanes 0..15 of each TMEM sub-partition, row = 16*sp + lane; the two warps that
    // share a sub-partition split the columns
    const int sp = warp & 3, half = warp >> 2;
    const bool own = lane < 16;
    const int mrow = sp * 16 + lane;
    const uint32_t tl = tmem_base + ((uint32_t)(sp * 32) << 16);
    const int ncols_half = p.Npad >> 1;
    const int col0 = half * ncols_half;
    float acc[NCH][8];
#pragma unroll
    for (int i = 0; i < NCH; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

    if (my_tiles > 0) split_tile(0);
    for (int it = 0; it < my_tiles; ++it) {
      // tile it+1 is split while the tensor core works on tile it: its image buffer and accumulator pair were released
      // when this warp drained tile it-1 (program order), and the MMA warp waits for all eight warps' arrivals
      if (it + 1 < my_tiles) split_tile(it + 1);
      mbar_wait(&mma_bar[it & 1], (uint32_t)(it >> 1) & 1u);
      fence_after_sync();
      const uint32_t ab = (uint32_t)((it & 1) * 2 * p.Npad);
#pragma unroll
      for (int i = 0; i < NCH; ++i) {
        if (i * 8 < ncols_half) {
          uint32_t v[8], t[8];
          tmem_ld8_async(tl + ab + (uint32_t)(p.Npad + col0 + i * 8), v);
          tmem_ld8_async(tl + ab + (uint32_t)(col0 + i * 8), t);
          tmem_ld_wait();
          tmem_ld_pin8(v);
          tmem_ld_pin8(t);
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[i][j] += __uint_as_float(v[j]) + __uint_as_float(t[j]);
        }
      }
    }
    // ---- one (vector) atomic per owned element group ----
    float* const dWo = DET ? a.det_ws + (size_t)blockIdx.x * a.Ks * a.Kc * L * Hout : a.dW;
    const bool dw_v4 = (Hout & 3) == 0 && (col0 & 3) == 0 && (reinterpret_cast<uintptr_t>(dWo) & 15) == 0;
    if (own && mrow < p.M1) {
      const int k = mrow / p.KBL, kb = mrow - k * p.KBL;
      const int l = kb < h ? Din + kb : (kb - h < Din ? kb - h : -1);
      if (l >= 0) {
#pragma unroll
        for (int i = 0; i < NCH; ++i) {
          if (i * 8 >= ncols_half) break;
#pragma unroll
          for (int j = 0; j < 8; j += 4) {
            const int n = col0 + i * 8 + j;
            const int c = n / Hout, o = n - c * Hout;
            float* dst = &dWo[((size_t)(k * a.Kc + c) * L + l) * Hout + o];
            // Hout % 4 == 0 and n % 4 == 0: the four columns stay inside one categorical block and one 16-byte slot
            if (dw_v4 && n + 3 < p.N1) {
              grad_out_v4<DET>(dst, acc[i][j], acc[i][j + 1], acc[i][j + 2], acc[i][j + 3]);
            } else {
#pragma unroll
              for (int e = 0; e < 4; ++e)
                if (n + e < p.N1) {
                  const int ce = (n + e) / Hout, oe = (n + e) - ce * Hout;
                  grad_out<DET>(&dWo[((size_t)(k * a.Kc + ce) * L + l) * Hout + oe], acc[i][j + e]);
                }
            }
          }
        }
      }
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
}

template <int NCH>
__global__ void __launch_bounds__(DWP_THREADS, 1)
tc_conv_bwd_dw_pipe_kernel(const ConvArgs a, const TcDwPipePlan p) { tc_conv_bwd_dw_pipe_body<NCH, false>(a, p); }
// the deterministic-mode instantiation, under a name of its own (the convolution variant list names the default
// kernels)
template <int NCH>
__global__ void __launch_bounds__(DWP_THREADS, 1)
tc_det_bwd_dw_pipe_kernel(const ConvArgs a, const TcDwPipePlan p) { tc_conv_bwd_dw_pipe_body<NCH, true>(a, p); }

static bool aligned16d(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// one dW launch (timed as tc_conv_bwd_dw); with a.det_ws (deterministic mode) the slot form, then the fixed-order sum of
// its grid slots into a.dW
template <typename Plan, typename K>
static int launch_dw(K plain, K det, const ConvArgs& a, const Plan& p, int grid, int threads, double bytes, cudaStream_t st) {
  const bool dm = a.det_ws != nullptr;
  if (dm && grid > det_conv_slots()) {
    set_error("tc_conv_bwd_dw: %d CTAs but %d partial slots", grid, det_conv_slots());
    return STC_ERR_WORKSPACE;
  }
  K kern = dm ? det : plain;
  STC_TRY(set_smem(kern, p.smem_bytes));
  {
    ScopedKernelTimer _t(KK_TC_CONV_BWD_DW, st, bytes);
    kern<<<grid, threads, p.smem_bytes, st>>>(a, p);
    STC_LAUNCH_OK("tc_conv_bwd_dw_kernel");
  }
  if (!dm) return STC_OK;
  const long long n = (long long)a.Ks * a.Kc * (a.Din + a.h) * a.Hout;
  return launch_det_reduce(a.dW, a.det_ws, grid, n, n, st);
}

// Pipelined dW kernel: every bulk copy must start 16-byte aligned and move a multiple of 16 bytes.
static int try_launch_dw_pipe(const ConvArgs& a, cudaStream_t st, bool* piped) {
  *piped = false;
  if (getenv("STC_DW_NO_PIPE")) return STC_OK;
  const long long R = (long long)a.B * a.N * a.C;
  const long long sample_x = (long long)a.N * a.C * a.Din;
  if (a.h % 4 != 0 || sample_x % 4 != 0 || a.x0_bs % 4 != 0 || (R * a.Din) % 4 != 0 || (R * a.h) % 4 != 0 ||
      ((long long)a.N * a.C * a.h) % 4 != 0 || (DW_TR * a.Din) % 4 != 0 || !aligned16d(a.x0) || !aligned16d(a.yx))
    return STC_OK;
  // a tile may start inside a sample: rows_before * Din floats must stay a multiple of 4 at every sample boundary
  if (a.Din % 4 != 0 && ((long long)a.N * a.C) % 4 != 0) return STC_OK;
  const int L = a.Din + a.h;
  TcDwPipePlan p;
  p.Dp = (a.Din + 7) & ~7;
  p.KBL = a.h + p.Dp;
  p.M1 = a.Ks * p.KBL;
  p.N1 = a.Kc * a.Hout;
  p.Npad = (p.N1 + 15) & ~15;
  p.mblk = 2;
  p.nblk = (p.Npad + 31) / 32;
  p.tmem_cols = 32;
  while (p.tmem_cols < 4 * p.Npad) p.tmem_cols *= 2;
  p.ntiles = (R + DW_TR - 1) / DW_TR;
  p.off_xk = (uint32_t)(a.Ks * DW_TR * a.h);
  p.off_d = (uint32_t)round_up((size_t)p.off_xk + (size_t)a.Ks * DW_TR * a.Din, 4);
  p.stage_floats = (uint32_t)round_up((size_t)p.off_d + (size_t)DW_TR * p.N1, 32);
  p.img_bytes = 2 * (uint32_t)(p.mblk + p.nblk) * DW_TR * ATOM_ROW_BYTES;
  const size_t fixed = 2 * (size_t)p.img_bytes + 8 * (2 * DWP_MAX_STAGES + 4) + 64;
  p.stages = DWP_MAX_STAGES;
  while (p.stages > 2 && fixed + (size_t)p.stages * p.stage_floats * 4 > 227 * 1024) --p.stages;
  if (fixed + (size_t)p.stages * p.stage_floats * 4 > 227 * 1024) return STC_OK;
  size_t o = 0;
  p.off_img = (uint32_t)o; o += 2 * (size_t)p.img_bytes;
  p.off_raw = (uint32_t)o; o += (size_t)p.stages * p.stage_floats * 4;
  p.off_bar = (uint32_t)o; o += 8 * (2 * DWP_MAX_STAGES + 4) + 16;
  p.smem_bytes = (uint32_t)o;
  const int nch = (p.Npad / 2 + 7) / 8;
  long long grid = device_sm_count();
  if (grid > p.ntiles) grid = p.ntiles;
  const double bytes = 4.0 * (double)R * (a.Ks * L + a.Kc * a.Hout) + 4.0 * a.Ks * a.Kc * L * a.Hout;
  switch (nch) {
    case 1: STC_TRY(launch_dw(tc_conv_bwd_dw_pipe_kernel<1>, tc_det_bwd_dw_pipe_kernel<1>, a, p, (int)grid, DWP_THREADS, bytes, st)); break;
    case 2: STC_TRY(launch_dw(tc_conv_bwd_dw_pipe_kernel<2>, tc_det_bwd_dw_pipe_kernel<2>, a, p, (int)grid, DWP_THREADS, bytes, st)); break;
    default: STC_TRY(launch_dw(tc_conv_bwd_dw_pipe_kernel<4>, tc_det_bwd_dw_pipe_kernel<4>, a, p, (int)grid, DWP_THREADS, bytes, st)); break;
  }
  *piped = true;
  return STC_OK;
}

bool conv_tc_dw_shape_ok(const ConvArgs& a) {
  const int Dp = (a.Din + 7) & ~7, KBL = a.h + Dp;
  return a.Ks * KBL <= 64 && a.Kc * a.Hout <= 64 && a.h % 8 == 0 && a.Hout % 16 == 0;
}

int try_launch_conv_bwd_dw_tc(const ConvArgs& a, cudaStream_t st, bool* handled) {
  *handled = false;
  if (!conv_tc_eligible(a) || !conv_tc_dw_shape_ok(a)) return STC_OK;   // FFMA kernel (it honours dpre_ld)
  if (!aligned16d(a.h0) || !aligned16d(a.yh) || !aligned16d(a.dpre)) {
    set_error("tcgen05 dW kernel needs 16-byte aligned state / workspace tensors");
    return STC_ERR_BAD_ARG;
  }
  const int L = a.Din + a.h;
  {
    bool piped = false;
    STC_TRY(try_launch_dw_pipe(a, st, &piped));
    if (piped) {
      *handled = true;
      return STC_OK;
    }
  }
  TcDwPlan p;
  p.Dp = (a.Din + 7) & ~7;
  p.KBL = a.h + p.Dp;
  p.M1 = a.Ks * p.KBL;
  p.Mpad = 64;
  p.N1 = a.Kc * a.Hout;
  p.Npad = (p.N1 + 15) & ~15;
  p.mblk = p.Mpad / 32;
  p.nblk = (p.Npad + 31) / 32;
  p.tmem_cols = 32;
  while (p.tmem_cols < 2 * p.Npad) p.tmem_cols *= 2;
  const long long R = (long long)a.B * a.N * a.C;
  p.ntiles = (R + DW_TR - 1) / DW_TR;
  p.x_vec = (a.Din % 4 == 0) && (a.x0_bs % 4 == 0) && aligned16d(a.x0) && aligned16d(a.yx);
  p.idx32 = R < (1LL << 31) ? 1 : 0;
  p.divC = make_fastdiv((uint32_t)a.C);
  p.divN = make_fastdiv((uint32_t)a.N);
  size_t o = 0;
  p.off_a = (uint32_t)o; o += 2 * (size_t)p.mblk * DW_TR * ATOM_ROW_BYTES;
  p.off_b = (uint32_t)o; o += 2 * (size_t)p.nblk * DW_TR * ATOM_ROW_BYTES;
  p.off_bar = (uint32_t)o; o += 32;
  p.smem_bytes = (uint32_t)o;
  const int nch = (p.Npad / 2 + 7) / 8;   // 8-column chunks per thread
  int ctas_per_sm = 2;
  if (ctas_per_sm * p.tmem_cols > 512) ctas_per_sm = 512 / p.tmem_cols;
  long long grid = (long long)device_sm_count() * ctas_per_sm;
  if (grid > p.ntiles) grid = p.ntiles;
  // compulsory traffic per row: the Ks spatial terms of [x|h] once and the (unmixed) pre-activation gradient once
  const double bytes = 4.0 * (double)R * (a.Ks * L + a.Kc * a.Hout) + 4.0 * a.Ks * a.Kc * L * a.Hout;
  switch (nch) {
    case 1: STC_TRY(launch_dw(tc_conv_bwd_dw_kernel<1>, tc_det_bwd_dw_kernel<1>, a, p, (int)grid, CV_THREADS, bytes, st)); break;
    case 2: STC_TRY(launch_dw(tc_conv_bwd_dw_kernel<2>, tc_det_bwd_dw_kernel<2>, a, p, (int)grid, CV_THREADS, bytes, st)); break;
    default: STC_TRY(launch_dw(tc_conv_bwd_dw_kernel<4>, tc_det_bwd_dw_kernel<4>, a, p, (int)grid, CV_THREADS, bytes, st)); break;
  }
  *handled = true;
  return STC_OK;
}

}  // namespace stc
