// tcgen05 / TMEM backward kernels of the gate / candidate convolution (the adjoint of stc_conv_tc.cu).
//
// tc_conv_bwd_dx_kernel, per 128-row tile (whole nodes x all categories):
//   1. CUDA cores: GRU / activation adjoint -> pre-activation gradient Ds [rows][Hout] (also written to HBM for
//      the dW kernel), bias-gradient column sums, the direct dH terms;
//      (Ds and its unmixed copies Dm_c are also written to HBM for the dW kernel, stc_conv_tc_dw.cu)
//   2. the categorical mix is pulled onto the K side:  dY_k = [Ds | Dm_1 | ...] x [W_{k,0}^T ; W_{k,1}^T ; ...]
//      with Dm_c[(node,c')] = sum_d T_c(Gc)[c',d] Ds[(node,d)]  (adjoint of 'bmcl,cd->bmdl', STC_GNN.py:38),
//      so one 3xTF32 tensor-core GEMM [rows x Kc*Hout] x [Kc*Hout x Ks*KBL] yields every spatial-term adjoint;
//   3. epilogue: TMEM -> registers -> dY_k tiles in HBM (x-part accumulated across the two convolutions);
//   4. dT_c(Gc) from the partial outputs P_c the forward kernel saved:  dQ_c[c',d] = sum P_c[(n,c')][o] Ds[(n,d)][o].
#include "stc_conv_common.cuh"
#include "stc_tc.cuh"

namespace stc {

using namespace tc;

constexpr int DX_APM = 3;  // atoms chained into one main accumulator (12 K-steps; see TC_APM in stc_conv_tc.cu)

struct TcDxPlan {
  int npt, Dp, KBL;
  int N1;         // Ks * KBL  (GEMM N: every spatial term's [h | x] block)
  int Npad;       // N1 rounded up to 16
  int Kdd;        // Kc * Hout (GEMM K)
  int KA;         // 32-wide atoms along K
  int nmain;      // main accumulators = ceil(KA / DX_APM); the cross-term accumulator follows them
  int tmem_cols, ntiles;
  int DP;         // row stride of the plain Ds tile (floats)
  int PW;         // (Kc-1) * Hout: width of the saved partial-output tile
  int x_vec;      // x-part adjoints can be written (and accumulated) with 16-byte accesses
  uint32_t off_a, off_b, off_ds, off_dh, off_ps, off_q, off_acc, off_bar, smem_bytes;
};

// operands of one prologue item (4 hidden channels of one row)
struct DxIn {
  float4 dhn, uu, cc, hp, rr, drh;
};
__device__ __forceinline__ void dx_load(const ConvArgs& a, long long o, DxIn& in) {
  in.dhn = *reinterpret_cast<const float4*>(a.dHn + o);
  in.uu = *reinterpret_cast<const float4*>(a.u + o);
  in.cc = *reinterpret_cast<const float4*>(a.c + o);
  if (a.phase == 0) {
    in.hp = *reinterpret_cast<const float4*>(a.Hprev + o);
    in.rr = *reinterpret_cast<const float4*>(a.r + o);
    in.drh = *reinterpret_cast<const float4*>(a.drH + o);
  }
}
// GRU / activation adjoint (SURVEY 2.2): g0v = pre-activation gradient of the candidate (phase 1) or of u (phase 0),
// g1v = of r, dir = the direct dH terms
__device__ __forceinline__ void dx_adjoint(const ConvArgs& a, const DxIn& in, float4& g0v, float4& g1v, float4& dir) {
  const float4 dhn = in.dhn, uu = in.uu, cc = in.cc;
  if (a.phase == 1) {
    g0v = make_float4(dhn.x * uu.x * (1.f - cc.x * cc.x), dhn.y * uu.y * (1.f - cc.y * cc.y),
                      dhn.z * uu.z * (1.f - cc.z * cc.z), dhn.w * uu.w * (1.f - cc.w * cc.w));
    if (a.act == STC_ACT_RELU) {
      if (!(cc.x > 0.f)) g0v.x = 0.f;
      if (!(cc.y > 0.f)) g0v.y = 0.f;
      if (!(cc.z > 0.f)) g0v.z = 0.f;
      if (!(cc.w > 0.f)) g0v.w = 0.f;
    }
  } else {
    const float4 hp = in.hp, rr = in.rr, drh = in.drh;
    g0v = make_float4(dhn.x * (cc.x - hp.x) * uu.x * (1.f - uu.x), dhn.y * (cc.y - hp.y) * uu.y * (1.f - uu.y),
                      dhn.z * (cc.z - hp.z) * uu.z * (1.f - uu.z), dhn.w * (cc.w - hp.w) * uu.w * (1.f - uu.w));
    g1v = make_float4(drh.x * hp.x * rr.x * (1.f - rr.x), drh.y * hp.y * rr.y * (1.f - rr.y),
                      drh.z * hp.z * rr.z * (1.f - rr.z), drh.w * hp.w * rr.w * (1.f - rr.w));
    if (a.act == STC_ACT_RELU) {
      if (!(uu.x > 0.5f)) g0v.x = 0.f;
      if (!(uu.y > 0.5f)) g0v.y = 0.f;
      if (!(uu.z > 0.5f)) g0v.z = 0.f;
      if (!(uu.w > 0.5f)) g0v.w = 0.f;
      if (!(rr.x > 0.5f)) g1v.x = 0.f;
      if (!(rr.y > 0.5f)) g1v.y = 0.f;
      if (!(rr.z > 0.5f)) g1v.z = 0.f;
      if (!(rr.w > 0.5f)) g1v.w = 0.f;
    }
    dir = make_float4(dhn.x * (1.f - uu.x) + drh.x * rr.x, dhn.y * (1.f - uu.y) + drh.y * rr.y,
                      dhn.z * (1.f - uu.z) + drh.z * rr.z, dhn.w * (1.f - uu.w) + drh.w * rr.w);
  }
}

// one lane: pull the next tile's operands (and the x-part adjoints the gates pass accumulates into) towards L2
__device__ __forceinline__ void dx_prefetch_tile(const ConvArgs& a, const TcDxPlan& p, int tile, bool want_dQ) {
  const long long total_nodes = (long long)a.B * a.N;
  const long long g0 = (long long)tile * p.npt;
  const int nv = (int)min((long long)p.npt, total_nodes - g0);
  const long long row0 = g0 * a.C;
  const uint32_t hb = (uint32_t)(nv * a.C * a.h * 4);
  l2_prefetch(a.dHn + row0 * a.h, hb);
  l2_prefetch(a.u + row0 * a.h, hb);
  l2_prefetch(a.c + row0 * a.h, hb);
  if (a.phase == 0) {
    l2_prefetch(a.Hprev + row0 * a.h, hb);
    l2_prefetch(a.r + row0 * a.h, hb);
    l2_prefetch(a.drH + row0 * a.h, hb);
  }
  if (want_dQ) l2_prefetch(a.Psave + row0 * p.PW, (uint32_t)(nv * a.C * p.PW * 4));
  const long long R = total_nodes * a.C;
  if (a.accum_x && p.x_vec) {
    const uint32_t xb = (uint32_t)(nv * a.C * a.Din * 4);
    if (a.dYx0) l2_prefetch(a.dYx0 + row0 * a.Din, xb);
    if (a.dYx)
      for (int k = 1; k < a.Ks; ++k) l2_prefetch(a.dYx + (size_t)(k - 1) * R * a.Din + row0 * a.Din, xb);
  } else if (a.dYx_add && p.x_vec) {
    const uint32_t xb = (uint32_t)(nv * a.C * a.Din * 4);
    for (int k = 1; k < a.Ks; ++k) l2_prefetch(a.dYx_add + (size_t)(k - 1) * R * a.Din + row0 * a.Din, xb);
  }
  if (a.dYh_add)
    for (int k = 1; k < a.Ks; ++k) l2_prefetch(a.dYh_add + (size_t)(k - 1) * R * a.h + row0 * a.h, hb);
}

// FAST: contiguous-column epilogue of the common shape (Ks = 2, h = 16, Din <= 16, one main accumulator)
// AT (implies FAST, Kc = 2): the A operand [Ds | Dm_1] goes from registers straight into TENSOR MEMORY (tcgen05.st) and
//     the MMAs read it from there -- no A atoms in shared memory, no proxy fence, no MMA round trip between atoms
//     (see tc_conv_fwd_at_kernel in stc_conv_tc.cu for the measurements behind this)
template <bool FAST, bool AT>
__global__ void __launch_bounds__(CV_THREADS, 2)
tc_conv_bwd_dx_kernel(const ConvArgs a, const TcDxPlan p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((smem_u32(smem) & 1023u) != 0u) __trap();
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int C = a.C, L = a.Din + a.h, h = a.h, Din = a.Din, Hout = a.Hout, DP = p.DP;
  const bool want_dQ = a.dQ != nullptr && a.Kc > 1;
  const uint32_t atomA = 128 * ATOM_ROW_BYTES;
  const uint32_t atomB = (uint32_t)p.Npad * ATOM_ROW_BYTES;
  uint8_t* A_hi = smem + p.off_a;
  uint8_t* A_lo = A_hi + atomA;
  // resident weight atoms: [KA][hi] then [KA][lo]; AT: per atom [hi | lo] so that one descriptor over both is the
  // N = 2 Npad operand [W_hi ; W_lo] (A_hi x [W_hi ; W_lo] fills the main and the cross-term accumulator in one MMA)
  uint8_t* B_hi = smem + p.off_b;
  uint8_t* B_lo = B_hi + (AT ? (size_t)atomB : (size_t)p.KA * atomB);
  const size_t bstride = AT ? 2 * (size_t)atomB : (size_t)atomB;   // distance between consecutive atoms
  float* Dsm = reinterpret_cast<float*>(smem + p.off_ds);       // [128][DP]  plain Ds
  float* Dh = reinterpret_cast<float*>(smem + p.off_dh);        // [128][h]   direct dH terms (gates)
  float* Psm = reinterpret_cast<float*>(smem + p.off_ps);       // [128][PW]  saved P_c tile (bulk copied)
  float* Qs = reinterpret_cast<float*>(smem + p.off_q);         // [(Kc-1)][C][C]
  float* dQacc = reinterpret_cast<float*>(smem + p.off_acc);    // [(Kc-1)][C][C] per-CTA accumulators
  uint64_t* mma_bar = reinterpret_cast<uint64_t*>(smem + p.off_bar);
  uint64_t* load_bar = mma_bar + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(mma_bar + 2);

  if (tid == 0) {
    mbar_init(mma_bar, 1);
    mbar_init(load_bar, 1);
    mbar_fence_init();
  }
  if (warp == 0) tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols);
  for (int i = tid; i < (a.Kc - 1) * C * C; i += CV_THREADS) {
    Qs[i] = a.Q[C * C + i];
    dQacc[i] = 0.f;
  }
  // resident B atoms:  Bt[(k,kb)][(c,o)] = W[((k*Kc + c)*L + l(kb))*Hout + o]
  for (int ja = 0; ja < p.KA; ++ja) {
    uint8_t* bh = B_hi + (size_t)ja * bstride;
    uint8_t* bl = B_lo + (size_t)ja * bstride;
    for (int it = tid; it < p.Npad * 8; it += CV_THREADS) {
      const int n = it >> 3, qq = it & 7;
      const int k = n / p.KBL, kb = n - k * p.KBL;
      const int l = kb < h ? Din + kb : (kb - h < Din ? kb - h : -1);
      float v[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int kk = ja * ATOM_K + qq * 4 + i;
        const int c = kk / Hout, o = kk - c * Hout;
        v[i] = (n < p.N1 && l >= 0 && kk < p.Kdd) ? a.W[((size_t)(k * a.Kc + c) * L + l) * Hout + o] : 0.f;
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
  const uint32_t d_small = tmem_base + (uint32_t)(p.nmain * p.Npad);
  // operand descriptors are launch constants: only the 16-byte-granular address field moves (K-step: +32 B, atom: +atomB)
  const uint64_t dA_hi = make_smem_desc_sw128(smem_u32(A_hi)), dA_lo = make_smem_desc_sw128(smem_u32(A_lo));
  const uint64_t dB_hi = make_smem_desc_sw128(smem_u32(B_hi)), dB_lo = make_smem_desc_sw128(smem_u32(B_lo));
  const long long total_nodes = (long long)a.B * a.N;
  const long long R = total_nodes * C;

  const int q = tid & 7, r0 = tid >> 3;
  uint32_t aoff[4];
  int rnode[4], rcat[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    aoff[i] = atom_chunk_offset(r0 + 32 * i, q);
    rnode[i] = (r0 + 32 * i) / C;
    rcat[i] = (r0 + 32 * i) - rnode[i] * C;
  }
  const int lane_base = (warp & 3) * 32, half = warp >> 2;
  const int erow = lane_base + lane;
  const uint32_t tl = tmem_base + ((uint32_t)lane_base << 16);
  // bias gradient: a thread's column chunk j is the same for every prologue item it handles (CV_THREADS % (h/4) == 0),
  // so the column sums live in registers for the whole kernel; otherwise a per-tile pass over the Ds tile is used
  const bool db_fast = a.dbias != nullptr && (CV_THREADS % (h >> 2)) == 0;
  float4 dbs0 = make_float4(0.f, 0.f, 0.f, 0.f), dbs1 = dbs0;
  float db_acc = 0.f;  // slow path: thread (group g, column j) owns rows g, g + groups, ... of bias-gradient column j
  const int db_groups = CV_THREADS / Hout, db_col = tid % Hout, db_grp = tid / Hout;
  // dT_1(Gc) fast path (Kc == 2, C <= DQ_C): thread (node slot, 4-channel chunk) keeps the C x C partial sums in
  // registers across tiles -- conflict-free 16-byte reads of the P and Ds tiles, one reduction at the end
  constexpr int DQ_C = 5;
  const int dq_chunks = Hout >> 2;
  const bool dq_fast = want_dQ && a.Kc == 2 && C <= DQ_C && p.npt * dq_chunks <= CV_THREADS;
  const int dq_node = tid / dq_chunks, dq_oc = (tid - dq_node * dq_chunks) << 2;
  float dq[DQ_C * DQ_C];
#pragma unroll
  for (int i = 0; i < DQ_C * DQ_C; ++i) dq[i] = 0.f;
  uint32_t mma_phase = 0, load_phase = 0;
  bool mma_pending = false;
  const bool tracing = a.trace != nullptr && blockIdx.x == 0 && tid == 0;
  int trace_it = 0;

  for (int tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x) {
    const long long g0 = (long long)tile * p.npt;
    const int nodes_valid = (int)min((long long)p.npt, total_nodes - g0);
    const int rows_valid = nodes_valid * C;
    const long long row0 = g0 * C;
    if (warp_u == 1 && elect_one_sync()) {  // a lane of warp 1 owns the bulk copy and the prefetches, warp 0 only issues MMAs
      if (want_dQ) {  // stage the saved partial outputs of this tile while the prologue runs
        const uint32_t bytes = (uint32_t)(rows_valid * p.PW * 4);
        mbar_arrive_expect_tx(load_bar, bytes);
        bulk_g2s(Psm, a.Psave + row0 * p.PW, bytes, load_bar);
      }
      if ((a.opt & OPT_L2_PREFETCH) && tile + (int)gridDim.x < p.ntiles) dx_prefetch_tile(a, p, tile + gridDim.x, want_dQ);
    }
    STC_TRACE(0);
    // ---- 1. elementwise adjoint: one float4 of hidden channels per item ----
    const int cpr = h >> 2;
    auto emit_item = [&](int row, int j, const float4& g0v, const float4& g1v, const float4& dir, bool live) {
      if (live) {
        *reinterpret_cast<float4*>(a.dpre + (row0 + row) * p.Kdd + j) = g0v;
        if (a.phase == 0) *reinterpret_cast<float4*>(a.dpre + (row0 + row) * p.Kdd + h + j) = g1v;
      }
      if (db_fast) {
        dbs0.x += g0v.x; dbs0.y += g0v.y; dbs0.z += g0v.z; dbs0.w += g0v.w;
        dbs1.x += g1v.x; dbs1.y += g1v.y; dbs1.z += g1v.z; dbs1.w += g1v.w;
      }
      *reinterpret_cast<float4*>(Dsm + row * DP + j) = g0v;
      if (a.phase == 0) {
        *reinterpret_cast<float4*>(Dsm + row * DP + h + j) = g1v;
        *reinterpret_cast<float4*>(Dh + row * h + j) = dir;
      }
    };
    // (issuing both rounds' loads before the first use was measured: shorter prologue, slower kernel -- the extra
    //  48 live registers spill)
    for (int it = tid; it < 128 * cpr; it += CV_THREADS) {
      const int row = it / cpr, j = (it - row * cpr) << 2;
      float4 g0v = make_float4(0.f, 0.f, 0.f, 0.f), g1v = g0v, dir = g0v;
      const bool live = row < rows_valid;
      if (live) {
        DxIn in;
        dx_load(a, (row0 + row) * h + j, in);
        dx_adjoint(a, in, g0v, g1v, dir);
      }
      emit_item(row, j, g0v, g1v, dir, live);
    }
    __syncthreads();
    STC_TRACE(1);
    if (a.dbias && !db_fast && tid < db_groups * Hout) {   // every thread sums a strided slice of rows of its column
      float s = 0.f;
      for (int row = db_grp; row < rows_valid; row += db_groups) s += Dsm[row * DP + db_col];
      db_acc += s;
    }
    if constexpr (AT) {
      // ---- 2'. my row's share of the A operand: Ds columns [cw*half, +cw) and the same columns of Dm_1 ----
      const int cw = Hout >> 1;                        // 8 (candidate) or 16 (gates)
      const int cbase = cw * half;
      const int enode = erow / C, ecat = erow - enode * C;
      const float* qrow = Qs + ecat * C;               // Dm_1[(node,c')][o] = sum_d Q_1[c'][d] Ds[(node,d)][o]
      const uint32_t tA = tl + (uint32_t)(2 * p.Npad);
      // both 8-column parts of a 16-column share (gates) advance through the category loop together: twice the
      // independent FMA chains and loads in flight per thread
      const bool two = cw == 16;
      float dm[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) dm[i] = 0.f;
      {
        const float* sp = Dsm + (enode * C) * DP + cbase;
#pragma unroll 5
        for (int d = 0; d < C; ++d) {
          const float w = qrow[d];
          const float4 x0 = *reinterpret_cast<const float4*>(sp + d * DP);
          const float4 x1 = *reinterpret_cast<const float4*>(sp + d * DP + 4);
          dm[0] = fmaf(w, x0.x, dm[0]); dm[1] = fmaf(w, x0.y, dm[1]); dm[2] = fmaf(w, x0.z, dm[2]); dm[3] = fmaf(w, x0.w, dm[3]);
          dm[4] = fmaf(w, x1.x, dm[4]); dm[5] = fmaf(w, x1.y, dm[5]); dm[6] = fmaf(w, x1.z, dm[6]); dm[7] = fmaf(w, x1.w, dm[7]);
          if (two) {
            const float4 x2 = *reinterpret_cast<const float4*>(sp + d * DP + 8);
            const float4 x3 = *reinterpret_cast<const float4*>(sp + d * DP + 12);
            dm[8] = fmaf(w, x2.x, dm[8]); dm[9] = fmaf(w, x2.y, dm[9]); dm[10] = fmaf(w, x2.z, dm[10]); dm[11] = fmaf(w, x2.w, dm[11]);
            dm[12] = fmaf(w, x3.x, dm[12]); dm[13] = fmaf(w, x3.y, dm[13]); dm[14] = fmaf(w, x3.z, dm[14]); dm[15] = fmaf(w, x3.w, dm[15]);
          }
        }
      }
      if (erow < rows_valid) {   // the dW kernel contracts Y_k^T with [Ds | Dm_1] straight from HBM
        float* dp = a.dpre + (row0 + erow) * p.Kdd + Hout + cbase;
        *reinterpret_cast<float4*>(dp) = make_float4(dm[0], dm[1], dm[2], dm[3]);
        *reinterpret_cast<float4*>(dp + 4) = make_float4(dm[4], dm[5], dm[6], dm[7]);
        if (two) {
          *reinterpret_cast<float4*>(dp + 8) = make_float4(dm[8], dm[9], dm[10], dm[11]);
          *reinterpret_cast<float4*>(dp + 12) = make_float4(dm[12], dm[13], dm[14], dm[15]);
        }
      }
#pragma unroll
      for (int part = 0; part < 2; ++part) {           // 8 columns at a time (cw == 8: one part)
        if (part * 8 < cw) {
          const int col = cbase + part * 8;
          float hi[8], lo[8];
          {
            const float4 x0 = *reinterpret_cast<const float4*>(Dsm + erow * DP + col);
            const float4 x1 = *reinterpret_cast<const float4*>(Dsm + erow * DP + col + 4);
            split_tf32(x0.x, hi[0], lo[0]); split_tf32(x0.y, hi[1], lo[1]); split_tf32(x0.z, hi[2], lo[2]); split_tf32(x0.w, hi[3], lo[3]);
            split_tf32(x1.x, hi[4], lo[4]); split_tf32(x1.y, hi[5], lo[5]); split_tf32(x1.z, hi[6], lo[6]); split_tf32(x1.w, hi[7], lo[7]);
          }
          tmem_st8(tA + (uint32_t)col, hi);
          tmem_st8(tA + 64u + (uint32_t)col, lo);
#pragma unroll
          for (int i = 0; i < 8; ++i) split_tf32(dm[part * 8 + i], hi[i], lo[i]);
          tmem_st8(tA + (uint32_t)(Hout + col), hi);
          tmem_st8(tA + 64u + (uint32_t)(Hout + col), lo);
        }
      }
      tmem_st_wait();
      STC_TRACE(12);
      fence_before_sync();
      STC_TRACE(13);
      __syncthreads();
      STC_TRACE(2);
      if (warp_u == 0 && elect_one_sync()) {
        fence_after_sync();
        const uint32_t a0 = tmem_base + (uint32_t)(2 * p.Npad);
        uint32_t acc = 0u;
        const int nks = p.Kdd >> 3;
        for (int ks = 0; ks < nks; ++ks) {
          const uint64_t bo = (uint64_t)((((uint32_t)(ks >> 2)) * 2u * atomB) >> 4) + (uint64_t)((ks & 3) * 2);
          const uint32_t ah = a0 + (uint32_t)(ks * 8), al = ah + 64u;
          mma_tf32_atmem(tmem_base, ah, dB_hi + bo, idesc2, acc);   // [main | cross] (+)= A_hi x [W_hi ; W_lo]
          mma_tf32_atmem(d_small, al, dB_hi + bo, idesc, 1u);       // cross += A_lo x W_hi
          acc = 1u;
        }
        STC_TRACE(8);
        STC_TRACE(10);
        mma_commit(mma_bar);
        STC_TRACE(9);
        STC_TRACE(11);
      }
      mma_pending = true;
    } else {
      // ---- 2. DD atoms + MMAs ----
      bool acc_small = false;
      for (int ja = 0; ja < p.KA; ++ja) {
        const int kk = ja * ATOM_K + q * 4;
        const int c = kk / Hout, o0 = kk - c * Hout;
        float4 vv[4];   // the atom's values are formed while the previous atom's MMAs still read the single A buffer
  #pragma unroll
        for (int i = 0; i < 4; ++i) {
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (kk < p.Kdd) {
            if (c == 0) {
              v = *reinterpret_cast<const float4*>(Dsm + (r0 + 32 * i) * DP + o0);
            } else {  // Dm_c[(node,c')][o] = sum_d Q_c[c'][d] Ds[(node,d)][o]
              const float* Qc = Qs + (size_t)(c - 1) * C * C + rcat[i] * C;
              const float* sp = Dsm + rnode[i] * C * DP + o0;
              for (int d = 0; d < C; ++d) {
                const float w = Qc[d];
                const float4 x = *reinterpret_cast<const float4*>(sp + d * DP);
                v.x = fmaf(w, x.x, v.x); v.y = fmaf(w, x.y, v.y); v.z = fmaf(w, x.z, v.z); v.w = fmaf(w, x.w, v.w);
              }
              if (r0 + 32 * i < rows_valid)   // the dW kernel contracts Y_k^T with [Ds | Dm_1 | ...] straight from HBM
                *reinterpret_cast<float4*>(a.dpre + (row0 + r0 + 32 * i) * p.Kdd + kk) = v;
            }
          }
          vv[i] = v;
        }
        if (mma_pending) {
          mbar_wait(mma_bar, mma_phase);
          mma_phase ^= 1u;
          mma_pending = false;
        }
  #pragma unroll
        for (int i = 0; i < 4; ++i) store_split4(A_hi, A_lo, aoff[i], vv[i]);
        if (ja == 0) STC_TRACE(12);
        fence_async_smem();
        if (ja == 0) STC_TRACE(13);
        __syncthreads();
        if (ja == 0) STC_TRACE(2);
        if (warp_u == 0 && elect_one_sync()) {   // one lane of converged warp 0: descriptors stay in uniform registers
          fence_after_sync();
          const int kleft = p.Kdd - ja * ATOM_K;
          const int ksteps = kleft >= ATOM_K ? 4 : (kleft + 7) / 8;
          const uint64_t bo = (uint64_t)(((uint32_t)ja * atomB) >> 4);
          const uint32_t d_main = tmem_base + (uint32_t)((ja / DX_APM) * p.Npad);
          uint32_t acc_main = (ja % DX_APM) != 0 ? 1u : 0u;
  #pragma unroll 4
          for (int ks = 0; ks < ksteps; ++ks) {   // small cross terms into their own accumulator, then the main product
            const uint64_t ko = (uint64_t)(ks * 2);
            mma_tf32(d_small, dA_lo + ko, dB_hi + bo + ko, idesc, acc_small ? 1u : 0u);
            mma_tf32(d_small, dA_hi + ko, dB_lo + bo + ko, idesc, 1u);
            mma_tf32(d_main, dA_hi + ko, dB_hi + bo + ko, idesc, acc_main);
            acc_main = 1u;
            acc_small = true;
          }
          if (ja == 0) STC_TRACE(8);
          if (ja == p.KA - 1) STC_TRACE(10);
          mma_commit(mma_bar);
          if (ja == 0) STC_TRACE(9);
          if (ja == p.KA - 1) STC_TRACE(11);
        }
        acc_small = true;
        mma_pending = true;
      }
    }
    STC_TRACE(3);
    // x-part adjoint this pass adds to (the other convolution's contribution): requested now, consumed in the epilogue --
    // the read-modify-write latency travels under the MMAs and the dQ pass instead of sitting at the end of every tile
    // (or, for term 1, the adjoint another cell folds into it)
    float4 xprev[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) xprev[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    if constexpr (FAST) {
      if (p.x_vec && erow < rows_valid) {
        const float* dbase_pf = a.accum_x ? (half == 0 ? a.dYx0 : a.dYx) : (half == 0 ? nullptr : a.dYx_add);
        if (dbase_pf != nullptr) {
          const float* src = dbase_pf + (row0 + erow) * Din;
#pragma unroll
          for (int i = 0; i < 4; ++i)
            if (4 * i < Din) xprev[i] = *reinterpret_cast<const float4*>(src + 4 * i);
        }
      }
    }
    // ---- 4 (overlaps the MMAs). dQ_c[c'][d] += sum_{node,o} P_c[(node,c')][o] * Ds[(node,d)][o] ----
    if (want_dQ) {
      mbar_wait(load_bar, load_phase);
      load_phase ^= 1u;
      const int npairs = (a.Kc - 1) * C * C;
      const int groups = CV_THREADS / npairs;      // node groups working on the same pair
      if (dq_fast) {
        if (dq_node < nodes_valid) {
          float4 pv[DQ_C], dv[DQ_C];
#pragma unroll
          for (int i = 0; i < DQ_C; ++i) {
            const int ci = i < C ? i : 0;
            pv[i] = *reinterpret_cast<const float4*>(Psm + (dq_node * C + ci) * p.PW + dq_oc);
            dv[i] = *reinterpret_cast<const float4*>(Dsm + (dq_node * C + ci) * DP + dq_oc);
          }
#pragma unroll
          for (int cp = 0; cp < DQ_C; ++cp)
#pragma unroll
            for (int d = 0; d < DQ_C; ++d) {
              float s = dq[cp * DQ_C + d];
              s = fmaf(pv[cp].x, dv[d].x, s); s = fmaf(pv[cp].y, dv[d].y, s);
              s = fmaf(pv[cp].z, dv[d].z, s); s = fmaf(pv[cp].w, dv[d].w, s);
              dq[cp * DQ_C + d] = s;
            }
        }
      } else if (groups >= 1) {
        const int pr = tid % npairs, grp = tid / npairs;
        if (grp < groups) {
          const int c = pr / (C * C), rem = pr - c * C * C, cp = rem / C, d = rem - cp * C;
          float s = 0.f;
          for (int node = grp; node < nodes_valid; node += groups) {
            const float* pp = Psm + (node * C + cp) * p.PW + c * Hout;
            const float* dd = Dsm + (node * C + d) * DP;
            for (int o = 0; o < Hout; o += 4) {
              const float4 x = *reinterpret_cast<const float4*>(pp + o);
              const float4 y = *reinterpret_cast<const float4*>(dd + o);
              s = fmaf(x.x, y.x, s); s = fmaf(x.y, y.y, s); s = fmaf(x.z, y.z, s); s = fmaf(x.w, y.w, s);
            }
          }
          atomicAdd(&dQacc[pr], s);
        }
      } else {  // more pairs than threads (large C): each thread walks several pairs
        for (int pr = tid; pr < npairs; pr += CV_THREADS) {
          const int c = pr / (C * C), rem = pr - c * C * C, cp = rem / C, d = rem - cp * C;
          float s = 0.f;
          for (int node = 0; node < nodes_valid; ++node) {
            const float* pp = Psm + (node * C + cp) * p.PW + c * Hout;
            const float* dd = Dsm + (node * C + d) * DP;
            for (int o = 0; o < Hout; ++o) s = fmaf(pp[o], dd[o], s);
          }
          dQacc[pr] += s;
        }
      }
    }
    // ---- 3. epilogue: dY_k tiles ----
    STC_TRACE(4);
    mbar_wait(mma_bar, mma_phase);
    mma_phase ^= 1u;
    mma_pending = false;
    fence_after_sync();
    STC_TRACE(5);
    const bool valid = erow < rows_valid;
    const long long gr = row0 + erow;
    if constexpr (FAST) {
      // thread (erow, half) owns spatial term k = half: columns [k*KBL, k*KBL + 16) are its h-part, the next Dp its x-part
      const int k = half;
      const uint32_t nb = (uint32_t)(k * p.KBL);
      {
        uint32_t sm[16], mn[16];
        tmem_ld16_async(tl + (uint32_t)p.Npad + nb, sm);
        tmem_ld16_async(tl + nb, mn);
        tmem_ld_wait();
        tmem_ld_pin16(sm); tmem_ld_pin16(mn);
        if (valid) {
          float v[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(sm[i]) + __uint_as_float(mn[i]);
          if (k == 0 && a.phase == 0) {
#pragma unroll
            for (int i = 0; i < 16; i += 4) {
              const float4 d = *reinterpret_cast<const float4*>(Dh + erow * 16 + i);
              v[i] += d.x; v[i + 1] += d.y; v[i + 2] += d.z; v[i + 3] += d.w;
            }
          }
          if (k == 1 && a.dYh_add != nullptr) {   // the folded adjoint of term 1 (pulled into L2 one tile ahead)
            const float4* ap = reinterpret_cast<const float4*>(a.dYh_add + gr * 16);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const float4 q = ap[i];
              v[4 * i] += q.x; v[4 * i + 1] += q.y; v[4 * i + 2] += q.z; v[4 * i + 3] += q.w;
            }
          }
          float* dst = (k == 0 ? a.dYh0 : a.dYh) + gr * 16;
#pragma unroll
          for (int i = 0; i < 16; i += 4) *reinterpret_cast<float4*>(dst + i) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
        }
      }
      float* dbase = (k == 0 ? a.dYx0 : a.dYx);
      {
        uint32_t sm[16], mn[16];
        if (p.Dp == 16) {
          tmem_ld16_async(tl + (uint32_t)p.Npad + nb + 16u, sm);
          tmem_ld16_async(tl + nb + 16u, mn);
          tmem_ld_wait();
          tmem_ld_pin16(sm); tmem_ld_pin16(mn);
        } else {   // Dp == 8
          uint32_t s8[8], m8[8];
          tmem_ld8_async(tl + (uint32_t)p.Npad + nb + 16u, s8);
          tmem_ld8_async(tl + nb + 16u, m8);
          tmem_ld_wait();
          tmem_ld_pin8(s8); tmem_ld_pin8(m8);
#pragma unroll
          for (int i = 0; i < 8; ++i) { sm[i] = s8[i]; mn[i] = m8[i]; sm[i + 8] = 0u; mn[i + 8] = 0u; }
        }
        if (valid && dbase != nullptr) {
          float* dst = dbase + gr * Din;
          if (p.x_vec) {   // Din % 4 == 0: 16-byte read-modify-writes, every read in flight before the first add
            float4 o[4];
#pragma unroll
            for (int i = 0; i < 4; ++i)
              o[i] = make_float4(__uint_as_float(sm[4 * i]) + __uint_as_float(mn[4 * i]),
                                 __uint_as_float(sm[4 * i + 1]) + __uint_as_float(mn[4 * i + 1]),
                                 __uint_as_float(sm[4 * i + 2]) + __uint_as_float(mn[4 * i + 2]),
                                 __uint_as_float(sm[4 * i + 3]) + __uint_as_float(mn[4 * i + 3]));
            if (a.accum_x || (k == 1 && a.dYx_add != nullptr)) {
#pragma unroll
              for (int i = 0; i < 4; ++i)
                if (4 * i < Din) { o[i].x += xprev[i].x; o[i].y += xprev[i].y; o[i].z += xprev[i].z; o[i].w += xprev[i].w; }
            }
#pragma unroll
            for (int i = 0; i < 4; ++i)
              if (4 * i < Din) *reinterpret_cast<float4*>(dst + 4 * i) = o[i];
          } else {
            const float* prior = a.accum_x ? dst : (k == 1 && a.dYx_add != nullptr) ? a.dYx_add + gr * Din : nullptr;
#pragma unroll
            for (int i = 0; i < 16; ++i)
              if (i < Din) {
                const float vi = __uint_as_float(sm[i]) + __uint_as_float(mn[i]);
                dst[i] = prior ? prior[i] + vi : vi;
              }
          }
        }
      }
    } else {
      int k = 0, kb = half * 8;                      // (spatial term, column within its [h | x] block) of chunk n0
      for (int n0 = half * 8; n0 < p.Npad; n0 += 16, kb += 16) {
        float v[8];
        if (p.nmain == 1) {                            // the common case: both accumulators in flight, one wait
          uint32_t t0[8], t1[8];
          tmem_ld8_async(tl + (uint32_t)(p.Npad + n0), t1);
          tmem_ld8_async(tl + (uint32_t)n0, t0);
          tmem_ld_wait();
          tmem_ld_pin8(t0); tmem_ld_pin8(t1);
#pragma unroll
          for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(t1[i]) + __uint_as_float(t0[i]);
        } else {
          float t[8];
          tmem_ld8(tl + (uint32_t)(p.nmain * p.Npad + n0), v);
          for (int m = 0; m < p.nmain; ++m) {
            tmem_ld8(tl + (uint32_t)(m * p.Npad + n0), t);
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] += t[i];
          }
        }
        while (kb >= p.KBL) { kb -= p.KBL; ++k; }      // KBL % 8 == 0: a chunk never straddles terms or parts
        if (!valid || n0 >= p.N1) continue;
        if (kb < h) {
          float* dst = (k == 0 ? a.dYh0 : a.dYh + (size_t)(k - 1) * R * h) + gr * h + kb;
          if (k == 0 && a.phase == 0) {
            const float* dp = Dh + erow * h + kb;
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] += dp[i];
          }
          if (k >= 1 && a.dYh_add != nullptr) {
            const float4* ap = reinterpret_cast<const float4*>(a.dYh_add + (size_t)(k - 1) * R * h + gr * h + kb);
            const float4 p0 = ap[0], p1 = ap[1];
            v[0] += p0.x; v[1] += p0.y; v[2] += p0.z; v[3] += p0.w;
            v[4] += p1.x; v[5] += p1.y; v[6] += p1.z; v[7] += p1.w;
          }
          reinterpret_cast<float4*>(dst)[0] = make_float4(v[0], v[1], v[2], v[3]);
          reinterpret_cast<float4*>(dst)[1] = make_float4(v[4], v[5], v[6], v[7]);
        } else {
          const int xi = kb - h;
          float* dbase = (k == 0 ? a.dYx0 : a.dYx + (size_t)(k - 1) * R * Din);
          if (dbase == nullptr) continue;
          float* dst = dbase + gr * Din + xi;
          const float* prior = a.accum_x ? dst
                               : (k >= 1 && a.dYx_add != nullptr) ? a.dYx_add + (size_t)(k - 1) * R * Din + gr * Din + xi
                                                                   : nullptr;
          if (p.x_vec && xi + 8 <= Din) {   // both 16-byte halves in flight at once (the accumulate is a read-modify-write)
            float4 o0 = make_float4(v[0], v[1], v[2], v[3]), o1 = make_float4(v[4], v[5], v[6], v[7]);
            if (prior != nullptr) {
              const float4 p0 = reinterpret_cast<const float4*>(prior)[0], p1 = reinterpret_cast<const float4*>(prior)[1];
              o0.x += p0.x; o0.y += p0.y; o0.z += p0.z; o0.w += p0.w;
              o1.x += p1.x; o1.y += p1.y; o1.z += p1.z; o1.w += p1.w;
            }
            reinterpret_cast<float4*>(dst)[0] = o0;
            reinterpret_cast<float4*>(dst)[1] = o1;
          } else {
#pragma unroll
            for (int i = 0; i < 8; ++i)
              if (xi + i < Din) dst[i] = prior ? prior[i] + v[i] : v[i];
          }
        }
      }
    }
    STC_TRACE(6);
    fence_before_sync();
    fence_async_smem();   // this tile's reads of Psm precede the next tile's bulk copy into it
    __syncthreads();  // Dsm / Dh / Psm are rewritten by the next tile's prologue
    STC_TRACE(7);
    ++trace_it;
  }
  if (a.dbias && !db_fast && tid < db_groups * Hout) atomicAdd(&a.dbias[db_col], db_acc);
  __syncthreads();   // every tile is done: Dsm is free and serves as the reduction scratch
  // End-of-kernel reductions.  Shared-memory float atomics are compare-and-swap loops: with every thread of the CTA
  // adding into the same few addresses at once (the first version) the loops serialise -- ~100 us per launch, at any batch
  // size (profiles/r3b_launches_b32.txt: 110 us per dx launch at B = 32 against 10 us for the forward).  Lanes that
  // share an address are therefore summed with warp shuffles first; one lane per warp and address touches memory.
  if (db_fast) {
    for (int i = tid; i < Hout; i += CV_THREADS) Dsm[i] = 0.f;
    __syncthreads();
    const int cprw = h >> 2;                         // lanes l and l + cprw (mod 32) hold the same column chunk
    float v[8] = {dbs0.x, dbs0.y, dbs0.z, dbs0.w, dbs1.x, dbs1.y, dbs1.z, dbs1.w};
    for (int off = cprw; off < 32; off <<= 1) {
#pragma unroll
      for (int i = 0; i < 8; ++i) v[i] += __shfl_xor_sync(0xffffffffu, v[i], off);
    }
    if (lane < cprw || cprw >= 32) {
      const int j = (tid % cprw) << 2;
      atomicAdd(&Dsm[j + 0], v[0]); atomicAdd(&Dsm[j + 1], v[1]); atomicAdd(&Dsm[j + 2], v[2]); atomicAdd(&Dsm[j + 3], v[3]);
      if (a.phase == 0) {
        atomicAdd(&Dsm[h + j + 0], v[4]); atomicAdd(&Dsm[h + j + 1], v[5]);
        atomicAdd(&Dsm[h + j + 2], v[6]); atomicAdd(&Dsm[h + j + 3], v[7]);
      }
    }
    __syncthreads();
    for (int i = tid; i < Hout; i += CV_THREADS) atomicAdd(&a.dbias[i], Dsm[i]);
  }
  if (dq_fast) {   // CTA-uniform: every lane takes part in the shuffles (threads without a node slot hold zeros)
#pragma unroll
    for (int cp = 0; cp < DQ_C; ++cp)
#pragma unroll
      for (int d = 0; d < DQ_C; ++d) {
        float s = dq[cp * DQ_C + d];
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
        if (lane == 0 && cp < C && d < C) atomicAdd(&dQacc[cp * C + d], s);
      }
  }
  __syncthreads();
  if (want_dQ)
    for (int i = tid; i < (a.Kc - 1) * C * C; i += CV_THREADS) atomicAdd(&a.dQ[C * C + i], dQacc[i]);
  if (warp == 0) tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
}

static bool aligned16b(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

int try_launch_conv_bwd_dx_tc(const ConvArgs& a, cudaStream_t st, bool* handled) {
  *handled = false;
  if (!conv_tc_eligible(a)) return STC_OK;
  if (!aligned16b(a.dHn) || !aligned16b(a.u) || !aligned16b(a.c) || !aligned16b(a.Hprev) || !aligned16b(a.dpre) ||
      !aligned16b(a.dYh0) || !aligned16b(a.dYh) || !aligned16b(a.dYh_add) || !aligned16b(a.Psave) ||
      (a.phase == 0 && (!aligned16b(a.r) || !aligned16b(a.drH)))) {
    set_error("tcgen05 backward needs 16-byte aligned gradient / workspace tensors");
    return STC_ERR_BAD_ARG;
  }
  const int L = a.Din + a.h;
  TcDxPlan p;
  p.npt = 128 / a.C;
  p.Dp = (a.Din + 7) & ~7;
  p.KBL = a.h + p.Dp;
  p.N1 = a.Ks * p.KBL;
  p.Npad = (p.N1 + 15) & ~15;
  p.Kdd = a.Kc * a.Hout;
  p.KA = (p.Kdd + ATOM_K - 1) / ATOM_K;
  p.nmain = (p.KA + DX_APM - 1) / DX_APM;
  p.tmem_cols = 32;
  while (p.tmem_cols < (p.nmain + 1) * p.Npad) p.tmem_cols *= 2;
  p.DP = a.Hout + 4;
  p.PW = (a.Kc - 1) * a.Hout;
  p.x_vec = (a.Din % 4 == 0) && aligned16b(a.dYx0) && aligned16b(a.dYx) && aligned16b(a.dYx_add);
  const long long total_nodes = (long long)a.B * a.N;
  p.ntiles = ceil_div(total_nodes, p.npt);
  const size_t atomB = (size_t)p.Npad * ATOM_ROW_BYTES;
  size_t o = 0;
  p.off_a = (uint32_t)o; o += 2 * 128 * ATOM_ROW_BYTES;
  p.off_b = (uint32_t)o; o += 2 * (size_t)p.KA * atomB;
  p.off_ds = (uint32_t)o; o += (size_t)128 * p.DP * sizeof(float);
  p.off_dh = (uint32_t)o; o += (size_t)128 * a.h * sizeof(float);
  p.off_ps = (uint32_t)o; o += round_up((size_t)128 * p.PW * sizeof(float), 16);
  p.off_q = (uint32_t)o; o += round_up((size_t)(a.Kc > 1 ? a.Kc - 1 : 0) * a.C * a.C * sizeof(float), 16);
  p.off_acc = (uint32_t)o; o += round_up((size_t)(a.Kc > 1 ? a.Kc - 1 : 0) * a.C * a.C * sizeof(float), 16);
  p.off_bar = (uint32_t)o; o += 32;
  p.smem_bytes = (uint32_t)o;
  if (p.smem_bytes > 200 * 1024) {
    set_error("tcgen05 backward tile does not fit (%u B) although the forward ran on the tensor-core path", p.smem_bytes);
    return STC_ERR_UNSUPPORTED;
  }
  const bool fast = a.Ks == 2 && a.h == 16 && a.Din <= 16 && p.nmain == 1 && !(a.opt & OPT_GENERIC_EPILOGUE);
  const bool at = fast && a.Kc == 2 && p.Kdd <= 64 && (a.Hout == 16 || a.Hout == 32) && !(a.opt & OPT_SMEM_A);
  auto kern = at ? tc_conv_bwd_dx_kernel<true, true>
                 : (fast ? tc_conv_bwd_dx_kernel<true, false> : tc_conv_bwd_dx_kernel<false, false>);
  if (at) p.tmem_cols = 256;   // 2 Npad accumulator columns + 64 A_hi + 64 A_lo
  STC_TRY(set_smem(kern, p.smem_bytes));
  int ctas_per_sm = (int)((228 * 1024) / (p.smem_bytes + 1024));
  if (ctas_per_sm < 1) ctas_per_sm = 1;
  if (ctas_per_sm > 2) ctas_per_sm = 2;
  if (ctas_per_sm * p.tmem_cols > 512) ctas_per_sm = 512 / p.tmem_cols;
  int grid = device_sm_count() * ctas_per_sm;
  if (grid > p.ntiles) grid = p.ntiles;
  // compulsory traffic per row: candidate reads dH',u,c (3h), gates reads dH',u,c,H,r,d(rH) (6h); both write dpre
  // (Hout) and the Ks adjoint terms (Ks*L; the gates pass re-reads the x-part it accumulates into) and, for dGc,
  // read the saved partial outputs ((Kc-1)*Hout).
  const double R = (double)total_nodes * a.C;
  ScopedKernelTimer _t(KK_TC_CONV_BWD_DX, st,
                       4.0 * R * ((a.phase == 0 ? 6 * a.h + a.Ks * a.Din : 3 * a.h) + a.Hout + a.Ks * L +
                                  ((a.dQ && a.Kc > 1) ? p.PW : 0)) + 4.0 * a.Ks * a.Kc * L * a.Hout);
  kern<<<grid, CV_THREADS, p.smem_bytes, st>>>(a, p);
  STC_LAUNCH_OK("tc_conv_bwd_dx_kernel");
  *handled = true;
  return STC_OK;
}

}  // namespace stc
