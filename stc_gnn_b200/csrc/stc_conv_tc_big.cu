// tcgen05 / TMEM forward gate / candidate convolution for WIDE hidden states (h = 32 ... 128, e.g. F = 64 of the
// synthetic grid and kNN configurations): the reference's 'bmdk,kh->bmdh' (/root/reference/framework/STC_GNN.py:42)
// with K = Ks * (h + Din) up to 512 and N = Kc * Hout up to 256 -- the one shape where the contraction is a real GEMM.
//
// Differences from the SF-class kernels (stc_conv_tc.cu):
//   * the split weights (hi | lo) do not fit in shared memory (512 KB at F = 64): a preparation kernel writes them
//     once per launch as ready-to-use K-major SW128 atoms into a scratch image, and the main kernel streams one
//     32-wide K chunk at a time through a 3-stage TMA (1-D bulk copy) ring;
//   * the data rows are the TMEM A operand (tcgen05.st), double-buffered per K chunk;
//   * N is processed per categorical block (c = 1 first, then c = 0): accumulators main0 | main1 | cross terms
//     = 3 Hout <= 384 TMEM columns, A buffers in columns [384, 512); chunks alternate between the two main
//     accumulators so that no chain exceeds K/2 (accumulate-truncation, profiles/r1_tc_precision.txt);
//   * the categorical mix is applied to the GEMM output as in the SF kernels: P_1 goes to shared memory, the c = 0
//     epilogue adds T_1(Gc)^T-mix(P_1), bias, activation, sigmoid / tanh and the GRU blend (STC_GNN.py:44-46, 71-78).
// Forward only: backward for these shapes runs on the general path (stc_conv.cu), which saves nothing extra.
#include "stc_conv_common.cuh"
#include "stc_tc.cuh"

#include <stdlib.h>
#include <string.h>

namespace stc {

using namespace tc;

constexpr int BG_STAGES = 3;
constexpr int BG_THREADS = 512;   // 16 warps: four threads per tile row (one per 8 K-values of a chunk / per quarter of the output columns)
constexpr int BG_FWD_THREADS = BG_THREADS + 32;   // forward: + one warp that only issues MMAs and refills the weight ring
constexpr int BG_ACOL = 384;   // first TMEM column of the A buffers: buffer b = [hi 32 | lo 32] at BG_ACOL + 64 b

struct BigPlan {
  int npt, Dp, KBL;
  int nchk;       // 32-wide K chunks per spatial term
  int nch;        // chunks per categorical block = Ks * nchk
  int ntiles;
  int PS;         // row stride (floats) of the P_1 exchange tile
  int x_vec;
  uint32_t stage_bytes;   // one weight chunk: [hi: Hout rows x 128 B | lo: Hout rows x 128 B]
  uint32_t off_b, off_pm, off_q, off_bias, off_bar, smem_bytes;
  int land;               // depth of the per-thread cp.async landing ring for the row chunks (0: register double buffer)
  uint32_t off_land;
};

__device__ __forceinline__ void bg_cp_async16(uint32_t smem_dst, const void* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_dst), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void bg_cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bg_cp_async_wait_depth(int pending) {   // wait until at most `pending` groups are in flight
  switch (pending) {
    case 0: asm volatile("cp.async.wait_group 0;" ::: "memory"); break;
    case 1: asm volatile("cp.async.wait_group 1;" ::: "memory"); break;
    case 2: asm volatile("cp.async.wait_group 2;" ::: "memory"); break;
    default: asm volatile("cp.async.wait_group 3;" ::: "memory"); break;
  }
}

// img[(cb, ch)][hi | lo][o][kb]  <-  W[((k*Kc + cb)*L + l(kb))*Hout + o],  k = ch / nchk, kb = 32 (ch % nchk) + ...
__global__ void tc_big_prep_kernel(const float* __restrict__ W, uint8_t* __restrict__ img, int Din, int h, int Ks, int Kc,
                                   int Hout, int KBL, int nchk) {
  const int L = Din + h, nch = Ks * nchk;
  const long long total = (long long)Kc * nch * Hout * 8;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int q = (int)(idx & 7);
    long long r = idx >> 3;
    const int o = (int)(r % Hout);
    r /= Hout;
    const int ch = (int)(r % nch), cb = (int)(r / nch);
    const int k = ch / nchk, j = ch - k * nchk;
    float v[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int kb = 32 * j + 4 * q + i;
      const int l = kb >= KBL ? -1 : (kb < h ? Din + kb : (kb - h < Din ? kb - h : -1));
      v[i] = l >= 0 ? W[((size_t)(k * Kc + cb) * L + l) * Hout + o] : 0.f;
    }
    uint8_t* base = img + (size_t)(cb * nch + ch) * 2 * Hout * ATOM_ROW_BYTES;
    store_split4(base, base + (size_t)Hout * ATOM_ROW_BYTES, atom_chunk_offset(o, q), make_float4(v[0], v[1], v[2], v[3]));
  }
}

// Round 2: the MMA issue moved out of the producers' loop.  Before, every chunk ended in a block barrier behind warp 0,
// which both staged its rows AND issued the chunk's 12 MMAs (tensor-execution-paced, ~800 cycles): a chunk cost
// staging + issue in series (ncu: 20 % barrier stalls, tensor pipe 13-21 %).  Now warp 16 only waits for "A staged"
// (a_full, one arrive per producer warp) and "weights landed" (b_full), issues, commits, and refills the weight ring;
// the 16 producer warps run ahead by the two TMEM A buffers and meet the issuer only through mbarriers (a_free,
// acc_full, acc_empty).  Producer-only block syncs use named barrier 1.
__device__ __forceinline__ void bg_producer_sync() { asm volatile("bar.sync 1, %0;" ::"n"(BG_THREADS) : "memory"); }

__global__ void __launch_bounds__(BG_FWD_THREADS, 1)
tc_conv_fwd_big_kernel(const ConvArgs a, const BigPlan p, const uint8_t* __restrict__ img) {
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((smem_u32(smem) & 1023u) != 0u) __trap();
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int C = a.C, h = a.h, Din = a.Din, Hout = a.Hout;
  uint8_t* Bring = smem + p.off_b;
  float* Pm = reinterpret_cast<float*>(smem + p.off_pm);        // [128 + C][PS]  P_1 tile (rows past 128 stay zero)
  float* Qs = reinterpret_cast<float*>(smem + p.off_q);         // [C][C] = T_1(Gc)
  float* bias_s = reinterpret_cast<float*>(smem + p.off_bias);
  uint64_t* b_full = reinterpret_cast<uint64_t*>(smem + p.off_bar);
  uint64_t* b_free = b_full + BG_STAGES;
  uint64_t* a_free = b_free + BG_STAGES;
  uint64_t* acc_full = a_free + 2;
  uint64_t* a_full = acc_full + 1;                               // [2] producers -> issuer: A buffer staged in TMEM
  uint64_t* acc_empty = a_full + 2;                              // producers -> issuer: the block's epilogue has read the accumulators
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 1);

  if (tid == 0) {
    for (int i = 0; i < BG_STAGES; ++i) {
      mbar_init(&b_full[i], 1);
      mbar_init(&b_free[i], 1);
    }
    mbar_init(&a_free[0], 1);
    mbar_init(&a_free[1], 1);
    mbar_init(acc_full, 1);
    mbar_init(&a_full[0], BG_THREADS / 32);
    mbar_init(&a_full[1], BG_THREADS / 32);
    mbar_init(acc_empty, BG_THREADS / 32);
    mbar_fence_init();
  }
  if (warp == 0) tmem_alloc(tmem_slot, 512u);
  for (int i = tid; i < C * C; i += BG_FWD_THREADS) Qs[i] = a.Q[C * C + i];
  for (int i = tid; i < Hout; i += BG_FWD_THREADS) bias_s[i] = a.bias ? a.bias[i] : 0.f;
  for (int i = tid; i < (128 + C) * p.PS; i += BG_FWD_THREADS) Pm[i] = 0.f;
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const int warp_u = uniform_warp_index();
  const uint32_t tmem_base = uniform_u32(*tmem_slot);
  const uint32_t idesc = make_idesc_tf32(128, Hout);
  const uint32_t d_small = tmem_base + (uint32_t)(2 * Hout);
  const long long total_nodes = (long long)a.B * a.N;
  const long long R = total_nodes * C;

  const int sp = warp & 3, qtr = warp >> 2;            // TMEM lane quarter / which of the row's four threads
  const int erow = sp * 32 + lane;                     // accumulator lane = tile row
  const int enode = erow / C, ecat = erow - enode * C;
  const uint32_t tl = tmem_base + ((uint32_t)(sp * 32) << 16);
  const bool xvec = p.x_vec != 0;

  const int my_tiles = (p.ntiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  const uint32_t total_chunks = (uint32_t)my_tiles * 2u * (uint32_t)p.nch;
  auto img_of = [&](uint32_t g) {                      // chunk g of this CTA -> its weight image (periodic in the tile)
    const uint32_t w = g % (2u * (uint32_t)p.nch);
    const uint32_t cbi = w / (uint32_t)p.nch, ch = w - cbi * (uint32_t)p.nch;
    return img + (size_t)((1u - cbi) * (uint32_t)p.nch + ch) * p.stage_bytes;   // c = 1 first, then c = 0
  };
  if (warp_u == BG_THREADS / 32) {
    // =============================== issuer: MMAs + weight ring ===============================
    if (elect_one_sync()) {
      for (uint32_t g = 0; g < (uint32_t)(BG_STAGES - 1) && g < total_chunks; ++g) {   // ring prologue
        mbar_arrive_expect_tx(&b_full[g], p.stage_bytes);
        bulk_g2s(Bring + (size_t)g * p.stage_bytes, img_of(g), p.stage_bytes, &b_full[g]);
      }
      uint32_t g = 0, blocks = 0;
      for (int t_ = 0; t_ < my_tiles; ++t_) {
        for (int cbi = 0; cbi < 2; ++cbi, ++blocks) {
          for (int ch = 0; ch < p.nch; ++ch, ++g) {
            const int buf = (int)(g & 1u), st = (int)(g % (uint32_t)BG_STAGES);
            if (ch == 0 && blocks > 0) mbar_wait(acc_empty, (blocks - 1u) & 1u);   // previous block's epilogue is done
            mbar_wait(&a_full[buf], (g >> 1) & 1u);
            mbar_wait(&b_full[st], (g / (uint32_t)BG_STAGES) & 1u);
            fence_after_sync();
            const int j = ch % p.nchk;
            const int kleft = p.KBL - 32 * j;
            const int ksteps = kleft >= 32 ? 4 : (kleft + 7) / 8;
            const uint32_t a_hi0 = tmem_base + (uint32_t)(BG_ACOL + 64 * buf);
            const uint64_t dBh = make_smem_desc_sw128(smem_u32(Bring + (size_t)st * p.stage_bytes));
            const uint64_t dBl = dBh + (uint64_t)(((uint32_t)Hout * ATOM_ROW_BYTES) >> 4);
            // consecutive MMAs never touch the same accumulator twice in a row: the main product alternates between the
            // two main accumulators per K-step and sits between the two cross-term products
            for (int ks = 0; ks < ksteps; ++ks) {
              const uint64_t ko = (uint64_t)(ks * 2);
              const uint32_t ah = a_hi0 + (uint32_t)(ks * 8), al = ah + 32u;
              const uint32_t d_main = tmem_base + (uint32_t)((ks & 1) * Hout);
              mma_tf32_atmem(d_small, al, dBh + ko, idesc, (ch > 0 || ks > 0) ? 1u : 0u);
              mma_tf32_atmem(d_main, ah, dBh + ko, idesc, (ch > 0 || ks >= 2) ? 1u : 0u);
              mma_tf32_atmem(d_small, ah, dBl + ko, idesc, 1u);
            }
            mma_commit(&a_free[buf]);                     // A buffer and weight stage are free once these MMAs have read them
            mma_commit(&b_free[st]);
            if (ch == p.nch - 1) mma_commit(acc_full);    // ... and the block's accumulators are complete
            const uint32_t t = g + (uint32_t)(BG_STAGES - 1);   // refill the ring BG_STAGES - 1 chunks ahead
            if (t < total_chunks) {
              const uint32_t ts = t % (uint32_t)BG_STAGES, tu = t / (uint32_t)BG_STAGES;
              if (tu >= 1u) mbar_wait(&b_free[ts], (tu - 1u) & 1u);
              mbar_arrive_expect_tx(&b_full[ts], p.stage_bytes);
              bulk_g2s(Bring + (size_t)ts * p.stage_bytes, img_of(t), p.stage_bytes, &b_full[ts]);
            }
          }
        }
      }
    }
    __syncwarp();
  } else {
  // =============================== producers + epilogue (16 warps) ===============================
  uint32_t g = 0;                                      // running chunk counter of this CTA
  uint32_t acc_phase = 0;
  // ---- row chunks, asynchronous form: every thread owns one 32-byte slot per ring stage; its 8 K-values of a chunk
  //      travel global -> shared with cp.async, `land - 1` chunks ahead and ACROSS block / tile boundaries (the register
  //      double buffer restarts at every categorical block and exposes one round trip per chunk, 30 % of the kernel's
  //      stall samples in profiles/r3o_config3_wide_ncu.txt).  Only the owner touches a slot: no barriers.
  const int LD = p.land;
  const uint32_t land0 = smem_u32(smem + p.off_land) + (uint32_t)tid * 32u;
  int c_tile = blockIdx.x, c_cbi = 0, c_ch = 0;        // the chunk the next copy is for
  uint32_t c_seq = 0;
  auto issue_copy = [&]() {
    if (c_tile < p.ntiles) {
      const long long cg0 = (long long)c_tile * p.npt;
      const int cnodes = (int)min((long long)p.npt, total_nodes - cg0);
      const bool cvalid = erow < cnodes * C;
      const long long cgr = cg0 * C + erow;
      const uint32_t dst = land0 + (c_seq % (uint32_t)LD) * (uint32_t)(BG_THREADS * 32);
      const int k = c_ch / p.nchk, j = c_ch - k * p.nchk;
      const int kb0 = 32 * j + 8 * qtr;
      bool z0 = true, z1 = true;
      if (cvalid) {
        if (kb0 < h) {
          const float* hs = (k == 0 ? a.h0 : a.yh + (size_t)(k - 1) * R * h) + cgr * h + kb0;
          bg_cp_async16(dst, hs);
          bg_cp_async16(dst + 16u, hs + 4);
          z0 = z1 = false;
        } else {
          const int xi = kb0 - h;
          const float* xs;
          if (k == 0) {
            const long long gn = cg0 + enode;
            const long long b = gn / a.N;
            xs = a.x0 + b * a.x0_bs + ((gn - b * a.N) * C + ecat) * Din;
          } else {
            xs = a.yx + (size_t)(k - 1) * R * Din + cgr * Din;
          }
          if (xvec) {
            if (xi < Din) { bg_cp_async16(dst, xs + xi); z0 = false; }
            if (xi + 4 < Din) { bg_cp_async16(dst + 16u, xs + xi + 4); z1 = false; }
          } else {   // unaligned x-part (layer-0 cells, Din = 1): plain loads, it is tiny
            float e[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) e[i] = (xi + i < Din) ? xs[xi + i] : 0.f;
            asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(dst), "f"(e[0]), "f"(e[1]), "f"(e[2]), "f"(e[3]) : "memory");
            asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(dst + 16u), "f"(e[4]), "f"(e[5]), "f"(e[6]), "f"(e[7]) : "memory");
            z0 = z1 = false;
          }
        }
      }
      if (z0) asm volatile("st.shared.v4.f32 [%0], {%1, %1, %1, %1};" ::"r"(dst), "f"(0.f) : "memory");
      if (z1) asm volatile("st.shared.v4.f32 [%0], {%1, %1, %1, %1};" ::"r"(dst + 16u), "f"(0.f) : "memory");
      if (++c_ch == p.nch) {
        c_ch = 0;
        if (++c_cbi == 2) {
          c_cbi = 0;
          c_tile += gridDim.x;
        }
      }
    }
    ++c_seq;
    bg_cp_async_commit();
  };
  if (LD > 0)
    for (int i = 0; i < LD - 1; ++i) issue_copy();
  for (int tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x) {
    const long long g0 = (long long)tile * p.npt;
    const int nodes_valid = (int)min((long long)p.npt, total_nodes - g0);
    const int rows_valid = nodes_valid * C;
    const bool valid = erow < rows_valid;
    const long long gr = g0 * C + erow;
    // x-part source of my row for spatial term 0 (Xt carries a batch stride)
    const float* xs0 = a.x0;
    if (valid) {
      const long long gn = g0 + enode;
      const long long b = gn / a.N;
      xs0 = a.x0 + b * a.x0_bs + ((gn - b * a.N) * C + ecat) * Din;
    }
    // my 8 K-values of chunk ch: K range [32 j + 8 qtr, +8) of spatial term k
    auto load_chunk = [&](int ch, float4 (&v)[2]) {
      v[0] = v[1] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (!valid) return;
      const int k = ch / p.nchk, j = ch - k * p.nchk;
      const int kb0 = 32 * j + 8 * qtr;
      if (kb0 < h) {        // h % 16 == 0: the run lies entirely in the h-part
        const float* hs = (k == 0 ? a.h0 : a.yh + (size_t)(k - 1) * R * h) + gr * h + kb0;
        v[0] = *reinterpret_cast<const float4*>(hs);
        v[1] = *reinterpret_cast<const float4*>(hs + 4);
      } else {
        const int xi = kb0 - h;
        const float* xs = (k == 0 ? xs0 : a.yx + (size_t)(k - 1) * R * Din + gr * Din);
        if (xvec) {
          if (xi < Din) v[0] = *reinterpret_cast<const float4*>(xs + xi);
          if (xi + 4 < Din) v[1] = *reinterpret_cast<const float4*>(xs + xi + 4);
        } else {
          float e[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) e[i] = (xi + i < Din) ? xs[xi + i] : 0.f;
          v[0] = make_float4(e[0], e[1], e[2], e[3]);
          v[1] = make_float4(e[4], e[5], e[6], e[7]);
        }
      }
    };

    for (int cbi = 0; cbi < 2; ++cbi) {                // categorical block c = 1, then c = 0
      const int cb = 1 - cbi;
      float4 cur[2], nxt[2];
      nxt[0] = nxt[1] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (LD == 0) load_chunk(0, cur);
      for (int ch = 0; ch < p.nch; ++ch, ++g) {
        if (LD > 0) {
          issue_copy();                                  // chunk g + LD - 1 (a group is committed even past the end)
          bg_cp_async_wait_depth(LD - 1);                // my piece of chunk g has landed
          const uint32_t src = land0 + (g % (uint32_t)LD) * (uint32_t)(BG_THREADS * 32);
          asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(cur[0].x), "=f"(cur[0].y), "=f"(cur[0].z), "=f"(cur[0].w) : "r"(src) : "memory");
          asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(cur[1].x), "=f"(cur[1].y), "=f"(cur[1].z), "=f"(cur[1].w) : "r"(src + 16u) : "memory");
        } else if (ch + 1 < p.nch) {
          load_chunk(ch + 1, nxt);   // register double buffer: next chunk's loads travel under this chunk's work
        }
        const int buf = (int)(g & 1u);
        const uint32_t ua = g >> 1;
        if (ua >= 1u) {                                // the MMAs that read this A buffer two chunks ago are done
          mbar_wait(&a_free[buf], (ua - 1u) & 1u);
          fence_after_sync();
        }
        const uint32_t tA = tl + (uint32_t)(BG_ACOL + 64 * buf + 8 * qtr);
        {                                              // my 8 columns: hi, and lo 32 columns further
          float hi[8], lo[8];
          split_tf32(cur[0].x, hi[0], lo[0]); split_tf32(cur[0].y, hi[1], lo[1]);
          split_tf32(cur[0].z, hi[2], lo[2]); split_tf32(cur[0].w, hi[3], lo[3]);
          split_tf32(cur[1].x, hi[4], lo[4]); split_tf32(cur[1].y, hi[5], lo[5]);
          split_tf32(cur[1].z, hi[6], lo[6]); split_tf32(cur[1].w, hi[7], lo[7]);
          tmem_st8(tA, hi);
          tmem_st8(tA + 32u, lo);
        }
        tmem_st_wait();
        fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(&a_full[buf]);       // one arrive per producer warp: the issuer takes it from here
        if (LD == 0) {
          cur[0] = nxt[0];
          cur[1] = nxt[1];
        }
      }
      // ---- epilogue of this categorical block ----
      mbar_wait(acc_full, acc_phase);
      acc_phase ^= 1u;
      fence_after_sync();
      for (int c0 = 8 * qtr; c0 < Hout; c0 += 32) {   // this thread's 8-column groups: qtr, qtr + 4, ...
        float v[8];
        {
          uint32_t t0[8], t1[8], t2[8];
          tmem_ld8_async(tl + (uint32_t)(2 * Hout + c0), t2);
          tmem_ld8_async(tl + (uint32_t)c0, t0);
          tmem_ld8_async(tl + (uint32_t)(Hout + c0), t1);
          tmem_ld_wait();
          tmem_ld_pin8(t0); tmem_ld_pin8(t1); tmem_ld_pin8(t2);
#pragma unroll
          for (int i = 0; i < 8; ++i) v[i] = (__uint_as_float(t2[i]) + __uint_as_float(t0[i])) + __uint_as_float(t1[i]);
        }
        if (cb == 1) {                                   // P_1: parked in shared memory for the mix
          *reinterpret_cast<float4*>(Pm + erow * p.PS + c0) = make_float4(v[0], v[1], v[2], v[3]);
          *reinterpret_cast<float4*>(Pm + erow * p.PS + c0 + 4) = make_float4(v[4], v[5], v[6], v[7]);
          if (a.Psave && valid) {                        // the wide-state dx kernel forms dGc from these partials
            float4* ps = reinterpret_cast<float4*>(a.Psave + gr * (long long)Hout + c0);
            ps[0] = make_float4(v[0], v[1], v[2], v[3]);
            ps[1] = make_float4(v[4], v[5], v[6], v[7]);
          }
          continue;
        }
        {                                                // P_0 + T_1(Gc)^T-mix of P_1 over the node's categories
          const float* pp = Pm + (enode * C) * p.PS + c0;
          for (int cp = 0; cp < C; ++cp) {
            const float w = Qs[cp * C + ecat];
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
            const float4 h0 = *reinterpret_cast<const float4*>(a.Hprev + o);
            const float4 h1 = *reinterpret_cast<const float4*>(a.Hprev + o + 4);
            float4* dr = reinterpret_cast<float4*>(a.r + o);
            dr[0] = make_float4(v[0], v[1], v[2], v[3]);
            dr[1] = make_float4(v[4], v[5], v[6], v[7]);
            float4* drh = reinterpret_cast<float4*>(a.rH + o);
            drh[0] = make_float4(v[0] * h0.x, v[1] * h0.y, v[2] * h0.z, v[3] * h0.w);
            drh[1] = make_float4(v[4] * h1.x, v[5] * h1.y, v[6] * h1.z, v[7] * h1.w);
          }
        } else {
          const long long o = gr * h + c0;
          const float4 u0 = *reinterpret_cast<const float4*>(a.u + o), u1 = *reinterpret_cast<const float4*>(a.u + o + 4);
          const float4 p0 = *reinterpret_cast<const float4*>(a.Hprev + o), p1 = *reinterpret_cast<const float4*>(a.Hprev + o + 4);
          const float uu[8] = {u0.x, u0.y, u0.z, u0.w, u1.x, u1.y, u1.z, u1.w};
          const float hp[8] = {p0.x, p0.y, p0.z, p0.w, p1.x, p1.y, p1.z, p1.w};
          float cc[8], hn[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            cc[i] = tanhf_fast(v[i]);
            hn[i] = fmaf(uu[i], cc[i] - hp[i], hp[i]);
          }
          float4* dc = reinterpret_cast<float4*>(a.c + o);
          dc[0] = make_float4(cc[0], cc[1], cc[2], cc[3]);
          dc[1] = make_float4(cc[4], cc[5], cc[6], cc[7]);
          float4* dh = reinterpret_cast<float4*>(a.Hnew + o);
          dh[0] = make_float4(hn[0], hn[1], hn[2], hn[3]);
          dh[1] = make_float4(hn[4], hn[5], hn[6], hn[7]);
        }
      }
      fence_before_sync();   // accumulator reads precede the next block's overwriting MMAs; P_1 is complete / consumed
      __syncwarp();
      if (lane == 0) mbar_arrive(acc_empty);
      bg_producer_sync();    // the P_1 tile is rewritten by the next block's epilogue
    }
  }
  if (LD > 0) bg_cp_async_wait_depth(0);
  }   // producers
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, 512u);
}

static bool aligned16g(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// shape-only test (also sizes the weight image inside the `saved` buffer, so it must not depend on pointers)
bool conv_big_shape_ok(int C, int Din, int h, int Ks, int Kc, int Hout) {
  const char* e = getenv("STC_DISABLE_TC");
  if (e && e[0] && e[0] != '0') return false;
  if (Kc != 2 || h % 16 != 0 || h < 32 || Hout % 16 != 0 || Hout > 128 || C > 128 || Ks < 1) return false;
  const int Dp = (Din + 7) & ~7, KBL = h + Dp, nchk = (KBL + 31) / 32;
  if (Ks * nchk < 2) return false;
  const size_t smem = (size_t)BG_STAGES * 2 * Hout * ATOM_ROW_BYTES + (size_t)(128 + C) * (Hout + 4) * sizeof(float) +
                      (size_t)C * C * sizeof(float) + (size_t)Hout * sizeof(float) + 2048;
  return smem <= 220 * 1024;
}

size_t conv_big_img_floats(int C, int Din, int h, int Ks, int Kc, int Hout) {
  if (!conv_big_shape_ok(C, Din, h, Ks, Kc, Hout)) return 0;
  const int Dp = (Din + 7) & ~7, KBL = h + Dp, nchk = (KBL + 31) / 32;
  return (size_t)Kc * Ks * nchk * 2 * Hout * (ATOM_ROW_BYTES / sizeof(float));
}

int try_launch_conv_fwd_big(const ConvArgs& a, cudaStream_t st, bool* handled) {
  *handled = false;
  if (a.Wimg == nullptr || !conv_big_shape_ok(a.C, a.Din, a.h, a.Ks, a.Kc, a.Hout)) return STC_OK;
  if (!aligned16g(a.u) || !aligned16g(a.Hprev) || !aligned16g(a.r) || !aligned16g(a.rH) || !aligned16g(a.c) ||
      !aligned16g(a.Hnew) || !aligned16g(a.h0) || !aligned16g(a.yh) || !aligned16g(a.Psave) ||
      ((reinterpret_cast<uintptr_t>(a.Wimg) & 127) != 0)) {
    // forward and backward must take the same path for a shape (backward reads what this kernel saves)
    set_error("tcgen05 wide-state path needs 16-byte aligned state / workspace tensors");
    return STC_ERR_BAD_ARG;
  }
  BigPlan p;
  p.npt = 128 / a.C;
  p.Dp = (a.Din + 7) & ~7;
  p.KBL = a.h + p.Dp;
  p.nchk = (p.KBL + 31) / 32;
  p.nch = a.Ks * p.nchk;
  p.PS = a.Hout + 4;
  p.x_vec = (a.Din % 4 == 0) && (a.x0_bs % 4 == 0) && aligned16g(a.x0) && aligned16g(a.yx);
  const long long total_nodes = (long long)a.B * a.N;
  p.ntiles = ceil_div(total_nodes, p.npt);
  p.stage_bytes = (uint32_t)(2 * a.Hout * ATOM_ROW_BYTES);
  size_t o = 0;
  p.off_b = (uint32_t)o; o += (size_t)BG_STAGES * p.stage_bytes;
  p.off_pm = (uint32_t)o; o += round_up((size_t)(128 + a.C) * p.PS * sizeof(float), 16);
  p.off_q = (uint32_t)o; o += round_up((size_t)a.C * a.C * sizeof(float), 16);
  p.off_bias = (uint32_t)o; o += round_up((size_t)a.Hout * sizeof(float), 16);
  p.off_bar = (uint32_t)o; o += 8 * (2 * BG_STAGES + 6) + 16;
  o = round_up(o, 128);
  {   // as many landing stages (16 KB each: 512 threads x 32 B) as fit, at most 4; fewer than 2: register double buffer
    static int land_max = -1;
    if (land_max < 0) {
      const char* e = getenv("STC_BIG_LAND");
      land_max = (e && e[0]) ? atoi(e) : 4;
    }
    int land = (int)(((size_t)226 * 1024 - o) / (BG_THREADS * 32));
    if (land > land_max) land = land_max;
    if (land < 2) land = 0;
    p.land = land;
    p.off_land = (uint32_t)o;
    o += (size_t)land * BG_THREADS * 32;
  }
  p.smem_bytes = (uint32_t)o;
  if (p.smem_bytes > 226 * 1024) return STC_OK;
  {
    const long long items = (long long)a.Kc * p.nch * a.Hout * 8;
    tc_big_prep_kernel<<<(int)min((items + 255) / 256, (long long)1024), 256, 0, st>>>(
        a.W, reinterpret_cast<uint8_t*>(a.Wimg), a.Din, a.h, a.Ks, a.Kc, a.Hout, p.KBL, p.nchk);
    STC_LAUNCH_OK("tc_big_prep_kernel");
  }
  STC_TRY(set_smem(tc_conv_fwd_big_kernel, p.smem_bytes));
  int grid = device_sm_count();
  if (grid > p.ntiles) grid = p.ntiles;
  const int L = a.Din + a.h, P = a.Ks * a.Kc;
  const double R = (double)total_nodes * a.C;
  ScopedKernelTimer _t(KK_TC_CONV_FWD, st,
                       4.0 * R * (a.Ks * L + (a.phase == 0 ? 3 * a.h : 4 * a.h)) + 4.0 * P * L * a.Hout);
  tc_conv_fwd_big_kernel<<<grid, BG_FWD_THREADS, p.smem_bytes, st>>>(a, p, reinterpret_cast<const uint8_t*>(a.Wimg));
  STC_LAUNCH_OK("tc_conv_fwd_big_kernel");
  *handled = true;
  return STC_OK;
}

// =================================================================================================
// backward dx for wide hidden states: the adjoint of the kernel above.
//   dY_k = [Ds | Dm_1] x [W_{k,0}^T ; W_{k,1}^T]      (K = 2 Hout, one N block of KBLp columns per spatial term k)
// Prologue (GRU / activation adjoint -> Ds tile in shared memory, dpre for the dW kernel, direct dH terms, bias
// column sums), dT_1(Gc) from the forward's saved P_1, then per spatial term the same streamed-weight mainloop as
// the forward with A = my row's 8 columns of [Ds | Dm_1] (Dm_1 mixed on the fly from the Ds tile) and an epilogue
// that writes the h-part / x-part adjoints (x-part accumulated across the two convolutions).
// =================================================================================================
struct BigDxPlan {
  int npt, Dp, KBL, KBLp;   // KBLp = KBL rounded up to 16: GEMM N per spatial term
  int nkc;                  // 32-wide K chunks = 2 Hout / 32
  int ntiles, DP, x_vec;
  int stages;               // depth of the weight-chunk ring (3, or 2 when the Ds tile of a wide category axis needs the room)
  uint32_t stage_bytes;     // [hi: KBLp rows x 128 B | lo]
  uint32_t off_b, off_ds, off_q, off_qacc, off_bar, smem_bytes;
};

// img[(k, kc)][hi | lo][n = kb][kk]  <-  W[((k*Kc + c)*L + l(kb))*Hout + o],  32 kc + kk = c*Hout + o
__global__ void tc_big_dx_prep_kernel(const float* __restrict__ W, uint8_t* __restrict__ img, int Din, int h, int Ks,
                                      int Kc, int Hout, int KBL, int KBLp, int nkc) {
  const int L = Din + h;
  const long long total = (long long)Ks * nkc * KBLp * 8;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int q = (int)(idx & 7);
    long long r = idx >> 3;
    const int n = (int)(r % KBLp);
    r /= KBLp;
    const int kc = (int)(r % nkc), k = (int)(r / nkc);
    const int l = n >= KBL ? -1 : (n < h ? Din + n : (n - h < Din ? n - h : -1));
    float v[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int kk = 32 * kc + 4 * q + i;
      const int c = kk / Hout, o = kk - c * Hout;
      v[i] = (l >= 0 && c < Kc) ? W[((size_t)(k * Kc + c) * L + l) * Hout + o] : 0.f;
    }
    uint8_t* base = img + (size_t)(k * nkc + kc) * 2 * KBLp * ATOM_ROW_BYTES;
    store_split4(base, base + (size_t)KBLp * ATOM_ROW_BYTES, atom_chunk_offset(n, q), make_float4(v[0], v[1], v[2], v[3]));
  }
}

// (same role split as the forward kernel: warp 16 issues the MMAs and refills the weight ring, the 16 producer warps
//  meet it only through mbarriers)
__global__ void __launch_bounds__(BG_FWD_THREADS, 1)
tc_conv_bwd_dx_big_kernel(const ConvArgs a, const BigDxPlan p, const uint8_t* __restrict__ img) {
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((smem_u32(smem) & 1023u) != 0u) __trap();
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int C = a.C, h = a.h, Din = a.Din, Hout = a.Hout, DP = p.DP;
  const bool want_dQ = a.dQ != nullptr;
  uint8_t* Bring = smem + p.off_b;
  float* Dsm = reinterpret_cast<float*>(smem + p.off_ds);       // [128 + C][DP]  Ds tile (rows past 128 stay zero)
  float* Qs = reinterpret_cast<float*>(smem + p.off_q);         // [C][C] = T_1(Gc)
  float* dQacc = reinterpret_cast<float*>(smem + p.off_qacc);   // [C][C] per-CTA partial sums of dT_1(Gc)
  uint64_t* b_full = reinterpret_cast<uint64_t*>(smem + p.off_bar);
  uint64_t* b_free = b_full + BG_STAGES;   // (arrays sized for the deepest ring)
  uint64_t* a_free = b_free + BG_STAGES;
  uint64_t* acc_full = a_free + 2;
  uint64_t* a_full = acc_full + 1;                               // [2] producers -> issuer: A buffer staged in TMEM
  uint64_t* acc_empty = a_full + 2;                              // producers -> issuer: a term's epilogue has read the accumulators
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 1);

  if (tid == 0) {
    for (int i = 0; i < BG_STAGES; ++i) {
      mbar_init(&b_full[i], 1);
      mbar_init(&b_free[i], 1);
    }
    mbar_init(&a_free[0], 1);
    mbar_init(&a_free[1], 1);
    mbar_init(acc_full, 1);
    mbar_init(&a_full[0], BG_THREADS / 32);
    mbar_init(&a_full[1], BG_THREADS / 32);
    mbar_init(acc_empty, BG_THREADS / 32);
    mbar_fence_init();
  }
  if (warp == 0) tmem_alloc(tmem_slot, 512u);
  for (int i = tid; i < C * C; i += BG_FWD_THREADS) {
    Qs[i] = a.Q[C * C + i];
    dQacc[i] = 0.f;
  }
  for (int i = tid; i < (128 + C) * DP; i += BG_FWD_THREADS) Dsm[i] = 0.f;
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const int warp_u = uniform_warp_index();
  const uint32_t tmem_base = uniform_u32(*tmem_slot);
  const int Nb = p.KBLp;
  const uint32_t idesc = make_idesc_tf32(128, Nb);
  const uint32_t d_small = tmem_base + (uint32_t)(2 * Nb);
  const long long total_nodes = (long long)a.B * a.N;
  const long long R = total_nodes * C;

  const int sp = warp & 3, qtr = warp >> 2;
  const int erow = sp * 32 + lane;
  const int enode = erow / C, ecat = erow - enode * C;
  const uint32_t tl = tmem_base + ((uint32_t)(sp * 32) << 16);
  const float* qrow = Qs + ecat * C;                    // Dm_1[(node,c')][o] = sum_d Q_1[c'][d] Ds[(node,d)][o]
  const bool xvec = p.x_vec != 0;
  float db_acc = 0.f;                                   // thread j < Hout owns bias-gradient column j

  const int my_tiles = (p.ntiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  const uint32_t per_tile = (uint32_t)(a.Ks * p.nkc);
  const uint32_t total_chunks = (uint32_t)my_tiles * per_tile;
  auto img_of = [&](uint32_t g) { return img + (size_t)(g % per_tile) * p.stage_bytes; };   // (k, kc) order = issue order
  if (warp_u == BG_THREADS / 32) {
    // =============================== issuer: MMAs + weight ring ===============================
    if (elect_one_sync()) {
      for (uint32_t g = 0; g < (uint32_t)(p.stages - 1) && g < total_chunks; ++g) {
        mbar_arrive_expect_tx(&b_full[g], p.stage_bytes);
        bulk_g2s(Bring + (size_t)g * p.stage_bytes, img_of(g), p.stage_bytes, &b_full[g]);
      }
      uint32_t g = 0, terms = 0;
      for (int t_ = 0; t_ < my_tiles; ++t_) {
        for (int k = 0; k < a.Ks; ++k, ++terms) {
          for (int kc = 0; kc < p.nkc; ++kc, ++g) {
            const int buf = (int)(g & 1u), st = (int)(g % (uint32_t)p.stages);
            if (kc == 0 && terms > 0) mbar_wait(acc_empty, (terms - 1u) & 1u);   // previous term's epilogue is done
            mbar_wait(&a_full[buf], (g >> 1) & 1u);
            mbar_wait(&b_full[st], (g / (uint32_t)p.stages) & 1u);
            fence_after_sync();
            const uint32_t a_hi0 = tmem_base + (uint32_t)(BG_ACOL + 64 * buf);
            const uint64_t dBh = make_smem_desc_sw128(smem_u32(Bring + (size_t)st * p.stage_bytes));
            const uint64_t dBl = dBh + (uint64_t)(((uint32_t)Nb * ATOM_ROW_BYTES) >> 4);
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
              const uint64_t ko = (uint64_t)(ks * 2);
              const uint32_t ah = a_hi0 + (uint32_t)(ks * 8), al = ah + 32u;
              const uint32_t d_main = tmem_base + (uint32_t)((ks & 1) * Nb);
              mma_tf32_atmem(d_small, al, dBh + ko, idesc, (kc > 0 || ks > 0) ? 1u : 0u);
              mma_tf32_atmem(d_main, ah, dBh + ko, idesc, (kc > 0 || ks >= 2) ? 1u : 0u);
              mma_tf32_atmem(d_small, ah, dBl + ko, idesc, 1u);
            }
            mma_commit(&a_free[buf]);
            mma_commit(&b_free[st]);
            if (kc == p.nkc - 1) mma_commit(acc_full);
            const uint32_t t = g + (uint32_t)(p.stages - 1);
            if (t < total_chunks) {
              const uint32_t ts = t % (uint32_t)p.stages, tu = t / (uint32_t)p.stages;
              if (tu >= 1u) mbar_wait(&b_free[ts], (tu - 1u) & 1u);
              mbar_arrive_expect_tx(&b_full[ts], p.stage_bytes);
              bulk_g2s(Bring + (size_t)ts * p.stage_bytes, img_of(t), p.stage_bytes, &b_full[ts]);
            }
          }
        }
      }
    }
    __syncwarp();
  } else {
  // =============================== producers + epilogue (16 warps) ===============================
  uint32_t g = 0;
  uint32_t acc_phase = 0;
  for (int tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x) {
    const long long g0 = (long long)tile * p.npt;
    const int nodes_valid = (int)min((long long)p.npt, total_nodes - g0);
    const int rows_valid = nodes_valid * C;
    const long long row0 = g0 * C;
    const bool valid = erow < rows_valid;
    const long long gr = row0 + erow;
    // ---- 1. elementwise adjoint: one float4 of hidden channels per item ----
    const int cpr = h >> 2;
    for (int it = tid; it < 128 * cpr; it += BG_THREADS) {
      const int row = it / cpr, j = (it - row * cpr) << 2;
      float4 g0v = make_float4(0.f, 0.f, 0.f, 0.f), g1v = g0v;
      if (row < rows_valid) {
        const long long o = (row0 + row) * h + j;
        const float4 dhn = *reinterpret_cast<const float4*>(a.dHn + o);
        const float4 uu = *reinterpret_cast<const float4*>(a.u + o);
        const float4 cc = *reinterpret_cast<const float4*>(a.c + o);
        if (a.phase == 1) {
          g0v = make_float4(dhn.x * uu.x * (1.f - cc.x * cc.x), dhn.y * uu.y * (1.f - cc.y * cc.y),
                            dhn.z * uu.z * (1.f - cc.z * cc.z), dhn.w * uu.w * (1.f - cc.w * cc.w));
          if (a.act == STC_ACT_RELU) {
            if (!(cc.x > 0.f)) g0v.x = 0.f;
            if (!(cc.y > 0.f)) g0v.y = 0.f;
            if (!(cc.z > 0.f)) g0v.z = 0.f;
            if (!(cc.w > 0.f)) g0v.w = 0.f;
          }
          *reinterpret_cast<float4*>(a.dpre + (row0 + row) * a.dpre_ld + j) = g0v;
        } else {
          const float4 hp = *reinterpret_cast<const float4*>(a.Hprev + o);
          const float4 rr = *reinterpret_cast<const float4*>(a.r + o);
          const float4 drh = *reinterpret_cast<const float4*>(a.drH + o);
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
          *reinterpret_cast<float4*>(a.dpre + (row0 + row) * a.dpre_ld + j) = g0v;
          *reinterpret_cast<float4*>(a.dpre + (row0 + row) * a.dpre_ld + h + j) = g1v;
          // direct terms of dH; the k = 0 epilogue adds the convolution adjoint (after the block barrier below)
          *reinterpret_cast<float4*>(a.dYh0 + o) =
              make_float4(dhn.x * (1.f - uu.x) + drh.x * rr.x, dhn.y * (1.f - uu.y) + drh.y * rr.y,
                          dhn.z * (1.f - uu.z) + drh.z * rr.z, dhn.w * (1.f - uu.w) + drh.w * rr.w);
        }
      }
      *reinterpret_cast<float4*>(Dsm + row * DP + j) = g0v;
      if (a.phase == 0) *reinterpret_cast<float4*>(Dsm + row * DP + h + j) = g1v;
    }
    bg_producer_sync();
    if (a.dbias && tid < Hout) {
      float sacc = 0.f;
      for (int row = 0; row < rows_valid; ++row) sacc += Dsm[row * DP + tid];
      db_acc += sacc;
    }
    // ---- 2. dT_1(Gc)[c'][d] += sum_{node,o} P_1[(node,c')][o] * Ds[(node,d)][o]  (P_1 saved by the forward kernel) ----
    if (want_dQ && (C & 7) == 0) {
      // Register-blocked form (C % 8 == 0; C = 64 of config 5: one (c', 8 d's) item per thread).  One 16-byte piece of
      // P_1[(node,c')] serves eight pairs: 9 loads per 32 FMAs instead of 2 per 4, and the eight Ds rows d = dblk + 8 j a
      // warp reads at a time are eight CONSECUTIVE rows (row pitch DP = Hout + 4 words: conflict-free 16-byte reads).
      const int nblk = C >> 3;
      for (int item = tid; item < C * nblk; item += BG_THREADS) {
        const int cp = item / nblk, dblk = item - cp * nblk;
        float sacc[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) sacc[j] = 0.f;
        for (int node = 0; node < nodes_valid; ++node) {
          const float* pp = a.Psave + (row0 + node * C + cp) * (long long)Hout;
          const float* dd = Dsm + (node * C + dblk) * DP;
          for (int o = 0; o < Hout; o += 4) {
            const float4 x = *reinterpret_cast<const float4*>(pp + o);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float4 y = *reinterpret_cast<const float4*>(dd + (size_t)(j * nblk) * DP + o);
              sacc[j] = fmaf(x.x, y.x, sacc[j]); sacc[j] = fmaf(x.y, y.y, sacc[j]);
              sacc[j] = fmaf(x.z, y.z, sacc[j]); sacc[j] = fmaf(x.w, y.w, sacc[j]);
            }
          }
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) dQacc[cp * C + dblk + j * nblk] += sacc[j];   // each pair has exactly one owner thread
      }
    } else if (want_dQ) {
      for (int pr = tid; pr < C * C; pr += BG_THREADS) {
        const int cp = pr / C, d = pr - cp * C;
        float sacc = 0.f;
        for (int node = 0; node < nodes_valid; ++node) {
          const float* pp = a.Psave + (row0 + node * C + cp) * (long long)Hout;
          const float* dd = Dsm + (node * C + d) * DP;
          for (int o = 0; o < Hout; o += 4) {
            const float4 x = *reinterpret_cast<const float4*>(pp + o);
            const float4 y = *reinterpret_cast<const float4*>(dd + o);
            sacc = fmaf(x.x, y.x, sacc); sacc = fmaf(x.y, y.y, sacc); sacc = fmaf(x.z, y.z, sacc); sacc = fmaf(x.w, y.w, sacc);
          }
        }
        dQacc[pr] += sacc;   // pair pr is only ever touched by this thread
      }
    }
    // ---- 3. per spatial term: streamed-weight GEMM + epilogue ----
    // my 8 columns of [Ds | Dm_1] for chunk kc: K range [32 kc + 8 qtr, +8).  Terms k > 0 reload Dm_1 from dpre (this
    // thread left it there during term 0): that global load is issued ONE CHUNK AHEAD (`nx`), so its latency travels
    // under the current chunk's split / TMEM store / barrier instead of being exposed 3 x nkc times per tile
    // (profiles/r3o_config3_wide_ncu.txt: 13 % of the kernel's stall samples sat on the first use of that load).
    auto reload_ok = [&](int k_, int kc_) {
      return k_ > 0 && kc_ < p.nkc && (32 * kc_ + 8 * qtr) >= Hout && valid && a.dpre_ld >= 2 * Hout;
    };
    float4 nx0 = make_float4(0.f, 0.f, 0.f, 0.f), nx1 = nx0;
    for (int k = 0; k < a.Ks; ++k) {
      // prior contents the epilogue of this term adds to (direct dH terms / the other convolution's x-part adjoint):
      // requested here, consumed after nkc chunks of work
      float4 prev[4][2];
#pragma unroll
      for (int gi = 0; gi < 4; ++gi) {
        prev[gi][0] = prev[gi][1] = make_float4(0.f, 0.f, 0.f, 0.f);
        const int c0 = 8 * qtr + 32 * gi;
        if (c0 < Nb && valid) {
          if (c0 < h) {
            if (k == 0 && a.phase == 0) {
              const float4* src = reinterpret_cast<const float4*>(a.dYh0 + gr * h + c0);
              prev[gi][0] = src[0];
              prev[gi][1] = src[1];
            } else if (k >= 1 && a.dYh_add != nullptr) {   // adjoint another cell folds into this term
              const float4* src = reinterpret_cast<const float4*>(a.dYh_add + (size_t)(k - 1) * R * h + gr * h + c0);
              prev[gi][0] = src[0];
              prev[gi][1] = src[1];
            }
          } else {
            const int xi = c0 - h;
            const float* xsrc = a.accum_x ? (k == 0 ? a.dYx0 : a.dYx + (size_t)(k - 1) * R * Din)
                                : (k >= 1 && a.dYx_add != nullptr) ? a.dYx_add + (size_t)(k - 1) * R * Din : nullptr;
            if (xi < Din && xvec && xsrc != nullptr) {
              const float* src = xsrc + gr * Din + xi;
              prev[gi][0] = *reinterpret_cast<const float4*>(src);
              if (xi + 4 < Din) prev[gi][1] = *reinterpret_cast<const float4*>(src + 4);
            }
          }
        }
      }
      if (reload_ok(k, 0)) {
        const float4* dp = reinterpret_cast<const float4*>(a.dpre + gr * a.dpre_ld + 8 * qtr);
        nx0 = dp[0];
        nx1 = dp[1];
      }
      for (int kc = 0; kc < p.nkc; ++kc, ++g) {
        const int kk0 = 32 * kc + 8 * qtr;
        float av[8];
        if (kk0 < Hout) {
          const float4 x0 = *reinterpret_cast<const float4*>(Dsm + erow * DP + kk0);
          const float4 x1 = *reinterpret_cast<const float4*>(Dsm + erow * DP + kk0 + 4);
          av[0] = x0.x; av[1] = x0.y; av[2] = x0.z; av[3] = x0.w; av[4] = x1.x; av[5] = x1.y; av[6] = x1.z; av[7] = x1.w;
        } else if (k > 0 && valid && a.dpre_ld >= 2 * Hout) {
          // Dm_1 does not depend on the spatial term: requested one chunk ago
          av[0] = nx0.x; av[1] = nx0.y; av[2] = nx0.z; av[3] = nx0.w; av[4] = nx1.x; av[5] = nx1.y; av[6] = nx1.z; av[7] = nx1.w;
        } else {
          const float* spm = Dsm + (enode * C) * DP + (kk0 - Hout);
#pragma unroll
          for (int i = 0; i < 8; ++i) av[i] = 0.f;
          if (valid) {
#pragma unroll 4
            for (int d = 0; d < C; ++d) {
              const float w = qrow[d];
              const float4 x0 = *reinterpret_cast<const float4*>(spm + d * DP);
              const float4 x1 = *reinterpret_cast<const float4*>(spm + d * DP + 4);
              av[0] = fmaf(w, x0.x, av[0]); av[1] = fmaf(w, x0.y, av[1]); av[2] = fmaf(w, x0.z, av[2]); av[3] = fmaf(w, x0.w, av[3]);
              av[4] = fmaf(w, x1.x, av[4]); av[5] = fmaf(w, x1.y, av[5]); av[6] = fmaf(w, x1.z, av[6]); av[7] = fmaf(w, x1.w, av[7]);
            }
          }
        }
        if (reload_ok(k, kc + 1)) {   // next chunk's Dm_1 piece
          const float4* dp = reinterpret_cast<const float4*>(a.dpre + gr * a.dpre_ld + kk0 + 32);
          nx0 = dp[0];
          nx1 = dp[1];
        }
        if (k == 0 && kk0 >= Hout && valid && a.dpre_ld >= 2 * Hout) {   // the wide dW kernel contracts Y_k^T with [Ds | Dm_1]
          float4* dp = reinterpret_cast<float4*>(a.dpre + gr * a.dpre_ld + kk0);
          dp[0] = make_float4(av[0], av[1], av[2], av[3]);
          dp[1] = make_float4(av[4], av[5], av[6], av[7]);
        }
        const int buf = (int)(g & 1u);
        const uint32_t ua = g >> 1;
        if (ua >= 1u) {
          mbar_wait(&a_free[buf], (ua - 1u) & 1u);
          fence_after_sync();
        }
        {
          const uint32_t tA = tl + (uint32_t)(BG_ACOL + 64 * buf + 8 * qtr);
          float hi[8], lo[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) split_tf32(av[i], hi[i], lo[i]);
          tmem_st8(tA, hi);
          tmem_st8(tA + 32u, lo);
        }
        tmem_st_wait();
        fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(&a_full[buf]);       // one arrive per producer warp: the issuer takes it from here
      }
      // ---- epilogue of spatial term k: columns [0,h) -> h-part adjoint, [h, h+Din) -> x-part adjoint ----
      mbar_wait(acc_full, acc_phase);
      acc_phase ^= 1u;
      fence_after_sync();
#pragma unroll
      for (int gi = 0; gi < 4; ++gi) {
        const int c0 = 8 * qtr + 32 * gi;
        if (c0 >= Nb) break;
        float v[8];
        {
          uint32_t t0[8], t1[8], t2[8];
          tmem_ld8_async(tl + (uint32_t)(2 * Nb + c0), t2);
          tmem_ld8_async(tl + (uint32_t)c0, t0);
          tmem_ld8_async(tl + (uint32_t)(Nb + c0), t1);
          tmem_ld_wait();
          tmem_ld_pin8(t0); tmem_ld_pin8(t1); tmem_ld_pin8(t2);
#pragma unroll
          for (int i = 0; i < 8; ++i) v[i] = (__uint_as_float(t2[i]) + __uint_as_float(t0[i])) + __uint_as_float(t1[i]);
        }
        if (!valid) continue;
        const float4 p0 = prev[gi][0], p1 = prev[gi][1];   // zeros unless this group accumulates (requested before the chunks)
        if (c0 < h) {
          float* dst = (k == 0 ? a.dYh0 : a.dYh + (size_t)(k - 1) * R * h) + gr * h + c0;
          reinterpret_cast<float4*>(dst)[0] = make_float4(v[0] + p0.x, v[1] + p0.y, v[2] + p0.z, v[3] + p0.w);
          reinterpret_cast<float4*>(dst)[1] = make_float4(v[4] + p1.x, v[5] + p1.y, v[6] + p1.z, v[7] + p1.w);
        } else {
          const int xi = c0 - h;
          if (xi >= Din) continue;
          float* dst = (k == 0 ? a.dYx0 : a.dYx + (size_t)(k - 1) * R * Din) + gr * Din + xi;
          if (xvec) {
            reinterpret_cast<float4*>(dst)[0] = make_float4(v[0] + p0.x, v[1] + p0.y, v[2] + p0.z, v[3] + p0.w);
            if (xi + 4 < Din) reinterpret_cast<float4*>(dst)[1] = make_float4(v[4] + p1.x, v[5] + p1.y, v[6] + p1.z, v[7] + p1.w);
          } else {
            const float* prior = a.accum_x ? dst
                                 : (k >= 1 && a.dYx_add != nullptr) ? a.dYx_add + (size_t)(k - 1) * R * Din + gr * Din + xi
                                                                     : nullptr;
#pragma unroll
            for (int i = 0; i < 8; ++i)
              if (xi + i < Din) dst[i] = prior ? prior[i] + v[i] : v[i];
          }
        }
      }
      fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(acc_empty);
      bg_producer_sync();    // the Ds tile is rewritten by the next tile's prologue
    }
  }
  if (a.dbias && tid < Hout) atomicAdd(&a.dbias[tid], db_acc);
  if (want_dQ)
    for (int i = tid; i < C * C; i += BG_THREADS) atomicAdd(&a.dQ[C * C + i], dQacc[i]);
  }   // producers
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, 512u);
}

static bool big_dx_shape_ok(const ConvArgs& a) {
  if (!conv_big_shape_ok(a.C, a.Din, a.h, a.Ks, a.Kc, a.Hout)) return false;
  const int KBLp = (a.h + ((a.Din + 7) & ~7) + 15) & ~15;
  if (KBLp > 128) return false;
  const size_t smem = (size_t)2 * 2 * KBLp * ATOM_ROW_BYTES + (size_t)(128 + a.C) * (a.Hout + 4) * sizeof(float) +
                      2 * (size_t)a.C * a.C * sizeof(float) + 2048;   // with the shallowest (2-stage) ring
  return smem <= 220 * 1024;
}

size_t conv_big_dx_img_floats(int C, int Din, int h, int Ks, int Kc, int Hout) {
  ConvArgs a;
  memset(&a, 0, sizeof(a));
  a.C = C; a.Din = Din; a.h = h; a.Ks = Ks; a.Kc = Kc; a.Hout = Hout;
  if (!big_dx_shape_ok(a)) return 0;
  const int KBLp = (h + ((Din + 7) & ~7) + 15) & ~15;
  return (size_t)Ks * (2 * Hout / 32) * 2 * KBLp * (ATOM_ROW_BYTES / sizeof(float));
}

int try_launch_conv_bwd_dx_big(const ConvArgs& a, cudaStream_t st, bool* handled) {
  *handled = false;
  if (a.Wimg == nullptr || !big_dx_shape_ok(a) || (a.opt & OPT_WIDE_DX_FFMA)) return STC_OK;
  if (!aligned16g(a.dHn) || !aligned16g(a.u) || !aligned16g(a.c) || !aligned16g(a.Hprev) || !aligned16g(a.dpre) ||
      !aligned16g(a.dYh0) || !aligned16g(a.dYh) || !aligned16g(a.dYh_add) || !aligned16g(a.Psave) || (a.dpre_ld % 4) != 0 ||
      (a.phase == 0 && (!aligned16g(a.r) || !aligned16g(a.drH))) || ((reinterpret_cast<uintptr_t>(a.Wimg) & 127) != 0)) {
    set_error("tcgen05 wide-state backward needs 16-byte aligned gradient / workspace tensors");
    return STC_ERR_BAD_ARG;
  }
  BigDxPlan p;
  p.npt = 128 / a.C;
  p.Dp = (a.Din + 7) & ~7;
  p.KBL = a.h + p.Dp;
  p.KBLp = (p.KBL + 15) & ~15;
  p.nkc = 2 * a.Hout / 32;
  p.DP = a.Hout + 4;
  p.x_vec = (a.Din % 4 == 0) && aligned16g(a.dYx0) && aligned16g(a.dYx) && aligned16g(a.dYx_add);
  const long long total_nodes = (long long)a.B * a.N;
  p.ntiles = ceil_div(total_nodes, p.npt);
  p.stage_bytes = (uint32_t)(2 * p.KBLp * ATOM_ROW_BYTES);
  const size_t rest = round_up((size_t)(128 + a.C) * p.DP * sizeof(float), 16) +
                      2 * round_up((size_t)a.C * a.C * sizeof(float), 16) + 8 * (2 * BG_STAGES + 3) + 16;
  p.stages = ((size_t)BG_STAGES * p.stage_bytes + rest <= 226 * 1024) ? BG_STAGES : 2;
  size_t o = 0;
  p.off_b = (uint32_t)o; o += (size_t)p.stages * p.stage_bytes;
  p.off_ds = (uint32_t)o; o += round_up((size_t)(128 + a.C) * p.DP * sizeof(float), 16);
  p.off_q = (uint32_t)o; o += round_up((size_t)a.C * a.C * sizeof(float), 16);
  p.off_qacc = (uint32_t)o; o += round_up((size_t)a.C * a.C * sizeof(float), 16);
  p.off_bar = (uint32_t)o; o += 8 * (2 * BG_STAGES + 6) + 16;
  p.smem_bytes = (uint32_t)o;
  if (p.smem_bytes > 226 * 1024) return STC_OK;
  {
    const long long items = (long long)a.Ks * p.nkc * p.KBLp * 8;
    tc_big_dx_prep_kernel<<<(int)min((items + 255) / 256, (long long)1024), 256, 0, st>>>(
        a.W, reinterpret_cast<uint8_t*>(a.Wimg), a.Din, a.h, a.Ks, a.Kc, a.Hout, p.KBL, p.KBLp, p.nkc);
    STC_LAUNCH_OK("tc_big_dx_prep_kernel");
  }
  STC_TRY(set_smem(tc_conv_bwd_dx_big_kernel, p.smem_bytes));
  int grid = device_sm_count();
  if (grid > p.ntiles) grid = p.ntiles;
  const int L = a.Din + a.h;
  const double R = (double)total_nodes * a.C;
  ScopedKernelTimer _t(KK_TC_CONV_BWD_DX, st,
                       4.0 * R * ((a.phase == 0 ? 6 * a.h + a.Ks * a.Din : 3 * a.h) + a.Hout + a.Ks * L +
                                  (a.dQ ? a.Hout : 0)) + 4.0 * a.Ks * a.Kc * L * a.Hout);
  tc_conv_bwd_dx_big_kernel<<<grid, BG_FWD_THREADS, p.smem_bytes, st>>>(a, p, reinterpret_cast<const uint8_t*>(a.Wimg));
  STC_LAUNCH_OK("tc_conv_bwd_dx_big_kernel");
  *handled = true;
  return STC_OK;
}

// =================================================================================================
// weight gradient for wide hidden states:  dW_{k,c} = Y_k^T x DD_c,  DD = [Ds | Dm_1] as left in `dpre` by the kernel
// above ([R][2 Hout]).  The contraction runs over rows, so both operands change with every chunk: each CTA owns one
// 128 x 128 output tile (spatial term k x a 128-column slice of [Ds | Dm_1]) and a contiguous range of rows; per
// 32-row chunk every thread loads two 16-byte pieces of each operand (next chunk's loads in flight), splits them and
// stores them MN-major (rows = K, SWIZZLE_128B_BASE32B, as tc_conv_bwd_dw_pipe_kernel) into one of two image buffers;
// 12 MMAs per chunk into main0 / main1 / cross accumulators, drained into fp32 registers every BG_DW_DRAIN chunks
// (bounded accumulation chains), one atomicAdd per element at the end.
// =================================================================================================
constexpr int BG_DW_CR = 32;       // rows per chunk (K extent of one image)
constexpr int BG_DW_DRAIN = 4;     // chunks per accumulation chain: 8 K-steps (64 rows) into each main accumulator.  The tensor core
                                   // truncates when it adds into the accumulator, so the error grows with the chain: at 32 chunks one
                                   // dWg element of the N = 4096 parity case sat at 3.0e-5 x mean|ref| against an allowance of 3e-5

struct BigDwPlan {
  int Dp, KBL, N1, NH;             // N1 = 2 Hout, NH = 128-column slices of it
  int nsplit;                      // row ranges per output tile
  long long rows_per;              // rows per range (multiple of BG_DW_CR)
  int x_vec;
  uint32_t img_bytes;              // one buffer: [A_hi | A_lo | B_hi | B_lo], 16 KB each
  uint32_t off_img, off_bar, smem_bytes;
};

__global__ void __launch_bounds__(BG_THREADS, 1)
tc_conv_bwd_dw_big_kernel(const ConvArgs a, const BigDwPlan p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((smem_u32(smem) & 1023u) != 0u) __trap();
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int C = a.C, h = a.h, Din = a.Din, Hout = a.Hout, L = a.Din + a.h;
  constexpr uint32_t IMG1 = 4u * BG_DW_CR * ATOM_ROW_BYTES;          // one hi or lo image: 4 column blocks x 32 rows
  uint8_t* img = smem + p.off_img;
  uint64_t* img_free = reinterpret_cast<uint64_t*>(smem + p.off_bar);   // [2] MMAs that read an image buffer are done
  uint64_t* acc_full = img_free + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_full + 1);
  if (tid == 0) {
    mbar_init(&img_free[0], 1);
    mbar_init(&img_free[1], 1);
    mbar_init(acc_full, 1);
    mbar_fence_init();
  }
  if (warp == 0) tmem_alloc(tmem_slot, 512u);
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const int warp_u = uniform_warp_index();
  const uint32_t tmem_base = uniform_u32(*tmem_slot);
  const uint32_t idesc = make_idesc_tf32_mn(128, 128);
  const uint32_t d_small = tmem_base + 256u;
  const long long total_nodes = (long long)a.B * a.N;
  const long long R = total_nodes * C;

  // which output tile / row range
  const int T = a.Ks * p.NH;
  const int tile = (int)blockIdx.x % T, split = (int)blockIdx.x / T;
  const int k = tile / p.NH, nh = tile - k * p.NH;
  const long long rbeg = (long long)split * p.rows_per;
  const long long rend = min(R, rbeg + p.rows_per);
  const int nchunks = rbeg < rend ? (int)((rend - rbeg + BG_DW_CR - 1) / BG_DW_CR) : 0;

  // staging map: 16-byte piece cq of rows r0 + 16 i (i = 0, 1) of either operand
  const int cq = tid & 31, r0 = tid >> 5;
  const int m0 = 4 * cq;                                  // feature index kb (A) / column within the slice (B)
  const uint32_t soff0 = (uint32_t)(m0 >> 5) * (BG_DW_CR * ATOM_ROW_BYTES);
  // A source: feature kb of spatial term k -> h-part (kb < h), x-part, or zero padding
  int apart = 2;                                          // 0 = h-part, 1 = x-part, 2 = zero
  int aoff = 0;
  if (m0 < h) { apart = 0; aoff = m0; }
  else if (m0 - h < Din) { apart = 1; aoff = m0 - h; }
  const int anvalid = apart == 1 ? min(4, Din - aoff) : 4;
  const bool avec = apart == 0 || (apart == 1 && p.x_vec && anvalid == 4);
  const int bn = nh * 128 + m0;                           // column of [Ds | Dm_1]
  const bool blive = bn < p.N1;
  const float* hsrc = (k == 0 ? a.h0 : a.yh + (size_t)(k - 1) * R * h);
  const float* xsrc = (k == 0 ? a.x0 : a.yx + (size_t)(k - 1) * R * Din);

  auto fetch = [&](int ch, float4 (&fa)[2], float4 (&fb)[2]) {
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const long long row = rbeg + (long long)ch * BG_DW_CR + r0 + 16 * i;
      fa[i] = fb[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (row >= rend) continue;
      if (apart == 0) {
        fa[i] = *reinterpret_cast<const float4*>(hsrc + row * h + aoff);
      } else if (apart == 1) {
        const float* xs;
        if (k == 0) {     // Xt carries a batch stride: row -> (sample, row within the sample)
          const long long rows_per_sample = (long long)a.N * C;
          const long long b = row / rows_per_sample;
          xs = xsrc + b * a.x0_bs + (row - b * rows_per_sample) * Din + aoff;
        } else {
          xs = xsrc + row * Din + aoff;
        }
        if (avec) {
          fa[i] = *reinterpret_cast<const float4*>(xs);
        } else {
          fa[i].x = xs[0];
          if (anvalid > 1) fa[i].y = xs[1];
          if (anvalid > 2) fa[i].z = xs[2];
          if (anvalid > 3) fa[i].w = xs[3];
        }
      }
      if (blive) fb[i] = *reinterpret_cast<const float4*>(a.dpre + row * a.dpre_ld + bn);
    }
  };

  // accumulator ownership: TMEM lane = feature kb, four threads per lane split the 128 columns
  const int sp = warp & 3, qtr = warp >> 2;
  const int mrow = sp * 32 + lane;
  const uint32_t tl = tmem_base + ((uint32_t)(sp * 32) << 16);
  float acc[4][8];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
  uint32_t acc_phase = 0;
  auto drain = [&]() {          // every MMA issued so far has been committed to acc_full by the issuer
    mbar_wait(acc_full, acc_phase);
    acc_phase ^= 1u;
    fence_after_sync();
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      uint32_t t0[8], t1[8], t2[8];
      const uint32_t c0 = (uint32_t)(32 * qtr + 8 * i);
      tmem_ld8_async(tl + 256u + c0, t2);
      tmem_ld8_async(tl + c0, t0);
      tmem_ld8_async(tl + 128u + c0, t1);
      tmem_ld_wait();
      tmem_ld_pin8(t0); tmem_ld_pin8(t1); tmem_ld_pin8(t2);
#pragma unroll
      for (int j = 0; j < 8; ++j)
        acc[i][j] += (__uint_as_float(t2[j]) + __uint_as_float(t0[j])) + __uint_as_float(t1[j]);
    }
    fence_before_sync();
    __syncthreads();            // the next chain's first MMAs overwrite the accumulators
  };

  float4 ca[2], cb[2], na[2], nb[2];
  if (nchunks > 0) fetch(0, ca, cb);
  int in_chain = 0;
  for (int ch = 0; ch < nchunks; ++ch) {
    if (ch + 1 < nchunks) fetch(ch + 1, na, nb);
    const int buf = ch & 1;
    const uint32_t ub = (uint32_t)ch >> 1;
    if (ub >= 1u) mbar_wait(&img_free[buf], (ub - 1u) & 1u);
    uint8_t* A_hi = img + (size_t)buf * p.img_bytes;
    uint8_t* A_lo = A_hi + IMG1;
    uint8_t* B_hi = A_lo + IMG1;
    uint8_t* B_lo = B_hi + IMG1;
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const uint32_t off = soff0 + mn32_chunk_offset(r0 + 16 * i, (m0 & 31) >> 2);
      store_split4(A_hi, A_lo, off, ca[i]);
      store_split4(B_hi, B_lo, off, cb[i]);
    }
    fence_async_smem();
    __syncthreads();
    if (warp_u == 0 && elect_one_sync()) {
      fence_after_sync();
      const uint32_t lbo = BG_DW_CR * ATOM_ROW_BYTES;
      const uint32_t base = smem_u32(A_hi);
#pragma unroll
      for (int ks = 0; ks < BG_DW_CR / 8; ++ks) {
        const uint32_t o = (uint32_t)ks * 2u * MN32_GROUP_BYTES;
        const uint64_t ah = make_smem_desc_mn32(base + o, lbo, MN32_GROUP_BYTES);
        const uint64_t al = make_smem_desc_mn32(base + IMG1 + o, lbo, MN32_GROUP_BYTES);
        const uint64_t bh = make_smem_desc_mn32(base + 2 * IMG1 + o, lbo, MN32_GROUP_BYTES);
        const uint64_t bl = make_smem_desc_mn32(base + 3 * IMG1 + o, lbo, MN32_GROUP_BYTES);
        const uint32_t d_main = tmem_base + (uint32_t)((ks & 1) * 128);
        mma_tf32(d_small, al, bh, idesc, (in_chain > 0 || ks > 0) ? 1u : 0u);
        mma_tf32(d_main, ah, bh, idesc, (in_chain > 0 || ks >= 2) ? 1u : 0u);
        mma_tf32(d_small, ah, bl, idesc, 1u);
      }
      mma_commit(&img_free[buf]);
      if (in_chain == BG_DW_DRAIN - 1 || ch == nchunks - 1) mma_commit(acc_full);
    }
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      ca[i] = na[i];
      cb[i] = nb[i];
    }
    if (++in_chain == BG_DW_DRAIN || ch == nchunks - 1) {
      drain();
      in_chain = 0;
    }
  }
  // ---- one atomicAdd per owned element: dW[((k*Kc + c)*L + l)*Hout + o] ----
  if (nchunks > 0 && mrow < p.KBL) {
    const int l = mrow < h ? Din + mrow : (mrow - h < Din ? mrow - h : -1);
    if (l >= 0) {
      const bool v4 = (Hout & 3) == 0 && (reinterpret_cast<uintptr_t>(a.dW) & 15) == 0;   // 16-byte vector reductions
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 8; j += 4) {
          const int n = nh * 128 + 32 * qtr + 8 * i + j;
          const int c = n / Hout, o = n - c * Hout;
          float* dst = &a.dW[((size_t)(k * a.Kc + c) * L + l) * Hout + o];
          if (v4 && n + 3 < p.N1) {
            red_add_v4(dst, acc[i][j], acc[i][j + 1], acc[i][j + 2], acc[i][j + 3]);
          } else {
#pragma unroll
            for (int e = 0; e < 4; ++e)
              if (n + e < p.N1) {
                const int ce = (n + e) / Hout, oe = (n + e) - ce * Hout;
                atomicAdd(&a.dW[((size_t)(k * a.Kc + ce) * L + l) * Hout + oe], acc[i][j + e]);
              }
          }
        }
    }
  }
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, 512u);
}

bool conv_big_bwd_shape_ok(int C, int Din, int h, int Ks, int Kc, int Hout) {
  ConvArgs a;
  memset(&a, 0, sizeof(a));
  a.C = C; a.Din = Din; a.h = h; a.Ks = Ks; a.Kc = Kc; a.Hout = Hout;
  return big_dx_shape_ok(a);
}

int try_launch_conv_bwd_dw_big(const ConvArgs& a, cudaStream_t st, bool* handled) {
  *handled = false;
  if (a.Wimg == nullptr || !big_dx_shape_ok(a) || a.dpre_ld < 2 * a.Hout || (a.opt & OPT_WIDE_DX_FFMA)) return STC_OK;
  if (!aligned16g(a.dpre) || !aligned16g(a.h0) || !aligned16g(a.yh) || (a.dpre_ld % 4) != 0) return STC_OK;
  BigDwPlan p;
  p.Dp = (a.Din + 7) & ~7;
  p.KBL = a.h + p.Dp;
  p.N1 = 2 * a.Hout;
  p.NH = (p.N1 + 127) / 128;
  p.x_vec = (a.Din % 4 == 0) && (a.x0_bs % 4 == 0) && aligned16g(a.x0) && aligned16g(a.yx);
  const long long R = (long long)a.B * a.N * a.C;
  const int T = a.Ks * p.NH;
  p.nsplit = device_sm_count() / T;
  if (p.nsplit < 1) p.nsplit = 1;
  p.rows_per = (R + p.nsplit - 1) / p.nsplit;
  p.rows_per = (p.rows_per + BG_DW_CR - 1) / BG_DW_CR * BG_DW_CR;
  p.img_bytes = 4u * 4u * BG_DW_CR * ATOM_ROW_BYTES;
  size_t o = 0;
  p.off_img = (uint32_t)o; o += 2 * (size_t)p.img_bytes;
  p.off_bar = (uint32_t)o; o += 8 * 3 + 16;
  p.smem_bytes = (uint32_t)o;
  STC_TRY(set_smem(tc_conv_bwd_dw_big_kernel, p.smem_bytes));
  const int L = a.Din + a.h;
  ScopedKernelTimer _t(KK_TC_CONV_BWD_DW, st, 4.0 * (double)R * (a.Ks * L + a.Kc * a.Hout));
  tc_conv_bwd_dw_big_kernel<<<T * p.nsplit, BG_THREADS, p.smem_bytes, st>>>(a, p);
  STC_LAUNCH_OK("tc_conv_bwd_dw_big_kernel");
  *handled = true;
  return STC_OK;
}

}  // namespace stc
