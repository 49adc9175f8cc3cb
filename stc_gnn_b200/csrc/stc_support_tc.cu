// tcgen05 / TMEM spatial-support kernels for a dense learned support that fits one tile (N <= ~104: the shipped
// SF grid has N = 100).
//
//  tc_support_kernel   Y[b,m,:] = alpha * sum_n A(m,n) X[b,n,:] + beta * Z[b,m,:],  A = Gs^T (forward mode product
//                      'bncl,nm->bmcl', /root/reference/framework/STC_GNN.py:37) or A = Gs (its adjoint).
//      GEMM orientation: D[m][(b,j)] = sum_n A(m,n) * X[b][n][j] -- the output node is the M axis (128 lanes),
//      the flattened (sample, feature) index the N axis (64 per tile), the input node the K axis.  Both operands
//      are MN-major (SWIZZLE_128B_BASE32B): the support image [n][m] is built once per CTA, X rows are contiguous
//      in j.  3xTF32, one short TMEM chain per tile.
//      Warp-specialised, mbarrier-pipelined:  warp 0 issues the MMAs, warps 1-8 stream X (16-byte loads two tiles
//      ahead, hi/lo split, swizzled stores into a 2-deep ring), warps 9-12 drain the 2-deep TMEM accumulator ring:
//      each epilogue thread owns one output node and writes 256 contiguous bytes per tile with 16-byte stores.
#include "stc_conv_common.cuh"
#include "stc_tc.cuh"

#include <stdlib.h>

namespace stc {

using namespace tc;

constexpr int TS_NT = 64;                    // (b,j) columns per tile = GEMM N
constexpr int TS_PROD_WARPS = 8, TS_EPI_WARPS = 4;
constexpr int TS_THREADS = 32 * (1 + TS_PROD_WARPS + TS_EPI_WARPS);
constexpr int TS_SLOTS = 8;                  // 16-byte chunks per producer thread per tile (Kp <= 128)
constexpr int TS_MAX_STAGES = 4;             // X ring depth (as many as fit)
constexpr int TS_ACC_COLS = 4 * TS_NT;       // 2 accumulator buffers x (main + cross-term)
constexpr int TS_OLD = TS_NT + 4;            // row stride (floats) of the output staging tile: conflict-free both ways

struct TcSupPlan {
  int N, Kp, W, transpose, stages;
  long long total_cols, ntiles;
  int tmem_cols;
  uint32_t off_x, off_o, off_bar, smem_bytes, imgX;
};

__global__ void __launch_bounds__(TS_THREADS, 1)
tc_support_kernel(const float* __restrict__ G, const float* __restrict__ X, long long x_bs, const float* Z,
                  long long z_bs, float* Y, float alpha, float beta, const TcSupPlan p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((smem_u32(smem) & 1023u) != 0u) __trap();
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int N = p.N, Kp = p.Kp, W = p.W;
  uint8_t* Xbuf = smem + p.off_x;               // [stages][hi | lo][2 column blocks][Kp][128 B]
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + p.off_bar);   // [stages] producers -> MMA
  uint64_t* empty = full + TS_MAX_STAGES;                           // [stages] MMA -> producers
  uint64_t* accfull = empty + TS_MAX_STAGES;                        // [2] MMA -> epilogue
  uint64_t* accempty = accfull + 2;                                 // [2] epilogue -> MMA
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(accempty + 2);
  const uint32_t colblk = (uint32_t)Kp * ATOM_ROW_BYTES;

  if (tid == 0) {
    for (int i = 0; i < TS_MAX_STAGES; ++i) {
      mbar_init(&full[i], TS_PROD_WARPS);
      mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&accfull[i], 1);
      mbar_init(&accempty[i], TS_EPI_WARPS);
    }
    mbar_fence_init();
  }
  if (warp == 0) tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols);
  // rows N..Kp-1 of the X images are never written by the producers: zero them once
  for (uint32_t i = tid * 16u; i < 2u * (uint32_t)p.stages * p.imgX; i += TS_THREADS * 16u)
    *reinterpret_cast<float4*>(Xbuf + i) = make_float4(0.f, 0.f, 0.f, 0.f);
  fence_async_smem();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  // The support is the A operand and lives in TENSOR MEMORY for the whole kernel: lane m = output node, column k =
  // input node, A(m,k) = Gs[k][m] (transpose) or Gs[m][k]; hi part in columns [TS_ACC_COLS, +Kp), lo part right after.
  // (Shared memory then only holds the streamed X ring, and each MMA reads a third of the bytes from it.)
  const uint32_t tG = tmem_base + TS_ACC_COLS;
  if (warp < 12) {   // three warps per TMEM lane quarter share the K columns
    const int q = warp & 3, part = warp >> 2;
    const int m = q * 32 + lane;
    const uint32_t tl = tG + ((uint32_t)(q * 32) << 16);
    for (int k0 = part * 8; k0 < Kp; k0 += 24) {
      float hi[8], lo[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int k = k0 + i;
        const float v = (k < N && m < N) ? (p.transpose ? G[(size_t)k * N + m] : G[(size_t)m * N + k]) : 0.f;
        split_tf32(v, hi[i], lo[i]);
      }
      tmem_st8(tl + (uint32_t)k0, hi);
      tmem_st8(tl + (uint32_t)(Kp + k0), lo);
    }
    tmem_st_wait();
  }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const long long stride = gridDim.x;

  if (uniform_warp_index() == 0) {
    // =========================== MMA issuer (one elected lane of a converged warp) ===========================
    const uint32_t tmem_base = uniform_u32(*tmem_slot);
    const uint32_t tG = tmem_base + TS_ACC_COLS;
    if (elect_one_sync()) {
      const uint32_t idesc = make_idesc_tf32_atmem_bmn(128, TS_NT);
      // the hi and lo images of an X stage are adjacent with one column-block pitch, and so are the main and the
      // cross-term accumulator: G_hi x [X_hi | X_lo] is ONE N = 2 TS_NT MMA, i.e. 2 MMAs per K-step instead of 3.
      // (Measured neutral, profiles/r3l_outer_support_ncu.txt: this kernel is bound neither by MMA issue nor by its
      //  load structure -- the tensor work is the same three products either way.)
      const uint32_t idesc2 = make_idesc_tf32_atmem_bmn(128, 2 * TS_NT);
      int it = 0;
      for (long long tile = blockIdx.x; tile < p.ntiles; tile += stride, ++it) {
        const int st = it % p.stages, ab = it & 1;
        mbar_wait(&accempty[ab], ((uint32_t)(it >> 1) & 1u) ^ 1u);   // the epilogue drained this accumulator pair
        mbar_wait(&full[st], (uint32_t)(it / p.stages) & 1u);        // the producers staged this X tile
        fence_after_sync();
        const uint32_t xhi = smem_u32(Xbuf + (size_t)st * 2 * p.imgX);
        const uint64_t xh0 = make_smem_desc_mn32(xhi, colblk, MN32_GROUP_BYTES);
        const uint32_t d_main = tmem_base + (uint32_t)(ab * 2 * TS_NT), d_small = d_main + TS_NT;
#pragma unroll 1
        for (int ks = 0; ks < Kp / 8; ++ks) {
          const uint64_t o = (uint64_t)(ks * ((2 * MN32_GROUP_BYTES) >> 4));   // K = 8 rows further down
          const uint32_t gh = tG + (uint32_t)(ks * 8), gl = gh + (uint32_t)Kp;
          mma_tf32_atmem(d_main, gh, xh0 + o, idesc2, ks > 0 ? 1u : 0u);   // [main | cross] (+)= G_hi x [X_hi | X_lo]
          mma_tf32_atmem(d_small, gl, xh0 + o, idesc, 1u);                  // cross += G_lo x X_hi
        }
        mma_commit(&empty[st]);       // X stage may be refilled once these MMAs have read it
        mma_commit(&accfull[ab]);     // ... and the accumulators are complete
      }
    }
  } else if (warp <= TS_PROD_WARPS) {
    // =========================== producers ===========================
    const int pt = tid - 32;
    const int c0 = (pt & 15) << 2, r0 = pt >> 4;       // chunk column of the 64-wide tile, rows r0 + 16 i
    const uint32_t soff0 = (uint32_t)(c0 >> 5) * colblk + mn32_chunk_offset(r0, (c0 & 31) >> 2);
    float4 ra[2][TS_SLOTS];
    auto fetch = [&](long long tile, float4 (&r)[TS_SLOTS]) {
      const long long cg = tile * TS_NT + c0;
      const bool ok = tile < p.ntiles && cg < p.total_cols;     // W % 4 == 0: a chunk never straddles samples
      const long long b = ok ? cg / W : 0;
      const float* src = X + b * x_bs + (cg - b * W);
#pragma unroll
      for (int i = 0; i < TS_SLOTS; ++i) {
        const int n = r0 + 16 * i;
        r[i] = (ok && n < N) ? __ldg(reinterpret_cast<const float4*>(src + (long long)n * W)) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    };
    auto stage = [&](int it, const float4 (&r)[TS_SLOTS]) {
      const int st = it % p.stages;
      mbar_wait(&empty[st], ((uint32_t)(it / p.stages) & 1u) ^ 1u);   // MMAs of the tile `stages` back have read it
      uint8_t* hi = Xbuf + (size_t)st * 2 * p.imgX;
      uint8_t* lo = hi + p.imgX;
#pragma unroll
      for (int i = 0; i < TS_SLOTS; ++i)
        if (r0 + 16 * i < N) store_split4(hi, lo, soff0 + (uint32_t)(16 * i) * ATOM_ROW_BYTES, r[i]);
      fence_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&full[st]);
    };
    long long tile = blockIdx.x;
    fetch(tile, ra[0]);
    fetch(tile + stride, ra[1]);
    for (int it = 0; tile < p.ntiles; it += 2) {
      stage(it, ra[0]);
      fetch(tile + 2 * stride, ra[0]);
      tile += stride;
      if (tile >= p.ntiles) break;
      stage(it + 1, ra[1]);
      fetch(tile + 2 * stride, ra[1]);
      tile += stride;
    }
  } else {
    // =========================== epilogue: TMEM -> staging tile -> coalesced rows ===========================
    // A thread can only read its own TMEM lane (= output node m), but writing Y one node-row per thread makes every
    // 16-byte store of a warp land in a different 128-byte line (and likewise every Z load).  So the tile goes through
    // a padded shared-memory image [128 nodes][TS_NT + 4]: row-per-thread on the TMEM side, 16 consecutive lanes per
    // 256-byte row segment on the global side.
    const int sp = warp & 3;                       // TMEM sub-partition this warp may read
    const int m = sp * 32 + lane;
    const bool live = m < N;
    const uint32_t tl = tmem_base + ((uint32_t)(sp * 32) << 16);
    const bool use_z = beta != 0.f;
    float* Obuf = reinterpret_cast<float*>(smem + p.off_o);
    const int et = tid - 32 * (1 + TS_PROD_WARPS);   // 0..127
    const int ch = et & 15, er0 = et >> 4;           // global side: 16-byte chunk `ch` of rows er0 + 8 i
    // Z travels one tile ahead in registers (same coalesced chunk pattern as the Y stores): its latency is covered by
    // the previous tile's drain instead of being exposed once per tile
    constexpr int ZR = 16;                           // rows er0 + 8 i, i < ZR  (N <= 128)
    float4 zreg[ZR];
    auto fetch_z = [&](long long tile) {
      const long long cg = tile * TS_NT + 4 * ch;
      const bool ok = tile < p.ntiles && cg < p.total_cols;
      const long long b = ok ? cg / W : 0;
      const float* zsrc = Z + b * z_bs + (cg - b * W);
#pragma unroll
      for (int i = 0; i < ZR; ++i) {
        const int r = er0 + 8 * i;
        zreg[i] = (ok && r < N) ? *reinterpret_cast<const float4*>(zsrc + (long long)r * W)   // plain load: Y may alias Z
                                : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    };
    if (use_z) fetch_z(blockIdx.x);
    int it = 0;
    for (long long tile = blockIdx.x; tile < p.ntiles; tile += stride, ++it) {
      const int ab = it & 1;
      const long long cgc = tile * TS_NT + 4 * ch;   // this thread's chunk column (never straddles samples: W % 4 == 0)
      const bool cok = cgc < p.total_cols;
      const long long bc = cok ? cgc / W : 0;
      const int jc = (int)(cgc - bc * W);
      if (use_z) {
#pragma unroll
        for (int i = 0; i < ZR; ++i) {
          const int r = er0 + 8 * i;
          if (r < N) *reinterpret_cast<float4*>(Obuf + r * TS_OLD + 4 * ch) = zreg[i];
        }
        asm volatile("bar.sync 1, 128;" ::: "memory");
        fetch_z(tile + stride);
      }
      mbar_wait(&accfull[ab], (uint32_t)(it >> 1) & 1u);
      fence_after_sync();
      float* orow = Obuf + m * TS_OLD;
#pragma unroll
      for (int hh = 0; hh < TS_NT / 16; ++hh) {    // 16 columns at a time
        uint32_t vm[16], vs[16];
        const uint32_t a0 = tl + (uint32_t)(ab * 2 * TS_NT + hh * 16);
        tmem_ld16_async(a0, vm);
        tmem_ld16_async(a0 + TS_NT, vs);
        tmem_ld_wait();
        tmem_ld_pin16(vm);
        tmem_ld_pin16(vs);
        if (live) {
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            float4 o;
            o.x = alpha * (__uint_as_float(vm[4 * g + 0]) + __uint_as_float(vs[4 * g + 0]));
            o.y = alpha * (__uint_as_float(vm[4 * g + 1]) + __uint_as_float(vs[4 * g + 1]));
            o.z = alpha * (__uint_as_float(vm[4 * g + 2]) + __uint_as_float(vs[4 * g + 2]));
            o.w = alpha * (__uint_as_float(vm[4 * g + 3]) + __uint_as_float(vs[4 * g + 3]));
            float4* slot = reinterpret_cast<float4*>(orow + hh * 16 + 4 * g);
            if (use_z) {
              const float4 z = *slot;
              o.x = fmaf(beta, z.x, o.x); o.y = fmaf(beta, z.y, o.y); o.z = fmaf(beta, z.z, o.z); o.w = fmaf(beta, z.w, o.w);
            }
            *slot = o;
          }
        }
      }
      fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(&accempty[ab]);   // the accumulators are free again while the tile is still being stored
      asm volatile("bar.sync 1, 128;" ::: "memory");
      if (cok) {
        float* ydst = Y + bc * (long long)N * W + jc;
#pragma unroll 4
        for (int r = er0; r < N; r += 8)
          *reinterpret_cast<float4*>(ydst + (long long)r * W) = *reinterpret_cast<const float4*>(Obuf + r * TS_OLD + 4 * ch);
      }
      asm volatile("bar.sync 1, 128;" ::: "memory");   // the staging tile is rewritten by the next tile
    }
  }
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
}

static bool aligned16s(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

static bool tc_support_disabled() {
  static int cached = -1;
  if (cached < 0) {
    const char* e = getenv("STC_DISABLE_TC");
    cached = (e && e[0] && e[0] != '0') ? 1 : 0;
  }
  return cached == 1;
}

// Dense support on the tensor cores when the whole support fits one resident image; *handled tells the caller.
int try_launch_support_tc(const float* G, int N, int B, int width, bool transpose, const float* x, int64_t x_bs,
                          const float* z, int64_t z_bs, float* y, float alpha, float beta, cudaStream_t st,
                          bool* handled) {
  *handled = false;
  if (tc_support_disabled()) return STC_OK;
  if (width % 4 != 0 || x_bs % 4 != 0 || !aligned16s(x) || !aligned16s(y) || N < 8 || N > 128) return STC_OK;
  if (beta != 0.f && (z == nullptr || z_bs % 4 != 0 || !aligned16s(z))) return STC_OK;
  TcSupPlan p;
  p.N = N;
  p.Kp = (N + 7) & ~7;
  if (p.Kp > 16 * TS_SLOTS) return STC_OK;
  p.W = width;
  p.transpose = transpose ? 1 : 0;
  p.total_cols = (long long)B * width;
  p.ntiles = (p.total_cols + TS_NT - 1) / TS_NT;
  p.imgX = (uint32_t)(TS_NT / 32) * p.Kp * ATOM_ROW_BYTES;
  p.tmem_cols = 512;   // 2 x (main + cross-term) x 64 accumulator columns + the support (2 x Kp <= 256 columns)
  const size_t obytes = (size_t)128 * TS_OLD * sizeof(float);
  const size_t fixed = 8 * (2 * TS_MAX_STAGES + 4) + 32 + obytes;
  p.stages = TS_MAX_STAGES;
  while (p.stages > 2 && 2 * (size_t)p.stages * p.imgX + fixed > 227 * 1024) --p.stages;
  size_t o = 0;
  p.off_x = (uint32_t)o; o += 2 * (size_t)p.stages * p.imgX;
  o = round_up(o, 16);
  p.off_o = (uint32_t)o; o += obytes;
  p.off_bar = (uint32_t)o; o += 8 * (2 * TS_MAX_STAGES + 4) + 16;
  p.smem_bytes = (uint32_t)o;
  if (p.smem_bytes > 227 * 1024) return STC_OK;   // larger N: the FFMA kernel tiles it
  STC_TRY(set_smem(tc_support_kernel, p.smem_bytes));
  long long grid = device_sm_count();
  if (grid > p.ntiles) grid = p.ntiles;
  ScopedKernelTimer _t(KK_TC_SUPPORT, st, 4.0 * B * N * width * (2 + (beta != 0.f ? 1 : 0)) + 4.0 * N * N);
  tc_support_kernel<<<(int)grid, TS_THREADS, p.smem_bytes, st>>>(G, x, x_bs, z, z_bs, y, alpha, beta, p);
  STC_LAUNCH_OK("tc_support_kernel");
  *handled = true;
  return STC_OK;
}

// ------------------------------------------------------------------------------------------------
//  tc_outer_kernel     dGs[n][m] += coef * sum_{b,j} A[b][n][j] * Bm[b][m][j]
//      (gradient of the mode product of STC_GNN.py:37 w.r.t. the support; the reference gets it from autograd).
//      GEMM: M = n, N = m, K = (b, j).  Both operands are K-major as stored (a node's feature slab is contiguous),
//      one SW128 atom = 32 features of one sample.  Three main TMEM accumulators are used round-robin plus one for
//      the 3xTF32 cross terms; every TO_DRAIN atoms they are drained into fp32 registers (bounded chains, see
//      profiles/r1_tc_precision.txt); one atomicAdd per element per CTA at the end.
// ------------------------------------------------------------------------------------------------
constexpr int TO_DRAIN = 32;          // atoms per accumulation chain set (two slots: 16 atoms = 64 K-steps per accumulator)
constexpr int TO_SH = 5;              // ring of raw -> hi operand images (cp.async landing zones)
constexpr int TO_SL = 2;              // ring of lo images
constexpr int TO_THREADS = CV_THREADS + 32;   // 8 producer / drain warps + 1 MMA-issue warp

struct TcOuterPlan {
  int N, Npad, W, B, atoms_per_sample;
  int nblk;       // 128-node blocks per side (1 when the support fits one tile); blockIdx.y = block row * nblk + block column
  int tmem_cols;
  int drain;      // atoms per chain set
  uint32_t imgA, imgB, off_lo, off_bar, smem_bytes;
};

// Round-2 structure (profiles/r3l_outer_support_ncu.txt): with 16-byte loads into registers two atoms ahead the
// compiler's register reuse serialised every fetch behind the previous one (long-scoreboard stalls on address
// arithmetic, 0.27-0.35 of HBM whatever the MMA count).  Now the operand chunks travel global -> shared with cp.async
// (no registers held, TO_SH - 2 = 3 atoms = 77 KB in flight per SM); every producer thread converts the chunks IT
// requested in place (raw -> hi in the landing zone, lo into a second, shorter ring), so no block-wide barrier is needed
// between the copy and the conversion; warp 8 only issues MMAs, paced by full / done mbarriers.  TMEM: two slots of
// [main | cross] used round-robin, drained into fp32 registers every `drain` atoms (bounded chains).
// BLOCKS = false: the support fits one tile (n0 = m0 = 0, every row bound is N -- exactly the one-tile code);
// BLOCKS = true: gridDim.y walks the 128 x 128 blocks of a larger support.
template <bool BLOCKS>
__global__ void __launch_bounds__(TO_THREADS, 1)
tc_outer_kernel(const float* __restrict__ A, long long a_bs, const float* __restrict__ Bm, float coef, float* dG,
                const TcOuterPlan p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((smem_u32(smem) & 1023u) != 0u) __trap();
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int N = p.N, W = p.W;
  const uint32_t hsz = p.imgA + p.imgB;              // one stage of either ring: [A image | B image]
  uint8_t* Hring = smem;                             // [TO_SH][A raw->hi | B raw->hi]
  uint8_t* Lring = smem + p.off_lo;                  // [TO_SL][A lo | B lo]
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + p.off_bar);   // [TO_SH] producers -> MMA warp
  uint64_t* done = full + TO_SH;                                     // [TO_SH] MMA commit -> producers
  uint64_t* drained = done + TO_SH;                                  // producers have read the accumulators
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(drained + 1);
  if (tid == 0) {
    for (int i = 0; i < TO_SH; ++i) {
      mbar_init(&full[i], CV_THREADS / 32);
      mbar_init(&done[i], 1);
    }
    mbar_init(drained, CV_THREADS / 32);
    mbar_fence_init();
  }
  if (warp == 0) tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols);
  for (uint32_t i = tid * 16u; i < (TO_SH + TO_SL) * hsz; i += TO_THREADS * 16u)   // rows >= N stay zero for good
    *reinterpret_cast<float4*>(smem + i) = make_float4(0.f, 0.f, 0.f, 0.f);
  fence_async_smem();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const int warp_u = uniform_warp_index();
  const uint32_t tmem_base = uniform_u32(*tmem_slot);
  // N > 128: this CTA owns the 128 x 128 block (n0.., m0..) of dGs; rows past the edge of an operand block stay zero
  const int n0 = BLOCKS ? ((int)blockIdx.y / p.nblk) * 128 : 0, m0 = BLOCKS ? ((int)blockIdx.y % p.nblk) * 128 : 0;
  const int rowsA = BLOCKS ? min(128, N - n0) : N, rowsB = BLOCKS ? min(128, N - m0) : N;
  const int rows_both = BLOCKS ? min(rowsA, rowsB) : N;
  const int nsamples = (p.B - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  const long long natoms = (long long)nsamples * p.atoms_per_sample;

  if (warp_u == CV_THREADS / 32) {
    // =============================== MMA issuer ===============================
    const uint32_t idesc = make_idesc_tf32(128, p.Npad);
    int at = 0, in_set = 0;
    uint32_t drain_parity = 0;
    for (long long seq = 0; seq < natoms; ++seq) {
      const int hb = (int)(seq % TO_SH), lb = (int)(seq % TO_SL);
      mbar_wait(&full[hb], (uint32_t)(seq / TO_SH) & 1u);
      if (seq > 0 && in_set == 0) {   // first atom of a new chain set: the producers must have drained the accumulators
        mbar_wait(drained, drain_parity);
        drain_parity ^= 1u;
      }
      const int kleft = W - at * ATOM_K;
      const int ksteps = kleft >= ATOM_K ? 4 : (kleft + 7) / 8;
      const int slot = in_set & 1;
      const bool fresh = in_set < 2;  // first atom into this slot since the drain
      if (elect_one_sync()) {
        fence_after_sync();
        const uint32_t a_hi = smem_u32(Hring + (size_t)hb * hsz), b_hi = a_hi + p.imgA;
        const uint32_t a_lo = smem_u32(Lring + (size_t)lb * hsz), b_lo = a_lo + p.imgA;
        const uint32_t d_main = tmem_base + (uint32_t)(slot * 2 * p.Npad), d_cross = d_main + (uint32_t)p.Npad;
        for (int ks = 0; ks < ksteps; ++ks) {
          const uint32_t o = ks * 32;
          const uint64_t ah = make_smem_desc_sw128(a_hi + o), al = make_smem_desc_sw128(a_lo + o);
          const uint64_t bh = make_smem_desc_sw128(b_hi + o), bl = make_smem_desc_sw128(b_lo + o);
          const uint32_t accf = (fresh && ks == 0) ? 0u : 1u;
          mma_tf32(d_cross, al, bh, idesc, accf);
          mma_tf32(d_cross, ah, bl, idesc, 1u);
          mma_tf32(d_main, ah, bh, idesc, accf);
        }
        mma_commit(&done[hb]);
      }
      __syncwarp();
      if (++at == p.atoms_per_sample) at = 0;
      if (++in_set == p.drain) in_set = 0;
    }
  } else {
    // =============================== producers / drain / epilogue ===============================
    // copy / conversion map: chunk q of rows r0 + 32 i of either operand -- a thread converts exactly what it copied
    const int q = tid & 7, r0 = tid >> 3;
    uint32_t soff[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) soff[i] = atom_chunk_offset(r0 + 32 * i, q);
    int cs = 0, cat = 0;                  // (sample, atom) of the next copy to issue
    auto issue_copy = [&](long long seq) {   // atom seq -> H ring (nothing for seq >= natoms: the group is still committed)
      if (seq < natoms) {
        const long long b = blockIdx.x + cs * (long long)gridDim.x;
        const int j = cat * ATOM_K + q * 4;
        if (j < W) {                       // W % 4 == 0; chunks past W are never read (the MMAs stop at ceil(kleft / 8))
          const float* pa = A + b * a_bs + (long long)n0 * W + j;
          const float* pb = Bm + (b * (long long)N + m0) * W + j;
          const uint32_t base = smem_u32(Hring + (size_t)(seq % TO_SH) * hsz);
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int r = r0 + 32 * i;
            if (r < rows_both) {   // the common case (always, when the support fits one tile): one branch for both operands
              cp_async16(base + soff[i], pa + (long long)r * W);
              cp_async16(base + p.imgA + soff[i], pb + (long long)r * W);
            } else {               // edge blocks of a large support: the operands have different row counts
              if (r < rowsA) cp_async16(base + soff[i], pa + (long long)r * W);
              if (r < rowsB) cp_async16(base + p.imgA + soff[i], pb + (long long)r * W);
            }
          }
        }
        if (++cat == p.atoms_per_sample) {
          cat = 0;
          ++cs;
        }
      }
      cp_async_commit();
    };
    // accumulators: thread (sub-partition sp, half) owns row 32 sp + lane and Npad/2 columns
    const int sp = warp & 3, half = warp >> 2;
    const int nrow = sp * 32 + lane;
    const uint32_t tl = tmem_base + ((uint32_t)(sp * 32) << 16);
    const int ncols_half = p.Npad >> 1, col0 = half * ncols_half;
    float acc[8][8];   // Npad <= 128 -> at most 64 columns per thread
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

    int in_set = 0;
    auto drain = [&](long long last_seq) {   // every atom up to last_seq has been handed to the MMA warp
      mbar_wait(&done[last_seq % TO_SH], (uint32_t)(last_seq / TO_SH) & 1u);   // commits complete in order
      fence_after_sync();
      const int slots = in_set >= 2 ? 2 : in_set;
#pragma unroll
      for (int ch = 0; ch < 8; ++ch) {
        if (ch * 8 < ncols_half) {
          const uint32_t cc = (uint32_t)(col0 + ch * 8);
          for (int sl = 0; sl < slots; ++sl) {
            float v[8], t[8];
            tmem_ld8(tl + (uint32_t)(sl * 2 * p.Npad + p.Npad) + cc, v);
            tmem_ld8(tl + (uint32_t)(sl * 2 * p.Npad) + cc, t);
#pragma unroll
            for (int i = 0; i < 8; ++i) acc[ch][i] += v[i] + t[i];
          }
        }
      }
      fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(drained);
      in_set = 0;
    };

    for (int k = 0; k < TO_SH - 2; ++k) issue_copy(k);      // the ring starts empty: no waits
    int at = 0;
    for (long long seq = 0; seq < natoms; ++seq) {
      // (a) Once the MMAs of atom seq - 2 are complete, its H stage can take the copy of atom seq + TO_SH - 2 and its L
      //     stage (TO_SL = 2: the same index parity as seq) the lo image of atom seq.  Waiting for seq - 2 rather than
      //     seq - 1 lets this conversion run beside the MMAs of atom seq - 1; TO_SH - 2 = 3 atoms (77 KB) stay in flight.
      if (seq >= 2) mbar_wait(&done[(seq - 2) % TO_SH], (uint32_t)((seq - 2) / TO_SH) & 1u);
      issue_copy(seq + TO_SH - 2);
      // (b) this thread's chunks of atom seq have landed
      cp_async_wait<TO_SH - 2>();
      const int j = at * ATOM_K + q * 4;
      if (j < W) {
        uint8_t* hb = Hring + (size_t)(seq % TO_SH) * hsz;
        uint8_t* lbp = Lring + (size_t)(seq % TO_SL) * hsz;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          // both raw chunks are read before either is rewritten: the in-place stores would otherwise order the second
          // load behind them (measured: 5.6 -> 6.6 ms per step when the two operands were converted one after the other)
          if (r0 + 32 * i < rows_both) {
            const float4 va = *reinterpret_cast<const float4*>(hb + soff[i]);
            const float4 vb = *reinterpret_cast<const float4*>(hb + p.imgA + soff[i]);
            store_split4(hb, lbp, soff[i], va);
            store_split4(hb + p.imgA, lbp + p.imgA, soff[i], vb);
          } else if (r0 + 32 * i < rowsA) {
            store_split4(hb, lbp, soff[i], *reinterpret_cast<const float4*>(hb + soff[i]));
          } else if (r0 + 32 * i < rowsB) {
            store_split4(hb + p.imgA, lbp + p.imgA, soff[i], *reinterpret_cast<const float4*>(hb + p.imgA + soff[i]));
          }
        }
      } else if (j < ((W + 7) & ~7)) {
        // W % 8 == 4: the last K-step of the sample's last atom reads 4 columns past W.  Nothing was copied there, so the
        // stage still holds a column of an earlier atom (any CTA with more than one sample): zero it in both images.
        uint8_t* hb = Hring + (size_t)(seq % TO_SH) * hsz;
        uint8_t* lbp = Lring + (size_t)(seq % TO_SL) * hsz;
        const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          if (r0 + 32 * i < rowsA) store_split4(hb, lbp, soff[i], z);
          if (r0 + 32 * i < rowsB) store_split4(hb + p.imgA, lbp + p.imgA, soff[i], z);
        }
      }
      fence_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&full[seq % TO_SH]);
      if (++at == p.atoms_per_sample) at = 0;
      if (++in_set == p.drain || seq == natoms - 1) drain(seq);
    }
    cp_async_wait<0>();

    if (nrow < rowsA) {
      const bool v4 = (N & 3) == 0 && (col0 & 3) == 0 && (reinterpret_cast<uintptr_t>(dG) & 15) == 0;
#pragma unroll
      for (int ch = 0; ch < 8; ++ch) {
        if (ch * 8 < ncols_half) {
#pragma unroll
          for (int i = 0; i < 8; i += 4) {
            const int m = col0 + ch * 8 + i;
            float* dst = &dG[(size_t)(n0 + nrow) * N + m0 + m];
            if (v4 && m + 3 < rowsB) {
              red_add_v4(dst, coef * acc[ch][i], coef * acc[ch][i + 1], coef * acc[ch][i + 2], coef * acc[ch][i + 3]);
            } else {
#pragma unroll
              for (int e = 0; e < 4; ++e)
                if (m + e < rowsB) atomicAdd(dst + e, coef * acc[ch][i + e]);
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

int try_launch_outer_tc(int N, int B, int width, const float* a, int64_t a_bs, const float* bmat, float coef, float* dG,
                        cudaStream_t st, bool* handled) {
  *handled = false;
  if (tc_support_disabled()) return STC_OK;
  if (width % 4 != 0 || a_bs % 4 != 0 || !aligned16s(a) || !aligned16s(bmat) || N < 8) return STC_OK;
  TcOuterPlan p;
  p.N = N;
  p.nblk = (N + 127) / 128;
  if ((long long)p.nblk * p.nblk > 65535) return STC_OK;
  if (N > 128) {   // A/B switch for tools/bench_dense_support.py (shared with the N > 128 support kernel)
    static int big_off = -1;
    if (big_off < 0) {
      const char* e = getenv("STC_DISABLE_TC_SUPPORT_BIG");
      big_off = (e && e[0] && e[0] != '0') ? 1 : 0;
    }
    if (big_off == 1) return STC_OK;
  }
  p.Npad = N > 128 ? 128 : (N + 15) & ~15;
  p.W = width;
  p.B = B;
  p.atoms_per_sample = (width + ATOM_K - 1) / ATOM_K;
  {
    static int v_drain = -1;
    if (v_drain < 0) {
      const char* e = getenv("STC_OUTER_DRAIN");
      v_drain = (e && atoi(e) > 1) ? atoi(e) : TO_DRAIN;
    }
    p.drain = v_drain;
  }
  p.tmem_cols = 32;
  while (p.tmem_cols < 4 * p.Npad) p.tmem_cols *= 2;
  p.imgA = 128 * ATOM_ROW_BYTES;
  p.imgB = (uint32_t)round_up((size_t)p.Npad * ATOM_ROW_BYTES, 1024);
  const uint32_t hsz = p.imgA + p.imgB;
  p.off_lo = TO_SH * hsz;
  p.off_bar = (TO_SH + TO_SL) * hsz;
  p.smem_bytes = p.off_bar + 8 * (2 * TO_SH + 1) + 16;
  if (p.smem_bytes > 227 * 1024) return STC_OK;
  auto kern = p.nblk > 1 ? tc_outer_kernel<true> : tc_outer_kernel<false>;
  STC_TRY(set_smem(kern, p.smem_bytes));
  // one tile: the CTAs split the samples.  N > 128: one CTA per 128 x 128 block of dGs and sample slice -- as few slices
  // as still fill the device twice over (long K runs per CTA, one pass of vector reductions per CTA at the end)
  const int nblocks = p.nblk * p.nblk;
  int grid = device_sm_count();
  if (nblocks > 1) grid = (2 * grid + nblocks - 1) / nblocks;
  if (grid > B) grid = B;
  ScopedKernelTimer _t(KK_TC_OUTER, st, 4.0 * B * N * width * 2 + 4.0 * N * N);
  kern<<<dim3(grid, nblocks), TO_THREADS, p.smem_bytes, st>>>(a, a_bs, bmat, coef, dG, p);
  STC_LAUNCH_OK("tc_outer_kernel");
  *handled = true;
  return STC_OK;
}

}  // namespace stc
