// Top-k pair scores of the graph generator over ALL candidate columns: the pattern-choosing step of the sparse MGP_Gen
// (stc_gnn_b200/sparse_mgp.py topk_pattern).  Nothing of size N^2 ever reaches HBM.  The query rows may be a block
// [row0, row0 + n_rows) of the N nodes (a rank of the row-partitioned generator selects its own rows only); the column
// tiles always start at column 0, so each row's K chains, tiles and result are those of the full selection.
//
//  tc_pair_topk_kernel      S[n][m] = <U_n, V_m> - <V_n, U_m> = [U | V]_n . [V | -U]_m: one 3xTF32 GEMM with K = 2W over
//      128 x 128 tiles.  A CTA owns the 128 query rows of block blockIdx.x and sweeps the column tiles of segment
//      blockIdx.y; its A rows are re-streamed from L2 for every tile.  Two epilogue threads own a row, each half of every
//      tile's columns, and keep the row's running top-k list (k <= 32, sorted best-first) in shared memory: the 64
//      accumulator registers leave no room for it in the 168 a thread of 288 may have.  A tile's scores enter the list
//      with one compare each against its k-th entry, the common case; the halves insert one after the other.  The CTA
//      writes the k best (score, col) pairs of each row to the workspace.
//  pair_topk_merge_kernel   merges the segments' lists of a row in segment order and writes the k best in ascending
//      column order.
//
// Order of the selection: larger score first, equal scores to the smaller column.  It is a total order on (score, col),
// so the merge result does not depend on how the columns were split into segments.  A tile's scores depend only on the fixed K-chain order; there are no atomics, so the output
// is a pure function of (U, V, k): bitwise the same on every call and for any segment count.
//
// Structure (tc_outer_kernel in stc_support_tc.cu, which contracts the same node-major K-major operands): 8 producer /
// drain warps + 1 MMA-issue warp; operand chunks land with cp.async and every producer thread converts the chunks it
// copied in place (raw -> hi, lo into a second ring).  The operands are never concatenated in memory: K-atoms
// [0, aph) of the A image read U and [aph, 2 aph) read V; the B image reads V, then U negated during the hi / lo split.
// TMEM holds two [main | cross] slots used round-robin per atom and drained into fp32 registers every TK_DRAIN atoms
// (<= 64 K-steps per chain, profiles/r1_tc_precision.txt) and at the end of every tile.
#include "stc_conv_common.cuh"
#include "stc_tc.cuh"

#include <math.h>

namespace stc {

using namespace tc;

constexpr int TK_SH = 4;                      // ring of raw -> hi operand images (cp.async landing zones)
constexpr int TK_SL = 2;                      // ring of lo images
constexpr int TK_DRAIN = 32;                  // atoms per chain set (two slots: 16 atoms = 64 K-steps per accumulator)
constexpr int TK_PROD_WARPS = 8;
constexpr int TK_THREADS = 32 * (TK_PROD_WARPS + 1);
constexpr int TK_TILE = 128;                  // rows per block and columns per tile
constexpr uint32_t TK_IMG = TK_TILE * ATOM_ROW_BYTES;   // one operand image: 128 rows x one 32-float atom
constexpr uint32_t TK_HSZ = 2 * TK_IMG;                 // one ring stage: [A | B]
constexpr int TK_KMAX = 32;
constexpr int TK_LD = TK_KMAX + 1;            // row pitch of the lists (odd: the 32 rows of a warp hit 32 banks)
constexpr uint32_t TK_OFF_LIST = (TK_SH + TK_SL) * TK_HSZ;
constexpr uint32_t TK_OFF_BAR = TK_OFF_LIST + 2 * TK_TILE * TK_LD * 4;   // [128 rows][TK_LD] scores, then columns
constexpr uint32_t TK_SMEM = TK_OFF_BAR + 8 * (2 * TK_SH + 1) + 16;

struct TopkPlan {
  int N, W, k;
  int row0, n_rows;    // the query rows [row0, row0 + n_rows); the columns are always all N
  int aph;             // K-atoms per half (ceil(W / 32)); a tile takes 2 aph atoms
  int ntiles, tiles_per_seg;
};

// the selection order: (s, c) comes before (s2, c2)
__device__ __forceinline__ bool tk_better(float s, int c, float s2, int c2) { return s > s2 || (s == s2 && c < c2); }

// insert (s, c) into a list of k entries kept best-first (the caller has checked that it beats the last entry)
__device__ __forceinline__ void tk_insert(float* ls, int* lc, int k, float s, int c) {
  int i = k - 1;
  for (; i > 0 && tk_better(s, c, ls[i - 1], lc[i - 1]); --i) {
    ls[i] = ls[i - 1];
    lc[i] = lc[i - 1];
  }
  ls[i] = s;
  lc[i] = c;
}

__global__ void __launch_bounds__(TK_THREADS, 1)
tc_pair_topk_kernel(const float* __restrict__ U, const float* __restrict__ V, float* __restrict__ ws_s,
                    int* __restrict__ ws_c, const TopkPlan p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((smem_u32(smem) & 1023u) != 0u) __trap();
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int N = p.N, W = p.W, k = p.k, aph = p.aph, apt = 2 * p.aph;
  uint8_t* Hring = smem;                                              // [TK_SH][A raw->hi | B raw->hi]
  uint8_t* Lring = smem + TK_SH * TK_HSZ;                             // [TK_SL][A lo | B lo]
  float* Ls = reinterpret_cast<float*>(smem + TK_OFF_LIST);          // [128 rows][TK_LD] running top-k of each row
  int* Lc = reinterpret_cast<int*>(Ls + TK_TILE * TK_LD);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + TK_OFF_BAR);   // [TK_SH] producers -> MMA warp
  uint64_t* done = full + TK_SH;                                      // [TK_SH] MMA commit -> producers
  uint64_t* drained = done + TK_SH;                                   // producers have read the accumulators
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(drained + 1);
  if (tid == 0) {
    for (int i = 0; i < TK_SH; ++i) {
      mbar_init(&full[i], TK_PROD_WARPS);
      mbar_init(&done[i], 1);
    }
    mbar_init(drained, TK_PROD_WARPS);
    mbar_fence_init();
  }
  if (warp == 0) tmem_alloc(tmem_slot, 512u);   // 2 slots x [main | cross] x 128 columns
  for (uint32_t i = tid * 16u; i < TK_OFF_LIST; i += TK_THREADS * 16u)   // A rows >= N stay zero for good
    *reinterpret_cast<float4*>(smem + i) = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int i = tid; i < TK_TILE * TK_LD; i += TK_THREADS) {
    Ls[i] = -INFINITY;
    Lc[i] = 0x7fffffff;
  }
  fence_async_smem();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const int warp_u = uniform_warp_index();
  const uint32_t tmem_base = uniform_u32(*tmem_slot);
  const int n0 = p.row0 + (int)blockIdx.x * TK_TILE, rowsA = min(TK_TILE, p.row0 + p.n_rows - n0);
  const int t0 = (int)blockIdx.y * p.tiles_per_seg, t1 = min(p.ntiles, t0 + p.tiles_per_seg);
  const long long natoms = (long long)(t1 - t0) * apt;

  if (warp_u == TK_PROD_WARPS) {
    // =============================== MMA issuer ===============================
    const uint32_t idesc = make_idesc_tf32(TK_TILE, TK_TILE);
    int at = 0;
    uint32_t drain_parity = 0;
    for (long long seq = 0; seq < natoms; ++seq) {
      const int hb = (int)(seq % TK_SH), lb = (int)(seq % TK_SL);
      mbar_wait(&full[hb], (uint32_t)(seq / TK_SH) & 1u);
      const int in_set = at % TK_DRAIN;
      if (seq > 0 && in_set == 0) {   // first atom of a chain set: the producers must have drained the accumulators
        mbar_wait(drained, drain_parity);
        drain_parity ^= 1u;
      }
      const int kleft = W - (at < aph ? at : at - aph) * ATOM_K;
      const int ksteps = kleft >= ATOM_K ? 4 : (kleft + 7) / 8;   // chunks past W are zero in both images
      const int slot = in_set & 1;
      const bool fresh = in_set < 2;   // first atom into this slot since the drain
      if (elect_one_sync()) {
        fence_after_sync();
        const uint32_t a_hi = smem_u32(Hring + (size_t)hb * TK_HSZ), b_hi = a_hi + TK_IMG;
        const uint32_t a_lo = smem_u32(Lring + (size_t)lb * TK_HSZ), b_lo = a_lo + TK_IMG;
        const uint32_t d_main = tmem_base + (uint32_t)(slot * 2 * TK_TILE), d_cross = d_main + (uint32_t)TK_TILE;
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
      if (++at == apt) at = 0;
    }
  } else {
    // =============================== producers / drain / selection ===============================
    const int q = tid & 7, r0 = tid >> 3;   // chunk q of rows r0 + 32 i of either operand
    uint32_t soff[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) soff[i] = atom_chunk_offset(r0 + 32 * i, q);
    int ctile = t0, cat = 0;                // (tile, atom) of the next copy to issue
    auto issue_copy = [&](long long seq) {   // nothing for seq >= natoms: the group is still committed
      if (seq < natoms) {
        const bool second = cat >= aph;
        const int j = (second ? cat - aph : cat) * ATOM_K + q * 4;
        if (j < W) {
          const int m0 = ctile * TK_TILE, rowsB = min(TK_TILE, N - m0);
          const float* pa = (second ? V : U) + (long long)n0 * W + j;
          const float* pb = (second ? U : V) + (long long)m0 * W + j;
          const uint32_t base = smem_u32(Hring + (size_t)(seq % TK_SH) * TK_HSZ);
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int r = r0 + 32 * i;
            if (r < rowsA) cp_async16(base + soff[i], pa + (long long)r * W);
            if (r < rowsB) cp_async16(base + TK_IMG + soff[i], pb + (long long)r * W);
          }
        }
        if (++cat == apt) {
          cat = 0;
          ++ctile;
        }
      }
      cp_async_commit();
    };
    // accumulators: thread (sub-partition sp, half) owns row 32 sp + lane and the 64 columns [64 half, 64 half + 64)
    const int sp = warp & 3, half = warp >> 2;
    const int nrow = sp * 32 + lane;
    const uint32_t tl = tmem_base + ((uint32_t)(sp * 32) << 16);
    const int col0 = half * (TK_TILE / 2);
    float acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
    float* ls = Ls + nrow * TK_LD;
    int* lc = Lc + nrow * TK_LD;

    auto drain = [&](long long last_seq, int atoms_in_set) {   // every atom up to last_seq went to the MMA warp
      mbar_wait(&done[last_seq % TK_SH], (uint32_t)(last_seq / TK_SH) & 1u);   // commits complete in order
      fence_after_sync();
      const int slots = atoms_in_set >= 2 ? 2 : 1;
#pragma unroll
      for (int ch = 0; ch < 8; ++ch) {
        const uint32_t cc = (uint32_t)(col0 + ch * 8);
        for (int sl = 0; sl < slots; ++sl) {
          float v[8], t[8];
          tmem_ld8(tl + (uint32_t)(sl * 2 * TK_TILE + TK_TILE) + cc, v);
          tmem_ld8(tl + (uint32_t)(sl * 2 * TK_TILE) + cc, t);
#pragma unroll
          for (int i = 0; i < 8; ++i) acc[ch][i] += v[i] + t[i];
        }
      }
      fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(drained);
    };
    for (int a = 0; a < TK_SH - 2; ++a) issue_copy(a);      // the ring starts empty: no waits
    int at = 0, tile = t0;
    for (long long seq = 0; seq < natoms; ++seq) {
      // as in tc_outer: once the MMAs of atom seq - 2 are complete, its H stage takes the copy of atom seq + TK_SH - 2
      // and its L stage (TK_SL = 2) the lo image of atom seq
      if (seq >= 2) mbar_wait(&done[(seq - 2) % TK_SH], (uint32_t)((seq - 2) / TK_SH) & 1u);
      issue_copy(seq + TK_SH - 2);
      cp_async_wait<TK_SH - 2>();
      const bool second = at >= aph;
      const int j = (second ? at - aph : at) * ATOM_K + q * 4;
      const int rowsB = min(TK_TILE, N - tile * TK_TILE);
      uint8_t* hb = Hring + (size_t)(seq % TK_SH) * TK_HSZ;
      uint8_t* lbp = Lring + (size_t)(seq % TK_SL) * TK_HSZ;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int r = r0 + 32 * i;
        if (j >= W) {   // past the end of a partial atom: zero in both images (the K-step that reads it adds nothing)
          const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
          store_split4(hb, lbp, soff[i], z);
          store_split4(hb + TK_IMG, lbp + TK_IMG, soff[i], z);
          continue;
        }
        // both raw chunks are read before either is rewritten (see tc_outer)
        float4 va = make_float4(0.f, 0.f, 0.f, 0.f), vb = va;
        if (r < rowsA) va = *reinterpret_cast<const float4*>(hb + soff[i]);
        if (r < rowsB) vb = *reinterpret_cast<const float4*>(hb + TK_IMG + soff[i]);
        if (second) {
          vb.x = -vb.x; vb.y = -vb.y; vb.z = -vb.z; vb.w = -vb.w;
        }
        if (r < rowsA) store_split4(hb, lbp, soff[i], va);
        // B rows past N keep an earlier tile's values: they only reach columns >= N, which the selection skips
        if (r < rowsB) store_split4(hb + TK_IMG, lbp + TK_IMG, soff[i], vb);
      }
      fence_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&full[seq % TK_SH]);
      const bool last = at == apt - 1;
      if (at % TK_DRAIN == TK_DRAIN - 1 || last) drain(seq, at % TK_DRAIN + 1);
      if (last) {   // the tile's scores of this thread's row enter the row's list, first half 0, then half 1
        const int grow = n0 + nrow, cbase = tile * TK_TILE + col0;
        for (int turn = 0; turn < 2; ++turn) {
          if (turn == half && nrow < rowsA) {
            float ts = ls[k - 1];
            int tc = lc[k - 1];
#pragma unroll
            for (int ch = 0; ch < 8; ++ch)
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                const int c = cbase + ch * 8 + i;
                // S[n][n] = 0 exactly; a NaN score (NaN or inf in U / V) ranks as -inf, so it loses every comparison
                // it can lose and the column tie rule still fills the list with valid columns
                const float v = acc[ch][i];
                const float s = c == grow ? 0.f : (v != v ? -INFINITY : v);
                if (c < N && tk_better(s, c, ts, tc)) {
                  tk_insert(ls, lc, k, s, c);
                  ts = ls[k - 1];
                  tc = lc[k - 1];
                }
              }
          }
          asm volatile("bar.sync 1, 256;" ::: "memory");
        }
#pragma unroll
        for (int ch = 0; ch < 8; ++ch)
#pragma unroll
          for (int i = 0; i < 8; ++i) acc[ch][i] = 0.f;
      }
      if (++at == apt) {
        at = 0;
        ++tile;
      }
    }
    cp_async_wait<0>();

    if (half == 0 && nrow < rowsA) {   // the last tile's barrier has passed: the list is complete
      const size_t o = ((size_t)blockIdx.y * p.n_rows + (n0 - p.row0) + nrow) * k;
      for (int i = 0; i < k; ++i) {
        ws_s[o + i] = ls[i];
        ws_c[o + i] = lc[i];
      }
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, 512u);
}

__global__ void __launch_bounds__(128)
pair_topk_merge_kernel(const float* __restrict__ ws_s, const int* __restrict__ ws_c, int n_rows, int nseg, int k,
                       int32_t* __restrict__ cols, float* __restrict__ scores) {
  __shared__ float Ms[128 * TK_LD];
  __shared__ int Mc[128 * TK_LD];
  const int n = (int)(blockIdx.x * blockDim.x + threadIdx.x);
  if (n >= n_rows) return;
  float* ls = Ms + threadIdx.x * TK_LD;
  int* lc = Mc + threadIdx.x * TK_LD;
  for (int i = 0; i < k; ++i) {   // segment 0's list is sorted already
    ls[i] = ws_s[(size_t)n * k + i];
    lc[i] = ws_c[(size_t)n * k + i];
  }
  for (int sg = 1; sg < nseg; ++sg) {
    const size_t o = ((size_t)sg * n_rows + n) * k;
    for (int i = 0; i < k; ++i) {
      const float s = ws_s[o + i];
      const int c = ws_c[o + i];
      if (!tk_better(s, c, ls[k - 1], lc[k - 1])) break;   // a segment's list is sorted: nothing after it beats it
      tk_insert(ls, lc, k, s, c);
    }
  }
  // ascending column order: entry i goes to the position of its rank among the k columns
  for (int i = 0; i < k; ++i) {
    const int c = lc[i];
    int rank = 0;
    for (int j = 0; j < k; ++j) rank += lc[j] < c ? 1 : 0;
    cols[(size_t)n * k + rank] = c;
    if (scores) scores[(size_t)n * k + rank] = ls[i];
  }
}

namespace {
struct TopkGeom {
  int rblocks, ntiles, tiles_per_seg, nseg;
};
// Row blocks alone fill the device when there are at least twice as many as SMs (config 4: 512); otherwise the column
// range is split into segments until the grid does (config 3, N = 4,096: 32 row blocks x 8 segments of 4 tiles; config
// 4 with a rank's n_rows = N / 8: 64 row blocks x 5 segments).  Only the row blocks count: a rank selecting a block of
// rows still sweeps all ceil(N / 128) column tiles.
TopkGeom topk_geom(int N, int n_rows) {
  TopkGeom g;
  g.rblocks = ceil_div(n_rows, TK_TILE);
  g.ntiles = ceil_div(N, TK_TILE);
  int nseg = ceil_div(2 * device_sm_count(), g.rblocks);
  if (nseg < 1) nseg = 1;
  if (nseg > g.ntiles) nseg = g.ntiles;
  g.tiles_per_seg = ceil_div(g.ntiles, nseg);
  g.nseg = ceil_div(g.ntiles, g.tiles_per_seg);
  return g;
}
}  // namespace

size_t pair_topk_ws_bytes(int N, int n_rows, int k) {
  if (n_rows == 0) return 0;
  return (size_t)topk_geom(N, n_rows).nseg * n_rows * k * (sizeof(float) + sizeof(int));
}

int launch_pair_topk(int N, int width, const float* u, const float* v, int row0, int n_rows, int k, int32_t* cols,
                     float* scores, void* ws, cudaStream_t st) {
  if (n_rows == 0) return STC_OK;
  const TopkGeom g = topk_geom(N, n_rows);
  float* ws_s = static_cast<float*>(ws);
  int* ws_c = reinterpret_cast<int*>(ws_s + (size_t)g.nseg * n_rows * k);
  TopkPlan p;
  p.N = N;
  p.W = width;
  p.k = k;
  p.row0 = row0;
  p.n_rows = n_rows;
  p.aph = ceil_div(width, ATOM_K);
  p.ntiles = g.ntiles;
  p.tiles_per_seg = g.tiles_per_seg;
  STC_TRY(set_smem(tc_pair_topk_kernel, TK_SMEM));
  // compulsory HBM traffic: U and V read once (8 N W: every column row is a B operand; the block's A rows are among
  // them) and the [n_rows][k] columns and scores written (8 n_rows k); the A rows re-read for every tile and the
  // workspace lists stay in L2 at the shapes the benchmark runs
  const bool full = row0 == 0 && n_rows == N;
  ScopedKernelTimer _t(full ? KK_PAIR_TOPK : KK_PAIR_TOPK_ROWS, st, 8.0 * N * width + 8.0 * n_rows * k);
  tc_pair_topk_kernel<<<dim3(g.rblocks, g.nseg), TK_THREADS, TK_SMEM, st>>>(u, v, ws_s, ws_c, p);
  STC_LAUNCH_OK("tc_pair_topk_kernel");
  pair_topk_merge_kernel<<<ceil_div(n_rows, 128), 128, 0, st>>>(ws_s, ws_c, n_rows, g.nseg, k, cols, scores);
  STC_LAUNCH_OK("pair_topk_merge_kernel");
  return STC_OK;
}

}  // namespace stc
