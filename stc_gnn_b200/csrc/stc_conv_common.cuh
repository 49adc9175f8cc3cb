// Device/host helpers shared by the convolution kernels (FFMA general path and tcgen05 path).
#pragma once
#include "stc_common.cuh"

namespace stc {

constexpr int CV_THREADS = 256;
constexpr int CV_MAX_NI = 4;

// ---- tile geometry shared by host and device -----------------------------------------------------
struct ConvTile {
  int npt;     // nodes per tile
  int rows;    // npt * C
  int rowsP;   // rows rounded up to 4
  int L;       // Din + h
  int LP;      // odd-padded row stride of feature tiles
  int LP4;     // L rounded up to 4
  int HoutP;   // Hout rounded up to 4
};

static inline ConvTile make_tile(const ConvArgs& a, int rows_target) {
  ConvTile t;
  t.L = a.Din + a.h;
  t.LP = t.L | 1;
  t.LP4 = (t.L + 3) & ~3;
  t.HoutP = (a.Hout + 3) & ~3;
  t.npt = rows_target / a.C;
  if (t.npt < 1) t.npt = 1;
  long long total_nodes = (long long)a.B * a.N;
  if (t.npt > total_nodes) t.npt = (int)total_nodes;
  t.rows = t.npt * a.C;
  t.rowsP = (t.rows + 3) & ~3;
  return t;
}

// ---- device helpers -------------------------------------------------------------------------------
struct FeatSrc {
  const float* x0;
  long long x0_bs;
  const float* yx;
  const float* h0;
  const float* yh;
  int N, C, Din, h;
  long long R;  // B*N*C
};

__device__ __forceinline__ FeatSrc feat_src(const ConvArgs& a) {
  FeatSrc s;
  s.x0 = a.x0; s.x0_bs = a.x0_bs; s.yx = a.yx; s.h0 = a.h0; s.yh = a.yh;
  s.N = a.N; s.C = a.C; s.Din = a.Din; s.h = a.h;
  s.R = (long long)a.B * a.N * a.C;
  return s;
}

// dst[(node*C+cat)*ld + l] = k-th spatial term of [Xt | H-like] for nodes g0 .. g0+nodes_valid-1;
// rows >= nodes_valid*C up to rows_alloc are zero-filled.
__device__ inline void load_feat_tile(const FeatSrc& s, int k, long long g0, int nodes_valid, int rows_alloc, float* dst,
                               int ld) {
  const int L = s.Din + s.h;
  const int rows_valid = nodes_valid * s.C;
  // x-part
  {
    const int per_node = s.C * s.Din;
    const int total = nodes_valid * per_node;
    for (int idx = threadIdx.x; idx < total; idx += blockDim.x) {
      int node = idx / per_node, rem = idx - node * per_node;
      int cat = rem / s.Din, l = rem - cat * s.Din;
      long long g = g0 + node;
      const float* src;
      if (k == 0) {
        long long b = g / s.N;
        src = s.x0 + b * s.x0_bs + (g - b * s.N) * per_node;
      } else {
        src = s.yx + (long long)(k - 1) * s.R * s.Din + g * per_node;
      }
      dst[(node * s.C + cat) * ld + l] = src[rem];
    }
  }
  // h-part
  {
    const float* base = (k == 0) ? s.h0 : s.yh + (long long)(k - 1) * s.R * s.h;
    base += g0 * s.C * s.h;
    const int total = rows_valid * s.h;
    for (int idx = threadIdx.x; idx < total; idx += blockDim.x) {
      int row = idx / s.h, l = idx - row * s.h;
      dst[row * ld + s.Din + l] = base[idx];
    }
  }
  // zero the tail rows
  const int tail = (rows_alloc - rows_valid) * L;
  for (int idx = threadIdx.x; idx < tail; idx += blockDim.x) {
    int row = rows_valid + idx / L, l = idx % L;
    dst[row * ld + l] = 0.f;
  }
}

// dst[(node,d)][l] = sum_c' Qc[c'*C + d] * src[(node,c')][l]      (apply Qc^T on the category axis)
__device__ inline void mix_tile(const float* src, float* dst, const float* Qc, int rows, int C, int L, int ld) {
  const int total = rows * L;
  for (int idx = threadIdx.x; idx < total; idx += blockDim.x) {
    int row = idx / L, l = idx - row * L;
    int node = row / C, d = row - node * C;
    const float* sp = src + node * C * ld + l;
    float acc = 0.f;
    for (int c = 0; c < C; ++c) acc = fmaf(Qc[c * C + d], sp[c * ld], acc);
    dst[row * ld + l] = acc;
  }
}

// dst[(node,c')][l] += sum_d Qc[c'*C + d] * src[(node,d)][l]      (adjoint of mix_tile)
__device__ inline void unmix_add_tile(const float* src, float* dst, const float* Qc, int rows, int C, int L, int ld) {
  const int total = rows * L;
  for (int idx = threadIdx.x; idx < total; idx += blockDim.x) {
    int row = idx / L, l = idx - row * L;
    int node = row / C, cp = row - node * C;
    const float* sp = src + node * C * ld + l;
    float acc = 0.f;
    for (int d = 0; d < C; ++d) acc = fmaf(Qc[cp * C + d], sp[d * ld], acc);
    dst[row * ld + l] += acc;
  }
}

__device__ __forceinline__ float sigmoidf_acc(float x) { return 1.f / (1.f + expf(-x)); }
// MUFU.EX2 / MUFU.RCP forms for the tensor-core epilogues (7 instructions instead of ~45): relative error ~1e-6 for
// the sigmoid, absolute error ~2e-7 for tanh -- two orders below the parity tolerance (rtol 1e-4 + 1e-5 mean|ref|)
__device__ __forceinline__ float sigmoidf_fast(float x) { return __fdividef(1.f, 1.f + __expf(-x)); }
__device__ __forceinline__ float tanhf_fast(float x) { return __fdividef(2.f, 1.f + __expf(-2.f * x)) - 1.f; }

template <typename K>
static inline int set_smem(K kernel, size_t smem) {
  if (smem > 48 * 1024) STC_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  return STC_OK;
}

// phase trace of the tcgen05 kernels (stc_debug_trace_set): `tracing` / `trace_it` are locals of the kernel
#define STC_TRACE(slot)                                                                              \
  do {                                                                                               \
    if (tracing && trace_it < a.trace_tiles) a.trace[trace_it * TRACE_SLOTS + (slot)] = clock64();   \
  } while (0)

// deterministic mode: after a dx kernel that stored its bias / dT_c(Gc) partials into `grid` slots of a.det_ws
// ([Hout | (Kc-1)*C*C] floats each), their fixed-order sums are added into a.dbias and a.dQ[C*C..]
int det_reduce_dx(const ConvArgs& a, int grid, cudaStream_t st);

// tcgen05 path (stc_conv_tc.cu): returns STC_OK and sets *handled when it took the launch
int try_launch_conv_fwd_tc(const ConvArgs& a, cudaStream_t st, bool* handled);
int try_launch_conv_bwd_dx_tc(const ConvArgs& a, cudaStream_t st, bool* handled);
int try_launch_conv_bwd_dw_tc(const ConvArgs& a, cudaStream_t st, bool* handled);

}  // namespace stc
