// C ABI of libstc_b200.so (declared in include/stc_b200.h): argument checking, workspace layout and the
// launch sequence of one cell forward / backward on the general path.
#include "stc_common.cuh"

#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <mutex>
#include <vector>

namespace stc {

static thread_local char g_err[512] = "";
static thread_local int g_launches = 0;

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
void count_launch(int n) { g_launches += n; }
void reset_launch_count() { g_launches = 0; }

// ---- per-kernel timing record (process-wide, guarded; only touched when enabled) ----
struct TimedLaunch {
  int kind;
  double bytes;
  cudaEvent_t e0, e1;
};
static std::mutex g_tmu;
static std::atomic<bool> g_timing{false};
static std::vector<TimedLaunch> g_timed;
static std::vector<cudaEvent_t> g_event_pool;

static cudaEvent_t take_event() {   // g_tmu held
  if (!g_event_pool.empty()) {
    cudaEvent_t e = g_event_pool.back();
    g_event_pool.pop_back();
    return e;
  }
  cudaEvent_t e = nullptr;
  cudaEventCreate(&e);
  return e;
}

// The timer holds its own event pair (a concurrent stc_timing_collect cannot invalidate it) and appends the finished
// pair to the record in its destructor.  Nothing is recorded while the stream is being captured into a CUDA graph:
// events recorded during capture cannot be synchronised or timed afterwards.
ScopedKernelTimer::ScopedKernelTimer(int kind_, cudaStream_t st_, double alg_bytes)
    : e0(nullptr), e1(nullptr), kind(kind_), bytes(alg_bytes), st(st_) {
  if (!g_timing.load(std::memory_order_relaxed)) return;
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(st, &cap) != cudaSuccess || cap != cudaStreamCaptureStatusNone) {
    cudaGetLastError();
    return;
  }
  {
    std::lock_guard<std::mutex> lk(g_tmu);
    e0 = take_event();
    e1 = take_event();
  }
  if (!e0 || !e1 || cudaEventRecord(e0, st) != cudaSuccess) {
    std::lock_guard<std::mutex> lk(g_tmu);
    if (e0) g_event_pool.push_back(e0);
    if (e1) g_event_pool.push_back(e1);
    e0 = e1 = nullptr;
  }
}
ScopedKernelTimer::~ScopedKernelTimer() {
  if (!e0) return;
  const bool ok = cudaEventRecord(e1, st) == cudaSuccess;
  std::lock_guard<std::mutex> lk(g_tmu);
  if (ok) {
    g_timed.push_back(TimedLaunch{kind, bytes, e0, e1});
  } else {
    g_event_pool.push_back(e0);
    g_event_pool.push_back(e1);
  }
}

int device_sm_count() {
  static thread_local int cached_dev = -1, cached = 0;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 148;
  if (dev != cached_dev) {
    cudaDeviceProp p;
    if (cudaGetDeviceProperties(&p, dev) != cudaSuccess) return 148;
    cached = p.multiProcessorCount;
    cached_dev = dev;
  }
  return cached;
}

int check_arch() {
  static thread_local int ok_dev = -1;
  int dev = 0;
  STC_CUDA_OK(cudaGetDevice(&dev));
  if (dev == ok_dev) return STC_OK;
  int major = 0;
  STC_CUDA_OK(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  if (major != 10) {
    set_error("libstc_b200 is built for sm_100a only; device %d has compute capability major %d", dev, major);
    return STC_ERR_ARCH;
  }
  ok_dev = dev;
  return STC_OK;
}

// ---- tuning switches and the phase trace ----
static long long* g_trace_buf = nullptr;
static int g_trace_tiles = 0;
int conv_opt_flags() {
  static int cached = -1;
  if (cached < 0) {
    const char* e = getenv("STC_OPT");
    cached = (e && e[0]) ? (atoi(e) & 0x7fffffff) : OPT_L2_PREFETCH;   // default: measured-best switches
  }
  return cached;
}
void conv_trace_target(long long** buf, int* tiles) {
  *buf = g_trace_buf;
  *tiles = g_trace_tiles;
}

// ---- small-problem concurrency: independent kernels of one cell call on side streams ---------------------------------
// At the reference's own batch size (32 windows -> 128 row tiles) no kernel fills the 148 SMs and a cell backward is a
// chain of ten ~10 us launches.  Several of them are independent (dW needs only dx's output, the three dGs outer
// products and the adjoint hops of Xt / H touch disjoint buffers), so they are forked onto side streams with events and
// joined back before anything they read is overwritten: the critical path of a backward call drops from 10 to 4
// kernels.  Everything stays ordered after prior work on the caller's stream and is complete, as seen from that stream,
// when the call's last event wait has been enqueued; event fork/join is also what CUDA-graph capture expects.
// Large problems (every kernel fills the device) keep the single-stream order.  STC_CONCURRENCY=0 / 1 forces it off / on.
struct SidePool {
  int dev = -1;
  cudaStream_t side[4] = {nullptr, nullptr, nullptr, nullptr};
  cudaEvent_t ev[16] = {};
  int next_ev = 0;
  bool ok = false;
};
static thread_local SidePool g_pool;

static SidePool* side_pool() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return nullptr;
  SidePool& p = g_pool;
  if (p.dev != dev) {   // first use on this thread / device (streams of another device are simply left behind)
    p = SidePool();
    p.dev = dev;
    p.ok = true;
    for (auto& s_ : p.side) p.ok = p.ok && cudaStreamCreateWithFlags(&s_, cudaStreamNonBlocking) == cudaSuccess;
    for (auto& e : p.ev) p.ok = p.ok && cudaEventCreateWithFlags(&e, cudaEventDisableTiming) == cudaSuccess;
    if (!p.ok) cudaGetLastError();
  }
  return p.ok ? &p : nullptr;
}

static std::atomic<int> g_concurrency{-2};   // -2: not read yet; -1 auto, 0 off, 1 on
static int concurrency_mode() {
  int m = g_concurrency.load(std::memory_order_relaxed);
  if (m == -2) {
    const char* e = getenv("STC_CONCURRENCY");
    m = (e && e[0]) ? (atoi(e) != 0 ? 1 : 0) : -1;
    g_concurrency.store(m, std::memory_order_relaxed);
  }
  return m;
}

// Fork / join helper of one cell call.  Inactive (every stream() is the caller's stream, fork / join are no-ops) when the
// problem is large or the pool could not be created.
struct Lanes {
  cudaStream_t main;
  SidePool* pool;
  bool forked[4] = {false, false, false, false};
  Lanes(cudaStream_t st, const StcDims& d) : main(st), pool(nullptr) {
    const int mode = concurrency_mode();
    const long long rows = (long long)d.B * d.N * d.C;
    // measured on the SF stack (profiles/r3g_*): +4 % at B = 512 (256 K rows), -1 % at B = 4096; threshold ~ B = 600
    const bool small = rows * (d.Din + 2 * d.h) < (long long)device_sm_count() * 2 * 128 * 48 * 8;
    if (mode == 1 || (mode == -1 && small)) pool = side_pool();
  }
  bool active() const { return pool != nullptr; }
  cudaStream_t stream(int i) const { return pool ? pool->side[i] : main; }
  cudaEvent_t next_event() { cudaEvent_t e = pool->ev[pool->next_ev]; pool->next_ev = (pool->next_ev + 1) & 15; return e; }
  int fork_from(cudaStream_t src, int i) {   // side[i] additionally waits for everything queued on src so far
    if (!pool || src == pool->side[i]) return STC_OK;
    cudaEvent_t e = next_event();
    STC_CUDA_OK(cudaEventRecord(e, src));
    STC_CUDA_OK(cudaStreamWaitEvent(pool->side[i], e, 0));
    forked[i] = true;
    return STC_OK;
  }
  int fork(int i) { return fork_from(main, i); }   // side[i] continues from the caller's stream's current position
  int join(int i) {          // the caller's stream waits for everything queued on side[i]
    if (!pool || !forked[i]) return STC_OK;
    cudaEvent_t e = next_event();
    STC_CUDA_OK(cudaEventRecord(e, pool->side[i]));
    STC_CUDA_OK(cudaStreamWaitEvent(main, e, 0));
    forked[i] = false;
    return STC_OK;
  }
  int join_all() {
    for (int i = 0; i < 4; ++i) STC_TRY(join(i));
    return STC_OK;
  }
};

static std::atomic<int> g_det{0};
bool det_mode() { return g_det.load(std::memory_order_relaxed) != 0; }
// every dW / dx kernel with a fixed-order form runs at most two CTAs per SM
int det_conv_slots() { return 2 * device_sm_count(); }

WsLayout make_layout(const StcDims& d, bool fwd_only) {
  WsLayout w;
  const size_t A = 64;  // 256-byte alignment of every region
  w.R = (size_t)d.B * d.N * d.C;
  const size_t Rh = w.R * d.h, Rx = w.R * d.Din;
  const size_t km1 = d.Ks > 1 ? (size_t)(d.Ks - 1) : 0;
  const size_t bwd = fwd_only ? 0 : 1;   // regions only the backward reads
  size_t o = 0;
  auto take = [&](size_t n) { size_t at = o; o = round_up(o + n, A); return at; };
  w.u = take(Rh);
  w.r = take(bwd * Rh);
  w.c = take(bwd * Rh);
  w.Yr = take((size_t)d.Ks * Rh);   // Yr[0] = r*H, then its spatial terms
  w.Yx = take(km1 * Rx);
  w.Yh = take(km1 * Rh);
  w.Q = take((size_t)d.Kc * d.C * d.C);
  const size_t kcm1 = d.Kc > 1 ? (size_t)(d.Kc - 1) : 0;
  w.Pg = take(bwd * w.R * kcm1 * 2 * d.h);
  w.Pc = take(bwd * w.R * kcm1 * d.h);
  {  // weight images of the wide-hidden-state forward: only for shapes the SF-class tensor-core kernels do not take
    ConvArgs t;
    memset(&t, 0, sizeof(t));
    t.B = d.B; t.N = d.N; t.C = d.C; t.Din = d.Din; t.h = d.h; t.Ks = d.Ks; t.Kc = d.Kc;
    t.Hout = 2 * d.h;
    const bool small_g = conv_tc_eligible(t);
    t.Hout = d.h;
    const bool small_c = conv_tc_eligible(t);
    w.Wimg_g = take(small_g ? 0 : conv_big_img_floats(d.C, d.Din, d.h, d.Ks, d.Kc, 2 * d.h));
    w.Wimg_c = take(small_c ? 0 : conv_big_img_floats(d.C, d.Din, d.h, d.Ks, d.Kc, d.h));
  }
  w.saved_total = o;
  o = 0;
  w.dpre = take(w.R * 2 * d.h * d.Kc);   // tcgen05 path keeps the Kc unmixed copies side by side
  w.dYx0 = take(Rx);
  w.dYx = take(km1 * Rx);
  w.dYh = take(km1 * Rh);
  w.dYr = take((size_t)d.Ks * Rh);
  w.dQ = take((size_t)d.Kc * d.C * d.C);
  {  // weight image of the wide-state backward dx (candidate pass, then gates pass: stream-ordered reuse)
    const size_t ig = w.Wimg_c > w.Wimg_g ? conv_big_dx_img_floats(d.C, d.Din, d.h, d.Ks, d.Kc, 2 * d.h) : 0;
    const size_t ic = w.saved_total > w.Wimg_c ? conv_big_dx_img_floats(d.C, d.Din, d.h, d.Ks, d.Kc, d.h) : 0;
    w.Wimg_dx = take(ig > ic ? ig : ic);
  }
  {  // deterministic mode: partial slots of the cross-CTA reductions (after every region of the default layout)
    const bool det = det_mode();
    const size_t P = (size_t)d.Ks * d.Kc, L = (size_t)d.Din + d.h, S = det ? (size_t)det_conv_slots() : 0;
    size_t dw = S * P * L * 2 * d.h, dx = S * (2 * (size_t)d.h + (size_t)(d.Kc - 1) * d.C * d.C);
    if (det) {   // the general (FFMA) kernels: one slot per CTA (dx) / per row chunk and row group (dW)
      ConvArgs t;
      memset(&t, 0, sizeof(t));
      t.B = d.B; t.N = d.N; t.C = d.C; t.Din = d.Din; t.h = d.h; t.Ks = d.Ks; t.Kc = d.Kc;
      for (int hout : {2 * d.h, d.h}) {
        t.Hout = hout;
        dw = std::max(dw, conv_dw_general_det_floats(t));
        dx = std::max(dx, conv_dx_general_det_floats(t));
      }
    }
    w.det_dw = take(dw);
    w.det_dx = take(dx);
    long long g = 0;
    if (det)
      for (int width : {d.C * d.Din, d.C * d.h}) {
        const long long f = support_outer_det_floats(d.N, d.B, width);
        if (f > g) g = f;
      }
    w.det_dgs = take((size_t)g);
  }
  w.scratch_total = o;
  return w;
}

static int check_dims(const StcDims* d) {
  if (!d) {
    set_error("dims is NULL");
    return STC_ERR_BAD_ARG;
  }
  if (d->B < 0 || d->N <= 0 || d->C <= 0 || d->Din <= 0 || d->h <= 0 || d->Ks <= 0 || d->Kc <= 0) {
    set_error("bad dims B=%d N=%d C=%d Din=%d h=%d Ks=%d Kc=%d", d->B, d->N, d->C, d->Din, d->h, d->Ks, d->Kc);
    return STC_ERR_BAD_ARG;
  }
  if (d->act != STC_ACT_NONE && d->act != STC_ACT_RELU) {
    set_error("unsupported activation code %d (none=0, relu=1)", d->act);
    return STC_ERR_UNSUPPORTED;
  }
  if ((long long)d->B * d->N * d->C * (long long)(2 * d->h > d->Din ? 2 * d->h : d->Din) >= (1LL << 40)) {
    set_error("problem too large");
    return STC_ERR_UNSUPPORTED;
  }
  return STC_OK;
}

static ConvArgs base_args(const StcDims& d, const float* xt, int64_t xt_bs, const float* W, const float* Q,
                          float* ws, const WsLayout& w, int phase) {
  ConvArgs a;
  memset(&a, 0, sizeof(a));
  a.B = d.B; a.N = d.N; a.C = d.C; a.Din = d.Din; a.h = d.h; a.Ks = d.Ks; a.Kc = d.Kc;
  a.act = d.act;
  a.phase = phase;
  a.Hout = phase == 0 ? 2 * d.h : d.h;
  a.x0 = xt;
  a.x0_bs = xt_bs;
  a.yx = ws + w.Yx;
  a.W = W;
  a.Q = Q;
  // dx leaves [Ds | Dm_1 ...] side by side for the tensor-core dW kernels; the general path only the plain Ds
  a.opt = conv_opt_flags();
  const bool wide_bwd = !(a.opt & OPT_WIDE_DX_FFMA) && conv_big_bwd_shape_ok(a.C, a.Din, a.h, a.Ks, a.Kc, a.Hout);
  a.dpre_ld = (conv_tc_eligible(a) || wide_bwd) ? a.Kc * a.Hout : a.Hout;
  conv_trace_target(&a.trace, &a.trace_tiles);
  if (a.trace) a.trace += (size_t)phase * a.trace_tiles * TRACE_SLOTS;   // gates stamps first, candidate stamps after them
  return a;
}

}  // namespace stc

using namespace stc;

extern "C" {

int stc_timing_enable(int32_t on) {
  g_timing.store(on != 0);
  return STC_OK;
}

int stc_timing_collect(double* ms, int64_t* launches, double* bytes, int32_t n_kinds) {
  std::lock_guard<std::mutex> lk(g_tmu);
  for (auto& t : g_timed) {
    float m = 0.f;
    if (cudaEventSynchronize(t.e1) == cudaSuccess && cudaEventElapsedTime(&m, t.e0, t.e1) == cudaSuccess &&
        t.kind < n_kinds) {
      if (ms) ms[t.kind] += m;
      if (launches) launches[t.kind] += 1;
      if (bytes) bytes[t.kind] += t.bytes;
    }
    g_event_pool.push_back(t.e0);
    g_event_pool.push_back(t.e1);
  }
  g_timed.clear();
  return KK_COUNT;
}

const char* stc_kernel_kind_name(int32_t kind) {
  static const char* names[KK_COUNT] = {"support_dense", "support_csr", "support_outer", "cheby_small",
                                        "conv_fwd",      "conv_bwd_dx", "conv_bwd_dw", "tc_conv_fwd", "tc_conv_bwd_dx", "tc_conv_bwd_dw",
                                        "tc_support", "tc_gemm_test", "tc_outer", "tc_support_big", "support_csr_grad",
                                        "pair_scores_csr", "edge_softmax", "pair_topk", "tc_support_adj", "pair_topk_rows",
                                        "det_reduce"};
  return (kind >= 0 && kind < KK_COUNT) ? names[kind] : "?";
}

int stc_debug_trace_set(void* dev_buf, int64_t n_slots) {
  std::lock_guard<std::mutex> lk(g_tmu);
  g_trace_buf = (long long*)dev_buf;
  g_trace_tiles = dev_buf ? (int)(n_slots / (2 * TRACE_SLOTS)) : 0;
  return STC_OK;
}

int stc_concurrency_set(int32_t mode) {
  if (mode < -1 || mode > 1) {
    set_error("stc_concurrency_set: mode %d (use -1 = by problem size, 0 = one stream, 1 = always fork)", mode);
    return STC_ERR_BAD_ARG;
  }
  g_concurrency.store(mode, std::memory_order_relaxed);
  return STC_OK;
}

int stc_deterministic_set(int32_t on) {
  if (on != 0 && on != 1) {
    set_error("stc_deterministic_set: %d (use 0 = atomics, 1 = fixed-order reductions)", on);
    return STC_ERR_BAD_ARG;
  }
  g_det.store(on, std::memory_order_relaxed);
  return STC_OK;
}

int stc_abi_version(void) { return STC_ABI_VERSION; }
const char* stc_last_error(void) { return g_err; }
int stc_last_launch_count(void) { return g_launches; }

size_t stc_cell_saved_bytes(const StcDims* d) {
  if (check_dims(d) != STC_OK) return 0;
  return make_layout(*d).saved_total * sizeof(float);
}
size_t stc_cell_bwd_scratch_bytes(const StcDims* d) {
  if (check_dims(d) != STC_OK) return 0;
  return make_layout(*d).scratch_total * sizeof(float);
}

int stc_support_apply(const StcSupport* gs, int32_t N, int32_t B, int32_t width, int32_t transpose,
                      const float* x, int64_t x_batch_stride, const float* z, int64_t z_batch_stride, float* y,
                      float alpha, float beta, void* stream) {
  reset_launch_count();
  if (!gs || !x || !y) {
    set_error("stc_support_apply: NULL argument");
    return STC_ERR_BAD_ARG;
  }
  STC_TRY(check_arch());
  return launch_support_apply(*gs, N, B, width, transpose != 0, x, x_batch_stride, z, z_batch_stride, y, alpha,
                              beta, nullptr, 0.f, (cudaStream_t)stream);
}

int stc_support_apply_rows(const StcSupport* gs, int32_t N, int32_t B, int32_t width, int32_t transpose, const float* x,
                           int64_t x_batch_stride, const float* z, int64_t z_batch_stride, float* y, float alpha,
                           float beta, const int32_t* rows, int32_t n_rows, void* stream) {
  reset_launch_count();
  if (!gs || !x || !y || !rows) {
    set_error("stc_support_apply_rows: NULL argument");
    return STC_ERR_BAD_ARG;
  }
  if (gs->kind == STC_SUPPORT_CSR_PER_SAMPLE) {
    set_error("stc_support_apply_rows: a per-sample CSR support (STC_SUPPORT_CSR_PER_SAMPLE) takes no row list");
    return STC_ERR_UNSUPPORTED;
  }
  if (n_rows < 0 || n_rows > N) {
    set_error("stc_support_apply_rows: n_rows %d outside [0, N = %d]", n_rows, N);
    return STC_ERR_BAD_ARG;
  }
  STC_TRY(check_arch());
  return launch_support_apply(*gs, N, B, width, transpose != 0, x, x_batch_stride, z, z_batch_stride, y, alpha, beta,
                              nullptr, 0.f, (cudaStream_t)stream, rows, n_rows);
}

int stc_halo_pack(const float* x_ext, int64_t x_batch_stride, int32_t width, int32_t B, const int32_t* idx, int32_t n_rows,
                  float* send, void* stream) {
  reset_launch_count();
  if (n_rows > 0 && (!x_ext || !idx || !send)) {
    set_error("stc_halo_pack: NULL argument");
    return STC_ERR_BAD_ARG;
  }
  STC_TRY(check_arch());
  return launch_halo_rows(true, const_cast<float*>(x_ext), x_batch_stride, width, B, idx, 0, n_rows, send, (cudaStream_t)stream);
}

int stc_halo_unpack(const float* recv, int32_t width, int32_t B, int32_t row0, int32_t n_rows, float* x_ext,
                    int64_t x_batch_stride, void* stream) {
  reset_launch_count();
  if (n_rows > 0 && (!x_ext || !recv)) {
    set_error("stc_halo_unpack: NULL argument");
    return STC_ERR_BAD_ARG;
  }
  STC_TRY(check_arch());
  return launch_halo_rows(false, x_ext, x_batch_stride, width, B, nullptr, row0, n_rows, const_cast<float*>(recv), (cudaStream_t)stream);
}

int stc_tf32x3_gemm(const float* a, const float* b, float* d, int32_t M, int32_t N, int32_t K, void* stream) {
  reset_launch_count();
  if (!a || !b || !d) {
    set_error("stc_tf32x3_gemm: NULL argument");
    return STC_ERR_BAD_ARG;
  }
  STC_TRY(check_arch());
  return launch_tf32x3_gemm(a, b, d, M, N, K, (cudaStream_t)stream);
}

// ---- forward pieces (stc_cell_fwd runs all four; the row-partitioned path runs the two node-local ones and does
//      the spatial hops itself, with a halo exchange before each) ----
struct FwdCtx {
  const StcDims& d;
  const WsLayout& w;
  const StcSupport* gs;
  const float* gc;
  const float* xt;
  int64_t xt_bs;
  const float* h_prev;
  float* ws;
  cudaStream_t st;
  Lanes* lanes = nullptr;   // set by stc_cell_fwd: the Xt-side terms and the Gc terms may run beside the H-side terms
  const float* yx_pre = nullptr;   // caller-supplied spatial terms of Xt ([Ks-1][B][N][C][Din]): skip the Xt-side hops
  const float* yh_pre = nullptr;   // caller-supplied spatial terms of H ([Ks-1][B][N][C][h]): skip the H-side hops
  bool fwd_only = false;   // `ws` has the forward-only layout: r, c and the P_1 partials (backward-only) are not stored
};

// spatial Chebyshev terms of Xt and H:  Y_1 = Gs^T Y_0,  Y_k = 2 Gs^T Y_{k-1} - Y_{k-2}
static int fwd_terms_xh(const FwdCtx& f) {
  const StcDims& d = f.d;
  const WsLayout& w = f.w;
  float* ws = f.ws;
  const size_t Rh = w.R * d.h, Rx = w.R * d.Din;
  const int CD = d.C * d.Din, CH = d.C * d.h;
  const long long nbs_h = (long long)d.N * CH;
  // the two recurrences are independent of each other: Xt's on side stream 0 (when lanes are active), H's on the caller's
  cudaStream_t sx = f.st;
  if (f.lanes && f.lanes->active() && d.Ks > 1 && !f.yx_pre && !f.yh_pre) {
    STC_TRY(f.lanes->fork(0));
    sx = f.lanes->stream(0);
  }
  for (int k = 1; k < d.Ks && !f.yx_pre; ++k) {
    const float alpha = k == 1 ? 1.f : 2.f, beta = k == 1 ? 0.f : -1.f;
    const float* xin = k == 1 ? f.xt : ws + w.Yx + (size_t)(k - 2) * Rx;
    const int64_t xin_bs = k == 1 ? f.xt_bs : (int64_t)d.N * CD;
    const float* xz = k == 1 ? nullptr : (k == 2 ? f.xt : ws + w.Yx + (size_t)(k - 3) * Rx);
    const int64_t xz_bs = k == 2 ? f.xt_bs : (int64_t)d.N * CD;
    STC_TRY(launch_support_apply(*f.gs, d.N, d.B, CD, true, xin, xin_bs, xz, xz_bs, ws + w.Yx + (size_t)(k - 1) * Rx,
                                 alpha, beta, nullptr, 0.f, sx));
  }
  for (int k = 1; k < d.Ks && !f.yh_pre; ++k) {
    const float alpha = k == 1 ? 1.f : 2.f, beta = k == 1 ? 0.f : -1.f;
    const float* hin = k == 1 ? f.h_prev : ws + w.Yh + (size_t)(k - 2) * Rh;
    const float* hz = k == 1 ? nullptr : (k == 2 ? f.h_prev : ws + w.Yh + (size_t)(k - 3) * Rh);
    STC_TRY(launch_support_apply(*f.gs, d.N, d.B, CH, true, hin, nbs_h, hz, nbs_h, ws + w.Yh + (size_t)(k - 1) * Rh,
                                 alpha, beta, nullptr, 0.f, f.st));
  }
  if (f.lanes) STC_TRY(f.lanes->join(0));
  return STC_OK;
}

// gates:  [u|r] = sigmoid(conv([Xt,H])),  rH = r*H   (also builds the Chebyshev terms of Gc)
static int fwd_gates(const FwdCtx& f, const float* Wg, const float* bg) {
  const StcDims& d = f.d;
  const WsLayout& w = f.w;
  float* ws = f.ws;
  if (d.Kc > 1) STC_TRY(launch_cheby_small(f.gc, d.C, d.Kc, ws + w.Q, f.st));
  ConvArgs a = base_args(d, f.xt, f.xt_bs, Wg, ws + w.Q, ws, w, 0);
  if (f.yx_pre) a.yx = f.yx_pre;
  a.h0 = f.h_prev;
  a.yh = f.yh_pre ? f.yh_pre : ws + w.Yh;
  a.bias = d.has_bias ? bg : nullptr;
  a.Hprev = f.h_prev;
  a.u = ws + w.u;
  a.r = f.fwd_only ? nullptr : ws + w.r;
  a.rH = ws + w.Yr;
  a.Psave = f.fwd_only ? nullptr : ws + w.Pg;
  a.Wimg = (w.Wimg_c > w.Wimg_g) ? ws + w.Wimg_g : nullptr;   // region is empty when the shape is not eligible
  return launch_conv_fwd(a, f.st);
}

// spatial terms of r*H
static int fwd_terms_rh(const FwdCtx& f) {
  const StcDims& d = f.d;
  const WsLayout& w = f.w;
  float* ws = f.ws;
  const size_t Rh = w.R * d.h;
  const int CH = d.C * d.h;
  const long long nbs_h = (long long)d.N * CH;
  for (int k = 1; k < d.Ks; ++k) {
    const float alpha = k == 1 ? 1.f : 2.f, beta = k == 1 ? 0.f : -1.f;
    const float* in = ws + w.Yr + (size_t)(k - 1) * Rh;
    const float* z = k == 1 ? nullptr : ws + w.Yr + (size_t)(k - 2) * Rh;
    STC_TRY(launch_support_apply(*f.gs, d.N, d.B, CH, true, in, nbs_h, z, nbs_h, ws + w.Yr + (size_t)k * Rh, alpha, beta,
                                 nullptr, 0.f, f.st));
  }
  return STC_OK;
}

// candidate:  c = tanh(conv([Xt, rH])),  H' = (1-u) H + u c
static int fwd_candi(const FwdCtx& f, const float* Wc, const float* bc, float* h_out) {
  const StcDims& d = f.d;
  const WsLayout& w = f.w;
  float* ws = f.ws;
  const size_t Rh = w.R * d.h;
  ConvArgs a = base_args(d, f.xt, f.xt_bs, Wc, ws + w.Q, ws, w, 1);
  if (f.yx_pre) a.yx = f.yx_pre;
  a.h0 = ws + w.Yr;
  a.yh = ws + w.Yr + Rh;
  a.bias = d.has_bias ? bc : nullptr;
  a.Hprev = f.h_prev;
  a.u = ws + w.u;
  a.c = f.fwd_only ? nullptr : ws + w.c;
  a.Hnew = h_out;
  a.Psave = f.fwd_only ? nullptr : ws + w.Pc;
  a.Wimg = (w.saved_total > w.Wimg_c) ? ws + w.Wimg_c : nullptr;
  return launch_conv_fwd(a, f.st);
}

static int check_fwd_args(const StcDims* dp, const float* gc, const float* xt, const float* h_prev, const float* Wg,
                          const float* bg, const float* Wc, const float* bc, float* h_out, void* wsv, size_t ws_bytes,
                          const char* who, bool fwd_only = false) {
  STC_TRY(check_dims(dp));
  if (!gc || !xt || !h_prev || !Wg || !Wc || !h_out || !wsv) {
    set_error("%s: NULL argument", who);
    return STC_ERR_BAD_ARG;
  }
  if (dp->has_bias && (!bg || !bc)) {
    set_error("%s: has_bias set but bias pointer is NULL", who);
    return STC_ERR_BAD_ARG;
  }
  const WsLayout w = make_layout(*dp, fwd_only);
  if (ws_bytes < w.saved_total * sizeof(float)) {
    if (fwd_only)
      set_error("%s: workspace too small (STC_ERR_WORKSPACE): %zu < %zu bytes (stc_cell_fwd_only_bytes)", who, ws_bytes,
                w.saved_total * sizeof(float));
    else
      set_error("saved buffer too small: %zu < %zu bytes", ws_bytes, w.saved_total * sizeof(float));
    return STC_ERR_WORKSPACE;
  }
  return STC_OK;
}

static int cell_fwd_impl(const StcDims* dp, const StcSupport* gs, const float* gc, const float* xt,
                         int64_t xt_batch_stride, const float* h_prev, const float* Wg, const float* bg, const float* Wc,
                         const float* bc, float* h_out, void* wsv, size_t ws_bytes, const float* yx_terms,
                         const float* yh_terms, void* stream, const char* who, bool fwd_only = false) {
  reset_launch_count();
  STC_TRY(check_fwd_args(dp, gc, xt, h_prev, Wg, bg, Wc, bc, h_out, wsv, ws_bytes, who, fwd_only));
  if (!gs) {
    set_error("%s: NULL support", who);
    return STC_ERR_BAD_ARG;
  }
  const StcDims& d = *dp;
  if (d.B == 0) return STC_OK;
  STC_TRY(check_arch());
  const WsLayout w = make_layout(d, fwd_only);
  Lanes lanes((cudaStream_t)stream, d);
  FwdCtx f{d, w, gs, gc, xt, xt_batch_stride, h_prev, (float*)wsv, (cudaStream_t)stream};
  f.lanes = &lanes;
  f.fwd_only = fwd_only;
  f.yx_pre = d.Ks > 1 ? yx_terms : nullptr;
  f.yh_pre = d.Ks > 1 ? yh_terms : nullptr;
  STC_TRY(fwd_terms_xh(f));
  STC_TRY(fwd_gates(f, Wg, bg));
  STC_TRY(fwd_terms_rh(f));
  STC_TRY(fwd_candi(f, Wc, bc, h_out));
  return STC_OK;
}

int stc_cell_fwd(const StcDims* dp, const StcSupport* gs, const float* gc, const float* xt,
                 int64_t xt_batch_stride, const float* h_prev, const float* Wg, const float* bg, const float* Wc,
                 const float* bc, float* h_out, void* wsv, size_t ws_bytes, void* stream) {  // wsv = `saved`
  return cell_fwd_impl(dp, gs, gc, xt, xt_batch_stride, h_prev, Wg, bg, Wc, bc, h_out, wsv, ws_bytes, nullptr, nullptr,
                       stream, "stc_cell_fwd");
}

int stc_cell_fwd_x(const StcDims* dp, const StcSupport* gs, const float* gc, const float* xt,
                   int64_t xt_batch_stride, const float* h_prev, const float* Wg, const float* bg, const float* Wc,
                   const float* bc, float* h_out, void* wsv, size_t ws_bytes, const float* yx_terms,
                   const float* yh_terms, void* stream) {
  return cell_fwd_impl(dp, gs, gc, xt, xt_batch_stride, h_prev, Wg, bg, Wc, bc, h_out, wsv, ws_bytes, yx_terms, yh_terms,
                       stream, "stc_cell_fwd_x");
}

int stc_cell_saved_layout(const StcDims* dp, int64_t* offsets, int32_t n_offsets) {
  STC_TRY(check_dims(dp));
  if (!offsets || n_offsets < STC_SAVED_REGIONS) {
    set_error("stc_cell_saved_layout: need room for %d offsets", (int)STC_SAVED_REGIONS);
    return STC_ERR_BAD_ARG;
  }
  const WsLayout w = make_layout(*dp);
  const size_t v[STC_SAVED_REGIONS] = {w.u, w.r, w.c, w.Yr, w.Yx, w.Yh, w.Q, w.Pg, w.Pc};
  for (int i = 0; i < STC_SAVED_REGIONS; ++i) offsets[i] = (int64_t)v[i];
  return STC_OK;
}

static int cell_fwd_stage_impl(const StcDims* dp, int32_t stage, const float* gc, const float* xt,
                               int64_t xt_batch_stride, const float* h_prev, const float* Wg, const float* bg,
                               const float* Wc, const float* bc, float* h_out, void* wsv, size_t ws_bytes, void* stream,
                               const char* who, bool fwd_only) {
  reset_launch_count();
  STC_TRY(check_fwd_args(dp, gc, xt, h_prev, Wg, bg, Wc, bc, h_out, wsv, ws_bytes, who, fwd_only));
  if (stage != STC_STAGE_GATES && stage != STC_STAGE_CANDI) {
    set_error("%s: bad stage %d", who, stage);
    return STC_ERR_BAD_ARG;
  }
  const StcDims& d = *dp;
  if (d.B == 0) return STC_OK;
  STC_TRY(check_arch());
  const WsLayout w = make_layout(d, fwd_only);
  FwdCtx f{d, w, nullptr, gc, xt, xt_batch_stride, h_prev, (float*)wsv, (cudaStream_t)stream};
  f.fwd_only = fwd_only;
  return stage == STC_STAGE_GATES ? fwd_gates(f, Wg, bg) : fwd_candi(f, Wc, bc, h_out);
}

int stc_cell_fwd_stage(const StcDims* dp, int32_t stage, const float* gc, const float* xt, int64_t xt_batch_stride,
                       const float* h_prev, const float* Wg, const float* bg, const float* Wc, const float* bc,
                       float* h_out, void* wsv, size_t ws_bytes, void* stream) {
  return cell_fwd_stage_impl(dp, stage, gc, xt, xt_batch_stride, h_prev, Wg, bg, Wc, bc, h_out, wsv, ws_bytes, stream,
                             "stc_cell_fwd_stage", false);
}

// ---- forward-only calls: the same launches on the smaller workspace of make_layout(d, true) ----
size_t stc_cell_fwd_only_bytes(const StcDims* d) {
  if (check_dims(d) != STC_OK) return 0;
  return make_layout(*d, true).saved_total * sizeof(float);
}

int stc_cell_fwd_only_layout(const StcDims* dp, int64_t* offsets, int32_t n_offsets) {
  STC_TRY(check_dims(dp));
  if (!offsets || n_offsets < STC_SAVED_REGIONS) {
    set_error("stc_cell_fwd_only_layout: need room for %d offsets", (int)STC_SAVED_REGIONS);
    return STC_ERR_BAD_ARG;
  }
  const WsLayout w = make_layout(*dp, true);
  const int64_t v[STC_SAVED_REGIONS] = {(int64_t)w.u, -1, -1, (int64_t)w.Yr, (int64_t)w.Yx, (int64_t)w.Yh,
                                        (int64_t)w.Q, -1, -1};
  for (int i = 0; i < STC_SAVED_REGIONS; ++i) offsets[i] = v[i];
  return STC_OK;
}

int stc_cell_fwd_only(const StcDims* dp, const StcSupport* gs, const float* gc, const float* xt,
                      int64_t xt_batch_stride, const float* h_prev, const float* Wg, const float* bg, const float* Wc,
                      const float* bc, float* h_out, void* wsv, size_t ws_bytes, const float* yx_terms,
                      const float* yh_terms, void* stream) {
  return cell_fwd_impl(dp, gs, gc, xt, xt_batch_stride, h_prev, Wg, bg, Wc, bc, h_out, wsv, ws_bytes, yx_terms, yh_terms,
                       stream, "stc_cell_fwd_only", true);
}

int stc_cell_fwd_only_stage(const StcDims* dp, int32_t stage, const float* gc, const float* xt, int64_t xt_batch_stride,
                            const float* h_prev, const float* Wg, const float* bg, const float* Wc, const float* bc,
                            float* h_out, void* wsv, size_t ws_bytes, void* stream) {
  return cell_fwd_stage_impl(dp, stage, gc, xt, xt_batch_stride, h_prev, Wg, bg, Wc, bc, h_out, wsv, ws_bytes, stream,
                             "stc_cell_fwd_only_stage", true);
}

// reverse of the feature-side recurrence Y_k = 2 A^T Y_{k-1} - Y_{k-2} (Y_1 = A^T Y_0) for one operand:
//   ybar[k-1] += (k>=2 ? 2 : 1) * Gs * ybar[k];  ybar[k-2] -= ybar[k];  dGs += coef * Y_{k-1} (x) ybar[k]
// For a CSR support dGs is the [nnz] gradient of its edge values, and that product is only needed at the edges: the
// adjoint hop already gathers every ybar[k][b,m,:] it needs, so the hop computes it (launch_support_csr_edge_grad).
static int adjoint_chain(const StcDims& d, const StcSupport& gs, int width, const float* y0, int64_t y0_bs,
                         const float* yk /* terms k>=1, contiguous */, float* ybar0, float* ybark /* k>=1 */,
                         float* dGs, cudaStream_t st, Lanes* lanes = nullptr, int outer_lane = 1,
                         float* det_dgs = nullptr) {
  const size_t Rw = (size_t)d.B * d.N * width;
  const int64_t nbs = (int64_t)d.N * width;
  for (int k = d.Ks - 1; k >= 1; --k) {
    const float coef = k >= 2 ? 2.f : 1.f;
    float* yb_k = ybark + (size_t)(k - 1) * Rw;
    float* yb_km1 = k == 1 ? ybar0 : ybark + (size_t)(k - 2) * Rw;
    float* axpy = nullptr;
    if (k >= 2) axpy = k == 2 ? ybar0 : ybark + (size_t)(k - 3) * Rw;
    if (dGs && is_csr_kind(gs.kind)) {
      const float* yprev = k == 1 ? y0 : yk + (size_t)(k - 2) * Rw;
      const int64_t yprev_bs = k == 1 ? y0_bs : nbs;
      STC_TRY(launch_support_csr_edge_grad(gs, d.N, d.B, width, yb_k, nbs, yb_km1, nbs, yb_km1, coef, 1.f, axpy, -1.f,
                                           yprev, yprev_bs, coef, dGs, st));
      continue;
    }
    if (dGs) {
      const float* yprev = k == 1 ? y0 : yk + (size_t)(k - 2) * Rw;
      const int64_t yprev_bs = k == 1 ? y0_bs : nbs;
      // One pass over ybar[k] for both of its readers (dense N <= 112).  Not when the lanes are active: there the outer
      // product runs beside the hops, off the critical path that fusing would lengthen.
      if (gs.kind == STC_SUPPORT_DENSE && gs.vals && !(lanes && lanes->active())) {
        bool handled = false;
        STC_TRY(try_launch_support_adj_tc(gs.vals, d.N, d.B, width, yb_k, nbs, yb_km1, axpy, yprev, yprev_bs, coef, dGs,
                                          st, &handled));
        if (handled) continue;
      }
      // the outer product only READS ybar[k] (final once the previous hop on `st` is queued) and Y[k-1]; nothing later in
      // the chain writes either, so it runs beside the hops on the outer lane and is joined at the end of the call
      cudaStream_t so = st;
      if (lanes && lanes->active()) {
        STC_TRY(lanes->fork_from(st, outer_lane));
        so = lanes->stream(outer_lane);
      }
      STC_TRY(launch_support_outer(d.N, d.B, width, yprev, yprev_bs, yb_k, coef, dGs, so, det_dgs));
    }
    STC_TRY(launch_support_apply(gs, d.N, d.B, width, false, yb_k, nbs, yb_km1, nbs, yb_km1, coef, 1.f, axpy, -1.f,
                                 st));
  }
  return STC_OK;
}

// ---- backward pieces (stc_cell_bwd runs all of them; the row-partitioned path runs the two node-local stages and
//      does the adjoint spatial hops itself, with a halo exchange before each) ----
struct BwdCtx {
  const StcDims& d;
  const WsLayout& w;
  const float* gc;
  const float* xt;
  int64_t xt_bs;
  const float* h_prev;
  const float* d_h_out;
  float* d_xt;        // may be NULL: the x-part adjoint then lives in scratch
  float* d_h_prev;
  float* dGc;
  float* sv;          // saved (read-only here)
  float* sc;          // scratch
  cudaStream_t st;
  Lanes* lanes = nullptr;   // set by stc_cell_bwd: dW runs beside the adjoint hops on side stream 0
  const float* yx_pre = nullptr;   // caller-supplied spatial terms of Xt (as in forward)
  float* dyx_out = nullptr;        // caller's buffer for the x-part adjoints of terms k >= 1 (the caller folds them)
  const float* yh_pre = nullptr;   // the same for H
  float* dyh_out = nullptr;
  const float* dyx_fold = nullptr; // adjoints of this call's own Xt-side terms k >= 1 from another reader: folded in
  const float* dyh_fold = nullptr; //   the dx epilogue before the adjoint chain of that side
  bool want_dGc() const { return dGc != nullptr && d.Kc > 1; }
  float* dYx0() const { return d_xt ? d_xt : sc + w.dYx0; }
};

static int check_bwd_args(const StcDims* dp, const float* gc, const float* xt, const float* h_prev, const float* Wg,
                          const float* Wc, const float* d_h_out, float* d_h_prev, float* dWg, float* dbg, float* dWc,
                          float* dbc, const void* savedv, size_t saved_bytes, void* scratchv, size_t scratch_bytes,
                          const char* who) {
  STC_TRY(check_dims(dp));
  const StcDims& d = *dp;
  if (!gc || !xt || !h_prev || !Wg || !Wc || !d_h_out || !d_h_prev || !dWg || !dWc || !savedv || !scratchv) {
    set_error("%s: NULL argument", who);
    return STC_ERR_BAD_ARG;
  }
  if (d.has_bias && (!dbg || !dbc)) {
    set_error("%s: has_bias set but a bias-gradient pointer is NULL", who);
    return STC_ERR_BAD_ARG;
  }
  const WsLayout w = make_layout(d);
  if (saved_bytes < w.saved_total * sizeof(float) || scratch_bytes < w.scratch_total * sizeof(float)) {
    set_error("buffers too small: saved %zu (need %zu), scratch %zu (need %zu) bytes", saved_bytes,
              w.saved_total * sizeof(float), scratch_bytes, w.scratch_total * sizeof(float));
    return STC_ERR_WORKSPACE;
  }
  return STC_OK;
}

// zero the parameter / support gradients unless the caller accumulates over a time loop; zero the dT_k(Gc) partials
// (dGs holds dGs_floats: N*N for a dense support, nnz for a CSR support)
static int bwd_begin(const BwdCtx& b, float* dWg, float* dbg, float* dWc, float* dbc, float* dGs, size_t dGs_floats,
                     int accumulate_params) {
  const StcDims& d = b.d;
  const int L = d.Din + d.h, P = d.Ks * d.Kc;
  if (!accumulate_params) {
    STC_CUDA_OK(cudaMemsetAsync(dWg, 0, sizeof(float) * P * L * 2 * d.h, b.st));
    STC_CUDA_OK(cudaMemsetAsync(dWc, 0, sizeof(float) * P * L * d.h, b.st));
    if (d.has_bias) {
      STC_CUDA_OK(cudaMemsetAsync(dbg, 0, sizeof(float) * 2 * d.h, b.st));
      STC_CUDA_OK(cudaMemsetAsync(dbc, 0, sizeof(float) * d.h, b.st));
    }
    if (dGs && dGs_floats) STC_CUDA_OK(cudaMemsetAsync(dGs, 0, sizeof(float) * dGs_floats, b.st));
    if (b.dGc) STC_CUDA_OK(cudaMemsetAsync(b.dGc, 0, sizeof(float) * d.C * d.C, b.st));
  }
  if (d.B > 0 && b.want_dGc()) STC_CUDA_OK(cudaMemsetAsync(b.sc + b.w.dQ, 0, sizeof(float) * d.Kc * d.C * d.C, b.st));
  return STC_OK;
}

// dW = Y_k^T [Ds | Dm_c] needs only what dx just wrote (dpre) and forward's saved terms: side stream 0 when lanes are active
// (deterministic mode: dx and dW each reduce through their own slot region, so the two may run side by side)
static int launch_dw_beside(const BwdCtx& b, const ConvArgs& dx_args) {
  ConvArgs a = dx_args;
  if (det_mode()) a.det_ws = b.sc + b.w.det_dw;
  if (b.lanes && b.lanes->active()) {
    STC_TRY(b.lanes->fork(0));
    return launch_conv_bwd_dw(a, b.lanes->stream(0));
  }
  return launch_conv_bwd_dw(a, b.st);
}

// candidate conv adjoint: leaves d(r*H terms) in scratch dYr[0..Ks-1], the x-part adjoint in dYx0 / scratch dYx
static int bwd_candi(const BwdCtx& b, const float* Wc, float* dWc, float* dbc) {
  const StcDims& d = b.d;
  const WsLayout& w = b.w;
  const size_t Rh = w.R * d.h;
  ConvArgs a = base_args(d, b.xt, b.xt_bs, Wc, b.sv + w.Q, b.sv, w, 1);
  if (b.yx_pre) a.yx = b.yx_pre;
  a.h0 = b.sv + w.Yr;
  a.yh = b.sv + w.Yr + Rh;
  a.Hprev = b.h_prev;
  a.u = b.sv + w.u;
  a.c = b.sv + w.c;
  a.dHn = b.d_h_out;
  a.dpre = b.sc + w.dpre;
  a.dbias = d.has_bias ? dbc : nullptr;
  a.dYx0 = b.dYx0();
  a.dYx = b.dyx_out ? b.dyx_out : b.sc + w.dYx;
  a.accum_x = 0;
  a.dYx_add = b.dyx_fold;
  a.dYh0 = b.sc + w.dYr;
  a.dYh = b.sc + w.dYr + Rh;
  a.dQ = b.want_dGc() ? b.sc + w.dQ : nullptr;
  a.dW = dWc;
  a.Psave = b.sv + w.Pc;
  a.Wimg = (w.saved_total > w.Wimg_c && w.scratch_total > w.Wimg_dx) ? b.sc + w.Wimg_dx : nullptr;   // wide forward ran
  if (det_mode()) a.det_ws = b.sc + w.det_dx;
  STC_TRY(launch_conv_bwd_dx(a, b.st));
  return launch_dw_beside(b, a);
}

// GRU elementwise adjoint + gates conv adjoint (reads d(r*H) = scratch dYr[0]); then dGc from the dT_k(Gc) partials
static int bwd_gates(const BwdCtx& b, const float* Wg, float* dWg, float* dbg) {
  const StcDims& d = b.d;
  const WsLayout& w = b.w;
  ConvArgs a = base_args(d, b.xt, b.xt_bs, Wg, b.sv + w.Q, b.sv, w, 0);
  if (b.yx_pre) a.yx = b.yx_pre;
  a.h0 = b.h_prev;
  a.yh = b.yh_pre ? b.yh_pre : b.sv + w.Yh;
  a.Hprev = b.h_prev;
  a.u = b.sv + w.u;
  a.r = b.sv + w.r;
  a.c = b.sv + w.c;
  a.dHn = b.d_h_out;
  a.drH = b.sc + w.dYr;
  a.dpre = b.sc + w.dpre;
  a.dbias = d.has_bias ? dbg : nullptr;
  a.dYx0 = b.dYx0();
  a.dYx = b.dyx_out ? b.dyx_out : b.sc + w.dYx;
  a.accum_x = 1;
  a.dYh0 = b.d_h_prev;
  a.dYh = b.dyh_out ? b.dyh_out : b.sc + w.dYh;
  a.dYh_add = b.dyh_fold;
  a.dQ = b.want_dGc() ? b.sc + w.dQ : nullptr;
  a.dW = dWg;
  a.Psave = b.sv + w.Pg;
  a.Wimg = (w.Wimg_c > w.Wimg_g && w.scratch_total > w.Wimg_dx) ? b.sc + w.Wimg_dx : nullptr;   // wide forward ran
  if (det_mode()) a.det_ws = b.sc + w.det_dx;
  if (b.lanes) STC_TRY(b.lanes->join(0));   // the candidate's dW reads dpre, which this dx overwrites
  STC_TRY(launch_conv_bwd_dx(a, b.st));
  STC_TRY(launch_dw_beside(b, a));
  if (b.want_dGc()) STC_TRY(launch_cheby_small_bwd(b.gc, b.sv + w.Q, b.sc + w.dQ, d.C, d.Kc, b.dGc, b.st));
  return STC_OK;
}

static int cell_bwd_impl(const StcDims* dp, const StcSupport* gs, const float* gc, const float* xt,
                         int64_t xt_batch_stride, const float* h_prev, const float* Wg, const float* Wc,
                         const float* d_h_out, float* d_xt, float* d_h_prev, float* dWg, float* dbg, float* dWc, float* dbc,
                         float* dGs, float* dGc, int32_t accumulate_params, const void* savedv, size_t saved_bytes,
                         void* scratchv, size_t scratch_bytes, const float* yx_terms, float* dyx_terms_out,
                         const float* dyx_fold, const float* yh_terms, float* dyh_terms_out, const float* dyh_fold,
                         void* stream, const char* who) {
  reset_launch_count();
  STC_TRY(check_bwd_args(dp, gc, xt, h_prev, Wg, Wc, d_h_out, d_h_prev, dWg, dbg, dWc, dbc, savedv, saved_bytes, scratchv,
                         scratch_bytes, who));
  const StcDims& d = *dp;
  if (!gs) {
    set_error("%s: NULL argument", who);
    return STC_ERR_BAD_ARG;
  }
  if (dGs && is_csr_kind(gs->kind) && (!gs->rowptr || !gs->col || !gs->vals || gs->nnz < 0)) {
    set_error("%s: the edge-value gradient of a CSR support needs its rowptr/col/vals and nnz", who);
    return STC_ERR_BAD_ARG;
  }
  if ((yx_terms && dyx_fold) || (yh_terms && dyh_fold)) {
    set_error("%s: a side either takes supplied terms or folds an adjoint into its own terms, not both", who);
    return STC_ERR_BAD_ARG;
  }
  const WsLayout w = make_layout(d);
  STC_TRY(check_arch());
  cudaStream_t st = (cudaStream_t)stream;
  Lanes lanes(st, d);
  BwdCtx b{d, w, gc, xt, xt_batch_stride, h_prev, d_h_out, d_xt, d_h_prev, dGc,
           const_cast<float*>((const float*)savedv), (float*)scratchv, st};
  b.lanes = &lanes;
  const bool hoisted = d.Ks > 1 && yx_terms != nullptr;
  const bool h_given = d.Ks > 1 && yh_terms != nullptr;
  if (hoisted) {
    b.yx_pre = yx_terms;
    b.dyx_out = dyx_terms_out;
  }
  if (h_given) {
    b.yh_pre = yh_terms;
    b.dyh_out = dyh_terms_out;
  }
  if (d.Ks > 1) {
    b.dyx_fold = dyx_fold;
    b.dyh_fold = dyh_fold;
  }
  // a per-sample CSR support's gradient is [B][nnz]: one row per sample
  const size_t dGs_floats = gs->kind == STC_SUPPORT_CSR_PER_SAMPLE ? (size_t)d.B * gs->nnz
                            : gs->kind == STC_SUPPORT_CSR           ? (size_t)gs->nnz
                                                                    : (size_t)d.N * d.N;
  STC_TRY(bwd_begin(b, dWg, dbg, dWc, dbc, dGs, dGs_floats, accumulate_params));
  if (d.B == 0) return STC_OK;
  const size_t Rh = w.R * d.h;
  const int CD = d.C * d.Din, CH = d.C * d.h;

  // Lanes (small problems only; otherwise everything below is one stream in program order):
  //   caller's stream   dx_c -> hops of d(rH) -> dx_g -> Gc chain -> hops of dH
  //   side 0            dW_c (joined before dx_g rewrites dpre), then dW_g
  //   side 1            the dGs outer products of all three chains (atomics into dGs)
  //   side 2            hops of dXt
  STC_TRY(bwd_candi(b, Wc, dWc, dbc));
  // d(rH) through the spatial recurrence
  float* const det_dgs = det_mode() ? b.sc + w.det_dgs : nullptr;   // (all outer products run on one lane)
  STC_TRY(adjoint_chain(d, *gs, CH, b.sv + w.Yr, (int64_t)d.N * CH, b.sv + w.Yr + Rh, b.sc + w.dYr, b.sc + w.dYr + Rh,
                        dGs, st, &lanes, 1, det_dgs));
  STC_TRY(bwd_gates(b, Wg, dWg, dbg));
  if (!hoisted) {   // (hoisted: the x-part adjoints of terms k >= 1 sit in the caller's buffer; d_xt holds term 0 only)
    cudaStream_t sx = st;
    // deterministic mode, learnable CSR support: both chains add their edge gradient into the same dGs in their hops,
    // so the Xt-side chain stays on the caller's stream, ordered after the H-side additions
    const bool csr_grad = dGs && is_csr_kind(gs->kind);
    if (lanes.active() && d.Ks > 1 && !(det_mode() && csr_grad)) {
      STC_TRY(lanes.fork(2));
      sx = lanes.stream(2);
    }
    STC_TRY(adjoint_chain(d, *gs, CD, xt, xt_batch_stride, b.sv + w.Yx, b.dYx0(), b.sc + w.dYx, dGs, sx, &lanes, 1, det_dgs));
  }
  if (!h_given)   // (given: the h-part adjoints of terms k >= 1 sit in dyh_terms_out, or are dropped when it is NULL)
    STC_TRY(adjoint_chain(d, *gs, CH, h_prev, (int64_t)d.N * CH, b.sv + w.Yh, d_h_prev, b.sc + w.dYh, dGs, st, &lanes, 1,
                          det_dgs));
  return lanes.join_all();
}

int stc_cell_bwd(const StcDims* dp, const StcSupport* gs, const float* gc, const float* xt,
                 int64_t xt_batch_stride, const float* h_prev, const float* Wg, const float* Wc,
                 const float* d_h_out, float* d_xt, float* d_h_prev, float* dWg, float* dbg, float* dWc, float* dbc,
                 float* dGs, float* dGc, int32_t accumulate_params, const void* savedv, size_t saved_bytes,
                 void* scratchv, size_t scratch_bytes, void* stream) {
  return cell_bwd_impl(dp, gs, gc, xt, xt_batch_stride, h_prev, Wg, Wc, d_h_out, d_xt, d_h_prev, dWg, dbg, dWc, dbc, dGs, dGc,
                       accumulate_params, savedv, saved_bytes, scratchv, scratch_bytes, nullptr, nullptr, nullptr, nullptr,
                       nullptr, nullptr, stream, "stc_cell_bwd");
}

int stc_cell_bwd_x(const StcDims* dp, const StcSupport* gs, const float* gc, const float* xt,
                   int64_t xt_batch_stride, const float* h_prev, const float* Wg, const float* Wc,
                   const float* d_h_out, float* d_xt, float* d_h_prev, float* dWg, float* dbg, float* dWc, float* dbc,
                   float* dGs, float* dGc, int32_t accumulate_params, const void* savedv, size_t saved_bytes,
                   void* scratchv, size_t scratch_bytes, const float* yx_terms, float* dyx_terms_out,
                   const float* dyx_fold, const float* yh_terms, float* dyh_terms_out, const float* dyh_fold, void* stream) {
  return cell_bwd_impl(dp, gs, gc, xt, xt_batch_stride, h_prev, Wg, Wc, d_h_out, d_xt, d_h_prev, dWg, dbg, dWc, dbc, dGs, dGc,
                       accumulate_params, savedv, saved_bytes, scratchv, scratch_bytes, yx_terms, dyx_terms_out, dyx_fold,
                       yh_terms, dyh_terms_out, dyh_fold, stream, "stc_cell_bwd_x");
}

int stc_support_outer(int32_t N, int32_t B, int32_t width, const float* a, int64_t a_batch_stride, const float* b,
                      float coef, float* dGs, void* stream) {
  reset_launch_count();
  if (!a || !b || !dGs) {
    set_error("stc_support_outer: NULL argument");
    return STC_ERR_BAD_ARG;
  }
  if (det_mode()) {
    set_error("stc_support_outer: deterministic mode needs the partial-slot workspace: use stc_support_outer_ws");
    return STC_ERR_UNSUPPORTED;
  }
  STC_TRY(check_arch());
  return launch_support_outer(N, B, width, a, a_batch_stride, b, coef, dGs, (cudaStream_t)stream);
}

size_t stc_support_outer_workspace_bytes(int32_t N, int32_t B, int32_t width) {
  if (N <= 0 || B < 0 || width <= 0 || !det_mode()) return 0;
  return (size_t)support_outer_det_floats(N, B, width) * sizeof(float);
}

int stc_support_outer_ws(int32_t N, int32_t B, int32_t width, const float* a, int64_t a_batch_stride, const float* b,
                         float coef, float* dGs, void* ws, size_t ws_bytes, void* stream) {
  reset_launch_count();
  if (!a || !b || !dGs) {
    set_error("stc_support_outer_ws: NULL argument");
    return STC_ERR_BAD_ARG;
  }
  const size_t need = stc_support_outer_workspace_bytes(N, B, width);
  if (ws_bytes < need || (need > 0 && ws == nullptr)) {
    set_error("stc_support_outer_ws: workspace of %zu bytes, %zu needed", ws ? ws_bytes : (size_t)0, need);
    return STC_ERR_WORKSPACE;
  }
  if ((reinterpret_cast<uintptr_t>(ws) & 15) != 0) {
    set_error("stc_support_outer_ws: ws must be 16-byte aligned");
    return STC_ERR_BAD_ARG;
  }
  STC_TRY(check_arch());
  return launch_support_outer(N, B, width, a, a_batch_stride, b, coef, dGs, (cudaStream_t)stream,
                              need > 0 ? (float*)ws : nullptr);
}

int stc_support_apply_edge_grad(const StcSupport* gs, int32_t N, int32_t B, int32_t width, const float* x,
                                int64_t x_batch_stride, const float* z, int64_t z_batch_stride, float* y, float alpha,
                                float beta, const float* a, int64_t a_batch_stride, float coef, float* dvals,
                                void* stream) {
  reset_launch_count();
  if (!gs || !x || !y || !a || !dvals) {
    set_error("stc_support_apply_edge_grad: NULL argument");
    return STC_ERR_BAD_ARG;
  }
  if (!is_csr_kind(gs->kind)) {
    set_error("stc_support_apply_edge_grad: CSR supports only (a dense support's gradient is stc_support_outer)");
    return STC_ERR_UNSUPPORTED;
  }
  STC_TRY(check_arch());
  return launch_support_csr_edge_grad(*gs, N, B, width, x, x_batch_stride, z, z_batch_stride, y, alpha, beta, nullptr,
                                      0.f, a, a_batch_stride, coef, dvals, (cudaStream_t)stream);
}

int stc_support_apply_rows_edge_grad(const StcSupport* gs, int32_t N, int32_t B, int32_t width, const float* x,
                                     int64_t x_batch_stride, const float* z, int64_t z_batch_stride, float* y,
                                     float alpha, float beta, const float* a, int64_t a_batch_stride, float coef,
                                     float* dvals, const int32_t* rows, int32_t n_rows, void* stream) {
  reset_launch_count();
  if (!gs || !x || !y || !a || !dvals || !rows) {
    set_error("stc_support_apply_rows_edge_grad: NULL argument");
    return STC_ERR_BAD_ARG;
  }
  if (gs->kind == STC_SUPPORT_CSR_PER_SAMPLE) {
    set_error("stc_support_apply_rows_edge_grad: a per-sample CSR support (STC_SUPPORT_CSR_PER_SAMPLE) takes no row list");
    return STC_ERR_UNSUPPORTED;
  }
  if (gs->kind != STC_SUPPORT_CSR) {
    set_error("stc_support_apply_rows_edge_grad: CSR supports only");
    return STC_ERR_UNSUPPORTED;
  }
  if (n_rows < 0 || n_rows > N) {
    set_error("stc_support_apply_rows_edge_grad: n_rows %d outside [0, N = %d]", n_rows, N);
    return STC_ERR_BAD_ARG;
  }
  STC_TRY(check_arch());
  return launch_support_csr_edge_grad(*gs, N, B, width, x, x_batch_stride, z, z_batch_stride, y, alpha, beta, nullptr,
                                      0.f, a, a_batch_stride, coef, dvals, (cudaStream_t)stream, rows, n_rows);
}

static int check_pattern(const StcSupport* gs, int32_t N, const char* who, bool any_csr = false) {
  if (!gs) {
    set_error("%s: NULL pattern", who);
    return STC_ERR_BAD_ARG;
  }
  if (any_csr ? !is_csr_kind(gs->kind) : gs->kind != STC_SUPPORT_CSR) {
    set_error("%s: the pattern must be a CSR support (kind %d)", who, gs->kind);
    return STC_ERR_UNSUPPORTED;
  }
  if (!gs->rowptr || !gs->col || gs->nnz < 0) {
    set_error("%s: the pattern needs rowptr / col and nnz >= 0", who);
    return STC_ERR_BAD_ARG;
  }
  if (N <= 0) {
    set_error("%s: N = %d must be positive", who, N);
    return STC_ERR_BAD_ARG;
  }
  return STC_OK;
}

int stc_pair_scores_csr(const StcSupport* gs, int32_t N, int64_t width, const float* u, const float* v, float* scores,
                        void* stream) {
  reset_launch_count();
  STC_TRY(check_pattern(gs, N, "stc_pair_scores_csr"));
  if (!u || !v || !scores) {
    set_error("stc_pair_scores_csr: NULL argument");
    return STC_ERR_BAD_ARG;
  }
  if (width <= 0) {
    set_error("stc_pair_scores_csr: width = %lld must be positive", (long long)width);
    return STC_ERR_BAD_ARG;
  }
  STC_TRY(check_arch());
  return launch_pair_scores_csr(gs->rowptr, gs->col, gs->nnz, N, width, u, v, scores, (cudaStream_t)stream);
}

int stc_pair_scores_csr_rows(const StcSupport* gs, int32_t N, int64_t width, int64_t ld, const float* u, const float* v,
                             float* scores, const int32_t* rows, int32_t n_rows, void* stream) {
  reset_launch_count();
  STC_TRY(check_pattern(gs, N, "stc_pair_scores_csr_rows"));
  if (!u || !v || !scores || !rows) {
    set_error("stc_pair_scores_csr_rows: NULL argument");
    return STC_ERR_BAD_ARG;
  }
  if (width <= 0) {
    set_error("stc_pair_scores_csr_rows: width = %lld must be positive", (long long)width);
    return STC_ERR_BAD_ARG;
  }
  if (ld < width) {
    set_error("stc_pair_scores_csr_rows: row stride ld = %lld is smaller than width = %lld", (long long)ld,
              (long long)width);
    return STC_ERR_BAD_ARG;
  }
  if (n_rows < 0 || n_rows > N) {
    set_error("stc_pair_scores_csr_rows: n_rows %d outside [0, N = %d]", n_rows, N);
    return STC_ERR_BAD_ARG;
  }
  STC_TRY(check_arch());
  return launch_pair_scores_csr_rows(gs->rowptr, gs->col, gs->nnz, N, width, ld, u, v, scores, rows, n_rows,
                                     (cudaStream_t)stream);
}

int stc_edge_softmax_fwd(const StcSupport* gs, int32_t N, const float* scores, float* p, void* stream) {
  reset_launch_count();
  STC_TRY(check_pattern(gs, N, "stc_edge_softmax_fwd"));
  if (!scores || !p) {
    set_error("stc_edge_softmax_fwd: NULL argument");
    return STC_ERR_BAD_ARG;
  }
  STC_TRY(check_arch());
  return launch_edge_softmax(false, gs->rowptr, gs->nnz, N, scores, nullptr, nullptr, p, (cudaStream_t)stream);
}

int stc_edge_softmax_bwd(const StcSupport* gs, int32_t N, const float* scores, const float* p, const float* dp,
                         float* dscores, void* stream) {
  reset_launch_count();
  STC_TRY(check_pattern(gs, N, "stc_edge_softmax_bwd"));
  if (!scores || !p || !dp || !dscores) {
    set_error("stc_edge_softmax_bwd: NULL argument");
    return STC_ERR_BAD_ARG;
  }
  STC_TRY(check_arch());
  return launch_edge_softmax(true, gs->rowptr, gs->nnz, N, scores, p, dp, dscores, (cudaStream_t)stream);
}

static int check_batch(int32_t B, const char* who) {
  if (B < 0 || B > 65535) {
    set_error("%s: B = %d outside [0, 65535]", who, B);
    return STC_ERR_BAD_ARG;
  }
  return STC_OK;
}

int stc_pair_scores_csr_batched(const StcSupport* gs, int32_t N, int32_t B, int64_t width, const float* u,
                                const float* v, float* scores, void* stream) {
  reset_launch_count();
  STC_TRY(check_pattern(gs, N, "stc_pair_scores_csr_batched", true));
  STC_TRY(check_batch(B, "stc_pair_scores_csr_batched"));
  if (B == 0) return STC_OK;
  if (!u || !v || !scores) {
    set_error("stc_pair_scores_csr_batched: NULL argument");
    return STC_ERR_BAD_ARG;
  }
  if (width <= 0) {
    set_error("stc_pair_scores_csr_batched: width = %lld must be positive", (long long)width);
    return STC_ERR_BAD_ARG;
  }
  STC_TRY(check_arch());
  return launch_pair_scores_csr_batched(gs->rowptr, gs->col, gs->nnz, N, B, width, u, v, scores, (cudaStream_t)stream);
}

int stc_edge_softmax_fwd_batched(const StcSupport* gs, int32_t N, int32_t B, const float* scores, float* p, void* stream) {
  reset_launch_count();
  STC_TRY(check_pattern(gs, N, "stc_edge_softmax_fwd_batched", true));
  STC_TRY(check_batch(B, "stc_edge_softmax_fwd_batched"));
  if (B == 0) return STC_OK;
  if (!scores || !p) {
    set_error("stc_edge_softmax_fwd_batched: NULL argument");
    return STC_ERR_BAD_ARG;
  }
  STC_TRY(check_arch());
  return launch_edge_softmax(false, gs->rowptr, gs->nnz, N, scores, nullptr, nullptr, p, (cudaStream_t)stream, B);
}

int stc_edge_softmax_bwd_batched(const StcSupport* gs, int32_t N, int32_t B, const float* scores, const float* p,
                                 const float* dp, float* dscores, void* stream) {
  reset_launch_count();
  STC_TRY(check_pattern(gs, N, "stc_edge_softmax_bwd_batched", true));
  STC_TRY(check_batch(B, "stc_edge_softmax_bwd_batched"));
  if (B == 0) return STC_OK;
  if (!scores || !p || !dp || !dscores) {
    set_error("stc_edge_softmax_bwd_batched: NULL argument");
    return STC_ERR_BAD_ARG;
  }
  STC_TRY(check_arch());
  return launch_edge_softmax(true, gs->rowptr, gs->nnz, N, scores, p, dp, dscores, (cudaStream_t)stream, B);
}

static int check_topk_shape(int32_t N, int64_t width, int32_t k, const char* who) {
  if (N <= 0 || width <= 0 || width % 4 != 0 || width > (1 << 28)) {
    set_error("%s: N = %d must be positive and width = %lld a positive multiple of 4 (at most 2^28)", who, N,
              (long long)width);
    return STC_ERR_BAD_ARG;
  }
  if (k > 32) {
    set_error("%s: k = %d: at most 32 columns a row are kept on chip", who, k);
    return STC_ERR_UNSUPPORTED;
  }
  if (k < 1 || k > N) {
    set_error("%s: k = %d outside [1, N = %d]", who, k, N);
    return STC_ERR_BAD_ARG;
  }
  return STC_OK;
}

size_t stc_pair_topk_workspace_bytes(int32_t N, int64_t width, int32_t k) {
  if (check_topk_shape(N, width, k, "stc_pair_topk_workspace_bytes") != STC_OK) return 0;
  return pair_topk_ws_bytes(N, N, k);
}

size_t stc_pair_topk_rows_workspace_bytes(int32_t N, int64_t width, int32_t n_rows, int32_t k) {
  if (check_topk_shape(N, width, k, "stc_pair_topk_rows_workspace_bytes") != STC_OK || n_rows < 0 || n_rows > N)
    return 0;
  return pair_topk_ws_bytes(N, n_rows, k);
}

int stc_pair_topk(int32_t N, int64_t width, const float* u, const float* v, int32_t k, int32_t* cols, float* scores,
                  void* ws, size_t ws_bytes, void* stream) {
  reset_launch_count();
  STC_TRY(check_topk_shape(N, width, k, "stc_pair_topk"));
  if (!u || !v || !cols || !ws) {
    set_error("stc_pair_topk: NULL argument");
    return STC_ERR_BAD_ARG;
  }
  if ((reinterpret_cast<uintptr_t>(u) | reinterpret_cast<uintptr_t>(v) | reinterpret_cast<uintptr_t>(ws)) & 15) {
    set_error("stc_pair_topk: u, v and ws must be 16-byte aligned");
    return STC_ERR_BAD_ARG;
  }
  STC_TRY(check_arch());
  const size_t need = pair_topk_ws_bytes(N, N, k);
  if (ws_bytes < need) {
    set_error("stc_pair_topk: workspace of %zu bytes, %zu needed", ws_bytes, need);
    return STC_ERR_WORKSPACE;
  }
  return launch_pair_topk(N, (int)width, u, v, 0, N, k, cols, scores, ws, (cudaStream_t)stream);
}

int stc_pair_topk_rows(int32_t N, int64_t width, const float* u, const float* v, int32_t row0, int32_t n_rows,
                       int32_t k, int32_t* cols, float* scores, void* ws, size_t ws_bytes, void* stream) {
  reset_launch_count();
  STC_TRY(check_topk_shape(N, width, k, "stc_pair_topk_rows"));
  if (row0 < 0 || n_rows < 0 || (int64_t)row0 + n_rows > N) {
    set_error("stc_pair_topk_rows: rows [%d, %d + %d) outside [0, N = %d)", row0, row0, n_rows, N);
    return STC_ERR_BAD_ARG;
  }
  if (n_rows == 0) return STC_OK;
  if (!u || !v || !cols || !ws) {
    set_error("stc_pair_topk_rows: NULL argument");
    return STC_ERR_BAD_ARG;
  }
  if ((reinterpret_cast<uintptr_t>(u) | reinterpret_cast<uintptr_t>(v) | reinterpret_cast<uintptr_t>(ws)) & 15) {
    set_error("stc_pair_topk_rows: u, v and ws must be 16-byte aligned");
    return STC_ERR_BAD_ARG;
  }
  STC_TRY(check_arch());
  const size_t need = pair_topk_ws_bytes(N, n_rows, k);
  if (ws_bytes < need) {
    set_error("stc_pair_topk_rows: workspace of %zu bytes, %zu needed", ws_bytes, need);
    return STC_ERR_WORKSPACE;
  }
  return launch_pair_topk(N, (int)width, u, v, row0, n_rows, k, cols, scores, ws, (cudaStream_t)stream);
}

int stc_cell_bwd_scratch_layout(const StcDims* dp, int64_t* offsets, int32_t n_offsets) {
  STC_TRY(check_dims(dp));
  if (!offsets || n_offsets < STC_SCRATCH_REGIONS) {
    set_error("stc_cell_bwd_scratch_layout: need room for %d offsets", (int)STC_SCRATCH_REGIONS);
    return STC_ERR_BAD_ARG;
  }
  const WsLayout w = make_layout(*dp);
  const size_t v[STC_SCRATCH_REGIONS] = {w.dYr, w.dYx, w.dYh};
  for (int i = 0; i < STC_SCRATCH_REGIONS; ++i) offsets[i] = (int64_t)v[i];
  if (n_offsets > STC_SCRATCH_DET) offsets[STC_SCRATCH_DET] = (int64_t)w.det_dw;
  return STC_OK;
}

int stc_cell_bwd_stage(const StcDims* dp, int32_t stage, const float* gc, const float* xt, int64_t xt_batch_stride,
                       const float* h_prev, const float* Wg, const float* Wc, const float* d_h_out, float* d_xt,
                       float* d_h_prev, float* dWg, float* dbg, float* dWc, float* dbc, float* dGc,
                       int32_t accumulate_params, const void* savedv, size_t saved_bytes, void* scratchv,
                       size_t scratch_bytes, void* stream) {
  reset_launch_count();
  STC_TRY(check_bwd_args(dp, gc, xt, h_prev, Wg, Wc, d_h_out, d_h_prev, dWg, dbg, dWc, dbc, savedv, saved_bytes, scratchv,
                         scratch_bytes, "stc_cell_bwd_stage"));
  if (stage != STC_STAGE_GATES && stage != STC_STAGE_CANDI) {
    set_error("stc_cell_bwd_stage: bad stage %d", stage);
    return STC_ERR_BAD_ARG;
  }
  if (!d_xt) {
    set_error("stc_cell_bwd_stage: d_xt must be given (the caller runs the adjoint hops on it)");
    return STC_ERR_BAD_ARG;
  }
  const StcDims& d = *dp;
  const WsLayout w = make_layout(d);
  STC_TRY(check_arch());
  const BwdCtx b{d, w, gc, xt, xt_batch_stride, h_prev, d_h_out, d_xt, d_h_prev, dGc,
                 const_cast<float*>((const float*)savedv), (float*)scratchv, (cudaStream_t)stream};
  if (stage == STC_STAGE_CANDI) {   // the first backward stage: also clears the gradients it and the gates stage add into
    STC_TRY(bwd_begin(b, dWg, dbg, dWc, dbc, nullptr, 0, accumulate_params));
    if (d.B == 0) return STC_OK;
    return bwd_candi(b, Wc, dWc, dbc);
  }
  if (d.B == 0) return STC_OK;
  return bwd_gates(b, Wg, dWg, dbg);
}

}  // extern "C"
