// tcgen05 / TMEM helpers for the tensor-core kernels (sm_100a only).
//
// Precision scheme ("3xTF32"): every fp32 operand a is split as a = hi + lo with hi = a with the low 13
// mantissa bits cleared (exactly a TF32 value) and lo = a - hi (exact in fp32), again cleared to TF32.
// A product is evaluated as hi*hi + hi*lo + lo*hi with fp32 accumulation in TMEM; the dropped lo*lo term
// is ~2^-20 relative, which keeps the reference's rtol 1e-4 with margin (single-pass TF32 does not).
//
// Operand layout in shared memory: K-major, 128-byte swizzle.  One "atom" is 32 fp32 along K (128 bytes)
// by R rows; rows are grouped by 8 (1024 contiguous bytes per group), the 16-byte chunk index inside a
// 128-byte row is XOR-ed with (row % 8).  Atoms must be 1024-byte aligned.  One tcgen05.mma of
// kind::tf32 consumes K = 8 (32 bytes): K-steps inside an atom advance the descriptor start address by
// 32 bytes.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace stc {
namespace tc {

constexpr int ATOM_K = 32;            // fp32 elements along K per 128-byte swizzle row
constexpr int ATOM_ROW_BYTES = 128;
constexpr int GROUP_BYTES = 1024;     // 8 rows x 128 B

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// byte offset of (row, 16-byte chunk q in [0,8)) inside a K-major SW128 atom
__device__ __forceinline__ uint32_t atom_chunk_offset(int row, int q) {
  return (uint32_t)((row >> 3) * GROUP_BYTES + (row & 7) * ATOM_ROW_BYTES + ((q ^ (row & 7)) << 4));
}

// round-to-nearest TF32 (cvt.rna): the result has its low 13 mantissa bits clear
__device__ __forceinline__ float to_tf32_rn(float v) {
  // the integer form of cvt.rna.tf32.f32 (round to nearest, ties away from zero, on the sign-magnitude bits): two
  // instructions instead of the four the cvt expands to (it also special-cases inf/nan, which never occur here)
  return __uint_as_float((__float_as_uint(v) + 0x1000u) & 0xFFFFE000u);
}
// hi = RN_tf32(v), lo = v - hi (exact).  The tensor core ignores lo's 13 low mantissa bits; because hi is
// rounded to nearest, lo has no preferred sign and that truncation is unbiased: |v - hi - tf32(lo)| <= 2^-21 |v|
__device__ __forceinline__ void split_tf32(float v, float& hi, float& lo) {
  hi = to_tf32_rn(v);
  lo = v - hi;
}
__device__ __forceinline__ void split_tf32_trunc(float v, float& hi, float& lo) {  // experiment only
  hi = __uint_as_float(__float_as_uint(v) & 0xFFFFE000u);
  lo = __uint_as_float(__float_as_uint(v - hi) & 0xFFFFE000u);
}

__device__ __forceinline__ void store_split4(uint8_t* a_hi, uint8_t* a_lo, uint32_t off, float4 v) {
  float4 h, l;
  split_tf32(v.x, h.x, l.x);
  split_tf32(v.y, h.y, l.y);
  split_tf32(v.z, h.z, l.z);
  split_tf32(v.w, h.w, l.w);
  *reinterpret_cast<float4*>(a_hi + off) = h;
  *reinterpret_cast<float4*>(a_lo + off) = l;
}

// ---- descriptors ---------------------------------------------------------------------------------
// shared-memory matrix descriptor: K-major, SWIZZLE_128B, SBO = 1024 B (8-row group pitch), LBO unused (=1)
__device__ __forceinline__ uint64_t make_smem_desc_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);        // start address  [0,14)
  d |= (uint64_t)1 << 16;                            // leading byte offset (ignored for swizzled K-major)
  d |= (uint64_t)(GROUP_BYTES >> 4) << 32;           // stride byte offset [32,46)
  d |= (uint64_t)1 << 46;                            // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;                            // layout type: SWIZZLE_128B
  return d;
}

// MN-major operand (the K index is the slow one: tile rows = K, 128-byte rows hold 32 consecutive M/N elements).
// For 32-bit (tf32) operands the only MN-major swizzle the tensor core accepts is SWIZZLE_128B_BASE32B
// (layout type 1): rows of 128 bytes in groups of FOUR K-rows (512 bytes, 512-byte aligned); inside a group the
// 32-byte chunk index (address bits [5,7)) is XOR-ed with the row index (address bits [7,9)).  LBO = pitch between
// 32-element column blocks along M/N, SBO = pitch between 4-row groups along K.  One MMA (K = 8) consumes two groups.
constexpr int MN32_GROUP_BYTES = 512;
// byte offset of the 16-byte chunk q in [0,8) (elements 4q..4q+3 of the 32-wide block) of K-row k
__device__ __forceinline__ uint32_t mn32_chunk_offset(int k, int q) {
  return (uint32_t)(k * ATOM_ROW_BYTES + ((((q >> 1) ^ (k & 3)) << 5) | ((q & 1) << 4)));
}
__device__ __forceinline__ uint64_t make_smem_desc_mn32(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;                            // descriptor version (Blackwell)
  d |= (uint64_t)1 << 61;                            // layout type: SWIZZLE_128B_BASE32B
  return d;
}
__host__ __device__ constexpr uint32_t make_idesc_tf32_mn(int M, int N) {  // both operands MN-major
  return (1u << 4) | (2u << 7) | (2u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(N >> 3) << 17) |
         ((uint32_t)(M >> 4) << 24);
}

// A operand resident in TMEM (lane = M row, one 32-bit column per K element), B MN-major in shared memory
__host__ __device__ constexpr uint32_t make_idesc_tf32_atmem_bmn(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | (1u << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// instruction descriptor: kind::tf32, fp32 accumulate, A and B K-major, M x N
__host__ __device__ constexpr uint32_t make_idesc_tf32(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// ---- TMEM ----------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {  // one full warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {  // the same warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// 32 lanes x 8 consecutive fp32 columns -> 8 registers per thread (thread t of warp w <-> lane 32*(w%4)+t)
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float (&v)[8]) {
  uint32_t r0, r1, r2, r3, r4, r5, r6, r7;
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3), "=r"(r4), "=r"(r5), "=r"(r6), "=r"(r7)
               : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
  v[0] = __uint_as_float(r0); v[1] = __uint_as_float(r1); v[2] = __uint_as_float(r2); v[3] = __uint_as_float(r3);
  v[4] = __uint_as_float(r4); v[5] = __uint_as_float(r5); v[6] = __uint_as_float(r6); v[7] = __uint_as_float(r7);
}

// asynchronous form: the registers are valid only after tmem_ld_wait(); follow it with tmem_ld_pin8 on the same array
__device__ __forceinline__ void tmem_ld8_async(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_pin8(uint32_t (&r)[8]) {
  asm volatile("" : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]));
}

// 32 lanes x 16 consecutive columns, asynchronous: the registers are valid only after tmem_ld_wait16 on the same array
__device__ __forceinline__ void tmem_ld16_async(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// compiler-level dependency: uses of r[] cannot be scheduled above this point (place it right after tmem_ld_wait)
__device__ __forceinline__ void tmem_ld_pin16(uint32_t (&r)[16]) {
  asm volatile("" : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                    "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]));
}

// ---- MMA issue (one thread) ------------------------------------------------------------------------
// One lane of a fully converged warp.  Issuing tcgen05.mma from `if (lane == 0)` makes the compiler treat every
// operand as lane-varying: each MMA is then wrapped in an ELECT / R2UR loop of ~25 dependent instructions (~200
// cycles per MMA measured with clock64 -- more than the 32 cycles the MMA itself takes).  With the warp index made
// warp-uniform (uniform_warp_index) and the lane chosen by elect.sync, descriptors stay in uniform registers and the
// MMAs issue back to back.
__device__ __forceinline__ int uniform_warp_index() { return __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0); }
__device__ __forceinline__ uint32_t uniform_u32(uint32_t v) { return __shfl_sync(0xffffffffu, v, 0); }
__device__ __forceinline__ bool elect_one_sync() {   // call from warp-uniform control flow only
  uint32_t pred;
  __syncwarp();   // lanes may have diverged on an earlier lane-dependent branch (e.g. the trace stamps)
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      "elect.sync _|P1, 0xFFFFFFFF;\n\t"
      "selp.b32 %0, 1, 0, P1;\n\t"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

__device__ __forceinline__ void mma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// same with the A operand read from tensor memory (a_tmem = address of its first K column, lane 0)
__device__ __forceinline__ void mma_tf32_atmem(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t"
      "}\n" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// registers -> TMEM: 32 lanes x 8 consecutive 32-bit columns (thread t of warp w <-> lane 32*(w%4)+t)
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const float (&v)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr),
               "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])),
               "r"(__float_as_uint(v[3])), "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])),
               "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7]))
               : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// all previously issued MMAs of this thread arrive on the mbarrier when complete
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// same product with the two small cross terms going to their own accumulator (d_small) so that the main
// accumulator only ever adds hi*hi products (fewer, larger, equally scaled additions)
__device__ __forceinline__ void mma_atom_3x_split(uint32_t d_main, uint32_t d_small, uint32_t a_hi, uint32_t a_lo,
                                                  uint32_t b_hi, uint32_t b_lo, int ksteps, uint32_t idesc,
                                                  bool& acc_main, bool& acc_small) {
  for (int ks = 0; ks < ksteps; ++ks) {
    const uint32_t o = ks * 32;
    const uint64_t ah = make_smem_desc_sw128(a_hi + o), al = make_smem_desc_sw128(a_lo + o);
    const uint64_t bh = make_smem_desc_sw128(b_hi + o), bl = make_smem_desc_sw128(b_lo + o);
    mma_tf32(d_small, al, bh, idesc, acc_small ? 1u : 0u);
    mma_tf32(d_small, ah, bl, idesc, 1u);
    mma_tf32(d_main, ah, bh, idesc, acc_main ? 1u : 0u);
    acc_main = true;
    acc_small = true;
  }
}

// 3xTF32 product of one atom pair over `ksteps` K-steps of 8: D (+)= A_hi B_hi + A_hi B_lo + A_lo B_hi
__device__ __forceinline__ void mma_atom_3x(uint32_t d_tmem, uint32_t a_hi, uint32_t a_lo, uint32_t b_hi,
                                            uint32_t b_lo, int ksteps, uint32_t idesc, bool& accumulate) {
  for (int ks = 0; ks < ksteps; ++ks) {
    const uint32_t o = ks * 32;
    const uint64_t ah = make_smem_desc_sw128(a_hi + o), al = make_smem_desc_sw128(a_lo + o);
    const uint64_t bh = make_smem_desc_sw128(b_hi + o), bl = make_smem_desc_sw128(b_lo + o);
    mma_tf32(d_tmem, al, bh, idesc, accumulate ? 1u : 0u);  // small terms first
    mma_tf32(d_tmem, ah, bl, idesc, 1u);
    mma_tf32(d_tmem, ah, bh, idesc, 1u);
    accumulate = true;
  }
}

// ---- bulk async copy global -> shared (TMA 1-D), completion counted in bytes on an mbarrier --------
// dst, src 16-byte aligned, bytes a multiple of 16
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
// shared -> global bulk store (TMA 1-D), tracked by the issuing thread's bulk async-group
__device__ __forceinline__ void bulk_s2g(void* gdst, const void* smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_u32(smem_src)),
               "r"(bytes)
               : "memory");
}
// hint: pull [gsrc, gsrc + bytes) into L2 (no destination, no completion to wait for).  gsrc 16-byte aligned, bytes a
// multiple of 16.  Used one tile ahead so that the tile's own loads see L2 latency instead of HBM latency.
__device__ __forceinline__ void l2_prefetch(const void* gsrc, uint32_t bytes) {
  if (bytes) asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(gsrc), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// all of this thread's committed bulk stores have finished READING their shared-memory source
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}

// ---- cp.async global -> shared (16 bytes, L2 only), completion tracked per thread in commit groups -----------
__device__ __forceinline__ void cp_async16(uint32_t smem_dst, const void* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_dst), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// ---- vector reduction into global memory ----------------------------------------------------------------
// red.global.add.v4.f32 (sm_90+): one L2 atomic transaction for four consecutive floats.  The end-of-kernel
// accumulations (dW, dGs: every CTA adds its partial sums into the same few thousand addresses) are bound by the
// number of atomic operations the L2 slices retire, not by bytes -- a quarter of the operations is a quarter of that
// fixed per-launch cost.  p must be 16-byte aligned.
__device__ __forceinline__ void red_add_v4(float* p, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
// The end-of-kernel gradient output of one CTA: a vector reduction into the destination, or (DET, deterministic mode) a
// plain store into the CTA's own partial slot, summed in slot order afterwards (launch_det_reduce).
template <bool DET>
__device__ __forceinline__ void grad_out_v4(float* p, float a, float b, float c, float d) {
  if constexpr (DET) *reinterpret_cast<float4*>(p) = make_float4(a, b, c, d);
  else red_add_v4(p, a, b, c, d);
}
template <bool DET>
__device__ __forceinline__ void grad_out(float* p, float v) {
  if constexpr (DET) *p = v;
  else atomicAdd(p, v);
}

// ---- mbarrier --------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
      "@P1 bra WAIT_DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "WAIT_DONE:\n\t"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}

// Waiting with back-off for warps that are AHEAD of the pipeline (producers waiting for a free stage, epilogue warps
// waiting for a whole accumulation chain): a bare try_wait loop issues an instruction every ~3 cycles (measured on
// tc_support_big, profiles/r4k_tc_support_big_ncu.txt: the four waiting epilogue warps executed as many instructions as
// the eight working warps) in a scheduler it shares with working warps.  ns == 0 spins like mbar_wait.
// (A/B on the one-tile kernels tc_support / tc_outer, whose waits are short: neutral at 0 / 32 / 128 ns --
//  profiles/r4o_wait_backoff_ab.txt -- so they keep mbar_wait.)
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, P1;\n\t"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait_backoff(uint64_t* bar, uint32_t parity, uint32_t ns) {
  while (!mbar_try_wait(bar, parity)) {
    if (ns) __nanosleep(ns);
  }
}

}  // namespace tc
}  // namespace stc
