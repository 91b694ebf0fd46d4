// sm_100a building blocks for the tensor-core kernels: mbarrier, TMA (cp.async.bulk.tensor),
// tcgen05 (TMEM alloc / mma / commit / ld) and the shared-memory / instruction descriptors.
// Everything is inline PTX; the bit layouts follow the PTX ISA "tcgen05" matrix / instruction
// descriptor tables (the same fields CuTe's mma_sm100_desc.hpp names).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ------------------------------------------------------------------ mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug must surface as an error flag, never as a hung GPU.
// Returns false on timeout (~ a few seconds); callers bail out of the kernel.
__device__ __forceinline__ bool mbar_wait(uint64_t* bar, uint32_t parity, int* err_flag, int code) {
  for (uint32_t it = 0; it < (1u << 24); ++it) {
    if (mbar_try_wait(bar, parity)) return true;
    if (it > 1024) __nanosleep(64);
    if ((it & 0xffff) == 0xffff && err_flag && *reinterpret_cast<volatile int*>(err_flag) != 0) return false;
  }
  if (err_flag) atomicCAS(err_flag, 0, code);
  return false;
}

// Bounded wait WITHOUT an early-exit branch: on timeout it records the error and simply returns, so the
// caller's loops keep warp-uniform control flow (ptxas can then keep loop-carried address arithmetic in
// uniform registers, which the single-thread tcgen05.mma issue path depends on).  After a timeout every
// later wait of the CTA returns after a short spin (shared `abort` flag): wrong results, but no hang.
__device__ __forceinline__ void mbar_wait_soft(uint64_t* bar, uint32_t parity, int* err_flag, int code,
                                               volatile uint32_t* abort_flag) {
  for (uint32_t it = 0;; ++it) {
    if (mbar_try_wait(bar, parity)) return;
    if ((it & 0xfffu) == 0xfffu) {
      if (*abort_flag) return;
      if (it >= (1u << 24)) {
        *abort_flag = 1u;
        if (err_flag) atomicCAS(err_flag, 0, code);
        return;
      }
      __nanosleep(64);
    }
  }
}

// generic-proxy smem writes -> visible to the async proxy (TMA / tcgen05.mma operand reads)
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// ------------------------------------------------------------------ TMA
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1,
                                            int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cta.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1,
                                            int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cta.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2),
      "r"(c3)
      : "memory");
}

// plain 1-D bulk copy global -> shared (size multiple of 16 bytes), completion on an mbarrier
__device__ __forceinline__ void bulk_load_1d(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(gsrc)), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// ------------------------------------------------------------------ tcgen05 / TMEM
template <int NCOLS>
__device__ __forceinline__ void tmem_alloc(uint32_t* slot_in_smem) {  // whole warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot_in_smem)),
               "n"(NCOLS));
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
}
template <int NCOLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {  // same warp that allocated
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(NCOLS));
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem]^T ; one thread issues on behalf of the CTA
__device__ __forceinline__ void mma_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                        uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Same instruction for warp-converged issue loops: every lane executes the (uniform) address
// arithmetic so that ptxas keeps descriptors in uniform registers, and only the lane whose `guard`
// is non-zero issues.  (Guarding the whole loop with `if (lane == 0)` instead makes every operand a
// per-thread value: each MMA then pays an ELECT loop plus five R2UR broadcasts, ~150+ cycles.)
__device__ __forceinline__ void mma_f16_guarded(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                                uint32_t accumulate, uint32_t guard) {
  asm volatile(
      "{\n\t.reg .pred p, q;\n\tsetp.ne.b32 p, %4, 0;\n\tsetp.ne.b32 q, %5, 0;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(guard)
      : "memory");
}
// FOUR MMAs of a host-built issue program in one instruction group: w.x .. w.w = (A offset | B offset << 16) in 16-byte
// units relative to a_base / b_base, 0xffffffff = no MMA (padding of the program to a multiple of four).  One election
// and one 128-bit constant load per four MMAs; the first MMA takes `accumulate_first`, the others accumulate.
// (`elect.sync` inside the group tells ptxas that exactly one lane issues: no per-lane ELECT / BRA.U.ANY loop around the
// UTCHMMA, uniform operands stay in uniform registers.  All 32 lanes must execute this, converged.)
// (Measured on the one-word-per-iteration loop, ncu source view: ~105 issue cycles per MMA against 61 of tensor time -
// the indexed constant load sat on the critical path of every MMA, plus ELECT / VOTEU / 4 x R2UR each.)
__device__ __forceinline__ void mma_f16_x4(uint32_t d_tmem, uint32_t a_base, uint32_t a_hi, uint32_t b_base, uint32_t b_hi,
                                           uint32_t idesc, uint4 w, uint32_t accumulate_first) {
  asm volatile(
      "{\n\t.reg .pred q, p0, e1, e2, e3, pt;\n\t.reg .b64 da, db;\n\t.reg .b32 al, bl;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "setp.ne.b32 p0, %10, 0;\n\t"
      "setp.eq.b32 pt, %5, %5;\n\t"
      "setp.ne.and.b32 e1, %7, 0xffffffff, q;\n\t"
      "setp.ne.and.b32 e2, %8, 0xffffffff, q;\n\t"
      "setp.ne.and.b32 e3, %9, 0xffffffff, q;\n\t"
      "and.b32 al, %6, 0xffff;\n\tadd.u32 al, al, %1;\n\tshr.u32 bl, %6, 16;\n\tadd.u32 bl, bl, %3;\n\t"
      "mov.b64 da, {al, %2};\n\tmov.b64 db, {bl, %4};\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p0;\n\t"
      "and.b32 al, %7, 0xffff;\n\tadd.u32 al, al, %1;\n\tshr.u32 bl, %7, 16;\n\tadd.u32 bl, bl, %3;\n\t"
      "mov.b64 da, {al, %2};\n\tmov.b64 db, {bl, %4};\n\t"
      "@e1 tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, pt;\n\t"
      "and.b32 al, %8, 0xffff;\n\tadd.u32 al, al, %1;\n\tshr.u32 bl, %8, 16;\n\tadd.u32 bl, bl, %3;\n\t"
      "mov.b64 da, {al, %2};\n\tmov.b64 db, {bl, %4};\n\t"
      "@e2 tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, pt;\n\t"
      "and.b32 al, %9, 0xffff;\n\tadd.u32 al, al, %1;\n\tshr.u32 bl, %9, 16;\n\tadd.u32 bl, bl, %3;\n\t"
      "mov.b64 da, {al, %2};\n\tmov.b64 db, {bl, %4};\n\t"
      "@e3 tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, pt;\n\t}"
      ::"r"(d_tmem), "r"(a_base), "r"(a_hi), "r"(b_base), "r"(b_hi), "r"(idesc), "r"(w.x), "r"(w.y), "r"(w.z), "r"(w.w),
        "r"(accumulate_first)
      : "memory");
}
// Up to four MMAs that share the A operand and the accumulate flag and differ in the B offset and the accumulator
// (weight gradient: one accumulator per filter tap, d_tmem + i * d_step): boff.x .. boff.w are added to b_row,
// 0xffffffff = no MMA.  One election / one 128-bit program load per group, see mma_f16_x4.
__device__ __forceinline__ void mma_f16_x4_taps(uint32_t d_tmem, uint32_t d_step, uint32_t a_lo, uint32_t a_hi, uint32_t b_row,
                                                uint32_t b_hi, uint32_t idesc, uint4 boff, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred q, p, e0, e1, e2, e3;\n\t.reg .b64 da, db;\n\t.reg .b32 bl, dd;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "setp.ne.b32 p, %11, 0;\n\t"
      "setp.ne.and.b32 e0, %7, 0xffffffff, q;\n\t"
      "setp.ne.and.b32 e1, %8, 0xffffffff, q;\n\t"
      "setp.ne.and.b32 e2, %9, 0xffffffff, q;\n\t"
      "setp.ne.and.b32 e3, %10, 0xffffffff, q;\n\t"
      "mov.b64 da, {%2, %3};\n\t"
      "add.u32 bl, %4, %7;\n\tmov.b64 db, {bl, %5};\n\t"
      "@e0 tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %6, p;\n\t"
      "add.u32 bl, %4, %8;\n\tmov.b64 db, {bl, %5};\n\tadd.u32 dd, %0, %1;\n\t"
      "@e1 tcgen05.mma.cta_group::1.kind::f16 [dd], da, db, %6, p;\n\t"
      "add.u32 bl, %4, %9;\n\tmov.b64 db, {bl, %5};\n\tadd.u32 dd, dd, %1;\n\t"
      "@e2 tcgen05.mma.cta_group::1.kind::f16 [dd], da, db, %6, p;\n\t"
      "add.u32 bl, %4, %10;\n\tmov.b64 db, {bl, %5};\n\tadd.u32 dd, dd, %1;\n\t"
      "@e3 tcgen05.mma.cta_group::1.kind::f16 [dd], da, db, %6, p;\n\t}"
      ::"r"(d_tmem), "r"(d_step), "r"(a_lo), "r"(a_hi), "r"(b_row), "r"(b_hi), "r"(idesc), "r"(boff.x), "r"(boff.y), "r"(boff.z),
        "r"(boff.w), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void mma_i8(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                       uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// all previously issued MMAs of this thread arrive on `bar` when they complete
// (implies tcgen05.fence::before_thread_sync)
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// commit issued by the SAME elected lane as the elect.sync issue groups above (elect.sync is deterministic for a given member
// mask): the commit tracks the MMAs of the executing thread only.  Warp-converged.
__device__ __forceinline__ void mma_commit_elect(uint64_t* bar) {
  asm volatile(
      "{\n\t.reg .pred q;\n\telect.sync _|q, 0xffffffff;\n\t"
      "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}"
      ::"r"(smem_u32(bar))
      : "memory");
}

// TMEM -> registers: warp w (w % 4 selects the 32-lane quarter) reads 32 consecutive columns
// of its 32 lanes; thread i gets lane (quarter*32 + i).
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ------------------------------------------------------------------ descriptors
// Shared-memory matrix descriptor, K-major, no swizzle ("interleaved" canonical layout):
//   core matrix = 8 rows x 16 bytes stored contiguously (row r at +16*r);
//   SBO = byte distance between consecutive 8-row groups along M/N;
//   LBO = byte distance between the two 16-byte K-chunks of one MMA K-step.
__device__ __forceinline__ uint64_t smem_desc_kmajor_noswz(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3fff);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3fff) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3fff) << 32;
  d |= (uint64_t)1 << 46;  // descriptor version (Blackwell)
  return d;                // base_offset = 0, lbo_mode = 0, layout_type = 0 (no swizzle)
}

// Instruction descriptor (32-bit).  fmt: kind::f16 -> 0 F16, 1 BF16, 2 TF32 ; kind::i8 -> 0 U8, 1 S8.
// cfmt: 0 F16, 1 F32, 2 S32.  Both operands K-major, dense, no negate, no saturate.
__host__ __device__ constexpr uint32_t make_idesc(uint32_t cfmt, uint32_t afmt, uint32_t bfmt, uint32_t M,
                                                  uint32_t N) {
  return (cfmt << 4) | (afmt << 7) | (bfmt << 10) | ((N >> 3) << 17) | ((M >> 4) << 24);
}

// same, with explicit operand majors (0 = K-major, 1 = MN-major)
__host__ __device__ constexpr uint32_t make_idesc_major(uint32_t cfmt, uint32_t afmt, uint32_t bfmt, uint32_t M,
                                                        uint32_t N, uint32_t a_mn, uint32_t b_mn) {
  return make_idesc(cfmt, afmt, bfmt, M, N) | (a_mn << 15) | (b_mn << 16);
}
// MN-major no-swizzle canonical layout: 16-byte vectors hold 8 consecutive M (or N) elements,
// 8 consecutive K rows are 16 bytes apart (128-byte core matrix);
//   LBO = byte distance between consecutive 8-row K groups,
//   SBO = byte distance between consecutive 8-element M/N groups.
// The bit layout of the descriptor is the same as the K-major one.
__device__ __forceinline__ uint64_t smem_desc_mnmajor_noswz(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return smem_desc_kmajor_noswz(saddr, lbo_bytes, sbo_bytes);
}

}  // namespace tc

// host: rank-`rank` tiled tensor map over a dense tensor (dims / box innermost-first)
int mnb_make_tmap(CUtensorMap* out, const void* base, int elem_bytes, int rank, const uint64_t* dims,
                  const uint32_t* box);
// same with explicit byte strides of dimensions 1 .. rank-1 (any order, multiples of 16): lets the box traversal
// order differ from the memory order (e.g. a channel-octet dimension declared last)
int mnb_make_tmap_strided(CUtensorMap* out, const void* base, int elem_bytes, int rank, const uint64_t* dims,
                          const uint64_t* strides_bytes, const uint32_t* box);
