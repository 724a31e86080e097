// Thin inline-PTX wrappers for the sm_100a features the tensor-core path uses:
// mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (alloc / mma / commit / ld / st / fence).
// Descriptor bit layouts follow the PTX ISA "tcgen05 matrix descriptor" / "instruction descriptor"
// tables (cross-checked against the CuTe headers shipped in this image).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cstdint>

namespace fgnn {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---- mbarrier -------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
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
// Bounded wait: a protocol bug must surface as a CUDA error, never as a hung GPU box.  The slow path is
// kept out of line so that every wait site costs a handful of instructions.
__device__ __noinline__ void mbar_wait_slow(uint32_t bar_addr, uint32_t parity) {
  // The loop is three instructions: a quarter of all issue slots of the conv-chain kernel used to go to polling
  // (try_wait + clock read + compare per spin, ~10 waiting warps per SM, and the waiting control warps have the
  // highest scheduling priority).  try_wait suspends the warp in hardware for a short, implementation-defined
  // time (a suspend-time hint turns it into NANOSLEEP.SYNCS, whose wake-up latency cost 3% end to end); the 2 s
  // watchdog is only evaluated every 1024 spins.
  const long long t0 = clock64();
  for (;;) {
#pragma unroll 1
    for (int spins = 0; spins < 1024; ++spins) {
      uint32_t ok;
      asm volatile(
          "{\n\t.reg .pred p;\n\t"
          "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
          "selp.u32 %0, 1, 0, p;\n\t}"
          : "=r"(ok)
          : "r"(bar_addr), "r"(parity)
          : "memory");
      if (ok) return;
    }
    if (clock64() - t0 > 4000000000LL) {  // ~2 s at 2 GHz
      printf("fgnn: mbarrier wait timed out (block %d thread %d bar %u parity %u)\n", blockIdx.x, threadIdx.x,
             bar_addr, parity);
      __trap();
    }
  }
}
// (A suspend-time hint on try_wait -- NANOSLEEP.SYNCS instead of polling -- was measured 3-5% slower end to end,
// for the control roles as well: every hand-off in the conv-chain kernel is latency-critical.)
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (!mbar_try_wait(bar, parity)) mbar_wait_slow(smem_u32(bar), parity);
}

// ---- TMA ------------------------------------------------------------------------------------
__device__ __forceinline__ void prefetch_tensormap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(m) : "memory");
}

__device__ __forceinline__ void tma_store_3d(const CUtensorMap* map, const void* smem_src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
               ::"l"(map), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_group_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_group_read1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_group0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ---- tcgen05: TMEM management -----------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_slot, uint32_t ncols) {  // whole warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_slot)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {  // whole warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---- tcgen05: descriptors ---------------------------------------------------------------------
// Shared-memory matrix descriptor, 128-byte swizzle.  Fields (bits): start>>4 [0,14), LBO>>4 [16,30),
// SBO>>4 [32,46), version=1 [46,48), base_offset [49,52)=0, layout_type [61,64)=2 (SWIZZLE_128B).
__device__ __forceinline__ uint64_t smem_desc_sw128(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr >> 4) & 0x3FFF);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}
// Same descriptor without swizzling (layout_type 0, "interleave"): 8-row x 16-byte core matrices stored contiguously
// (128 B each); for a K-major operand LBO = byte distance between the two core matrices of one K = 16 step, SBO =
// distance between 8-row groups.
__device__ __forceinline__ uint64_t smem_desc_nosw(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr >> 4) & 0x3FFF);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  return d;
}
// Instruction descriptor for kind::f16 with fp32 accumulation.
// c_format F32=1 [4,6); a_format [7,10), b_format [10,13) (0=f16, 1=bf16); a_major bit 15, b_major bit 16
// (0 = K-major, 1 = MN-major); N>>3 [17,23); M>>4 [24,29).
__host__ __device__ constexpr uint32_t make_idesc(int fmt, int a_mn_major, int b_mn_major, int M, int N) {
  return (1u << 4) | (static_cast<uint32_t>(fmt) << 7) | (static_cast<uint32_t>(fmt) << 10) |
         (static_cast<uint32_t>(a_mn_major) << 15) | (static_cast<uint32_t>(b_mn_major) << 16) |
         (static_cast<uint32_t>(N >> 3) << 17) | (static_cast<uint32_t>(M >> 4) << 24);
}

// ---- tcgen05: MMA / commit --------------------------------------------------------------------
// D[tmem] (+)= A[smem desc] * B[smem desc]      (single thread issues)
__device__ __forceinline__ void mma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                       uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// mma_ss with the 64-bit descriptors passed as (lo, hi) register pairs: the issuing thread is a single lane
// running dependent scalar code, so descriptor updates are kept to one 32-bit add.
__device__ __forceinline__ void mma_ss2(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                        uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\tsetp.ne.b32 p, %6, 0;\n\t"
      "mov.b64 da, {%1, %2};\n\tmov.b64 db, {%3, %4};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t}"
      ::"r"(d_tmem), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem desc]   (A: 128 lanes x K 16-bit values packed 2 per column; B descriptor as (lo, hi))
__device__ __forceinline__ void mma_ts2(uint32_t d_tmem, uint32_t a_tmem, uint32_t b_lo, uint32_t b_hi, uint32_t idesc,
                                        uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 db;\n\tsetp.ne.b32 p, %5, 0;\n\t"
      "mov.b64 db, {%2, %3};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], db, %4, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
// mbarrier arrives once all previously issued MMAs of this thread have completed
// (implies tcgen05.fence::before_thread_sync).
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// ---- warp-uniform issue ------------------------------------------------------------------------------
// tcgen05.mma / tcgen05.commit / cp.async.bulk.tensor take their operands from UNIFORM registers.  If the
// issuing code sits in a lane-divergent branch (`if (lane == 0)`), ptxas cannot prove the operands uniform
// and wraps every instruction in an elect / R2UR-broadcast / branch "waterfall" loop (~10 extra dependent
// instructions each).  The *_e variants are executed by the WHOLE warp under warp-uniform control flow and
// elect the issuing lane inside the asm statement, so operands stay in uniform registers.
__device__ __forceinline__ int uniform_warp_idx() { return __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0); }

__device__ __forceinline__ void mbar_arrive_expect_tx_e(uint64_t* bar, uint32_t bytes) {
  asm volatile(
      "{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\t"
      "@P mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n\t}"
      ::"r"(smem_u32(bar)), "r"(bytes)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d_e(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1,
                                              int c2) {
  asm volatile(
      "{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\t"
      "@P cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];\n\t}"
      ::"r"(smem_u32(smem_dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// 1-D bulk copy global -> shared (size a multiple of 16 bytes), completing on an mbarrier like a TMA load
__device__ __forceinline__ void bulk_load_1d_e(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\t"
      "@P cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n\t}"
      ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void mma_ss2_e(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                          uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p, P;\n\t.reg .b64 da, db;\n\tsetp.ne.b32 p, %6, 0;\n\t"
      "mov.b64 da, {%1, %2};\n\tmov.b64 db, {%3, %4};\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "@P tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t}"
      ::"r"(d_tmem), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void mma_commit_e(uint64_t* bar) {
  asm volatile(
      "{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\t"
      "@P tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}"
      ::"r"(smem_u32(bar))
      : "memory");
}

// ---- single-thread region: `if (elect_one_sync()) { ... }` executed by the WHOLE warp under warp-uniform control
// flow.  ptxas recognises the ELECT-derived predicate, so inside the region tcgen05.mma / commit / TMA operands move
// to uniform registers with a plain R2UR (no waterfall loop as for `if (lane == 0)`), and a run of MMAs pays for one
// election instead of one WARPSYNC.COLLECTIVE / ELECT / VOTEU sequence per instruction.
__device__ __forceinline__ bool elect_one_sync() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// ---- tcgen05: TMEM <-> registers (32 lanes x 32-bit, N consecutive columns per thread) ---------
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
// 16 lanes x 256 bit, repeated 8x along the columns: thread t receives, for k = 0..7, columns 8k + 2(t%4) and +1
// of lane (t/4) in r[4k], r[4k+1] and of lane (t/4 + 8) in r[4k+2], r[4k+3] -- the mma C-fragment layout, which is
// what stmatrix consumes.  The lane field of taddr selects lanes 0-15 or 16-31 of the warp's quadrant.
__device__ __forceinline__ void tmem_ld_16x256b_x8(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.16x256b.x8.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_16x256b_x4(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.16x256b.x4.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
// two transposed 8x8 b16 matrices: matrix i takes register r_i; thread t holds elements (col t/4, rows 2(t%4), +1)
// in the (low, high) halves of r_i; row r of matrix i (16 bytes) goes to the address supplied by thread 8i + r (threads 0-15)
__device__ __forceinline__ void stmatrix_x2_trans(uint32_t saddr, uint32_t r0, uint32_t r1) {
  asm volatile("stmatrix.sync.aligned.m8n8.x2.trans.shared.b16 [%0], {%1, %2};" ::"r"(saddr), "r"(r0), "r"(r1) : "memory");
}
__device__ __forceinline__ void tmem_ld64(uint32_t taddr, uint32_t (&r)[64]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x64.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32, %33, %34, %35, %36, %37, %38, %39, %40, %41, %42, %43, %44, %45, %46, %47, %48, %49, %50, %51, %52, %53, %54, %55, %56, %57, %58, %59, %60, %61, %62, %63}, [%64];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31]), "=r"(r[32]), "=r"(r[33]), "=r"(r[34]), "=r"(r[35]), "=r"(r[36]), "=r"(r[37]), "=r"(r[38]), "=r"(r[39]), "=r"(r[40]), "=r"(r[41]), "=r"(r[42]), "=r"(r[43]), "=r"(r[44]), "=r"(r[45]), "=r"(r[46]), "=r"(r[47]), "=r"(r[48]), "=r"(r[49]), "=r"(r[50]), "=r"(r[51]), "=r"(r[52]), "=r"(r[53]), "=r"(r[54]), "=r"(r[55]), "=r"(r[56]), "=r"(r[57]), "=r"(r[58]), "=r"(r[59]), "=r"(r[60]), "=r"(r[61]), "=r"(r[62]), "=r"(r[63])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
               ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
__device__ __forceinline__ uint32_t tmem_ld1(uint32_t taddr) {
  uint32_t r;
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(r) : "r"(taddr) : "memory");
  return r;
}

// ---- 16-bit element helpers ----------------------------------------------------------------------
// 16-byte load from a SHARED-space address.  A pointer that may point to one of several shared arrays is a
// generic pointer to the compiler, which then emits LD.E (generic) instead of LDS; volatile so that it is neither
// hoisted over the barrier that publishes the data nor merged with another load.
__device__ __forceinline__ uint4 lds128u(uint32_t saddr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(saddr));
  return v;
}
template <typename T> struct Elem;
// (qa, qb) += (x * x, y * y) and (sa, sb) += (x, y) as packed fp32x2 operations
__device__ __forceinline__ void sum_sq2(float& sa, float& sb, float& qa, float& qb, float x, float y) {
  asm("{\n\t.reg .b64 v, s, q;\n\tmov.b64 v, {%4, %5};\n\tmov.b64 s, {%0, %1};\n\tmov.b64 q, {%2, %3};\n\t"
      "add.rn.f32x2 s, s, v;\n\tfma.rn.f32x2 q, v, v, q;\n\tmov.b64 {%0, %1}, s;\n\tmov.b64 {%2, %3}, q;\n\t}"
      : "+f"(sa), "+f"(sb), "+f"(qa), "+f"(qb)
      : "f"(x), "f"(y));
}
template <> struct Elem<__nv_bfloat16> {
  static constexpr int kFmt = 1;
  __device__ static __forceinline__ uint32_t pack_relu(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
  }
  __device__ static __forceinline__ uint32_t pack(float lo, float hi) {
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
  }
  __device__ static __forceinline__ float to_float(__nv_bfloat16 v) { return __bfloat162float(v); }
  __device__ static __forceinline__ float2 unpack2(uint32_t w) {
    return make_float2(__uint_as_float(w << 16), __uint_as_float(w & 0xffff0000u));
  }
  __device__ static __forceinline__ uint16_t bits(float v) { return __bfloat16_as_ushort(__float2bfloat16_rn(v)); }
  __device__ static __forceinline__ __nv_bfloat16 from_float(float v) { return __float2bfloat16_rn(v); }
};
template <> struct Elem<__half> {
  static constexpr int kFmt = 0;
  __device__ static __forceinline__ uint32_t pack_relu(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
  }
  __device__ static __forceinline__ uint32_t pack(float lo, float hi) {
    __half2 v = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
  }
  __device__ static __forceinline__ float to_float(__half v) { return __half2float(v); }
  __device__ static __forceinline__ float2 unpack2(uint32_t w) {
    return __half22float2(*reinterpret_cast<const __half2*>(&w));
  }
  __device__ static __forceinline__ uint16_t bits(float v) { return __half_as_ushort(__float2half_rn(v)); }
  __device__ static __forceinline__ __half from_float(float v) { return __float2half_rn(v); }
};

}  // namespace ptx
}  // namespace fgnn
