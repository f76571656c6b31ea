// Shared helpers for the sm_100a kernels: error plumbing, PTX wrappers (mbarrier, TMA, tcgen05),
// exact-rounding fp32 intrinsics.  No torch types anywhere below the C-ABI (include/frcnn_b200.h).
#pragma once
#include <cuda_runtime.h>
#include <cuda.h>
#include <stdint.h>
#include <stdio.h>

namespace frcnn {

// ---- error plumbing: every C-ABI entry returns an int status; message kept per thread -------
enum Status : int {
  OK = 0, ERR_CUDA = -1, ERR_ARG = -2, ERR_NO_DEVICE = -3, ERR_DRIVER_ENTRY = -4, ERR_CAPACITY = -5
};
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what, const char* file, int line);

#define FRCNN_CUDA(expr)                                                        \
  do {                                                                          \
    cudaError_t _e = (expr);                                                    \
    if (_e != cudaSuccess) return ::frcnn::cuda_fail(_e, #expr, __FILE__, __LINE__); \
  } while (0)

#define FRCNN_LAUNCH_CHECK() FRCNN_CUDA(cudaGetLastError())

#define FRCNN_REQUIRE(cond, ...)                    \
  do {                                              \
    if (!(cond)) {                                  \
      ::frcnn::set_error(__VA_ARGS__);              \
      return ::frcnn::ERR_ARG;                      \
    }                                               \
  } while (0)

static inline int cdiv(int a, int b) { return (a + b - 1) / b; }

// ---- device-side PTX wrappers -------------------------------------------------------------
#if defined(__CUDACC__)

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// mbarrier ------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// arrive that the compiler must order after the computation of `dep` (an otherwise unused register operand)
__device__ __forceinline__ void mbar_arrive_after(uint64_t* bar, uint32_t dep) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0]; // after %1" ::"r"(smem_u32(bar)), "r"(dep) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t addr = smem_u32(bar);
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%0], %1;\n\t"
      "@P bra WAIT_DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "WAIT_DONE:\n\t}\n" ::"r"(addr), "r"(parity) : "memory");
}

// ---- development watchdog (builds with -DFRCNN_WATCHDOG only: libfrcnn_b200_wd.so) -------------------------------------
// A barrier-protocol bug in a warp-specialised kernel shows up as a hang, which on a leased GPU box is a lost call with no
// information.  In watchdog builds every tagged wait gives up after ~0.2 s, records who waited on what, and raises a
// device-wide abort flag that makes every other tagged wait fall through, so the kernel terminates (with garbage) and the
// host can read the record through frcnn_debug_watchdog().  Normal builds compile MBAR_WAIT to the plain wait.
#ifdef FRCNN_WATCHDOG
static __device__ unsigned int g_watchdog[16];   // per translation unit (only conv_gemm.cu uses it)
//   // [0] abort flag, [1] count, [2..7] first record: block, thread, tag, parity, kbt, spare
__device__ __forceinline__ void mbar_wait_wd(uint64_t* bar, uint32_t parity, uint32_t tag, uint32_t aux) {
  const uint32_t addr = smem_u32(bar);
  long long t0 = 0;
  for (uint32_t it = 0;; ++it) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred P;\n\tmbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\tselp.u32 %0, 1, 0, P;\n\t}\n"
                 : "=r"(ok) : "r"(addr), "r"(parity) : "memory");
    if (ok) return;
    if ((it & 63u) == 63u) {
      if (*(volatile unsigned int*)&g_watchdog[0]) return;
      const long long now = clock64();
      if (t0 == 0) t0 = now;
      else if (now - t0 > 400000000LL) {
        if (atomicAdd(&g_watchdog[1], 1u) == 0u) {
          g_watchdog[2] = blockIdx.x; g_watchdog[3] = threadIdx.x; g_watchdog[4] = tag; g_watchdog[5] = parity; g_watchdog[6] = aux;
        }
        __threadfence();
        atomicExch(&g_watchdog[0], 1u);
        return;
      }
    }
  }
}
#define MBAR_WAIT(bar, parity, tag, aux) mbar_wait_wd(bar, parity, tag, (uint32_t)(aux))
#else
#define MBAR_WAIT(bar, parity, tag, aux) mbar_wait(bar, parity)
#endif

// tcgen05 fences around thread synchronisation ---------------------------------------------------
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// TMA ------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

// tcgen05 ---------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem] (+)= A * B, TF32 operands, fp32 accumulate, single CTA; A operand read from tensor memory (lane = row, one 32-bit column per tf32 element), B from shared memory
__device__ __forceinline__ void umma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}\n"
      ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
// D[tmem] (+)= A * B, FP16 operands (K = 16 per instruction), fp32 accumulate, single CTA; A from tensor memory (lane = row,
// one 32-bit column per PAIR of K-consecutive fp16 values: 8 columns per instruction), B from shared memory
__device__ __forceinline__ void umma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n"
      ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
// same, the shared-memory descriptor given as (low word, constant high word); `accumulate` run-time
__device__ __forceinline__ void umma_f16_ts_lo(uint32_t tmem_d, uint32_t tmem_a, uint32_t desc_lo, uint32_t desc_hi, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 d;\n\t"
      "setp.ne.b32 p, %5, 0;\n\t"
      "mov.b64 d, {%2, %3};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], d, %4, p;\n\t}\n"
      ::"r"(tmem_d), "r"(tmem_a), "r"(desc_lo), "r"(desc_hi), "r"(idesc), "r"(accumulate) : "memory");
}
// ... and always accumulating
__device__ __forceinline__ void umma_f16_ts_acc(uint32_t tmem_d, uint32_t tmem_a, uint32_t desc_lo, uint32_t desc_hi, uint32_t idesc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 d;\n\t"
      "setp.eq.b32 p, 0, 0;\n\t"
      "mov.b64 d, {%2, %3};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], d, %4, p;\n\t}\n"
      ::"r"(tmem_d), "r"(tmem_a), "r"(desc_lo), "r"(desc_hi), "r"(idesc) : "memory");
}
// wait for TWO barriers with one pair of try_waits per round (their ~90-cycle latencies overlap)
__device__ __forceinline__ void mbar_wait2(uint32_t bar0, uint32_t par0, uint32_t bar1, uint32_t par1) {
  asm volatile(
      "{\n\t.reg .pred P0, P1;\n\t"
      "WAIT2_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P0, [%0], %1;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%2], %3;\n\t"
      "and.pred P0, P0, P1;\n\t"
      "@P0 bra WAIT2_DONE;\n\t"
      "bra WAIT2_LOOP;\n\t"
      "WAIT2_DONE:\n\t}\n" ::"r"(bar0), "r"(par0), "r"(bar1), "r"(par1) : "memory");
}
// register re-allocation between warp roles: every warp of a warpgroup (4 consecutive warps) executes the same one
template <int R> __device__ __forceinline__ void reg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(R)); }
template <int R> __device__ __forceinline__ void reg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(R)); }
// two fp32 -> packed fp16x2 (lo half = a, hi half = b), round to nearest even, IEEE overflow: |x| >= 65520 becomes +-Inf and
// NaN stays NaN (no .satfinite: a saturated operand would turn an out-of-range activation into a finite, wrong product)
__device__ __forceinline__ uint32_t pack_f16x2_rn(float a, float b) {
  uint32_t r;
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}
// one lane of a converged warp (the rest of the warp stays converged: operands remain in uniform registers)
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}\n" : "=r"(pred));
  return pred != 0;
}
// arrive on an mbarrier once all previously issued MMAs of this thread have completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// 32 lanes x 32 consecutive fp32 columns -> 32 registers per thread (thread = TMEM lane)
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t* v) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// 32 registers per thread -> this thread's TMEM lane, 32 consecutive columns
__device__ __forceinline__ void tmem_st_32x32(uint32_t taddr, const uint32_t* v) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
        "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]),
        "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]),
        "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
      : "memory");
}
// 16 registers per thread -> this thread's TMEM lane, 16 consecutive columns
__device__ __forceinline__ void tmem_st_32x16(uint32_t taddr, const uint32_t* v) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
        "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// read-only global loads the compiler may neither duplicate nor sink (asm volatile): used where the loads must be
// issued early, all together, to hide their latency (conv epilogue)
__device__ __forceinline__ float4 ld_nc_f4_pinned(const float* p) {
  float4 v;
  asm volatile("ld.global.nc.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  return v;
}
__device__ __forceinline__ float ld_nc_f32_pinned(const float* p) {
  float v;
  asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}

// 128-bit load from a 32-bit shared-space address
__device__ __forceinline__ float4 lds_f4(uint32_t saddr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(saddr));
  return v;
}

// programmatic dependent launch: let the next kernel in the stream start its prologue early / wait for the previous one's data
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// same rounding (nearest, ties away from zero) for finite inputs in two integer ops: add half a tf32 ulp to the magnitude
// bits, clear the low 13 bits.  cvt.rna.tf32 additionally special-cases Inf/NaN (an extra compare + select per element),
// which the operand splitter -- it shares its scheduler with the MMA-issuing warp -- does not need.
__device__ __forceinline__ float to_tf32_fast(float x) {
  return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u);
}

// round-to-nearest fp32 -> tf32 (result is an fp32 bit pattern with the low 13 mantissa bits clear)
__device__ __forceinline__ float to_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}

#endif  // __CUDACC__
}  // namespace frcnn
