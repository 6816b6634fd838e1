// aps_tc_ptx.cuh -- sm_100a PTX wrappers shared by the tensor-core kernels (aps_knn_tc.cu, aps_pair_screen.cu):
// mbarrier pipelines, TMA (cp.async.bulk.tensor) loads, tcgen05.mma / commit / ld, shared-memory matrix
// descriptors and the host-side tensor-map encoder.  Everything is static / inline: one copy per translation unit.
#pragma once
#include <cstdio>
#include <cuda.h>
#include <math_constants.h>

#include "aps_common.cuh"

namespace aps_tc {

constexpr int KSLAB = 64;      // 16-bit elements per 128-byte swizzle row

// ---- PTX helpers -------------------------------------------------------------------------------
static __device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// One thread of a fully active warp.  Guarding the single-thread TMA / tcgen05.mma issue loops with elect.sync instead of
// "lane == 0" lets the compiler keep descriptors and addresses in uniform registers; a lane-id guard makes it wrap
// every UTCHMMA / UTMALDG in a ~20-instruction R2UR "waterfall" loop (profiles/r2_ncu_history.txt).
static __device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
static __device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
// The uint32_t overloads take the barrier's 32-bit shared-window address: per-tile loops compute it once.
static __device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
static __device__ __forceinline__ void mbar_arrive(uint64_t* bar) { mbar_arrive(smem_u32(bar)); }
static __device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// try_wait suspends the thread in hardware until the phase completes or the hint (ns) elapses: the
// polling loops of the producer / MMA lanes then cost almost no issue slots (they were 21 % of all
// executed instructions with the default time limit -- profiles/r1_ncu_history.txt)
constexpr uint32_t kSuspendHintNs = 20000;
static __device__ __forceinline__ void mbar_wait(uint32_t addr, uint32_t parity) {
  uint32_t done;
#ifdef APS_TC_WATCHDOG
  uint32_t spins = 0;
#endif
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(addr), "r"(parity), "r"(kSuspendHintNs)
        : "memory");
#ifdef APS_TC_WATCHDOG   // debugging aid: name the barrier a deadlocked role is parked on, then trap
    if (!done && ++spins > (1u << 16)) {
      printf("mbar watchdog: block %d thread %d barrier smem+0x%x parity %u\n", (int)blockIdx.x, (int)threadIdx.x, addr, parity);
      __trap();
    }
#endif
  } while (!done);
}
static __device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) { mbar_wait(smem_u32(bar), parity); }
// producer / MMA-issuer flavour: back off between probes so the spinning lane does not steal issue
// slots from the epilogue warp that shares its SM sub-partition
static __device__ __forceinline__ void mbar_wait_backoff(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  uint32_t done;
  for (;;) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(addr), "r"(parity), "r"(kSuspendHintNs)
        : "memory");
    if (done) break;
    __nanosleep(40);
  }
}
static __device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(c0), "r"(c1), "r"(smem_u32(bar))
      : "memory");
}
static __device__ __forceinline__ void bulk_load_1d(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
static __device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
static __device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
static __device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
static __device__ __forceinline__ void tc_commit(uint64_t* bar) { tc_commit(smem_u32(bar)); }
// D[tmem] (+)= A[smem] * B[smem]^T ; kind::f16 (bf16 inputs, fp32 accumulate)
static __device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// 32 lanes x 32 columns of 32-bit accumulators: thread i <- TMEM lane (quadrant*32 + i)
static __device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
// 32 lanes x 8 columns (one column group of the selection epilogue, re-read on the rare candidate path)
static __device__ __forceinline__ void tmem_ld8(uint32_t taddr, float (&v)[8]) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
}
static __device__ __forceinline__ void tmem_wait_ld8(float (&v)[8]) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7])
               :
               : "memory");
}
// The wait names the destination registers as in/out operands so the compiler cannot schedule a use of
// them above the wait (tcgen05.ld is asynchronous).
static __device__ __forceinline__ void tmem_wait_ld(float (&v)[32]) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                 "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]),
                 "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]),
                 "+r"(r[23]), "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]),
                 "+r"(r[30]), "+r"(r[31])
               :
               : "memory");
}

// K-major, SWIZZLE_128B shared-memory matrix descriptor (sm_100 format: version 1 at bit 46,
// layout type 2 at bits 61-63, SBO = 1024 B between 8-row groups, LBO unused for swizzled K-major).
static __device__ __forceinline__ uint64_t make_kmajor_sw128_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);        // start address, bits [0,14)
  d |= (uint64_t)0 << 16;                             // leading byte offset (ignored)
  d |= (uint64_t)(1024 >> 4) << 32;                   // stride byte offset, bits [32,46)
  d |= (uint64_t)1 << 46;                             // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;                             // SWIZZLE_128B
  return d;
}

// instruction descriptor: kind::f16, A/B = BF16, D = F32, both K-major, M x N
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}


// instruction descriptor: kind::f16, A/B = F16, D = F32
__host__ __device__ constexpr uint32_t make_idesc_f16_f32acc(int M, int N) {
  return (1u << 4) | (0u << 7) | (0u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// instruction descriptor: kind::f16, A/B = F16, D = F16 (packed half accumulators), both K-major, M x N
__host__ __device__ constexpr uint32_t make_idesc_f16_f16acc(int M, int N) {
  return (0u << 4) | (0u << 7) | (0u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// ---- host side -----------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// Resolved once per process; the function-local static makes the first call thread-safe (several host threads build
// tensor maps at once when a device group runs its members in parallel).
static PFN_encodeTiled get_encode() {
  static const PFN_encodeTiled fn = []() -> PFN_encodeTiled {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      return (PFN_encodeTiled)p;
    return nullptr;
  }();
  return fn;
}

static int make_map(CUtensorMap* map, const void* base, int64_t rows, int dp, int box_rows,
                    CUtensorMapDataType dt = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) {
    aps_set_error(APS_ERR_CUDA, "", "cuTensorMapEncodeTiled is not available from the driver");
    return APS_ERR_CUDA;
  }
  cuuint64_t dims[2] = {(cuuint64_t)dp, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)dp * 2};
  cuuint32_t box[2] = {(cuuint32_t)KSLAB, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, dt, 2, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    aps_set_error(APS_ERR_CUDA, "", "cuTensorMapEncodeTiled failed (%d)", (int)r);
    return APS_ERR_CUDA;
  }
  return APS_OK;
}


}  // namespace aps_tc
