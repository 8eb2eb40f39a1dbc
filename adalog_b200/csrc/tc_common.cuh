// tcgen05 / TMA / mbarrier PTX wrappers and the tensor-map builder shared by the candidate GEMM kernels (sm_100a).
#pragma once
#include "common.cuh"
#include "quant_device.cuh"
#include <cuda.h>
#include <cudaTypedefs.h>

namespace adalog {

constexpr int kBM = 128;                // UMMA M = candidates per unit
constexpr int kBK = 64;                 // bf16 elements = one 128-byte swizzle row (128 int8 elements)

// ---------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// bounded wait: a pipeline bug traps (launch error) instead of hanging the GPU box.  try_wait carries a suspend-time
// hint so a waiting lane sleeps in hardware instead of spinning in the issue slots the epilogue warps need.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  uint32_t done = 0;
  long long t0 = 0;
  for (uint32_t it = 0;; ++it) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done) : "r"(addr), "r"(parity), "r"(0x989680u) : "memory");
    if (done) break;
    if ((it & 0xff) == 0xff) {
      if (t0 == 0) t0 = clock64();
      else if (clock64() - t0 > 4000000000ll) {  // ~2 s
        printf("adalog: mbarrier timeout (block %d,%d thread %d parity %u)\n", blockIdx.x, 0,
               threadIdx.x, parity);
        __trap();
      }
    }
  }
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tma_load_2d(const CUtensorMap* map, uint64_t* bar, void* dst, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

// K-major, SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor, sm_100 "version 1"):
//   [0,14) start>>4 | [16,30) LBO>>4 (=1, ignored for swizzled K-major) | [32,46) SBO>>4 (8 rows*128B = 1024)
//   [46,48) version=1 | [61,64) layout = 2 (SWIZZLE_128B)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// kind::f16 instruction descriptor: D=F32 (bit4), A=BF16 (bit7), B=BF16 (bit10), K-major both, N>>3 @17, M>>4 @24
__device__ __forceinline__ uint32_t make_idesc(int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(kBM >> 4) << 24);
}
// kind::i8: D=S32 (2 @ bit4), A = B = signed int8 (1 @ bit7, 1 @ bit10), no saturation, K-major both
__device__ __forceinline__ uint32_t make_idesc_i8(int n) {
  return (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(kBM >> 4) << 24);
}
__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
      : "memory");
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// Lean issue path for a CONVERGED warp (all 32 lanes in lock step, every operand warp-uniform): the four K slices of
// one 128-byte K block (the descriptor start address advances by 32 bytes = 2 units per slice) followed by the commit
// of `bar_addr`, issued by one elected lane inside a single asm block.  The one-lane form above (`if (lane == 0)`
// around umma_* / umma_commit) costs ~17 SASS instructions per MMA: ptxas wraps every tcgen05 instruction of a
// divergent region in an elect / R2UR / BRA.U.ANY "waterfall" because its operands must sit in uniform registers.
// ncu on the linear activation sweeps: the issuing warp ran 280 instructions per K block against 768 clocks of MMA
// work and was never found waiting at a barrier -- the tensor pipe (41-51% active) was bound by this instruction stream.
template <bool I8>
__device__ __forceinline__ void umma_kblock_commit(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                                   uint32_t acc_first, int ks, uint32_t bar_addr) {
  // ks = live K slices of this block (1..4; slices that are all K padding are skipped); bar_addr == 0: no commit
#define ADALOG_UMMA_KBLOCK(KIND)                                                                          \
  asm volatile(                                                                                           \
      "{\n\t.reg .pred pe, p0, pt, p1, p2, p3, pc;\n\t.reg .b64 a1, a2, a3, b1, b2, b3;\n\t"              \
      "elect.sync _|pe, 0xffffffff;\n\t"                                                                  \
      "setp.ne.b32 p0, %4, 0;\n\t"                                                                        \
      "setp.eq.b32 pt, %4, %4;\n\t"                                                                       \
      "setp.gt.and.s32 p1, %5, 1, pe;\n\t"                                                                \
      "setp.gt.and.s32 p2, %5, 2, pe;\n\t"                                                                \
      "setp.gt.and.s32 p3, %5, 3, pe;\n\t"                                                                \
      "setp.ne.and.b32 pc, %6, 0, pe;\n\t"                                                                \
      "add.s64 a1, %1, 2;\n\tadd.s64 a2, %1, 4;\n\tadd.s64 a3, %1, 6;\n\t"                                \
      "add.s64 b1, %2, 2;\n\tadd.s64 b2, %2, 4;\n\tadd.s64 b3, %2, 6;\n\t"                                \
      "@pe tcgen05.mma.cta_group::1.kind::" KIND " [%0], %1, %2, %3, p0;\n\t"                              \
      "@p1 tcgen05.mma.cta_group::1.kind::" KIND " [%0], a1, b1, %3, pt;\n\t"                              \
      "@p2 tcgen05.mma.cta_group::1.kind::" KIND " [%0], a2, b2, %3, pt;\n\t"                              \
      "@p3 tcgen05.mma.cta_group::1.kind::" KIND " [%0], a3, b3, %3, pt;\n\t"                              \
      "@pc tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%6];\n\t}"              \
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc_first), "r"(ks), "r"(bar_addr)          \
      : "memory")
  if (I8) ADALOG_UMMA_KBLOCK("i8");
  else    ADALOG_UMMA_KBLOCK("f16");
#undef ADALOG_UMMA_KBLOCK
}
// commit issued by one elected lane of a converged warp
__device__ __forceinline__ void umma_commit_elect(uint32_t bar_addr) {
  asm volatile(
      "{\n\t.reg .pred pe;\n\telect.sync _|pe, 0xffffffff;\n\t"
      "@pe tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}"
      ::"r"(bar_addr) : "memory");
}
// warp index the compiler can prove warp-uniform (so that everything derived from it may live in uniform registers)
__device__ __forceinline__ int uniform_warp_idx() { return __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0); }

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
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
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// 32 lanes x 32 columns of zeros (TMEM is not cleared by tcgen05.alloc)
__device__ __forceinline__ void tmem_st32_zero(uint32_t taddr) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, "
      "%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1};"
      ::"r"(taddr), "r"(0u) : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// (packed FP32 helpers fmul2 / fadd2 / ffma2 and the two-sum accumulator live in quant_device.cuh)


// ---------------------------------------------------------------- host side
inline PFN_cuTensorMapEncodeTiled_v12000 get_encode() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
  }
  return fn;
}

// 2-D row-major [rows, cols] operand (bf16 or int8), box [box_rows, 128 bytes], 128-byte swizzle
inline int make_map(CUtensorMap* m, const void* base, int64_t rows, int64_t cols, int box_rows, bool i8) {
  auto enc = get_encode();
  if (!enc) return fail(-20, "cuTensorMapEncodeTiled entry point not found");
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0) return fail(-21, "operand base not 16-byte aligned");
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)cols * (i8 ? 1 : 2)};
  cuuint32_t box[2] = {(cuuint32_t)(i8 ? 2 * kBK : kBK), (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, i8 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base),
                   dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(-22, "cuTensorMapEncodeTiled failed (%d) rows=%lld cols=%lld box_rows=%d", (int)r,
                                     (long long)rows, (long long)cols, box_rows);
  return 0;
}


}  // namespace adalog
