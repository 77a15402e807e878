// tc_common.cuh — shared tcgen05 / TMEM / TMA / mbarrier helpers (inline PTX, sm_100a) used by the
// score+select filter (score_select_tc.cu) and the tensor-core cross-entropy (ce_tc.cu).
#pragma once
#include "pcv_common.cuh"

namespace pcv {

constexpr int TC_BM = 128;
constexpr int TC_BN = 256;
constexpr int TC_D = 8;
constexpr int TC_STAGES = 16;  // 8 KB tiles: ~16 in flight to cover the L2/HBM latency (Little)
constexpr int TC_EPI_WARPS = 8;                      // multiple of 4 (each warp reads one TMEM lane quarter)
constexpr int TC_SLICES = TC_EPI_WARPS / 4;          // column slices of a 256-column tile
constexpr int TC_SW = TC_BN / TC_SLICES;             // columns per slice
constexpr int TC_THREADS = 64 + 32 * TC_EPI_WARPS;  // warp0 TMA, warp1 MMA/TMEM, 8 epilogue warps
constexpr uint32_t TC_TILE_BYTES = TC_BN * TC_D * 4;

// embedding dims served by the tcgen05 engines (filter and cross-entropy): 1, 2, 4, 8 or 16 k-atoms of 8 fp32
inline bool tc_dim_ok(int dim) { return dim == 8 || dim == 16 || dim == 32 || dim == 64 || dim == 128; }

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(void *bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(void *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(void *bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(void *bar, uint32_t parity) {
  uint32_t addr = smem_u32(bar);
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra WAIT_DONE;\n"
      "bra WAIT_LOOP;\n"
      "WAIT_DONE:\n"
      "}\n" ::"r"(addr), "r"(parity) : "memory");
}

// same, on a precomputed 32-bit shared address (keeps the generic->shared conversion out of hot loops)
__device__ __forceinline__ void mbar_wait_u32(uint32_t addr, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra WAIT_DONE;\n"
      "bra WAIT_LOOP;\n"
      "WAIT_DONE:\n"
      "}\n" ::"r"(addr), "r"(parity) : "memory");
}
__device__ __forceinline__ void mbar_arrive_u32(uint32_t addr) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(addr) : "memory");
}

// TMA bulk copy global -> shared (contiguous bytes), completion on an mbarrier
__device__ __forceinline__ void tma_bulk_load(void *dst, const void *src, uint32_t bytes, void *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// K-major, SWIZZLE_32B shared-memory matrix descriptor: rows of 32 B, 8-row groups 256 B apart.
__device__ __forceinline__ uint64_t umma_desc_sw32(const void *smem) {
  uint64_t d = (uint64_t)((smem_u32(smem) & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;          // leading byte offset (unused for swizzled K-major)
  d |= (uint64_t)(256 >> 4) << 32; // stride byte offset between 8-row groups
  d |= (uint64_t)1 << 46;          // descriptor version (Blackwell)
  d |= (uint64_t)6 << 61;          // LayoutType::SWIZZLE_32B
  return d;
}

// kind::tf32, fp32 accumulate, A and B K-major, M=128, N=256
constexpr uint32_t TC_IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(TC_BN >> 3) << 17) |
                              ((uint32_t)(TC_BM >> 4) << 24);

__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(void *bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// Converged issue: ALL 32 lanes of the MMA warp run the issue loop and one elected lane issues each tcgen05
// instruction.  With a single-lane branch around the loop the compiler moves every operand vector -> uniform register
// (R2UR) per MMA: ~25 latency-bound single-thread instructions per MMA, which bounds kernels that issue many small MMAs
// per tile (measured on the CE gradient MMAs: 1.09 ms -> 0.70 ms).
__device__ __forceinline__ void umma_tf32_elect(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                                uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p, q;\n"
      "elect.sync _|q, 0xffffffff;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit_elect(void *bar) {
  asm volatile(
      "{\n"
      ".reg .pred q;\n"
      "elect.sync _|q, 0xffffffff;\n"
      "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n"
      "}\n" ::"r"(smem_u32(bar)) : "memory");
}

#define TC_LD32(v, taddr)                                                                                   \
  asm volatile(                                                                                             \
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "                                                             \
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "                             \
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"             \
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),     \
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]),            \
        "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]),          \
        "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]),          \
        "=r"(v[29]), "=r"(v[30]), "=r"(v[31])                                                               \
      : "r"(taddr))

// The wait names the destination registers as in/out operands so the compiler
// cannot move any use of them above the wait.
#define TC_WAIT_LD(v)                                                                                       \
  asm volatile("tcgen05.wait::ld.sync.aligned;"                                                             \
               : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]),        \
                 "+r"(v[7]), "+r"(v[8]), "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]),    \
                 "+r"(v[14]), "+r"(v[15]), "+r"(v[16]), "+r"(v[17]), "+r"(v[18]), "+r"(v[19]), "+r"(v[20]), \
                 "+r"(v[21]), "+r"(v[22]), "+r"(v[23]), "+r"(v[24]), "+r"(v[25]), "+r"(v[26]), "+r"(v[27]), \
                 "+r"(v[28]), "+r"(v[29]), "+r"(v[30]), "+r"(v[31])::"memory")

__device__ __forceinline__ float max3(float a, float b, float c) { return fmaxf(fmaxf(a, b), c); }


}  // namespace pcv
