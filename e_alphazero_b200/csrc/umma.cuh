// umma.cuh -- hand-written sm_100a plumbing for the tensor-core network path:
// mbarriers, 1-D bulk async copies (UBLKCP), TMEM allocation, tcgen05.mma
// (kind::tf32, operands from shared memory), tcgen05.commit / ld, and the
// shared-memory operand layout used throughout:
//
//   K-major, SWIZZLE_NONE ("interleave") canonical layout, 4-byte elements:
//   core matrix = 8 rows x 16 B (4 elements), stored contiguously (128 B);
//   a [rows x 32] K-chunk is laid out [row/8][k/4][row%8][k%4]:
//       byte offset(row, k) = (row/8)*1024 + (k/4)*128 + (row%8)*16 + (k%4)*4
//   => descriptor LBO (K-adjacent core matrices) = 128 B, SBO (8-row groups) = 1024 B.
//   One tcgen05.mma kind::tf32 consumes K = 8 (two core matrices): K-step j starts at +256*j B.
//
// fp32 accuracy comes from the 3xTF32 split: x = hi + lo with hi = x & 0xFFFFE000,
// lo = x - hi (exact); D += A_hi*B_hi + A_hi*B_lo + A_lo*B_hi, fp32 accumulation in TMEM.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace eaz {
namespace umma {

constexpr int kChunkK = 32;                    // K elements per pipeline stage
constexpr int kRowGroupBytes = 1024;           // SBO: 8 rows x 32 k x 4 B
constexpr int kCoreBytes = 128;                // LBO
constexpr int kKStepBytes = 256;               // 8 tf32 = two core matrices
constexpr int kKSteps = kChunkK / 8;           // MMAs per chunk per product

__host__ __device__ inline int tile_offset(int row, int k) {  // bytes, within one [rows x 32] chunk
  return (row >> 3) * kRowGroupBytes + (k >> 2) * kCoreBytes + (row & 7) * 16 + (k & 3) * 4;
}
// same layout for a [rows x CK] chunk (CK = 16 or 32): the 8-row group stride (SBO) is CK/4 core matrices
template <int CK>
__host__ __device__ inline int tile_offset_ck(int row, int k) {
  return (row >> 3) * (CK / 4) * kCoreBytes + (k >> 2) * kCoreBytes + (row & 7) * 16 + (k & 3) * 4;
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}

// One lane polls (hundreds of polling threads starve the shared-memory pipe), but the LOOP is warp-uniform: the poll is a predicated
// instruction and the exit condition a vote.  `if (lane == 0) mbar_wait(); __syncwarp();` leaves lane 0 and lanes 1..31 as two
// separately scheduled groups whenever lane 0 actually had to loop; the code after it then issues every instruction twice and
// re-synchronises at every shuffle (measured in psearch.cuh: the same tree step took 4.8 us in warps whose first poll succeeded and
// 13 us in warps that had to wait; profiles/r2_summary.md).
__device__ __forceinline__ void mbar_wait_warp(uint64_t* bar, uint32_t parity) {
  const bool poller = (threadIdx.x & 31) == 0;
  while (true) {
    uint32_t ok = 0;
    if (poller) ok = mbar_try_wait(bar, parity) ? 1u : 0u;
    if (__any_sync(0xffffffffu, ok != 0)) break;
  }
}
// One lane of the (converged) warp.  tcgen05.mma issued under `if (elect_one())` from warp-uniform values takes its descriptors from
// uniform registers; inside an `if (lane == 0)` region the compiler wraps every tcgen05.mma in an ELECT / R2UR.BROADCAST loop
// (~100 cycles per instruction).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n"
      ".reg .pred P;\n"
      "elect.sync _|P, 0xffffffff;\n"
      "selp.u32 %0, 1, 0, P;\n"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

// ---- 1-D bulk async copy global -> shared (SASS UBLKCP), completion on an mbarrier
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
// generic-proxy writes (st.shared) -> visible to the async proxy (tcgen05.mma operand reads)
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {  // whole warp, ncols power of two >= 32
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() { asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ---- descriptors
// shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start>>4 [0,14), LBO>>4 [16,30), SBO>>4 [32,46),
// version=1 [46,48), layout_type=SWIZZLE_NONE [61,64)
__device__ __forceinline__ uint64_t smem_desc(uint32_t saddr, uint32_t sbo_bytes = kRowGroupBytes) {
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(kCoreBytes >> 4) << 16) | ((uint64_t)(sbo_bytes >> 4) << 32) | (1ull << 46);
}
// instruction descriptor (cute::UMMA::InstrDescriptor) for kind::tf32, fp32 accumulate, K-major A and B
__host__ __device__ inline uint32_t idesc_tf32(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// D[tmem] (+)= A[smem] * B[smem]^T ; one elected thread issues
__device__ __forceinline__ void mma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// all previously issued MMAs of this thread arrive on the mbarrier when complete (implies fence::before_thread_sync)
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// ---- TMEM -> registers: lane i of the warp reads TMEM lane (lane_base + i), 32 consecutive 32-bit columns
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
        "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// ---- registers -> TMEM: lane i of the warp writes TMEM lane (lane_base + i), 8 consecutive 32-bit columns
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint4& a, const uint4& b) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(a.x), "r"(a.y), "r"(a.z), "r"(a.w),
               "r"(b.x), "r"(b.y), "r"(b.z), "r"(b.w)
               : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---- 3xTF32 split
__device__ __forceinline__ void split_tf32(float x, uint32_t& hi, uint32_t& lo) {
  hi = __float_as_uint(x) & 0xFFFFE000u;
  lo = __float_as_uint(__fsub_rn(x, __uint_as_float(hi)));
}

}  // namespace umma
}  // namespace eaz

// ---- scaled 3xFP16 variant (mlp_tensor.cu): same byte geometry, 2-byte elements.
// x*S = hi + lo (hi, lo fp16, ~22 significant bits); D += A_hi*B_hi + A_hi*B_lo + A_lo*B_hi; S is a power of two
// removed exactly in the epilogue.  kind::f16 consumes K = 16 per instruction (two 16-byte core-matrix columns).
#include <cuda_fp16.h>
namespace eaz {
namespace umma {
__host__ __device__ inline uint32_t idesc_f16(int M, int N) {  // F16 x F16 -> F32, K-major A and B
  return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void mma_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// A operand from TENSOR MEMORY (row m = TMEM lane m, two consecutive-k fp16 per 32-bit column), B from shared memory
__device__ __forceinline__ void mma_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n"
      "}\n" ::"r"(d_tmem),
      "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// byte offset of element (row, k) in a [rows x 32] fp16 chunk tile (64 B per row = 4 core-matrix columns)
__host__ __device__ inline int tile_offset_h32(int row, int k) {
  return (row >> 3) * 512 + (k >> 3) * kCoreBytes + (row & 7) * 16 + (k & 7) * 2;
}
__device__ __forceinline__ void split_f16(float xs, __half& hi, __half& lo) {  // xs already scaled and range-clamped
  hi = __float2half_rn(xs);
  lo = __float2half_rn(__fsub_rn(xs, __half2float(hi)));
}
}  // namespace umma
}  // namespace eaz
