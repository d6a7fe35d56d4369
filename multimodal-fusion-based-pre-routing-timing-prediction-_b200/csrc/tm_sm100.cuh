// sm_100a primitives shared by the tcgen05 kernels: mbarriers, non-tensor bulk copies, async-proxy and
// tcgen05 fences, tensor-memory allocation and loads, tcgen05.mma and its shared-memory / instruction
// descriptors.  Every PTX statement of that kind in the library lives here, so the descriptor bit layouts
// and the barrier-wait policies are written down once.
#pragma once
#include <stdint.h>

namespace tmk {
namespace sm100 {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---------------------------------------------------------------------------------------------
// mbarriers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
// makes initialised barriers visible to the other threads and to the async proxy (TMA, tcgen05.commit)
__device__ __forceinline__ void fence_mbarrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// arrive and announce `bytes` of asynchronous copies that complete on this barrier
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// one probe: has the phase with this parity completed?
__device__ __forceinline__ bool mbar_try_wait(uint32_t addr, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(done) : "r"(addr), "r"(parity) : "memory");
  return done != 0;
}
// Every mbarrier wait is bounded: a lost arrival or a tensor-core fault must end the launch, not hang the
// GPU.  Two policies:
//   mbar_wait_trap<SPINS>   traps after SPINS probes (the launch fails with an error).
//   mbar_wait_abort         gives up after 2^24 probes, or as soon as another role of the CTA has given up
//                           (*abort != 0, polled every 1024 probes), and returns false; the caller raises its
//                           error flag and drains, so the failure is reported without killing the context.
template <uint32_t SPINS>
__device__ __forceinline__ void mbar_wait_trap(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  for (uint32_t spin = 0;; ++spin) {
    if (mbar_try_wait(addr, parity)) return;
    if (spin > SPINS) __trap();
  }
}
__device__ __forceinline__ bool mbar_wait_abort(uint64_t* bar, uint32_t parity, volatile int* abort) {
  const uint32_t addr = smem_u32(bar);
  for (uint32_t spin = 0; spin < (1u << 24); ++spin) {
    if ((spin & 1023u) == 1023u && *abort) return false;
    if (mbar_try_wait(addr, parity)) return true;
  }
  return false;
}

// non-tensor bulk copy global -> shared (dst: shared address), completing `bytes` on bar
__device__ __forceinline__ void bulk_copy_g2s(uint32_t dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// ---------------------------------------------------------------------------------------------
// fences
// ---------------------------------------------------------------------------------------------
// generic-proxy writes to shared memory -> visible to the async proxy (UMMA operand reads, bulk copies)
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ---------------------------------------------------------------------------------------------
// tensor memory
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {   // one full warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols));
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {     // same warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols));
}
// 32 lanes x 8 / 16 / 32 consecutive fp32 columns (lane = accumulator row)
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float (&v)[8]) {
  uint32_t r[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
      "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// ---------------------------------------------------------------------------------------------
// tcgen05.mma
// ---------------------------------------------------------------------------------------------
// Shared-memory matrix descriptor, version 1 (cute::UMMA::SmemDescriptor layout):
//   [0,14) start address >> 4 | [16,30) leading byte offset >> 4 | [32,46) stride byte offset >> 4 |
//   [46,48) version 1 | [61,64) layout: 0 = SWIZZLE_NONE, 1 = SWIZZLE_128B_BASE32B, 2 = SWIZZLE_128B,
//   4 = SWIZZLE_64B, 6 = SWIZZLE_32B.
// SWIZZLE_NONE, K-major: lbo = distance between the two 8-element k groups of one MMA, sbo = between 8-row groups.
__device__ __forceinline__ uint64_t smem_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo, uint32_t layout = 0) {
  return (uint64_t)((saddr & 0x3FFFF) >> 4) | ((uint64_t)(lbo >> 4) << 16) | ((uint64_t)(sbo >> 4) << 32) |
         (1ull << 46) | ((uint64_t)layout << 61);
}

// Operand format field of the instruction descriptor: kind::f16 takes F16 / BF16, kind::tf32 takes TF32.
enum class Fmt : uint32_t { F16 = 0, BF16 = 1, TF32 = 2 };
// Instruction descriptor, D = fp32, M = 128:
//   [4,6) D format (1 = f32) | [7,10) A format | [10,13) B format | 15 A MN-major | 16 B MN-major |
//   [17,23) N >> 3 | [24,29) M >> 4
__host__ __device__ constexpr uint32_t make_idesc(Fmt ab, int n, bool a_mn = false, bool b_mn = false) {
  return (1u << 4) | ((uint32_t)ab << 7) | ((uint32_t)ab << 10) | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16) |
         ((uint32_t)(n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}
// Values of the descriptors the kernels use (fp16: GNN / self-MLP, bf16: GEMM and convolutions, tf32: 3xTF32
// GEMM and convolutions), so a change of the bit packing fails the build.
static_assert(make_idesc(Fmt::F16, 32) == 0x08080010u, "fp16, K-major, N = 32");
static_assert(make_idesc(Fmt::F16, 64) == 0x08100010u, "fp16, K-major, N = 64");
static_assert(make_idesc(Fmt::F16, 96) == 0x08180010u, "fp16, K-major, N = 96");
static_assert(make_idesc(Fmt::F16, 128) == 0x08200010u, "fp16, K-major, N = 128");
static_assert(make_idesc(Fmt::F16, 256) == 0x08400010u, "fp16, K-major, N = 256");
static_assert(make_idesc(Fmt::BF16, 32) == 0x08080490u, "bf16, K-major, N = 32");
static_assert(make_idesc(Fmt::BF16, 64) == 0x08100490u, "bf16, K-major, N = 64");
static_assert(make_idesc(Fmt::BF16, 128) == 0x08200490u, "bf16, K-major, N = 128");
static_assert(make_idesc(Fmt::BF16, 256) == 0x08400490u, "bf16, K-major, N = 256");
static_assert(make_idesc(Fmt::BF16, 64, true, true) == 0x08118490u, "bf16, both MN-major, N = 64");
static_assert(make_idesc(Fmt::BF16, 128, true, true) == 0x08218490u, "bf16, both MN-major, N = 128");
static_assert(make_idesc(Fmt::TF32, 32) == 0x08080910u, "tf32, K-major, N = 32");
static_assert(make_idesc(Fmt::TF32, 128) == 0x08200910u, "tf32, K-major, N = 128");
static_assert(make_idesc(Fmt::TF32, 256) == 0x08400910u, "tf32, K-major, N = 256");
static_assert(make_idesc(Fmt::TF32, 64, false, true) == 0x08110910u, "tf32, B MN-major, N = 64");
static_assert(make_idesc(Fmt::TF32, 128, true, false) == 0x08208910u, "tf32, A MN-major, N = 128");
static_assert(make_idesc(Fmt::TF32, 128, true, true) == 0x08218910u, "tf32, both MN-major, N = 128");

// D[tmem] (+)= A[adesc] . B[bdesc]^T; acc == 0 overwrites D.  One thread issues.
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
}
// arrives on bar once every previously issued tcgen05.mma of this thread has completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

}  // namespace sm100
}  // namespace tmk
