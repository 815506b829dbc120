// tcgen05 (UMMA) plumbing shared by the tensor-core kernels that keep their accumulators in tensor memory: field_mixed_bwd_tc5.cu (the fused
// base-architecture backward) and mlp_mixed.cu (the layer-by-layer operator for MLPs wider than 64).
//
// Shared-memory operands use the no-swizzle canonical layouts proven in tests/micro/umma_chain_test.cu / umma_dw_test.cu:
//   a [rows][features] 16-bit matrix, rows = samples:  byte(s, f) = (f/8)*2048 + s*16 + (f%8)*2   (128 rows; a thread owning row s writes
//                                                       one conflict-free 16-byte chunk per 8-feature block)
//       K-major (K = features, e.g. the A of a layer)  : LBO 2048, SBO 128
//       MN-major (K = samples, an operand of dY^T X)   : LBO 128,  SBO 2048
//   a weight [out][in] 16-bit, OUT rows (padded to 16): byte(o, i) = (i/8)*(OUT*16) + o*16 + (i%8)*2
//       Y = X W^T (B K-major, K = in)                  : LBO OUT*16, SBO 128
//       dX = dY W (B MN-major, K = out)                : LBO 128,    SBO OUT*16
// i.e. LBO is always the stride between 8-element core matrices along K, SBO the stride along M / N.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>

namespace cnbumma {

// instruction descriptor of kind::f16 with an fp32 accumulator; major: 0 = K, 1 = MN.  A and B must have the same format (a bf16 A with an
// fp16 B is an illegal instruction: umma_chain_test).
__device__ __forceinline__ constexpr uint32_t idesc(int M, int N, int amajor, int bmajor) {   // bf16 x bf16
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)amajor << 15) | ((uint32_t)bmajor << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ constexpr uint32_t idesc_f16(int M, int N, int amajor, int bmajor) {   // fp16 x fp16
  return (1u << 4) | ((uint32_t)amajor << 15) | ((uint32_t)bmajor << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t id, uint32_t accumulate) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d), "l"(da),
               "l"(db), "r"(id), "r"(accumulate)
               : "memory");
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.b32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  while (!done)
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}" : "=r"(done) : "r"(bar), "r"(parity) : "memory");
}
// Shared-memory descriptor split in two words: a K step only adds to the 14-bit start-address field of the low word (shared addresses
// < 256 KB never carry out of it).
__device__ __forceinline__ uint32_t desc_lo(uint32_t addr, uint32_t lbo) { return ((addr >> 4) & 0x3FFFu) | ((lbo >> 4) << 16); }
__device__ __forceinline__ constexpr uint32_t desc_hi(uint32_t sbo) { return (sbo >> 4) | (1u << 14); }
__device__ __forceinline__ uint64_t desc64(uint32_t lo, uint32_t hi) { return ((uint64_t)hi << 32) | lo; }

// NC accumulator columns of this thread's TMEM lane (taddr carries the warp's lane quarter in bits 16+)
template <int NC>
__device__ __forceinline__ void tm_load(uint32_t taddr, float (&v)[NC]) {
  static_assert(NC % 16 == 0, "16-column chunks");
  uint32_t r[NC];
#pragma unroll
  for (int c = 0; c < NC; c += 16)
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(r[c]), "=r"(r[c + 1]), "=r"(r[c + 2]), "=r"(r[c + 3]), "=r"(r[c + 4]), "=r"(r[c + 5]), "=r"(r[c + 6]), "=r"(r[c + 7]), "=r"(r[c + 8]),
                   "=r"(r[c + 9]), "=r"(r[c + 10]), "=r"(r[c + 11]), "=r"(r[c + 12]), "=r"(r[c + 13]), "=r"(r[c + 14]), "=r"(r[c + 15])
                 : "r"(taddr + c));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int c = 0; c < NC; ++c) v[c] = __uint_as_float(r[c]);
}

__device__ __forceinline__ uint32_t pack_bf2(float a, float b) {
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}

}  // namespace cnbumma
