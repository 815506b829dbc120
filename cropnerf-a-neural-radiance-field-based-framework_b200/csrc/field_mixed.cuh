// Shared pieces of the mixed-precision (tensor-core) FruitField kernels: shared-memory weight layout, mma.sync wrappers,
// fragment plumbing.  See field_mixed.cu for the design notes.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "field_common.cuh"

namespace cnbmix {


constexpr int WARPS = 8;
constexpr int THREADS = WARPS * 32;
constexpr int H = 64;      // hidden width of every MLP
constexpr int S32 = 40;    // row stride (halves) of a K=32 weight matrix
constexpr int S64 = 72;    // K=64
constexpr int S16 = 24;    // K=16

// shared-memory layout (half offsets, then float offsets)
constexpr int O_WB1 = 0;                    // [64][S32]
constexpr int O_WB2 = O_WB1 + 64 * S32;     // [16][S64]
constexpr int O_WS1 = O_WB2 + 16 * S64;     // [64][S16]   K' = [0 | geo15]
constexpr int O_WS2 = O_WS1 + 64 * S16;     // [64][S64]
constexpr int O_WR1 = O_WS2 + 64 * S64;     // [64][S64]   K' = [SH16 | 0,geo15 | emb32]
constexpr int O_WR2 = O_WR1 + 64 * S64;     // [64][S64]
constexpr int O_WR3 = O_WR2 + 64 * S64;     // [8][S64]    rows 3..7 zero
constexpr int HALVES = O_WR3 + 8 * S64;
constexpr int F_BB1 = 0, F_BB2 = 64, F_BS1 = 80, F_BS2 = 144, F_WH = 208, F_BH = 272, F_BR1 = 276, F_BR2 = 340, F_BR3 = 404;
constexpr int FLOATS = 412;
constexpr size_t SMEM_FWD = HALVES * sizeof(__half) + FLOATS * sizeof(float);

struct MixArgs {
  const float* table;
  int L;
  uint32_t mask, T;
  float scalings[CNB_MAX_LEVELS];
  cnb_warp warp;
  cnb_samples sm;
  const float *Wb1, *bb1, *Wb2, *bb2, *Ws1, *bs1, *Ws2, *bs2, *Wh, *bh, *Wr1, *br1, *Wr2, *br2, *Wr3, *br3;
  const float* embedding;       // per-camera rows, or the mean row, or null (zeros)
  int app_mode;
  int in0;                      // 2L
  float* density; float* rgb; float* sem; float* pos_out;
  float* geo_out;               // optional [N][16] fp32: base-MLP output [density before activation | geo15] (FruitField.get_density's embedding)
  __half* x0_out;               // optional [N][32] fp16 copy of the encoded features (kept for the backward)
  float* stash_out;             // optional [N][4] fp32 for the backward: d(density)/d(pre-activation) (trunc_exp' times the selector) | rgb after sigmoid
  uint2* mask_out;              // optional [N][4] ReLU masks of the four 64-wide hidden layers (relu_flags / field_mixed_bwd_tc5.cu)
};

__device__ __forceinline__ uint32_t pack_h2(float a, float b) {
  __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}

__device__ __forceinline__ void mma_f16(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];\n" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x2(uint32_t (&r)[2], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.shared.b16 {%0,%1}, [%2];\n" : "=r"(r[0]), "=r"(r[1]) : "r"(addr));
}

// acc[NT][4] (+)= A[KT][4] x W^T, W = smem fp16 [8*NT rows][STRIDE].
// B fragments come from ldmatrix: one x4 fetches (k 0-7, k 8-15) of TWO n-tiles -- the thread (g, t) of matrix q receives W[row g][2t, 2t+1],
// which is exactly the col-major B fragment -- instead of four 32-bit shared loads and their address arithmetic (the MLP kernels are
// issue / latency bound: 15 % of their instructions were those LDS).  Rows are 16-byte aligned (STRIDE % 8 == 0) and STRIDE = 8 (mod 16)
// halves spreads the eight 16-byte rows of a matrix over all 32 banks.
template <int NT, int KT, int STRIDE>
__device__ __forceinline__ void layer(const __half* __restrict__ W, const uint32_t (&A)[KT][4], float (&acc)[NT][4], int g, int t) {
  (void)g; (void)t;
  static_assert(STRIDE % 8 == 0, "ldmatrix rows must be 16-byte aligned");
  const int lane = threadIdx.x & 31;
  const uint32_t base = (uint32_t)__cvta_generic_to_shared(W);
  if constexpr (NT == 1) {
    const uint32_t a0 = base + 2u * ((lane & 7) * STRIDE + ((lane >> 3) & 1) * 8);
#pragma unroll
    for (int kt = 0; kt < KT; ++kt) {
      uint32_t b[2];
      ldsm_x2(b, a0 + 2u * kt * 16);
      mma_f16(acc[0], A[kt], b[0], b[1]);
    }
  } else {
    static_assert(NT % 2 == 0, "n-tiles are fetched in pairs");
    const uint32_t a0 = base + 2u * (((lane >> 4) * 8 + (lane & 7)) * STRIDE + ((lane >> 3) & 1) * 8);
#pragma unroll
    for (int np = 0; np < NT / 2; ++np) {
#pragma unroll
      for (int kt = 0; kt < KT; ++kt) {
        uint32_t b[4];
        ldsm_x4(b, a0 + 2u * (np * 16 * STRIDE + kt * 16));
        mma_f16(acc[2 * np], A[kt], b[0], b[1]);
        mma_f16(acc[2 * np + 1], A[kt], b[2], b[3]);
      }
    }
  }
}

template <int NT>
__device__ __forceinline__ void init_bias(float (&acc)[NT][4], const float* __restrict__ b, int t) {
#pragma unroll
  for (int nt = 0; nt < NT; ++nt) {
    const float2 v = *reinterpret_cast<const float2*>(b + nt * 8 + 2 * t);
    acc[nt][0] = v.x; acc[nt][1] = v.y; acc[nt][2] = v.x; acc[nt][3] = v.y;
  }
}

// ReLU + pack the C fragments of 2*KT n-tiles into KT A-fragment k-tiles
template <int KT, bool RELU>
__device__ __forceinline__ void to_afrag(const float (&acc)[2 * KT][4], uint32_t (&A)[KT][4]) {
#pragma unroll
  for (int kt = 0; kt < KT; ++kt) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      float v0 = acc[2 * kt + h][0], v1 = acc[2 * kt + h][1], v2 = acc[2 * kt + h][2], v3 = acc[2 * kt + h][3];
      if (RELU) { v0 = fmaxf(v0, 0.f); v1 = fmaxf(v1, 0.f); v2 = fmaxf(v2, 0.f); v3 = fmaxf(v3, 0.f); }
      A[kt][2 * h] = pack_h2(v0, v1);      // row g
      A[kt][2 * h + 1] = pack_h2(v2, v3);  // row g+8
    }
  }
}

// ReLU flags of this thread's 16 values of each of its two fragment rows (A = the packed, already rectified fp16 activations of a 64-wide
// layer): bit nt <-> column 8 nt + 2 t, bit 16 + nt <-> column 8 nt + 2 t + 1.  A rectified half is +0 or positive, so "non-zero" is bit 15 of
// half + 0x7fff; three instructions per word.
__device__ __forceinline__ void relu_flags(const uint32_t (&A)[4][4], uint32_t& row_lo, uint32_t& row_hi) {
  uint32_t a0 = 0u, a1 = 0u;
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {   // n-tile nt = words A[nt/2][2 (nt%2)] (row g) and A[nt/2][2 (nt%2) + 1] (row g + 8)
    a0 = (a0 >> 1) | ((A[nt >> 1][2 * (nt & 1)] + 0x7FFF7FFFu) & 0x80008000u);
    a1 = (a1 >> 1) | ((A[nt >> 1][2 * (nt & 1) + 1] + 0x7FFF7FFFu) & 0x80008000u);
  }
  row_lo = (a0 >> 8) & 0x00FF00FFu;
  row_hi = (a1 >> 8) & 0x00FF00FFu;
}

__device__ __forceinline__ float pick4(int t, float a, float b, float c, float d) { return t == 0 ? a : (t == 1 ? b : (t == 2 ? c : d)); }

__device__ inline void load_weights(const MixArgs& a, __half* Wh_, float* Bf) {
  const int tid = threadIdx.x;
  for (int e = tid; e < 64 * S32; e += THREADS) { const int n = e / S32, k = e - n * S32; Wh_[O_WB1 + e] = __float2half_rn(k < a.in0 ? __ldg(a.Wb1 + n * a.in0 + k) : 0.f); }
  for (int e = tid; e < 16 * S64; e += THREADS) { const int n = e / S64, k = e - n * S64; Wh_[O_WB2 + e] = __float2half_rn(k < 64 ? __ldg(a.Wb2 + n * 64 + k) : 0.f); }
  for (int e = tid; e < 64 * S16; e += THREADS) { const int n = e / S16, k = e - n * S16; Wh_[O_WS1 + e] = __float2half_rn((k >= 1 && k < 16) ? __ldg(a.Ws1 + n * 15 + (k - 1)) : 0.f); }
  for (int e = tid; e < 64 * S64; e += THREADS) {
    const int n = e / S64, k = e - n * S64;
    Wh_[O_WS2 + e] = __float2half_rn(k < 64 ? __ldg(a.Ws2 + n * 64 + k) : 0.f);
    float w1 = 0.f;
    if (k < 16) w1 = __ldg(a.Wr1 + n * 63 + k);
    else if (k >= 17 && k < 64) w1 = __ldg(a.Wr1 + n * 63 + (k - 1));
    Wh_[O_WR1 + e] = __float2half_rn(w1);
    Wh_[O_WR2 + e] = __float2half_rn(k < 64 ? __ldg(a.Wr2 + n * 64 + k) : 0.f);
  }
  for (int e = tid; e < 8 * S64; e += THREADS) { const int n = e / S64, k = e - n * S64; Wh_[O_WR3 + e] = __float2half_rn((n < 3 && k < 64) ? __ldg(a.Wr3 + n * 64 + k) : 0.f); }
  for (int e = tid; e < 64; e += THREADS) {
    Bf[F_BB1 + e] = __ldg(a.bb1 + e); Bf[F_BS1 + e] = __ldg(a.bs1 + e); Bf[F_BS2 + e] = __ldg(a.bs2 + e); Bf[F_WH + e] = __ldg(a.Wh + e);
    Bf[F_BR1 + e] = __ldg(a.br1 + e); Bf[F_BR2 + e] = __ldg(a.br2 + e);
  }
  if (tid < 16) Bf[F_BB2 + tid] = __ldg(a.bb2 + tid);
  if (tid < 8) Bf[F_BR3 + tid] = tid < 3 ? __ldg(a.br3 + tid) : 0.f;
  if (tid < 4) Bf[F_BH + tid] = tid == 0 ? __ldg(a.bh) : 0.f;
}

// ctx (mixed, training): [x0: N*32 fp16][positions: N*3 floats][d_x0: 16 levels x N x 2 floats, level-major][stash: N*4 floats]
// [relu masks: N*8 words][partial weight gradients], every block 16-byte aligned
inline int64_t ctx_pos_off(int64_t n) { return n * 16; }
inline int64_t ctx_dx0_off(int64_t n) { return (n * 19 + 3) & ~(int64_t)3; }
inline int64_t ctx_stash_off(int64_t n) { return ctx_dx0_off(n) + n * 32; }
inline int64_t ctx_mask_off(int64_t n) { return ctx_stash_off(n) + n * 4; }
// [per-CTA partial weight gradients of field_mixed_bwd_tc5.cu: CTX_PART_CTAS images of CTX_PART_FLOATS]
constexpr int64_t CTX_PART_FLOATS = 16896, CTX_PART_CTAS = 160;
inline int64_t ctx_part_off(int64_t n) { return ctx_mask_off(n) + n * 8; }
inline int64_t ctx_total(int64_t n) { return ctx_part_off(n) + CTX_PART_FLOATS * CTX_PART_CTAS + 16; }

inline int fill_args(const cnb_field* f, const cnb_samples* s, MixArgs& a) {
  a.table = f->grid.table;
  a.L = f->grid.num_levels;
  a.T = 1u << f->grid.log2_hashmap_size;
  a.mask = a.T - 1u;
  for (int i = 0; i < CNB_MAX_LEVELS; ++i) a.scalings[i] = f->grid.scalings[i];
  a.warp = f->warp;
  a.sm = *s;
  a.Wb1 = f->base.W[0]; a.bb1 = f->base.b[0]; a.Wb2 = f->base.W[1]; a.bb2 = f->base.b[1];
  a.Ws1 = f->sem.W[0]; a.bs1 = f->sem.b[0]; a.Ws2 = f->sem.W[1]; a.bs2 = f->sem.b[1];
  a.Wh = f->sem_head.W[0]; a.bh = f->sem_head.b[0];
  a.Wr1 = f->rgb.W[0]; a.br1 = f->rgb.b[0]; a.Wr2 = f->rgb.W[1]; a.br2 = f->rgb.b[1]; a.Wr3 = f->rgb.W[2]; a.br3 = f->rgb.b[2];
  a.app_mode = f->appearance_mode;
  a.embedding = f->appearance_mode == CNB_APP_PER_CAMERA ? f->embedding : (f->appearance_mode == CNB_APP_MEAN ? f->mean_embedding : nullptr);
  a.in0 = f->base.dims[0];
  a.geo_out = nullptr;
  a.stash_out = nullptr;
  a.mask_out = nullptr;
  return CNB_OK;
}


}  // namespace cnbmix
