// Mixed-precision nn.Linear stack on tcgen05 for MLPs with layers wider than CNB_MAX_WIDTH (nerfstudio MLP, fruit_field.py:133-167 at the
// widths of the reference's fruit_nerf_big / fruit_nerf_huge presets: 32->64->31, 30->128->128->64, 78->64->64->3).  The tensor-core
// counterpart of mlp_wide.cu; the base preset keeps its fused kernels (field_mixed*.cu).
//
//   forward  : Y_l = act(X_l W_l^T + b_l)               fp16 operands, fp32 accumulator in TMEM, bias / activation in fp32       k_mx_fwd
//              hidden activations are kept in fp16 (row stride up8(width)) in the caller's scratch; the last layer is written in fp32, so
//              that sigmoid' sees the value the loss saw
//   backward : dZ_L = dY * act'(Y)                       computed while staging (never stored)
//              dW_l = dZ_l^T X_l , db_l = colsum(dZ_l)   bf16 operands; one fp32 accumulator per CTA in TMEM across all its tiles, the bias
//                                                        as one more column of X (= 1); per-CTA images, then one reduction   k_mx_dw, k_mx_reduce
//              dZ_{l-1} = (dZ_l W_l) * [X_l > 0]         bf16; the mask is the STORED forward activation (a bf16 recompute flips
//                                                        units: DESIGN section 4)                                              k_mx_dx
// Every GEMM is tcgen05.mma kind::f16 on 128-sample tiles (M = 128), operands in the canonical no-swizzle layouts of umma.cuh; K and N are
// padded to 16 inside the kernel (odd widths such as 3, 30, 31, 78 are zero-padded in shared memory).  kind::f16 needs A and B in one
// format, so the forward is fp16 x fp16 (the arithmetic of the fused mixed forward) and the backward bf16 x bf16 (gradients need bf16's
// range); the fp16 activations are converted to bf16 when they are staged for dW.
//
// One layer per launch, one 128-thread CTA per tile stream: thread r owns sample row r of the tile (staging, epilogue), thread 0 issues the
// MMAs.  Chaining all layers of an MLP in one CTA would save the activations' round trip through L2 / HBM, but the widths here differ per
// MLP and per layer (up to 128 x 144 accumulator columns, 32 KB weight images), and a per-layer kernel keeps shared memory and tensor
// memory small enough for three or four CTAs per SM, whose staging and epilogues then overlap each other's MMAs.
//
// Scratch (caller's, nothing allocated here): [hidden fp16 | dZ bf16 [n][up8(max width)] | DW_PARTS partial dW images].  The dZ buffer is
// updated in place: a CTA reads all rows of its tile into shared memory before it writes the tile's next dZ rows.
#include <cstdio>

#include "field_common.cuh"
#include "umma.cuh"

using namespace cnbumma;

namespace {

constexpr int ROWS = 128;                 // samples per tile = UMMA M = threads per CTA
constexpr int MX_MAX = 128;               // widest layer of this path
constexpr uint32_t FB = 2048;             // bytes of one 8-feature block of a [128][*] operand
constexpr int DW_PARTS = 296;             // partial dW images (two CTAs per SM on a 148-SM B200); a fixed count keeps the scratch size device-free
constexpr int CTAS_PER_SM = 4;

__host__ __device__ inline int up16(int v) { return (v + 15) & ~15; }
__host__ __device__ inline int up8(int v) { return (v + 7) & ~7; }
inline int64_t up4l(int64_t v) { return (v + 3) & ~(int64_t)3; }
__host__ __device__ inline uint32_t tmem_cols(int n) { uint32_t c = 32; while ((int)c < n) c <<= 1; return c; }

__device__ __forceinline__ float act_fwd(float v, int act) {
  if (act == CNB_ACT_RELU) return fmaxf(v, 0.0f);
  if (act == CNB_ACT_SIGMOID) return 1.0f / (1.0f + expf(-v));
  return v;
}
__device__ __forceinline__ float act_grad(float dy, float y, int act) {
  if (act == CNB_ACT_SIGMOID) return dy * y * (1.0f - y);
  if (act == CNB_ACT_RELU) return y > 0.0f ? dy : 0.0f;
  return dy;
}
__device__ __forceinline__ uint32_t pack_h2f(float a, float b) {
  __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}

// ---- per-CTA set-up / synchronisation -------------------------------------------------------------------------------------------------------
struct Sync {
  uint32_t tmem, bar, phase;
};
__device__ __forceinline__ void cta_setup(uint64_t* bar, uint32_t* slot, uint32_t cols, Sync& s) {
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"((uint32_t)__cvta_generic_to_shared(bar)));
    asm volatile("fence.mbarrier_init.release.cluster;");
  }
  if (threadIdx.x < 32) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(slot)), "r"(cols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("tcgen05.fence::before_thread_sync;");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;");
  s.tmem = *slot;
  s.bar = (uint32_t)__cvta_generic_to_shared(bar);
  s.phase = 0;
}
__device__ __forceinline__ void cta_teardown(const Sync& s, uint32_t cols) {
  asm volatile("tcgen05.fence::before_thread_sync;");
  __syncthreads();
  if (threadIdx.x < 32) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(s.tmem), "r"(cols));
}
// operands staged by every thread -> visible to the tensor core
__device__ __forceinline__ void operands_ready() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("tcgen05.fence::before_thread_sync;");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;");
}
// thread 0: the MMAs issued since the last commit -> mbarrier; every thread waits for them
__device__ __forceinline__ void commit_wait(Sync& s) {
  if (threadIdx.x == 0) asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.b64 [%0];" ::"l"((uint64_t)s.bar) : "memory");
  mbar_wait(s.bar, s.phase);
  s.phase ^= 1u;
  asm volatile("tcgen05.fence::after_thread_sync;");
}

// weight [OUT][IN] fp32 -> 16-bit image of OP x IP (zero padded), byte(o, i) = (i/8)*(OP*16) + o*16 + (i%8)*2
template <bool BF16>
__device__ __forceinline__ void stage_weight(const float* __restrict__ W, int OUT, int IN, int OP, int IP, unsigned char* dst) {
  const int pairs = OP * IP / 2;
  for (int p = threadIdx.x; p < pairs; p += ROWS) {
    const int o = p / (IP / 2), i = 2 * (p - o * (IP / 2));
    const float a = (o < OUT && i < IN) ? __ldg(W + (int64_t)o * IN + i) : 0.0f;
    const float b = (o < OUT && i + 1 < IN) ? __ldg(W + (int64_t)o * IN + i + 1) : 0.0f;
    *reinterpret_cast<uint32_t*>(dst + (i >> 3) * (OP * 16) + o * 16 + (i & 7) * 2) = BF16 ? pack_bf2(a, b) : pack_h2f(a, b);
  }
}

// 8 features [k0, k0 + 8) of one row as floats: fp32 rows (any stride) or fp16 rows (16-byte aligned, zero padded to up8(K))
__device__ __forceinline__ void load8_f32(const float* row, int k0, int K, float (&f)[8]) {
#pragma unroll
  for (int e = 0; e < 8; ++e) f[e] = (k0 + e < K) ? __ldg(row + k0 + e) : 0.0f;
}
__device__ __forceinline__ void load8_h16(const __half* row, int k0, int K, float (&f)[8]) {
  if (k0 < K) {
    const uint4 q = __ldg(reinterpret_cast<const uint4*>(row + k0));
    const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 v = __half22float2(*reinterpret_cast<const __half2*>(&w[e]));
      f[2 * e] = v.x; f[2 * e + 1] = v.y;
    }
  } else {
#pragma unroll
    for (int e = 0; e < 8; ++e) f[e] = 0.0f;
  }
}

// dZ rows: either dY * act'(Y) of the last layer (fp32, dense [n][K]) or the bf16 buffer of the layer above (row stride ldz, zero padded)
struct DzSrc {
  const float* dy;
  const float* y;
  int act;
  const __nv_bfloat16* dz;   // may alias the output of k_mx_dx: plain loads
  int64_t ldz;
};
__device__ __forceinline__ void load8_dz(const DzSrc& s, int64_t row, int k0, int K, float (&f)[8]) {
  if (s.dz == nullptr) {
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int k = k0 + e;
      f[e] = 0.0f;
      if (k < K) f[e] = act_grad(__ldg(s.dy + row * K + k), s.act == CNB_ACT_NONE ? 0.0f : __ldg(s.y + row * K + k), s.act);
    }
  } else if (k0 < K) {
    const uint4 q = *reinterpret_cast<const uint4*>(s.dz + row * s.ldz + k0);
    const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 v = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[e]));
      f[2 * e] = v.x; f[2 * e + 1] = v.y;
    }
  } else {
#pragma unroll
    for (int e = 0; e < 8; ++e) f[e] = 0.0f;
  }
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8], bool bf16) {
  if (bf16) return make_uint4(pack_bf2(f[0], f[1]), pack_bf2(f[2], f[3]), pack_bf2(f[4], f[5]), pack_bf2(f[6], f[7]));
  return make_uint4(pack_h2f(f[0], f[1]), pack_h2f(f[2], f[3]), pack_h2f(f[4], f[5]), pack_h2f(f[6], f[7]));
}

// ---- forward: Y = act(X W^T + b) ----------------------------------------------------------------------------------------------------------
// X: fp32 rows (x32, ldx floats) or fp16 hidden rows (x16, ldx halves).  Y: fp32 dense [n][N] (y32) or fp16 hidden rows (y16, ldy halves).
__global__ void __launch_bounds__(ROWS) k_mx_fwd(const float* __restrict__ x32, const __half* __restrict__ x16, int64_t ldx, int64_t n, int K, int N,
                                                 const float* __restrict__ W, const float* __restrict__ bias, int act, float* __restrict__ y32,
                                                 __half* __restrict__ y16, int64_t ldy) {
  extern __shared__ __align__(1024) unsigned char smem[];
  __shared__ __align__(8) uint64_t bar;
  __shared__ uint32_t slot;
  __shared__ float sb[MX_MAX];
  const int KP = up16(K), NP = up16(N);
  unsigned char* sA = smem;                         // [128][KP] fp16
  unsigned char* sW = smem + ROWS * KP * 2;         // [NP][KP] fp16
  stage_weight<false>(W, N, K, NP, KP, sW);
  for (int c = threadIdx.x; c < MX_MAX; c += ROWS) sb[c] = c < N ? __ldg(bias + c) : 0.0f;
  Sync s;
  const uint32_t cols = tmem_cols(NP);
  cta_setup(&bar, &slot, cols, s);
  const int r = threadIdx.x, warp = r >> 5;
  const uint32_t trow = s.tmem + ((uint32_t)(32 * warp) << 16);
  const uint32_t a_s = (uint32_t)__cvta_generic_to_shared(sA), w_s = (uint32_t)__cvta_generic_to_shared(sW);
  const uint32_t id = idesc_f16(ROWS, NP, 0, 0);
  const int64_t tiles = (n + ROWS - 1) / ROWS;
  for (int64_t t = blockIdx.x; t < tiles; t += gridDim.x) {
    const int64_t row = t * ROWS + r;
    const bool valid = row < n;
    for (int k0 = 0; k0 < KP; k0 += 8) {
      float f[8];
      if (!valid) { for (int e = 0; e < 8; ++e) f[e] = 0.0f; }
      else if (x32) load8_f32(x32 + row * ldx, k0, K, f);
      else load8_h16(x16 + row * ldx, k0, K, f);
      *reinterpret_cast<uint4*>(sA + (k0 >> 3) * FB + r * 16) = pack8(f, false);
    }
    operands_ready();
    if (threadIdx.x == 0)
      for (int ks = 0; ks < KP / 16; ++ks)
        umma(s.tmem, desc64(desc_lo(a_s + ks * 2 * FB, FB), desc_hi(128)), desc64(desc_lo(w_s + ks * 2 * NP * 16, NP * 16), desc_hi(128)), id, ks > 0 ? 1u : 0u);
    commit_wait(s);
    for (int c0 = 0; c0 < NP; c0 += 16) {
      float v[16];
      tm_load<16>(trow + c0, v);
#pragma unroll
      for (int j = 0; j < 16; ++j) v[j] = c0 + j < N ? act_fwd(v[j] + sb[c0 + j], act) : 0.0f;
      if (!valid) continue;
      if (y32) {
#pragma unroll
        for (int j = 0; j < 16; ++j) if (c0 + j < N) y32[row * N + c0 + j] = v[j];
      } else {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          if (c0 + 8 * h >= N) break;
          float f[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) f[e] = v[8 * h + e];
          *reinterpret_cast<uint4*>(y16 + row * ldy + c0 + 8 * h) = pack8(f, false);
        }
      }
    }
    asm volatile("tcgen05.fence::before_thread_sync;");
    __syncthreads();   // accumulator read and A consumed before the next tile overwrites them
    asm volatile("tcgen05.fence::after_thread_sync;");
  }
  cta_teardown(s, cols);
}

// ---- input gradient: dZ_prev = (dZ W) * [X > 0] (bf16 rows, ldo halves) or dX = dZ W (fp32, ldo floats) ------------------------------------
// OUT = K of this GEMM (the layer's outputs), IN = N (its inputs); mask = the layer's input as kept by the forward (fp16, ldm halves) or null
__global__ void __launch_bounds__(ROWS) k_mx_dx(DzSrc src, int64_t n, int OUT, int IN, const float* __restrict__ W, const __half* __restrict__ mask,
                                                int64_t ldm, __nv_bfloat16* dz_out, float* __restrict__ dx, int64_t ldo) {
  extern __shared__ __align__(1024) unsigned char smem[];
  __shared__ __align__(8) uint64_t bar;
  __shared__ uint32_t slot;
  const int KP = up16(OUT), NP = up16(IN);
  unsigned char* sA = smem;                         // dZ [128][KP] bf16
  unsigned char* sW = smem + ROWS * KP * 2;         // W [KP rows = out][NP] bf16
  stage_weight<true>(W, OUT, IN, KP, NP, sW);
  Sync s;
  const uint32_t cols = tmem_cols(NP);
  cta_setup(&bar, &slot, cols, s);
  const int r = threadIdx.x, warp = r >> 5;
  const uint32_t trow = s.tmem + ((uint32_t)(32 * warp) << 16);
  const uint32_t a_s = (uint32_t)__cvta_generic_to_shared(sA), w_s = (uint32_t)__cvta_generic_to_shared(sW);
  const uint32_t id = idesc(ROWS, NP, 0, 1);
  const int64_t tiles = (n + ROWS - 1) / ROWS;
  for (int64_t t = blockIdx.x; t < tiles; t += gridDim.x) {
    const int64_t row = t * ROWS + r;
    const bool valid = row < n;
    for (int k0 = 0; k0 < KP; k0 += 8) {
      float f[8];
      if (!valid) { for (int e = 0; e < 8; ++e) f[e] = 0.0f; }
      else load8_dz(src, row, k0, OUT, f);
      *reinterpret_cast<uint4*>(sA + (k0 >> 3) * FB + r * 16) = pack8(f, true);
    }
    operands_ready();   // (the in-place dZ rows of this tile are all read: the writes below cannot race them)
    if (threadIdx.x == 0)
      for (int ks = 0; ks < KP / 16; ++ks)
        umma(s.tmem, desc64(desc_lo(a_s + ks * 2 * FB, FB), desc_hi(128)), desc64(desc_lo(w_s + ks * 256, 128), desc_hi(KP * 16)), id, ks > 0 ? 1u : 0u);
    commit_wait(s);
    for (int c0 = 0; c0 < NP; c0 += 16) {
      float v[16];
      tm_load<16>(trow + c0, v);
      if (!valid) continue;
      if (dx) {
#pragma unroll
        for (int j = 0; j < 16; ++j) if (c0 + j < IN) dx[row * ldo + c0 + j] = v[j];
      } else {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int k0 = c0 + 8 * h;
          if (k0 >= IN) break;
          float m[8];
          load8_h16(mask + row * ldm, k0, IN, m);
          float f[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) f[e] = (k0 + e < IN && m[e] > 0.0f) ? v[8 * h + e] : 0.0f;
          *reinterpret_cast<uint4*>(dz_out + row * ldo + k0) = pack8(f, true);
        }
      }
    }
    asm volatile("tcgen05.fence::before_thread_sync;");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;");
  }
  cta_teardown(s, cols);
}

// ---- weight gradient: this CTA's image of [dW | db] = dZ^T [X | 1] over its tiles ----------------------------------------------------------
// M = 128 (dZ's OUT features, zero padded), N = up16(IN + 1): column IN of the staged X is 1, so accumulator column IN is colsum(dZ) = db.
// part: this CTA's image [OUT][IN] then [OUT]
__global__ void __launch_bounds__(ROWS) k_mx_dw(DzSrc src, const float* __restrict__ x32, const __half* __restrict__ x16, int64_t ldx, int64_t n,
                                                int OUT, int IN, float* __restrict__ part, int64_t img) {
  extern __shared__ __align__(1024) unsigned char smem[];
  __shared__ __align__(8) uint64_t bar;
  __shared__ uint32_t slot;
  const int ND = up16(IN + 1), OB = up8(OUT) / 8;
  unsigned char* sA = smem;                         // dZ [128 samples][128 features] bf16
  unsigned char* sX = smem + ROWS * MX_MAX * 2;     // X  [128 samples][ND] bf16
  for (int e = threadIdx.x; e < (int)(ROWS * MX_MAX * 2 / 16); e += ROWS) reinterpret_cast<uint4*>(sA)[e] = make_uint4(0u, 0u, 0u, 0u);
  Sync s;
  const uint32_t cols = tmem_cols(ND);
  cta_setup(&bar, &slot, cols, s);
  const int r = threadIdx.x, warp = r >> 5;
  const uint32_t trow = s.tmem + ((uint32_t)(32 * warp) << 16);
  const uint32_t a_s = (uint32_t)__cvta_generic_to_shared(sA), x_s = (uint32_t)__cvta_generic_to_shared(sX);
  const uint32_t id = idesc(ROWS, ND, 1, 1);
  const int64_t tiles = (n + ROWS - 1) / ROWS;
  bool first = true;
  for (int64_t t = blockIdx.x; t < tiles; t += gridDim.x) {
    const int64_t row = t * ROWS + r;
    const bool valid = row < n;
    for (int b = 0; b < OB; ++b) {
      float f[8];
      if (!valid) { for (int e = 0; e < 8; ++e) f[e] = 0.0f; }
      else load8_dz(src, row, 8 * b, OUT, f);
      *reinterpret_cast<uint4*>(sA + b * FB + r * 16) = pack8(f, true);
    }
    for (int k0 = 0; k0 < ND; k0 += 8) {
      float f[8];
      if (!valid) { for (int e = 0; e < 8; ++e) f[e] = 0.0f; }
      else {
        if (x32) load8_f32(x32 + row * ldx, k0, IN, f);
        else load8_h16(x16 + row * ldx, k0, IN, f);
#pragma unroll
        for (int e = 0; e < 8; ++e) if (k0 + e == IN) f[e] = 1.0f;
      }
      *reinterpret_cast<uint4*>(sX + (k0 >> 3) * FB + r * 16) = pack8(f, true);
    }
    operands_ready();
    if (threadIdx.x == 0)
      for (int ks = 0; ks < ROWS / 16; ++ks)
        umma(s.tmem, desc64(desc_lo(a_s + ks * 256, 128), desc_hi(FB)), desc64(desc_lo(x_s + ks * 256, 128), desc_hi(FB)), id, (ks > 0 || !first) ? 1u : 0u);
    commit_wait(s);   // operands consumed: the next tile may be staged
    first = false;
  }
  // accumulator row r = output r (TMEM loads are warp-collective: every lane loads, the lanes r >= OUT drop)
  float* out = part + (int64_t)blockIdx.x * img;
  for (int c0 = 0; c0 < ND; c0 += 16) {
    float v[16];
    tm_load<16>(trow + c0, v);
    if (r >= OUT) continue;
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const int c = c0 + j;
      if (c < IN) out[(int64_t)r * IN + c] = v[j];
      else if (c == IN) out[(int64_t)OUT * IN + r] = v[j];
    }
  }
  cta_teardown(s, cols);
}

// dW += sum of the images, db += ...  (one thread per element: deterministic, no atomics)
__global__ void __launch_bounds__(256) k_mx_reduce(const float* __restrict__ part, int nparts, int64_t img, int OUT, int IN, float* __restrict__ dW,
                                                   float* __restrict__ db) {
  const int64_t e = blockIdx.x * 256LL + threadIdx.x;
  const int64_t nw = (int64_t)OUT * IN;
  if (e >= nw + OUT) return;
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  int p = 0;
  for (; p + 4 <= nparts; p += 4) {
    s0 += __ldg(part + (int64_t)p * img + e); s1 += __ldg(part + (int64_t)(p + 1) * img + e);
    s2 += __ldg(part + (int64_t)(p + 2) * img + e); s3 += __ldg(part + (int64_t)(p + 3) * img + e);
  }
  for (; p < nparts; ++p) s0 += __ldg(part + (int64_t)p * img + e);
  const float sum = (s0 + s1) + (s2 + s3);
  if (e < nw) { if (dW) dW[e] += sum; }
  else if (db) db[e - nw] += sum;
}

// ---- host side -------------------------------------------------------------------------------------------------------------------------
int hidden_w(const cnb_mlp* m) { int w = 0; for (int l = 1; l < m->num_layers; ++l) w = max(w, up8(m->dims[l])); return w; }
int dz_w(const cnb_mlp* m) { int w = 0; for (int l = 1; l <= m->num_layers; ++l) w = max(w, up8(m->dims[l])); return w; }
int64_t img_floats(const cnb_mlp* m) {
  int64_t w = 0;
  for (int l = 0; l < m->num_layers; ++l) w = max(w, up4l((int64_t)m->dims[l + 1] * (m->dims[l] + 1)));
  return w;
}
// half offset of hidden layer l's rows: layer-major when training (kept for the backward), two ping-pong buffers for inference
int64_t hidden_off(const cnb_mlp* m, int64_t n, int l, bool training) {
  if (!training) return (l & 1) * n * hidden_w(m);
  int64_t off = 0;
  for (int q = 0; q < l; ++q) off += n * up8(m->dims[q + 1]);
  return off;
}
int64_t hidden_floats(const cnb_mlp* m, int64_t n, bool training) {
  if (m->num_layers < 2) return 0;
  const int64_t halves = training ? hidden_off(m, n, m->num_layers - 1, true) : 2 * n * hidden_w(m);
  return up4l((halves + 1) / 2);
}
int64_t work_floats(const cnb_mlp* m, int64_t n) { return up4l((n * dz_w(m) + 1) / 2) + DW_PARTS * img_floats(m); }

// Dynamic shared memory, with a floor that caps the CTAs per SM at what tensor memory holds (512 columns: four forward / dX CTAs of <= 128
// columns, two dW CTAs of 256), so that no CTA ever waits in tcgen05.alloc for another to finish.
constexpr size_t FLOOR_4 = 48 * 1024, FLOOR_2 = 80 * 1024;
size_t fwd_smem(int K, int N) { return max((size_t)ROWS * up16(K) * 2 + (size_t)up16(N) * up16(K) * 2, FLOOR_4); }
size_t dx_smem(int OUT, int IN) { return max((size_t)ROWS * up16(OUT) * 2 + (size_t)up16(OUT) * up16(IN) * 2, FLOOR_4); }
size_t dw_smem(int IN) { return max((size_t)ROWS * MX_MAX * 2 + (size_t)ROWS * up16(IN + 1) * 2, FLOOR_2); }
constexpr size_t SMEM_MAX = 96 * 1024;   // >= every size above (largest: 64 KB forward / dX, 68 KB dW)

int set_smem_attrs() {
  static bool done = false;
  if (done) return CNB_OK;
  if (cudaFuncSetAttribute(k_mx_fwd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_MAX) != cudaSuccess ||
      cudaFuncSetAttribute(k_mx_dx, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_MAX) != cudaSuccess ||
      cudaFuncSetAttribute(k_mx_dw, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_MAX) != cudaSuccess)
    return cnb_check_launch("mlp_mixed smem attributes");
  done = true;
  return CNB_OK;
}
int grid_for(int64_t n, int cap) {
  const int64_t tiles = (n + ROWS - 1) / ROWS;
  return (int)(tiles < cap ? tiles : cap);
}

int check_mlp(const cnb_mlp* m, const char* what) {
  CNB_REQUIRE(m != nullptr, "%s: null mlp", what);
  if (!cnb_mlp_mixed_supported(m)) {
    char shape[160];
    int o = 0;
    for (int l = 0; l <= m->num_layers && l <= CNB_MAX_LAYERS && o < 140; ++l) o += snprintf(shape + o, sizeof(shape) - o, l ? "->%d" : "%d", m->dims[l]);
    if (o == 0) snprintf(shape, sizeof(shape), "(%d layers)", m->num_layers);
    cnb_set_error("%s: MLP %s is outside the tensor-core operator (1..%d layers, every width 1..%d)", what, shape, CNB_MAX_LAYERS, MX_MAX);
    return CNB_ERR_UNSUPPORTED;
  }
  for (int l = 0; l < m->num_layers; ++l) CNB_REQUIRE(m->W[l] && m->b[l], "%s: null W/b for layer %d", what, l);
  return CNB_OK;
}

}  // namespace

bool cnb_mlp_mixed_supported(const cnb_mlp* m) {
  if (!m || m->num_layers < 1 || m->num_layers > CNB_MAX_LAYERS) return false;
  if (m->out_activation != CNB_ACT_NONE && m->out_activation != CNB_ACT_RELU && m->out_activation != CNB_ACT_SIGMOID) return false;
  for (int l = 0; l <= m->num_layers; ++l)
    if (m->dims[l] < 1 || m->dims[l] > MX_MAX) return false;
  return true;
}

int64_t cnb_mlp_mixed_hidden_floats(const cnb_mlp* m, int64_t n, int training) { return hidden_floats(m, n, training != 0); }
int64_t cnb_mlp_mixed_work_floats(const cnb_mlp* m, int64_t n) { return work_floats(m, n); }

int cnb_mlp_mixed_fwd_ws(const cnb_mlp* m, const float* x, int64_t x_stride, int64_t n, float* y, float* hidden, int training, cudaStream_t stream) {
  int rc = check_mlp(m, "mlp_mixed_fwd");
  if (rc) return rc;
  if (n <= 0) return CNB_OK;
  CNB_REQUIRE(x && y, "mlp_mixed_fwd: null x / y");
  CNB_REQUIRE(m->num_layers == 1 || hidden != nullptr, "mlp_mixed_fwd: null scratch (cnb_mlp_mixed_scratch_floats)");
  if ((rc = set_smem_attrs())) return rc;
  __half* h = reinterpret_cast<__half*>(hidden);
  const int grid = grid_for(n, cnb_num_sms() * CTAS_PER_SM);
  const __half* in16 = nullptr;
  int64_t ldin = x_stride;
  for (int l = 0; l < m->num_layers; ++l) {
    const int K = m->dims[l], N = m->dims[l + 1];
    const bool last = l == m->num_layers - 1;
    __half* out16 = last ? nullptr : h + hidden_off(m, n, l, training != 0);
    k_mx_fwd<<<grid, ROWS, fwd_smem(K, N), stream>>>(l == 0 ? x : nullptr, in16, ldin, n, K, N, m->W[l], m->b[l], last ? m->out_activation : CNB_ACT_RELU,
                                                     last ? y : nullptr, out16, up8(N));
    if ((rc = cnb_check_launch("mlp_mixed fwd"))) return rc;
    in16 = out16;
    ldin = up8(N);
  }
  return CNB_OK;
}

int cnb_mlp_mixed_bwd_ws(const cnb_mlp* m, const float* x, int64_t x_stride, const float* hidden, const float* y, const float* dy, int64_t n, float* dx,
                         int64_t dx_stride, float* work, cudaStream_t stream) {
  int rc = check_mlp(m, "mlp_mixed_bwd");
  if (rc) return rc;
  if (n <= 0) return CNB_OK;
  const int nl = m->num_layers;
  CNB_REQUIRE(x && dy && work, "mlp_mixed_bwd: null x / dy / scratch");
  CNB_REQUIRE(m->out_activation == CNB_ACT_NONE || y != nullptr, "mlp_mixed_bwd: the output activation's derivative needs y");
  CNB_REQUIRE(nl == 1 || hidden != nullptr, "mlp_mixed_bwd: null hidden activations");
  if ((rc = set_smem_attrs())) return rc;
  const __half* h = reinterpret_cast<const __half*>(hidden);
  __nv_bfloat16* dzb = reinterpret_cast<__nv_bfloat16*>(work);
  float* part = work + up4l((n * dz_w(m) + 1) / 2);
  const int64_t img = img_floats(m), ldz = dz_w(m);
  const int grid = grid_for(n, cnb_num_sms() * CTAS_PER_SM);
  const int grid_dw = grid_for(n, DW_PARTS);
  for (int l = nl - 1; l >= 0; --l) {
    const int IN = m->dims[l], OUT = m->dims[l + 1];
    DzSrc src{nullptr, nullptr, CNB_ACT_NONE, nullptr, 0};
    if (l == nl - 1) { src.dy = dy; src.y = y; src.act = m->out_activation; }
    else { src.dz = dzb; src.ldz = ldz; }
    const __half* xin16 = l > 0 ? h + hidden_off(m, n, l - 1, true) : nullptr;
    const int64_t ldx = l > 0 ? up8(IN) : x_stride;
    if (m->dW[l] != nullptr || m->db[l] != nullptr) {
      k_mx_dw<<<grid_dw, ROWS, dw_smem(IN), stream>>>(src, l == 0 ? x : nullptr, xin16, ldx, n, OUT, IN, part, img);
      if ((rc = cnb_check_launch("mlp_mixed dW"))) return rc;
      const int64_t elems = (int64_t)OUT * IN + OUT;
      k_mx_reduce<<<(unsigned)((elems + 255) / 256), 256, 0, stream>>>(part, grid_dw, img, OUT, IN, m->dW[l], m->db[l]);
      if ((rc = cnb_check_launch("mlp_mixed dW reduce"))) return rc;
    }
    if (l > 0) {
      k_mx_dx<<<grid, ROWS, dx_smem(OUT, IN), stream>>>(src, n, OUT, IN, m->W[l], xin16, up8(IN), dzb, nullptr, ldz);
      if ((rc = cnb_check_launch("mlp_mixed dX"))) return rc;
    } else if (dx != nullptr) {
      k_mx_dx<<<grid, ROWS, dx_smem(OUT, IN), stream>>>(src, n, OUT, IN, m->W[l], nullptr, 0, nullptr, dx, dx_stride);
      if ((rc = cnb_check_launch("mlp_mixed dX0"))) return rc;
    }
  }
  return CNB_OK;
}

// kernels launched by one call (stage timers of the fused pipeline)
int cnb_mlp_mixed_launches(const cnb_mlp* m, bool bwd, bool want_dx) {
  if (!bwd) return m->num_layers;
  int k = 0;
  for (int l = 0; l < m->num_layers; ++l) k += (m->dW[l] || m->db[l] ? 2 : 0) + ((l > 0 || want_dx) ? 1 : 0);
  return k;
}

// ---- C ABI: scratch = [hidden (training: kept for the backward) | backward work] ----------------------------------------------------------
extern "C" int64_t cnb_mlp_mixed_scratch_floats(const cnb_mlp* m, int64_t n, int32_t training) {
  if (!cnb_mlp_mixed_supported(m) || n <= 0) return 0;
  return hidden_floats(m, n, training != 0) + (training ? work_floats(m, n) : 0);
}

extern "C" int cnb_mlp_mixed_fwd(const cnb_mlp* m, const float* x, int64_t x_stride, int64_t n, float* y, float* scratch, int32_t training,
                                 cnb_stream_t stream) {
  return cnb_mlp_mixed_fwd_ws(m, x, x_stride, n, y, scratch, training, (cudaStream_t)stream);
}

extern "C" int cnb_mlp_mixed_bwd(const cnb_mlp* m, const float* x, int64_t x_stride, const float* y, const float* dy, int64_t n, float* dx,
                                 int64_t dx_stride, float* scratch, cnb_stream_t stream) {
  int rc = check_mlp(m, "mlp_mixed_bwd");
  if (rc) return rc;
  if (n <= 0) return CNB_OK;
  CNB_REQUIRE(scratch != nullptr, "mlp_mixed_bwd: null scratch (the one cnb_mlp_mixed_fwd(training=1) wrote)");
  return cnb_mlp_mixed_bwd_ws(m, x, x_stride, scratch, y, dy, n, dx, dx_stride, scratch + hidden_floats(m, n, true), (cudaStream_t)stream);
}
