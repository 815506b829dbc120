// FruitField backward entirely on tcgen05 / TMEM (rows a1/a5/a6 of SURVEY.md section 8, the autograd of fruit_field.py:169-302).
//
// An mma.sync design that keeps a 16-sample tile per warp and chains the 13 layers through register fragments needs 225 registers, runs 8 warps per SM
// and leaves a dependent HMMA -> F2FP -> HMMA chain with nothing to hide it behind (measured: tensor pipe 26 %, issue 31 %, 30 k cycles per 128-sample
// batch; DESIGN.md section 4).  Here a batch of 128 samples is ONE tcgen05.mma tile (M = 128): every layer is 1-4 asynchronous MMAs issued by a single
// thread, the accumulator lives in tensor memory, and the "epilogue" between two layers is row-parallel -- thread r of a 128-thread warpgroup owns
// sample r: it reads its accumulator row with tcgen05.ld, applies bias / ReLU / the ReLU mask, converts to bf16 and writes the row back to shared memory
// as the next layer's operand (8 conflict-free 16-byte stores).  No fragment layouts, no shuffles, ~150 instructions per thread and layer.  Two
// warpgroups work on two batches at once, so one batch's MMAs run under the other's epilogue.
//
// Shared-memory operand format (no-swizzle canonical UMMA layouts, tests/micro/umma_chain_test.cu):
//   activation / gradient matrices [128 samples][64 features] bf16:  byte(s, f) = (f/8)*2048 + s*16 + (f%8)*2
//       as the A operand of a layer (K-major: K = features)        : LBO 2048, SBO 128
//       as an operand of dW = dY^T X (MN-major: K = samples)       : LBO 128,  SBO 2048      -- the SAME bytes, no second copy
//   weights [out][in] bf16:                                          byte(o, i) = (i/8)*(OUT*16) + o*16 + (i%8)*2
//       forward  Y = X W^T  (B K-major)                             : LBO OUT*16, SBO 128
//       backward dX = dY W  (B MN-major)                            : LBO 128,    SBO OUT*16  -- the SAME bytes again
// kind::f16 needs A and B in one format (a bf16 A with an fp16 B is an illegal instruction: umma_chain_test), and the gradients need bf16's
// range, so everything here is bf16, including the forward recompute.  The two places where the recomputed pre-activation would enter a
// derivative with full weight -- trunc_exp' of the density and sigmoid' of the colour -- take the FORWARD's fp32 values instead (the
// 4-float-per-sample stash k_field_mixed_fwd writes in training), as autograd does.
//
// dW: eight accumulators stay in TMEM across all batches of the persistent CTA (304 of 512 columns; 2 x 64 more are the two warpgroups' layer
// accumulators) and are flushed once per CTA through a shared-memory image.  The bias gradients ride along as one extra row / column of each dW
// GEMM, read from a constant that sits behind (or inside) its operand -- see the buffer order below.
//
// Three single-thread issuers: one per warpgroup for the layer MMAs (the only thing the epilogue threads wait for), one for all dW / bias MMAs
// (every dW accumulator has one issuing thread; its completion is only needed before the next overwrite of D / DS / the X buffers).
// Per batch and warpgroup, 12 (operands ready -> MMAs -> accumulator ready) round trips, see `issue_chain` / `issue_dw` / the epilogue:
//   0 B1 fwd | 1 B2 fwd | 2 R1 fwd | 3 R2 fwd | 4 dWr3, dX r3 | 5 dWr2, dX r2 | 6 dWr1, dX r1 | 7 S1 fwd | 8 S2 fwd | 9 dWh, dWs2, dX s2 |
//   10 dWs1, dWb2, dX b2 | 11 dWb1, dX b1 (= d encoded features, written level-major for cnb_hashgrid_bwd_level_major)
#include <cstdio>
#include <cstdlib>
#include <type_traits>

#include "field_mixed.cuh"
#include "umma.cuh"

using namespace cnbmix;
using namespace cnbumma;

namespace {

constexpr int ROWS = 128;            // samples per batch = UMMA M = threads of one epilogue warpgroup
constexpr int NWG = 2;               // batches in flight per CTA
constexpr int EPI = NWG * ROWS;
// + two more warpgroups: warps 8, 9 = the layer-MMA issuers of the two epilogue warpgroups, warp 10 = the dW issuer, warps 11..15 idle.
// The idle warps pay for the epilogue's registers: setmaxnreg re-splits the register file after launch, and the sum must not exceed what
// the CTA was launched with, so 4 x 128 threads at 128 registers is what lets the epilogue warpgroups rise to 200 (200 + 200 + 56 + 56 =
// 4 x 128; the increase blocks until the decreases have released enough).
constexpr int KTHREADS = EPI + 256;
constexpr uint32_t FB = 2048;        // bytes of one 8-feature block of an activation matrix (128 rows x 16 B)
constexpr int NSTEP = 12;

// per-warpgroup activation buffers (byte offsets inside the warpgroup's region).  The ORDER carries the bias gradients: every dW GEMM gets
// its bias row / column from a block of the NEXT buffer (or a spare column of its own) that holds a constant --
//   AH | BO      : dWb2^T = [AH | BO ...]^T DS with M = 128: row 64 is BO's column 0, which is set to 1 (the cleared dba slot; its weight columns are 0)
//   R1 | ONES    : dWr2 / dWs2 = dY^T [R1 | ones] with N = 72: column 64;   dWb1 = dY^T [X0 (4 blocks) | ones written behind it], N = 40: column 32
//   R2 | AIN     : dWr3^T / dWh^T = [R2 | AIN ...]^T DS with M = 128: row 64 is AIN's column 0 = SH component 0, the constant 0.2820948 (bf16)
//   AIN itself   : column 16 (the dba slot, = BO's column 0 = 1): dWr1's column 16;   BO: dWs1's column 0
// (bias gradients as separate dY^T x ones GEMMs were 64 of the dW issuer's 128 MMAs per batch)
constexpr uint32_t B_DS = 0;                   // 16-feature matrices: d(rgb pre-activation) | [d_sem] | d(base output)
constexpr uint32_t B_AH = B_DS + 2 * FB;       // base hidden
constexpr uint32_t B_BO = B_AH + 8 * FB;       // [1 | geo15]
constexpr uint32_t B_R1 = B_BO + 2 * FB;       // rgb hidden 1      | later: semantic hidden 1 | later: encoded features + ones (for dWb1)
constexpr uint32_t B_ONES = B_R1 + 8 * FB;     // one block of ones, written once
constexpr uint32_t B_R2 = B_ONES + FB;         // rgb hidden 2      | later: semantic hidden 2
constexpr uint32_t B_AIN = B_R2 + 8 * FB;      // encoded features (step 0) | [SH16 | 1, geo15 | emb32]
constexpr uint32_t B_D = B_AIN + 8 * FB;       // every 64-wide dY
constexpr uint32_t WG_BYTES = B_D + 8 * FB;    // 92 160
// weights (bf16, layout above)
constexpr uint32_t W_B1 = 0;                   // [64][32]
constexpr uint32_t W_B2 = W_B1 + 64 * 32 * 2;  // [16][64]
constexpr uint32_t W_R1 = W_B2 + 16 * 64 * 2;  // [64][64]  in = [SH16 | 0, geo15 | emb32]
constexpr uint32_t W_R2 = W_R1 + 64 * 64 * 2;
constexpr uint32_t W_R3 = W_R2 + 64 * 64 * 2;  // [16][64]  rows 3..15 zero
constexpr uint32_t W_S1 = W_R3 + 16 * 64 * 2;  // [64][16]  in = [0 | geo15]
constexpr uint32_t W_S2 = W_S1 + 64 * 16 * 2;
constexpr uint32_t W_BYTES = W_S2 + 64 * 64 * 2;   // 34 816
// fp32 constants
constexpr int C_BB1 = 0, C_BB2 = 64, C_BR1 = 80, C_BR2 = 144, C_BS1 = 208, C_BS2 = 272, C_WH = 336, C_FLOATS = 400;
constexpr uint32_t O_WG = 0, O_W = NWG * WG_BYTES, O_CONST = O_W + W_BYTES, O_BAR = O_CONST + C_FLOATS * 4,
                   SMEM_TC5 = O_BAR + 128;   // 4 NWG mbarriers + the TMEM base slot
static_assert(SMEM_TC5 <= 232448, "227 KB of dynamic shared memory per CTA");
// TMEM columns
constexpr uint32_t T_CHAIN = 0;   // + 64 * warpgroup
// dW accumulators (fp32 columns).  M = 64 GEMMs keep row m in lane (m % 16) + 32 (m / 16); the three transposed ones are M = 128 (row r in lane r).
constexpr uint32_t T_R3 = 128;          // [64 in + bias row 64][16]   M = 128
constexpr uint32_t T_R2 = T_R3 + 16;    // [64 out][64 in | bias col 64 ...]  72 columns
constexpr uint32_t T_R1 = T_R2 + 72;    // [64][64], column 16 = bias
constexpr uint32_t T_H = T_R1 + 64;     // [64 in + bias row 64][8]    M = 128
constexpr uint32_t T_S2 = T_H + 8;      // 72 columns
constexpr uint32_t T_S1 = T_S2 + 72;    // [64][16], column 0 = bias
constexpr uint32_t T_B2 = T_S1 + 16;    // [64 in + bias row 64][16]   M = 128
constexpr uint32_t T_B1 = T_B2 + 16;    // [64][32 | bias col 32 ...]  40 columns
constexpr uint32_t T_END = T_B1 + 40;   // 432
static_assert(T_END <= 512, "TMEM columns");

// gradient image: every weight / bias gradient in its global element order (one image per CTA, reduced by k_tc5_reduce)
constexpr int I_WR3 = 0, I_BR3 = 192, I_WR2 = 196, I_BR2 = I_WR2 + 4096, I_WR1 = I_BR2 + 64, I_BR1 = I_WR1 + 4032, I_WH = I_BR1 + 64, I_BH = I_WH + 64,
              I_WS2 = I_BH + 4, I_BS2 = I_WS2 + 4096, I_WS1 = I_BS2 + 64, I_BS1 = I_WS1 + 960, I_WB2 = I_BS1 + 64, I_BB2 = I_WB2 + 1024,
              I_WB1 = I_BB2 + 16, I_BB1 = I_WB1 + 2048, I_END = I_BB1 + 64;
static_assert(I_END * 4 <= (int)(NWG * WG_BYTES), "gradient image must fit the activation buffers");
static_assert(I_END <= CTX_PART_FLOATS && I_END % 4 == 0, "partial image size");

struct BwdArgs {
  MixArgs m;
  float* part;      // [gridDim.x][CTX_PART_FLOATS] per-CTA gradient images
  const __half* x0;
  const float* stash;
  const uint4* masks;
  const float *d_density, *d_rgb, *d_sem;
  float* d_x0;
  float *dWb1, *dbb1, *dWb2, *dbb2, *dWs1, *dbs1, *dWs2, *dbs2, *dWh, *dbh, *dWr1, *dbr1, *dWr2, *dbr2, *dWr3, *dbr3;
  float* d_embedding;
  long long* dbg;   // CNB_TC5_DEBUG=1: cycle counters of CTA 0 (issuer wait / issue, epilogue wait / work per step)
};

// ---- tcgen05 plumbing (descriptors, umma, tm_load: umma.cuh) -----------------------------------------------------------------------------
// The issuer is ONE thread: what it executes per MMA is on the critical path of every layer.  A descriptor is built once per GEMM; a K step
// only adds to the start-address field of its low word.
template <int KS, uint32_t A_STEP, uint32_t B_STEP>
__device__ __forceinline__ void mm_loop(uint32_t tm, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi, uint32_t id, bool acc0) {
#pragma unroll
  for (int ks = 0; ks < KS; ++ks)
    umma(tm, desc64(a_lo + ks * (A_STEP >> 4), a_hi), desc64(b_lo + ks * (B_STEP >> 4), b_hi), id, (ks > 0 || acc0) ? 1u : 0u);
}
// forward layer: TM[128][OUT] = A[128][K] W^T
template <int K, int OUT>
__device__ __forceinline__ void mm_fwd(uint32_t tm, uint32_t a_s, uint32_t w_s) {
  mm_loop<K / 16, 2 * FB, 2 * OUT * 16>(tm, desc_lo(a_s, FB), desc_hi(128), desc_lo(w_s, OUT * 16), desc_hi(128), idesc(128, OUT, 0, 0), false);
}
// input gradient: TM[128][NIN] = dY[128][KOUT] W[:, first input block ...]   (w_s already points at the first 8-input block wanted)
template <int KOUT, int OUT, int NIN>
__device__ __forceinline__ void mm_dx(uint32_t tm, uint32_t dy_s, uint32_t w_s) {
  mm_loop<KOUT / 16, 2 * FB, 256>(tm, desc_lo(dy_s, FB), desc_hi(128), desc_lo(w_s, 128), desc_hi(OUT * 16), idesc(128, NIN, 0, 1), false);
}
// weight gradient: TM[M features of A][N features of B] (+)= A^T B over the 128 samples (M = 64, or 128 for the transposed GEMMs whose
// bias row lives in the block behind A's 64 features)
template <int N, int M = 64>
__device__ __forceinline__ void mm_dw(uint32_t tm, uint32_t a_s, uint32_t b_s, bool first) {
  mm_loop<ROWS / 16, 256, 256>(tm, desc_lo(a_s, 128), desc_hi(FB), desc_lo(b_s, 128), desc_hi(FB), idesc(M, N, 1, 1), !first);
}

// row-owner store of NB 8-feature blocks (bf16) of this thread's sample row
template <int NB>
__device__ __forceinline__ void row_store(unsigned char* mat, int r, const uint32_t (&w)[NB * 4]) {
#pragma unroll
  for (int fb = 0; fb < NB; ++fb) *reinterpret_cast<uint4*>(mat + fb * FB + r * 16) = make_uint4(w[4 * fb], w[4 * fb + 1], w[4 * fb + 2], w[4 * fb + 3]);
}
// y = relu?(acc + bias) -> bf16 row
template <int NC, bool RELU>
__device__ __forceinline__ void bias_act_pack(const float (&v)[NC], const float* __restrict__ bias, uint32_t (&w)[NC / 2]) {
#pragma unroll
  for (int c = 0; c < NC; c += 4) {
    const float4 b = *reinterpret_cast<const float4*>(bias + c);
    float y0 = v[c] + b.x, y1 = v[c + 1] + b.y, y2 = v[c + 2] + b.z, y3 = v[c + 3] + b.w;
    if (RELU) { y0 = fmaxf(y0, 0.f); y1 = fmaxf(y1, 0.f); y2 = fmaxf(y2, 0.f); y3 = fmaxf(y3, 0.f); }
    w[c / 2] = pack_bf2(y0, y1);
    w[c / 2 + 1] = pack_bf2(y2, y3);
  }
}
// dY = dX where the FORWARD's activation was positive: the forward kernel keeps one flag per hidden unit (relu_flags in field_mixed.cuh:
// for packed word j = columns 2j, 2j+1 the flags are bits (sh + j/4) and (16 + sh + j/4) of word P[j % 4]), so the masks are those of the
// function whose loss was evaluated, not of the bf16 recompute (a flipped unit is a full-size error in dY: the relative L2 error of the
// gradients goes with the square root of the flipped fraction)
template <int NC>
__device__ __forceinline__ void mask_pack(const float (&v)[NC], const uint32_t (&P)[4], int sh, uint32_t (&w)[NC / 2]) {
#pragma unroll
  for (int j = 0; j < NC / 2; ++j) {
    const uint32_t m = ((P[j & 3] >> (sh + (j >> 2))) & 0x10001u) * 0xFFFFu;
    w[j] = pack_bf2(v[2 * j], v[2 * j + 1]) & m;
  }
}

// One weight matrix into its UMMA layout, in two phases.  Consecutive threads take consecutive input PAIRS of one output row (coalesced
// global loads); ALL loads of ALL matrices are issued before the first conversion, so the prologue pays one memory round trip, not one per
// loop iteration (the parameters have usually left L2 since the optimiser wrote them: 14-22 k cycles per CTA with loads issued loop by loop).
template <int OUT, int IN>
struct WLoad {
  static constexpr int PAIRS = OUT * IN / 2;
  static constexpr int SLOTS = (PAIRS + KTHREADS - 1) / KTHREADS;   // blockDim.x = KTHREADS
  float v[SLOTS][2];
  template <typename Src>
  __device__ __forceinline__ void load(Src src) {
#pragma unroll
    for (int u = 0; u < SLOTS; ++u) {
      const int p = (int)threadIdx.x + u * KTHREADS;
      const int o = p / (IN / 2), i = 2 * (p - o * (IN / 2));
      v[u][0] = p < PAIRS ? src(o, i) : 0.f;
      v[u][1] = p < PAIRS ? src(o, i + 1) : 0.f;
    }
  }
  __device__ __forceinline__ void store(unsigned char* dst) const {
#pragma unroll
    for (int u = 0; u < SLOTS; ++u) {
      const int p = (int)threadIdx.x + u * KTHREADS;
      const int o = p / (IN / 2), i = 2 * (p - o * (IN / 2));
      if (p < PAIRS) *reinterpret_cast<uint32_t*>(dst + (i >> 3) * (OUT * 16) + o * 16 + (i & 7) * 2) = pack_bf2(v[u][0], v[u][1]);
    }
  }
};
__device__ inline void load_weights_tc5(const MixArgs& a, unsigned char* Wb, float* Cf, long long* tmark) {
  const int in0 = a.in0;
  const int tid = threadIdx.x;
  WLoad<64, 32> b1; WLoad<16, 64> b2, r3; WLoad<64, 64> r1, r2, s2; WLoad<64, 16> s1;
  b1.load([&](int o, int i) { return i < in0 ? __ldg(a.Wb1 + o * in0 + i) : 0.f; });
  b2.load([&](int o, int i) { return __ldg(a.Wb2 + o * 64 + i); });
  r3.load([&](int o, int i) { return o < 3 ? __ldg(a.Wr3 + o * 64 + i) : 0.f; });
  r1.load([&](int o, int i) { return i == 16 ? 0.f : __ldg(a.Wr1 + o * 63 + (i < 16 ? i : i - 1)); });
  r2.load([&](int o, int i) { return __ldg(a.Wr2 + o * 64 + i); });
  s2.load([&](int o, int i) { return __ldg(a.Ws2 + o * 64 + i); });
  s1.load([&](int o, int i) { return i >= 1 ? __ldg(a.Ws1 + o * 15 + (i - 1)) : 0.f; });
  float c[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, cb2 = 0.f;
  if (tid < 64) { c[0] = __ldg(a.bb1 + tid); c[1] = __ldg(a.br1 + tid); c[2] = __ldg(a.br2 + tid); c[3] = __ldg(a.bs1 + tid); c[4] = __ldg(a.bs2 + tid); c[5] = __ldg(a.Wh + tid); }
  if (tid < 16) cb2 = __ldg(a.bb2 + tid);
  if (tmark) tmark[0] = clock64();   // all loads issued
  b1.store(Wb + W_B1);
  if (tmark) tmark[1] = clock64();   // first matrix converted and stored: its loads have landed
  b2.store(Wb + W_B2); r3.store(Wb + W_R3); r1.store(Wb + W_R1); r2.store(Wb + W_R2); s2.store(Wb + W_S2); s1.store(Wb + W_S1);
  if (tid < 64) { Cf[C_BB1 + tid] = c[0]; Cf[C_BR1 + tid] = c[1]; Cf[C_BR2 + tid] = c[2]; Cf[C_BS1 + tid] = c[3]; Cf[C_BS2 + tid] = c[4]; Cf[C_WH + tid] = c[5]; }
  if (tid < 16) Cf[C_BB2 + tid] = cb2;
}

// 32 values per lane -> lane c ends with the warp-wide sum of value c (31 shuffles)
template <int OFF>
__device__ __forceinline__ void tr_step(float (&x)[32], int lane) {
  const bool up = (lane & OFF) != 0;
#pragma unroll
  for (int j = 0; j < OFF; ++j) {
    const float send = up ? x[j] : x[j + OFF];
    const float keep = up ? x[j + OFF] : x[j];
    x[j] = keep + __shfl_xor_sync(0xffffffffu, send, OFF);
  }
}
__device__ __forceinline__ float transpose_reduce32(float (&x)[32], int lane) {
  tr_step<16>(x, lane); tr_step<8>(x, lane); tr_step<4>(x, lane); tr_step<2>(x, lane); tr_step<1>(x, lane);
  return x[0];
}

// The layer MMA of one step of one warpgroup's batch: what the epilogue threads wait for.  Its descriptors are prepared BEFORE the issuer
// waits for the operands (`prepare_chain`), so that after the wake-up only the K-step adds and the MMAs themselves are on the critical path.
struct ChainOp {
  uint32_t a_lo, a_hi, b_lo, b_hi, id, a_step, b_step;
  int ks;
};
template <int K, int OUT>
__device__ __forceinline__ ChainOp op_fwd(uint32_t a_s, uint32_t w_s) {
  return ChainOp{desc_lo(a_s, FB), desc_hi(128), desc_lo(w_s, OUT * 16), desc_hi(128), idesc(128, OUT, 0, 0), (2 * FB) >> 4, (2 * OUT * 16) >> 4, K / 16};
}
template <int KOUT, int OUT, int NIN>
__device__ __forceinline__ ChainOp op_dx(uint32_t dy_s, uint32_t w_s) {
  return ChainOp{desc_lo(dy_s, FB), desc_hi(128), desc_lo(w_s, 128), desc_hi(OUT * 16), idesc(128, NIN, 0, 1), (2 * FB) >> 4, 256 >> 4, KOUT / 16};
}
__device__ __forceinline__ ChainOp prepare_chain(int step, uint32_t wg_s, uint32_t w_s) {
  const uint32_t DS = wg_s + B_DS, AH = wg_s + B_AH, BO = wg_s + B_BO, AIN = wg_s + B_AIN, R1 = wg_s + B_R1, D = wg_s + B_D;
  switch (step) {
    case 0: return op_fwd<32, 64>(AIN, w_s + W_B1);   // the encoded features are staged in the (still free) AIN buffer
    case 1: return op_fwd<64, 16>(AH, w_s + W_B2);
    case 2: return op_fwd<64, 64>(AIN, w_s + W_R1);
    case 3: return op_fwd<64, 64>(R1, w_s + W_R2);
    case 4: return op_dx<16, 16, 64>(DS, w_s + W_R3);
    case 5: return op_dx<64, 64, 64>(D, w_s + W_R2);
    case 6: return op_dx<64, 64, 48>(D, w_s + W_R1 + 2 * (64 * 16));   // inputs 16..63: [0, geo15 | emb32]
    case 7: return op_fwd<16, 64>(BO, w_s + W_S1);
    case 8: return op_fwd<64, 64>(R1, w_s + W_S2);
    case 9: return op_dx<64, 64, 64>(D, w_s + W_S2);
    case 10: return op_dx<16, 16, 64>(DS, w_s + W_B2);
    default: return op_dx<64, 64, 32>(D, w_s + W_B1);
  }
}
__device__ __forceinline__ void issue_chain(const ChainOp& o, uint32_t tm) {
  for (int ks = 0; ks < o.ks; ++ks) umma(tm, desc64(o.a_lo + ks * o.a_step, o.a_hi), desc64(o.b_lo + ks * o.b_step, o.b_hi), o.id, ks > 0 ? 1u : 0u);
}
// The weight-gradient MMAs of a step (steps 4-6 and 9-11): off the epilogue's critical path, issued by their own thread.
__device__ __forceinline__ constexpr bool step_has_dw(int step) { return (step >= 4 && step <= 6) || step >= 9; }
__device__ __forceinline__ void issue_dw(int step, uint32_t tmem, uint32_t wg_s, bool first) {
  const uint32_t DS = wg_s + B_DS, AH = wg_s + B_AH, BO = wg_s + B_BO, AIN = wg_s + B_AIN, R1 = wg_s + B_R1, R2 = wg_s + B_R2, D = wg_s + B_D;
  switch (step) {
    case 4: mm_dw<16, 128>(tmem + T_R3, R2, DS, first); break;       // dWr3^T [in | AIN col 0][out]
    case 5: mm_dw<72>(tmem + T_R2, D, R1, first); break;             // [R1 | ones]
    case 6: mm_dw<64>(tmem + T_R1, D, AIN, first); break;            // AIN column 16 = 1
    case 9:
      mm_dw<8, 128>(tmem + T_H, R2, DS, first);                      // dWh^T [in | AIN col 0][1]
      mm_dw<72>(tmem + T_S2, D, R1, first);
      break;
    case 10:
      mm_dw<16>(tmem + T_S1, D, BO, first);                          // BO column 0 = 1
      mm_dw<16, 128>(tmem + T_B2, AH, DS, first);                    // dWb2^T [in | BO col 0][out]
      break;
    default: mm_dw<40>(tmem + T_B1, D, R1, first); break;            // [X0 | ones]
  }
}

__global__ void __launch_bounds__(KTHREADS, 1) k_field_bwd_tc5(const __grid_constant__ BwdArgs b) {
  extern __shared__ __align__(1024) unsigned char smem[];
  const MixArgs& a = b.m;
  const long long t_start = b.dbg ? clock64() : 0;
  unsigned char* Wb = smem + O_W;
  float* Cf = reinterpret_cast<float*>(smem + O_CONST);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + O_BAR);   // ready[NWG], dwready[NWG] (128 arrivals), done[NWG], dwdone[NWG] (tcgen05.commit)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 4 * NWG);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  long long tmark[2] = {0, 0};
  load_weights_tc5(a, Wb, Cf, b.dbg ? tmark : nullptr);
  for (int e = threadIdx.x; e < (int)(NWG * FB / 4); e += KTHREADS)   // the ones block of each warpgroup, bf16 (1, 1)
    reinterpret_cast<uint32_t*>(smem + O_WG + (uint32_t)(e / (FB / 4)) * WG_BYTES + B_ONES)[e % (FB / 4)] = 0x3F803F80u;
  const long long t_w = b.dbg ? clock64() : 0;
  if (threadIdx.x == 0) {
    for (int w = 0; w < NWG; ++w) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(bars + w)), "r"(ROWS));
      asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(bars + NWG + w)), "r"(ROWS));
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"((uint32_t)__cvta_generic_to_shared(bars + 2 * NWG + w)));
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"((uint32_t)__cvta_generic_to_shared(bars + 3 * NWG + w)));
    }
    asm volatile("fence.mbarrier_init.release.cluster;");
  }
  if (warp == 0) {  // all 512 TMEM columns: the CTA owns the SM (214 KB of shared memory)
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"((uint32_t)__cvta_generic_to_shared(tmem_slot)));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("tcgen05.fence::before_thread_sync;");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;");
  const uint32_t tmem = *tmem_slot;
  if (b.dbg && blockIdx.x == 0 && threadIdx.x == 0) { b.dbg[49] = clock64() - t_start; b.dbg[52] = t_w - t_start; b.dbg[55] = tmark[0] - t_start; b.dbg[56] = tmark[1] - t_start; }
  const uint32_t smem_s = (uint32_t)__cvta_generic_to_shared(smem);
  const uint32_t bars_s = smem_s + O_BAR;
  const int S = a.sm.samples_per_ray;
  const int64_t N = a.sm.num_rays * S;
  const int64_t nbatches = (N + ROWS - 1) / ROWS;
  // batches of this CTA: blockIdx.x + j * gridDim.x ; warpgroup w takes j = w, w + 2, ...
  const int64_t nb_cta = nbatches > blockIdx.x ? (nbatches - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

  if (warp >= EPI / 32) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");   // 4 x 128 at launch = 200 + 200 + 56 + 56 per sub-partition lane
    // ===== three issuers (warp-uniform: all lanes wait, one elected lane issues -- no per-instruction election loop in the SASS) =====
    //   warp 8 + w : the layer MMAs of warpgroup w -- the epilogue's critical path, nothing else in this thread's queue
    //   warp 10    : every dW / bias MMA of both warpgroups -- each dW accumulator has ONE issuing thread
    const int iw = warp - EPI / 32;
    if (iw < NWG) {
      uint32_t ph = 0;
      for (int64_t j = iw; j < nb_cta; j += NWG) {
        for (int step = 0; step < NSTEP; ++step) {
          const long long tq0 = b.dbg ? clock64() : 0;
          const ChainOp op = prepare_chain(step, smem_s + O_WG + (uint32_t)iw * WG_BYTES, smem_s + O_W);
          mbar_wait(bars_s + 8 * iw, ph);
          ph ^= 1u;
          asm volatile("tcgen05.fence::after_thread_sync;");
          const long long tq1 = b.dbg ? clock64() : 0;
          if (elect_one()) {
            issue_chain(op, tmem + T_CHAIN + 64u * (uint32_t)iw);
            asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.b64 [%0];" ::"l"((uint64_t)(bars_s + 8 * (2 * NWG + iw))) : "memory");
            if (b.dbg && blockIdx.x == 0 && iw == 0) { b.dbg[step] += tq1 - tq0; b.dbg[12 + step] += clock64() - tq1; }
          }
          __syncwarp();
        }
      }
    } else if (iw == NWG) {
      uint32_t ph[NWG] = {0u, 0u};
      for (int64_t j0 = 0; j0 < nb_cta; j0 += NWG) {
        for (int step = 0; step < NSTEP; ++step) {
          if (!step_has_dw(step)) continue;
#pragma unroll
          for (int w = 0; w < NWG; ++w) {
            if (j0 + w >= nb_cta) continue;
            // dwready[w] completes one phase per dW step; the epilogue waits for this step's dwdone before it arrives for the next dW step,
            // so the barrier is never more than one phase ahead of this wait (no parity aliasing)
            mbar_wait(bars_s + 8 * (NWG + w), ph[w]);
            ph[w] ^= 1u;
            asm volatile("tcgen05.fence::after_thread_sync;");
            if (elect_one()) {
              uint32_t wg_s = smem_s + O_WG + (uint32_t)w * WG_BYTES;
              asm volatile("" : "+r"(wg_s));
              issue_dw(step, tmem, wg_s, j0 == 0 && w == 0);
              asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.b64 [%0];" ::"l"((uint64_t)(bars_s + 8 * (3 * NWG + w))) : "memory");
            }
            __syncwarp();
          }
        }
      }
    }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 200;");
    // ===== epilogue warpgroups: thread r owns sample row r of its warpgroup's batch =====
    const int wg = warp >> 2, r = threadIdx.x & (ROWS - 1);
    unsigned char* base = smem + O_WG + (uint32_t)wg * WG_BYTES;
    const uint32_t ready_s = bars_s + 8 * wg, dwready_s = bars_s + 8 * (NWG + wg), done_s = bars_s + 8 * (2 * NWG + wg);
    const uint32_t trow = tmem + ((uint32_t)(32 * (warp & 3)) << 16) + T_CHAIN + 64u * (uint32_t)wg;
    uint32_t dphase = 0;
    int estep = 0;
    long long te = 0;
    const bool dbg_on = b.dbg != nullptr && blockIdx.x == 0 && threadIdx.x == 0;
    long long t_fence = 0, t_dbgrmw = 0;
    auto ready = [&](bool dw = false) {   // this thread's operand rows are written and its accumulator reads are complete (dw: a dW step)
      if (dbg_on) { const long long t0 = clock64(); b.dbg[36 + estep] += t0 - te; ++estep; t_dbgrmw += clock64() - t0; }
      const long long tf = dbg_on ? clock64() : 0;
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      asm volatile("tcgen05.fence::before_thread_sync;");
      asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(ready_s) : "memory");
      if (dw) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(dwready_s) : "memory");
      if (dbg_on) t_fence += clock64() - tf;
    };
    const uint32_t dwdone_s = bars_s + 8 * (3 * NWG + wg);
    uint32_t wphase = 0;
    auto wait_dw = [&]() {   // the dW MMAs of the previous step have read their operands: D / DS / X buffers may be overwritten
      mbar_wait(dwdone_s, wphase);
      wphase ^= 1u;
    };
    auto wait_acc = [&]() {
      const long long tw = dbg_on ? clock64() : 0;
      mbar_wait(done_s, dphase);
      dphase ^= 1u;
      asm volatile("tcgen05.fence::after_thread_sync;");
      if (dbg_on) { te = clock64(); b.dbg[24 + estep - 1] += te - tw; }
    };
    // every global input of this thread's row; the NEXT batch's are requested right after step 0 of the current one (loop-carried registers,
    // so the compiler cannot sink the loads): fetched at the top of a batch they cost ~7 k exposed cycles per batch
    struct RowIn {
      uint4 xq[4];
      float4 st;
      uint4 mq[2];
      float drgb[3], dsem, ddens, dir[3];
      int cam;
    };
    auto load_row = [&](int64_t j, RowIn& in) {
      const int64_t i = (blockIdx.x + j * gridDim.x) * ROWS + r;
      const bool ok = j < nb_cta && i < N;
#pragma unroll
      for (int q = 0; q < 4; ++q) in.xq[q] = make_uint4(0u, 0u, 0u, 0u);
      in.st = make_float4(0.f, 0.f, 0.f, 0.f);
      in.mq[0] = in.mq[1] = make_uint4(0u, 0u, 0u, 0u);
      in.drgb[0] = in.drgb[1] = in.drgb[2] = 0.f; in.dsem = 0.f; in.ddens = 0.f;
      in.dir[0] = in.dir[1] = in.dir[2] = 0.f; in.cam = 0;
      if (j >= nb_cta) return;
      if (ok) {
#pragma unroll
        for (int q = 0; q < 4; ++q) in.xq[q] = __ldg(reinterpret_cast<const uint4*>(b.x0 + i * 32) + q);
        in.st = __ldg(reinterpret_cast<const float4*>(b.stash) + i);
        in.mq[0] = __ldg(b.masks + 2 * i); in.mq[1] = __ldg(b.masks + 2 * i + 1);
        if (b.d_rgb) { in.drgb[0] = __ldg(b.d_rgb + 3 * i); in.drgb[1] = __ldg(b.d_rgb + 3 * i + 1); in.drgb[2] = __ldg(b.d_rgb + 3 * i + 2); }
        if (b.d_sem) in.dsem = __ldg(b.d_sem + i);
        if (b.d_density) in.ddens = __ldg(b.d_density + i);
      }
      const int64_t ry = (i < N ? i : N - 1) / S;
      in.dir[0] = __ldg(a.sm.directions + 3 * ry); in.dir[1] = __ldg(a.sm.directions + 3 * ry + 1); in.dir[2] = __ldg(a.sm.directions + 3 * ry + 2);
      if (a.app_mode == CNB_APP_PER_CAMERA) in.cam = __ldg(a.sm.camera_indices + ry);
    };
    RowIn nxt;
    load_row(wg, nxt);
    for (int64_t j = wg; j < nb_cta; j += NWG) {
      const int64_t i = (blockIdx.x + j * gridDim.x) * ROWS + r;
      const bool valid = i < N;
      const int64_t ray = (valid ? i : N - 1) / S;
      const RowIn cur = nxt;
      const uint4 (&xq)[4] = cur.xq;
      const float4 st = cur.st;
      const uint4 (&mq)[2] = cur.mq;
      const float (&drgb)[3] = cur.drgb;
      const float dsem = cur.dsem, ddens = cur.ddens;
      const float dirx = cur.dir[0], diry = cur.dir[1], dirz = cur.dir[2];
      const int cam = cur.cam;
      const float* erow = a.app_mode == CNB_APP_PER_CAMERA ? a.embedding + (int64_t)cam * 32 : (a.app_mode == CNB_APP_MEAN ? a.embedding : nullptr);
      const uint32_t P0[4] = {mq[0].x, mq[0].z, mq[1].x, mq[1].z};   // base hidden | semantic hidden 1 << 8
      const uint32_t P1[4] = {mq[0].y, mq[0].w, mq[1].y, mq[1].w};   // rgb hidden 1 | rgb hidden 2 << 8
      uint32_t x0w[16];   // encoded features, bf16
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const uint32_t hw[4] = {xq[q].x, xq[q].y, xq[q].z, xq[q].w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&hw[e]));
          x0w[4 * q + e] = pack_bf2(f.x, f.y);
        }
      }
      if (dbg_on) { te = clock64(); estep = 0; }
      // ---- 0: encoded features -> AIN's first four blocks (free until step 2; D and R1 may still be read by the previous batch's dWb1 GEMM) ----
      row_store<4>(base + B_AIN, r, x0w);
      ready();
      load_row(j + NWG, nxt);
      // ---- 1: base hidden -----------------------------------------------------------------------------------------------------------
      {
        wait_acc();
        float v[64];
        tm_load<64>(trow, v);
        uint32_t w[32];
        bias_act_pack<64, true>(v, Cf + C_BB1, w);
        row_store<8>(base + B_AH, r, w);
        ready();
      }
      // ---- 2: base output -> BO = [0 | geo15], AIN = [SH16 | BO | emb32] --------------------------------------------------------------
      {
        float4 ev[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) ev[q] = erow ? __ldg(reinterpret_cast<const float4*>(erow) + q) : make_float4(0.f, 0.f, 0.f, 0.f);
        float sh[16];
        cnb_sh16(dirx, diry, dirz, sh);
        uint32_t ain[32];
#pragma unroll
        for (int c = 0; c < 8; ++c) ain[c] = pack_bf2(sh[2 * c], sh[2 * c + 1]);
#pragma unroll
        for (int q = 0; q < 8; ++q) { ain[16 + 2 * q] = pack_bf2(ev[q].x, ev[q].y); ain[16 + 2 * q + 1] = pack_bf2(ev[q].z, ev[q].w); }
        wait_acc();
        float v[16];
        tm_load<16>(trow, v);
        uint32_t w[8];
        bias_act_pack<16, false>(v, Cf + C_BB2, w);
        w[0] = (w[0] & 0xFFFF0000u) | 0x3F80u;   // column 0 is the density pre-activation: its slot in every downstream input has zero WEIGHTS, and
                                               // carries the constant 1 whose dW column / row is the bias gradient of the layers that read BO / AIN
        row_store<2>(base + B_BO, r, w);
#pragma unroll
        for (int c = 0; c < 8; ++c) ain[8 + c] = w[c];
        row_store<8>(base + B_AIN, r, ain);
        ready();
      }
      // ---- 3, 4: rgb hidden 1, 2 ; d(rgb pre-activation) from the forward's colours ----------------------------------------------------
      {
        wait_acc();
        float v[64];
        tm_load<64>(trow, v);
        uint32_t w[32];
        bias_act_pack<64, true>(v, Cf + C_BR1, w);
        if (j > wg) wait_dw();   // step 11 of this warpgroup's PREVIOUS batch (dWb1 reads D, R1): waited for here, three layers later, not at its end
        row_store<8>(base + B_R1, r, w);
        ready();
      }
      {
        wait_acc();
        float v[64];
        tm_load<64>(trow, v);
        uint32_t w[32];
        bias_act_pack<64, true>(v, Cf + C_BR2, w);
        row_store<8>(base + B_R2, r, w);
        uint32_t d3[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
        d3[0] = pack_bf2(drgb[0] * st.y * (1.f - st.y), drgb[1] * st.z * (1.f - st.z));
        d3[1] = pack_bf2(drgb[2] * st.w * (1.f - st.w), 0.f);
        row_store<2>(base + B_DS, r, d3);
        ready(true);
      }
      // ---- 5, 6: dY of rgb layers 2 and 1 ---------------------------------------------------------------------------------------------
      {
        wait_acc();
        float v[64];
        tm_load<64>(trow, v);
        uint32_t w[32];
        mask_pack<64>(v, P1, 8, w);
        wait_dw();   // step 4 (dWr3: R2, DS)
        row_store<8>(base + B_D, r, w);
        ready(true);
      }
      {
        wait_acc();
        float v[64];
        tm_load<64>(trow, v);
        uint32_t w[32];
        mask_pack<64>(v, P1, 0, w);

        wait_dw();   // step 5 (dWr2 reads D)
        row_store<8>(base + B_D, r, w);
        ready(true);
      }
      // ---- 7: d(rgb input) columns 16..63 = [d dba slot, d geo15 | d emb32] --------------------------------------------------------------
      float dbo[16];
      {
        wait_acc();
        float v[48];
        tm_load<48>(trow, v);
#pragma unroll
        for (int c = 0; c < 16; ++c) dbo[c] = v[c];
        if (a.app_mode == CNB_APP_PER_CAMERA && b.d_embedding != nullptr) {
          // appearance-embedding gradient (fruit_field.py:251-258): sum over the rows of a ray before the atomics
          const int64_t ray0 = __shfl_sync(0xffffffffu, ray, 0), ray1 = __shfl_sync(0xffffffffu, ray, 31);
          const int cam0 = __shfl_sync(0xffffffffu, cam, 0), cam1 = __shfl_sync(0xffffffffu, cam, 31);
          const bool two = __all_sync(0xffffffffu, ray == ray0 || ray == ray1);
          if (two) {
            float x[32];
#pragma unroll
            for (int c = 0; c < 32; ++c) x[c] = ray == ray0 ? v[16 + c] : 0.f;
            const float s0 = transpose_reduce32(x, lane);
            if (s0 != 0.f) atomicAdd(b.d_embedding + (int64_t)cam0 * 32 + lane, s0);
            if (ray0 != ray1) {
#pragma unroll
              for (int c = 0; c < 32; ++c) x[c] = ray == ray0 ? 0.f : v[16 + c];
              const float s1 = transpose_reduce32(x, lane);
              if (s1 != 0.f) atomicAdd(b.d_embedding + (int64_t)cam1 * 32 + lane, s1);
            }
          } else if (valid) {
#pragma unroll
            for (int c = 0; c < 32; ++c) atomicAdd(b.d_embedding + (int64_t)cam * 32 + c, v[16 + c]);
          }
        }
        wait_dw();   // step 6 (dWr1 reads D, AIN)
        ready();
      }
      // ---- 8, 9: semantic hidden 1, 2 (input detached: fruit_field.py:264-266) ; d_sem through the head -----------------------------------
      {
        wait_acc();
        float v[64];
        tm_load<64>(trow, v);
        uint32_t w[32];
        bias_act_pack<64, true>(v, Cf + C_BS1, w);
        row_store<8>(base + B_R1, r, w);
        ready();
      }
      {
        wait_acc();
        float v[64];
        tm_load<64>(trow, v);
        uint32_t w[32];
        bias_act_pack<64, false>(v, Cf + C_BS2, w);

        row_store<8>(base + B_R2, r, w);
        uint32_t dh[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
        dh[0] = pack_bf2(dsem, 0.f);
        row_store<2>(base + B_DS, r, dh);
#pragma unroll
        for (int c = 0; c < 64; c += 4) {
          const float4 wh = *reinterpret_cast<const float4*>(Cf + C_WH + c);
          w[c / 2] = pack_bf2(dsem * wh.x, dsem * wh.y);
          w[c / 2 + 1] = pack_bf2(dsem * wh.z, dsem * wh.w);
        }
        row_store<8>(base + B_D, r, w);
        ready(true);
      }
      // ---- 10: dY of semantic layer 1 ; d(base output) = [d_density * trunc_exp' * selector | d geo15] -------------------------------------
      {
        wait_acc();
        float v[64];
        tm_load<64>(trow, v);
        uint32_t w[32];
        mask_pack<64>(v, P0, 8, w);
        wait_dw();   // step 9 (dWh, dWs2: R2, DS, D, R1)
        row_store<8>(base + B_D, r, w);
        uint32_t db[8];
        dbo[0] = ddens * st.x;
#pragma unroll
        for (int c = 0; c < 8; ++c) db[c] = pack_bf2(dbo[2 * c], dbo[2 * c + 1]);
        row_store<2>(base + B_DS, r, db);
        ready(true);
      }
      // ---- 11: dY of base layer 1 ; the encoded features again (X of dWb1) -------------------------------------------------------------------
      {
        wait_acc();
        float v[64];
        tm_load<64>(trow, v);
        uint32_t w[32];
        mask_pack<64>(v, P0, 0, w);
        wait_dw();   // step 10 (dWs1, dWb2: D, BO, AH, DS)
        row_store<8>(base + B_D, r, w);
        row_store<4>(base + B_R1, r, x0w);
        *reinterpret_cast<uint4*>(base + B_R1 + 4 * FB + r * 16) = make_uint4(0x3F803F80u, 0x3F803F80u, 0x3F803F80u, 0x3F803F80u);   // dWb1's bias column
        ready(true);
      }
      // ---- 12: d(encoded features), level-major [L][N][2] -------------------------------------------------------------------------------------
      {
        wait_acc();
        float v[32];
        tm_load<32>(trow, v);
        if (valid) {
#pragma unroll
          for (int l = 0; l < 16; ++l)
            if (l < a.L) reinterpret_cast<float2*>(b.d_x0)[(int64_t)l * N + i] = make_float2(v[2 * l], v[2 * l + 1]);
        }
        asm volatile("tcgen05.fence::before_thread_sync;");
        if (dbg_on) { b.dbg[48] += clock64() - te; b.dbg[53] = t_fence; b.dbg[54] = t_dbgrmw; }
      }
    }
    if (wg < nb_cta) wait_dw();   // the last batch's dWb1
  }

  // ---- one read-out + flush per CTA ----------------------------------------------------------------------------------------------------
  // every epilogue thread has seen the commit of its last step, and the issuer's commits cover all earlier MMAs of both warpgroups
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;");
  if (b.dbg && blockIdx.x == 0 && threadIdx.x == 0) b.dbg[50] = clock64() - t_start;
  const int in0 = a.in0;
  float* img = reinterpret_cast<float*>(smem + O_WG);   // gradient image, every tensor in its global element order
  // M = 64 accumulators keep row m in TMEM lane (m % 16) + 32 * (m / 16): lanes 0..15 of the warps with warp % 4 == q hold rows 16 q + lane;
  // M = 128 accumulators (the transposed GEMMs) keep row r in lane r: warp quarter q holds rows 32 q + lane.  tcgen05.ld is warp-collective
  // (.sync.aligned): all 32 lanes take part and discard what they do not own.  Twelve warps read (the warp's quarter of the lanes, a third of
  // the accumulators each); column indices are compile-time, so a value costs one shared store.
  if (nb_cta > 0) {
    const int q = warp & 3, m = 16 * q + (lane & 15), r128 = 32 * q + lane;
    const bool own = lane < 16;
    const uint32_t taddr = tmem + ((uint32_t)(32 * q) << 16);
    // the bias row of dWr3^T / dWh^T was accumulated against AIN's column 0 = SH component 0 (bf16): a constant
    const float inv_sh0 = 1.0f / __bfloat162float(__float2bfloat16_rn(0.28209479177387814f));
    auto rd = [&](auto ncols_tag, uint32_t col0, bool mine, auto put) {
      constexpr int NC = decltype(ncols_tag)::value;
#pragma unroll
      for (int c0 = 0; c0 < NC; c0 += 8) {
        uint32_t v[8];
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                     : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                     : "r"(taddr + col0 + c0));
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        if (mine) {
#pragma unroll
          for (int e = 0; e < 8; ++e) put(c0 + e, __uint_as_float(v[e]));
        }
        __syncwarp();
      }
    };
    using C8 = std::integral_constant<int, 8>; using C16 = std::integral_constant<int, 16>;
    using C40 = std::integral_constant<int, 40>; using C64 = std::integral_constant<int, 64>; using C72 = std::integral_constant<int, 72>;
    const int grp = warp >> 2;
    const bool t_own = r128 <= 64;   // transposed accumulators: rows 0..63 = the layer's inputs, row 64 = the bias
    if (grp == 0) {
      rd(C72{}, T_R2, own, [&](int k, float v) { if (k < 64) img[I_WR2 + m * 64 + k] = v; else if (k == 64) img[I_BR2 + m] = v; });
      rd(C16{}, T_R3, t_own, [&](int k, float v) { if (k < 3) { if (r128 < 64) img[I_WR3 + k * 64 + r128] = v; else img[I_BR3 + k] = v * inv_sh0; } });
      rd(C8{}, T_H, t_own, [&](int k, float v) { if (k == 0) { if (r128 < 64) img[I_WH + r128] = v; else img[I_BH] = v * inv_sh0; } });
    } else if (grp == 1) {
      rd(C64{}, T_R1, own, [&](int k, float v) { if (k == 16) img[I_BR1 + m] = v; else img[I_WR1 + m * 63 + (k < 16 ? k : k - 1)] = v; });
      rd(C16{}, T_S1, own, [&](int k, float v) { if (k == 0) img[I_BS1 + m] = v; else img[I_WS1 + m * 15 + (k - 1)] = v; });
      rd(C16{}, T_B2, t_own, [&](int k, float v) { if (r128 < 64) img[I_WB2 + k * 64 + r128] = v; else img[I_BB2 + k] = v; });
    } else if (grp == 2) {
      rd(C72{}, T_S2, own, [&](int k, float v) { if (k < 64) img[I_WS2 + m * 64 + k] = v; else if (k == 64) img[I_BS2 + m] = v; });
      rd(C40{}, T_B1, own, [&](int k, float v) { if (k < 32) { if (k < in0) img[I_WB1 + m * in0 + k] = v; } else if (k == 32) img[I_BB1 + m] = v; });
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;");
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem));
  // the image goes to this CTA's slot of the partial-gradient scratch with plain coalesced stores; k_tc5_reduce sums the slots.  (148 CTAs
  // adding 16.8 k floats each straight into the gradients is 2.5 M same-address-contended atomics: measured 84 k cycles per CTA, a third of
  // the kernel.)
  {
    float4* dst = reinterpret_cast<float4*>(b.part + (int64_t)blockIdx.x * CTX_PART_FLOATS);
    const float4* src = reinterpret_cast<const float4*>(img);
    for (int e = threadIdx.x; e < I_END / 4; e += KTHREADS) dst[e] = src[e];
  }
  if (b.dbg && blockIdx.x == 0 && threadIdx.x == 0) b.dbg[51] = clock64() - t_start;
}

// gradients += sum over the CTAs' images.  grid (ceil(I_END / 256), 4): blockIdx.y takes a quarter of the images (4 atomics per element).
__global__ void __launch_bounds__(256) k_tc5_reduce(const __grid_constant__ BwdArgs b, int nimg) {
  const int e = blockIdx.x * 256 + threadIdx.x;
  if (e >= I_END) return;
  float* g = nullptr;
  int off = 0, n = 0;
  auto seg = [&](float* p, int o, int len) { if (e >= o && e < o + len) { g = p; off = o; n = len; } };
  seg(b.dWr3, I_WR3, 192); seg(b.dbr3, I_BR3, 3);
  seg(b.dWr2, I_WR2, 4096); seg(b.dbr2, I_BR2, 64);
  seg(b.dWr1, I_WR1, 4032); seg(b.dbr1, I_BR1, 64);
  seg(b.dWh, I_WH, 64); seg(b.dbh, I_BH, 1);
  seg(b.dWs2, I_WS2, 4096); seg(b.dbs2, I_BS2, 64);
  seg(b.dWs1, I_WS1, 960); seg(b.dbs1, I_BS1, 64);
  seg(b.dWb2, I_WB2, 1024); seg(b.dbb2, I_BB2, 16);
  seg(b.dWb1, I_WB1, 64 * b.m.in0); seg(b.dbb1, I_BB1, 64);
  if (g == nullptr || n == 0) return;
  const int per = (nimg + gridDim.y - 1) / gridDim.y;
  const int c0 = blockIdx.y * per, c1 = min(nimg, c0 + per);
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  int c = c0;
  for (; c + 4 <= c1; c += 4) {
    s0 += __ldg(b.part + (int64_t)c * CTX_PART_FLOATS + e);
    s1 += __ldg(b.part + (int64_t)(c + 1) * CTX_PART_FLOATS + e);
    s2 += __ldg(b.part + (int64_t)(c + 2) * CTX_PART_FLOATS + e);
    s3 += __ldg(b.part + (int64_t)(c + 3) * CTX_PART_FLOATS + e);
  }
  for (; c < c1; ++c) s0 += __ldg(b.part + (int64_t)c * CTX_PART_FLOATS + e);
  const float s = (s0 + s1) + (s2 + s3);
  if (s != 0.f) atomicAdd(g + (e - off), s);
}

}  // namespace

int cnb_field_mixed_bwd(const cnb_field* f, const cnb_samples* s, const float* d_density, const float* d_rgb, const float* d_sem, float* ctx,
                        cudaStream_t stream) {
  BwdArgs b;
  fill_args(f, s, b.m);
  const int64_t N = s->num_rays * s->samples_per_ray;
  b.x0 = reinterpret_cast<const __half*>(ctx);
  b.stash = ctx + ctx_stash_off(N);
  b.masks = reinterpret_cast<const uint4*>(ctx + ctx_mask_off(N));
  b.part = ctx + ctx_part_off(N);
  b.d_x0 = ctx + ctx_dx0_off(N);
  b.d_density = d_density; b.d_rgb = d_rgb; b.d_sem = d_sem;
  b.dWb1 = f->base.dW[0]; b.dbb1 = f->base.db[0]; b.dWb2 = f->base.dW[1]; b.dbb2 = f->base.db[1];
  b.dWs1 = f->sem.dW[0]; b.dbs1 = f->sem.db[0]; b.dWs2 = f->sem.dW[1]; b.dbs2 = f->sem.db[1];
  b.dWh = f->sem_head.dW[0]; b.dbh = f->sem_head.db[0];
  b.dWr1 = f->rgb.dW[0]; b.dbr1 = f->rgb.db[0]; b.dWr2 = f->rgb.dW[1]; b.dbr2 = f->rgb.db[1]; b.dWr3 = f->rgb.dW[2]; b.dbr3 = f->rgb.db[2];
  b.d_embedding = f->appearance_mode == CNB_APP_PER_CAMERA ? f->d_embedding : nullptr;
  static const bool want_dbg = [] { const char* e = getenv("CNB_TC5_DEBUG"); return e != nullptr && e[0] == '1'; }();
  static long long* dbg_dev = nullptr;
  b.dbg = nullptr;
  if (want_dbg) {
    if (!dbg_dev) cudaMalloc(&dbg_dev, 64 * sizeof(long long));
    cudaMemsetAsync(dbg_dev, 0, 64 * sizeof(long long), stream);
    b.dbg = dbg_dev;
  }
  static bool configured = false;
  if (!configured) {
    if (cudaFuncSetAttribute(k_field_bwd_tc5, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_TC5) != cudaSuccess)
      return cnb_check_launch("field_bwd_tc5 attr");
    configured = true;
  }
  const int64_t nbatches = (N + ROWS - 1) / ROWS;
  int64_t blocks = nbatches < (int64_t)cnb_num_sms() ? nbatches : (int64_t)cnb_num_sms();
  if (blocks > CTX_PART_CTAS) blocks = CTX_PART_CTAS;
  k_field_bwd_tc5<<<(int)blocks, KTHREADS, SMEM_TC5, stream>>>(b);
  int rc = cnb_check_launch("field_bwd_tc5");
  if (rc) return rc;
  k_tc5_reduce<<<dim3((I_END + 255) / 256, 4), 256, 0, stream>>>(b, (int)blocks);
  if ((rc = cnb_check_launch("field_bwd_tc5 reduce"))) return rc;
  if (want_dbg) {
    long long h[64];
    cudaStreamSynchronize(stream);
    cudaMemcpy(h, dbg_dev, sizeof(h), cudaMemcpyDeviceToHost);
    fprintf(stderr, "[tc5] N=%lld  step: issuer_wait issuer_issue | epi_wait epi_work (cycles summed over CTA 0's wg0 batches)\n", (long long)N);
    for (int i = 0; i < 12; ++i) fprintf(stderr, "[tc5] %2d: %8lld %8lld | %8lld %8lld\n", i, h[i], h[12 + i], h[24 + i], h[36 + i]);
    fprintf(stderr, "[tc5] final epilogue work %lld ; CTA 0: prologue %lld, batch loop end %lld, kernel end %lld cycles\n", h[48], h[49], h[50], h[51]);
    fprintf(stderr, "[tc5] weights: loads issued at %lld, first matrix stored at %lld, all stored at %lld cycles; fence+arrive total %lld; dbg RMW total %lld\n", h[55], h[56], h[52], h[53], h[54]);
  }
  return cnb_hashgrid_bwd_level_major(&f->grid, ctx + ctx_pos_off(N), b.d_x0, N, stream);
}
