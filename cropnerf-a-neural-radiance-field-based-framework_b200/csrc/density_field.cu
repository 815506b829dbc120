// Proposal-network density, fused: position warp -> hash grid (L levels) -> MLP 2L->H->1 -> trunc_exp * selector.
// Row a7 of SURVEY.md section 8: replaces nerfstudio/fields/density_fields.py HashMLPDensityField.get_density /
// Field.density_fn as built at fruit_nerf.py:118-142 and called by the ProposalNetworkSampler (fruit_nerf.py:549).
// 70 % of all corner fetches of a training step happen here (256+96 of 400 samples per ray).
//
// One thread per sample; everything between the ray description and the density stays in registers.  The tiny
// MLP (193 parameters for H=16) is read from shared memory as warp-wide broadcasts.  Backward recomputes the
// forward, scatters the table gradient with vector reductions (red.global.add.v2.f32) and reduces the MLP
// parameter gradients per CTA through a shared-memory tile before one atomic flush per CTA.
#include <cuda_bf16.h>

#include <type_traits>

#include "cnb_common.cuh"

namespace {

constexpr int BLOCK = 128;

struct DfArgs {
  const float* table;
  float* d_table;
  int L;
  uint32_t mask, T;
  float scalings[CNB_MAX_LEVELS];
  cnb_warp warp;
  float avg;
  const float *W1, *b1, *W2, *b2;
  float *dW1, *db1, *dW2, *db2;
  int in;  // 2L
  cnb_samples sm;
  float* d_feat_out;  // optional [N, 2L]: gradient reaching the encoded features (consumed by cnb_position_grad_rays)
  float* feat_keep;       // forward, optional: encoded features written LEVEL-MAJOR [L][N] float2 (coalesced) for the backward
  const float* feat_kept; // backward, optional: features kept by the forward -> no re-gather
  int mixed;              // CNB_PREC_MIXED: MLP parameter gradients contracted with plain bf16 operands (no hi/lo split)
};

// Kernels are compiled for LMAX levels.  The fruit_nerf proposal grids (hidden 16, <= 7 levels) run kernels compiled for their
// exact level count (nl = LMAX: every level loop has a fixed trip count); the other shapes run LMAX = 8 / 16 kernels with
// nl = a.L <= LMAX, zero features past nl and zero-padded weights.
template <int LMAX>
__device__ __forceinline__ void encode(const DfArgs& a, int nl, float x, float y, float z, float (&feat)[2 * LMAX]) {
#pragma unroll
  for (int l = 0; l < LMAX; ++l) {
    if (l < nl) {
      const CnbCell c = cnb_cell(x, y, z, a.scalings[l]);
      uint32_t h[8];
      cnb_corner_rows(c, a.mask, (uint32_t)l * a.T, h);
      float f0[8], f1[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) { const float2 v = cnb_ldg2(a.table, h[k]); f0[k] = v.x; f1[k] = v.y; }
      feat[2 * l] = cnb_blend(f0, c.ox, c.oy, c.oz);
      feat[2 * l + 1] = cnb_blend(f1, c.ox, c.oy, c.oz);
    } else {
      feat[2 * l] = 0.0f;
      feat[2 * l + 1] = 0.0f;
    }
  }
}

// row stride of W1 in shared memory: 2*LMAX rounded up to whole float4s
__host__ __device__ constexpr int w1_stride(int lmax) { return (2 * lmax + 3) & ~3; }

// smem weights: W1 [H][w1_stride] (zero padded), b1 [H], W2 [H], b2 [4]
template <int LMAX, int H>
__device__ __forceinline__ void load_weights(const DfArgs& a, float* Ws) {
  constexpr int WS = w1_stride(LMAX);
  for (int e = threadIdx.x; e < H * WS; e += BLOCK) {
    const int j = e / WS, k = e - j * WS;
    Ws[e] = k < a.in ? __ldg(a.W1 + j * a.in + k) : 0.0f;
  }
  for (int j = threadIdx.x; j < H; j += BLOCK) {
    Ws[H * WS + j] = __ldg(a.b1 + j);
    Ws[H * WS + H + j] = __ldg(a.W2 + j);
  }
  if (threadIdx.x == 0) Ws[H * WS + 2 * H] = __ldg(a.b2);
}

// Row j of W1 against the 2*LMAX inputs, in ascending k: float4 reads, and a float2 tail when 2*LMAX is not a multiple of 4.
// acc + sum_k W1[j][k] * feat[k]
template <int LMAX>
__device__ __forceinline__ float w1_dot(const float* Wj, const float (&feat)[2 * LMAX], float acc) {
  constexpr int IN = 2 * LMAX;
#pragma unroll
  for (int k = 0; k + 4 <= IN; k += 4) {
    const float4 w = *reinterpret_cast<const float4*>(Wj + k);
    acc = fmaf(w.x, feat[k], acc); acc = fmaf(w.y, feat[k + 1], acc);
    acc = fmaf(w.z, feat[k + 2], acc); acc = fmaf(w.w, feat[k + 3], acc);
  }
  if (IN % 4 != 0) {
    const float2 w = *reinterpret_cast<const float2*>(Wj + IN - 2);
    acc = fmaf(w.x, feat[IN - 2], acc); acc = fmaf(w.y, feat[IN - 1], acc);
  }
  return acc;
}

// dfeat[k] += dh * W1[j][k]
template <int LMAX>
__device__ __forceinline__ void w1_axpy(const float* Wj, float dh, float (&dfeat)[2 * LMAX]) {
  constexpr int IN = 2 * LMAX;
#pragma unroll
  for (int k = 0; k + 4 <= IN; k += 4) {
    const float4 w = *reinterpret_cast<const float4*>(Wj + k);
    dfeat[k] = fmaf(dh, w.x, dfeat[k]); dfeat[k + 1] = fmaf(dh, w.y, dfeat[k + 1]);
    dfeat[k + 2] = fmaf(dh, w.z, dfeat[k + 2]); dfeat[k + 3] = fmaf(dh, w.w, dfeat[k + 3]);
  }
  if (IN % 4 != 0) {
    const float2 w = *reinterpret_cast<const float2*>(Wj + IN - 2);
    dfeat[IN - 2] = fmaf(dh, w.x, dfeat[IN - 2]); dfeat[IN - 1] = fmaf(dh, w.y, dfeat[IN - 1]);
  }
}

template <int LMAX, int H>
__device__ __forceinline__ float mlp_forward(const float* Ws, const float (&feat)[2 * LMAX], float (&hid)[H]) {
  constexpr int WS = w1_stride(LMAX);
  float out = Ws[H * WS + 2 * H];
#pragma unroll
  for (int j = 0; j < H; ++j) {
    hid[j] = fmaxf(w1_dot<LMAX>(Ws + j * WS, feat, Ws[H * WS + j]), 0.0f);
    out = fmaf(Ws[H * WS + H + j], hid[j], out);
  }
  return out;
}

// EXACT: a.L == LMAX (see encode)
template <int LMAX, int H, bool KEEP, bool EXACT>
__global__ void __launch_bounds__(BLOCK) k_density_fwd(DfArgs a, float* __restrict__ density, float* __restrict__ pos_out) {
  constexpr int INP = 2 * LMAX;
  __shared__ __align__(16) float Ws[H * w1_stride(LMAX) + 2 * H + 4];
  load_weights<LMAX, H>(a, Ws);
  __syncthreads();
  const int nl = EXACT ? LMAX : a.L;
  const int S = a.sm.samples_per_ray;
  const int64_t total = a.sm.num_rays * S;
  for (int64_t i = blockIdx.x * (int64_t)BLOCK + threadIdx.x; i < total; i += (int64_t)gridDim.x * BLOCK) {
    const int64_t r = cnb_ray_of(i, S);
    const int s = (int)(i - r * S);
    float x, y, z;
    const bool sel = cnb_sample_position(a.sm, a.warp, r, s, x, y, z);
    if (pos_out) { pos_out[3 * i] = x; pos_out[3 * i + 1] = y; pos_out[3 * i + 2] = z; }
    float feat[INP], hid[H];
    encode<LMAX>(a, nl, x, y, z, feat);
    if (KEEP) {  // compile-time: the render path keeps its 64-register forward
#pragma unroll
      for (int l = 0; l < LMAX; ++l)
        if (l < nl) reinterpret_cast<float2*>(a.feat_keep)[(int64_t)l * total + i] = make_float2(feat[2 * l], feat[2 * l + 1]);
    }
    const float out = mlp_forward<LMAX, H>(Ws, feat, hid);
    density[i] = sel ? a.avg * expf(out) : 0.0f;
  }
}

// Backward.  Per tile of BLOCK samples the per-sample factors are staged in shared memory as
//   U_s = [dh_s (H) | g_s]      V_s = [x_s (in) | 1 | h_s (H)]
// and the parameter gradients are the pair sums (dh_j,x_k) (dh_j,1) (g,h_j) (g,1).
template <int LMAX, int H>
__global__ void __launch_bounds__(BLOCK, (H <= 16 && LMAX <= 8) ? 5 : 1) k_density_bwd(DfArgs a, const float* __restrict__ d_density) {
  constexpr int INP = 2 * LMAX, WS = w1_stride(LMAX);
  constexpr int LD = BLOCK + 1;
  extern __shared__ float4 smem4[];
  float* Ws = reinterpret_cast<float*>(smem4);       // H*WS + 2H + 4
  float* U = Ws + (H * WS + 2 * H + 4);              // (H+1) x LD
  float* V = U + (H + 1) * LD;                       // (in+1+H) x LD
  const int nv = a.in + 1 + H;
  float* acc = V + nv * LD;                          // nout
  const int nout = H * a.in + 2 * H + 1;
  load_weights<LMAX, H>(a, Ws);
  for (int o = threadIdx.x; o < nout; o += BLOCK) acc[o] = 0.0f;
  __syncthreads();
  const int tid = threadIdx.x;
  const int S = a.sm.samples_per_ray;
  const int64_t total = a.sm.num_rays * S;
  const int64_t ntiles = (total + BLOCK - 1) / BLOCK;
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t i = tile * BLOCK + tid;
    float g = 0.0f;
    float feat[INP], hid[H];
    float x = 0.f, y = 0.f, z = 0.f;
    bool active = false;
    if (i < total) {
      const float dd = __ldg(d_density + i);
      if (dd != 0.0f) {
        const int64_t r = cnb_ray_of(i, S);
        const int s = (int)(i - r * S);
        const bool sel = cnb_sample_position(a.sm, a.warp, r, s, x, y, z);
        if (sel) {
          encode<LMAX>(a, a.L, x, y, z, feat);
          const float out = mlp_forward<LMAX, H>(Ws, feat, hid);
          g = dd * a.avg * cnb_trunc_exp_grad(out);
          active = (g != 0.0f);
        }
      }
    }
    float dfeat[INP];
#pragma unroll
    for (int k = 0; k < INP; ++k) dfeat[k] = 0.0f;
    if (active) {
#pragma unroll
      for (int j = 0; j < H; ++j) {
        const float dh = hid[j] > 0.0f ? g * Ws[H * WS + H + j] : 0.0f;
        U[j * LD + tid] = dh;
        V[(a.in + 1 + j) * LD + tid] = hid[j];
        w1_axpy<LMAX>(Ws + j * WS, dh, dfeat);
      }
      U[H * LD + tid] = g;
#pragma unroll
      for (int k = 0; k < INP; ++k)
        if (k < a.in) V[k * LD + tid] = feat[k];
      V[a.in * LD + tid] = 1.0f;
    } else {
      for (int j = 0; j <= H; ++j) U[j * LD + tid] = 0.0f;
      for (int k = 0; k < nv; ++k) V[k * LD + tid] = 0.0f;
    }
    if (a.d_feat_out != nullptr && i < total) {
#pragma unroll
      for (int l = 0; l < LMAX; ++l)
        if (l < a.L) reinterpret_cast<float2*>(a.d_feat_out)[i * a.L + l] = make_float2(dfeat[2 * l], dfeat[2 * l + 1]);
    }
    // table gradient: the lanes of a warp are consecutive samples of a ray -> warp-aggregated scatter (all lanes take part)
#pragma unroll
    for (int l = 0; l < LMAX; ++l) {
      if (l < a.L) {
        const float d0 = dfeat[2 * l], d1 = dfeat[2 * l + 1];
        const bool on = active && (d0 != 0.0f || d1 != 0.0f);
        CnbCell c = {};
        if (on) c = cnb_cell(x, y, z, a.scalings[l]);
        cnb_scatter_cell(a.d_table, c, a.mask, (uint32_t)l * a.T, d0, d1, on);
      }
    }
    __syncthreads();
    for (int o = tid; o < nout; o += BLOCK) {
      int u, v;
      if (o < H * a.in) { u = o / a.in; v = o - u * a.in; }
      else if (o < H * a.in + H) { u = o - H * a.in; v = a.in; }
      else if (o < H * a.in + 2 * H) { u = H; v = a.in + 1 + (o - H * a.in - H); }
      else { u = H; v = a.in; }
      const float* up = U + u * LD;
      const float* vp = V + v * LD;
      float sacc = 0.0f;
#pragma unroll 8
      for (int s = 0; s < BLOCK; ++s) sacc = fmaf(up[s], vp[s], sacc);
      acc[o] += sacc;
    }
    __syncthreads();
  }
  for (int o = tid; o < nout; o += BLOCK) {
    const float v = acc[o];
    if (v == 0.0f) continue;
    if (o < H * a.in) { if (a.dW1) atomicAdd(a.dW1 + o, v); }
    else if (o < H * a.in + H) { if (a.db1) atomicAdd(a.db1 + (o - H * a.in), v); }
    else if (o < H * a.in + 2 * H) { if (a.dW2) atomicAdd(a.dW2 + (o - H * a.in - H), v); }
    else { if (a.db2) atomicAdd(a.db2, v); }
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// Backward for the fruit_nerf proposal architecture (<= 7 levels, hidden 16): the MLP parameter gradients dW1, db1 and dW2
// are the products U^T V of the per-sample rows
//     U_s = [dh_s (16) | h_s (16)] (32 cols)        V_s = [x_s (in <= 14) | 0.. | g_s (col 14) | 1 (col 15)] (16 cols)
// contracted over SAMPLES, i.e. a GEMM whose K dimension is the 128 samples of the CTA's tile: the rows are staged in
// shared memory and contracted with mma.sync.m16n8k16 through ldmatrix.trans.  To keep fp32-level accuracy (this kernel
// also serves the exact-fp32 mode, 5e-4 gradient parity) every value is split into bf16 hi + bf16 lo and the three
// significant cross products are accumulated (relative error ~1e-5).  Each warp takes two of the tile's eight 16-sample
// k-steps and keeps its 3 output tiles in registers across the whole kernel; one cross-warp reduction + flush per CTA.
// db2 = sum_s g_s is a plain fp32 sum per thread.
constexpr int TC_SW = 40;  // staging row stride in halves (32 + 8 pad): 80-byte rows, 16-byte aligned, conflict-free

__device__ __forceinline__ void tc_ldsm_x4_t(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];\n" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void tc_mma_bf16(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// 8 floats -> 8 bf16 hi (uint4) + 8 bf16 lo (uint4)
__device__ __forceinline__ void tc_split8(const float (&v)[8], uint4& hi, uint4& lo) {
  uint32_t h[4], l[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const __nv_bfloat162 hh = __floats2bfloat162_rn(v[2 * q], v[2 * q + 1]);
    const float2 back = __bfloat1622float2(hh);
    const __nv_bfloat162 ll = __floats2bfloat162_rn(v[2 * q] - back.x, v[2 * q + 1] - back.y);
    h[q] = *reinterpret_cast<const uint32_t*>(&hh);
    l[q] = *reinterpret_cast<const uint32_t*>(&ll);
  }
  hi = make_uint4(h[0], h[1], h[2], h[3]);
  lo = make_uint4(l[0], l[1], l[2], l[3]);
}

// Run-aggregation cap of the table scatter per level: a larger cap merges longer runs into fewer reductions, and costs scan
// rounds only in the warps whose runs are that long.  Finer levels have shorter runs.  Measured on one B200 (1000 W), 4096 rays,
// cnb_density_field_bwd_kept in us, proposal0 mixed / fp32, proposal1 mixed / fp32 (tests/time_proposal_bwd.py):
// {8,8,4,2,2} 139.0 / 149.6 / 66.2 / 71.8, {16,16,8,4,4} 143.3 / 157.0 / 66.4 / 70.4, {32,32,32,32,32} 146.3 / 159.0 / 65.8 / 68.1
__device__ __forceinline__ void prop_scatter(int l, float* d_table, const CnbCell& c, uint32_t mask, uint32_t level_offset, float d0, float d1,
                                             bool on) {
  if (l < 2) cnb_scatter_cell<8>(d_table, c, mask, level_offset, d0, d1, on);
  else if (l < 3) cnb_scatter_cell<4>(d_table, c, mask, level_offset, d0, d1, on);
  else cnb_scatter_cell<2>(d_table, c, mask, level_offset, d0, d1, on);
}

// SPLIT = true: exact mode (bf16 hi + lo operands, three cross products, 42 KB of staging, 5 CTAs/SM).  SPLIT = false: mixed-precision mode --
// plain bf16 operands like the field's mixed backward (2e-3-class parameter gradients), half the staging and conversions, one product, and
// with them enough shared memory and registers for 6 CTAs/SM on this latency-bound kernel.
// Compiled for the exact level count L (a.L == L, in = 2L): the MLP recompute, dfeat and the level scatter run exact trip counts.
template <int L, bool SPLIT>
__global__ void __launch_bounds__(BLOCK, SPLIT ? 5 : 6) k_density_bwd_tc(DfArgs a, const float* __restrict__ d_density) {
  constexpr int H = 16, IN = 2 * L, WS = w1_stride(L);
  static_assert(IN <= 14, "V holds the inputs in columns 0..14, column 15 is the bias");
  extern __shared__ float4 smem4[];
  float* Ws = reinterpret_cast<float*>(smem4);                         // H*WS + 2H + 4 floats (<= 292)
  __nv_bfloat16* stg = reinterpret_cast<__nv_bfloat16*>(Ws + 296);     // Uh, Ul, Vh, Vl: 4 x [BLOCK][TC_SW]
  load_weights<L, H>(a, Ws);
  __syncthreads();
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t stg_s = (uint32_t)__cvta_generic_to_shared(stg);
  constexpr uint32_t MAT = BLOCK * TC_SW * 2;  // bytes per staged matrix
  const int S = a.sm.samples_per_ray;
  const int64_t total = a.sm.num_rays * S;
  const int64_t ntiles = (total + BLOCK - 1) / BLOCK;
  // output tiles: t0 = dh x V[0:8] (dW1), t1 = dh x V[8:16] (dW1, col 15: db1), t2 = h x V[8:16] (col 14: dW2)
  constexpr int NT = 3;
  float acc[NT][4];
#pragma unroll
  for (int q = 0; q < NT; ++q) { acc[q][0] = 0.f; acc[q][1] = 0.f; acc[q][2] = 0.f; acc[q][3] = 0.f; }
  float gsum = 0.0f;
  const int j = lane >> 3, r8 = lane & 7;
  constexpr int MATQ = BLOCK * TC_SW / 8;  // uint4 per matrix
  constexpr int VQ = SPLIT ? 2 * MATQ : MATQ;  // staged matrices: Uh, (Ul), Vh, (Vl)
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t i = tile * BLOCK + tid;
    uint4* row = reinterpret_cast<uint4*>(stg + tid * TC_SW);
    float g = 0.0f;
    uint32_t hpos = 0;  // bit jj: h_jj > 0 (ReLU open)
    float x = 0.f, y = 0.f, z = 0.f;
    bool active = false;
    uint4 hi, lo;
    float v8[8];
    if (i < total) {
      const float dd = __ldg(d_density + i);
      if (dd != 0.0f) {
        const int64_t r = cnb_ray_of(i, S);
        const int s = (int)(i - r * S);
        const bool sel = cnb_sample_position(a.sm, a.warp, r, s, x, y, z);
        if (sel) {
          float feat[IN];
          if (a.feat_kept != nullptr) {
            // the forward of this step kept the encoded features (level-major, coalesced): no second gather pass
#pragma unroll
            for (int l = 0; l < L; ++l) {
              const float2 fv = __ldg(reinterpret_cast<const float2*>(a.feat_kept) + (int64_t)l * total + i);
              feat[2 * l] = fv.x; feat[2 * l + 1] = fv.y;
            }
          } else {
            encode<L>(a, L, x, y, z, feat);
          }
          float hid[H];
          const float out = mlp_forward<L, H>(Ws, feat, hid);
          g = dd * a.avg * cnb_trunc_exp_grad(out);
          active = (g != 0.0f);
          if (active) {
            // V = [x0..x(in-1) 0.. g 1] and U[16:32] = h, staged here so that the features and activations are dead before the backward
#pragma unroll
            for (int c = 0; c < 2; ++c) {
#pragma unroll
              for (int k = 0; k < 8; ++k) v8[k] = (8 * c + k < IN) ? feat[8 * c + k] : 0.0f;
              if (c == 1) { v8[6] = g; v8[7] = 1.0f; }
              tc_split8(v8, hi, lo);
              row[VQ + c] = hi;
              if (SPLIT) row[VQ + MATQ + c] = lo;
            }
#pragma unroll
            for (int c = 0; c < 2; ++c) {
#pragma unroll
              for (int k = 0; k < 8; ++k) v8[k] = hid[8 * c + k];
              tc_split8(v8, hi, lo);
              row[2 + c] = hi;
              if (SPLIT) row[MATQ + 2 + c] = lo;
            }
#pragma unroll
            for (int jj = 0; jj < H; ++jj) hpos |= (hid[jj] > 0.0f ? 1u : 0u) << jj;
          }
        }
      }
    }
    float dfeat[IN];
#pragma unroll
    for (int k = 0; k < IN; ++k) dfeat[k] = 0.0f;
    if (active) {
      gsum += g;
      // U[0:16] = dh
#pragma unroll
      for (int c = 0; c < 2; ++c) {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const int jj = 8 * c + k;
          v8[k] = (hpos >> jj) & 1u ? g * Ws[H * WS + H + jj] : 0.0f;
          w1_axpy<L>(Ws + jj * WS, v8[k], dfeat);
        }
        tc_split8(v8, hi, lo);
        row[c] = hi;
        if (SPLIT) row[MATQ + c] = lo;
      }
    } else {
      const uint4 zq = make_uint4(0, 0, 0, 0);
#pragma unroll
      for (int m = 0; m < (SPLIT ? 2 : 1); ++m) {
#pragma unroll
        for (int c = 0; c < 4; ++c) row[m * MATQ + c] = zq;
        row[VQ + m * MATQ] = zq;
        row[VQ + m * MATQ + 1] = zq;
      }
    }
    if (a.d_feat_out != nullptr && i < total) {
#pragma unroll
      for (int l = 0; l < L; ++l) reinterpret_cast<float2*>(a.d_feat_out)[i * L + l] = make_float2(dfeat[2 * l], dfeat[2 * l + 1]);
    }
    // table gradient: the lanes of a warp are consecutive samples of a ray -> warp-aggregated scatter (all lanes take part)
#pragma unroll
    for (int l = 0; l < L; ++l) {
      const float d0 = dfeat[2 * l], d1 = dfeat[2 * l + 1];
      const bool on = active && (d0 != 0.0f || d1 != 0.0f);
      CnbCell c = {};
      if (on) c = cnb_cell(x, y, z, a.scalings[l]);
      prop_scatter(l, a.d_table, c, a.mask, (uint32_t)l * a.T, d0, d1, on);  // l is a constant of the unrolled loop
    }
    __syncthreads();
    // ---- parameter gradients: this warp contracts k-steps 2*warp, 2*warp+1 of the tile ----------------------------------------
#pragma unroll
    for (int kk = 0; kk < 2; ++kk) {
      const int ks = 2 * warp + kk;
      uint32_t A0[2][4], A1[2][4], B01[2][4];  // [hi/lo]
#pragma unroll
      for (int p = 0; p < (SPLIT ? 2 : 1); ++p) {
        const uint32_t ubase = stg_s + p * MAT, vbase = stg_s + ((SPLIT ? 2 : 1) + p) * MAT;
        const uint32_t arow = 2u * ((16 * ks + (j >> 1) * 8 + r8) * TC_SW + (j & 1) * 8);
        tc_ldsm_x4_t(A0[p], ubase + arow);
        tc_ldsm_x4_t(A1[p], ubase + arow + 2u * 16);
        const uint32_t brow = 2u * ((16 * ks + (j & 1) * 8 + r8) * TC_SW + 8 * (j >> 1));
        tc_ldsm_x4_t(B01[p], vbase + brow);
      }
#pragma unroll
      for (int c = 0; c < (SPLIT ? 3 : 1); ++c) {  // hi*hi, hi*lo, lo*hi
        const int pa = c == 2 ? 1 : 0, pb = c == 1 ? 1 : 0;
        tc_mma_bf16(acc[0], A0[pa], B01[pb][0], B01[pb][1]);
        tc_mma_bf16(acc[1], A0[pa], B01[pb][2], B01[pb][3]);
        tc_mma_bf16(acc[2], A1[pa], B01[pb][2], B01[pb][3]);
      }
    }
    __syncthreads();
  }
  // ---- cross-warp reduction + one flush per CTA -----------------------------------------------------------------------------------
  constexpr int NO = NT * 4 * 32;  // accumulator values per warp
  float* red = reinterpret_cast<float*>(stg);  // [4 warps][NT][4][32], then the 4 warps' db2 sums
#pragma unroll
  for (int q = 0; q < NT; ++q)
#pragma unroll
    for (int e = 0; e < 4; ++e) red[((warp * NT + q) * 4 + e) * 32 + lane] = acc[q][e];
#pragma unroll
  for (int m = 16; m > 0; m >>= 1) gsum += __shfl_xor_sync(0xffffffffu, gsum, m);
  if (lane == 0) red[4 * NO + warp] = gsum;
  __syncthreads();
  if (tid == 0 && a.db2) {
    const float v = red[4 * NO] + red[4 * NO + 1] + red[4 * NO + 2] + red[4 * NO + 3];
    if (v != 0.0f) atomicAdd(a.db2, v);
  }
  for (int o = tid; o < NO; o += BLOCK) {
    const float v = red[o] + red[NO + o] + red[2 * NO + o] + red[3 * NO + o];
    if (v == 0.0f) continue;
    const int q = o / 128, e = (o >> 5) & 3, ln = o & 31;
    const int rowi = (ln >> 2) + (e >> 1) * 8, col = 2 * (ln & 3) + (e & 1);  // within the 16x8 tile
    if (q == 0) { if (col < a.in && a.dW1) atomicAdd(a.dW1 + rowi * a.in + col, v); }
    else if (q == 1) {
      if (8 + col < a.in) { if (a.dW1) atomicAdd(a.dW1 + rowi * a.in + 8 + col, v); }
      else if (col == 7 && a.db1) atomicAdd(a.db1 + rowi, v);
    } else if (col == 6 && a.dW2) atomicAdd(a.dW2 + rowi, v);
  }
}

int make_args(const cnb_density_field* f, const cnb_samples* s, bool bwd, DfArgs& a) {
  CNB_REQUIRE(f && s, "density_field: null descriptor");
  const cnb_grid& g = f->grid;
  CNB_REQUIRE(g.table != nullptr, "density_field: null table");
  CNB_REQUIRE(g.num_levels >= 1 && g.num_levels <= CNB_MAX_LEVELS, "density_field: num_levels %d unsupported", g.num_levels);
  CNB_REQUIRE(g.log2_hashmap_size >= 1 && g.log2_hashmap_size <= 24, "density_field: log2_hashmap_size %d unsupported", g.log2_hashmap_size);
  const cnb_mlp& m = f->mlp;
  if (m.num_layers != 2 || m.dims[2] != 1 || m.out_activation != CNB_ACT_NONE) {
    cnb_set_error("density_field: fused kernel supports MLP 2L->H->1 only (got %d layers); compose cnb_hashgrid_* + cnb_mlp_* instead", m.num_layers);
    return CNB_ERR_UNSUPPORTED;
  }
  CNB_REQUIRE(m.dims[0] == 2 * g.num_levels, "density_field: mlp in dim %d != 2*num_levels", m.dims[0]);
  CNB_REQUIRE(m.W[0] && m.b[0] && m.W[1] && m.b[1], "density_field: null mlp weights");
  CNB_REQUIRE(s->samples_per_ray >= 1 && s->num_rays >= 0, "density_field: bad sample counts");
  // an empty batch has no arrays: torch hands out null pointers for zero-size tensors
  CNB_REQUIRE(s->num_rays == 0 || (s->origins && s->directions && s->starts && s->ends), "density_field: null sample arrays");
  CNB_REQUIRE(!bwd || g.d_table != nullptr, "density_field_bwd: d_table required");
  if (bwd)
    for (int i = 0; i < g.num_levels; ++i) CNB_REQUIRE(g.scalings[i] < 65535.0f, "density_field_bwd: level resolution %g too large for the aggregated scatter", g.scalings[i]);
  a.table = g.table; a.d_table = g.d_table; a.L = g.num_levels;
  a.T = 1u << g.log2_hashmap_size; a.mask = a.T - 1u;
  for (int i = 0; i < CNB_MAX_LEVELS; ++i) a.scalings[i] = g.scalings[i];
  a.warp = f->warp; a.avg = f->average_init_density;
  a.W1 = m.W[0]; a.b1 = m.b[0]; a.W2 = m.W[1]; a.b2 = m.b[1];
  a.dW1 = m.dW[0]; a.db1 = m.db[0]; a.dW2 = m.dW[1]; a.db2 = m.db[1];
  a.in = m.dims[0];
  a.sm = *s;
  a.d_feat_out = nullptr;
  a.feat_keep = nullptr;
  a.feat_kept = nullptr;
  a.mixed = f->precision == CNB_PREC_MIXED;
  return CNB_OK;
}

// f(std::integral_constant<int, L>{}) for the level counts L = 1..7 that run exact-level kernels (hidden 16)
template <class F>
int with_exact_levels(int L, F&& f) {
  switch (L) {
    case 1: return f(std::integral_constant<int, 1>{});
    case 2: return f(std::integral_constant<int, 2>{});
    case 3: return f(std::integral_constant<int, 3>{});
    case 4: return f(std::integral_constant<int, 4>{});
    case 5: return f(std::integral_constant<int, 5>{});
    case 6: return f(std::integral_constant<int, 6>{});
    case 7: return f(std::integral_constant<int, 7>{});
  }
  cnb_set_error("density_field: no exact-level kernel for %d levels (1..7)", L);
  return CNB_ERR_UNSUPPORTED;
}

template <int LMAX, int H, bool EXACT>
int launch_fwd_k(const DfArgs& a, float* density, float* pos_out, cudaStream_t st) {
  const int64_t total = a.sm.num_rays * a.sm.samples_per_ray;
  int64_t blocks = (total + BLOCK - 1) / BLOCK;
  const int64_t cap = (int64_t)cnb_num_sms() * 16;
  if (blocks > cap) blocks = cap;
  if (a.feat_keep != nullptr) k_density_fwd<LMAX, H, true, EXACT><<<(int)blocks, BLOCK, 0, st>>>(a, density, pos_out);
  else k_density_fwd<LMAX, H, false, EXACT><<<(int)blocks, BLOCK, 0, st>>>(a, density, pos_out);
  return cnb_check_launch("density_field_fwd");
}

template <int LMAX, int H>
int launch_fwd(const DfArgs& a, float* density, float* pos_out, cudaStream_t st) {
  if constexpr (LMAX == 8 && H == 16) {
    if (a.L <= 7) return with_exact_levels(a.L, [&](auto l) { return launch_fwd_k<decltype(l)::value, H, true>(a, density, pos_out, st); });
  }
  return launch_fwd_k<LMAX, H, false>(a, density, pos_out, st);
}

template <int L>
int launch_bwd_tc(const DfArgs& a, const float* d_density, cudaStream_t st) {
  const int64_t total = a.sm.num_rays * a.sm.samples_per_ray;
  const bool split = !a.mixed;
  const size_t smem = sizeof(float) * 296 + (size_t)(split ? 4 : 2) * BLOCK * TC_SW * 2;
  int64_t blocks = (total + BLOCK - 1) / BLOCK;
  const int64_t cap = (int64_t)cnb_num_sms() * (split ? 5 : 6);
  if (blocks > cap) blocks = cap;
  if (split) k_density_bwd_tc<L, true><<<(int)blocks, BLOCK, smem, st>>>(a, d_density);
  else k_density_bwd_tc<L, false><<<(int)blocks, BLOCK, smem, st>>>(a, d_density);
  return cnb_check_launch("density_field_bwd");
}

template <int LMAX, int H>
int launch_bwd(const DfArgs& a, const float* d_density, cudaStream_t st) {
  if constexpr (LMAX == 8 && H == 16) {
    if (a.L <= 7) return with_exact_levels(a.L, [&](auto l) { return launch_bwd_tc<decltype(l)::value>(a, d_density, st); });
  }
  const int64_t total = a.sm.num_rays * a.sm.samples_per_ray;
  const int nv = a.in + 1 + H, nout = H * a.in + 2 * H + 1;
  const size_t smem = sizeof(float) * ((H * w1_stride(LMAX) + 2 * H + 4) + (size_t)(H + 1 + nv) * (BLOCK + 1) + nout + 4);
  static size_t configured = 0;
  if (smem > configured) {
    if (cudaFuncSetAttribute(k_density_bwd<LMAX, H>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
      return cnb_check_launch("density_field_bwd attr");
    configured = smem;
  }
  int64_t blocks = (total + BLOCK - 1) / BLOCK;
  const int64_t cap = (int64_t)cnb_num_sms() * 8;  // 8 resident CTAs/SM (smem 25 KB, 76 regs): the gathers and reds need the warps
  if (blocks > cap) blocks = cap;
  k_density_bwd<LMAX, H><<<(int)blocks, BLOCK, smem, st>>>(a, d_density);
  return cnb_check_launch("density_field_bwd");
}

#define DISPATCH(FN, ...)                                                                   \
  do {                                                                                      \
    const int H = f->mlp.dims[1];                                                           \
    const bool small = a.L <= 8;                                                            \
    if (small && H == 16) return FN<8, 16>(__VA_ARGS__);                                    \
    if (small && H == 32) return FN<8, 32>(__VA_ARGS__);                                    \
    if (small && H == 64) return FN<8, 64>(__VA_ARGS__);                                    \
    if (!small && H == 16) return FN<16, 16>(__VA_ARGS__);                                  \
    if (!small && H == 32) return FN<16, 32>(__VA_ARGS__);                                  \
    if (!small && H == 64) return FN<16, 64>(__VA_ARGS__);                                  \
    cnb_set_error("density_field: hidden width %d not compiled (16/32/64)", H);             \
    return CNB_ERR_UNSUPPORTED;                                                             \
  } while (0)

}  // namespace

static int density_fwd_impl(const cnb_density_field* f, const cnb_samples* s, float* density, float* positions_out, float* feat_keep, cnb_stream_t stream) {
  DfArgs a;
  int rc = make_args(f, s, false, a);
  if (rc) return rc;
  if (a.sm.num_rays == 0) return CNB_OK;
  CNB_REQUIRE(density != nullptr, "density_field_fwd: null output");
  a.feat_keep = feat_keep;
  DISPATCH(launch_fwd, a, density, positions_out, stream);
}

extern "C" int cnb_density_field_fwd(const cnb_density_field* f, const cnb_samples* s, float* density, float* positions_out, cnb_stream_t stream) {
  return density_fwd_impl(f, s, density, positions_out, nullptr, stream);
}

extern "C" int cnb_density_field_fwd_keep(const cnb_density_field* f, const cnb_samples* s, float* density, float* features_keep, cnb_stream_t stream) {
  CNB_REQUIRE(features_keep != nullptr, "density_field_fwd_keep: null feature buffer");
  return density_fwd_impl(f, s, density, nullptr, features_keep, stream);
}

extern "C" int cnb_density_field_kept_supported(const cnb_density_field* f) {
  // the backward that consumes kept features is the tensor-core kernel of the fruit_nerf proposal architecture
  return f && f->grid.num_levels <= 7 && f->mlp.num_layers == 2 && f->mlp.dims[1] == 16 && f->mlp.dims[2] == 1;
}

static int density_bwd_impl(const cnb_density_field* f, const cnb_samples* s, const float* d_density, float* d_feat_out, const float* feat_kept,
                            cnb_stream_t stream) {
  DfArgs a;
  int rc = make_args(f, s, true, a);
  if (rc) return rc;
  if (a.sm.num_rays == 0) return CNB_OK;
  CNB_REQUIRE(d_density != nullptr, "density_field_bwd: null d_density");
  CNB_REQUIRE(feat_kept == nullptr || cnb_density_field_kept_supported(f), "density_field_bwd_kept: architecture outside the kept-feature kernel (<= 7 levels, hidden 16)");
  a.d_feat_out = d_feat_out;
  a.feat_kept = feat_kept;
  DISPATCH(launch_bwd, a, d_density, stream);
}

extern "C" int cnb_density_field_bwd_kept(const cnb_density_field* f, const cnb_samples* s, const float* d_density, const float* features_kept,
                                          cnb_stream_t stream) {
  CNB_REQUIRE(features_kept != nullptr, "density_field_bwd_kept: null feature buffer");
  return density_bwd_impl(f, s, d_density, nullptr, features_kept, stream);
}

extern "C" int cnb_density_field_bwd(const cnb_density_field* f, const cnb_samples* s, const float* d_density, cnb_stream_t stream) {
  return density_bwd_impl(f, s, d_density, nullptr, nullptr, stream);
}

extern "C" int cnb_density_field_bwd_rays(const cnb_density_field* f, const cnb_samples* s, const float* d_density, float* scratch, float* d_origins,
                                          float* d_directions, cnb_stream_t stream) {
  CNB_REQUIRE(scratch && d_origins && d_directions, "density_field_bwd_rays: null scratch / ray gradients");
  int rc = density_bwd_impl(f, s, d_density, scratch, nullptr, stream);
  if (rc) return rc;
  return cnb_position_grad_rays(&f->grid, &f->warp, s, scratch, d_origins, d_directions, stream);
}
