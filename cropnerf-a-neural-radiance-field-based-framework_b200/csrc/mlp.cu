// Generic fp32 nn.Linear stack, forward and backward (rows a3/a4 of SURVEY.md section 8).
// Replaces nerfstudio/field_components/mlp.py MLP (torch path; ctor calls fruit_field.py:133-141,146-154,
// 159-167) and FieldHead (components/field_heads.py:29-40).  This is the exact-fp32 path (1e-4 parity mode);
// the mixed-precision hot path fuses the same layers on tensor cores in field_mixed.cu.
//
// The layers run on tensor cores as 3xTF32.  Every fp32 operand is split into a tf32 "hi" part and a tf32 "lo"
// residual (x = hi + lo up to 2^-22 relative) and each product is accumulated as hi*hi + lo*hi + hi*lo on
// mma.sync.m16n8k8.tf32 with fp32 accumulators: ~2^-21 relative error per product (the dropped lo*lo term), i.e. fp32-class
// results -- the tests' 1e-5 / 2e-5 bounds against the oracle are unchanged -- at tensor-core rate instead of FFMA rate.
// (bf16 hi+lo, which the mixed kernels' fragment layout would allow, keeps 16 mantissa bits: not enough for the 1e-4 mode.)
//
// Forward: warp-autonomous.  A warp owns 16 rows at a time in a private pair of shared-memory activation tiles and chains the
// layers through them (C fragment -> bias / activation -> tile -> A fragment of the next layer); no block barrier in the loop.
// Backward: CTA tile of 128 rows.  dW = dOut^T In is a contraction over the tile's 128 SAMPLES (m = output feature, n = input
// feature, k = sample) with its output tiles dealt round-robin to the 8 warps and accumulated in a per-CTA shared-memory copy of the
// gradients (fixed ownership, no atomics until the flush); the bias gradient is one more n-tile against a column of ones;
// dIn = dOut W is row-parallel again (warp = 16 rows).
#include "cnb_common.cuh"

namespace {

__device__ __forceinline__ int up16_dev(int v) { return (v + 15) & ~15; }

__device__ __forceinline__ float apply_act(float v, int act) {
  if (act == CNB_ACT_RELU) return fmaxf(v, 0.0f);
  if (act == CNB_ACT_SIGMOID) return 1.0f / (1.0f + expf(-v));
  return v;
}

namespace tc {

constexpr int WARPS = 8;
constexpr int THREADS = WARPS * 32;
constexpr int ROWS = 128;     // backward CTA tile
constexpr int RS = 68;        // activation tile row stride (floats): conflict-free A-fragment reads (bank = 4 g + t)

struct Args {
  int nl;
  int dims[CNB_MAX_LAYERS + 1];
  int in8[CNB_MAX_LAYERS], out8[CNB_MAX_LAYERS], ws[CNB_MAX_LAYERS];  // padded dims, weight row stride (in8 + 4: bank = 4 g' + t)
  int wo[CNB_MAX_LAYERS], bo[CNB_MAX_LAYERS];
  int total_w;
  int act;
  const float* W[CNB_MAX_LAYERS];
  const float* b[CNB_MAX_LAYERS];
  float* dW[CNB_MAX_LAYERS];
  float* db[CNB_MAX_LAYERS];
};

inline int up8(int v) { return (v + 7) & ~7; }
inline int up16(int v) { return (v + 15) & ~15; }

int make_args(const cnb_mlp* m, Args& a) {
  CNB_REQUIRE(m != nullptr, "mlp: null descriptor");
  CNB_REQUIRE(m->num_layers >= 1 && m->num_layers <= CNB_MAX_LAYERS, "mlp: num_layers %d outside 1..%d", m->num_layers, CNB_MAX_LAYERS);
  a.nl = m->num_layers;
  a.act = m->out_activation;
  for (int l = 0; l <= a.nl; ++l) {
    CNB_REQUIRE(m->dims[l] >= 1 && m->dims[l] <= CNB_MAX_WIDTH, "mlp: dims[%d]=%d outside 1..%d", l, m->dims[l], CNB_MAX_WIDTH);
    a.dims[l] = m->dims[l];
  }
  int off = 0;
  for (int l = 0; l < CNB_MAX_LAYERS; ++l) {
    if (l < a.nl) {
      CNB_REQUIRE(m->W[l] && m->b[l], "mlp: null W/b for layer %d", l);
      a.in8[l] = up8(a.dims[l]); a.out8[l] = up8(a.dims[l + 1]); a.ws[l] = a.in8[l] + 4;
      a.wo[l] = off; off += up16(a.dims[l + 1]) * a.ws[l];   // rows padded to 16: the dW contraction uses m16 tiles
      a.bo[l] = off; off += up16(a.dims[l + 1]);
      a.W[l] = m->W[l]; a.b[l] = m->b[l]; a.dW[l] = m->dW[l]; a.db[l] = m->db[l];
    } else {
      a.in8[l] = a.out8[l] = a.ws[l] = a.wo[l] = a.bo[l] = 0;
      a.W[l] = a.b[l] = nullptr; a.dW[l] = a.db[l] = nullptr;
    }
  }
  a.total_w = (off + 3) & ~3;
  return CNB_OK;
}

// x = hi + lo with hi a tf32 number (10 mantissa bits) rounded to nearest: two integer ops instead of cvt.rna.tf32.f32 (a conversion-unit
// instruction at a quarter of the ALU rate, and there are four of them per three MMAs in the inner loops).  lo = x - hi is exact in fp32
// and is handed to the tensor core as it is: the hardware reads the upper 19 bits of a tf32 operand, i.e. truncates lo's 13-bit tail,
// an error of 2^-11 |lo| <= 2^-22 |x|.
__device__ __forceinline__ void split(float x, uint32_t& hi, uint32_t& lo) {
  hi = (__float_as_uint(x) + 0x1000u) & 0xffffe000u;
  lo = __float_as_uint(x - __uint_as_float(hi));
}
__device__ __forceinline__ void mma_tf32(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// c += A B with both operands given as fp32 values (a: 4 fragment registers, b: 2)
__device__ __forceinline__ void mma3(float (&c)[4], const uint32_t (&ah)[4], const uint32_t (&al)[4], float b0, float b1) {
  uint32_t bh0, bl0, bh1, bl1;
  split(b0, bh0, bl0);
  split(b1, bh1, bl1);
  mma_tf32(c, al, bh0, bh1);
  mma_tf32(c, ah, bl0, bl1);
  mma_tf32(c, ah, bh0, bh1);
}

// the same with B already split (the backward keeps tf32 hi / lo images of the weights in shared memory: two extra loads instead of six ALU
// instructions per product triple)
__device__ __forceinline__ void mma3_presplit(float (&c)[4], const uint32_t (&ah)[4], const uint32_t (&al)[4], uint32_t bh0, uint32_t bh1, uint32_t bl0,
                                              uint32_t bl1) {
  mma_tf32(c, al, bh0, bh1);
  mma_tf32(c, ah, bl0, bl1);
  mma_tf32(c, ah, bh0, bh1);
}

__device__ __forceinline__ void load_weights(const Args& m, float* Ws) {
  for (int e = threadIdx.x; e < m.total_w; e += blockDim.x) Ws[e] = 0.0f;
  __syncthreads();
  for (int l = 0; l < m.nl; ++l) {
    const int in = m.dims[l], out = m.dims[l + 1];
    for (int e = threadIdx.x; e < out * in; e += blockDim.x) {
      const int j = e / in, k = e - j * in;
      Ws[m.wo[l] + j * m.ws[l] + k] = __ldg(m.W[l] + e);
    }
    for (int j = threadIdx.x; j < out; j += blockDim.x) Ws[m.bo[l] + j] = __ldg(m.b[l] + j);
  }
}

// global rows -> activation tile [rows][RS], zero padded to in8 columns / `rows` rows.  Eight loads are in flight per thread before the first
// store: with one element per loop iteration every iteration was an exposed memory round trip (1 CTA / SM in the backward, nothing to hide it).
template <int NTHR>
__device__ __forceinline__ void stage_rows(float* __restrict__ dst, const float* __restrict__ src, int64_t sstride, int rows, int cnt, int in, int in8, int tid) {
  const int total = rows * in8;
  for (int e0 = tid; e0 < total; e0 += 8 * NTHR) {
    float v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int e = e0 + u * NTHR;
      const int r = e / in8, k = e - r * in8;
      v[u] = (e < total && r < cnt && k < in) ? __ldg(src + (int64_t)r * sstride + k) : 0.0f;
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int e = e0 + u * NTHR;
      if (e < total) { const int r = e / in8, k = e - r * in8; dst[r * RS + k] = v[u]; }
    }
  }
}

// rows [16 rows of `cur`, stride RS] x W^T + b -> act -> `nxt`; K = in8, N = out8.  All 32 lanes of one warp.
__device__ __forceinline__ void dense16(const float* __restrict__ cur, const float* __restrict__ W, const float* __restrict__ b, int in8, int out8, int ws,
                                        int act, float* __restrict__ nxt, int g, int t) {
  const int NT = out8 >> 3;
  float acc[8][4];
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
    if (nt < NT) {
      const float2 bb = *reinterpret_cast<const float2*>(b + 8 * nt + 2 * t);
      acc[nt][0] = bb.x; acc[nt][1] = bb.y; acc[nt][2] = bb.x; acc[nt][3] = bb.y;
    }
  }
  for (int k0 = 0; k0 < in8; k0 += 8) {
    uint32_t ah[4], al[4];
    split(cur[g * RS + k0 + t], ah[0], al[0]);
    split(cur[(g + 8) * RS + k0 + t], ah[1], al[1]);
    split(cur[g * RS + k0 + t + 4], ah[2], al[2]);
    split(cur[(g + 8) * RS + k0 + t + 4], ah[3], al[3]);
#pragma unroll
    for (int nt = 0; nt < 8; ++nt)
      if (nt < NT) {
        const float* wr = W + (8 * nt + g) * ws + k0 + t;
        mma3(acc[nt], ah, al, wr[0], wr[4]);
      }
  }
#pragma unroll
  for (int nt = 0; nt < 8; ++nt)
    if (nt < NT) {
      *reinterpret_cast<float2*>(nxt + g * RS + 8 * nt + 2 * t) = make_float2(apply_act(acc[nt][0], act), apply_act(acc[nt][1], act));
      *reinterpret_cast<float2*>(nxt + (g + 8) * RS + 8 * nt + 2 * t) = make_float2(apply_act(acc[nt][2], act), apply_act(acc[nt][3], act));
    }
}

__global__ void __launch_bounds__(THREADS, 2) k_mlp_fwd_tc(const __grid_constant__ Args m, const float* __restrict__ x, int64_t x_stride, int64_t n,
                                                           float* __restrict__ y, float* __restrict__ hidden) {
  extern __shared__ float4 smem4[];
  float* Ws = reinterpret_cast<float*>(smem4);
  load_weights(m, Ws);
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  float* tA = Ws + m.total_w + warp * 2 * 16 * RS;
  float* tB = tA + 16 * RS;
  const int64_t ntiles = (n + 15) >> 4;
  const int in0 = m.dims[0], in80 = m.in8[0];
  for (int64_t tile = (int64_t)blockIdx.x * WARPS + warp; tile < ntiles; tile += (int64_t)gridDim.x * WARPS) {
    const int64_t n0 = tile * 16;
    const int cnt = (int)min((int64_t)16, n - n0);
    stage_rows<32>(tA, x + n0 * x_stride, x_stride, 16, cnt, in0, in80, lane);
    __syncwarp();
    float* cur = tA;
    float* nxt = tB;
    int64_t hoff = 0;
    for (int l = 0; l < m.nl; ++l) {
      const bool last = (l == m.nl - 1);
      dense16(cur, Ws + m.wo[l], Ws + m.bo[l], m.in8[l], m.out8[l], m.ws[l], last ? m.act : CNB_ACT_RELU, nxt, g, t);
      __syncwarp();
      if (!last && hidden != nullptr) {
        const int w = m.dims[l + 1];
        float* dst = hidden + hoff + n0 * w;
        for (int e = lane; e < cnt * w; e += 32) {
          const int r = e / w, k = e - r * w;
          dst[e] = nxt[r * RS + k];
        }
        hoff += n * (int64_t)w;
      }
      float* sw = cur; cur = nxt; nxt = sw;
    }
    const int out = m.dims[m.nl];
    for (int e = lane; e < cnt * out; e += 32) {
      const int r = e / out, k = e - r * out;
      y[n0 * out + e] = cur[r * RS + k];
    }
    __syncwarp();
  }
}

// PRESPLIT: tf32 hi / lo images of the weights in shared memory (3 x total_w floats; every fruit_nerf MLP fits), else split on the fly
template <bool PRESPLIT>
__global__ void __launch_bounds__(THREADS, 1) k_mlp_bwd_tc(const __grid_constant__ Args m, const float* __restrict__ x, int64_t x_stride,
                                                           const float* __restrict__ hidden, const float* __restrict__ y, const float* __restrict__ dy,
                                                           int64_t n, float* __restrict__ dx, int64_t dx_stride) {
  extern __shared__ float4 smem4[];
  float* Ws = reinterpret_cast<float*>(smem4);     // after the prologue: the tf32 hi parts of the weights
  float* dWs = Ws + m.total_w;
  float* Wlo = dWs + m.total_w;                    // their lo parts (x - hi)
  float* tIn = Wlo + (PRESPLIT ? m.total_w : 0);
  float* tD = tIn + ROWS * RS;
  float* tN = tD + ROWS * RS;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  load_weights(m, Ws);
  for (int e = tid; e < m.total_w; e += THREADS) dWs[e] = 0.0f;
  __syncthreads();
  if (PRESPLIT) {
    for (int e = tid; e < m.total_w; e += THREADS) {
      uint32_t hi, lo;
      split(Ws[e], hi, lo);
      Ws[e] = __uint_as_float(hi);
      Wlo[e] = __uint_as_float(lo);
    }
    __syncthreads();
  }
  const int64_t ntiles = (n + ROWS - 1) / ROWS;
  auto layer_input = [&](int l, int64_t row0, const float*& src, int64_t& sstride) {
    if (l == 0) { src = x + row0 * x_stride; sstride = x_stride; }
    else {
      int64_t hoff = 0;
      for (int q = 0; q < l - 1; ++q) hoff += n * (int64_t)m.dims[q + 1];
      src = hidden + hoff + row0 * m.dims[l]; sstride = m.dims[l];
    }
  };
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t n0 = tile * ROWS;
    const int cnt = (int)min((int64_t)ROWS, n - n0);
    {
      const int out = m.dims[m.nl], oc = up16_dev(out);
      const int total = ROWS * oc;
      for (int e0 = tid; e0 < total; e0 += 4 * THREADS) {
        float v[4], yy[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int e = e0 + u * THREADS;
          const int r = e / oc, j = e - r * oc;
          const bool ok = e < total && r < cnt && j < out;
          v[u] = ok ? __ldg(dy + (n0 + r) * out + j) : 0.0f;
          yy[u] = (ok && m.act != CNB_ACT_NONE) ? __ldg(y + (n0 + r) * out + j) : 1.0f;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int e = e0 + u * THREADS;
          if (e >= total) continue;
          const int r = e / oc, j = e - r * oc;
          float w = v[u];
          if (m.act == CNB_ACT_SIGMOID) w *= yy[u] * (1.0f - yy[u]);
          else if (m.act == CNB_ACT_RELU) { if (!(yy[u] > 0.0f)) w = 0.0f; }
          tD[r * RS + j] = w;
        }
      }
    }
    for (int l = m.nl - 1; l >= 0; --l) {
      const int in = m.dims[l], in8 = m.in8[l], out16 = up16_dev(m.dims[l + 1]), ws = m.ws[l];
      {
        // (requesting the NEXT step's tile into 32 registers per thread before the MMAs and committing it after them was measured: 1.62 vs 1.55 ms
        // for the field backward stage -- the loads are already batched below, and 159 registers cost more than the overlap gains)
        const float* src;
        int64_t sstride;
        layer_input(l, n0, src, sstride);
        stage_rows<THREADS>(tIn, src, sstride, ROWS, cnt, in, in8, tid);
      }
      __syncthreads();
      // (a) dW[j][k] += sum_s dOut[s][j] In[s][k]; tiles (m-tile of 16 output features) x (n-tile of 8 inputs, + 1 bias tile).  A warp owns one
      // m-tile and a contiguous share of its n-tiles: the A fragments (dOut) are split into tf32 hi / lo ONCE per k step and reused over the
      // share (they were re-split for every (m, n) tile pair: 6 -> 2.8 splits per product triple)
      {
        const int MT = out16 >> 4, NTT = (in8 >> 3) + 1;
        const int WPM = WARPS / MT > 0 ? WARPS / MT : 1;          // warps per m-tile (MT <= 4: widths <= 64)
        const int per = (NTT + WPM - 1) / WPM;                    // <= 5 n-tiles per warp
        const int mi = warp % MT, part = warp / MT;
        const int nj0 = part * per, njn = min(NTT, nj0 + per) - nj0;
        if (part < WPM && njn > 0) {
          float c[5][4];
#pragma unroll
          for (int q = 0; q < 5; ++q) { c[q][0] = 0.f; c[q][1] = 0.f; c[q][2] = 0.f; c[q][3] = 0.f; }
          const float* ap = tD + 16 * mi + g;
          const float* bp = tIn + 8 * nj0 + g;
          const float one = (g == 0) ? 1.0f : 0.0f;
          for (int k0 = 0; k0 < ROWS; k0 += 8) {
            uint32_t ah[4], al[4];
            split(ap[(k0 + t) * RS], ah[0], al[0]);
            split(ap[(k0 + t) * RS + 8], ah[1], al[1]);
            split(ap[(k0 + t + 4) * RS], ah[2], al[2]);
            split(ap[(k0 + t + 4) * RS + 8], ah[3], al[3]);
#pragma unroll
            for (int q = 0; q < 5; ++q)
              if (q < njn) {
                if (nj0 + q == NTT - 1) mma3(c[q], ah, al, one, one);
                else mma3(c[q], ah, al, bp[(k0 + t) * RS + 8 * q], bp[(k0 + t + 4) * RS + 8 * q]);
              }
          }
#pragma unroll
          for (int q = 0; q < 5; ++q)
            if (q < njn) {
              const int nj = nj0 + q;
              if (nj == NTT - 1) {
                if (t == 0) { dWs[m.bo[l] + 16 * mi + g] += c[q][0]; dWs[m.bo[l] + 16 * mi + g + 8] += c[q][2]; }
              } else {
                float* dst = dWs + m.wo[l] + (16 * mi + g) * ws + 8 * nj + 2 * t;
                dst[0] += c[q][0]; dst[1] += c[q][1];
                dst[8 * ws] += c[q][2]; dst[8 * ws + 1] += c[q][3];
              }
            }
        }
      }
      // (b) dIn = dOut W (rows 16 warp .. +15), masked by the ReLU of the producing layer
      if (l > 0 || dx != nullptr) {
        const int NT = in8 >> 3, out8 = m.out8[l];
        const float* dr = tD + 16 * warp * RS;
        const float* W = Ws + m.wo[l];
        const float* WL = Wlo + m.wo[l];
        float acc[8][4];
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) { acc[nt][0] = 0.f; acc[nt][1] = 0.f; acc[nt][2] = 0.f; acc[nt][3] = 0.f; }
        for (int k0 = 0; k0 < out8; k0 += 8) {
          uint32_t ah[4], al[4];
          split(dr[g * RS + k0 + t], ah[0], al[0]);
          split(dr[(g + 8) * RS + k0 + t], ah[1], al[1]);
          split(dr[g * RS + k0 + t + 4], ah[2], al[2]);
          split(dr[(g + 8) * RS + k0 + t + 4], ah[3], al[3]);
#pragma unroll
          for (int nt = 0; nt < 8; ++nt)
            if (nt < NT) {
              const int i0 = (k0 + t) * ws + 8 * nt + g, i1 = (k0 + t + 4) * ws + 8 * nt + g;
              if (PRESPLIT) mma3_presplit(acc[nt], ah, al, __float_as_uint(W[i0]), __float_as_uint(W[i1]), __float_as_uint(WL[i0]), __float_as_uint(WL[i1]));
              else mma3(acc[nt], ah, al, W[i0], W[i1]);
            }
        }
        const float* hin = tIn + 16 * warp * RS;
        float* dn = tN + 16 * warp * RS;
#pragma unroll
        for (int nt = 0; nt < 8; ++nt)
          if (nt < NT) {
            float v0 = acc[nt][0], v1 = acc[nt][1], v2 = acc[nt][2], v3 = acc[nt][3];
            if (l > 0) {
              const float2 h0 = *reinterpret_cast<const float2*>(hin + g * RS + 8 * nt + 2 * t);
              const float2 h1 = *reinterpret_cast<const float2*>(hin + (g + 8) * RS + 8 * nt + 2 * t);
              if (!(h0.x > 0.f)) v0 = 0.f;
              if (!(h0.y > 0.f)) v1 = 0.f;
              if (!(h1.x > 0.f)) v2 = 0.f;
              if (!(h1.y > 0.f)) v3 = 0.f;
            }
            *reinterpret_cast<float2*>(dn + g * RS + 8 * nt + 2 * t) = make_float2(v0, v1);
            *reinterpret_cast<float2*>(dn + (g + 8) * RS + 8 * nt + 2 * t) = make_float2(v2, v3);
          }
        // the next layer's dW contraction reads columns up to up16(in): clear the pad columns of this warp's rows
        const int c16 = up16_dev(in);
        for (int e = lane; e < 16 * (c16 - in8); e += 32) {
          const int r = e / (c16 - in8), k = in8 + e - r * (c16 - in8);
          dn[r * RS + k] = 0.0f;
        }
      }
      __syncthreads();
      float* sw = tD; tD = tN; tN = sw;
    }
    if (dx != nullptr) {
      const int in0 = m.dims[0];
      for (int e = tid; e < cnt * in0; e += THREADS) {
        const int r = e / in0, k = e - r * in0;
        dx[(n0 + r) * dx_stride + k] = tD[r * RS + k];
      }
    }
    __syncthreads();
  }
  for (int l = 0; l < m.nl; ++l) {
    const int in = m.dims[l], out = m.dims[l + 1];
    if (m.dW[l])
      for (int e = tid; e < out * in; e += THREADS) {
        const int j = e / in, k = e - j * in;
        const float v = dWs[m.wo[l] + j * m.ws[l] + k];
        if (v != 0.0f) atomicAdd(m.dW[l] + e, v);
      }
    if (m.db[l])
      for (int j = tid; j < out; j += THREADS) {
        const float v = dWs[m.bo[l] + j];
        if (v != 0.0f) atomicAdd(m.db[l] + j, v);
      }
  }
}

}  // namespace tc

}  // namespace

// mlp_wide.cu: layer-by-layer path for MLPs with a dimension above CNB_MAX_WIDTH
bool cnb_mlp_is_wide(const cnb_mlp* m);
int cnb_mlp_wide_fwd(const cnb_mlp* m, const float* x, int64_t x_stride, int64_t n, float* y, float* hidden, cudaStream_t stream);
int cnb_mlp_wide_bwd(const cnb_mlp* m, const float* x, int64_t x_stride, const float* hidden, const float* y, const float* dy, int64_t n, float* dx,
                     int64_t dx_stride, cudaStream_t stream);
bool cnb_mlp_is_lin1(const cnb_mlp* m);   // Linear(in -> 1): the semantic head
int cnb_mlp_lin1_fwd(const cnb_mlp* m, const float* x, int64_t x_stride, int64_t n, float* y, cudaStream_t stream);
int cnb_mlp_lin1_bwd(const cnb_mlp* m, const float* x, int64_t x_stride, const float* y, const float* dy, int64_t n, float* dx, int64_t dx_stride,
                     cudaStream_t stream);

extern "C" int64_t cnb_mlp_hidden_floats(const cnb_mlp* m) {
  if (!m) return 0;
  int64_t s = 0;
  for (int l = 1; l < m->num_layers; ++l) s += m->dims[l];
  return s;
}

extern "C" int cnb_mlp_fwd(const cnb_mlp* m, const float* x, int64_t x_stride, int64_t n, float* y, float* hidden, cnb_stream_t stream) {
  if (cnb_mlp_is_lin1(m) || cnb_mlp_is_wide(m)) {
    CNB_REQUIRE(n >= 0 && (n == 0 || (x && y)), "mlp_fwd: null x/y");
    CNB_REQUIRE(x_stride >= m->dims[0], "mlp_fwd: x_stride %lld < in dim %d", (long long)x_stride, m->dims[0]);
    if (n == 0) return CNB_OK;
    return cnb_mlp_is_lin1(m) ? cnb_mlp_lin1_fwd(m, x, x_stride, n, y, stream) : cnb_mlp_wide_fwd(m, x, x_stride, n, y, hidden, stream);
  }
  tc::Args a;
  int rc = tc::make_args(m, a);
  if (rc) return rc;
  CNB_REQUIRE(n >= 0 && (n == 0 || (x && y)), "mlp_fwd: null x/y");
  CNB_REQUIRE(x_stride >= a.dims[0], "mlp_fwd: x_stride %lld < in dim %d", (long long)x_stride, a.dims[0]);
  if (n == 0) return CNB_OK;
  const size_t smem = sizeof(float) * ((size_t)a.total_w + (size_t)tc::WARPS * 2 * 16 * tc::RS);
  static size_t configured = 0;
  if (smem > configured) {
    if (cudaFuncSetAttribute(tc::k_mlp_fwd_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return cnb_check_launch("mlp_fwd_tc attr");
    configured = smem;
  }
  const int64_t nt16 = (n + 15) / 16;
  const int64_t want = (nt16 + tc::WARPS - 1) / tc::WARPS;
  const int grid = (int)min(want, (int64_t)cnb_num_sms() * 2);
  tc::k_mlp_fwd_tc<<<grid, tc::THREADS, smem, stream>>>(a, x, x_stride, n, y, hidden);
  return cnb_check_launch("mlp_fwd_tc");
}

extern "C" int cnb_mlp_bwd(const cnb_mlp* m, const float* x, int64_t x_stride, const float* hidden, const float* y, const float* dy, int64_t n,
                           float* dx, int64_t dx_stride, cnb_stream_t stream) {
  if (cnb_mlp_is_lin1(m)) {
    CNB_REQUIRE(n >= 0 && (n == 0 || (x && dy)), "mlp_bwd: null x/dy");
    CNB_REQUIRE(m->out_activation == CNB_ACT_NONE || y != nullptr, "mlp_bwd: forward output required for the output activation");
    CNB_REQUIRE(dx == nullptr || dx_stride >= m->dims[0], "mlp_bwd: dx_stride too small");
    return n == 0 ? CNB_OK : cnb_mlp_lin1_bwd(m, x, x_stride, y, dy, n, dx, dx_stride, stream);
  }
  if (cnb_mlp_is_wide(m)) {
    CNB_REQUIRE(n >= 0 && (n == 0 || (x && dy)), "mlp_bwd: null x/dy");
    CNB_REQUIRE(m->num_layers == 1 || hidden != nullptr, "mlp_bwd: hidden activations required for %d layers", m->num_layers);
    CNB_REQUIRE(m->out_activation == CNB_ACT_NONE || y != nullptr, "mlp_bwd: forward output required for the output activation");
    CNB_REQUIRE(dx == nullptr || dx_stride >= m->dims[0], "mlp_bwd: dx_stride too small");
    for (int l = 0; l < m->num_layers; ++l) CNB_REQUIRE(m->W[l] != nullptr, "mlp_bwd: null W for layer %d", l);
    return n == 0 ? CNB_OK : cnb_mlp_wide_bwd(m, x, x_stride, hidden, y, dy, n, dx, dx_stride, stream);
  }
  tc::Args a;
  int rc = tc::make_args(m, a);
  if (rc) return rc;
  CNB_REQUIRE(n >= 0 && (n == 0 || (x && dy)), "mlp_bwd: null x/dy");
  CNB_REQUIRE(a.nl == 1 || hidden != nullptr, "mlp_bwd: hidden activations required for %d layers", a.nl);
  CNB_REQUIRE(a.act == CNB_ACT_NONE || y != nullptr, "mlp_bwd: forward output required for the output activation");
  CNB_REQUIRE(dx == nullptr || dx_stride >= a.dims[0], "mlp_bwd: dx_stride too small");
  if (n == 0) return CNB_OK;
  const size_t tiles = 3 * (size_t)tc::ROWS * tc::RS;
  const bool presplit = sizeof(float) * (3 * (size_t)a.total_w + tiles) <= 232448;   // W hi, dW, W lo + three activation tiles
  const size_t smem = sizeof(float) * ((presplit ? 3 : 2) * (size_t)a.total_w + tiles);
  static size_t configured[2] = {0, 0};
  if (smem > configured[presplit]) {
    const cudaError_t e = presplit ? cudaFuncSetAttribute(tc::k_mlp_bwd_tc<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
                                   : cudaFuncSetAttribute(tc::k_mlp_bwd_tc<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return cnb_check_launch("mlp_bwd_tc attr");
    configured[presplit] = smem;
  }
  const int64_t nt = (n + tc::ROWS - 1) / tc::ROWS;
  const int grid = (int)min(nt, (int64_t)cnb_num_sms());
  if (presplit) tc::k_mlp_bwd_tc<true><<<grid, tc::THREADS, smem, stream>>>(a, x, x_stride, hidden, y, dy, n, dx, dx_stride);
  else tc::k_mlp_bwd_tc<false><<<grid, tc::THREADS, smem, stream>>>(a, x, x_stride, hidden, y, dy, n, dx, dx_stride);
  return cnb_check_launch("mlp_bwd_tc");
}
