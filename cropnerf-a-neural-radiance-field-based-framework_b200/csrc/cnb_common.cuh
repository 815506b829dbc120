// Shared device helpers for the cropnerf_b200 kernels (sm_100a).
//
// Bit-exactness notes (SURVEY.md App. B): everything that decides a hash index is written with explicit
// round-to-nearest intrinsics (__fmul_rn/__fadd_rn/__fdiv_rn) so nvcc cannot contract it into FMAs; the
// torch reference evaluates each elementwise op as a separately rounded fp32 operation.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/cropnerf_b200.h"

#define CNB_HASH_P1 2654435761u
#define CNB_HASH_P2 805459861u

void cnb_set_error(const char* fmt, ...);
int cnb_check_launch(const char* what);

#define CNB_REQUIRE(cond, ...)      \
  do {                              \
    if (!(cond)) {                  \
      cnb_set_error(__VA_ARGS__);   \
      return CNB_ERR_ARG;           \
    }                               \
  } while (0)

static inline int cnb_num_sms() {
  static int sms = 0;
  if (sms == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0)
      sms = 148;
  }
  return sms;
}

// ---------------------------------------------------------------------------------------------------------
// positions
// ---------------------------------------------------------------------------------------------------------

// Frustums.get_positions (nerfstudio rays.py): o + d * (start + end) / 2, each op rounded separately.
__device__ __forceinline__ float cnb_axis_position(float o, float d, float start, float end) {
  return __fadd_rn(o, __fmul_rn(__fmul_rn(d, __fadd_rn(start, end)), 0.5f));
}

// fruit_field.py:171-180: contraction / aabb normalisation, strict (0,1) selector, masked positions -> 0.
// Returns the selector.
__device__ __forceinline__ bool cnb_warp_position(const cnb_warp& w, float& x, float& y, float& z) {
  if (w.mode == CNB_WARP_CONTRACT_LINF) {
    // SceneContraction(order=inf): where(mag < 1, x, (2 - 1/mag) * (x / mag))
    float mag = fmaxf(fabsf(x), fmaxf(fabsf(y), fabsf(z)));
    if (!(mag < 1.0f)) {
      float s = __fsub_rn(2.0f, __fdiv_rn(1.0f, mag));
      x = __fmul_rn(s, __fdiv_rn(x, mag));
      y = __fmul_rn(s, __fdiv_rn(y, mag));
      z = __fmul_rn(s, __fdiv_rn(z, mag));
    }
    x = __fmul_rn(__fadd_rn(x, 2.0f), 0.25f);
    y = __fmul_rn(__fadd_rn(y, 2.0f), 0.25f);
    z = __fmul_rn(__fadd_rn(z, 2.0f), 0.25f);
  } else {
    x = __fdiv_rn(__fsub_rn(x, w.aabb_min[0]), __fsub_rn(w.aabb_max[0], w.aabb_min[0]));
    y = __fdiv_rn(__fsub_rn(y, w.aabb_min[1]), __fsub_rn(w.aabb_max[1], w.aabb_min[1]));
    z = __fdiv_rn(__fsub_rn(z, w.aabb_min[2]), __fsub_rn(w.aabb_max[2], w.aabb_min[2]));
  }
  bool sel = (x > 0.0f) && (x < 1.0f) && (y > 0.0f) && (y < 1.0f) && (z > 0.0f) && (z < 1.0f);
  if (!sel) { x = 0.0f; y = 0.0f; z = 0.0f; }
  return sel;
}

// flat sample index -> ray index: a 32-bit division whenever the index fits (a 64-bit one is an ~50-instruction subroutine per thread)
__device__ __forceinline__ int64_t cnb_ray_of(int64_t i, int S) {
  if (i <= 0x7fffffffLL) return (int64_t)((uint32_t)i / (uint32_t)S);
  return i / S;
}

// normalised + masked position of sample i (= r*S + s) of a cnb_samples description
__device__ __forceinline__ bool cnb_sample_position(const cnb_samples& sm, const cnb_warp& w, int64_t r, int32_t s,
                                                    float& x, float& y, float& z) {
  const float st = __ldg(sm.starts + r * sm.row_stride + s);
  const float en = __ldg(sm.ends + r * sm.row_stride + s);
  x = cnb_axis_position(__ldg(sm.origins + 3 * r + 0), __ldg(sm.directions + 3 * r + 0), st, en);
  y = cnb_axis_position(__ldg(sm.origins + 3 * r + 1), __ldg(sm.directions + 3 * r + 1), st, en);
  z = cnb_axis_position(__ldg(sm.origins + 3 * r + 2), __ldg(sm.directions + 3 * r + 2), st, en);
  return cnb_warp_position(w, x, y, z);
}

// ---------------------------------------------------------------------------------------------------------
// hash grid (nerfstudio encodings.py HashEncoding.pytorch_fwd / hash_fn)
// ---------------------------------------------------------------------------------------------------------

struct CnbCell {
  uint32_t cx, cy, cz, fx, fy, fz;  // ceil / floor integer coordinates (>= 0)
  float ox, oy, oz;                 // scaled - floor
};

__device__ __forceinline__ CnbCell cnb_cell(float x, float y, float z, float scale) {
  CnbCell c;
  const float sx = __fmul_rn(x, scale), sy = __fmul_rn(y, scale), sz = __fmul_rn(z, scale);
  const float flx = floorf(sx), fly = floorf(sy), flz = floorf(sz);
  c.cx = (uint32_t)(int32_t)ceilf(sx); c.cy = (uint32_t)(int32_t)ceilf(sy); c.cz = (uint32_t)(int32_t)ceilf(sz);
  c.fx = (uint32_t)(int32_t)flx; c.fy = (uint32_t)(int32_t)fly; c.fz = (uint32_t)(int32_t)flz;
  c.ox = __fsub_rn(sx, flx); c.oy = __fsub_rn(sy, fly); c.oz = __fsub_rn(sz, flz);
  return c;
}

// int64 (x*1 ^ y*2654435761 ^ z*805459861) % 2^T of the reference == uint32 wrap-around arithmetic for
// non-negative coordinates and power-of-two tables (SURVEY.md App. A.1, verified there on 1.6 M triples).
__device__ __forceinline__ uint32_t cnb_hash(uint32_t x, uint32_t y, uint32_t z, uint32_t mask) {
  return (x ^ (y * CNB_HASH_P1) ^ (z * CNB_HASH_P2)) & mask;
}

// the 8 corner rows in the reference's h0..h7 order: ccc cfc ffc fcc ccf cff fff fcf
__device__ __forceinline__ void cnb_corner_rows(const CnbCell& c, uint32_t mask, uint32_t level_offset, uint32_t (&h)[8]) {
  const uint32_t xc = c.cx, xf = c.fx;
  const uint32_t yc = c.cy * CNB_HASH_P1, yf = c.fy * CNB_HASH_P1;
  const uint32_t zc = c.cz * CNB_HASH_P2, zf = c.fz * CNB_HASH_P2;
  h[0] = ((xc ^ yc ^ zc) & mask) + level_offset;
  h[1] = ((xc ^ yf ^ zc) & mask) + level_offset;
  h[2] = ((xf ^ yf ^ zc) & mask) + level_offset;
  h[3] = ((xf ^ yc ^ zc) & mask) + level_offset;
  h[4] = ((xc ^ yc ^ zf) & mask) + level_offset;
  h[5] = ((xc ^ yf ^ zf) & mask) + level_offset;
  h[6] = ((xf ^ yf ^ zf) & mask) + level_offset;
  h[7] = ((xf ^ yc ^ zf) & mask) + level_offset;
}

// trilinear blend in the reference's exact operation order (separately rounded ops)
__device__ __forceinline__ float cnb_blend(const float (&f)[8], float ox, float oy, float oz) {
  const float mx = __fsub_rn(1.0f, ox), my = __fsub_rn(1.0f, oy), mz = __fsub_rn(1.0f, oz);
  const float f03 = __fadd_rn(__fmul_rn(f[0], ox), __fmul_rn(f[3], mx));
  const float f12 = __fadd_rn(__fmul_rn(f[1], ox), __fmul_rn(f[2], mx));
  const float f56 = __fadd_rn(__fmul_rn(f[5], ox), __fmul_rn(f[6], mx));
  const float f47 = __fadd_rn(__fmul_rn(f[4], ox), __fmul_rn(f[7], mx));
  const float f0312 = __fadd_rn(__fmul_rn(f03, oy), __fmul_rn(f12, my));
  const float f4756 = __fadd_rn(__fmul_rn(f47, oy), __fmul_rn(f56, my));
  return __fadd_rn(__fmul_rn(f0312, oz), __fmul_rn(f4756, mz));
}

// corner weights matching cnb_blend (d out / d f[i])
__device__ __forceinline__ void cnb_corner_weights(float ox, float oy, float oz, float (&w)[8]) {
  const float mx = 1.0f - ox, my = 1.0f - oy, mz = 1.0f - oz;
  w[0] = ox * oy * oz;  w[3] = mx * oy * oz;
  w[1] = ox * my * oz;  w[2] = mx * my * oz;
  w[4] = ox * oy * mz;  w[7] = mx * oy * mz;
  w[5] = ox * my * mz;  w[6] = mx * my * mz;
}

__device__ __forceinline__ float2 cnb_ldg2(const float* table, uint32_t row) {
  return __ldg(reinterpret_cast<const float2*>(table) + row);
}

// fp16 copy of a table (one __half2 per row): the row widened to fp32 exactly, so a blend of these values is the fp32 blend of a table holding
// table.half().float()
__device__ __forceinline__ float2 cnb_ldg2(const __half2* table, uint32_t row) { return __half22float2(__ldg(table + row)); }

// The 8 corner rows of a cell.  The hash prime of x is 1, so the ceil-x / floor-x rows of a corner pair differ only in
// bit 0 whenever floor(x) is even: those pairs -- (0,3) (1,2) (5,6) (4,7) in the reference's corner order -- are fetched
// with ONE 16-byte load.  The gathers are bound by the L1TEX data pipe (one wavefront per distinct sector per request),
// so where the lanes of a request hit unrelated sectors (fine levels of the 16-level field grid) this removes up to a
// quarter of the wavefronts.  Measured: field forward -5 %; proposal forward +20 % (its lanes are consecutive samples
// that already share sectors, so the divergent second path only adds requests) -- used by the field kernel only.
// Values are bit-identical to eight 8-byte loads.
__device__ __forceinline__ void cnb_gather8(const float* __restrict__ table, const CnbCell& c, const uint32_t (&h)[8], float2 (&v)[8]) {
  if (c.cx == c.fx + 1u && (c.fx & 1u) == 0u) {
    const int pc[4] = {0, 1, 5, 4}, pf[4] = {3, 2, 6, 7};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float4 w = __ldg(reinterpret_cast<const float4*>(table) + (h[pf[q]] >> 1));
      const bool f_even = (h[pf[q]] & 1u) == 0u;
      v[pf[q]] = f_even ? make_float2(w.x, w.y) : make_float2(w.z, w.w);
      v[pc[q]] = f_even ? make_float2(w.z, w.w) : make_float2(w.x, w.y);
    }
  } else {
#pragma unroll
    for (int k = 0; k < 8; ++k) v[k] = cnb_ldg2(table, h[k]);
  }
}

// cnb_gather8 on an fp16 copy of the table: the x-neighbour pair of a corner (adjacent rows when floor(x) is even) is ONE 8-byte load.
__device__ __forceinline__ void cnb_gather8(const __half2* __restrict__ table, const CnbCell& c, const uint32_t (&h)[8], float2 (&v)[8]) {
  if (c.cx == c.fx + 1u && (c.fx & 1u) == 0u) {
    const int pc[4] = {0, 1, 5, 4}, pf[4] = {3, 2, 6, 7};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const uint2 w = __ldg(reinterpret_cast<const uint2*>(table) + (h[pf[q]] >> 1));
      const float2 lo = __half22float2(*reinterpret_cast<const __half2*>(&w.x)), hi = __half22float2(*reinterpret_cast<const __half2*>(&w.y));
      const bool f_even = (h[pf[q]] & 1u) == 0u;
      v[pf[q]] = f_even ? lo : hi;
      v[pc[q]] = f_even ? hi : lo;
    }
  } else {
#pragma unroll
    for (int k = 0; k < 8; ++k) v[k] = cnb_ldg2(table, h[k]);
  }
}

// vector reduction into the gradient table: one red.global.add.v2.f32 (sm_90+) per corner
__device__ __forceinline__ void cnb_red2(float* table, uint32_t row, float a, float b) {
  asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(reinterpret_cast<float2*>(table) + row), "f"(a), "f"(b) : "memory");
}

__device__ __forceinline__ void cnb_red4(float* table, uint32_t even_row, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(reinterpret_cast<float2*>(table) + even_row), "f"(a), "f"(b), "f"(c), "f"(d)
               : "memory");
}

// Gradient scatter of one (sample, level) with WARP AGGREGATION.  Must be called by all 32 lanes (inactive lanes pass
// active = false).  Lanes are consecutive samples of a ray, so samples that fall into the same grid cell form runs of
// consecutive lanes; a run (capped at CAP lanes) is summed with a segmented warp scan and only its last lane issues the
// reductions.  The scan stops after the rounds the warp's longest run needs: a round of offset off >= that length adds
// nothing on any lane, so the sums are those of the full log2(CAP) rounds, bit for bit, and a large cap costs shuffles
// only in the warps whose runs are long.  The two x-neighbours of a corner pair (hash prime of x is 1, SURVEY.md
// section 7) are adjacent table rows whenever floor(x) is even: those go out as ONE 16-byte red.global.add.v4.f32.
// Requires integer cell coordinates < 65536 (scalings < 65535).
template <int CAP = 8>
__device__ __forceinline__ void cnb_scatter_cell(float* d_table, const CnbCell& c, uint32_t mask, uint32_t level_offset, float d0, float d1,
                                                 bool active) {
  const unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  if (!active) { d0 = 0.0f; d1 = 0.0f; }
  // cell identity: floor coordinates + which coordinates are exact integers (ceil == floor)
  const uint32_t k0 = active ? (c.fx | (c.fy << 16)) : FULL;
  const uint32_t k1 = active ? (c.fz | ((c.cx - c.fx) << 16) | ((c.cy - c.fy) << 17) | ((c.cz - c.fz) << 18)) : (uint32_t)lane;
  const uint32_t p0 = __shfl_up_sync(FULL, k0, 1), p1 = __shfl_up_sync(FULL, k1, 1);
  const bool head = (lane & (CAP - 1)) == 0 || k0 != p0 || k1 != p1;
  const uint32_t heads = __ballot_sync(FULL, head);
  float w[8];
  cnb_corner_weights(c.ox, c.oy, c.oz, w);
  float v0[8], v1[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) { v0[k] = w[k] * d0; v1[k] = w[k] * d1; }
  // lane 0 is always a head, so every lane has a run start; depth + 1 is the warp's longest run (warp-uniform)
  const int start = 31 - __clz(heads & (FULL >> (31 - lane)));
  const int depth = (int)__reduce_max_sync(FULL, (unsigned)(lane - start));
#pragma unroll
  for (int off = 1; off < CAP; off <<= 1) {
    if (off > depth) break;
    const bool take = lane - off >= start;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float t0 = __shfl_up_sync(FULL, v0[k], off), t1 = __shfl_up_sync(FULL, v1[k], off);
      if (take) { v0[k] += t0; v1[k] += t1; }
    }
  }
  const bool tail = lane == 31 || ((heads >> (lane + 1)) & 1u);
  if (!tail || !active) return;
  uint32_t h[8];
  cnb_corner_rows(c, mask, level_offset, h);
  if (c.cx == c.fx + 1u && (c.fx & 1u) == 0u) {
    // pairs (ceil-x, floor-x) of the reference's corner order: (0,3) (1,2) (5,6) (4,7)
    const int pc[4] = {0, 1, 5, 4}, pf[4] = {3, 2, 6, 7};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int kc = pc[q], kf = pf[q];
      if (v0[kc] == 0.0f && v1[kc] == 0.0f && v0[kf] == 0.0f && v1[kf] == 0.0f) continue;
      if ((h[kf] & 1u) == 0u) cnb_red4(d_table, h[kf], v0[kf], v1[kf], v0[kc], v1[kc]);
      else cnb_red4(d_table, h[kc], v0[kc], v1[kc], v0[kf], v1[kf]);
    }
  } else {
#pragma unroll
    for (int k = 0; k < 8; ++k)
      if (v0[k] != 0.0f || v1[k] != 0.0f) cnb_red2(d_table, h[k], v0[k], v1[k]);
  }
}

// trunc_exp (nerfstudio activations.py): exp forward, g*exp(clamp(x,-15,15)) backward
__device__ __forceinline__ float cnb_trunc_exp_grad(float x) { return expf(fminf(fmaxf(x, -15.0f), 15.0f)); }

__device__ __forceinline__ float cnb_nan_to_num(float v) {
  if (isnan(v)) return 0.0f;
  if (isinf(v)) return v > 0 ? 3.4028234663852886e38f : -3.4028234663852886e38f;
  return v;
}

// spacing functions (nerfstudio ray_samplers.py UniformLinDispPiecewiseSampler / UniformSampler)
__device__ __forceinline__ float cnb_spacing_fn(int kind, float x) {
  if (kind == CNB_SPACING_LINDISP_PIECEWISE) return x < 1.0f ? __fmul_rn(x, 0.5f) : __fsub_rn(1.0f, __fdiv_rn(1.0f, __fmul_rn(2.0f, x)));
  return x;
}
__device__ __forceinline__ float cnb_spacing_inv(int kind, float x) {
  if (kind == CNB_SPACING_LINDISP_PIECEWISE) return x < 0.5f ? __fmul_rn(2.0f, x) : __fdiv_rn(1.0f, __fsub_rn(2.0f, __fmul_rn(2.0f, x)));
  return x;
}
// spacing_to_euclidean_fn(x) = inv(x * s_far + (1 - x) * s_near)
__device__ __forceinline__ float cnb_spacing_to_euclid(int kind, float x, float s_near, float s_far) {
  return cnb_spacing_inv(kind, __fadd_rn(__fmul_rn(x, s_far), __fmul_rn(__fsub_rn(1.0f, x), s_near)));
}
