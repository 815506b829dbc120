// Multiresolution hash-grid encoding, forward and backward (row a2 of SURVEY.md section 8).
// Replaces nerfstudio/field_components/encodings.py HashEncoding.pytorch_fwd + its autograd
// (constructed at fruit_field.py:125-132 and, through HashMLPDensityField, fruit_nerf.py:124-141).
//
// One thread per (sample, level): 8 independent 8-byte gathers in flight per thread, coalesced 8-byte
// stores of the [n, 2L] feature rows.  HBM/L2-bound: 8 corners * 8 B per (sample, level).
#include <type_traits>

#include "cnb_common.cuh"

namespace {

// Row = float: the fp32 table (two floats per row); Row = __half2: its fp16 copy (cnb_table_to_half), same layout otherwise
template <typename Row>
struct GridArgsT {
  const Row* table;
  float* d_table;
  int32_t L;
  uint32_t mask;
  uint32_t T;
  float scalings[CNB_MAX_LEVELS];
};
using GridArgs = GridArgsT<float>;

template <typename Row = float>
GridArgsT<Row> make_args(const cnb_grid* g, const Row* table = nullptr) {
  GridArgsT<Row> a;
  a.table = table;
  if constexpr (std::is_same<Row, float>::value) a.table = g->table;
  a.d_table = g->d_table;
  a.L = g->num_levels;
  a.T = 1u << g->log2_hashmap_size;
  a.mask = a.T - 1u;
  for (int i = 0; i < CNB_MAX_LEVELS; ++i) a.scalings[i] = g->scalings[i];
  return a;
}

// Forward: a warp owns 32 CONSECUTIVE samples of one level, so one load instruction touches few distinct 128-byte lines at
// the coarse / middle levels (the gathers are bound by the L1TEX t-stage: one wavefront per distinct line per request).
// The fp16 rows are gathered with cnb_gather8 (x-neighbour pairs as one 8-byte load); the fp32 rows keep eight 8-byte loads.
template <typename Row>
__global__ void __launch_bounds__(256) k_hashgrid_fwd(const __grid_constant__ GridArgsT<Row> g, const float* __restrict__ pos, int64_t n, float* __restrict__ out,
                                                       int32_t* __restrict__ indices) {
  const int lane = threadIdx.x & 31;
  const int64_t nblk = (n + 31) >> 5;
  const int64_t nwork = nblk * g.L;
  const int64_t wstride = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t w = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5); w < nwork; w += wstride) {
    const int64_t sb = w / g.L;
    const int l = (int)(w - sb * g.L);
    const int64_t s = sb * 32 + lane;
    if (s >= n) continue;
    const int64_t i = s * g.L + l;
    const float x = __ldg(pos + 3 * s), y = __ldg(pos + 3 * s + 1), z = __ldg(pos + 3 * s + 2);
    const CnbCell c = cnb_cell(x, y, z, g.scalings[l]);
    uint32_t h[8];
    cnb_corner_rows(c, g.mask, (uint32_t)l * g.T, h);
    float2 v[8];
    if constexpr (std::is_same<Row, float>::value) {
#pragma unroll
      for (int k = 0; k < 8; ++k) v[k] = cnb_ldg2(g.table, h[k]);
    } else {
      cnb_gather8(g.table, c, h, v);
    }
    float f0[8], f1[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) { f0[k] = v[k].x; f1[k] = v[k].y; }
    float2 r;
    r.x = cnb_blend(f0, c.ox, c.oy, c.oz);
    r.y = cnb_blend(f1, c.ox, c.oy, c.oz);
    reinterpret_cast<float2*>(out)[i] = r;
    if (indices) {
      int4* dst = reinterpret_cast<int4*>(indices + i * 8);
      dst[0] = make_int4((int)h[0], (int)h[1], (int)h[2], (int)h[3]);
      dst[1] = make_int4((int)h[4], (int)h[5], (int)h[6], (int)h[7]);
    }
  }
}

// Backward: a warp owns 32 CONSECUTIVE samples of one level (samples are ray-major, so neighbouring lanes are
// neighbouring samples of a ray and often share a cell): cnb_scatter_cell aggregates those runs before the reductions.
// LM = d_out is level-major [L][n][2] (what the fused field backward writes: a warp's 32 loads are one 256-byte run
// instead of 32 sectors of a [n, 2L] row-major matrix).
template <bool LM>
__global__ void __launch_bounds__(256) k_hashgrid_bwd(const __grid_constant__ GridArgs g, const float* __restrict__ pos, const float* __restrict__ d_out, int64_t n) {
  const int lane = threadIdx.x & 31;
  const int64_t nblk = (n + 31) >> 5;
  const int64_t nwork = nblk * g.L;
  const int64_t wstride = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t w = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5); w < nwork; w += wstride) {
    const int64_t sb = w / g.L;
    const int l = (int)(w - sb * g.L);
    const int64_t s = sb * 32 + lane;
    bool active = s < n;
    float2 d = make_float2(0.f, 0.f);
    if (active) {
      d = __ldg(reinterpret_cast<const float2*>(d_out) + (LM ? (int64_t)l * n + s : s * g.L + l));
      active = d.x != 0.0f || d.y != 0.0f;  // zero gradients add nothing (masked samples, App. B-3)
    }
    CnbCell c = {};
    if (active) c = cnb_cell(__ldg(pos + 3 * s), __ldg(pos + 3 * s + 1), __ldg(pos + 3 * s + 2), g.scalings[l]);
    cnb_scatter_cell(g.d_table, c, g.mask, (uint32_t)l * g.T, d.x, d.y, active);
  }
}

// Row a17 (camera optimizer, fruit_nerf.py:114-116,547): gradient of the loss with respect to the RAYS.  Given the gradient
// d_feat [N, 2L] that reaches a grid's encoded features, one thread per sample
//   * re-derives the sample's world position p = o + d (s+e)/2 and its normalised grid position (cnb_sample_position),
//   * differentiates the trilinear blend of every level w.r.t. the offsets (offset = x*scale - floor(x*scale), so
//     d offset / d x = scale; floor/ceil carry no gradient, exactly as torch autograd sees HashEncoding.pytorch_fwd),
//   * applies the selector mask, the (c+2)/4 or AABB normalisation and the Jacobian of SceneContraction(order=inf),
//   * reduces dL/dp over the ray (d_origins += dL/dp, d_directions += (s+e)/2 * dL/dp): warp shuffle when the 32 lanes
//     share the ray, atomics otherwise.
template <bool LM, typename Row = float>  // LM: d_feat is level-major [L][total][2]; Row: the rows the forward gathered
__global__ void __launch_bounds__(128) k_position_grad_rays(const __grid_constant__ GridArgsT<Row> g, cnb_warp wp, cnb_samples sm, const float* __restrict__ d_feat,
                                                            float* __restrict__ d_origins, float* __restrict__ d_directions) {
  const int S = sm.samples_per_ray;
  const int64_t total = sm.num_rays * S;
  const int64_t nround = (total + 127) / 128 * 128;
  const int lane = threadIdx.x & 31;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < nround; i += (int64_t)gridDim.x * blockDim.x) {
    const bool in = i < total;
    const int64_t ii = in ? i : total - 1;
    const int64_t r = cnb_ray_of(ii, S);
    const int s = (int)(ii - r * S);
    float gx = 0.f, gy = 0.f, gz = 0.f, tt = 0.f;
    if (in) {
      const float st = __ldg(sm.starts + r * sm.row_stride + s), en = __ldg(sm.ends + r * sm.row_stride + s);
      tt = 0.5f * (st + en);
      const float ox = __ldg(sm.origins + 3 * r), oy = __ldg(sm.origins + 3 * r + 1), oz = __ldg(sm.origins + 3 * r + 2);
      const float dx = __ldg(sm.directions + 3 * r), dy = __ldg(sm.directions + 3 * r + 1), dz = __ldg(sm.directions + 3 * r + 2);
      const float px = cnb_axis_position(ox, dx, st, en), py = cnb_axis_position(oy, dy, st, en), pz = cnb_axis_position(oz, dz, st, en);
      float x = px, y = py, z = pz;
      const bool sel = cnb_warp_position(wp, x, y, z);
      if (sel) {
        float ax = 0.f, ay = 0.f, az = 0.f;  // dL / d(normalised position)
        for (int l = 0; l < g.L; ++l) {
          const float2 d = __ldg(reinterpret_cast<const float2*>(d_feat) + (LM ? (int64_t)l * total + i : i * g.L + l));
          if (d.x == 0.0f && d.y == 0.0f) continue;
          const float scale = g.scalings[l];
          const CnbCell c = cnb_cell(x, y, z, scale);
          uint32_t h[8];
          cnb_corner_rows(c, g.mask, (uint32_t)l * g.T, h);
          float2 v[8];
#pragma unroll
          for (int k = 0; k < 8; ++k) v[k] = cnb_ldg2(g.table, h[k]);
          const float mx = 1.f - c.ox, my = 1.f - c.oy, mz = 1.f - c.oz;
          float u[8];  // corner values weighted by the feature gradients
#pragma unroll
          for (int k = 0; k < 8; ++k) u[k] = d.x * v[k].x + d.y * v[k].y;
          const float f03 = u[0] * c.ox + u[3] * mx, f12 = u[1] * c.ox + u[2] * mx, f56 = u[5] * c.ox + u[6] * mx, f47 = u[4] * c.ox + u[7] * mx;
          const float f0312 = f03 * c.oy + f12 * my, f4756 = f47 * c.oy + f56 * my;
          const float dox = ((u[0] - u[3]) * c.oy + (u[1] - u[2]) * my) * c.oz + ((u[4] - u[7]) * c.oy + (u[5] - u[6]) * my) * mz;
          const float doy = (f03 - f12) * c.oz + (f47 - f56) * mz;
          const float doz = f0312 - f4756;
          ax = fmaf(scale, dox, ax); ay = fmaf(scale, doy, ay); az = fmaf(scale, doz, az);
        }
        if (wp.mode == CNB_WARP_CONTRACT_LINF) {
          ax *= 0.25f; ay *= 0.25f; az *= 0.25f;
          const float apx = fabsf(px), apy = fabsf(py), apz = fabsf(pz);
          const float m = fmaxf(apx, fmaxf(apy, apz));
          if (!(m < 1.0f)) {
            // c = f(m) p with f = 2/m - 1/m^2 ; dc_i/dp_j = f delta_ij + p_i f'(m) dm/dp_j ; dm/dp_j = sign(p_k) [j == argmax]
            const float f = 2.0f / m - 1.0f / (m * m), fp = -2.0f / (m * m) + 2.0f / (m * m * m);
            const float dot = ax * px + ay * py + az * pz;
            gx = f * ax; gy = f * ay; gz = f * az;
            if (apx >= apy && apx >= apz) gx += copysignf(1.0f, px) * fp * dot;
            else if (apy >= apz) gy += copysignf(1.0f, py) * fp * dot;
            else gz += copysignf(1.0f, pz) * fp * dot;
          } else { gx = ax; gy = ay; gz = az; }
        } else {
          gx = ax / (wp.aabb_max[0] - wp.aabb_min[0]); gy = ay / (wp.aabb_max[1] - wp.aabb_min[1]); gz = az / (wp.aabb_max[2] - wp.aabb_min[2]);
        }
      }
    }
    // ---- reduce over the ray ---------------------------------------------------------------------------------------------------
    const int64_t r0 = __shfl_sync(0xffffffffu, r, 0);
    const bool uniform = __all_sync(0xffffffffu, r == r0 && in);
    float vals[6] = {gx, gy, gz, tt * gx, tt * gy, tt * gz};
    if (uniform) {
#pragma unroll
      for (int q = 0; q < 6; ++q) {
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) vals[q] += __shfl_xor_sync(0xffffffffu, vals[q], off);
      }
      if (lane == 0) {
#pragma unroll
        for (int q = 0; q < 3; ++q) {
          if (vals[q] != 0.0f) atomicAdd(d_origins + 3 * r + q, vals[q]);
          if (vals[3 + q] != 0.0f) atomicAdd(d_directions + 3 * r + q, vals[3 + q]);
        }
      }
    } else if (in) {
#pragma unroll
      for (int q = 0; q < 3; ++q) {
        if (vals[q] != 0.0f) atomicAdd(d_origins + 3 * r + q, vals[q]);
        if (vals[3 + q] != 0.0f) atomicAdd(d_directions + 3 * r + q, vals[3 + q]);
      }
    }
  }
}

int grid_for(int64_t work_items, int block) {
  int64_t blocks = (work_items + block - 1) / block;
  int64_t cap = (int64_t)cnb_num_sms() * 16;  // multiple of the SM count; grid-stride beyond that
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

}  // namespace

static int check_grid(const cnb_grid* g, bool need_grad) {
  CNB_REQUIRE(g != nullptr && g->table != nullptr, "hashgrid: null grid/table");
  CNB_REQUIRE(g->num_levels >= 1 && g->num_levels <= CNB_MAX_LEVELS, "hashgrid: num_levels %d outside 1..%d", g->num_levels, CNB_MAX_LEVELS);
  CNB_REQUIRE(g->log2_hashmap_size >= 1 && g->log2_hashmap_size <= 24, "hashgrid: log2_hashmap_size %d outside 1..24", g->log2_hashmap_size);
  CNB_REQUIRE(!need_grad || g->d_table != nullptr, "hashgrid: backward needs d_table");
  return CNB_OK;
}

extern "C" int cnb_hashgrid_fwd(const cnb_grid* g, const float* positions, int64_t n, float* out, int32_t* indices, cnb_stream_t stream) {
  return cnb_hashgrid_fwd_half(g, nullptr, positions, n, out, indices, stream);
}

extern "C" int cnb_hashgrid_fwd_half(const cnb_grid* g, const void* table_half, const float* positions, int64_t n, float* out, int32_t* indices,
                                     cnb_stream_t stream) {
  int rc = check_grid(g, false);
  if (rc) return rc;
  CNB_REQUIRE(n >= 0 && (n == 0 || (positions && out)), "hashgrid_fwd: null positions/out");
  if (n == 0) return CNB_OK;
  const int blocks = grid_for(((n + 31) / 32) * 32 * g->num_levels, 256);
  if (table_half != nullptr) {
    CNB_REQUIRE(((uintptr_t)table_half & 7) == 0, "hashgrid_fwd: the fp16 table must be 8-byte aligned");
    k_hashgrid_fwd<__half2><<<blocks, 256, 0, stream>>>(make_args(g, static_cast<const __half2*>(table_half)), positions, n, out, indices);
  } else {
    k_hashgrid_fwd<float><<<blocks, 256, 0, stream>>>(make_args(g), positions, n, out, indices);
  }
  return cnb_check_launch("hashgrid_fwd");
}

static int hashgrid_bwd_impl(const cnb_grid* g, const float* positions, const float* d_out, int64_t n, bool level_major, cnb_stream_t stream) {
  int rc = check_grid(g, true);
  if (rc) return rc;
  CNB_REQUIRE(n >= 0 && (n == 0 || (positions && d_out)), "hashgrid_bwd: null positions/d_out");
  if (n == 0) return CNB_OK;
  GridArgs a = make_args(g);
  for (int i = 0; i < a.L; ++i) CNB_REQUIRE(a.scalings[i] < 65535.0f, "hashgrid_bwd: level resolution %g too large for the aggregated scatter", a.scalings[i]);
  const int blocks = grid_for(((n + 31) / 32) * 32 * a.L, 256);
  if (level_major) k_hashgrid_bwd<true><<<blocks, 256, 0, stream>>>(a, positions, d_out, n);
  else k_hashgrid_bwd<false><<<blocks, 256, 0, stream>>>(a, positions, d_out, n);
  return cnb_check_launch("hashgrid_bwd");
}

extern "C" int cnb_hashgrid_bwd(const cnb_grid* g, const float* positions, const float* d_out, int64_t n, cnb_stream_t stream) {
  return hashgrid_bwd_impl(g, positions, d_out, n, false, stream);
}

// library-internal: d_out level-major [L][n][2] (scratch of the fused field backward)
int cnb_hashgrid_bwd_level_major(const cnb_grid* g, const float* positions, const float* d_out, int64_t n, cudaStream_t stream) {
  return hashgrid_bwd_impl(g, positions, d_out, n, true, stream);
}

static int position_grad_rays_impl(const cnb_grid* g, const __half2* table_half, const cnb_warp* warp, const cnb_samples* s, const float* d_feat,
                                   float* d_origins, float* d_directions, bool level_major, cnb_stream_t stream) {
  int rc = check_grid(g, false);
  if (rc) return rc;
  CNB_REQUIRE(warp && s && d_feat && d_origins && d_directions, "position_grad_rays: null pointer");
  CNB_REQUIRE(s->origins && s->directions && s->starts && s->ends && s->samples_per_ray >= 1 && s->num_rays >= 0, "position_grad_rays: bad samples");
  const int64_t total = s->num_rays * s->samples_per_ray;
  if (total == 0) return CNB_OK;
  const int blocks = grid_for(total, 128);
  if (table_half != nullptr) {
    CNB_REQUIRE(!level_major, "position_grad_rays: the fp16 table is read by the layer-by-layer field path only");
    k_position_grad_rays<false, __half2><<<blocks, 128, 0, stream>>>(make_args(g, table_half), *warp, *s, d_feat, d_origins, d_directions);
    return cnb_check_launch("position_grad_rays");
  }
  GridArgs a = make_args(g);
  if (level_major) k_position_grad_rays<true><<<blocks, 128, 0, stream>>>(a, *warp, *s, d_feat, d_origins, d_directions);
  else k_position_grad_rays<false><<<blocks, 128, 0, stream>>>(a, *warp, *s, d_feat, d_origins, d_directions);
  return cnb_check_launch("position_grad_rays");
}

extern "C" int cnb_position_grad_rays(const cnb_grid* g, const cnb_warp* warp, const cnb_samples* s, const float* d_feat, float* d_origins,
                                      float* d_directions, cnb_stream_t stream) {
  return position_grad_rays_impl(g, nullptr, warp, s, d_feat, d_origins, d_directions, false, stream);
}

extern "C" int cnb_position_grad_rays_half(const cnb_grid* g, const void* table_half, const cnb_warp* warp, const cnb_samples* s, const float* d_feat,
                                           float* d_origins, float* d_directions, cnb_stream_t stream) {
  return position_grad_rays_impl(g, static_cast<const __half2*>(table_half), warp, s, d_feat, d_origins, d_directions, false, stream);
}

// library-internal: d_feat level-major [L][total][2]
int cnb_position_grad_rays_level_major(const cnb_grid* g, const cnb_warp* warp, const cnb_samples* s, const float* d_feat, float* d_origins,
                                       float* d_directions, cudaStream_t stream) {
  return position_grad_rays_impl(g, nullptr, warp, s, d_feat, d_origins, d_directions, true, stream);
}

// ---------------------------------------------------------------------------------------------------------------------
// Reachable rows.  nerfstudio's torch HashEncoding hashes EVERY level into its 2^T slots, also the coarse ones whose lattice has far fewer
// points than slots (level 0 of the field grid: 17^3 = 4913 corners for 524 288 rows).  A row no lattice point hashes to never receives a
// gradient: its Adam moments stay exactly 0 and torch.optim.Adam leaves the parameter exactly unchanged, step after step.  The optimiser and the
// data-parallel exchange can therefore skip such rows without changing a single bit -- ~21 % of the field table, ~29 % of the proposal tables.
// This kernel ORs one bit per 16-byte unit (float4 = two rows) of the table into `bitmap`; bit index = first_unit + row / 2.
namespace {
__global__ void __launch_bounds__(256) k_mark_reachable(uint32_t* __restrict__ bitmap, int64_t first_unit, uint32_t level_offset, uint32_t mask, int side) {
  const int64_t total = (int64_t)side * side * side;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t x = (uint32_t)(i % side), y = (uint32_t)((i / side) % side), z = (uint32_t)(i / ((int64_t)side * side));
    const uint32_t row = cnb_hash(x, y, z, mask) + level_offset;
    const int64_t unit = first_unit + (row >> 1);
    atomicOr(bitmap + (unit >> 5), 1u << (unit & 31));
  }
}
__global__ void __launch_bounds__(256) k_mark_range(uint32_t* __restrict__ bitmap, int64_t first_unit, int64_t units) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < units; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t unit = first_unit + i;
    atomicOr(bitmap + (unit >> 5), 1u << (unit & 31));
  }
}
}  // namespace

extern "C" int cnb_hashgrid_mark_reachable(const cnb_grid* g, uint32_t* bitmap, int64_t first_unit, cnb_stream_t stream) {
  CNB_REQUIRE(g && bitmap && first_unit >= 0, "hashgrid_mark_reachable: null / negative argument");
  CNB_REQUIRE(g->num_levels >= 1 && g->num_levels <= CNB_MAX_LEVELS && g->log2_hashmap_size >= 1 && g->log2_hashmap_size <= 24, "hashgrid_mark_reachable: bad grid");
  const uint32_t T = 1u << g->log2_hashmap_size;
  for (int l = 0; l < g->num_levels; ++l) {
    const double side = floor((double)g->scalings[l]) + 2.0;  // coordinates 0 .. ceil(scale); one spare plane against rounding at the top face
    const int64_t first = first_unit + ((int64_t)l * T) / 2;
    if (side * side * side >= 8.0 * (double)T) {
      // (almost) every slot is hit: the level is dense in the table
      int64_t blocks = (T / 2 + 255) / 256;
      k_mark_range<<<(int)blocks, 256, 0, stream>>>(bitmap, first, T / 2);
    } else {
      const int sd = (int)side;
      int64_t blocks = ((int64_t)sd * sd * sd + 255) / 256;
      const int64_t cap = (int64_t)cnb_num_sms() * 32;
      if (blocks > cap) blocks = cap;
      k_mark_reachable<<<(int)blocks, 256, 0, stream>>>(bitmap, first_unit, (uint32_t)l * T, T - 1u, sd);
    }
    int rc = cnb_check_launch("hashgrid_mark_reachable");
    if (rc) return rc;
  }
  return CNB_OK;
}

extern "C" int cnb_bitmap_mark_range(uint32_t* bitmap, int64_t first_unit, int64_t units, cnb_stream_t stream) {
  CNB_REQUIRE(bitmap && first_unit >= 0 && units >= 0, "bitmap_mark_range: bad argument");
  if (units == 0) return CNB_OK;
  int64_t blocks = (units + 255) / 256;
  const int64_t cap = (int64_t)cnb_num_sms() * 32;
  if (blocks > cap) blocks = cap;
  k_mark_range<<<(int)blocks, 256, 0, stream>>>(bitmap, first_unit, units);
  return cnb_check_launch("bitmap_mark_range");
}

// ---------------------------------------------------------------------------------------------------------------------
// fp16 copy of a table (initialisation, checkpoint load, writes made outside the optimiser): dst[i] = __float2half_rn(src[i]).  With `live`, only
// the 16-byte units whose bit (first_unit + i / 4) is set are written -- the rows the optimiser updates; the others keep what they hold.
namespace {
__global__ void __launch_bounds__(256) k_table_to_half(const float4* __restrict__ src, int64_t n4, const uint32_t* __restrict__ live, int64_t first_unit,
                                                       uint2* __restrict__ dst) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    if (live != nullptr) {
      const int64_t u = first_unit + i;
      if (!((__ldg(live + (u >> 5)) >> (u & 31)) & 1u)) continue;
    }
    const float4 v = __ldg(src + i);
    const __half2 a = __floats2half2_rn(v.x, v.y), b = __floats2half2_rn(v.z, v.w);
    dst[i] = make_uint2(*reinterpret_cast<const uint32_t*>(&a), *reinterpret_cast<const uint32_t*>(&b));
  }
}
}  // namespace

extern "C" int cnb_table_to_half(const float* table, int64_t n, const uint32_t* live, int64_t first_unit, void* table_half, cnb_stream_t stream) {
  CNB_REQUIRE(n >= 0 && n % 4 == 0 && first_unit >= 0, "table_to_half: n = %lld must be a multiple of 4", (long long)n);
  if (n == 0) return CNB_OK;
  CNB_REQUIRE(table && table_half, "table_to_half: null pointer");
  CNB_REQUIRE((((uintptr_t)table & 15) | ((uintptr_t)table_half & 7)) == 0, "table_to_half: table must be 16-byte, table_half 8-byte aligned");
  const int64_t n4 = n / 4;
  int64_t blocks = (n4 + 255) / 256;
  const int64_t cap = (int64_t)cnb_num_sms() * 16;
  if (blocks > cap) blocks = cap;
  k_table_to_half<<<(int)blocks, 256, 0, stream>>>(reinterpret_cast<const float4*>(table), n4, live, first_unit, static_cast<uint2*>(table_half));
  return cnb_check_launch("table_to_half");
}
