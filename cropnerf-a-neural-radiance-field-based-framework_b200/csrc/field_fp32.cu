// FruitField forward/backward, exact-fp32 path (rows a1, a5, a6 of SURVEY.md section 8) and the C-ABI entry
// points cnb_field_* that dispatch between this path and the tensor-core path (field_mixed.cu).
//
// Replaces fruit_field.py:169-194 (get_density), :196-233 (get_inference_outputs), :235-282 (get_outputs) and
// :284-302 (forward).  The fp32 path is the 1e-4-parity mode: it chains the exact building blocks
// (position warp -> cnb_hashgrid -> cnb_mlp(base) -> trunc_exp/SH/embedding glue -> cnb_mlp(sem)+head, cnb_mlp(rgb))
// through a caller-provided scratch buffer `ctx`, which also keeps the activations the backward needs.
#include <algorithm>

#include "field_common.cuh"

namespace {

inline int up4(int v) { return (v + 3) & ~3; }

struct CtxLayout {
  int64_t pos, sel, x0, hb, bo, hs, s2, semv, rin, hr, rgbv;  // forward (float offsets)
  int64_t d_bo, d_rin, d_s2, d_x0, d_gs;                      // backward scratch
  int64_t work;                                               // mixed: the MLP operator's backward work space, shared by the three MLPs
  int64_t total;
  int in0, ob, os, ri, rip;
};

// exact fp32 (mixed = false) or the mixed path for architectures outside the fused kernels (mixed = true): the same chain and layout, with
// the MLPs' kept activations in the tensor-core operator's fp16 format (inference: one ping-pong region that the three MLPs take in turn)
CtxLayout make_layout(const cnb_field* f, int64_t n, bool training, bool mixed = false) {
  CtxLayout c;
  c.in0 = f->base.dims[0];
  c.ob = f->base.dims[f->base.num_layers];
  c.os = f->sem.dims[f->sem.num_layers];
  c.ri = f->rgb.dims[0];
  c.rip = up4(c.ri);
  int64_t o = 0;
  auto take = [&](int64_t per) { int64_t r = o; o += per * n; o = (o + 3) & ~(int64_t)3; return r; };
  auto take_total = [&](int64_t floats) { int64_t r = o; o += floats; o = (o + 3) & ~(int64_t)3; return r; };
  auto hidden = [&](const cnb_mlp* m) {
    if (!mixed) return take(training ? cnb_mlp_hidden_floats(m) : 0);
    return take_total(cnb_mlp_mixed_hidden_floats(m, n, 1));
  };
  c.pos = take(3); c.sel = take(1); c.x0 = take(c.in0);
  if (mixed && !training) {
    const int64_t h = std::max(cnb_mlp_mixed_hidden_floats(&f->base, n, 0),
                               std::max(cnb_mlp_mixed_hidden_floats(&f->sem, n, 0), cnb_mlp_mixed_hidden_floats(&f->rgb, n, 0)));
    c.hb = c.hs = c.hr = take_total(h);
  } else {
    c.hb = hidden(&f->base);
  }
  c.bo = take(c.ob);
  if (training || !mixed) c.hs = hidden(&f->sem);
  c.s2 = take(c.os); c.semv = take(1); c.rin = take(c.rip);
  if (training || !mixed) c.hr = hidden(&f->rgb);
  c.rgbv = take(3);
  if (training) {
    c.d_bo = take(c.ob); c.d_rin = take(c.rip); c.d_s2 = take(c.os); c.d_x0 = take(c.in0);
    c.d_gs = take(f->pass_semantic_gradients && !mixed ? c.ob : 0);
    c.work = take_total(mixed ? std::max(cnb_mlp_mixed_work_floats(&f->base, n),
                                         std::max(cnb_mlp_mixed_work_floats(&f->sem, n), cnb_mlp_mixed_work_floats(&f->rgb, n)))
                              : 0);
  } else {
    c.d_bo = c.d_rin = c.d_s2 = c.d_x0 = c.d_gs = c.work = o;
  }
  c.total = o;
  return c;
}

__global__ void __launch_bounds__(256) k_positions(cnb_samples sm, cnb_warp w, float* __restrict__ pos, float* __restrict__ sel, float* __restrict__ pos_out) {
  const int S = sm.samples_per_ray;
  const int64_t total = sm.num_rays * S;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = cnb_ray_of(i, S);
    float x, y, z;
    const bool s = cnb_sample_position(sm, w, r, (int)(i - r * S), x, y, z);
    pos[3 * i] = x; pos[3 * i + 1] = y; pos[3 * i + 2] = z;
    sel[i] = s ? 1.0f : 0.0f;
    if (pos_out) { pos_out[3 * i] = x; pos_out[3 * i + 1] = y; pos_out[3 * i + 2] = z; }
  }
}

// density = trunc_exp(bo[:,0]) * selector ; rgb_in = [SH16 | geo | appearance] (fruit_field.py:186-193,244-279)
// One WARP per sample, lanes = columns of the row: the 256-byte rows go out as coalesced stores (a thread per sample wrote 32 rows per store
// instruction, 256 bytes apart: 87 us for 196 608 samples, several times its HBM time).  Every lane evaluates the 16 SH components of the
// ray (40 flops) and keeps the one of its column.
__global__ void __launch_bounds__(256) k_mid_fwd(cnb_samples sm, const float* __restrict__ bo, int ob, const float* __restrict__ sel,
                                                 const float* __restrict__ embedding, const float* __restrict__ mean_embedding, int app_mode,
                                                 int app_dim, int rip, float* __restrict__ density, float* __restrict__ geo_out,
                                                 float* __restrict__ rin) {
  const int S = sm.samples_per_ray;
  const int64_t total = sm.num_rays * S;
  const int geo = ob - 1, lane = threadIdx.x & 31;
  const int64_t wstride = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t i = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5); i < total; i += wstride) {
    const int64_t r = cnb_ray_of(i, S);
    const float* b = bo + i * ob;
    if (lane == 0) density[i] = sel[i] != 0.0f ? expf(b[0]) : 0.0f;
    if (geo_out) for (int k = lane; k < ob; k += 32) geo_out[i * ob + k] = b[k];
    float c[16];
    cnb_sh16(__ldg(sm.directions + 3 * r), __ldg(sm.directions + 3 * r + 1), __ldg(sm.directions + 3 * r + 2), c);
    float mine = 0.0f;
#pragma unroll
    for (int q = 0; q < 16; ++q) mine = (lane == q) ? c[q] : mine;
    const float* e = nullptr;
    if (app_mode == CNB_APP_PER_CAMERA) e = embedding + (int64_t)__ldg(sm.camera_indices + r) * app_dim;
    else if (app_mode == CNB_APP_MEAN) e = mean_embedding;
    float* o = rin + i * rip;
    for (int k = lane; k < rip; k += 32) {
      float v = 0.0f;
      if (k < 16) v = mine;
      else if (k < 16 + geo) v = b[1 + (k - 16)];
      else if (k < 16 + geo + app_dim) v = e ? __ldg(e + (k - 16 - geo)) : 0.0f;
      o[k] = v;
    }
  }
}

// d_bo = [d_density * exp(clamp(bo0)) * sel | d_rin[geo slice] (+ semantic / external geo gradients)]
__global__ void __launch_bounds__(256) k_mid_bwd(int64_t total, const float* __restrict__ bo, int ob, const float* __restrict__ sel,
                                                 const float* __restrict__ d_density, const float* __restrict__ d_rin, int rip,
                                                 const float* __restrict__ d_gs, const float* __restrict__ d_geo_ext, float* __restrict__ d_bo) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    float g0 = 0.0f;
    if (d_density && sel[i] != 0.0f) g0 = __ldg(d_density + i) * cnb_trunc_exp_grad(bo[i * ob]);
    if (d_geo_ext) g0 += __ldg(d_geo_ext + i * ob);
    d_bo[i * ob] = g0;
    for (int k = 1; k < ob; ++k) {
      float g = d_rin ? d_rin[i * rip + 15 + k] : 0.0f;
      if (d_gs) g += d_gs[i * ob + k];
      if (d_geo_ext) g += __ldg(d_geo_ext + i * ob + k);
      d_bo[i * ob + k] = g;
    }
  }
}

// d_embedding[cam] += sum over the ray's samples of d_rin[appearance slice]; one warp per ray, lanes = embedding dims
__global__ void __launch_bounds__(128) k_emb_bwd(const int32_t* __restrict__ cams, int64_t R, int S, const float* __restrict__ d_rin, int rip,
                                                 int app_off, int app_dim, float* __restrict__ d_embedding) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int64_t r = blockIdx.x * 4LL + warp; r < R; r += gridDim.x * 4LL) {
    const int64_t cam = __ldg(cams + r);
    for (int k0 = 0; k0 < app_dim; k0 += 32) {
      const int k = k0 + lane;
      if (k >= app_dim) continue;
      float acc = 0.0f;
      for (int s = 0; s < S; ++s) acc += d_rin[(r * S + s) * rip + app_off + k];
      if (acc != 0.0f) atomicAdd(d_embedding + cam * app_dim + k, acc);
    }
  }
}

int grid1d(int64_t items, int block) {
  int64_t blocks = (items + block - 1) / block;
  const int64_t cap = (int64_t)cnb_num_sms() * 16;
  if (blocks > cap) blocks = cap;
  return (int)(blocks < 1 ? 1 : blocks);
}

}  // namespace

int cnb_field_check(const cnb_field* f, const cnb_samples* s, bool bwd) {
  CNB_REQUIRE(f && s, "field: null descriptor");
  CNB_REQUIRE(f->grid.table != nullptr, "field: null table");
  CNB_REQUIRE(f->grid.num_levels >= 1 && f->grid.num_levels <= CNB_MAX_LEVELS, "field: num_levels %d unsupported", f->grid.num_levels);
  CNB_REQUIRE(f->base.dims[0] == 2 * f->grid.num_levels, "field: base mlp in dim %d != 2*num_levels", f->base.dims[0]);
  CNB_REQUIRE(f->base.dims[f->base.num_layers] == 1 + f->geo_feat_dim, "field: base mlp out dim != 1+geo_feat_dim");
  CNB_REQUIRE(f->sem.dims[0] == f->geo_feat_dim, "field: semantic mlp in dim != geo_feat_dim");
  CNB_REQUIRE(f->sem_head.num_layers == 1 && f->sem_head.dims[0] == f->sem.dims[f->sem.num_layers] && f->sem_head.dims[1] == 1,
              "field: semantic head must be Linear(sem_out, 1) (num_semantic_classes=1, fruit_nerf.py:110)");
  CNB_REQUIRE(f->rgb.dims[0] == 16 + f->geo_feat_dim + f->appearance_dim, "field: rgb mlp in dim != 16+geo+appearance");
  CNB_REQUIRE(f->rgb.dims[f->rgb.num_layers] == 3 && f->rgb.out_activation == CNB_ACT_SIGMOID, "field: rgb mlp must end in 3 sigmoid outputs");
  CNB_REQUIRE(f->appearance_mode != CNB_APP_PER_CAMERA || (f->embedding && s->camera_indices), "field: per-camera appearance needs embedding + camera_indices");
  CNB_REQUIRE(f->appearance_mode != CNB_APP_MEAN || f->mean_embedding, "field: mean appearance needs mean_embedding");
  CNB_REQUIRE(s->origins && s->directions && s->starts && s->ends, "field: null sample arrays");
  CNB_REQUIRE(s->samples_per_ray >= 1 && s->num_rays >= 0, "field: bad sample counts");
  CNB_REQUIRE(!bwd || f->grid.d_table != nullptr, "field_bwd: d_table required");
  return CNB_OK;
}

bool cnb_field_mixed_wide_supported(const cnb_field* f) {
  return f && cnb_mlp_mixed_supported(&f->base) && cnb_mlp_mixed_supported(&f->sem) && cnb_mlp_mixed_supported(&f->rgb);
}

// kernels launched by cnb_field_fwd / cnb_field_bwd(_rays) on the mixed path for the wide architectures (stage timers of pipeline.cu)
int cnb_field_mixed_wide_launches(const cnb_field* f, bool bwd, bool rays) {
  if (!bwd) return 4 + cnb_mlp_mixed_launches(&f->base, false, false) + cnb_mlp_mixed_launches(&f->sem, false, false) +
                   cnb_mlp_mixed_launches(&f->rgb, false, false);
  return 4 + (rays ? 1 : 0) + cnb_mlp_mixed_launches(&f->rgb, true, true) + cnb_mlp_mixed_launches(&f->sem, true, false) +
         cnb_mlp_mixed_launches(&f->base, true, true);
}

namespace {
// the mixed path of a field that the fused kernels do not cover
bool mixed_wide(const cnb_field* f) { return f->precision == CNB_PREC_MIXED && !cnb_field_mixed_supported(f) && cnb_field_mixed_wide_supported(f); }
}  // namespace

extern "C" int64_t cnb_field_ctx_floats(const cnb_field* f, int64_t n, int32_t training) {
  if (!f || n <= 0) return 0;
  if (mixed_wide(f)) return make_layout(f, n, training != 0, true).total;
  if (f->precision == CNB_PREC_MIXED) return cnb_field_mixed_ctx_floats(n, training);
  return make_layout(f, n, training != 0).total;
}

extern "C" int cnb_field_fwd(const cnb_field* f, const cnb_samples* s, float* density, float* geo, float* rgb, float* sem, float* positions_out,
                             float* ctx, int32_t training, cnb_stream_t stream) {
  int rc = cnb_field_check(f, s, false);
  if (rc) return rc;
  const int64_t N = s->num_rays * s->samples_per_ray;
  if (N == 0) return CNB_OK;
  CNB_REQUIRE(density != nullptr, "field_fwd: null density output");
  const bool wide = mixed_wide(f);
  if (f->precision == CNB_PREC_MIXED && !wide) {
    if (!cnb_field_mixed_supported(f)) {
      cnb_set_error("field_fwd: mixed precision is compiled for the base fruit_nerf architecture (L<=16, widths 64, geo 15, app 32) and for "
                    "MLPs up to 128 wide");
      return CNB_ERR_UNSUPPORTED;
    }
    CNB_REQUIRE(geo == nullptr || f->geo_feat_dim == 15, "field_fwd: the mixed path exports geo as [N,16]");
    CNB_REQUIRE(!training || ctx != nullptr, "field_fwd: mixed training forward needs ctx scratch (cnb_field_ctx_floats)");
    CNB_REQUIRE(!training || (rgb != nullptr && sem != nullptr), "field_fwd: the mixed training forward keeps both heads' activations for the backward");
    return cnb_field_mixed_fwd(f, s, density, geo, rgb, sem, positions_out, ctx, training, stream);
  }
  CNB_REQUIRE(ctx != nullptr, "field_fwd: this path needs ctx scratch (cnb_field_ctx_floats)");
  const CtxLayout c = make_layout(f, N, training != 0, wide);
  // the three MLPs: exact (mlp.cu / mlp_wide.cu) or the tensor-core operator (mlp_mixed.cu)
  auto mlp_fwd = [&](const cnb_mlp* m, const float* x, int64_t ld, float* y, int64_t hidden) {
    if (wide) return cnb_mlp_mixed_fwd_ws(m, x, ld, N, y, ctx + hidden, training, stream);
    return cnb_mlp_fwd(m, x, ld, N, y, training ? ctx + hidden : nullptr, stream);
  };
  float* pos = ctx + c.pos; float* sel = ctx + c.sel; float* x0 = ctx + c.x0; float* bo = ctx + c.bo;
  k_positions<<<grid1d(N, 256), 256, 0, stream>>>(*s, f->warp, pos, sel, positions_out);
  if ((rc = cnb_check_launch("field positions"))) return rc;
  if ((rc = cnb_hashgrid_fwd(&f->grid, pos, N, x0, nullptr, stream))) return rc;
  if ((rc = mlp_fwd(&f->base, x0, c.in0, bo, c.hb))) return rc;
  k_mid_fwd<<<grid1d(N, 256), 256, 0, stream>>>(*s, bo, c.ob, sel, f->embedding, f->mean_embedding, f->appearance_mode, f->appearance_dim, c.rip, density,
                                                 geo, ctx + c.rin);
  if ((rc = cnb_check_launch("field mid"))) return rc;
  if (sem != nullptr || training) {
    float* semv = ctx + c.semv;
    if ((rc = mlp_fwd(&f->sem, bo + 1, c.ob, ctx + c.s2, c.hs))) return rc;
    if ((rc = cnb_mlp_fwd(&f->sem_head, ctx + c.s2, c.os, N, sem ? sem : semv, nullptr, stream))) return rc;
  }
  if (rgb != nullptr || training) {
    float* rgbv = ctx + c.rgbv;
    if ((rc = mlp_fwd(&f->rgb, ctx + c.rin, c.rip, rgbv, c.hr))) return rc;
    if (rgb != nullptr && cudaMemcpyAsync(rgb, rgbv, sizeof(float) * 3 * N, cudaMemcpyDeviceToDevice, stream) != cudaSuccess)
      return cnb_check_launch("field rgb copy");
  }
  return CNB_OK;
}

extern "C" int cnb_field_bwd(const cnb_field* f, const cnb_samples* s, const float* d_density, const float* d_rgb, const float* d_sem,
                             const float* d_geo, float* ctx, cnb_stream_t stream) {
  int rc = cnb_field_check(f, s, true);
  if (rc) return rc;
  const int64_t N = s->num_rays * s->samples_per_ray;
  if (N == 0) return CNB_OK;
  const bool wide = mixed_wide(f);
  if (f->precision == CNB_PREC_MIXED) {
    if (!cnb_field_mixed_supported(f) && !wide) {
      cnb_set_error("field_bwd: mixed precision is compiled for the base fruit_nerf architecture and for MLPs up to 128 wide");
      return CNB_ERR_UNSUPPORTED;
    }
    CNB_REQUIRE(d_geo == nullptr, "field_bwd: mixed precision path takes no external geo gradient");
    CNB_REQUIRE(ctx != nullptr, "field_bwd: mixed path needs the ctx written by cnb_field_fwd(training=1)");
    CNB_REQUIRE(!f->pass_semantic_gradients, "field_bwd: pass_semantic_gradients is not compiled for the mixed path");
    if (!wide) return cnb_field_mixed_bwd(f, s, d_density, d_rgb, d_sem, ctx, stream);
  }
  CNB_REQUIRE(ctx != nullptr, "field_bwd: fp32 path needs the ctx written by cnb_field_fwd(training=1)");
  const CtxLayout c = make_layout(f, N, true, wide);
  auto mlp_bwd = [&](const cnb_mlp* m, const float* x, int64_t ld, int64_t hidden, const float* y, const float* dy, float* dx, int64_t dx_ld) {
    if (wide) return cnb_mlp_mixed_bwd_ws(m, x, ld, ctx + hidden, y, dy, N, dx, dx_ld, ctx + c.work, stream);
    return cnb_mlp_bwd(m, x, ld, ctx + hidden, y, dy, N, dx, dx_ld, stream);
  };
  float* pos = ctx + c.pos; float* sel = ctx + c.sel; float* x0 = ctx + c.x0; float* bo = ctx + c.bo;
  float* d_rin = nullptr;
  if (d_rgb != nullptr) {
    d_rin = ctx + c.d_rin;
    if ((rc = mlp_bwd(&f->rgb, ctx + c.rin, c.rip, c.hr, ctx + c.rgbv, d_rgb, d_rin, c.rip))) return rc;
    if (f->appearance_mode == CNB_APP_PER_CAMERA && f->d_embedding != nullptr) {
      k_emb_bwd<<<grid1d(s->num_rays, 4), 128, 0, stream>>>(s->camera_indices, s->num_rays, s->samples_per_ray, d_rin, c.rip, 16 + f->geo_feat_dim,
                                                            f->appearance_dim, f->d_embedding);
      if ((rc = cnb_check_launch("field emb bwd"))) return rc;
    }
  }
  float* d_gs = nullptr;
  if (d_sem != nullptr) {
    if ((rc = cnb_mlp_bwd(&f->sem_head, ctx + c.s2, c.os, nullptr, nullptr, d_sem, N, ctx + c.d_s2, c.os, stream))) return rc;
    if (f->pass_semantic_gradients) {
      d_gs = ctx + c.d_gs;
      if (cudaMemsetAsync(d_gs, 0, sizeof(float) * c.ob * N, stream) != cudaSuccess) return cnb_check_launch("field memset");
    }
    if ((rc = mlp_bwd(&f->sem, bo + 1, c.ob, c.hs, nullptr, ctx + c.d_s2, d_gs ? d_gs + 1 : nullptr, c.ob))) return rc;
  }
  k_mid_bwd<<<grid1d(N, 256), 256, 0, stream>>>(N, bo, c.ob, sel, d_density, d_rin, c.rip, d_gs, d_geo, ctx + c.d_bo);
  if ((rc = cnb_check_launch("field mid bwd"))) return rc;
  if ((rc = mlp_bwd(&f->base, x0, c.in0, c.hb, nullptr, ctx + c.d_bo, ctx + c.d_x0, c.in0))) return rc;
  return cnb_hashgrid_bwd(&f->grid, pos, ctx + c.d_x0, N, stream);
}

// Same as cnb_field_bwd, plus the gradient with respect to the rays (row a17: camera optimizer): the hash-grid input
// gradient is chained through the position normalisation / contraction and reduced per ray into d_origins / d_directions
// (accumulated).  Not compiled for the 16-level limit of the fused mixed kernel's d_x0 layout when num_levels > 16; the other paths keep
// d(features) row-major.
extern "C" int cnb_field_bwd_rays(const cnb_field* f, const cnb_samples* s, const float* d_density, const float* d_rgb, const float* d_sem,
                                  const float* d_geo, float* ctx, float* d_origins, float* d_directions, cnb_stream_t stream) {
  CNB_REQUIRE(d_origins && d_directions, "field_bwd_rays: null ray gradients");
  int rc = cnb_field_bwd(f, s, d_density, d_rgb, d_sem, d_geo, ctx, stream);
  if (rc) return rc;
  const int64_t N = s->num_rays * s->samples_per_ray;
  if (N == 0) return CNB_OK;
  const bool wide = mixed_wide(f);
  if (f->precision == CNB_PREC_MIXED && !wide) {
    CNB_REQUIRE(f->grid.num_levels == 16, "field_bwd_rays: the mixed path stores d(features) as [16][N][2]; num_levels must be 16");
    return cnb_position_grad_rays_level_major(&f->grid, &f->warp, s, cnb_field_mixed_dx0(ctx, N), d_origins, d_directions, stream);
  }
  return cnb_position_grad_rays(&f->grid, &f->warp, s, ctx + make_layout(f, N, true, wide).d_x0, d_origins, d_directions, stream);
}
