// The ray-render loop body as ONE C call (row a15 of SURVEY.md section 8): what FruitModel.get_outputs /
// get_inference_outputs (fruit_nerf.py:497-599) do per chunk of rays, plus -- for training -- get_loss_dict /
// get_metrics_dict (fruit_nerf.py:601-615,639-645) and the full backward.  Everything is enqueued on the caller's
// stream into a caller-provided workspace: no allocation, no host synchronisation, CUDA-graph capturable.
//
// Workspace layout (floats, every block 64-float aligned), for S_l = samples of level l (proposal levels then the field):
//   nears,fars [R] | per level: spacing edges [R,S_l+1], euclid edges [R,S_l+1], density [R,S_l], weights [R,S_l]
//   | field rgb [R,S,3], sem [R,S] | per-ray outputs | (training) per-ray output grads, d_weights/d_density per level,
//   d_rgb, d_sem | field ctx (cnb_field_ctx_floats)
#include "field_common.cuh"

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

namespace {

constexpr int MAX_LEVELS_P = 3;

// Optional per-stage device timing of the calls below (cudaEvents on the launching stream); off by default and never
// enabled during graph capture.  Read with cnb_profile_read.
struct StageEv { const char* name; int kernels; cudaEvent_t e0, e1; };
bool g_prof_on = false;
std::vector<StageEv> g_prof;

struct StageTimer {
  cudaStream_t st; bool on; StageEv ev;
  StageTimer(const char* name, int kernels, cudaStream_t s) : st(s), on(g_prof_on) {
    if (!on) return;
    ev.name = name; ev.kernels = kernels;
    cudaEventCreate(&ev.e0); cudaEventCreate(&ev.e1);
    cudaEventRecord(ev.e0, st);
  }
  ~StageTimer() {
    if (!on) return;
    cudaEventRecord(ev.e1, st);
    g_prof.push_back(ev);
  }
};
#define STAGE(name, kernels, call) do { StageTimer _t(name, kernels, st); rc = (call); } while (0)

struct Layout {
  int levels;            // proposal iterations + 1
  int S[MAX_LEVELS_P];
  int64_t nears, fars;
  int64_t sp[MAX_LEVELS_P], eu[MAX_LEVELS_P], dens[MAX_LEVELS_P], w[MAX_LEVELS_P];
  int64_t rgb, sem;
  int64_t o_rgb, o_acc, o_sem, o_depth, o_pd[2];
  int64_t g_rgb, g_sem, d_w[MAX_LEVELS_P], d_dens[MAX_LEVELS_P], d_rgb, d_sem;
  int64_t ctx, ctx_floats;
  int64_t pg_scratch;    // (= pg_level[0]; kept for the workspace-size accounting)
  int64_t pg_level[MAX_LEVELS_P];  // one scratch per proposal level: the levels back-propagate concurrently
  int64_t pfeat[MAX_LEVELS_P];  // (training) encoded features of each proposal level kept by the forward for the backward; -1 = not kept
  int64_t total;
};

int make_layout(const cnb_model* m, int64_t R, bool training, Layout& L) {
  const cnb_sampler& s = m->sampler;
  CNB_REQUIRE(s.num_proposal_iterations >= 1 && s.num_proposal_iterations <= 2, "render: num_proposal_iterations %d outside 1..2", s.num_proposal_iterations);
  L.levels = s.num_proposal_iterations + 1;
  for (int i = 0; i < s.num_proposal_iterations; ++i) L.S[i] = s.proposal_samples[i];
  L.S[L.levels - 1] = s.nerf_samples;
  for (int i = 0; i < L.levels; ++i) CNB_REQUIRE(L.S[i] >= 1 && L.S[i] <= 4096, "render: samples per ray %d outside 1..4096", L.S[i]);
  int64_t o = 0;
  auto take = [&](int64_t n) { int64_t r = o; o += (n + 63) & ~(int64_t)63; return r; };
  L.nears = take(R); L.fars = take(R);
  for (int i = 0; i < L.levels; ++i) {
    L.sp[i] = take(R * (L.S[i] + 1)); L.eu[i] = take(R * (L.S[i] + 1));
    L.dens[i] = take(R * L.S[i]); L.w[i] = take(R * L.S[i]);
  }
  const int Sf = L.S[L.levels - 1];
  L.rgb = take(R * Sf * 3); L.sem = take(R * Sf);
  L.o_rgb = take(R * 3); L.o_acc = take(R); L.o_sem = take(R); L.o_depth = take(R); L.o_pd[0] = take(R); L.o_pd[1] = take(R);
  if (training) {
    L.g_rgb = take(R * 3); L.g_sem = take(R);
    for (int i = 0; i < L.levels; ++i) { L.d_w[i] = take(R * L.S[i]); L.d_dens[i] = take(R * L.S[i]); }
    L.d_rgb = take(R * Sf * 3); L.d_sem = take(R * Sf);
  }
  for (int i = 0; i < MAX_LEVELS_P; ++i) L.pfeat[i] = -1;
  if (training)
    for (int i = 0; i + 1 < L.levels; ++i)
      if (cnb_density_field_kept_supported(&m->proposal[i])) L.pfeat[i] = take(R * L.S[i] * 2 * m->proposal[i].grid.num_levels);
  L.pg_scratch = o;
  for (int i = 0; i < MAX_LEVELS_P; ++i) L.pg_level[i] = o;
  if (training && m->ray_gradients) {
    for (int i = 0; i + 1 < L.levels; ++i) L.pg_level[i] = take(R * L.S[i] * 2 * m->proposal[i].grid.num_levels);
    L.pg_scratch = L.pg_level[0];
  }
  L.ctx_floats = cnb_field_ctx_floats(&m->field, R * Sf, training ? 1 : 0);
  L.ctx = take(L.ctx_floats);
  L.total = o;
  return CNB_OK;
}


// losses[4] = PSNR of the batch (get_metrics_dict, fruit_nerf.py:639-645: 10 log10(1 / mse)), losses[5] = rgb + semantics + interlevel
// (what the Trainer sums from get_loss_dict): the scalars a training loop logs, so it reads one buffer instead of launching its own kernels
__global__ void k_finalize_losses(float* __restrict__ l) {
  if (threadIdx.x == 0) {
    l[4] = -10.0f * log10f(l[0]);
    l[5] = l[0] + l[1] + l[2] + l[6];   // l[6] = camera-optimizer regulariser (0 unless it runs inside the step)
  }
}

__global__ void k_scale(float* __restrict__ v, int n, float s) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) v[i] *= s;
}

// Side stream + events for the fork / join inside cnb_train_step (one set per device, created on first use, never destroyed).
struct ForkState { cudaStream_t side[2] = {nullptr, nullptr}; cudaEvent_t fork = nullptr, join[2] = {nullptr, nullptr}, fork2 = nullptr; bool failed = false; };
ForkState g_fork[64];

ForkState* fork_state(cudaStream_t main) {
  static const bool disabled = [] { const char* e = getenv("CNB_TRAIN_NO_OVERLAP"); return e && e[0] == '1'; }();
  if (disabled) return nullptr;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  ForkState& f = g_fork[dev];
  if (f.failed) return nullptr;
  if (f.side[0] == nullptr) {
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(main, &cap) != cudaSuccess || cap != cudaStreamCaptureStatusNone) return nullptr;  // create outside captures (eager warm-up call)
    bool ok = cudaEventCreateWithFlags(&f.fork, cudaEventDisableTiming) == cudaSuccess && cudaEventCreateWithFlags(&f.fork2, cudaEventDisableTiming) == cudaSuccess;
    for (int i = 0; i < 2 && ok; ++i)
      ok = cudaStreamCreateWithFlags(&f.side[i], cudaStreamNonBlocking) == cudaSuccess && cudaEventCreateWithFlags(&f.join[i], cudaEventDisableTiming) == cudaSuccess;
    if (!ok) {
      f.failed = true;
      f.side[0] = nullptr;
      (void)cudaGetLastError();
      return nullptr;
    }
  }
  return &f;
}

// `to` waits for everything enqueued on `from` so far
bool stream_after(cudaStream_t to, cudaStream_t from, cudaEvent_t ev) {
  if (cudaEventRecord(ev, from) != cudaSuccess || cudaStreamWaitEvent(to, ev, 0) != cudaSuccess) { (void)cudaGetLastError(); return false; }
  return true;
}

cnb_samples make_samples(const cnb_rays* rays, const float* edges, int S) {
  cnb_samples sm;
  sm.origins = rays->origins; sm.directions = rays->directions;
  sm.starts = edges; sm.ends = edges + 1;
  sm.camera_indices = rays->camera_indices;
  sm.num_rays = rays->num_rays; sm.row_stride = S + 1; sm.samples_per_ray = S; sm._pad = 0;
  return sm;
}

int check_common(const cnb_model* m, const cnb_rays* rays, const float* ws) {
  CNB_REQUIRE(m && rays, "render: null model/rays");
  CNB_REQUIRE(rays->num_rays >= 0, "render: negative ray count");
  if (rays->num_rays == 0) return CNB_OK;
  CNB_REQUIRE(rays->origins && rays->directions, "render: null ray arrays");
  CNB_REQUIRE(ws != nullptr, "render: null workspace (cnb_render_workspace_floats)");
  CNB_REQUIRE(m->sampler.lin_bins != nullptr, "render: sampler.lin_bins missing");
  for (int i = 1; i <= m->sampler.num_proposal_iterations; ++i) CNB_REQUIRE(m->sampler.u_base[i - 1] != nullptr, "render: sampler.u_base[%d] missing", i - 1);
  return CNB_OK;
}

// sampler + proposal networks + field + compositing.  jitter == nullptr: deterministic (eval) samplers.
int forward_chain(const cnb_model* m, const cnb_rays* rays, const Layout& L, float* ws, bool training, const float* jitter, float anneal,
                  const cnb_ray_outputs* out, cudaStream_t st, bool keep_proposal_features = false, int part = 0) {
  // part 0: everything; 1: samplers + proposal networks only (reads no field parameter); 2: field level + compositing on what part 1 left
  const int64_t R = rays->num_rays;
  const cnb_sampler& sp = m->sampler;
  int rc = CNB_OK;
  const bool mixed = m->field.precision == CNB_PREC_MIXED;
  const bool mixed_wide = mixed && !cnb_field_mixed_supported(&m->field);   // the layer-by-layer tensor-core path (big / huge presets)
  const float* jit = jitter;
  const int lf = L.levels - 1;
  const bool user = out != nullptr;
  if (part != 2) {
    // NearFarCollider + the initial sampler in one kernel (per-ray near / far land in the workspace for the resampling levels)
    const int rstride = sp.single_jitter ? 1 : L.S[0] + 1;
    STAGE("sample_spaced", 1, cnb_sample_spaced_collide(rays->nears, rays->fars, rays->near_plane, rays->far_plane, sp.lin_bins, jit, rstride, sp.initial_spacing, R,
                                                        L.S[0], ws + L.nears, ws + L.fars, ws + L.sp[0], ws + L.eu[0], st));
    if (rc) return rc;
  }
  for (int lv = (part == 2 ? lf : 0); lv < (part == 1 ? lf : L.levels); ++lv) {
    const int S = L.S[lv];
    const cnb_samples sm = make_samples(rays, ws + L.eu[lv], S);
    if (lv < lf) {
      if (keep_proposal_features && L.pfeat[lv] >= 0)
        STAGE(lv == 0 ? "proposal0_fwd" : "proposal1_fwd", 1, cnb_density_field_fwd_keep(&m->proposal[lv], &sm, ws + L.dens[lv], ws + L.pfeat[lv], st));
      else
        STAGE(lv == 0 ? "proposal0_fwd" : "proposal1_fwd", 1, cnb_density_field_fwd(&m->proposal[lv], &sm, ws + L.dens[lv], nullptr, st));
      if (rc) return rc;
      // get_weights -> median depth -> PDF resampling of the next level, one kernel
      const int Sn = L.S[lv + 1];
      const int rstride = sp.single_jitter ? 1 : Sn + 1;
      if (jitter) {  // draws are laid out in sampler order: the initial sampler's, then one block per PDF resampling
        jit = jitter + R * (sp.single_jitter ? 1 : L.S[0] + 1);
        for (int q = 0; q < lv; ++q) jit += R * (sp.single_jitter ? 1 : L.S[q + 1] + 1);
      }
      STAGE("level_resample", 1, cnb_level_resample(ws + L.dens[lv], ws + L.eu[lv], ws + L.sp[lv], ws + L.nears, ws + L.fars, sp.initial_spacing, anneal,
                                                    sp.u_base[lv], jit, rstride, R, S, Sn, sp.histogram_padding, sp.pdf_eps, training ? ws + L.w[lv] : nullptr,
                                                    user ? out->prop_depth[lv] : nullptr, ws + L.sp[lv + 1], ws + L.eu[lv + 1],
                                                    (lv + 1 == lf && user) ? out->pdf_inds : nullptr, st));
      if (rc) return rc;
    } else {
      STAGE("field_fwd", mixed_wide ? cnb_field_mixed_wide_launches(&m->field, false, false) : (mixed ? 1 : 7), cnb_field_fwd(&m->field, &sm, ws + L.dens[lv], nullptr, ws + L.rgb, ws + L.sem, nullptr,
                                                        L.ctx_floats > 0 ? ws + L.ctx : nullptr, training ? 1 : 0, st));
      if (rc) return rc;
    }
  }
  if (part == 1) return rc;
  const int Sf = L.S[lf];
  float* o_rgb = (user && out->rgb) ? out->rgb : ws + L.o_rgb;
  float* o_acc = (user && out->accumulation) ? out->accumulation : ws + L.o_acc;
  float* o_sem = (user && out->semantics) ? out->semantics : ws + L.o_sem;
  float* o_depth = (user && out->depth) ? out->depth : nullptr;
  // get_weights -> RGB / accumulation / semantic / median-depth renderers of the final level, one kernel
  STAGE("final_composite", 1, cnb_final_composite(ws + L.dens[lf], ws + L.rgb, ws + L.sem, ws + L.eu[lf], R, Sf, m->bg_mode, m->bg_color, training ? 0 : 1,
                                                  training ? ws + L.w[lf] : nullptr, o_rgb, o_depth, o_acc, o_sem, st));
  return rc;
}

}  // namespace

extern "C" int64_t cnb_render_workspace_floats(const cnb_model* m, int64_t num_rays, int32_t training) {
  if (!m || num_rays <= 0) return 0;
  Layout L;
  if (make_layout(m, num_rays, training != 0, L)) return 0;
  return L.total;
}

extern "C" int cnb_render_rays(const cnb_model* m, const cnb_rays* rays, const cnb_ray_outputs* out, float* workspace, cnb_stream_t stream) {
  int rc = check_common(m, rays, workspace);
  if (rc) return rc;
  if (rays->num_rays == 0) return CNB_OK;
  Layout L;
  if ((rc = make_layout(m, rays->num_rays, false, L))) return rc;
  return forward_chain(m, rays, L, workspace, false, nullptr, 1.0f, out, stream);
}

extern "C" int cnb_train_step(const cnb_model* m, const cnb_rays* rays, const cnb_train_cfg* cfg, const cnb_ray_outputs* out, float* losses_out,
                              float* workspace, cnb_stream_t stream) {
  int rc = check_common(m, rays, workspace);
  if (rc) return rc;
  CNB_REQUIRE(cfg && cfg->image && cfg->fruit_mask && losses_out, "train_step: null cfg/image/fruit_mask/losses_out");
  const int64_t R = rays->num_rays;
  if (R == 0) return CNB_OK;
  Layout L;
  if ((rc = make_layout(m, R, true, L))) return rc;
  float* ws = workspace;
  const bool mixed = m->field.precision == CNB_PREC_MIXED;
  const bool mixed_wide = mixed && !cnb_field_mixed_supported(&m->field);   // the layer-by-layer tensor-core path (big / huge presets)
  CNB_REQUIRE(cfg->phase >= 0 && cfg->phase <= 4, "train_step: phase %d outside 0..4", cfg->phase);
  CNB_REQUIRE(cfg->num_opt_groups >= 0 && cfg->num_opt_groups <= CNB_MAX_OPT_GROUPS, "train_step: num_opt_groups %d outside 0..%d", cfg->num_opt_groups, CNB_MAX_OPT_GROUPS);
  // ---- camera optimizer inside the step (row a17): rays are corrected by cnb_camera_opt_apply before the samplers, the kernels return
  // dLoss/d(corrected rays) and cnb_camera_opt_bwd turns that into the pose-adjustment gradient (camera_opt.cu) ----------------------
  const bool camopt = cfg->pose_adjustment != nullptr;
  const float* const cfg_orig_directions = rays->directions;   // dR is contracted with the UNcorrected directions
  cnb_rays adjusted = *rays;
  float* d_origins = cfg->d_origins;
  float* d_directions = cfg->d_directions;
  if (camopt) {
    CNB_REQUIRE(cfg->d_pose_adjustment && cfg->camopt_scratch && cfg->num_cameras >= 1 && rays->camera_indices, "train_step: camera optimizer needs d_pose_adjustment, camopt_scratch, num_cameras and camera indices");
    CNB_REQUIRE(cfg->phase == 0 || cfg->phase == 3 || cfg->phase == 4, "train_step: the camera optimizer is combined with phase 0 or 3/4 only");
    CNB_REQUIRE(cfg->d_origins == nullptr, "train_step: d_origins / d_directions are internal when the camera optimizer is inside the step");
    float* sc = cfg->camopt_scratch;   // [R,3] origins', [R,3] directions', [R,3] d_origins', [R,3] d_directions', [C,12] per-camera accumulators
    adjusted.origins = sc; adjusted.directions = sc + 3 * R;
    d_origins = sc + 6 * R; d_directions = sc + 9 * R;
    if (cfg->phase != 4) {
      if ((rc = cnb_camera_opt_apply(cfg->pose_adjustment, rays->camera_indices, rays->origins, rays->directions, R, cfg->num_cameras, sc, sc + 3 * R, stream))) return rc;
      if (cudaMemsetAsync(d_origins, 0, sizeof(float) * 6 * (size_t)R, stream) != cudaSuccess) return cnb_check_launch("train_step camopt memset");
    }
    rays = &adjusted;
  }
  const bool rays_grad = d_origins != nullptr;
  CNB_REQUIRE(!rays_grad || (d_directions != nullptr && m->ray_gradients), "train_step: ray gradients need d_directions and cnb_model.ray_gradients (workspace scratch)");
  const bool first = cfg->phase != 2, second = cfg->phase != 1;
  if (first) {
    if (cfg->phase != 4 && cudaMemsetAsync(losses_out, 0, 8 * sizeof(float), stream) != cudaSuccess) return cnb_check_launch("train_step memset");
    // on proposal-update steps the proposal forward keeps its encoded features for the backward (no second gather pass)
    const int part = cfg->phase == 3 ? 1 : (cfg->phase == 4 ? 2 : 0);
    if ((rc = forward_chain(m, rays, L, ws, true, cfg->jitter, cfg->anneal, out, stream, cfg->update_proposals != 0 && !rays_grad, part))) return rc;
    if (cfg->phase == 3) return CNB_OK;  // samplers + proposal forward only: the caller continues with phase 4 on the same workspace
  }
  const int lf = L.levels - 1, Sf = L.S[lf];
  const float gs = cfg->grad_scale == 0.0f ? 1.0f : cfg->grad_scale;
  const float* o_rgb = (out && out->rgb) ? out->rgb : ws + L.o_rgb;
  const float* o_sem = (out && out->semantics) ? out->semantics : ws + L.o_sem;
  // The backward splits into two independent chains after the forward: (A) pixel losses -> renderers -> field MLPs -> field table,
  // (B) interlevel loss -> proposal networks.  They share only read-only inputs (weights / samples of the forward) and write different
  // gradient tables, so with phase == 0 chain B is forked onto a side stream (event fork / join: still ONE stream-ordered call for the
  // caller, and capturable as two parallel branches of a CUDA graph).  Neither chain fills the GPU on its own (the field-MLP backward is a
  // latency-bound persistent kernel at 8 warps/SM, the per-ray kernels are one thin wave at 4096 rays); CNB_TRAIN_NO_OVERLAP=1 keeps them serial.
  // (ray gradients are atomically accumulated per ray by all three chains, and every proposal level has its own d(features) scratch: the fork
  // is as legal with them as without; callers that hand in their own d_origins keep the serial order they were tested with)
  ForkState* fk = ((cfg->phase == 0 || cfg->phase == 4) && (!rays_grad || camopt) && !g_prof_on) ? fork_state(stream) : nullptr;
  const bool overlap = fk != nullptr && stream_after(fk->side[0], stream, fk->fork);
  auto optimise = [&](int chain, cudaStream_t st) -> int {
    int rc = CNB_OK;
    for (int i = 0; i < cfg->num_opt_groups; ++i) {
      const cnb_opt_group& og = cfg->opt_groups[i];
      if (og.chain != chain) continue;
      if (og.peer_comm != nullptr)  // data parallel over peer memory: the group's whole exchange on this chain's branch
        STAGE(chain == CNB_CHAIN_FIELD ? "exchange_fields" : "exchange_proposals", 3, cnb_ddp_exchange_dev(og.peer_comm, og.peer_group, og.exp_avg, og.exp_avg_sq,
                                                                                                          og.grad, og.n, og.scalars, og.peer_flags, og.peer_channel, st));
      else
        STAGE(chain == CNB_CHAIN_FIELD ? "adam_fields" : "adam_proposals", 1, cnb_adam_step_zero_dev_live(og.param, og.grad, og.exp_avg, og.exp_avg_sq, og.n, og.scalars, og.live, st));
      if (rc) return rc;
    }
    return rc;
  };
  auto chain_field = [&](cudaStream_t st) -> int {
    int rc;
    // ---- losses + backward of the final level: MSE / BCE gradients -> renderers -> get_weights, one kernel (fruit_nerf.py:601-608) ----
    STAGE("final_composite_bwd", 1, cnb_final_composite_bwd(ws + L.dens[lf], ws + L.rgb, ws + L.sem, ws + L.eu[lf], ws + L.w[lf], o_rgb, o_sem, cfg->image,
                                                            cfg->fruit_mask, R, Sf, m->bg_mode, m->bg_color, cfg->semantic_loss_weight, gs,
                                                            m->field.pass_semantic_gradients, losses_out, ws + L.d_dens[lf], ws + L.d_rgb, ws + L.d_sem, st));
    if (rc) return rc;
    const cnb_samples sm = make_samples(rays, ws + L.eu[lf], Sf);
    if (rays_grad) STAGE("field_bwd", mixed_wide ? cnb_field_mixed_wide_launches(&m->field, true, true) : (mixed ? 3 : 9), cnb_field_bwd_rays(&m->field, &sm, ws + L.d_dens[lf], ws + L.d_rgb, ws + L.d_sem, nullptr, ws + L.ctx,
                                                                        d_origins, d_directions, st));
    else STAGE("field_bwd", mixed_wide ? cnb_field_mixed_wide_launches(&m->field, true, false) : (mixed ? 2 : 8), cnb_field_bwd(&m->field, &sm, ws + L.d_dens[lf], ws + L.d_rgb, ws + L.d_sem, nullptr, ws + L.ctx, st));
    if (rc) return rc;
    return optimise(CNB_CHAIN_FIELD, st);  // the field gradient is complete: its Adam pass overlaps the proposal chain
  };
  // one proposal level: interlevel loss (fruit_nerf.py:610) and, on "updated" steps, its backward into that proposal network
  auto proposal_level = [&](int lv, cudaStream_t st) -> int {
    int rc;
    const int S = L.S[lv];
    STAGE("interlevel", 1, cnb_interlevel_fused(ws + L.sp[lf], ws + L.w[lf], ws + L.sp[lv], ws + L.w[lv], ws + L.dens[lv], ws + L.eu[lv], R, Sf, S,
                                                gs * cfg->interlevel_loss_mult, losses_out + 2, cfg->update_proposals ? ws + L.d_dens[lv] : nullptr, st));
    if (rc) return rc;
    if (cfg->update_proposals) {
      const cnb_samples sm = make_samples(rays, ws + L.eu[lv], S);
      // every level has its OWN d(features) scratch: the two levels back-propagate on concurrent branches (handing both the first level's
      // buffer was the "7 % off, unexplained" pose gradient of the two-branch order: a plain race on that scratch)
      if (rays_grad) STAGE(lv == 0 ? "proposal0_bwd" : "proposal1_bwd", 2, cnb_density_field_bwd_rays(&m->proposal[lv], &sm, ws + L.d_dens[lv], ws + L.pg_level[lv],
                                                                                                     d_origins, d_directions, st));
      else if (L.pfeat[lv] >= 0) STAGE(lv == 0 ? "proposal0_bwd" : "proposal1_bwd", 1, cnb_density_field_bwd_kept(&m->proposal[lv], &sm, ws + L.d_dens[lv], ws + L.pfeat[lv], st));
      else STAGE(lv == 0 ? "proposal0_bwd" : "proposal1_bwd", 1, cnb_density_field_bwd(&m->proposal[lv], &sm, ws + L.d_dens[lv], st));
    }
    return rc;
  };
  auto proposals_tail = [&](cudaStream_t st) -> int {
    int rc = CNB_OK;
    if (cfg->interlevel_loss_mult != 1.0f) {
      k_scale<<<1, 32, 0, st>>>(losses_out + 2, 1, cfg->interlevel_loss_mult);
      if ((rc = cnb_check_launch("train_step scale"))) return rc;
    }
    if (cfg->want_metrics) {
      STAGE("distortion", 1, cnb_distortion_fwd(ws + L.sp[lf], ws + L.w[lf], R, Sf, losses_out + 3, st));
      if (rc) return rc;
    }
    return optimise(CNB_CHAIN_PROPOSALS, st);
  };
  auto chain_proposals = [&](cudaStream_t st) -> int {
    int rc = CNB_OK;
    for (int lv = 0; lv < lf; ++lv)
      if ((rc = proposal_level(lv, st))) return rc;
    return proposals_tail(st);
  };
  if (overlap) {
    // three branches: field chain on the caller's stream; proposal level 0 on side[0]; proposal level 1 on side[1] (the two proposal networks
    // are independent: each only needs its own interlevel gradient; the level-1 backward is a short, latency-bound kernel that fills the gaps
    // of the level-0 one); side[1] joins side[0] before the proposal group's tail (loss scaling, metrics, Adam), side[0] joins the caller's stream
    cudaStream_t s0 = fk->side[0], s1 = fk->side[1];
    bool two = lf >= 2 && cfg->update_proposals && stream_after(s1, stream, fk->fork2);
    rc = proposal_level(0, s0);
    if (lf >= 2) { const int r1 = proposal_level(1, two ? s1 : s0); if (!rc) rc = r1; }
    bool joined = true;
    if (two) joined = stream_after(s0, s1, fk->join[1]);
    if (!rc) rc = proposals_tail(s0);
    const int rc2 = chain_field(stream);
    joined = stream_after(stream, s0, fk->join[0]) && joined;  // always join, even after a failed launch
    if (!joined) { cnb_set_error("train_step: stream join failed"); return CNB_ERR_CUDA; }
    if (rc || rc2) return rc ? rc : rc2;
  } else {
    if (first && (rc = chain_field(stream))) return rc;
    if (!second) return CNB_OK;
    if ((rc = chain_proposals(stream))) return rc;
  }
  if (camopt) {
    // all three chains have joined: every ray's gradient is complete
    cudaStream_t st = stream;
    STAGE("camera_opt_bwd", 3, cnb_camera_opt_bwd(cfg->pose_adjustment, rays->camera_indices, cfg_orig_directions, d_origins,
                                                  d_directions, R, cfg->num_cameras, cfg->trans_l2_penalty, cfg->rot_l2_penalty, gs, cfg->camopt_scratch + 12 * R,
                                                  cfg->d_pose_adjustment, losses_out + 6, stream));
    if (rc) return rc;
    for (int i = 0; i < cfg->num_opt_groups; ++i) {
      const cnb_opt_group& og = cfg->opt_groups[i];
      if (og.chain != CNB_CHAIN_JOIN) continue;
      STAGE("adam_camera_opt", 1, cnb_adam_step_zero_dev_live(og.param, og.grad, og.exp_avg, og.exp_avg_sq, og.n, og.scalars, og.live, stream));
      if (rc) return rc;
    }
  }
  k_finalize_losses<<<1, 32, 0, stream>>>(losses_out);
  return cnb_check_launch("train_step finalize");
}

// ---- optional stage profiling ---------------------------------------------------------------------------------------------
extern "C" void cnb_profile_enable(int32_t on) {
  for (auto& e : g_prof) { cudaEventDestroy(e.e0); cudaEventDestroy(e.e1); }
  g_prof.clear();
  g_prof_on = on != 0;
}

// Synchronises the device, sums the recorded stages by name and writes "name:calls:kernels:ms;..." into buf; clears the log.
extern "C" int cnb_profile_read(char* buf, int32_t buflen) {
  if (!buf || buflen <= 0) return CNB_ERR_ARG;
  if (cudaDeviceSynchronize() != cudaSuccess) return cnb_check_launch("profile_read");
  struct Acc { std::string name; int calls; int kernels; double ms; };
  std::vector<Acc> acc;
  for (auto& e : g_prof) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e.e0, e.e1);
    cudaEventDestroy(e.e0); cudaEventDestroy(e.e1);
    bool found = false;
    for (auto& a : acc) if (a.name == e.name) { a.calls++; a.kernels += e.kernels; a.ms += ms; found = true; break; }
    if (!found) acc.push_back({e.name, 1, e.kernels, ms});
  }
  g_prof.clear();
  std::string out;
  char tmp[160];
  for (auto& a : acc) { snprintf(tmp, sizeof(tmp), "%s:%d:%d:%.6f;", a.name.c_str(), a.calls, a.kernels, a.ms); out += tmp; }
  if ((int)out.size() + 1 > buflen) return CNB_ERR_ARG;
  memcpy(buf, out.c_str(), out.size() + 1);
  return CNB_OK;
}
