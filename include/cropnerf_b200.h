/*
 * cropnerf_b200.h -- C ABI of the B200-native per-ray rendering hot path of FruitNeRF / CropNeRF.
 *
 * The reference (robotic-vision-lab/CropNeRF, /root/reference) is pure Python on top of nerfstudio 1.1.3; it
 * has no FFI of its own.  The entry points below are what a binding for this path would call: one per
 * nerfstudio primitive the reference imports (cited per function, paths relative to
 * /root/reference/crop_nerf/fruit_nerf unless prefixed "nerfstudio/").  INTEGRATION.md shows the ctypes
 * stubs a maintainer adds on the reference side.
 *
 * Conventions
 *  - plain pointers + sizes only; every pointer is DEVICE memory owned by the caller unless stated; the
 *    library never allocates persistent memory and never frees caller memory;
 *  - all work is enqueued on `stream` (no hidden syncs, graph-capturable); stateless and re-entrant (two documented exceptions keep a
 *    per-device side stream + events: cnb_train_step's forked backward chains and cnb_ddp_optimizer_step's deferred exchange);
 *  - return 0 on success, negative cnb_status otherwise; cnb_last_error() gives the thread-local message;
 *  - tensors are contiguous row-major fp32 unless stated; "[R,S]" sample arrays may carry a row stride so
 *    that bin-edge arrays [R,S+1] can be passed as starts (=edges) and ends (=edges+1) without copies;
 *  - gradient pointers inside descriptor structs are ACCUMULATED into (caller zeroes them per step).
 *  - there is no CPU fallback: without a CUDA device every compute entry returns CNB_ERR_CUDA.
 */
#ifndef CROPNERF_B200_H
#define CROPNERF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CNB_VERSION 100
#define CNB_MAX_LEVELS 16
#define CNB_MAX_LAYERS 4
#define CNB_MAX_WIDTH 64        /* widest layer of the fused (shared-memory resident) MLP operators */
#define CNB_WIDE_MAX_WIDTH 256  /* wider MLPs (the _big / _huge presets) run layer by layer in exact fp32: csrc/mlp_wide.cu */

typedef struct CUstream_st* cnb_stream_t;

typedef enum cnb_status {
  CNB_OK = 0,
  CNB_ERR_ARG = -1,         /* bad argument / unsupported configuration */
  CNB_ERR_CUDA = -2,        /* CUDA runtime error (message in cnb_last_error) */
  CNB_ERR_UNSUPPORTED = -3  /* configuration outside the compiled specialisations */
} cnb_status;

enum { CNB_PREC_FP32 = 0, CNB_PREC_MIXED = 1 };          /* MLP arithmetic: fp32 FFMA / fp16 tensor cores, fp32 accumulate */
enum { CNB_ACT_NONE = 0, CNB_ACT_RELU = 1, CNB_ACT_SIGMOID = 2 };
enum { CNB_WARP_AABB = 0, CNB_WARP_CONTRACT_LINF = 1 }; /* position normalisation (fruit_field.py:171-176) */
enum { CNB_SPACING_UNIFORM = 0, CNB_SPACING_LINDISP_PIECEWISE = 1 };
enum { CNB_BG_NONE = 0, CNB_BG_LAST_SAMPLE = 1, CNB_BG_CONSTANT = 2 };
enum { CNB_APP_PER_CAMERA = 0, CNB_APP_MEAN = 1, CNB_APP_ZERO = 2 }; /* fruit_field.py:251-261, 219-221 */

/* Multiresolution hash grid == nerfstudio/field_components/encodings.py HashEncoding (ctor: fruit_field.py:125-132;
 * proposal grids: fruit_nerf.py:124-141).  table row index = hash(level corner) + level * 2^log2_hashmap_size. */
typedef struct cnb_grid {
  const float* table;        /* [num_levels * 2^log2_hashmap_size, 2] */
  float* d_table;            /* same shape, accumulated by *_bwd; may be NULL for forward-only use */
  int32_t num_levels;        /* 1..CNB_MAX_LEVELS */
  int32_t log2_hashmap_size; /* <= 24 */
  float scalings[CNB_MAX_LEVELS]; /* floor(min_res * growth^level) evaluated in fp32 by the host (top field level = 2047) */
} cnb_grid;

/* nn.Linear stack == nerfstudio/field_components/mlp.py MLP torch path (fruit_field.py:133-141,146-154,159-167);
 * ReLU between layers, out_activation after the last.  W[l] is [dims[l+1], dims[l]] row-major (nn.Linear.weight). */
typedef struct cnb_mlp {
  int32_t num_layers;                 /* 1..CNB_MAX_LAYERS */
  int32_t dims[CNB_MAX_LAYERS + 1];   /* in, hidden..., out ; each <= CNB_WIDE_MAX_WIDTH (fused kernels up to CNB_MAX_WIDTH) */
  int32_t out_activation;             /* CNB_ACT_* */
  int32_t _pad;
  const float* W[CNB_MAX_LAYERS];
  const float* b[CNB_MAX_LAYERS];
  float* dW[CNB_MAX_LAYERS];          /* accumulated by *_bwd; NULL entries are skipped */
  float* db[CNB_MAX_LAYERS];
} cnb_mlp;

/* world position -> unit cube (fruit_field.py:171-180; nerfstudio/fields/density_fields.py get_density) */
typedef struct cnb_warp {
  int32_t mode;        /* CNB_WARP_* ; CONTRACT_LINF: x' = (contract(x) + 2) / 4 ; AABB: (x - min) / (max - min) */
  float aabb_min[3];
  float aabb_max[3];
} cnb_warp;

/* Ray samples == nerfstudio/cameras/rays.py RaySamples/Frustums restricted to what the field reads.
 * position(r,s) = origins[r] + directions[r] * (starts[r,s] + ends[r,s]) / 2 . */
typedef struct cnb_samples {
  const float* origins;          /* [R,3] */
  const float* directions;       /* [R,3] */
  const float* starts;           /* element (r,s) at starts[r*row_stride + s] */
  const float* ends;             /* same addressing */
  const int32_t* camera_indices; /* [R] or NULL */
  int64_t num_rays;
  int64_t row_stride;
  int32_t samples_per_ray;
  int32_t _pad;
} cnb_samples;

/* HashMLPDensityField (nerfstudio/fields/density_fields.py; built fruit_nerf.py:118-142) */
typedef struct cnb_density_field {
  cnb_grid grid;
  cnb_mlp mlp;               /* 2L -> hidden -> 1 (hidden <= 64), or a single Linear when use_linear */
  cnb_warp warp;
  float average_init_density;
  int32_t precision;         /* CNB_PREC_FP32 (0): exact gradients; CNB_PREC_MIXED: MLP parameter gradients contracted with bf16 operands */
} cnb_density_field;

/* FruitField (fruit_field.py:44-302) */
typedef struct cnb_field {
  cnb_grid grid;
  cnb_mlp base;              /* 2L -> 64 -> 1+geo     (fruit_field.py:133-141) */
  cnb_mlp sem;               /* geo -> 64 -> 64        (fruit_field.py:146-154) */
  cnb_mlp sem_head;          /* 64 -> 1                (components/field_heads.py:29-40, fruit_field.py:155-157) */
  cnb_mlp rgb;               /* 16+geo+app -> 64 -> 64 -> 3, sigmoid (fruit_field.py:159-167) */
  const float* embedding;    /* [num_images, appearance_dim] (fruit_field.py:106) */
  float* d_embedding;        /* accumulated (per-camera mode only); may be NULL */
  const float* mean_embedding; /* [appearance_dim], required for CNB_APP_MEAN */
  cnb_warp warp;
  int32_t num_images;
  int32_t appearance_dim;    /* 32 */
  int32_t geo_feat_dim;      /* 15 */
  int32_t appearance_mode;   /* CNB_APP_* */
  int32_t pass_semantic_gradients; /* fruit_field.py:264-266 */
  int32_t precision;         /* CNB_PREC_* */
} cnb_field;

int cnb_version(void);
const char* cnb_last_error(void);
/* number of CUDA devices visible, or a negative status; never throws */
int cnb_device_count(void);

/* ---- a2: HashEncoding.pytorch_fwd / its autograd (nerfstudio encodings.py; constructed fruit_field.py:125-132, and inside
 *      HashMLPDensityField fruit_nerf.py:124-141; called fruit_field.py:181-182) ------------------------------------------------ */
/* positions [n,3] in [0,1]; out [n, 2*L]; indices (optional) [n, L, 8] int32 table rows in h0..h7 order */
int cnb_hashgrid_fwd(const cnb_grid* g, const float* positions, int64_t n, float* out, int32_t* indices, cnb_stream_t stream);
/* accumulates g->d_table from d_out [n, 2*L] */
int cnb_hashgrid_bwd(const cnb_grid* g, const float* positions, const float* d_out, int64_t n, cnb_stream_t stream);
/* fp16 table rows (fruit_nerf_big / _huge with table_precision="fp16"): table_half [num_levels * 2^log2_hashmap_size] __half2 (8-byte aligned)
 * is gathered instead of g->table; each corner is widened to fp32 and blended as in cnb_hashgrid_fwd, so the result equals cnb_hashgrid_fwd on a
 * table holding table_half's values.  table_half NULL = cnb_hashgrid_fwd. */
int cnb_hashgrid_fwd_half(const cnb_grid* g, const void* table_half, const float* positions, int64_t n, float* out, int32_t* indices,
                          cnb_stream_t stream);
/* table_half[i] = __float2half_rn(table[i]) for n floats (n % 4 == 0; table 16-byte, table_half 8-byte aligned).  live (optional) = a flat
 * group's bitmap (cnb_hashgrid_mark_reachable) with the table at unit first_unit: only units whose bit is set are written. */
int cnb_table_to_half(const float* table, int64_t n, const uint32_t* live, int64_t first_unit, void* table_half, cnb_stream_t stream);

/* ---- a3/a4: MLP / FieldHead (nerfstudio mlp.py, field_heads.py; fruit_field.py:133-141,146-154,159-167;
 *      SemanticFieldHead components/field_heads.py:29-40, used fruit_field.py:155-157,207,269) ---------------------------------- */
/* floats of `hidden` needed per sample when training (sum of hidden widths) */
int64_t cnb_mlp_hidden_floats(const cnb_mlp* m);
/* x: element (i,k) at x[i*x_stride+k]; y [n, out] dense; hidden (optional, for bwd) [sum_l n*width_l] */
int cnb_mlp_fwd(const cnb_mlp* m, const float* x, int64_t x_stride, int64_t n, float* y, float* hidden, cnb_stream_t stream);
/* y is the forward output (needed for sigmoid'); dx optional, element (i,k) at dx[i*dx_stride+k] (overwritten) */
int cnb_mlp_bwd(const cnb_mlp* m, const float* x, int64_t x_stride, const float* hidden, const float* y, const float* dy,
                int64_t n, float* dx, int64_t dx_stride, cnb_stream_t stream);

/* ---- a3 in mixed precision for layers up to 128 wide (nerfstudio MLP, fruit_field.py:133-167 at the widths of the fruit_nerf_big /
 *      fruit_nerf_huge presets): tcgen05 tensor cores, fp16 forward operands, bf16 gradient operands, fp32 accumulation
 *      (csrc/mlp_mixed.cu).  Every width must be 1..128; other shapes return CNB_ERR_UNSUPPORTED with the shape in cnb_last_error.
 *      Nothing is allocated inside: `scratch` holds the forward's kept activations (training) and the backward's work space, so the calls
 *      are graph-capturable and independent across streams when each stream has its own scratch. */
/* floats of `scratch` for n rows; training = 1: what a forward(training=1) + backward pair needs, 0: a forward alone */
int64_t cnb_mlp_mixed_scratch_floats(const cnb_mlp* m, int64_t n, int32_t training);
/* as cnb_mlp_fwd; training = 1 keeps the hidden activations in scratch for cnb_mlp_mixed_bwd */
int cnb_mlp_mixed_fwd(const cnb_mlp* m, const float* x, int64_t x_stride, int64_t n, float* y, float* scratch, int32_t training,
                      cnb_stream_t stream);
/* as cnb_mlp_bwd; scratch = the one the forward(training=1) of the same x / n wrote; dW / db accumulated */
int cnb_mlp_mixed_bwd(const cnb_mlp* m, const float* x, int64_t x_stride, const float* y, const float* dy, int64_t n, float* dx,
                      int64_t dx_stride, float* scratch, cnb_stream_t stream);

/* ---- a7: HashMLPDensityField.get_density / density_fn (nerfstudio density_fields.py; built fruit_nerf.py:118-142,
 *      handed to the sampler as density_fns fruit_nerf.py:143-145,549) ----------------------------------------------------------- */
/* density [R*S]; positions_out (optional) [R*S,3] normalised+masked positions */
int cnb_density_field_fwd(const cnb_density_field* f, const cnb_samples* s, float* density, float* positions_out, cnb_stream_t stream);
/* recomputes the forward per sample; accumulates grid.d_table, mlp.dW/db */
int cnb_density_field_bwd(const cnb_density_field* f, const cnb_samples* s, const float* d_density, cnb_stream_t stream);
/* Same pair for callers that run forward and backward of ONE batch back to back (cnb_train_step on proposal-update steps): the
 * forward also writes the encoded features, level-major [num_levels][N] float2 (N = num_rays * samples_per_ray; 2*num_levels*N
 * floats), and the backward reads them instead of gathering the table a second time.  Bit-identical gradients.
 * cnb_density_field_kept_supported: 1 when the architecture has the kept-feature backward (<= 7 levels, MLP 2L->16->1). */
int cnb_density_field_fwd_keep(const cnb_density_field* f, const cnb_samples* s, float* density, float* features_keep, cnb_stream_t stream);
int cnb_density_field_bwd_kept(const cnb_density_field* f, const cnb_samples* s, const float* d_density, const float* features_kept,
                               cnb_stream_t stream);
int cnb_density_field_kept_supported(const cnb_density_field* f);

/* ---- a1/a5/a6: FruitField.forward (fruit_field.py:284-302) = get_density (:169-194) + get_outputs (:235-282) /
 *      get_inference_outputs (:196-233); called fruit_nerf.py:340,431,480,503,551 ---------------------------------------------- */
/* floats of `ctx` scratch per call (activations kept for backward + backward scratch); 0 => ctx may be NULL */
int64_t cnb_field_ctx_floats(const cnb_field* f, int64_t n, int32_t training);
/* outputs (each optional except density): density [N], geo [N,1+geo] (col 0 = pre-activation density),
 * rgb [N,3], sem [N], positions_out [N,3] (= FruitField._sample_locations) */
int cnb_field_fwd(const cnb_field* f, const cnb_samples* s, float* density, float* geo, float* rgb, float* sem,
                  float* positions_out, float* ctx, int32_t training, cnb_stream_t stream);
/* d_geo (optional) [N,1+geo] external gradient on the geo embedding; accumulates all parameter gradients */
int cnb_field_bwd(const cnb_field* f, const cnb_samples* s, const float* d_density, const float* d_rgb, const float* d_sem,
                  const float* d_geo, float* ctx, cnb_stream_t stream);
/* cnb_field_fwd gathering the fp16 copy of f->grid.table (see cnb_hashgrid_fwd_half); table_half NULL = cnb_field_fwd.  Compiled for
 * precision CNB_PREC_MIXED on the layer-by-layer path only (MLPs outside the fused base kernels); elsewhere CNB_ERR_UNSUPPORTED.  The backward
 * (cnb_field_bwd) reads no table; cnb_field_bwd_rays_half differentiates the same fp16 rows. */
int cnb_field_fwd_half(const cnb_field* f, const void* table_half, const cnb_samples* s, float* density, float* geo, float* rgb, float* sem,
                       float* positions_out, float* ctx, int32_t training, cnb_stream_t stream);

/* ---- a17: gradient with respect to the rays (camera optimizer, fruit_nerf.py:114-116,547,614) ---------------------- */
/* d_feat [N, 2L] = gradient reaching a grid's encoded features; accumulates d_origins / d_directions [R,3]:
 * trilinear-offset derivative of every level -> selector mask -> normalisation / SceneContraction Jacobian -> sum over the ray */
int cnb_position_grad_rays(const cnb_grid* g, const cnb_warp* warp, const cnb_samples* s, const float* d_feat, float* d_origins,
                           float* d_directions, cnb_stream_t stream);
/* cnb_density_field_bwd + ray gradients; scratch: R*S*2L floats */
int cnb_density_field_bwd_rays(const cnb_density_field* f, const cnb_samples* s, const float* d_density, float* scratch, float* d_origins,
                               float* d_directions, cnb_stream_t stream);
/* cnb_field_bwd + ray gradients (the SH direction encoding carries no gradient, as in nerfstudio's torch SHEncoding) */
int cnb_field_bwd_rays(const cnb_field* f, const cnb_samples* s, const float* d_density, const float* d_rgb, const float* d_sem,
                       const float* d_geo, float* ctx, float* d_origins, float* d_directions, cnb_stream_t stream);
/* the two with the fp16 table copy the forward gathered (cnb_field_fwd_half) */
int cnb_position_grad_rays_half(const cnb_grid* g, const void* table_half, const cnb_warp* warp, const cnb_samples* s, const float* d_feat,
                                float* d_origins, float* d_directions, cnb_stream_t stream);
int cnb_field_bwd_rays_half(const cnb_field* f, const void* table_half, const cnb_samples* s, const float* d_density, const float* d_rgb,
                            const float* d_sem, const float* d_geo, float* ctx, float* d_origins, float* d_directions, cnb_stream_t stream);

/* ---- a8/a9: samplers (nerfstudio ray_samplers.py; components/ray_samplers.py:54-104) ----------------------- */
/* SpacedSampler: lin_bins = torch.linspace(0,1,S+1) supplied by the host (bit-exact u); t_rand NULL (eval) or
 * [R*rand_stride] with rand_stride 1 (single_jitter) or S+1.  Outputs spacing/euclid bin edges [R,S+1]. */
int cnb_sample_spaced(const float* nears, const float* fars, const float* lin_bins, const float* t_rand, int32_t rand_stride,
                      int32_t spacing, int64_t R, int32_t S, float* spacing_bins, float* euclid_bins, cnb_stream_t stream);
/* the same with nerfstudio's NearFarCollider folded in (fruit_nerf.py:167): ray_nears / ray_fars [R] when the bundle carries them (AABB-clipped
 * projection rays), else the two planes; the values used are written to nears_out / fars_out [R] for the PDF resampling levels */
int cnb_sample_spaced_collide(const float* ray_nears, const float* ray_fars, float near_plane, float far_plane, const float* lin_bins,
                              const float* t_rand, int32_t rand_stride, int32_t spacing, int64_t R, int32_t S, float* nears_out, float* fars_out,
                              float* spacing_bins, float* euclid_bins, cnb_stream_t stream);
/* PDFSampler(include_original=False): weights [R,Sp] (raised to `anneal` in-kernel), prev spacing bins [R,Sp+1];
 * u_base = torch.linspace(0, 1-1/(S+1), S+1) from the host; rand NULL (eval: + 1/(2(S+1))) or [R*rand_stride];
 * inds (optional) [R,S+1] int32 = searchsorted(cdf,u,right). */
int cnb_sample_pdf(const float* weights, float anneal, const float* prev_spacing_bins, const float* nears, const float* fars,
                   int32_t spacing, const float* u_base, const float* rand, int32_t rand_stride, int64_t R, int32_t Sp, int32_t S,
                   float histogram_padding, float eps, float* spacing_bins, float* euclid_bins, int32_t* inds, cnb_stream_t stream);

/* ---- a10: RaySamples.get_weights (nerfstudio rays.py; called fruit_nerf.py:556,508,442,341 and inside the proposal sampler) */
int cnb_weights_fwd(const float* density, const float* starts, const float* ends, int64_t row_stride, int64_t R, int32_t S,
                    float* weights, cnb_stream_t stream);
int cnb_weights_bwd(const float* density, const float* starts, const float* ends, int64_t row_stride, int64_t R, int32_t S,
                    const float* d_weights, float* d_density, cnb_stream_t stream);

/* ---- a11-a14: RGB / Depth(median) / Accumulation / Semantic renderers (nerfstudio renderers.py; built fruit_nerf.py:170-174,
 *      called :560-591, :512-520, :446-452; background_color_override_context scripts/semantic_projection.py:51,169) ------------ */
/* Any of rgb/sem inputs and outputs may be NULL (that renderer is skipped).  eval_mode: nan_to_num(rgb) in, clamp out.
 * median_index (optional) [R] int32. */
int cnb_render_fwd(const float* weights, const float* rgb, const float* sem, const float* starts, const float* ends,
                   int64_t row_stride, int64_t R, int32_t S, int32_t bg_mode, const float* bg_color, int32_t eval_mode,
                   float* rgb_out, float* depth_out, float* acc_out, float* sem_out, int32_t* median_index, cnb_stream_t stream);
/* d_weights gets d(rgb,acc[,sem if sem_weight_grad]) ; d_rgb [R,S,3]; d_sem [R,S]; NULL outputs skipped */
int cnb_render_bwd(const float* weights, const float* rgb, const float* sem, int64_t R, int32_t S, int32_t bg_mode,
                   const float* bg_color, const float* d_rgb_out, const float* d_acc_out, const float* d_sem_out,
                   int32_t sem_weight_grad, float* d_weights, float* d_rgb, float* d_sem, cnb_stream_t stream);

/* ---- a16: losses (nerfstudio losses.py interlevel_loss / distortion_loss; fruit_nerf.py:601-615,639-645) --- */
/* loss_out[0] += sum_r mean-normalised lossfun_outer ; c [R,Sc+1], w [R,Sc] (final level, detached); cp/wp proposal */
int cnb_interlevel_fwd(const float* c, const float* w, const float* cp, const float* wp, int64_t R, int32_t Sc, int32_t Sp,
                       float* loss_out, cnb_stream_t stream);
/* d_wp [R,Sp] overwritten with grad_scale * dLoss/dwp */
int cnb_interlevel_bwd(const float* c, const float* w, const float* cp, const float* wp, int64_t R, int32_t Sc, int32_t Sp,
                       float grad_scale, float* d_wp, cnb_stream_t stream);
int cnb_distortion_fwd(const float* c, const float* w, int64_t R, int32_t S, float* loss_out, cnb_stream_t stream);
/* MSE(rgb) + weight*BCEWithLogits(sem) forward and gradients in one pass; losses_out[0]+=mse, [1]+=bce */
int cnb_pixel_losses(const float* rgb, const float* sem, const float* image, const float* mask, int64_t R, float sem_weight,
                     float grad_scale, float* losses_out, float* d_rgb, float* d_sem, cnb_stream_t stream);

/* ---- fused per-ray stages (csrc/fused_ray.cu): the same arithmetic as the per-primitive entries above, chained in one
 * warp-per-ray kernel per pipeline stage; results are bit-identical to calling the primitives one after the other ---- */
/* get_weights(density) -> DepthRenderer(median) [depth_out optional] -> PDFSampler to S bins; weights_out optional [R,Sp] */
int cnb_level_resample(const float* density, const float* euclid_bins_prev, const float* spacing_bins_prev, const float* nears,
                       const float* fars, int32_t spacing, float anneal, const float* u_base, const float* rand, int32_t rand_stride,
                       int64_t R, int32_t Sp, int32_t S, float histogram_padding, float eps, float* weights_out, float* depth_out,
                       float* spacing_bins, float* euclid_bins, int32_t* inds, cnb_stream_t stream);
/* get_weights -> RGB / accumulation / semantic / median-depth renderers of the final level (outputs optional) */
int cnb_final_composite(const float* density, const float* rgb, const float* sem, const float* euclid_bins, int64_t R, int32_t S,
                        int32_t bg_mode, const float* bg_color, int32_t eval_mode, float* weights_out, float* rgb_out, float* depth_out,
                        float* acc_out, float* sem_out, cnb_stream_t stream);
/* MSE + weighted BCE-with-logits (losses_out[0], [1] accumulated) and their gradients through the renderers and get_weights */
int cnb_final_composite_bwd(const float* density, const float* rgb, const float* sem, const float* euclid_bins, const float* weights,
                            const float* rgb_out, const float* sem_out, const float* image, const float* mask, int64_t R, int32_t S,
                            int32_t bg_mode, const float* bg_color, float sem_weight, float grad_scale, int32_t sem_weight_grad,
                            float* losses_out, float* d_density, float* d_rgb, float* d_sem, cnb_stream_t stream);
/* interlevel loss of one proposal level (loss_out[0] accumulated); d_density_p != NULL also runs its backward through
 * get_weights of that level and overwrites d_density_p [R,Sp] */
int cnb_interlevel_fused(const float* c, const float* w, const float* cp, const float* wp, const float* density_p, const float* euclid_bins_p,
                         int64_t R, int32_t Sc, int32_t Sp, float grad_scale, float* loss_out, float* d_density_p, cnb_stream_t stream);

/* ---- f1 ("next" row): ray generation + AABB clipping on the device (fruit_nerf.py:283-288) ------------------------------ */
/* nerfstudio Cameras.generate_rays for one perspective camera (without distortion; the *_lens entries add it) */
typedef struct cnb_camera {
  float c2w[12];   /* camera-to-world [3,4], row-major (OpenGL axes: +x right, +y up, camera looks down -z) */
  float fx, fy, cx, cy;
  int32_t width, height;
} cnb_camera;
/* Lens distortion of an OPENCV-style perspective camera, in the order of nerfstudio's camera_utils.get_distortion_params
 * (Cameras.distortion_params [..., 6]).  The *_lens entries undistort every normalised pixel coordinate (x, -y) -- the ray's and
 * both pixel-area offsets -- with camera_utils.radial_and_tangential_undistort (10 Newton steps, eps 1e-3, float32 in nerfstudio's
 * operation order) before forming the direction.  All six zero = no distortion (the solve is then the identity, bit for bit). */
typedef struct cnb_lens {
  float k1, k2, k3, k4, p1, p2;
} cnb_lens;
/* cam / aabb are HOST pointers (aabb = min xyz, max xyz; NULL = no clipping).  pixel_yx (device, optional) [n,2] integer pixel
 * rows/columns; NULL = every pixel of the image in row-major order (n = width*height).  Outputs (device): origins, directions
 * [n,3]; pixel_area [n] (optional); nears, fars [n] (with aabb: slab test, misses = 1e10 as nerfstudio's intersect_aabb);
 * valid_count (optional, device int32, ACCUMULATED) = rays that hit the box. */
int cnb_generate_rays(const cnb_camera* cam, const int32_t* pixel_yx, int64_t n, const float* aabb, float* origins, float* directions,
                      float* pixel_area, float* nears, float* fars, int32_t* valid_count, cnb_stream_t stream);
/* cnb_generate_rays with lens distortion: lens is a HOST pointer, NULL or all zero = cnb_generate_rays exactly. */
int cnb_generate_rays_lens(const cnb_camera* cam, const cnb_lens* lens, const int32_t* pixel_yx, int64_t n, const float* aabb, float* origins,
                           float* directions, float* pixel_area, float* nears, float* fars, int32_t* valid_count, cnb_stream_t stream);

/* ---- e2 / e3 / f1: the loop bodies of the two export workloads around the render call -------------------------------------- */
/* `ns-export pointcloud` (export/exporter_utils_nerfacto.py:153-176): point = origin + direction * depth; keep = (only_semantics ?
 * sigmoid(semantics) - threshold > 0 : true) && (obb ? OrientedBox.within(point) : true); kept points / colours / view directions are
 * appended IN RAY ORDER at out_*[*count_in ...]; *count_out = *count_in + kept (two distinct device counters, so the export loop chains
 * batches without a host round trip; entries past `capacity` are counted but not written).  obb: HOST pointer to 15 floats (R row-major
 * [3,3], T [3], S [3]) or NULL.  block_counts: device scratch of cnb_extract_points_scratch_ints(n) int32.  All other pointers device. */
int64_t cnb_extract_points_scratch_ints(int64_t n);
int cnb_extract_points(const float* origins, const float* directions, const float* depth, const float* semantics, const float* rgb, int64_t n,
                       const float* obb, int32_t only_semantics, float threshold, int32_t* block_counts, const int32_t* count_in,
                       int32_t* count_out, int64_t capacity, float* out_points, float* out_rgbs, float* out_dirs, cnb_stream_t stream);
/* fruit_nerf.py:281-288 for all `num_boxes` sub-cluster AABBs of a super-cluster in one pass over the camera's pixels: every (pixel, box)
 * hit of nerfstudio's intersect_aabb is appended (any order) to a compacted ray list -- origins, directions [cap,3], pixel_area, nears,
 * fars [cap], tags [cap] = box * width*height + pixel -- and counted in *count (device int32, ACCUMULATED; hits past `capacity` are counted,
 * not written).  cam: HOST pointer; boxes: DEVICE [num_boxes,6] (min xyz, max xyz). */
int cnb_generate_rays_boxes(const cnb_camera* cam, const float* boxes, int32_t num_boxes, int64_t capacity, float* origins, float* directions,
                            float* pixel_area, float* nears, float* fars, int32_t* tags, int32_t* count, cnb_stream_t stream);
/* cnb_generate_rays_boxes with lens distortion (see cnb_lens): each pixel's ray is undistorted before the slab tests, the pixel-area
 * offsets on its first hit.  lens: HOST pointer, NULL or all zero = cnb_generate_rays_boxes exactly. */
int cnb_generate_rays_boxes_lens(const cnb_camera* cam, const cnb_lens* lens, const float* boxes, int32_t num_boxes, int64_t capacity,
                                 float* origins, float* directions, float* pixel_area, float* nears, float* fars, int32_t* tags, int32_t* count,
                                 cnb_stream_t stream);
/* fruit_nerf.py:296-315: wo_occ[tag] = q(semantics), visible[tag] = front_opacity >= occlusion_threshold ? 0 : q(semantics), with
 * q(x) = uint8(clamp(x * 255 + 0.5, 0, 255)) (torchvision save_image); the two uint8 images [num_boxes, H*W] are cleared by the caller. */
int cnb_projection_scatter(const int32_t* tags, const float* semantics, const float* front_opacity, int64_t n, float occlusion_threshold,
                           uint8_t* wo_occ, uint8_t* visible, cnb_stream_t stream);
/* Volumetric export ray source (data/fruit_datamanager.py:71-120 sample_surface_points + components/ray_generators.py:46-66
 * OrthographicRayGenerator): rays first .. first+n of the nx x ny grid meshgrid(linspace(x0,x1,nx), linspace(y0,y1,ny), indexing="ij") on
 * the plane z, common direction (HOST pointer, 3 floats), nears = 0, fars = far.  Bit-equal to torch.linspace on the host. */
int cnb_volume_face_rays(float x0, float x1, int32_t nx, float y0, float y1, int32_t ny, float z, const float* direction, float far,
                         int64_t first, int64_t n, float* origins, float* directions, float* nears, float* fars, cnb_stream_t stream);

/* ---- f1, training side: FruitDataManager.next_train (data/fruit_datamanager.py:188-197) on the device ---------------------
 * = nerfstudio PixelSampler.sample (indices = (rand[R,3] * [N,H,W]).long(); value[c,y,x] of every per-pixel tensor) followed by
 * RayGenerator (image_coords[y,x] = pixel centre -> Cameras.generate_rays(camera_indices=c)).  All images of the split are resident
 * in device memory with one size (nerfstudio's PixelSampler assumes that too). */
typedef struct cnb_image_set {
  const uint8_t* images_u8;  /* device [N,H,W,3] uint8 (value / 255 = the float image of cotton_dataset.py), or NULL */
  const float* images_f32;   /* device [N,H,W,3] float32, or NULL; exactly one of the two when the image output is requested */
  const uint8_t* masks_u8;   /* device [N,H,W] fruit masks, non-zero = fruit (binary, cotton_dataset.py:34-39); NULL = all zero */
  const cnb_camera* cameras; /* device array [N] (width / height fields unused here) */
  int32_t num_images, height, width;
} cnb_image_set;
/* rand3 (device) [R,3] uniform in [0,1) (torch.rand).  Outputs (device): indices [R,3] int32 (camera, y, x) optional; origins,
 * directions [R,3]; pixel_area [R] optional; camera_indices [R] int32 optional; image [R,3] and fruit_mask [R] optional. */
int cnb_sample_train_batch(const cnb_image_set* set, const float* rand3, int64_t R, int32_t* indices, float* origins, float* directions,
                           float* pixel_area, int32_t* camera_indices, float* image, float* fruit_mask, cnb_stream_t stream);
/* cnb_sample_train_batch with per-camera lens distortion (see cnb_lens): lenses is a DEVICE array [num_images] (zero records = no
 * distortion for that camera) or NULL = cnb_sample_train_batch exactly. */
int cnb_sample_train_batch_lens(const cnb_image_set* set, const cnb_lens* lenses, const float* rand3, int64_t R, int32_t* indices, float* origins,
                                float* directions, float* pixel_area, int32_t* camera_indices, float* image, float* fruit_mask,
                                cnb_stream_t stream);

/* ---- f2: optimiser (torch.optim.Adam semantics; fruit_nerf_config.py:45-60) -------------------------------- */
int cnb_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float beta1,
                  float beta2, float eps, int32_t step, float inv_grad_scale, cnb_stream_t stream);

/* ---- a15: the ray-render loop body (FruitModel.get_outputs / get_inference_outputs, fruit_nerf.py:497-599) -------
 * One call = collider -> ProposalNetworkSampler (piecewise/uniform bins -> proposal density -> weights -> PDF resample,
 * per proposal iteration) -> FruitField -> get_weights -> RGB / accumulation / semantic / median-depth renderers, all
 * enqueued on `stream` into a caller-provided workspace.  The training entry also runs the losses of
 * FruitModel.get_loss_dict / get_metrics_dict (fruit_nerf.py:601-615,639-645) and the whole backward. */

/* RayBundle (nerfstudio/cameras/rays.py) restricted to what the path reads */
typedef struct cnb_rays {
  const float* origins;          /* [R,3] */
  const float* directions;       /* [R,3] */
  const float* nears;            /* [R] or NULL => near_plane (NearFarCollider, fruit_nerf.py:167) */
  const float* fars;             /* [R] or NULL => far_plane */
  const int32_t* camera_indices; /* [R]; required for per-camera appearance (training) */
  int64_t num_rays;
  float near_plane, far_plane;
} cnb_rays;

/* ProposalNetworkSampler configuration (fruit_nerf.py:155-164) */
typedef struct cnb_sampler {
  int32_t num_proposal_iterations; /* 1..2 */
  int32_t proposal_samples[2];     /* num_proposal_samples_per_ray */
  int32_t nerf_samples;            /* num_nerf_samples_per_ray */
  int32_t initial_spacing;         /* CNB_SPACING_* of the initial sampler */
  int32_t single_jitter;
  float histogram_padding;         /* 0.01 */
  float pdf_eps;                   /* 1e-5 */
  const float* lin_bins;           /* device [proposal_samples[0]+1] = torch.linspace(0,1,S0+1) */
  const float* u_base[2];          /* device [S+1] = torch.linspace(0, 1-1/(S+1), S+1) for resampled level 1, 2 */
} cnb_sampler;

typedef struct cnb_model {
  cnb_field field;
  cnb_density_field proposal[2];   /* use_same_proposal_network: both entries describe the same network */
  cnb_sampler sampler;
  int32_t bg_mode;                 /* CNB_BG_* (renderer_rgb background_color / override context) */
  float bg_color[3];
  int32_t ray_gradients;           /* training workspace also holds the scratch for cnb_train_cfg.d_origins / d_directions */
  const void* field_table_half;    /* fp16 copy of field.grid.table (cnb_field_fwd_half), or NULL = the fp32 table */
} cnb_model;

/* per-ray outputs, each optional (NULL = not wanted) */
typedef struct cnb_ray_outputs {
  float* rgb;            /* [R,3] */
  float* depth;          /* [R]  median depth of the final level */
  float* accumulation;   /* [R] */
  float* semantics;      /* [R]  composited semantic logit */
  float* prop_depth[2];  /* [R]  median depth of each proposal level */
  int32_t* pdf_inds;     /* [R, nerf_samples+1] searchsorted bins of the last resampling (bit-exactness tests) */
} cnb_ray_outputs;

/* floats of workspace for R rays (training != 0: forward activations + backward scratch are kept) */
int64_t cnb_render_workspace_floats(const cnb_model* m, int64_t num_rays, int32_t training);
/* eval-mode render (deterministic samplers, nan_to_num/clamp in the RGB renderer) */
int cnb_render_rays(const cnb_model* m, const cnb_rays* rays, const cnb_ray_outputs* out, float* workspace, cnb_stream_t stream);

/* Optional optimiser stage of cnb_train_step: one flat param group (engine.FlatGroup) updated by the fused Adam + gradient-clear pass
 * as soon as the backward chain that produces its gradient has finished -- the "fields" group right after the field backward, while
 * the proposal networks are still back-propagating on the forked stream, and vice versa.  The per-step scalars live in DEVICE memory
 * so a captured CUDA graph of the step picks up fresh values on every replay. */
#define CNB_MAX_OPT_GROUPS 4
enum { CNB_CHAIN_FIELD = 0, CNB_CHAIN_PROPOSALS = 1, CNB_CHAIN_JOIN = 2 /* after all chains: the camera-optimizer group */ };
struct cnb_p2p_comm;   /* section (e) below */
struct cnb_p2p_group;
typedef struct cnb_opt_group {
  float* param; float* grad; float* exp_avg; float* exp_avg_sq;  /* flat, 16-byte aligned, n % 4 == 0 */
  int64_t n;
  const float* scalars;      /* device, 8 floats: lr, beta1, beta2, eps, 1 - beta1^t, sqrt(1 - beta2^t), 1 / grad_scale, unused */
  int32_t chain;             /* CNB_CHAIN_*: which backward chain completes this group's gradient */
  int32_t _pad;
  const uint32_t* live;      /* optional: one bit per float4 of the group (cnb_hashgrid_mark_reachable); 0 = unreachable table rows, skipped */
  /* data-parallel training over peer memory (section (e)): when peer_comm != NULL the stage is the group's whole gradient exchange --
   * barrier -> reduce-scatter + Adam + all-gather (cnb_ddp_adam_update with the scalars read from `scalars`) -> barrier -> clear own
   * gradient -- enqueued on the chain's branch of the step, i.e. inside the captured graph and next to the other chain's backward.
   * HOST pointers to the caller's structs (copied at enqueue time); exp_avg / exp_avg_sq are then the owned-slice moments, param / grad
   * this rank's replicas (= peer_group->param[rank] / grad[rank]). */
  const struct cnb_p2p_comm* peer_comm;
  const struct cnb_p2p_group* peer_group;
  int32_t peer_flags;        /* CNB_P2P_* */
  int32_t peer_channel;      /* barrier channel 0..3 reserved for this stage */
} cnb_opt_group;

/* the fp16 copy of a hash table inside an optimiser group (cnb_adam_step_zero_dev_half): table_half = NULL for none */
typedef struct cnb_opt_half {
  void* table_half;
  int64_t first, count;      /* float range of the table inside the group, multiples of 4 */
} cnb_opt_half;

typedef struct cnb_train_cfg {
  const float* image;        /* [R,3] target colours */
  const float* fruit_mask;   /* [R] 0/1 */
  const float* jitter;       /* [levels][R] uniform(0,1) draws (single_jitter) in sampler order, or [levels][R*(S_l+1)] */
  float anneal;              /* proposal weight annealing exponent (fruit_nerf.py:202-216) */
  float semantic_loss_weight;
  float interlevel_loss_mult;
  float grad_scale;          /* GradScaler factor applied to every gradient (1 = none) */
  int32_t update_proposals;  /* ProposalNetworkSampler "updated": proposal networks receive gradients this step */
  int32_t want_metrics;      /* distortion metric + psnr inputs (get_metrics_dict) */
  float* d_origins;          /* optional [R,3], ACCUMULATED: dLoss/d origins (camera optimizer, row a17); needs d_directions too */
  float* d_directions;       /* optional [R,3], ACCUMULATED */
  int32_t phase;             /* 0 = whole step; 1 = forward + final-level/field backward only; 2 = the rest (interlevel loss,
                                proposal backward, metrics) on the workspace phase 1 left behind -- lets a data-parallel caller
                                start the all-reduce of the field gradients while the proposal networks back-propagate;
                                3 = samplers + proposal-network forward only (touches no field parameter); 4 = everything after that
                                (field forward, compositing, losses, the whole backward) on the workspace phase 3 left behind -- lets a
                                data-parallel caller begin the next step while the field group's parameter exchange is still in flight */
  int32_t num_opt_groups;    /* 0 = the caller runs the optimiser itself (cnb_adam_step_zero / cnb_ddp_adam_update) */
  cnb_opt_group opt_groups[CNB_MAX_OPT_GROUPS];
  /* camera optimizer inside the step (nerfstudio CameraOptimizer mode "SO3xR3", fruit_nerf.py:114-116,547,614): NULL = off.  The rays
   * are corrected per camera before the samplers (cnb_camera_opt_apply), dLoss/d(corrected rays) is collected by the backward kernels
   * (cnb_model.ray_gradients must be set; d_origins / d_directions above must be NULL) and chained into d_pose_adjustment together
   * with the regulariser's gradient (cnb_camera_opt_bwd); losses_out[6] = regulariser, included in [5]. */
  const float* pose_adjustment;  /* [num_cameras, 6] (translation | axis-angle) */
  float* d_pose_adjustment;      /* [num_cameras, 6], ACCUMULATED */
  float* camopt_scratch;         /* 12 * (R + num_cameras) floats */
  int32_t num_cameras;
  float trans_l2_penalty, rot_l2_penalty;
  int32_t _pad_camopt;
  cnb_opt_half opt_half[CNB_MAX_OPT_GROUPS];  /* per opt_groups entry; refused with peer-memory groups and the camera-optimizer group */
} cnb_train_cfg;

/* forward + losses + backward of one batch; parameter gradients are ACCUMULATED into the d_* pointers of `m`;
 * With phase 0 / 4 the independent backward chains (field | proposal level 0 | proposal level 1) are forked onto two library-owned side
 * streams per device and joined back with events before the call's last kernel: for the caller it remains ONE stream-ordered call
 * (and a CUDA graph capture of `stream` records the branches); the side streams are created on the first un-captured call and are the
 * only state the library keeps (calls from several host threads on one device share them: still correct, merely serialised there).
 * CNB_TRAIN_NO_OVERLAP=1 in the environment keeps everything on `stream`.
 * losses_out (device, 8 floats, overwritten): [0] rgb mse, [1] weighted semantic bce, [2] interlevel (x mult), [3] distortion,
 * [4] psnr = -10 log10([0]) (get_metrics_dict, fruit_nerf.py:639-645), [5] total = [0] + [1] + [2] + [6] (sum of get_loss_dict),
 * [6] camera-optimizer regulariser (0 unless cfg->pose_adjustment) */
int cnb_train_step(const cnb_model* m, const cnb_rays* rays, const cnb_train_cfg* cfg, const cnb_ray_outputs* out, float* losses_out,
                   float* workspace, cnb_stream_t stream);

/* ---- f2: fused optimiser over one flat parameter group: Adam update + gradient clear in one pass ----------------- */
int cnb_adam_step_zero(float* param, float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float beta1, float beta2,
                       float eps, int32_t step, float inv_grad_scale, cnb_stream_t stream);

/* the same pass with its per-step scalars read from device memory (cnb_opt_group.scalars layout): graph-replay safe */
int cnb_adam_step_zero_dev(float* param, float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, const float* scalars, cnb_stream_t stream);

/* Reachable rows of a hash table.  nerfstudio's torch HashEncoding hashes every level into 2^T slots, also coarse levels whose lattice has
 * far fewer corners than slots; a row no corner hashes to never receives a gradient, its Adam moments stay exactly 0 and torch.optim.Adam
 * leaves it exactly unchanged.  cnb_hashgrid_mark_reachable ORs one bit per 16-byte unit (two rows) of the table into `bitmap` (bit index =
 * first_unit + row / 2; first_unit = float offset of the table inside its flat group / 4); cnb_bitmap_mark_range marks `units` consecutive
 * units (MLP weights, embeddings: always live).  The *_live optimiser entries skip units whose bit is 0 -- bit-identical to the full pass. */
int cnb_hashgrid_mark_reachable(const cnb_grid* g, uint32_t* bitmap, int64_t first_unit, cnb_stream_t stream);
int cnb_bitmap_mark_range(uint32_t* bitmap, int64_t first_unit, int64_t units, cnb_stream_t stream);
int cnb_adam_step_zero_live(float* param, float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float beta1, float beta2,
                            float eps, int32_t step, float inv_grad_scale, const uint32_t* live, cnb_stream_t stream);
int cnb_adam_step_zero_dev_live(float* param, float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, const float* scalars, const uint32_t* live,
                                cnb_stream_t stream);

/* GradScaler support (nerfstudio Trainer: grad_scaler.scale(loss).backward(); grad_scaler.step(optimizer); grad_scaler.update()).
 * cnb_grad_check_finite ORs 1 into *found_inf (device int32, caller clears it) when any of the n gradients is inf / NaN;
 * cnb_adam_step_zero_guarded is cnb_adam_step_zero that, when *skip_flag != 0 (device), leaves param / moments untouched and only
 * clears the gradient -- GradScaler.step's "skip the optimizer step", decided on the device (no host sync, graph-capturable). */
int cnb_grad_check_finite(const float* grad, int64_t n, int32_t* found_inf, cnb_stream_t stream);
int cnb_adam_step_zero_guarded(float* param, float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float beta1, float beta2,
                               float eps, int32_t step, float inv_grad_scale, const int32_t* skip_flag, cnb_stream_t stream);

/* The flat-group updates of a group holding a hash table with an fp16 copy (cnb_table_to_half): the table occupies floats
 * [half_first, half_first + half_count) of the group (multiples of 4); every float4 of it the update writes is also stored, rounded to fp16, into
 * table_half -- from registers, without a second pass over the table.  Units left unchanged (live bit 0, a skipped step) keep their copy.
 * cnb_adam_step_zero_half = cnb_adam_step_zero / _live / _guarded (skip_flag, live optional); cnb_adam_step_zero_dev_half = _dev / _dev_live. */
int cnb_adam_step_zero_half(float* param, float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float beta1, float beta2, float eps,
                            int32_t step, float inv_grad_scale, const int32_t* skip_flag, const uint32_t* live, void* table_half, int64_t half_first,
                            int64_t half_count, cnb_stream_t stream);
int cnb_adam_step_zero_dev_half(float* param, float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, const float* scalars, const uint32_t* live,
                                void* table_half, int64_t half_first, int64_t half_count, cnb_stream_t stream);

/* ---- (e) data-parallel optimiser step over NVLink / NVSwitch peer memory: gradient reduce-scatter + Adam + parameter all-gather in ONE
 * kernel (replaces DDP's all-reduce, fruit_pipeline.py:119-121, followed by torch.optim.Adam, fruit_nerf_config.py:45-60).
 * Buffers are SYMMETRIC allocations mapped into every rank's address space (torch.distributed._symmetric_memory on the Python
 * side); rank r owns the float4-aligned slice cnb_p2p_owned_range(n, r, world) of a flat group, reads that slice of the gradient
 * from every rank, updates it with its shard of the Adam moments (exp_avg / exp_avg_sq are only maintained inside the owned
 * slice) and writes the new parameters into every replica.  Protocol per step, all on `stream`:
 *   cnb_p2p_barrier  (all backward passes done)  ->  cnb_ddp_adam_update per group  ->  cnb_p2p_barrier (all replicas written,
 *   all gradients consumed)  ->  caller clears its own gradient buffers. */
#define CNB_MAX_PEERS 16
enum { CNB_P2P_GRADS_ZERO = 1, /* the group's gradient is zero on every rank this step (frozen proposal networks): skip the peer reads */
       CNB_P2P_MULTIMEM = 2    /* NVLS: one multimem.ld_reduce / multimem.st through the multicast mappings instead of N peer loads / stores */ };
typedef struct cnb_p2p_comm {
  int32_t world, rank;
  uint32_t* flags[CNB_MAX_PEERS]; /* flags[k] = rank k's flag block (>= 4 * CNB_MAX_PEERS uint32, zero-initialised), peer-mapped here */
  uint32_t* state;                /* LOCAL device memory, 8 uint32, zero-initialised: [2c] barrier sequence of channel c, [2c+1] set to 1 when one timed out */
  int32_t timeout_ms;             /* spin limit of one barrier (0 = 10 s) */
  int32_t channel;                /* 0..3: barriers on different channels are independent (may run concurrently on different streams) */
} cnb_p2p_comm;
typedef struct cnb_p2p_group {
  float* grad[CNB_MAX_PEERS];     /* grad[k] = rank k's flat gradient buffer of this group (grad[rank] = own), peer-mapped here */
  float* param[CNB_MAX_PEERS];    /* likewise the flat parameter buffers */
  float* mc_grad;                 /* multicast mappings of the same buffers (NULL without NVLS) */
  float* mc_param;
  const uint32_t* live;           /* optional, LOCAL: one bit per float4 of the group (cnb_hashgrid_mark_reachable); 0 = unreachable table rows, skipped */
} cnb_p2p_group;
void cnb_p2p_owned_range(int64_t n, int32_t rank, int32_t world, int64_t* lo, int64_t* hi);
int cnb_p2p_barrier(const cnb_p2p_comm* comm, cnb_stream_t stream);
int cnb_ddp_adam_update(const cnb_p2p_comm* comm, const cnb_p2p_group* group, float* exp_avg, float* exp_avg_sq, int64_t n, float lr,
                        float beta1, float beta2, float eps, int32_t step, float inv_grad_scale, int32_t flags, cnb_stream_t stream);
/* One group's complete exchange on `stream`, graph-capturable: barrier(channel) -> the update above with its seven scalars read from DEVICE
 * memory (cnb_opt_group.scalars layout; [6] = 1 / (world * loss scale)) -> barrier(channel) -> grad_own cleared (unless CNB_P2P_GRADS_ZERO). */
int cnb_ddp_exchange_dev(const cnb_p2p_comm* comm, const cnb_p2p_group* group, float* exp_avg, float* exp_avg_sq, float* grad_own, int64_t n,
                         const float* scalars, int32_t flags, int32_t channel, cnb_stream_t stream);

/* The whole data-parallel optimiser step in one host call.  Groups with deferred != 0 are exchanged on a library-owned side stream that waits for
 * the work enqueued on `stream` so far and then runs barrier (channel 1) -> update -> barrier -> gradient clear by itself: nothing is added to
 * `stream`, later consumers are fenced with cnb_ddp_wait_deferred; the other groups take barrier (channel 0) -> update -> barrier -> clear on `stream`. */
typedef struct cnb_ddp_group_step {
  const cnb_p2p_group* group;
  float* exp_avg; float* exp_avg_sq;
  float* grad_own;           /* this rank's gradient buffer of the group (= group->grad[rank]); cleared after the exchange; NULL = leave */
  int64_t n;
  float lr, beta1, beta2, eps;
  int32_t step;              /* Adam step count (bias correction), >= 1 */
  float inv_grad_scale;      /* 1 / (world * loss scale) */
  int32_t flags;             /* CNB_P2P_* */
  int32_t deferred;
} cnb_ddp_group_step;
int cnb_ddp_optimizer_step(const cnb_p2p_comm* comm, const cnb_ddp_group_step* groups, int32_t n_groups, cnb_stream_t stream);
int cnb_ddp_wait_deferred(cnb_stream_t stream);

/* ---- a17: camera optimizer (nerfstudio cameras/camera_optimizers.py CameraOptimizer mode "SO3xR3", cameras/lie_groups.py exp_map_SO3xR3)
 * apply: origins_out[r] = origins[r] + t(c), directions_out[r] = R(c) directions[r] with [R|t] = exp_map(pose_adjustment[c]), c = camera_indices[r].
 * bwd: d_pose_adjustment[c] += dLoss/d pose from the ray gradients (d_origins / d_directions w.r.t. the CORRECTED rays; `directions` are the
 * uncorrected ones) + grad_scale * d(regulariser)/d pose, regulariser = mean_c |t_c| * trans_l2_penalty + mean_c |w_c| * rot_l2_penalty, whose
 * value is ADDED to *reg_loss (optional).  scratch: 12 * num_cameras floats. */
int cnb_camera_opt_apply(const float* pose_adjustment, const int32_t* camera_indices, const float* origins, const float* directions, int64_t R,
                         int32_t num_cameras, float* origins_out, float* directions_out, cnb_stream_t stream);
int cnb_camera_opt_bwd(const float* pose_adjustment, const int32_t* camera_indices, const float* directions, const float* d_origins,
                       const float* d_directions, int64_t R, int32_t num_cameras, float trans_l2_penalty, float rot_l2_penalty, float grad_scale,
                       float* scratch, float* d_pose_adjustment, float* reg_loss, cnb_stream_t stream);

/* ---- host -> device staging of one batch (rays, targets, optimiser scalars): n cudaMemcpyAsync on `stream` in one call.
 * dst[i] device, src[i] HOST (pinned for a truly asynchronous copy), bytes[i] sizes; the arrays themselves are host arrays. */
int cnb_upload(void* const* dst, const void* const* src, const int64_t* bytes, int32_t n, cnb_stream_t stream);
/* the device-resident variant: n (<= 8) device -> device copies (16-byte aligned buffers) and n_scalars (<= 32) floats written from the
 * HOST array `scalars` into `scalars_dst` (device) as kernel parameters -- ONE kernel launch instead of n + 1 stream operations
 * (the data manager's batch and the optimiser's per-step scalars of a graph-replayed step). */
int cnb_stage_inputs(void* const* dst, const void* const* src, const int64_t* bytes, int32_t n, float* scalars_dst, const float* scalars,
                     int32_t n_scalars, cnb_stream_t stream);

/* ---- measurement aid: per-stage device times of cnb_render_rays / cnb_train_step (CUDA events on the launching stream).
 * cnb_profile_read synchronises, writes "stage:calls:kernels:ms;..." (summed since enable) into buf and clears the log. */
void cnb_profile_enable(int32_t on);
int cnb_profile_read(char* buf, int32_t buflen);

#ifdef __cplusplus
}
#endif
#endif /* CROPNERF_B200_H */
