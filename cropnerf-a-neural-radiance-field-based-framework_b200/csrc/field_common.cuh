// Pieces shared by the fp32 and mixed-precision FruitField kernels.
#pragma once
#include "cnb_common.cuh"

// components_from_spherical_harmonics(degree=3) on the *shifted* direction (d+1)/2, exactly as the torch path of
// nerfstudio's SHEncoding evaluates it for fruit_field.py:116-119,244-246 (SURVEY.md App. A.4).
__device__ __forceinline__ void cnb_sh16(float dx, float dy, float dz, float (&c)[16]) {
  const float x = __fmul_rn(__fadd_rn(dx, 1.0f), 0.5f);
  const float y = __fmul_rn(__fadd_rn(dy, 1.0f), 0.5f);
  const float z = __fmul_rn(__fadd_rn(dz, 1.0f), 0.5f);
  const float xx = x * x, yy = y * y, zz = z * z;
  c[0] = 0.28209479177387814f;
  c[1] = 0.4886025119029199f * y;
  c[2] = 0.4886025119029199f * z;
  c[3] = 0.4886025119029199f * x;
  c[4] = 1.0925484305920792f * x * y;
  c[5] = 1.0925484305920792f * y * z;
  c[6] = 0.9461746957575601f * zz - 0.31539156525251999f;
  c[7] = 1.0925484305920792f * x * z;
  c[8] = 0.5462742152960396f * (xx - yy);
  c[9] = 0.5900435899266435f * y * (3.0f * xx - yy);
  c[10] = 2.890611442640554f * x * y * z;
  c[11] = 0.4570457994644658f * y * (5.0f * zz - 1.0f);
  c[12] = 0.3731763325901154f * z * (5.0f * zz - 3.0f);
  c[13] = 0.4570457994644658f * x * (5.0f * zz - 1.0f);
  c[14] = 1.445305721320277f * z * (xx - yy);
  c[15] = 0.5900435899266435f * x * (xx - 3.0f * yy);
}

int cnb_field_check(const cnb_field* f, const cnb_samples* s, bool bwd);

// mixed-precision (tensor-core) implementation: field_mixed.cu, the backward in field_mixed_bwd_tc5.cu
int cnb_field_mixed_fwd(const cnb_field* f, const cnb_samples* s, float* density, float* geo, float* rgb, float* sem, float* positions_out, float* ctx,
                        int training, cudaStream_t stream);
int cnb_field_mixed_bwd(const cnb_field* f, const cnb_samples* s, const float* d_density, const float* d_rgb, const float* d_sem, float* ctx,
                        cudaStream_t stream);
bool cnb_field_mixed_supported(const cnb_field* f);
int64_t cnb_field_mixed_ctx_floats(int64_t n, int training);
float* cnb_field_mixed_dx0(float* ctx, int64_t n);  // d(encoded features), LEVEL-MAJOR [16][n][2], written by the mixed backward

// mlp_mixed.cu: the tensor-core operator for MLPs wider than 64, with the kept activations (`hidden`) and the backward's transient scratch
// (`work`) in separate caller buffers, so that the field can share one work region between its MLPs
bool cnb_mlp_mixed_supported(const cnb_mlp* m);
int64_t cnb_mlp_mixed_hidden_floats(const cnb_mlp* m, int64_t n, int training);
int64_t cnb_mlp_mixed_work_floats(const cnb_mlp* m, int64_t n);
int cnb_mlp_mixed_fwd_ws(const cnb_mlp* m, const float* x, int64_t x_stride, int64_t n, float* y, float* hidden, int training, cudaStream_t stream);
int cnb_mlp_mixed_bwd_ws(const cnb_mlp* m, const float* x, int64_t x_stride, const float* hidden, const float* y, const float* dy, int64_t n, float* dx,
                         int64_t dx_stride, float* work, cudaStream_t stream);
int cnb_mlp_mixed_launches(const cnb_mlp* m, bool bwd, bool want_dx);
// field_fp32.cu: the mixed FruitField for architectures outside the fused kernels (the big / huge presets), and its launch counts
bool cnb_field_mixed_wide_supported(const cnb_field* f);
int cnb_field_mixed_wide_launches(const cnb_field* f, bool bwd, bool rays);

// hashgrid.cu, library-internal variants reading d(features) level-major [L][n][2]: the fused field backward's accumulator pair of a
// thread IS one level's two features, and the level-major scatter warps then read one contiguous 256-byte run per request.
int cnb_hashgrid_bwd_level_major(const cnb_grid* g, const float* positions, const float* d_out, int64_t n, cudaStream_t stream);
int cnb_position_grad_rays_level_major(const cnb_grid* g, const cnb_warp* warp, const cnb_samples* s, const float* d_feat, float* d_origins,
                                       float* d_directions, cudaStream_t stream);
