// Lens distortion of the perspective ray generators (raygen.cu, export_ops.cu, train_batch.cu): nerfstudio
// camera_utils.radial_and_tangential_undistort (eps = 1e-3, max_iterations = 10) with _compute_residual_and_jacobian, which
// Cameras._generate_rays_from_coords applies to the normalised coordinates (x, -y) of the ray and of both pixel-area offsets.
// Newton's method from the distorted point, float32 throughout, every operation rounded on its own in torch's left-to-right
// order (2*p1*x*y = ((2*p1)*x)*y), so nvcc cannot contract any of it into FMAs.  With all six parameters zero the solve returns
// its input bit for bit: d == 1, the residual is 0 and every step is +-0.
#pragma once
#include "cnb_common.cuh"

__device__ __forceinline__ float lens_mul(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float lens_add(float a, float b) { return __fadd_rn(a, b); }

// (x, y) in: distorted normalised coordinates; out: undistorted.
__device__ __forceinline__ void lens_undistort(const cnb_lens& l, float& x, float& y) {
  const float xd = x, yd = y;
  const float two_p1 = lens_mul(2.0f, l.p1), two_p2 = lens_mul(2.0f, l.p2);
  const float six_p1 = lens_mul(6.0f, l.p1), six_p2 = lens_mul(6.0f, l.p2);
  const float two_k2 = lens_mul(2.0f, l.k2), three_k3 = lens_mul(3.0f, l.k3);
  for (int it = 0; it < 10; ++it) {
    const float r = lens_add(lens_mul(x, x), lens_mul(y, y));
    // d = 1 + r*(k1 + r*(k2 + r*(k3 + r*k4)))
    const float d = lens_add(1.0f, lens_mul(r, lens_add(l.k1, lens_mul(r, lens_add(l.k2, lens_mul(r, lens_add(l.k3, lens_mul(r, l.k4))))))));
    // fx = d*x + 2*p1*x*y + p2*(r + 2*x*x) - xd ;  fy = d*y + 2*p2*x*y + p1*(r + 2*y*y) - yd
    const float fx = __fsub_rn(lens_add(lens_add(lens_mul(d, x), lens_mul(lens_mul(two_p1, x), y)),
                                        lens_mul(l.p2, lens_add(r, lens_mul(lens_mul(2.0f, x), x)))), xd);
    const float fy = __fsub_rn(lens_add(lens_add(lens_mul(d, y), lens_mul(lens_mul(two_p2, x), y)),
                                        lens_mul(l.p1, lens_add(r, lens_mul(lens_mul(2.0f, y), y)))), yd);
    // d_r = k1 + r*(2*k2 + r*(3*k3 + r*4*k4)) ;  d_x = 2*x*d_r ;  d_y = 2*y*d_r
    const float d_r = lens_add(l.k1, lens_mul(r, lens_add(two_k2, lens_mul(r, lens_add(three_k3, lens_mul(lens_mul(r, 4.0f), l.k4))))));
    const float d_x = lens_mul(lens_mul(2.0f, x), d_r), d_y = lens_mul(lens_mul(2.0f, y), d_r);
    // fx_x = d + d_x*x + 2*p1*y + 6*p2*x ;  fx_y = d_y*x + 2*p1*x + 2*p2*y
    const float fx_x = lens_add(lens_add(lens_add(d, lens_mul(d_x, x)), lens_mul(two_p1, y)), lens_mul(six_p2, x));
    const float fx_y = lens_add(lens_add(lens_mul(d_y, x), lens_mul(two_p1, x)), lens_mul(two_p2, y));
    // fy_x = d_x*y + 2*p2*y + 2*p1*x ;  fy_y = d + d_y*y + 2*p2*x + 6*p1*y
    const float fy_x = lens_add(lens_add(lens_mul(d_x, y), lens_mul(two_p2, y)), lens_mul(two_p1, x));
    const float fy_y = lens_add(lens_add(lens_add(d, lens_mul(d_y, y)), lens_mul(two_p2, x)), lens_mul(six_p1, y));
    const float den = __fsub_rn(lens_mul(fy_x, fx_y), lens_mul(fx_x, fy_y));
    const float num_x = __fsub_rn(lens_mul(fx, fy_y), lens_mul(fy, fx_y));
    const float num_y = __fsub_rn(lens_mul(fy, fx_x), lens_mul(fx, fy_x));
    const bool solve = fabsf(den) > 1e-3f;  // torch.where(|den| > eps, num / den, 0), eps compared in float32
    x = lens_add(x, solve ? __fdiv_rn(num_x, den) : 0.0f);
    y = lens_add(y, solve ? __fdiv_rn(num_y, den) : 0.0f);
  }
}

// "Some parameter is non-zero" ((distortion_params != 0).any() of nerfstudio; NaN counts as non-zero)
static inline bool lens_active(const cnb_lens* l) {
  return l != nullptr && (l->k1 != 0.0f || l->k2 != 0.0f || l->k3 != 0.0f || l->k4 != 0.0f || l->p1 != 0.0f || l->p2 != 0.0f);
}
