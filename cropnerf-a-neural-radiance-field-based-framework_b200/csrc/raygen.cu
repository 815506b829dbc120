// "Next" row f1 of SURVEY.md section 8: ray generation + AABB clipping on the device, the step immediately before the hot path
// in the projection export (fruit_nerf.py:283-288: cam.generate_rays(camera_indices=0, keep_shape=True, aabb_box=aabb), then
// valid = nears < 1e10), which runs once per (super-cluster, camera, sub-cluster) on full 2-2.8 MP images.
// One thread per pixel: nerfstudio Cameras._generate_rays_from_coords (perspective, no distortion; pixel centres at +0.5;
// OpenGL camera axes; pixel_area from the two neighbouring-pixel directions) fused with nerfstudio/utils/math.py
// intersect_aabb (slab test; misses get nears = fars = 1e10) and an optional count of the rays that hit the box.
// LENS = true (cnb_generate_rays_lens) undistorts the three normalised coordinates of every ray first (lens.cuh), as nerfstudio does
// for a camera with non-zero distortion_params; LENS = false is the pinhole kernel, which ignores the trailing lens argument.
#include "lens.cuh"

namespace {

struct RayGenArgs {
  float r[9];   // rotation, row-major
  float t[3];
  float fx, fy, cx, cy;
  int width, height;
  float aabb[6];
  int has_aabb;
};

__device__ __forceinline__ void dir_of(const RayGenArgs& a, float u, float v, float& dx, float& dy, float& dz) {
  // d_world = R * (u, v, -1), each product rounded then summed left to right like torch.sum over the last axis
  const float w = -1.0f;
  dx = __fadd_rn(__fadd_rn(__fmul_rn(u, a.r[0]), __fmul_rn(v, a.r[1])), __fmul_rn(w, a.r[2]));
  dy = __fadd_rn(__fadd_rn(__fmul_rn(u, a.r[3]), __fmul_rn(v, a.r[4])), __fmul_rn(w, a.r[5]));
  dz = __fadd_rn(__fadd_rn(__fmul_rn(u, a.r[6]), __fmul_rn(v, a.r[7])), __fmul_rn(w, a.r[8]));
  const float n = sqrtf(dx * dx + dy * dy + dz * dz);
  dx = __fdiv_rn(dx, n); dy = __fdiv_rn(dy, n); dz = __fdiv_rn(dz, n);
}

// The lens is the last parameter so that the LENS = false instantiation reads every other parameter at the offsets it always had.
template <bool LENS>
__global__ void __launch_bounds__(256) k_generate_rays(const __grid_constant__ RayGenArgs a, const int32_t* __restrict__ pixel_yx, int64_t n,
                                                       float* __restrict__ origins, float* __restrict__ directions, float* __restrict__ pixel_area,
                                                       float* __restrict__ nears, float* __restrict__ fars, int32_t* __restrict__ valid_count,
                                                       const __grid_constant__ cnb_lens lens) {
  int local_valid = 0;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    int py, px;
    if (pixel_yx) { py = __ldg(pixel_yx + 2 * i); px = __ldg(pixel_yx + 2 * i + 1); }
    else { py = (int)(i / a.width); px = (int)(i - (int64_t)py * a.width); }
    const float y = (float)py + 0.5f, x = (float)px + 0.5f;
    float u = __fdiv_rn(__fsub_rn(x, a.cx), a.fx), v = -__fdiv_rn(__fsub_rn(y, a.cy), a.fy);
    const float ux = __fdiv_rn(__fadd_rn(__fsub_rn(x, a.cx), 1.0f), a.fx), vy = -__fdiv_rn(__fadd_rn(__fsub_rn(y, a.cy), 1.0f), a.fy);
    // the offset coordinates share one of their two components with the ray's before undistortion, not after
    float u1 = ux, v1 = v, u2 = u, v2 = vy;
    if (LENS) {
      lens_undistort(lens, u, v);
      if (pixel_area) { lens_undistort(lens, u1, v1); lens_undistort(lens, u2, v2); }
    }
    float dx, dy, dz, ex, ey, ez, gx, gy, gz;
    dir_of(a, u, v, dx, dy, dz);
    if (LENS) {
      if (pixel_area) { dir_of(a, u1, v1, ex, ey, ez); dir_of(a, u2, v2, gx, gy, gz); }
    } else {
      dir_of(a, ux, v, ex, ey, ez);
      dir_of(a, u, vy, gx, gy, gz);
    }
    origins[3 * i] = a.t[0]; origins[3 * i + 1] = a.t[1]; origins[3 * i + 2] = a.t[2];
    directions[3 * i] = dx; directions[3 * i + 1] = dy; directions[3 * i + 2] = dz;
    if (pixel_area) {
      const float sx = sqrtf((dx - ex) * (dx - ex) + (dy - ey) * (dy - ey) + (dz - ez) * (dz - ez));
      const float sy = sqrtf((dx - gx) * (dx - gx) + (dy - gy) * (dy - gy) + (dz - gz) * (dz - gz));
      pixel_area[i] = sx * sy;
    }
    if (a.has_aabb && nears && fars) {
      const float o[3] = {a.t[0], a.t[1], a.t[2]}, d[3] = {dx, dy, dz};
      float tmin = -INFINITY, tmax = INFINITY;
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const float t0 = __fdiv_rn(__fsub_rn(a.aabb[k], o[k]), d[k]), t1 = __fdiv_rn(__fsub_rn(a.aabb[3 + k], o[k]), d[k]);
        tmin = fmaxf(tmin, fminf(t0, t1));
        tmax = fminf(tmax, fmaxf(t0, t1));
      }
      tmin = fminf(fmaxf(tmin, 0.0f), 1e10f);
      tmax = fminf(fmaxf(tmax, 0.0f), 1e10f);
      const bool miss = tmax <= tmin;
      nears[i] = miss ? 1e10f : tmin;
      fars[i] = miss ? 1e10f : tmax;
      local_valid += miss ? 0 : 1;
    }
  }
  if (valid_count) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) local_valid += __shfl_xor_sync(0xffffffffu, local_valid, off);
    if ((threadIdx.x & 31) == 0 && local_valid) atomicAdd(valid_count, local_valid);
  }
}

int launch_generate_rays(const cnb_camera* cam, const cnb_lens* lens, const int32_t* pixel_yx, int64_t n, const float* aabb, float* origins,
                         float* directions, float* pixel_area, float* nears, float* fars, int32_t* valid_count, cnb_stream_t stream) {
  CNB_REQUIRE(cam != nullptr && n >= 0, "generate_rays: null camera / negative count");
  if (n == 0) return CNB_OK;
  CNB_REQUIRE(origins && directions, "generate_rays: null outputs");
  CNB_REQUIRE(cam->width > 0 && cam->height > 0 && cam->fx != 0.0f && cam->fy != 0.0f, "generate_rays: bad intrinsics");
  CNB_REQUIRE(pixel_yx != nullptr || n == (int64_t)cam->width * cam->height, "generate_rays: without pixel_yx n must be width*height");
  CNB_REQUIRE(aabb == nullptr || (nears && fars), "generate_rays: aabb needs nears/fars outputs");
  RayGenArgs a;
  for (int i = 0; i < 3; ++i) {
    for (int j = 0; j < 3; ++j) a.r[3 * i + j] = cam->c2w[4 * i + j];
    a.t[i] = cam->c2w[4 * i + 3];
  }
  a.fx = cam->fx; a.fy = cam->fy; a.cx = cam->cx; a.cy = cam->cy; a.width = cam->width; a.height = cam->height;
  a.has_aabb = aabb != nullptr;
  for (int i = 0; i < 6; ++i) a.aabb[i] = aabb ? aabb[i] : 0.0f;
  int64_t blocks = (n + 255) / 256;
  const int64_t cap = (int64_t)cnb_num_sms() * 16;
  if (blocks > cap) blocks = cap;
  if (lens_active(lens))
    k_generate_rays<true><<<(int)blocks, 256, 0, stream>>>(a, pixel_yx, n, origins, directions, pixel_area, nears, fars, valid_count, *lens);
  else
    k_generate_rays<false><<<(int)blocks, 256, 0, stream>>>(a, pixel_yx, n, origins, directions, pixel_area, nears, fars, valid_count, cnb_lens{});
  return cnb_check_launch("generate_rays");
}

}  // namespace

extern "C" int cnb_generate_rays(const cnb_camera* cam, const int32_t* pixel_yx, int64_t n, const float* aabb, float* origins, float* directions,
                                 float* pixel_area, float* nears, float* fars, int32_t* valid_count, cnb_stream_t stream) {
  return launch_generate_rays(cam, nullptr, pixel_yx, n, aabb, origins, directions, pixel_area, nears, fars, valid_count, stream);
}

extern "C" int cnb_generate_rays_lens(const cnb_camera* cam, const cnb_lens* lens, const int32_t* pixel_yx, int64_t n, const float* aabb,
                                      float* origins, float* directions, float* pixel_area, float* nears, float* fars, int32_t* valid_count,
                                      cnb_stream_t stream) {
  return launch_generate_rays(cam, lens, pixel_yx, n, aabb, origins, directions, pixel_area, nears, fars, valid_count, stream);
}
