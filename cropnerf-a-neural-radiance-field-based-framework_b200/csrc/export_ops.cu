// Device side of the two export workloads' loop bodies around the render call (rows e2 / e3 / f1 of SURVEY.md section 8):
//
//  * cnb_extract_points       -- export/exporter_utils_nerfacto.py:153-176 (`ns-export pointcloud`, BASELINE configs[2]): after a batch is
//    rendered, point = origin + direction * depth, keep = semantic label is "fruit" (sigmoid(logit) - 0.9 > 0, fruit_nerf.py:594-597) and the
//    point lies inside the crop OrientedBox (nerfstudio OrientedBox.within), then an ORDER-PRESERVING compaction appended to the
//    output arrays.  The running count lives in device memory, so the export loop never synchronises per batch.
//  * cnb_generate_rays_boxes  -- fruit_nerf.py:281-288 for ALL k sub-cluster boxes of a super-cluster at once: one pass over the camera's
//    pixels builds each ray once, slab-tests it against every box and appends the hits (ray, near, far, box * npix + pixel) to one compacted
//    list -- one launch and one count read-back per (super-cluster, camera) instead of k full-image ray bundles, k masks and 2 k syncs.
//    cnb_generate_rays_boxes_lens undistorts the ray before the slab tests and the pixel-area offsets on the first hit (lens.cuh).
//  * cnb_projection_scatter   -- fruit_nerf.py:296-315: semantics of the hit rays back into the k un-occluded images and, where the opacity
//    accumulated in front of the box is below 0.5, into the k "visible" images, quantised like torchvision's save_image (x * 255 + 0.5,
//    clamped, truncated) -- the pixels stay on the device until the PNG encoder wants them.
//  * cnb_volume_face_rays     -- data/fruit_datamanager.py:71-120 + components/ray_generators.py:46-66 (volumetric export): the regular
//    grid of orthographic rays on the z_min face of the export box, torch.linspace's two-sided formula evaluated per thread.
#include "lens.cuh"

namespace {

constexpr int XB = 256;

struct ExtractArgs {
  const float *origins, *directions, *depth, *semantics, *rgb;
  int64_t n;
  float R[9], T[3], half[3];
  int has_obb, only_semantics;
  float threshold;
};

__device__ __forceinline__ bool extract_keep(const ExtractArgs& a, int64_t i, float (&p)[3]) {
#pragma unroll
  for (int k = 0; k < 3; ++k) p[k] = __fadd_rn(__ldg(a.origins + 3 * i + k), __fmul_rn(__ldg(a.directions + 3 * i + k), __ldg(a.depth + i)));
  bool keep = true;
  if (a.only_semantics) {
    // semantics_colormap = colormap[heaviside(sigmoid(logit) - 0.9, 0)] with colormap = (0, 1): label 1 iff sigmoid(logit) - 0.9 > 0
    const float sg = __fdiv_rn(1.0f, __fadd_rn(1.0f, expf(-__ldg(a.semantics + i))));
    keep = __fsub_rn(sg, a.threshold) > 0.0f;
  }
  if (keep && a.has_obb) {
    const float d0 = __fsub_rn(p[0], a.T[0]), d1 = __fsub_rn(p[1], a.T[1]), d2 = __fsub_rn(p[2], a.T[2]);
#pragma unroll
    for (int j = 0; j < 3; ++j) {  // local = (p - T) @ R
      const float l = fmaf(d2, a.R[6 + j], fmaf(d1, a.R[3 + j], d0 * a.R[j]));
      keep = keep && (l > -a.half[j]) && (l < a.half[j]);
    }
  }
  return keep;
}

__global__ void __launch_bounds__(XB) k_extract_count(const __grid_constant__ ExtractArgs a, int32_t* __restrict__ block_counts) {
  const int64_t i = blockIdx.x * (int64_t)XB + threadIdx.x;
  float p[3];
  const bool keep = i < a.n && extract_keep(a, i, p);
  const int c = __syncthreads_count(keep ? 1 : 0);
  if (threadIdx.x == 0) block_counts[blockIdx.x] = c;
}

__global__ void __launch_bounds__(XB) k_extract_write(const __grid_constant__ ExtractArgs a, const int32_t* __restrict__ block_counts,
                                                       const int32_t* __restrict__ count_in, int32_t* __restrict__ count_out, int64_t capacity,
                                                       float* __restrict__ out_points, float* __restrict__ out_rgbs, float* __restrict__ out_dirs) {
  __shared__ int s_part[XB / 32];
  __shared__ int s_prefix;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // kept rays in the blocks before this one
  int part = 0;
  for (int j = threadIdx.x; j < (int)blockIdx.x; j += XB) part += __ldg(block_counts + j);
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) part += __shfl_xor_sync(0xffffffffu, part, off);
  if (lane == 0) s_part[warp] = part;
  __syncthreads();
  if (threadIdx.x == 0) {
    int t = 0;
    for (int w = 0; w < XB / 32; ++w) t += s_part[w];
    s_prefix = t;
  }
  __syncthreads();
  const int64_t base = (int64_t)__ldg(count_in) + s_prefix;
  const int64_t i = blockIdx.x * (int64_t)XB + threadIdx.x;
  float p[3];
  const bool keep = i < a.n && extract_keep(a, i, p);
  const unsigned m = __ballot_sync(0xffffffffu, keep);
  __syncthreads();
  if (lane == 0) s_part[warp] = __popc(m);
  __syncthreads();
  int before = 0;
  for (int w = 0; w < warp; ++w) before += s_part[w];
  if (keep) {
    const int64_t slot = base + before + __popc(m & ((1u << lane) - 1u));
    if (slot < capacity) {
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        out_points[3 * slot + k] = p[k];
        if (out_rgbs) out_rgbs[3 * slot + k] = __ldg(a.rgb + 3 * i + k);
        if (out_dirs) out_dirs[3 * slot + k] = __ldg(a.directions + 3 * i + k);
      }
    }
  }
  if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) {
    int total = 0;
    for (int w = 0; w < XB / 32; ++w) total += s_part[w];
    *count_out = (int32_t)(base + total);  // may exceed capacity: the caller sees how many were dropped
  }
}

// ---------------------------------------------------------------------------------------------------------------------
struct BoxRayArgs {
  float r[9], t[3];
  float fx, fy, cx, cy;
  int width, height;
  const float* boxes;  // device [k][6]: min xyz, max xyz
  int k;
};

__device__ __forceinline__ void box_dir_of(const BoxRayArgs& a, float u, float v, float& dx, float& dy, float& dz) {
  const float w = -1.0f;  // same operation order as k_generate_rays (raygen.cu): nerfstudio's pinhole model op for op
  dx = __fadd_rn(__fadd_rn(__fmul_rn(u, a.r[0]), __fmul_rn(v, a.r[1])), __fmul_rn(w, a.r[2]));
  dy = __fadd_rn(__fadd_rn(__fmul_rn(u, a.r[3]), __fmul_rn(v, a.r[4])), __fmul_rn(w, a.r[5]));
  dz = __fadd_rn(__fadd_rn(__fmul_rn(u, a.r[6]), __fmul_rn(v, a.r[7])), __fmul_rn(w, a.r[8]));
  const float n = sqrtf(dx * dx + dy * dy + dz * dz);
  dx = __fdiv_rn(dx, n); dy = __fdiv_rn(dy, n); dz = __fdiv_rn(dz, n);
}

// The lens is the last parameter so that the LENS = false instantiation reads every other parameter at the offsets it always had.
template <bool LENS>
__global__ void __launch_bounds__(256) k_generate_rays_boxes(const __grid_constant__ BoxRayArgs a, int64_t capacity, float* __restrict__ origins,
                                                             float* __restrict__ directions, float* __restrict__ pixel_area, float* __restrict__ nears,
                                                             float* __restrict__ fars, int32_t* __restrict__ tags, int32_t* __restrict__ count,
                                                             const __grid_constant__ cnb_lens lens) {
  const int64_t npix = (int64_t)a.width * a.height;
  const int64_t nround = (npix + 31) / 32 * 32;
  const int lane = threadIdx.x & 31;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < nround; i += (int64_t)gridDim.x * blockDim.x) {
    const bool in = i < npix;
    const int py = (int)((in ? i : 0) / a.width), px = (int)((in ? i : 0) - (int64_t)py * a.width);
    const float y = (float)py + 0.5f, x = (float)px + 0.5f;
    const float u0 = __fdiv_rn(__fsub_rn(x, a.cx), a.fx), v0 = -__fdiv_rn(__fsub_rn(y, a.cy), a.fy);
    float u = u0, v = v0;
    if (LENS) lens_undistort(lens, u, v);
    float dx, dy, dz;
    box_dir_of(a, u, v, dx, dy, dz);
    float area = -1.0f;  // computed on the first hit only
    for (int b = 0; b < a.k; ++b) {
      const float* bx = a.boxes + 6 * b;
      const float o[3] = {a.t[0], a.t[1], a.t[2]}, d[3] = {dx, dy, dz};
      float tmin = -INFINITY, tmax = INFINITY;
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const float t0 = __fdiv_rn(__fsub_rn(__ldg(bx + k), o[k]), d[k]), t1 = __fdiv_rn(__fsub_rn(__ldg(bx + 3 + k), o[k]), d[k]);
        tmin = fmaxf(tmin, fminf(t0, t1));
        tmax = fminf(tmax, fmaxf(t0, t1));
      }
      tmin = fminf(fmaxf(tmin, 0.0f), 1e10f);
      tmax = fminf(fmaxf(tmax, 0.0f), 1e10f);
      const bool hit = in && !(tmax <= tmin);
      const unsigned m = __ballot_sync(0xffffffffu, hit);
      if (m == 0u) continue;
      int base = 0;
      if (lane == 0) base = atomicAdd(count, __popc(m));
      base = __shfl_sync(0xffffffffu, base, 0);
      if (!hit) continue;
      const int64_t slot = (int64_t)base + __popc(m & ((1u << lane) - 1u));
      if (slot >= capacity) continue;
      if (area < 0.0f) {
        const float ux = __fdiv_rn(__fadd_rn(__fsub_rn(x, a.cx), 1.0f), a.fx), vy = -__fdiv_rn(__fadd_rn(__fsub_rn(y, a.cy), 1.0f), a.fy);
        float ex, ey, ez, gx, gy, gz;
        if (LENS) {
          float u1 = ux, v1 = v0, u2 = u0, v2 = vy;
          lens_undistort(lens, u1, v1);
          lens_undistort(lens, u2, v2);
          box_dir_of(a, u1, v1, ex, ey, ez);
          box_dir_of(a, u2, v2, gx, gy, gz);
        } else {
          box_dir_of(a, ux, v, ex, ey, ez);
          box_dir_of(a, u, vy, gx, gy, gz);
        }
        const float sx = sqrtf((dx - ex) * (dx - ex) + (dy - ey) * (dy - ey) + (dz - ez) * (dz - ez));
        const float sy = sqrtf((dx - gx) * (dx - gx) + (dy - gy) * (dy - gy) + (dz - gz) * (dz - gz));
        area = sx * sy;
      }
      origins[3 * slot] = a.t[0]; origins[3 * slot + 1] = a.t[1]; origins[3 * slot + 2] = a.t[2];
      directions[3 * slot] = dx; directions[3 * slot + 1] = dy; directions[3 * slot + 2] = dz;
      pixel_area[slot] = area;
      nears[slot] = tmin;
      fars[slot] = tmax;
      tags[slot] = (int32_t)((int64_t)b * npix + i);
    }
  }
}

__device__ __forceinline__ uint8_t quantise_png(float x) {
  // torchvision.utils.save_image: img.mul(255).add_(0.5).clamp_(0, 255).to(uint8)
  const float q = fminf(fmaxf(__fadd_rn(__fmul_rn(x, 255.0f), 0.5f), 0.0f), 255.0f);
  return (uint8_t)(int)q;
}

__global__ void __launch_bounds__(256) k_projection_scatter(const int32_t* __restrict__ tags, const float* __restrict__ semantics,
                                                            const float* __restrict__ front, int64_t n, float occlusion, uint8_t* __restrict__ wo_occ,
                                                            uint8_t* __restrict__ visible) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int32_t tag = __ldg(tags + i);
    const uint8_t q = quantise_png(__ldg(semantics + i));
    wo_occ[tag] = q;
    visible[tag] = (__ldg(front + i) >= occlusion) ? (uint8_t)0 : q;
  }
}

// torch.linspace(start, end, steps) for float32 on the CPU: step = (end - start) / (steps - 1) in float; the first half counts up from
// start, the second half counts down from end, each element ONE fused multiply-add (the vectorised CPU kernel uses fmadd; checked
// against torch on 2000 random (start, end, steps) triples when this was written)
__device__ __forceinline__ float linspace_at(float start, float end, int steps, int i) {
  if (steps == 1) return start;
  const float step = __fdiv_rn(__fsub_rn(end, start), (float)(steps - 1));
  const int halfway = steps / 2;
  return i < halfway ? __fmaf_rn(step, (float)i, start) : __fmaf_rn(-step, (float)(steps - i - 1), end);
}

__global__ void __launch_bounds__(256) k_volume_face_rays(float x0, float x1, int nx, float y0, float y1, int ny, float z, float dirx, float diry,
                                                          float dirz, float far, int64_t first, int64_t n, float* __restrict__ origins,
                                                          float* __restrict__ directions, float* __restrict__ nears, float* __restrict__ fars) {
  for (int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; j < n; j += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = first + j;             // meshgrid(x, y, indexing="ij") flattened: x slowest
    const int ix = (int)(i / ny), iy = (int)(i - (int64_t)ix * ny);
    origins[3 * j] = linspace_at(x0, x1, nx, ix);
    origins[3 * j + 1] = linspace_at(y0, y1, ny, iy);
    origins[3 * j + 2] = z;
    directions[3 * j] = dirx; directions[3 * j + 1] = diry; directions[3 * j + 2] = dirz;
    nears[j] = 0.0f;
    fars[j] = far;
  }
}

int grid_cap(int64_t items, int block, int per_sm) {
  int64_t blocks = (items + block - 1) / block;
  const int64_t cap = (int64_t)cnb_num_sms() * per_sm;
  if (blocks > cap) blocks = cap;
  return (int)(blocks < 1 ? 1 : blocks);
}

}  // namespace

extern "C" int64_t cnb_extract_points_scratch_ints(int64_t n) { return n <= 0 ? 0 : (n + XB - 1) / XB; }

extern "C" int cnb_extract_points(const float* origins, const float* directions, const float* depth, const float* semantics, const float* rgb, int64_t n,
                                  const float* obb, int32_t only_semantics, float threshold, int32_t* block_counts, const int32_t* count_in,
                                  int32_t* count_out, int64_t capacity, float* out_points, float* out_rgbs, float* out_dirs, cnb_stream_t stream) {
  CNB_REQUIRE(n >= 0 && capacity >= 0, "extract_points: negative size");
  CNB_REQUIRE(count_in && count_out && count_in != count_out, "extract_points: count_in / count_out must be two distinct device counters");
  if (n == 0) return cudaMemcpyAsync(count_out, count_in, sizeof(int32_t), cudaMemcpyDeviceToDevice, stream) == cudaSuccess ? CNB_OK : cnb_check_launch("extract_points copy");
  CNB_REQUIRE(origins && directions && depth && out_points && block_counts, "extract_points: null pointer");
  CNB_REQUIRE(!only_semantics || semantics, "extract_points: only_semantics needs the semantic logits");
  CNB_REQUIRE(!out_rgbs || rgb, "extract_points: out_rgbs needs rgb");
  CNB_REQUIRE(n <= (int64_t)XB * 0x7fffffff, "extract_points: batch too large");
  ExtractArgs a;
  a.origins = origins; a.directions = directions; a.depth = depth; a.semantics = semantics; a.rgb = rgb; a.n = n;
  a.has_obb = obb != nullptr; a.only_semantics = only_semantics; a.threshold = threshold;
  for (int i = 0; i < 9; ++i) a.R[i] = obb ? obb[i] : 0.f;
  for (int i = 0; i < 3; ++i) { a.T[i] = obb ? obb[9 + i] : 0.f; a.half[i] = obb ? obb[12 + i] * 0.5f : 0.f; }
  const int blocks = (int)((n + XB - 1) / XB);
  k_extract_count<<<blocks, XB, 0, stream>>>(a, block_counts);
  int rc = cnb_check_launch("extract_points count");
  if (rc) return rc;
  k_extract_write<<<blocks, XB, 0, stream>>>(a, block_counts, count_in, count_out, capacity, out_points, out_rgbs, out_dirs);
  return cnb_check_launch("extract_points write");
}

extern "C" int cnb_generate_rays_boxes_lens(const cnb_camera* cam, const cnb_lens* lens, const float* boxes, int32_t num_boxes, int64_t capacity,
                                            float* origins, float* directions, float* pixel_area, float* nears, float* fars, int32_t* tags,
                                            int32_t* count, cnb_stream_t stream) {
  CNB_REQUIRE(cam && boxes && num_boxes >= 1 && capacity >= 0, "generate_rays_boxes: null camera / boxes");
  CNB_REQUIRE(origins && directions && pixel_area && nears && fars && tags && count, "generate_rays_boxes: null output");
  CNB_REQUIRE(cam->width > 0 && cam->height > 0 && cam->fx != 0.0f && cam->fy != 0.0f, "generate_rays_boxes: bad intrinsics");
  CNB_REQUIRE((int64_t)num_boxes * cam->width * cam->height <= 0x7fffffffLL, "generate_rays_boxes: boxes x pixels exceeds the 31-bit tag");
  BoxRayArgs a;
  for (int i = 0; i < 3; ++i) {
    for (int j = 0; j < 3; ++j) a.r[3 * i + j] = cam->c2w[4 * i + j];
    a.t[i] = cam->c2w[4 * i + 3];
  }
  a.fx = cam->fx; a.fy = cam->fy; a.cx = cam->cx; a.cy = cam->cy; a.width = cam->width; a.height = cam->height;
  a.boxes = boxes; a.k = num_boxes;
  const int blocks = grid_cap((int64_t)cam->width * cam->height, 256, 8);
  if (lens_active(lens))
    k_generate_rays_boxes<true><<<blocks, 256, 0, stream>>>(a, capacity, origins, directions, pixel_area, nears, fars, tags, count, *lens);
  else
    k_generate_rays_boxes<false><<<blocks, 256, 0, stream>>>(a, capacity, origins, directions, pixel_area, nears, fars, tags, count, cnb_lens{});
  return cnb_check_launch("generate_rays_boxes");
}

extern "C" int cnb_generate_rays_boxes(const cnb_camera* cam, const float* boxes, int32_t num_boxes, int64_t capacity, float* origins, float* directions,
                                       float* pixel_area, float* nears, float* fars, int32_t* tags, int32_t* count, cnb_stream_t stream) {
  return cnb_generate_rays_boxes_lens(cam, nullptr, boxes, num_boxes, capacity, origins, directions, pixel_area, nears, fars, tags, count, stream);
}

extern "C" int cnb_projection_scatter(const int32_t* tags, const float* semantics, const float* front_opacity, int64_t n, float occlusion_threshold,
                                      uint8_t* wo_occ, uint8_t* visible, cnb_stream_t stream) {
  CNB_REQUIRE(n >= 0, "projection_scatter: negative count");
  if (n == 0) return CNB_OK;
  CNB_REQUIRE(tags && semantics && front_opacity && wo_occ && visible, "projection_scatter: null pointer");
  k_projection_scatter<<<grid_cap(n, 256, 8), 256, 0, stream>>>(tags, semantics, front_opacity, n, occlusion_threshold, wo_occ, visible);
  return cnb_check_launch("projection_scatter");
}

extern "C" int cnb_volume_face_rays(float x0, float x1, int32_t nx, float y0, float y1, int32_t ny, float z, const float* direction, float far,
                                    int64_t first, int64_t n, float* origins, float* directions, float* nears, float* fars, cnb_stream_t stream) {
  CNB_REQUIRE(nx >= 1 && ny >= 1 && first >= 0 && n >= 0 && first + n <= (int64_t)nx * ny, "volume_face_rays: range outside the %d x %d grid", nx, ny);
  if (n == 0) return CNB_OK;
  CNB_REQUIRE(direction && origins && directions && nears && fars, "volume_face_rays: null pointer");
  k_volume_face_rays<<<grid_cap(n, 256, 8), 256, 0, stream>>>(x0, x1, nx, y0, y1, ny, z, direction[0], direction[1], direction[2], far, first, n, origins,
                                                             directions, nears, fars);
  return cnb_check_launch("volume_face_rays");
}
