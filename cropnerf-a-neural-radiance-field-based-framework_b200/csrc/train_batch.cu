// "Next" row f1 of SURVEY.md section 8, training side: the step immediately before the hot path in a training iteration,
// FruitDataManager.next_train (data/fruit_datamanager.py:188-197):
//     batch       = train_pixel_sampler.sample(image_batch)      nerfstudio PixelSampler: (camera, y, x) = (rand[R,3] * [N,H,W]).long(),
//                                                                 then value[c, y, x] for every per-pixel tensor of the batch
//     ray_bundle  = train_ray_generator(batch["indices"])        nerfstudio RayGenerator: image_coords[y, x] (pixel centres, +0.5) ->
//                                                                 Cameras.generate_rays(camera_indices=c, coords=...)
// With the images resident in HBM (300 x 1080p: 1.9 GB as uint8 RGB + 0.6 GB of masks) one thread per ray does index -> pixel gather ->
// per-camera pinhole ray -> pixel area; the outputs are exactly the tensors cnb_train_step reads (origins, directions, camera indices,
// image, fruit_mask), so a training step needs no host batch at all.  Ray arithmetic = k_generate_rays (raygen.cu), op for op,
// including the per-camera lens undistortion of cnb_sample_train_batch_lens (LENS = true; lens.cuh).
#include <cstddef>

#include "lens.cuh"

namespace {

struct TrainBatchArgs {
  const uint8_t* images_u8;
  const float* images_f32;
  const uint8_t* masks_u8;
  const cnb_camera* cameras;
  int32_t N, H, W;
};

// d_world = R (u, v, -1), each product rounded then summed left to right like torch.sum over the last axis; then normalised
__device__ __forceinline__ void camera_direction(const float (&r)[9], float u, float v, float& dx, float& dy, float& dz) {
  const float w = -1.0f;
  dx = __fadd_rn(__fadd_rn(__fmul_rn(u, r[0]), __fmul_rn(v, r[1])), __fmul_rn(w, r[2]));
  dy = __fadd_rn(__fadd_rn(__fmul_rn(u, r[3]), __fmul_rn(v, r[4])), __fmul_rn(w, r[5]));
  dz = __fadd_rn(__fadd_rn(__fmul_rn(u, r[6]), __fmul_rn(v, r[7])), __fmul_rn(w, r[8]));
  const float n = sqrtf(dx * dx + dy * dy + dz * dz);
  dx = __fdiv_rn(dx, n); dy = __fdiv_rn(dy, n); dz = __fdiv_rn(dz, n);
}

// (rand * extent).long() of the reference, clamped to the last valid index (a float32 product can round up to `extent`; torch would raise there)
__device__ __forceinline__ int scaled_index(float rnd, int extent) {
  const int v = (int)__fmul_rn(rnd, (float)extent);
  return min(max(v, 0), extent - 1);
}

// lenses [N] (device) is the last parameter so that the LENS = false instantiation reads every other parameter where it always did
template <bool LENS>
__global__ void __launch_bounds__(256) k_sample_train_batch(const __grid_constant__ TrainBatchArgs a, const float* __restrict__ rand3, int64_t R,
                                                            int32_t* __restrict__ indices, float* __restrict__ origins, float* __restrict__ directions,
                                                            float* __restrict__ pixel_area, int32_t* __restrict__ camera_indices,
                                                            float* __restrict__ image, float* __restrict__ fruit_mask,
                                                            const cnb_lens* __restrict__ lenses) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < R; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = scaled_index(__ldg(rand3 + 3 * i), a.N);
    const int py = scaled_index(__ldg(rand3 + 3 * i + 1), a.H);
    const int px = scaled_index(__ldg(rand3 + 3 * i + 2), a.W);
    if (indices) { indices[3 * i] = c; indices[3 * i + 1] = py; indices[3 * i + 2] = px; }
    if (camera_indices) camera_indices[i] = c;
    // ---- pixel gather (collate_image_dataset_batch: value[c, y, x]) -------------------------------------------------------------
    const int64_t p = ((int64_t)c * a.H + py) * a.W + px;
    if (image) {
      if (a.images_u8) {
        const uint8_t* s = a.images_u8 + 3 * p;
        image[3 * i] = __fdiv_rn((float)__ldg(s), 255.0f);          // = np.uint8 -> float32 / 255.0 of the dataset loader
        image[3 * i + 1] = __fdiv_rn((float)__ldg(s + 1), 255.0f);
        image[3 * i + 2] = __fdiv_rn((float)__ldg(s + 2), 255.0f);
      } else {
        const float* s = a.images_f32 + 3 * p;
        image[3 * i] = __ldg(s); image[3 * i + 1] = __ldg(s + 1); image[3 * i + 2] = __ldg(s + 2);
      }
    }
    if (fruit_mask) fruit_mask[i] = (a.masks_u8 != nullptr && __ldg(a.masks_u8 + p) != 0) ? 1.0f : 0.0f;
    // ---- RayGenerator: Cameras.generate_rays(camera_indices=c, coords=image_coords[y, x]) ------------------------------------------
    const float* cam = reinterpret_cast<const float*>(a.cameras + c);   // c2w[12] row-major [3,4], then fx, fy, cx, cy (72-byte records)
    float r[9], t[3];
#pragma unroll
    for (int row = 0; row < 3; ++row) {
      r[3 * row] = __ldg(cam + 4 * row); r[3 * row + 1] = __ldg(cam + 4 * row + 1); r[3 * row + 2] = __ldg(cam + 4 * row + 2);
      t[row] = __ldg(cam + 4 * row + 3);
    }
    const float fx = __ldg(cam + 12), fy = __ldg(cam + 13), cx = __ldg(cam + 14), cy = __ldg(cam + 15);
    const float y = (float)py + 0.5f, x = (float)px + 0.5f;
    float u = __fdiv_rn(__fsub_rn(x, cx), fx), v = -__fdiv_rn(__fsub_rn(y, cy), fy);
    const float ux = __fdiv_rn(__fadd_rn(__fsub_rn(x, cx), 1.0f), fx), vy = -__fdiv_rn(__fadd_rn(__fsub_rn(y, cy), 1.0f), fy);
    float dx, dy, dz, ex, ey, ez, gx, gy, gz;
    if (LENS) {
      // the three coordinates are undistorted independently (the offsets share one component with the ray's only before it)
      const float* lp = reinterpret_cast<const float*>(lenses + c);
      const cnb_lens l = {__ldg(lp), __ldg(lp + 1), __ldg(lp + 2), __ldg(lp + 3), __ldg(lp + 4), __ldg(lp + 5)};
      float u1 = ux, v1 = v, u2 = u, v2 = vy;
      lens_undistort(l, u, v);
      camera_direction(r, u, v, dx, dy, dz);
      if (pixel_area) {
        lens_undistort(l, u1, v1);
        lens_undistort(l, u2, v2);
        camera_direction(r, u1, v1, ex, ey, ez);
        camera_direction(r, u2, v2, gx, gy, gz);
      }
    } else {
      camera_direction(r, u, v, dx, dy, dz);
      camera_direction(r, ux, v, ex, ey, ez);
      camera_direction(r, u, vy, gx, gy, gz);
    }
    origins[3 * i] = t[0]; origins[3 * i + 1] = t[1]; origins[3 * i + 2] = t[2];
    directions[3 * i] = dx; directions[3 * i + 1] = dy; directions[3 * i + 2] = dz;
    if (pixel_area) {
      const float sx = sqrtf((dx - ex) * (dx - ex) + (dy - ey) * (dy - ey) + (dz - ez) * (dz - ez));
      const float sy = sqrtf((dx - gx) * (dx - gx) + (dy - gy) * (dy - gy) + (dz - gz) * (dz - gz));
      pixel_area[i] = sx * sy;
    }
  }
}

int launch_sample_train_batch(const cnb_image_set* set, const cnb_lens* lenses, const float* rand3, int64_t R, int32_t* indices, float* origins,
                              float* directions, float* pixel_area, int32_t* camera_indices, float* image, float* fruit_mask, cnb_stream_t stream) {
  CNB_REQUIRE(set != nullptr && R >= 0, "sample_train_batch: null image set / negative count");
  if (R == 0) return CNB_OK;
  CNB_REQUIRE(rand3 && origins && directions, "sample_train_batch: null rand / ray outputs");
  CNB_REQUIRE(set->cameras != nullptr && set->num_images > 0 && set->height > 0 && set->width > 0, "sample_train_batch: bad image set");
  CNB_REQUIRE(image == nullptr || (set->images_u8 != nullptr) != (set->images_f32 != nullptr),
              "sample_train_batch: image output needs exactly one of images_u8 / images_f32");
  static_assert(offsetof(cnb_camera, fx) == 48 && offsetof(cnb_camera, cy) == 60, "k_sample_train_batch reads cnb_camera as 16 leading floats");
  TrainBatchArgs a;
  a.images_u8 = set->images_u8; a.images_f32 = set->images_f32; a.masks_u8 = set->masks_u8; a.cameras = set->cameras;
  a.N = set->num_images; a.H = set->height; a.W = set->width;
  int64_t blocks = (R + 255) / 256;
  const int64_t cap = (int64_t)cnb_num_sms() * 16;
  if (blocks > cap) blocks = cap;
  static_assert(sizeof(cnb_lens) == 24, "k_sample_train_batch reads cnb_lens as 6 floats");
  if (lenses)
    k_sample_train_batch<true><<<(int)blocks, 256, 0, stream>>>(a, rand3, R, indices, origins, directions, pixel_area, camera_indices, image, fruit_mask,
                                                                lenses);
  else
    k_sample_train_batch<false><<<(int)blocks, 256, 0, stream>>>(a, rand3, R, indices, origins, directions, pixel_area, camera_indices, image, fruit_mask,
                                                                 nullptr);
  return cnb_check_launch("sample_train_batch");
}

}  // namespace

extern "C" int cnb_sample_train_batch(const cnb_image_set* set, const float* rand3, int64_t R, int32_t* indices, float* origins, float* directions,
                                      float* pixel_area, int32_t* camera_indices, float* image, float* fruit_mask, cnb_stream_t stream) {
  return launch_sample_train_batch(set, nullptr, rand3, R, indices, origins, directions, pixel_area, camera_indices, image, fruit_mask, stream);
}

extern "C" int cnb_sample_train_batch_lens(const cnb_image_set* set, const cnb_lens* lenses, const float* rand3, int64_t R, int32_t* indices,
                                           float* origins, float* directions, float* pixel_area, int32_t* camera_indices, float* image, float* fruit_mask,
                                           cnb_stream_t stream) {
  return launch_sample_train_batch(set, lenses, rand3, R, indices, origins, directions, pixel_area, camera_indices, image, fruit_mask, stream);
}
