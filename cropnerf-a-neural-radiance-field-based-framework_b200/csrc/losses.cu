// Losses of the training step (row a16 of SURVEY.md section 8) and the optimiser (row f2).
//  - cnb_interlevel_fwd/bwd : nerfstudio losses.py interlevel_loss / lossfun_outer / outer (fruit_nerf.py:610)
//  - cnb_distortion_fwd     : nerfstudio losses.py distortion_loss / lossfun_distortion (fruit_nerf.py:643, metric)
//  - cnb_pixel_losses       : MSELoss(image, rgb) + w * BCEWithLogitsLoss(sem, fruit_mask) (fruit_nerf.py:601-608)
//  - cnb_adam_step          : torch.optim.Adam(lr, eps=1e-15) update (fruit_nerf_config.py:45-60)
#include "cnb_common.cuh"
#include "warp_scan.cuh"

namespace {

constexpr int WARPS = 4;
constexpr float EPS7 = 1e-7f;

// smem per warp: cp [Sp+1], cy1 [Sp+1]
__global__ void __launch_bounds__(WARPS * 32) k_interlevel(const float* __restrict__ c, const float* __restrict__ w, const float* __restrict__ cp,
                                                           const float* __restrict__ wp, int64_t R, int Sc, int Sp, float grad_scale,
                                                           float* __restrict__ loss_out, float* __restrict__ d_wp) {
  extern __shared__ float smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* cps = smem + (size_t)warp * 3 * (Sp + 1);
  float* cy1 = cps + (Sp + 1);
  float* dcy = cy1 + (Sp + 1);
  const float norm = 1.0f / (float)((double)R * (double)Sc);
  float loss_acc = 0.0f;
  for (int64_t r = blockIdx.x * (int64_t)WARPS + warp; r < R; r += (int64_t)gridDim.x * WARPS) {
    for (int j = lane; j <= Sp; j += 32) { cps[j] = __ldg(cp + r * (Sp + 1) + j); dcy[j] = 0.0f; }
    for (int j = lane; j < Sp; j += 32) cy1[1 + j] = __ldg(wp + r * Sp + j);
    if (lane == 0) cy1[0] = 0.0f;
    __syncwarp();
    cnb_warp_cumsum(cy1 + 1, cy1 + 1, Sp, lane);
    __syncwarp();
    for (int i = lane; i < Sc; i += 32) {
      const float t0s = __ldg(c + r * (Sc + 1) + i), t0e = __ldg(c + r * (Sc + 1) + i + 1);
      int lo = cnb_search_right(cps, Sp, t0s) - 1;        // over t1_starts = cp[:-1]
      lo = min(max(lo, 0), Sp - 1);
      int hi = cnb_search_right(cps + 1, Sp, t0e);        // over t1_ends = cp[1:]
      hi = min(max(hi, 0), Sp - 1);
      const float w_outer = __fsub_rn(cy1[hi + 1], cy1[lo]);
      const float wi = __ldg(w + r * Sc + i);
      const float diff = fmaxf(__fsub_rn(wi, w_outer), 0.0f);
      const float denom = __fadd_rn(wi, EPS7);
      loss_acc += diff * diff / denom;
      if (d_wp != nullptr && diff > 0.0f) {
        const float g = -2.0f * diff / denom * norm * grad_scale;  // dL / d w_outer
        atomicAdd(dcy + hi + 1, g);
        atomicAdd(dcy + lo, -g);
      }
    }
    if (d_wp != nullptr) {
      __syncwarp();
      // cy1[m] = sum_{k<m} wp_k  =>  d wp_k = sum_{m>k} dcy[m]
      cnb_warp_suffix_excl(dcy, dcy, Sp + 1, lane);
      __syncwarp();
      for (int k = lane; k < Sp; k += 32) d_wp[r * Sp + k] = dcy[k];
    }
    __syncwarp();
  }
  if (loss_out != nullptr) {
    loss_acc = cnb_warp_sum(loss_acc);
    if (lane == 0 && loss_acc != 0.0f) atomicAdd(loss_out, loss_acc * norm);
  }
}

// lossfun_distortion: sum_i w_i sum_j w_j |ut_i - ut_j| + sum_i w_i^2 (t_{i+1}-t_i)/3 ; mean over rays
__global__ void __launch_bounds__(WARPS * 32) k_distortion(const float* __restrict__ c, const float* __restrict__ w, int64_t R, int S,
                                                           float* __restrict__ loss_out) {
  extern __shared__ float smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* ut = smem + (size_t)warp * 2 * S;
  float* ws = ut + S;
  float acc = 0.0f;
  for (int64_t r = blockIdx.x * (int64_t)WARPS + warp; r < R; r += (int64_t)gridDim.x * WARPS) {
    float intra = 0.0f;
    for (int j = lane; j < S; j += 32) {
      const float t0 = __ldg(c + r * (S + 1) + j), t1 = __ldg(c + r * (S + 1) + j + 1);
      const float wj = __ldg(w + r * S + j);
      ut[j] = (t1 + t0) * 0.5f;
      ws[j] = wj;
      intra += wj * wj * (t1 - t0);
    }
    __syncwarp();
    float inter = 0.0f;
    for (int i = lane; i < S; i += 32) {
      float inner = 0.0f;
      const float ui = ut[i];
      for (int j = 0; j < S; ++j) inner = fmaf(ws[j], fabsf(ui - ut[j]), inner);
      inter = fmaf(ws[i], inner, inter);
    }
    acc += inter + intra / 3.0f;
    __syncwarp();
  }
  acc = cnb_warp_sum(acc);
  if (lane == 0 && acc != 0.0f) atomicAdd(loss_out, acc / (float)R);
}

__global__ void __launch_bounds__(256) k_pixel_losses(const float* __restrict__ rgb, const float* __restrict__ sem, const float* __restrict__ image,
                                                      const float* __restrict__ mask, int64_t R, float sem_weight, float grad_scale,
                                                      float* __restrict__ losses_out, float* __restrict__ d_rgb, float* __restrict__ d_sem) {
  float mse = 0.0f, bce = 0.0f;
  const float inv3r = 1.0f / (3.0f * (float)R), invr = 1.0f / (float)R;
  for (int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; r < R; r += (int64_t)gridDim.x * blockDim.x) {
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
      const float d = __ldg(rgb + 3 * r + ch) - __ldg(image + 3 * r + ch);
      mse = fmaf(d, d, mse);
      if (d_rgb) d_rgb[3 * r + ch] = 2.0f * d * inv3r * grad_scale;
    }
    if (sem != nullptr) {
      // BCEWithLogits: max(x,0) - x*y + log1p(exp(-|x|)) ; d/dx = sigmoid(x) - y
      const float x = __ldg(sem + r), y = __ldg(mask + r);
      bce += fmaxf(x, 0.0f) - x * y + log1pf(expf(-fabsf(x)));
      if (d_sem) d_sem[r] = (1.0f / (1.0f + expf(-x)) - y) * invr * sem_weight * grad_scale;
    }
  }
  mse = cnb_warp_sum(mse);
  bce = cnb_warp_sum(bce);
  if ((threadIdx.x & 31) == 0 && losses_out != nullptr) {
    atomicAdd(losses_out, mse * inv3r);
    if (sem != nullptr) atomicAdd(losses_out + 1, bce * invr * sem_weight);
  }
}

__global__ void __launch_bounds__(256) k_adam(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                                              int64_t n, float lr, float b1, float b2, float eps, float bc1, float bc2_sqrt, float inv_scale) {
  const float step_size = lr / bc1;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float gi = g[i] * inv_scale;
    const float mi = m[i] + (1.0f - b1) * (gi - m[i]);  // torch: exp_avg.lerp_(grad, 1 - beta1)
    const float vi = b2 * v[i] + (1.0f - b2) * gi * gi;
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    p[i] -= step_size * (mi / denom);
  }
}

// Adam + gradient clear in one pass over a flat group (float4 lanes; n is a multiple of 4 for the flat groups):
// 4 reads + 4 writes of 16 B per 4 parameters, nothing else touches the group between backward and the next forward.
// The gradient clear is issued LAST, with a fake data dependency on the updated parameter: left to itself the compiler
// hoists the (independent) zero store right behind the loads, and a store to a line whose load is still in flight
// serialises the LSU -- the pass then runs at 2.0 TB/s instead of 6.3 TB/s on B200 (tests/micro/adam_bench.cu:
// a_current vs f_late_zero; store cache policy makes no difference).
// HALF: the group holds a hash table with an fp16 copy (cnb_table_to_half); every updated float4 of the table's range [first4, first4 + count4)
// is also stored rounded to fp16 (8 bytes, from registers).  Units the update skips (unreachable rows, a skipped step) keep their copy.
struct HalfDst {
  uint2* dst;
  int64_t first4, count4;
};

template <bool HALF>
__device__ __forceinline__ void store_half(const HalfDst& hd, int64_t i, const float4& p) {
  if constexpr (HALF) {
    const int64_t j = i - hd.first4;
    if (j >= 0 && j < hd.count4) {
      const __half2 a = __floats2half2_rn(p.x, p.y), b = __floats2half2_rn(p.z, p.w);
      hd.dst[j] = make_uint2(*reinterpret_cast<const uint32_t*>(&a), *reinterpret_cast<const uint32_t*>(&b));
    }
  }
}

template <bool HALF>
__global__ void __launch_bounds__(256) k_adam_zero4(float4* __restrict__ p, float4* __restrict__ g, float4* __restrict__ m, float4* __restrict__ v,
                                                    int64_t n4, float lr, float b1, float b2, float eps, float bc1, float bc2_sqrt, float inv_scale,
                                                    const int32_t* __restrict__ skip, const uint32_t* __restrict__ live, const HalfDst hd) {
  const float step_size = lr / bc1;
  if (skip != nullptr && __ldg(skip) != 0) {
    // GradScaler.step: a non-finite gradient was found -> the optimizer step is skipped, the gradient is still cleared
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) g[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    return;
  }
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    // unreachable hash-table rows (cnb_hashgrid_mark_reachable): gradient and moments are exactly 0 forever -> the update is the identity
    if (live != nullptr && !((__ldg(live + (i >> 5)) >> (i & 31)) & 1u)) continue;
    float4 gi = g[i], mi = m[i], vi = v[i], pi = p[i];
    float* gp = &gi.x; float* mp = &mi.x; float* vp = &vi.x; float* pp = &pi.x;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float gk = gp[k] * inv_scale;
      mp[k] = mp[k] + (1.0f - b1) * (gk - mp[k]);
      vp[k] = b2 * vp[k] + (1.0f - b2) * gk * gk;
      pp[k] -= step_size * (mp[k] / (sqrtf(vp[k]) / bc2_sqrt + eps));
    }
    float z;
    asm volatile("mov.f32 %0, 0f00000000;" : "=f"(z) : "f"(pi.w));  // zero that "depends" on the finished update
    m[i] = mi; v[i] = vi; p[i] = pi;
    store_half<HALF>(hd, i, pi);
    g[i] = make_float4(z, z, z, z);
  }
}

// k_adam_zero4 with the step's scalars in device memory (read once per thread through the constant-like path)
template <bool HALF>
__global__ void __launch_bounds__(256) k_adam_zero4_dev(float4* __restrict__ p, float4* __restrict__ g, float4* __restrict__ m, float4* __restrict__ v,
                                                        int64_t n4, const float* __restrict__ sc, const uint32_t* __restrict__ live, const HalfDst hd) {
  const float lr = __ldg(sc), b1 = __ldg(sc + 1), b2 = __ldg(sc + 2), eps = __ldg(sc + 3), bc1 = __ldg(sc + 4), bc2_sqrt = __ldg(sc + 5), inv_scale = __ldg(sc + 6);
  const float step_size = lr / bc1;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    if (live != nullptr && !((__ldg(live + (i >> 5)) >> (i & 31)) & 1u)) continue;  // unreachable table rows: identity update
    float4 gi = g[i], mi = m[i], vi = v[i], pi = p[i];
    float* gp = &gi.x; float* mp = &mi.x; float* vp = &vi.x; float* pp = &pi.x;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float gk = gp[k] * inv_scale;
      mp[k] = mp[k] + (1.0f - b1) * (gk - mp[k]);
      vp[k] = b2 * vp[k] + (1.0f - b2) * gk * gk;
      pp[k] -= step_size * (mp[k] / (sqrtf(vp[k]) / bc2_sqrt + eps));
    }
    float z;
    asm volatile("mov.f32 %0, 0f00000000;" : "=f"(z) : "f"(pi.w));  // see k_adam_zero4: the clear is issued last
    m[i] = mi; v[i] = vi; p[i] = pi;
    store_half<HALF>(hd, i, pi);
    g[i] = make_float4(z, z, z, z);
  }
}

// torch.amp GradScaler's inf check (_amp_foreach_non_finite_check_and_unscale_) over one flat gradient group: found_inf |= any !isfinite
__global__ void __launch_bounds__(256) k_grad_nonfinite(const float4* __restrict__ g, int64_t n4, const float* __restrict__ tail, int ntail,
                                                        int32_t* __restrict__ found_inf) {
  bool bad = false;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    const float4 v = __ldg(g + i);
    // (x - x) is 0 for finite x and NaN for inf / NaN
    const float t = (v.x - v.x) + (v.y - v.y) + (v.z - v.z) + (v.w - v.w);
    bad |= !(t == 0.0f);
  }
  if (blockIdx.x == 0 && (int)threadIdx.x < ntail) { const float x = tail[threadIdx.x]; bad |= !((x - x) == 0.0f); }
  if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) atomicOr(found_inf, 1);
}

int ray_grid(int64_t R) {
  int64_t blocks = (R + WARPS - 1) / WARPS;
  const int64_t cap = (int64_t)cnb_num_sms() * 16;
  if (blocks > cap) blocks = cap;
  return (int)(blocks < 1 ? 1 : blocks);
}

int launch_interlevel(const float* c, const float* w, const float* cp, const float* wp, int64_t R, int Sc, int Sp, float grad_scale, float* loss_out,
                      float* d_wp, cudaStream_t stream) {
  CNB_REQUIRE(R >= 0 && Sc >= 1 && Sp >= 1 && Sp <= 4096, "interlevel: bad sizes R=%lld Sc=%d Sp=%d", (long long)R, Sc, Sp);
  if (R == 0) return CNB_OK;
  CNB_REQUIRE(c && w && cp && wp, "interlevel: null pointer");
  const size_t smem = sizeof(float) * WARPS * 3 * (size_t)(Sp + 1);
  static size_t configured = 48 * 1024;
  if (smem > configured) {
    if (cudaFuncSetAttribute(k_interlevel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return cnb_check_launch("interlevel attr");
    configured = smem;
  }
  k_interlevel<<<ray_grid(R), WARPS * 32, smem, stream>>>(c, w, cp, wp, R, Sc, Sp, grad_scale, loss_out, d_wp);
  return cnb_check_launch("interlevel");
}

}  // namespace

extern "C" int cnb_interlevel_fwd(const float* c, const float* w, const float* cp, const float* wp, int64_t R, int32_t Sc, int32_t Sp,
                                  float* loss_out, cnb_stream_t stream) {
  CNB_REQUIRE(loss_out != nullptr, "interlevel_fwd: null loss_out");
  return launch_interlevel(c, w, cp, wp, R, Sc, Sp, 0.0f, loss_out, nullptr, stream);
}

extern "C" int cnb_interlevel_bwd(const float* c, const float* w, const float* cp, const float* wp, int64_t R, int32_t Sc, int32_t Sp,
                                  float grad_scale, float* d_wp, cnb_stream_t stream) {
  CNB_REQUIRE(d_wp != nullptr, "interlevel_bwd: null d_wp");
  return launch_interlevel(c, w, cp, wp, R, Sc, Sp, grad_scale, nullptr, d_wp, stream);
}

extern "C" int cnb_distortion_fwd(const float* c, const float* w, int64_t R, int32_t S, float* loss_out, cnb_stream_t stream) {
  CNB_REQUIRE(R >= 0 && S >= 1 && S <= 4096, "distortion: bad sizes R=%lld S=%d", (long long)R, S);
  if (R == 0) return CNB_OK;
  CNB_REQUIRE(c && w && loss_out, "distortion: null pointer");
  const size_t smem = sizeof(float) * WARPS * 2 * (size_t)S;
  static size_t configured = 48 * 1024;
  if (smem > configured) {
    if (cudaFuncSetAttribute(k_distortion, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return cnb_check_launch("distortion attr");
    configured = smem;
  }
  k_distortion<<<ray_grid(R), WARPS * 32, smem, stream>>>(c, w, R, S, loss_out);
  return cnb_check_launch("distortion");
}

extern "C" int cnb_pixel_losses(const float* rgb, const float* sem, const float* image, const float* mask, int64_t R, float sem_weight,
                                float grad_scale, float* losses_out, float* d_rgb, float* d_sem, cnb_stream_t stream) {
  CNB_REQUIRE(R >= 0, "pixel_losses: bad R");
  if (R == 0) return CNB_OK;
  CNB_REQUIRE(rgb && image && (sem == nullptr || mask != nullptr), "pixel_losses: null pointer");
  int64_t blocks = (R + 255) / 256;
  const int64_t cap = (int64_t)cnb_num_sms() * 4;
  if (blocks > cap) blocks = cap;
  k_pixel_losses<<<(int)blocks, 256, 0, stream>>>(rgb, sem, image, mask, R, sem_weight, grad_scale, losses_out, d_rgb, d_sem);
  return cnb_check_launch("pixel_losses");
}

extern "C" int cnb_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float beta1, float beta2,
                             float eps, int32_t step, float inv_grad_scale, cnb_stream_t stream) {
  CNB_REQUIRE(n >= 0 && step >= 1, "adam: bad n/step");
  if (n == 0) return CNB_OK;
  CNB_REQUIRE(param && grad && exp_avg && exp_avg_sq, "adam: null pointer");
  const double bc1 = 1.0 - pow((double)beta1, (double)step);
  const double bc2 = 1.0 - pow((double)beta2, (double)step);
  int64_t blocks = (n + 255) / 256;
  const int64_t cap = (int64_t)cnb_num_sms() * 16;
  if (blocks > cap) blocks = cap;
  k_adam<<<(int)blocks, 256, 0, stream>>>(param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, (float)bc1, (float)sqrt(bc2), inv_grad_scale);
  return cnb_check_launch("adam");
}

extern "C" int cnb_adam_step_zero_dev_live(float* param, float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, const float* scalars, const uint32_t* live,
                                           cnb_stream_t stream);
extern "C" int cnb_adam_step_zero_dev(float* param, float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, const float* scalars, cnb_stream_t stream) {
  return cnb_adam_step_zero_dev_live(param, grad, exp_avg, exp_avg_sq, n, scalars, nullptr, stream);
}
// the fp16 copy of a table inside a flat group: float range [first, first + count) of the group, both multiples of 4
static int half_dst(void* table_half, int64_t first, int64_t count, int64_t n, HalfDst& hd) {
  hd.dst = static_cast<uint2*>(table_half);
  hd.first4 = first / 4;
  hd.count4 = count / 4;
  CNB_REQUIRE(table_half != nullptr && ((uintptr_t)table_half & 7) == 0, "adam: the fp16 table copy must be a non-null 8-byte aligned pointer");
  CNB_REQUIRE(first >= 0 && count >= 0 && first % 4 == 0 && count % 4 == 0 && first + count <= n,
              "adam: fp16 table range [%lld, %lld) must lie inside the group (%lld floats) on 4-float boundaries", (long long)first,
              (long long)(first + count), (long long)n);
  return CNB_OK;
}

static int adam_dev_impl(float* param, float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, const float* scalars, const uint32_t* live,
                         const HalfDst* hd, cnb_stream_t stream);

extern "C" int cnb_adam_step_zero_dev_live(float* param, float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, const float* scalars, const uint32_t* live,
                                           cnb_stream_t stream) {
  return adam_dev_impl(param, grad, exp_avg, exp_avg_sq, n, scalars, live, nullptr, stream);
}

extern "C" int cnb_adam_step_zero_dev_half(float* param, float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, const float* scalars,
                                           const uint32_t* live, void* table_half, int64_t half_first, int64_t half_count, cnb_stream_t stream) {
  HalfDst hd;
  int rc = half_dst(table_half, half_first, half_count, n, hd);
  if (rc) return rc;
  return adam_dev_impl(param, grad, exp_avg, exp_avg_sq, n, scalars, live, &hd, stream);
}

static int adam_dev_impl(float* param, float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, const float* scalars, const uint32_t* live,
                         const HalfDst* hd, cnb_stream_t stream) {
  CNB_REQUIRE(n >= 0, "adam_dev: bad n");
  if (n == 0) return CNB_OK;
  CNB_REQUIRE(param && grad && exp_avg && exp_avg_sq && scalars, "adam_dev: null pointer");
  CNB_REQUIRE((n % 4 == 0) && ((((uintptr_t)param | (uintptr_t)grad | (uintptr_t)exp_avg | (uintptr_t)exp_avg_sq) & 15) == 0),
              "adam_dev: needs a 16-byte aligned flat group with n % 4 == 0");
  const int64_t n4 = n / 4;
  int64_t blocks = (n4 + 255) / 256;
  const int64_t cap = (int64_t)cnb_num_sms() * 16;
  if (blocks > cap) blocks = cap;
  if (hd != nullptr)
    k_adam_zero4_dev<true><<<(int)blocks, 256, 0, stream>>>(reinterpret_cast<float4*>(param), reinterpret_cast<float4*>(grad),
                                                            reinterpret_cast<float4*>(exp_avg), reinterpret_cast<float4*>(exp_avg_sq), n4, scalars, live, *hd);
  else
    k_adam_zero4_dev<false><<<(int)blocks, 256, 0, stream>>>(reinterpret_cast<float4*>(param), reinterpret_cast<float4*>(grad),
                                                             reinterpret_cast<float4*>(exp_avg), reinterpret_cast<float4*>(exp_avg_sq), n4, scalars, live, HalfDst{});
  return cnb_check_launch("adam_zero_dev");
}

extern "C" int cnb_grad_check_finite(const float* grad, int64_t n, int32_t* found_inf, cnb_stream_t stream) {
  CNB_REQUIRE(n >= 0, "grad_check_finite: bad n");
  if (n == 0) return CNB_OK;
  CNB_REQUIRE(grad && found_inf, "grad_check_finite: null pointer");
  CNB_REQUIRE(((uintptr_t)grad & 15) == 0, "grad_check_finite: gradient buffer must be 16-byte aligned");
  const int64_t n4 = n / 4;
  int64_t blocks = (n4 + 255) / 256;
  const int64_t cap = (int64_t)cnb_num_sms() * 16;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  k_grad_nonfinite<<<(int)blocks, 256, 0, stream>>>(reinterpret_cast<const float4*>(grad), n4, grad + 4 * n4, (int)(n - 4 * n4), found_inf);
  return cnb_check_launch("grad_check_finite");
}

static int adam_step_zero_impl(float* param, float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float beta1, float beta2,
                               float eps, int32_t step, float inv_grad_scale, const int32_t* skip_flag, cnb_stream_t stream, const uint32_t* live = nullptr,
                               const HalfDst* hd = nullptr);

extern "C" int cnb_adam_step_zero_half(float* param, float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float beta1, float beta2,
                                       float eps, int32_t step, float inv_grad_scale, const int32_t* skip_flag, const uint32_t* live, void* table_half,
                                       int64_t half_first, int64_t half_count, cnb_stream_t stream) {
  CNB_REQUIRE(n % 4 == 0 && ((((uintptr_t)param | (uintptr_t)grad | (uintptr_t)exp_avg | (uintptr_t)exp_avg_sq) & 15) == 0),
              "adam_step_zero_half: needs a 16-byte aligned flat group with n % 4 == 0");
  HalfDst hd;
  int rc = half_dst(table_half, half_first, half_count, n, hd);
  if (rc) return rc;
  return adam_step_zero_impl(param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, step, inv_grad_scale, skip_flag, stream, live, &hd);
}

extern "C" int cnb_adam_step_zero_live(float* param, float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float beta1, float beta2,
                                       float eps, int32_t step, float inv_grad_scale, const uint32_t* live, cnb_stream_t stream) {
  CNB_REQUIRE(live == nullptr || (n % 4 == 0 && ((((uintptr_t)param | (uintptr_t)grad | (uintptr_t)exp_avg | (uintptr_t)exp_avg_sq) & 15) == 0)),
              "adam_step_zero_live: the masked step needs a 16-byte aligned flat group with n % 4 == 0");
  return adam_step_zero_impl(param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, step, inv_grad_scale, nullptr, stream, live);
}

extern "C" int cnb_adam_step_zero(float* param, float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float beta1, float beta2,
                                  float eps, int32_t step, float inv_grad_scale, cnb_stream_t stream) {
  return adam_step_zero_impl(param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, step, inv_grad_scale, nullptr, stream);
}

extern "C" int cnb_adam_step_zero_guarded(float* param, float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float beta1, float beta2,
                                          float eps, int32_t step, float inv_grad_scale, const int32_t* skip_flag, cnb_stream_t stream) {
  CNB_REQUIRE(skip_flag == nullptr || (n % 4 == 0 && ((((uintptr_t)param | (uintptr_t)grad | (uintptr_t)exp_avg | (uintptr_t)exp_avg_sq) & 15) == 0)),
              "adam_step_zero_guarded: the guarded step needs a 16-byte aligned flat group with n % 4 == 0");
  return adam_step_zero_impl(param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, step, inv_grad_scale, skip_flag, stream);
}

static int adam_step_zero_impl(float* param, float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float beta1, float beta2,
                               float eps, int32_t step, float inv_grad_scale, const int32_t* skip_flag, cnb_stream_t stream, const uint32_t* live,
                               const HalfDst* hd) {
  CNB_REQUIRE(n >= 0 && step >= 1, "adam: bad n/step");
  if (n == 0) return CNB_OK;
  CNB_REQUIRE(param && grad && exp_avg && exp_avg_sq, "adam: null pointer");
  const bool vec = (n % 4 == 0) && ((((uintptr_t)param | (uintptr_t)grad | (uintptr_t)exp_avg | (uintptr_t)exp_avg_sq) & 15) == 0);
  if (!vec) {
    int rc = cnb_adam_step(param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, step, inv_grad_scale, stream);
    if (rc) return rc;
    if (cudaMemsetAsync(grad, 0, sizeof(float) * n, stream) != cudaSuccess) return cnb_check_launch("adam memset");
    return CNB_OK;
  }
  const double bc1 = 1.0 - pow((double)beta1, (double)step);
  const double bc2 = 1.0 - pow((double)beta2, (double)step);
  const int64_t n4 = n / 4;
  int64_t blocks = (n4 + 255) / 256;
  const int64_t cap = (int64_t)cnb_num_sms() * 16;
  if (blocks > cap) blocks = cap;
  if (hd != nullptr)
    k_adam_zero4<true><<<(int)blocks, 256, 0, stream>>>(reinterpret_cast<float4*>(param), reinterpret_cast<float4*>(grad), reinterpret_cast<float4*>(exp_avg),
                                                        reinterpret_cast<float4*>(exp_avg_sq), n4, lr, beta1, beta2, eps, (float)bc1, (float)sqrt(bc2),
                                                        inv_grad_scale, skip_flag, live, *hd);
  else
    k_adam_zero4<false><<<(int)blocks, 256, 0, stream>>>(reinterpret_cast<float4*>(param), reinterpret_cast<float4*>(grad), reinterpret_cast<float4*>(exp_avg),
                                                         reinterpret_cast<float4*>(exp_avg_sq), n4, lr, beta1, beta2, eps, (float)bc1, (float)sqrt(bc2),
                                                         inv_grad_scale, skip_flag, live, HalfDst{});
  return cnb_check_launch("adam_zero");
}
