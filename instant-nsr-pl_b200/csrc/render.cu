// Per-ray transmittance scans and compositing: nerfacc 0.3.3 `render_visibility`,
// `render_weight_from_density`, `render_weight_from_alpha`, `accumulate_along_rays`
// (models/nerf.py:87-92,105-109; models/neus.py:181-184,237-243).
// One warp per ray walks the ray's contiguous sample segment in chunks of 32 with shuffle scans and a
// running carry -- no CUB scan-by-key over the whole batch, no atomics, deterministic results.
#include "common.cuh"

namespace {

constexpr int kWarps = 8;

__device__ __forceinline__ float warp_incl_sum(float v, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const float t = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += t;
  }
  return v;
}
__device__ __forceinline__ float warp_incl_prod(float v, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const float t = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v *= t;
  }
  return v;
}
// inclusive suffix sum (lane i gets sum over lanes >= i)
__device__ __forceinline__ float warp_suffix_sum(float v, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const float t = __shfl_down_sync(0xffffffffu, v, o);
    if (lane + o < 32) v += t;
  }
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

#define RAY_PROLOGUE                                                      \
  const int lane = threadIdx.x & 31;                                      \
  const int64_t ray = blockIdx.x * (int64_t)kWarps + (threadIdx.x >> 5);  \
  if (ray >= n_rays) return;                                              \
  const int64_t beg = offsets[ray], end = offsets[ray + 1];

__global__ void __launch_bounds__(kWarps * 32) visibility_kernel(const float* __restrict__ alphas, const int64_t* __restrict__ offsets,
                                                                 uint8_t* __restrict__ keep, float* __restrict__ trans,
                                                                 int32_t* __restrict__ kept_counts, float eps, float alpha_thre,
                                                                 int64_t n_rays) {
  RAY_PROLOGUE
  float carry = 1.f;
  int kept = 0;
  for (int64_t b = beg; b < end; b += 32) {
    const int64_t i = b + lane;
    const float a = i < end ? alphas[i] : 0.f;
    const float incl = warp_incl_prod(1.f - a, lane);
    float excl = __shfl_up_sync(0xffffffffu, incl, 1);
    if (lane == 0) excl = 1.f;
    const float T = carry * excl;
    bool k = (i < end) && (T >= eps);
    if (alpha_thre > 0.f) k = k && (a >= alpha_thre);
    if (i < end) {
      keep[i] = k ? 1 : 0;
      if (trans) trans[i] = T;
    }
    kept += __popc(__ballot_sync(0xffffffffu, k));
    carry *= __shfl_sync(0xffffffffu, incl, 31);
    if (alpha_thre <= 0.f && carry < eps) {  // everything after is dropped: finish the bookkeeping
      for (int64_t j = b + 32 + lane; j < end; j += 32) {
        keep[j] = 0;
        if (trans) trans[j] = 0.f;  // below early_stop_eps; exact value is not part of the contract
      }
      break;
    }
  }
  if (lane == 0 && kept_counts) kept_counts[ray] = kept;
}

__global__ void __launch_bounds__(kWarps * 32) weight_density_fwd_kernel(const float* __restrict__ t_starts, const float* __restrict__ t_ends,
                                                                         const float* __restrict__ sigmas, const int64_t* __restrict__ offsets,
                                                                         float* __restrict__ weights, float* __restrict__ trans,
                                                                         int64_t n_rays) {
  RAY_PROLOGUE
  float carry = 0.f;
  for (int64_t b = beg; b < end; b += 32) {
    const int64_t i = b + lane;
    const float sd = i < end ? sigmas[i] * (t_ends[i] - t_starts[i]) : 0.f;
    const float incl = warp_incl_sum(sd, lane);
    // exclusive sum from the neighbour, not incl - sd: after a sample with a huge sigma * delta (an opaque surface) that difference loses
    // every earlier term to rounding, and inf - inf is NaN
    float excl = __shfl_up_sync(0xffffffffu, incl, 1);
    if (lane == 0) excl = 0.f;
    const float T = __expf(-(carry + excl));
    if (i < end) {
      weights[i] = T * (1.f - __expf(-sd));
      if (trans) trans[i] = T;
    }
    carry += __shfl_sync(0xffffffffu, incl, 31);
  }
}

// d sigma_i = delta_i * [ g_i * (T_i - w_i) - sum_{j>i} g_j w_j ]
__global__ void __launch_bounds__(kWarps * 32) weight_density_bwd_kernel(const float* __restrict__ t_starts, const float* __restrict__ t_ends,
                                                                         const float* __restrict__ weights, const float* __restrict__ trans,
                                                                         const float* __restrict__ grad_weights,
                                                                         const int64_t* __restrict__ offsets, float* __restrict__ grad_sigmas,
                                                                         int64_t n_rays) {
  RAY_PROLOGUE
  float carry = 0.f;  // sum of g_j w_j over the chunks after the current one
  const int64_t n = end - beg;
  for (int64_t cb = ((n - 1) / 32) * 32; cb >= 0 && n > 0; cb -= 32) {
    const int64_t i = beg + cb + lane;
    const bool ok = i < end;
    const float w = ok ? weights[i] : 0.f, g = ok ? grad_weights[i] : 0.f;
    const float gw = g * w;
    const float suf = warp_suffix_sum(gw, lane);  // includes own
    float after = __shfl_down_sync(0xffffffffu, suf, 1);  // sum over the later lanes (suf - gw cancels when g_i w_i dominates it)
    if (lane == 31) after = 0.f;
    if (ok) grad_sigmas[i] = (t_ends[i] - t_starts[i]) * (g * (trans[i] - w) - (carry + after));
    carry += __shfl_sync(0xffffffffu, suf, 0);
  }
}

__global__ void __launch_bounds__(kWarps * 32) weight_alpha_fwd_kernel(const float* __restrict__ alphas, const int64_t* __restrict__ offsets,
                                                                       float* __restrict__ weights, float* __restrict__ trans, int64_t n_rays) {
  RAY_PROLOGUE
  float carry = 1.f;
  for (int64_t b = beg; b < end; b += 32) {
    const int64_t i = b + lane;
    const float a = i < end ? alphas[i] : 0.f;
    const float incl = warp_incl_prod(1.f - a, lane);
    float excl = __shfl_up_sync(0xffffffffu, incl, 1);
    if (lane == 0) excl = 1.f;
    const float T = carry * excl;
    if (i < end) {
      weights[i] = T * a;
      if (trans) trans[i] = T;
    }
    carry *= __shfl_sync(0xffffffffu, incl, 31);
  }
}

// d alpha_i = g_i T_i - (sum_{j>i} g_j w_j) / (1 - alpha_i)
__global__ void __launch_bounds__(kWarps * 32) weight_alpha_bwd_kernel(const float* __restrict__ alphas, const float* __restrict__ weights,
                                                                       const float* __restrict__ trans, const float* __restrict__ grad_weights,
                                                                       const int64_t* __restrict__ offsets, float* __restrict__ grad_alphas,
                                                                       int64_t n_rays) {
  RAY_PROLOGUE
  float carry = 0.f;
  const int64_t n = end - beg;
  for (int64_t cb = ((n - 1) / 32) * 32; cb >= 0 && n > 0; cb -= 32) {
    const int64_t i = beg + cb + lane;
    const bool ok = i < end;
    const float w = ok ? weights[i] : 0.f, g = ok ? grad_weights[i] : 0.f;
    const float gw = g * w;
    const float suf = warp_suffix_sum(gw, lane);
    if (ok) grad_alphas[i] = g * trans[i] - (carry + suf - gw) / fmaxf(1.f - alphas[i], 1e-10f);
    carry += __shfl_sync(0xffffffffu, suf, 0);
  }
}

__global__ void __launch_bounds__(kWarps * 32) accumulate_kernel(const float* __restrict__ weights, const float* __restrict__ values,
                                                                 const int64_t* __restrict__ offsets, float* __restrict__ out, int d,
                                                                 int64_t n_rays) {
  RAY_PROLOGUE
  for (int c0 = 0; c0 < d; c0 += 4) {
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    for (int64_t i = beg + lane; i < end; i += 32) {
      const float w = weights[i];
#pragma unroll
      for (int c = 0; c < 4; ++c)
        if (c0 + c < d) acc[c] += values ? w * values[i * d + c0 + c] : w;
    }
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const float s = warp_sum(acc[c]);
      if (lane == 0 && c0 + c < d) out[ray * d + c0 + c] = s;
    }
  }
}

// ---- NeuS compositing in one pass per direction (models/neus.py:237-243: render_weight_from_alpha + 4x accumulate_along_rays).
// forward: weights, transmittance, opacity, depth, rgb and (un-normalised) normal sums per ray.
__global__ void __launch_bounds__(kWarps * 32) neus_composite_fwd_kernel(const float* __restrict__ alphas, const float* __restrict__ rgbs,
                                                                         const float* __restrict__ normals, const float* __restrict__ t_starts,
                                                                         const float* __restrict__ t_ends, const int64_t* __restrict__ offsets,
                                                                         float* __restrict__ weights, float* __restrict__ trans,
                                                                         float* __restrict__ opacity, float* __restrict__ depth,
                                                                         float* __restrict__ comp_rgb, float* __restrict__ comp_normal,
                                                                         int64_t n_rays) {
  RAY_PROLOGUE
  float carry = 1.f;
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};  // opacity, depth, rgb, normal
  for (int64_t b = beg; b < end; b += 32) {
    const int64_t i = b + lane;
    const bool ok = i < end;
    const float a = ok ? alphas[i] : 0.f;
    const float incl = warp_incl_prod(1.f - a, lane);
    float excl = __shfl_up_sync(0xffffffffu, incl, 1);
    if (lane == 0) excl = 1.f;
    const float T = carry * excl;
    const float w = T * a;
    if (ok) {
      weights[i] = w;
      trans[i] = T;
      acc[0] += w;
      acc[1] += w * ((t_starts[i] + t_ends[i]) * 0.5f);
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        acc[2 + c] += w * rgbs[i * 3 + c];
        acc[5 + c] += w * normals[i * 3 + c];
      }
    }
    carry *= __shfl_sync(0xffffffffu, incl, 31);
  }
#pragma unroll
  for (int c = 0; c < 8; ++c) acc[c] = warp_sum(acc[c]);
  if (lane == 0) {
    opacity[ray] = acc[0];
    depth[ray] = acc[1];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      comp_rgb[ray * 3 + c] = acc[2 + c];
      comp_normal[ray * 3 + c] = acc[5 + c];
    }
  }
}

// backward: g_w = g_opacity + g_depth * mid + g_rgb . rgb + g_normal . n (+ g_weights); d alpha as in weight_alpha_bwd_kernel;
// d rgb_i = w_i g_rgb[ray], d normal_i = w_i g_normal[ray].
__global__ void __launch_bounds__(kWarps * 32) neus_composite_bwd_kernel(const float* __restrict__ alphas, const float* __restrict__ rgbs,
                                                                         const float* __restrict__ normals, const float* __restrict__ t_starts,
                                                                         const float* __restrict__ t_ends, const float* __restrict__ weights,
                                                                         const float* __restrict__ trans, const int64_t* __restrict__ offsets,
                                                                         const float* __restrict__ g_weights, const float* __restrict__ g_opacity,
                                                                         const float* __restrict__ g_depth, const float* __restrict__ g_rgb,
                                                                         const float* __restrict__ g_normal, float* __restrict__ d_alphas,
                                                                         float* __restrict__ d_rgbs, float* __restrict__ d_normals,
                                                                         int64_t n_rays) {
  RAY_PROLOGUE
  const float go = g_opacity ? g_opacity[ray] : 0.f, gd = g_depth ? g_depth[ray] : 0.f;
  float gc[3] = {0.f, 0.f, 0.f}, gn[3] = {0.f, 0.f, 0.f};
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    if (g_rgb) gc[c] = g_rgb[ray * 3 + c];
    if (g_normal) gn[c] = g_normal[ray * 3 + c];
  }
  float carry = 0.f;
  const int64_t n = end - beg;
  for (int64_t cb = ((n - 1) / 32) * 32; cb >= 0 && n > 0; cb -= 32) {
    const int64_t i = beg + cb + lane;
    const bool ok = i < end;
    float w = 0.f, g = 0.f;
    if (ok) {
      w = weights[i];
      g = go + gd * ((t_starts[i] + t_ends[i]) * 0.5f);
#pragma unroll
      for (int c = 0; c < 3; ++c) g += gc[c] * rgbs[i * 3 + c] + gn[c] * normals[i * 3 + c];
      if (g_weights) g += g_weights[i];
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        d_rgbs[i * 3 + c] = w * gc[c];
        d_normals[i * 3 + c] = w * gn[c];
      }
    }
    const float gw = g * w;
    const float suf = warp_suffix_sum(gw, lane);
    if (ok) d_alphas[i] = g * trans[i] - (carry + suf - gw) / fmaxf(1.f - alphas[i], 1e-10f);
    carry += __shfl_sync(0xffffffffu, suf, 0);
  }
}

}  // namespace

#define RAY_LAUNCH(kernel, name, ...)                                                                       \
  do {                                                                                                      \
    if (n_rays == 0) return 0;                                                                              \
    kernel<<<nsr_blocks(n_rays, kWarps), kWarps * 32, 0, (cudaStream_t)stream>>>(__VA_ARGS__);              \
    NSR_CHECK_LAUNCH(name);                                                                                 \
    return 0;                                                                                               \
  } while (0)

extern "C" int nsr_visibility(const float* alphas, const int64_t* offsets, uint8_t* keep, float* trans, int32_t* kept_counts,
                              float early_stop_eps, float alpha_thre, int64_t n_rays, void* stream) {
  RAY_LAUNCH(visibility_kernel, "nsr_visibility", alphas, offsets, keep, trans, kept_counts, early_stop_eps, alpha_thre, n_rays);
}
extern "C" int nsr_weight_from_density_fwd(const float* t_starts, const float* t_ends, const float* sigmas, const int64_t* offsets,
                                           float* weights, float* trans, int64_t n_rays, void* stream) {
  RAY_LAUNCH(weight_density_fwd_kernel, "nsr_weight_from_density_fwd", t_starts, t_ends, sigmas, offsets, weights, trans, n_rays);
}
extern "C" int nsr_weight_from_density_bwd(const float* t_starts, const float* t_ends, const float* weights, const float* trans,
                                           const float* grad_weights, const int64_t* offsets, float* grad_sigmas, int64_t n_rays,
                                           void* stream) {
  RAY_LAUNCH(weight_density_bwd_kernel, "nsr_weight_from_density_bwd", t_starts, t_ends, weights, trans, grad_weights, offsets,
             grad_sigmas, n_rays);
}
extern "C" int nsr_weight_from_alpha_fwd(const float* alphas, const int64_t* offsets, float* weights, float* trans, int64_t n_rays,
                                         void* stream) {
  RAY_LAUNCH(weight_alpha_fwd_kernel, "nsr_weight_from_alpha_fwd", alphas, offsets, weights, trans, n_rays);
}
extern "C" int nsr_weight_from_alpha_bwd(const float* alphas, const float* weights, const float* trans, const float* grad_weights,
                                         const int64_t* offsets, float* grad_alphas, int64_t n_rays, void* stream) {
  RAY_LAUNCH(weight_alpha_bwd_kernel, "nsr_weight_from_alpha_bwd", alphas, weights, trans, grad_weights, offsets, grad_alphas, n_rays);
}
extern "C" int nsr_accumulate(const float* weights, const float* values, const int64_t* offsets, float* out, int32_t d, int64_t n_rays,
                              void* stream) {
  NSR_REQUIRE(d >= 1, "nsr_accumulate: d must be >= 1");
  RAY_LAUNCH(accumulate_kernel, "nsr_accumulate", weights, values, offsets, out, d, n_rays);
}

extern "C" int nsr_neus_composite_fwd(const float* alphas, const float* rgbs, const float* normals, const float* t_starts,
                                      const float* t_ends, const int64_t* offsets, float* weights, float* trans, float* opacity,
                                      float* depth, float* comp_rgb, float* comp_normal, int64_t n_rays, void* stream) {
  RAY_LAUNCH(neus_composite_fwd_kernel, "nsr_neus_composite_fwd", alphas, rgbs, normals, t_starts, t_ends, offsets, weights, trans, opacity,
             depth, comp_rgb, comp_normal, n_rays);
}
extern "C" int nsr_neus_composite_bwd(const float* alphas, const float* rgbs, const float* normals, const float* t_starts,
                                      const float* t_ends, const float* weights, const float* trans, const int64_t* offsets,
                                      const float* g_weights, const float* g_opacity, const float* g_depth, const float* g_rgb,
                                      const float* g_normal, float* d_alphas, float* d_rgbs, float* d_normals, int64_t n_rays,
                                      void* stream) {
  RAY_LAUNCH(neus_composite_bwd_kernel, "nsr_neus_composite_bwd", alphas, rgbs, normals, t_starts, t_ends, weights, trans, offsets,
             g_weights, g_opacity, g_depth, g_rgb, g_normal, d_alphas, d_rgbs, d_normals, n_rays);
}
