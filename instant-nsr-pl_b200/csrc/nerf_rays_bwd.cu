// Persistent per-ray NeRF backward: compositing backward + both MLPs + hash-grid scatter in ONE kernel
// (autograd of models/nerf.py:95-109 through models/texture.py:23-30 and models/geometry.py:122-130).
//
// A warp owns a ray (atomic ticket queue) and walks its kept samples 16 at a time from the LAST chunk to the first,
// carrying the suffix sum  S_i = sum_{j>i} g_j w_j  in a register, so
//     d sigma_i = delta_i [ g_i (T_i - w_i) - S_i ],   d rgb_i = w_i dL/dC       (g_i = dL/dw_i)
// is produced in-kernel (no separate ray-backward launch, no d_sigma / d_rgb round trip through HBM).  The rest is
// the tile machinery of nerf_fused_bwd.cu: reload the saved 64 B/sample encoding, recompute all five layers on tensor
// cores, dgrad chain in registers, run-merged 8-byte REDs into the fp32 gradient table straight from the accumulator
// layout, weight gradients accumulated in registers across the whole kernel.  Four warps (four rays) form a CTA tile of
// 64 rows for the wgrad GEMMs; a warp that has run out of rays simply contributes no rows.
#include "nerf_fused.cuh"

namespace {

constexpr int kWarps = 4;
constexpr int kThreads = kWarps * 32;
constexpr int kRows = kWarps * 16;
constexpr int kCtasPerSm = 2;

constexpr int T_X0 = 0;
constexpr int T_H1 = T_X0 + kRows * NF_LD32;
constexpr int T_CI = T_H1 + kRows * NSR_LD64;
constexpr int T_G1 = T_CI + kRows * NF_LD32;
constexpr int T_G2 = T_G1 + kRows * NSR_LD64;
constexpr int T_DC3 = T_G2 + kRows * NSR_LD64;
constexpr int T_DG2 = T_DC3 + kRows * 24;
constexpr int T_DG1 = T_DG2 + kRows * NSR_LD64;
constexpr int T_DO = T_DG1 + kRows * NSR_LD64;
constexpr int T_DH1 = T_DO + kRows * 24;
constexpr int T_TOTAL = T_DH1 + kRows * NSR_LD64;
// per-warp scratch after the tiles (floats): d_sraw[16], d_rgb[16][3], k[16] (as float)
constexpr int kScratchFloats = 16 + 48 + 16;
constexpr size_t kSmemBytes = (size_t)(NF_W_TOTAL + T_TOTAL) * sizeof(__half) + (size_t)kWarps * kScratchFloats * sizeof(float);
constexpr int kSlots = 40 / kWarps;

struct WgradTile {
  int dy_off, ldy, x_off, ldx, m0, n0, net, base, in_dim;
};
__device__ __forceinline__ WgradTile wgrad_tile(int t) {
  WgradTile w;
  if (t < 8) {
    w = {T_DH1, NSR_LD64, T_X0, NF_LD32, (t / 2) * 16, (t % 2) * 16, 0, 0, 32};
  } else if (t < 12) {
    w = {T_DO, 24, T_H1, NSR_LD64, 0, (t - 8) * 16, 0, 64 * 32, 64};
  } else if (t < 20) {
    const int u = t - 12;
    w = {T_DG1, NSR_LD64, T_CI, NF_LD32, (u / 2) * 16, (u % 2) * 16, 1, 0, 32};
  } else if (t < 36) {
    const int u = t - 20;
    w = {T_DG2, NSR_LD64, T_G1, NSR_LD64, (u / 4) * 16, (u % 4) * 16, 1, 64 * 32, 64};
  } else {
    w = {T_DC3, 24, T_G2, NSR_LD64, 0, (t - 36) * 16, 1, 64 * 32 + 64 * 64, 64};
  }
  return w;
}

__device__ __forceinline__ void relu_mask_pack(const float (&acc)[1][8][4], const uint32_t (&post)[1][4][4], uint32_t (&out)[1][4][4]) {
#pragma unroll
  for (int k = 0; k < 4; ++k)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const __half2 hv = *reinterpret_cast<const __half2*>(&post[0][k][j]);
      const int nt = 2 * k + (j >> 1), i0 = (j & 1) * 2;
      out[0][k][j] = nsr_pack_h2(__low2float(hv) > 0.f ? acc[0][nt][i0] : 0.f, __high2float(hv) > 0.f ? acc[0][nt][i0 + 1] : 0.f);
    }
}

// wgrad over the row blocks (16 rows each) of the warps that worked this round
__device__ __forceinline__ void wgrad_tile_masked(float (&acc0)[4], float (&acc1)[4], const __half* dY, int ldy, int m0, const __half* X,
                                                  int ldx, int n0, uint32_t active_mask) {
  const int lane = threadIdx.x & 31, mi = lane >> 3, r = lane & 7;
#pragma unroll
  for (int blk = 0; blk < kWarps; ++blk) {
    if (!((active_mask >> blk) & 1u)) continue;
    const int s0 = blk * 16;
    uint32_t a[4], b[4];
    nsr_ldmatrix_x4_trans(a, dY + (size_t)(s0 + (mi >> 1) * 8 + r) * ldy + m0 + (mi & 1) * 8);
    nsr_ldmatrix_x4_trans(b, X + (size_t)(s0 + (mi & 1) * 8 + r) * ldx + n0 + (mi >> 1) * 8);
    nsr_mma16816(acc0, a, b[0], b[1]);
    nsr_mma16816(acc1, a, b[2], b[3]);
  }
}

struct RaysBwdArgs {
  const float* rays;
  const float* t_min;
  const int64_t* offsets_m;
  const int32_t* kept;
  const __half* enc_save;
  const float* sigmas;
  const float* rgbs;
  const float* weights;
  const float* trans;
  const int32_t* kidx;
  const __half* dparams;
  const __half* cparams;
  const float* g_rgb;      // [n_rays,3] or NULL
  const float* g_opacity;  // [n_rays] or NULL
  const float* g_depth;    // [n_rays] or NULL
  const float* g_weights;  // [cap] (loose layout) or NULL
  float* grad_dparams;
  float* grad_cparams;
  const float* amax;       // device scalar: bound on |dL/dw| over the kept samples (loss-scale selection)
  uint32_t* ticket;        // ray queue head (zero on entry)
  float step, loss_scale;
  int64_t n_rays;
};

__global__ void __launch_bounds__(kThreads, kCtasPerSm) nerf_rays_bwd_kernel(const __grid_constant__ nsr_nerf_t P, const RaysBwdArgs a) {
  extern __shared__ __align__(16) __half smem[];
  __shared__ int s_active[kWarps];
  __half* T = smem + NF_W_TOTAL;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, c = lane & 3;
  float* scratch = reinterpret_cast<float*>(smem + NF_W_TOTAL + T_TOTAL) + warp * kScratchFloats;
  float* s_dsraw = scratch;
  float* s_drgb = scratch + 16;
  float* s_kf = scratch + 64;
  const int r0 = warp * 16;
  float loss_scale = a.loss_scale;
  if (loss_scale <= 0.f) {
    const float amax = fmaxf(__ldg(a.amax), 1e-30f);
    loss_scale = exp2f(fminf(fmaxf(floorf(log2f(64.f / amax)), -24.f), 60.f));
  }
  const float inv_scale = 1.f / loss_scale;
  nf_stage_weights(smem, a.dparams, a.cparams, true);
  float* grad_table = a.grad_dparams + NF_DENSITY_PARAMS;
  const float inv2r = 1.f / (2.f * P.radius);

  float wacc[kSlots][2][4];
#pragma unroll
  for (int s = 0; s < kSlots; ++s)
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
      for (int i = 0; i < 4; ++i) wacc[s][j][i] = 0.f;

  // per-warp ray state
  int64_t ray = -1, base = 0;
  int chunk = -1, kept = 0;
  bool exhausted = false;
  float carry = 0.f, ox = 0.f, oy = 0.f, oz = 0.f, dx = 0.f, dy = 0.f, dz = 1.f, tmin = 0.f;
  float gr = 0.f, gg = 0.f, gb = 0.f, go = 0.f, gd = 0.f;

  for (;;) {
    __syncthreads();  // the previous round's wgrad has finished reading the tiles (first round: weights are staged)
    // ---- make sure this warp has a (ray, chunk) to work on
    while (chunk < 0 && !exhausted) {
      int64_t nr = 0;
      if (lane == 0) nr = atomicAdd(a.ticket, 1u);
      nr = __shfl_sync(0xffffffffu, nr, 0);
      if (nr >= a.n_rays) {
        exhausted = true;
        break;
      }
      const int kp = __ldg(a.kept + nr);
      if (kp <= 0) continue;
      ray = nr;
      kept = kp;
      chunk = (kp - 1) >> 4;
      carry = 0.f;
      base = a.offsets_m[ray];
      const float* rr = a.rays + ray * 6;
      ox = __ldg(rr + 0); oy = __ldg(rr + 1); oz = __ldg(rr + 2);
      dx = __ldg(rr + 3); dy = __ldg(rr + 4); dz = __ldg(rr + 5);
      tmin = __ldg(a.t_min + ray);
      gr = a.g_rgb ? __ldg(a.g_rgb + ray * 3 + 0) : 0.f;
      gg = a.g_rgb ? __ldg(a.g_rgb + ray * 3 + 1) : 0.f;
      gb = a.g_rgb ? __ldg(a.g_rgb + ray * 3 + 2) : 0.f;
      go = a.g_opacity ? __ldg(a.g_opacity + ray) : 0.f;
      gd = a.g_depth ? __ldg(a.g_depth + ray) : 0.f;
      // the SH row is the same for every sample of the ray: write this warp's 16 rows of the colour-input tile once
      float s[16];
      nsr_sh4(dx, dy, dz, s);
      if (lane < 16) {
        uint4* sp = reinterpret_cast<uint4*>(T + T_CI + (r0 + lane) * NF_LD32 + 16);
        sp[0] = make_uint4(nsr_pack_h2(s[0], s[1]), nsr_pack_h2(s[2], s[3]), nsr_pack_h2(s[4], s[5]), nsr_pack_h2(s[6], s[7]));
        sp[1] = make_uint4(nsr_pack_h2(s[8], s[9]), nsr_pack_h2(s[10], s[11]), nsr_pack_h2(s[12], s[13]), nsr_pack_h2(s[14], s[15]));
      }
    }
    const bool have = chunk >= 0;
    if (lane == 0) s_active[warp] = have ? 1 : 0;
    __syncthreads();
    uint32_t active_mask = 0u;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) active_mask |= (uint32_t)s_active[w] << w;
    if (active_mask == 0u) break;
    if (have) {
      // ---- compositing backward for the 16 rows of this chunk (both half-warps compute the same 16 rows)
      const int row = lane & 15;
      const int sidx = chunk * 16 + row;
      const bool ok = sidx < kept;
      const int64_t p = base + sidx;
      float w = 0.f, gi = 0.f, Tt = 0.f, sg = 0.f, delta = 0.f, kf = 0.f;
      if (ok) {
        w = a.weights[p];
        Tt = a.trans[p];
        sg = a.sigmas[p];
        kf = (float)a.kidx[p];
        const float t0 = __fmaf_rn(kf, a.step, tmin), t1 = __fmaf_rn(kf + 1.f, a.step, tmin);
        delta = t1 - t0;
        gi = gr * a.rgbs[p * 3 + 0] + gg * a.rgbs[p * 3 + 1] + gb * a.rgbs[p * 3 + 2] + go + gd * ((t0 + t1) * 0.5f) +
             (a.g_weights ? a.g_weights[p] : 0.f);
      }
      const float gw = gi * w;
      float suf = gw;
#pragma unroll
      for (int o = 1; o < 16; o <<= 1) {
        const float t = __shfl_down_sync(0xffffffffu, suf, o, 16);
        if (row + o < 16) suf += t;
      }
      const float ds = delta * (gi * (Tt - w) - (carry + suf - gw));
      if (lane < 16) {
        s_dsraw[row] = ds * fminf(sg, 3269017.37f) * loss_scale;  // trunc_exp backward folded in
        s_drgb[row * 3 + 0] = w * gr * loss_scale;
        s_drgb[row * 3 + 1] = w * gg * loss_scale;
        s_drgb[row * 3 + 2] = w * gb * loss_scale;
        s_kf[row] = ok ? kf : -1.f;
      }
      carry += __shfl_sync(0xffffffffu, suf, 0);
      // ---- stage the encoded features of the 16 rows
      for (int v = lane; v < 64; v += 32) {
        const int r = v >> 2, q = v & 3;
        uint4 val = make_uint4(0, 0, 0, 0);
        if (chunk * 16 + r < kept) val = __ldg(reinterpret_cast<const uint4*>(a.enc_save + (base + chunk * 16 + r) * 32) + q);
        *reinterpret_cast<uint4*>(T + T_X0 + (r0 + r) * NF_LD32 + q * 8) = val;
      }
      __syncwarp();

      // ---- forward recompute
      uint32_t a_h1[1][4][4], a_o[1][1][4], a_g1[1][4][4], a_g2[1][4][4];
      float acc[1][8][4], acc16[1][2][4];
      {
        uint32_t a_in[1][2][4];
        nsr_load_afrag<1, 2>(a_in, T + T_X0, NF_LD32, r0);
        nsr_zero_acc(acc);
        nsr_gemm_w<1, 2, 8>(acc, a_in, smem + NF_OFF_DW1, NF_LD32);
        nsr_acc_to_afrag<1, 8>(acc, a_h1, NSR_ACT_RELU);
        nsr_store_afrag<1, 4>(a_h1, T + T_H1, NSR_LD64, r0);
        nsr_zero_acc(acc16);
        nsr_gemm_w<1, 4, 2>(acc16, a_h1, smem + NF_OFF_DW2, NSR_LD64);
        nsr_acc_to_afrag<1, 2>(acc16, a_o, NSR_ACT_NONE);
        nsr_store_afrag<1, 1>(a_o, T + T_CI, NF_LD32, r0, 0);
      }
      {
        uint32_t a_c[1][2][4], a_sh[1][1][4];
        nsr_load_afrag<1, 1>(a_sh, T + T_CI + 16, NF_LD32, r0);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          a_c[0][0][j] = a_o[0][0][j];
          a_c[0][1][j] = a_sh[0][0][j];
        }
        nsr_zero_acc(acc);
        nsr_gemm_w<1, 2, 8>(acc, a_c, smem + NF_OFF_CW1, NF_LD32);
        nsr_acc_to_afrag<1, 8>(acc, a_g1, NSR_ACT_RELU);
        nsr_store_afrag<1, 4>(a_g1, T + T_G1, NSR_LD64, r0);
        nsr_zero_acc(acc);
        nsr_gemm_w<1, 4, 8>(acc, a_g1, smem + NF_OFF_CW2, NSR_LD64);
        nsr_acc_to_afrag<1, 8>(acc, a_g2, NSR_ACT_RELU);
        nsr_store_afrag<1, 4>(a_g2, T + T_G2, NSR_LD64, r0);
        nsr_zero_acc(acc16);
        nsr_gemm_w<1, 4, 2>(acc16, a_g2, smem + NF_OFF_CW3, NSR_LD64);
      }
      // ---- d(rgb pre-activation) = d_rgb * s (1 - s)
      uint32_t a_dc3[1][1][4];
      {
        float dp[4] = {0.f, 0.f, 0.f, 0.f};
        if (c < 2) {
#pragma unroll
          for (int hh = 0; hh < 2; ++hh)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
              const int col = c * 2 + e;
              if (col < 3) {
                const float raw = __half2float(__float2half_rn(acc16[0][0][hh * 2 + e]));
                const float sgm = 1.f / (1.f + expf(-raw));
                dp[hh * 2 + e] = s_drgb[(g + hh * 8) * 3 + col] * sgm * (1.f - sgm);
              }
            }
        }
        a_dc3[0][0][0] = nsr_pack_h2(dp[0], dp[1]);
        a_dc3[0][0][1] = nsr_pack_h2(dp[2], dp[3]);
        a_dc3[0][0][2] = 0u;
        a_dc3[0][0][3] = 0u;
        nsr_store_afrag<1, 1>(a_dc3, T + T_DC3, 24, r0);
      }
      // ---- dgrad chain
      uint32_t a_d[1][4][4];
      nsr_zero_acc(acc);
      nsr_gemm_wt<1, 1, 8>(acc, a_dc3, smem + NF_OFF_CW3, NSR_LD64);
      relu_mask_pack(acc, a_g2, a_d);
      nsr_store_afrag<1, 4>(a_d, T + T_DG2, NSR_LD64, r0);
      nsr_zero_acc(acc);
      nsr_gemm_wt<1, 4, 8>(acc, a_d, smem + NF_OFF_CW2, NSR_LD64);
      relu_mask_pack(acc, a_g1, a_d);
      nsr_store_afrag<1, 4>(a_d, T + T_DG1, NSR_LD64, r0);
      nsr_zero_acc(acc16);
      nsr_gemm_wt<1, 4, 2>(acc16, a_d, smem + NF_OFF_CW1, NF_LD32);
      if (c == 0) {
        acc16[0][0][0] += s_dsraw[g];
        acc16[0][0][2] += s_dsraw[g + 8];
      }
      uint32_t a_do[1][1][4];
      nsr_acc_to_afrag<1, 2>(acc16, a_do, NSR_ACT_NONE);
      nsr_store_afrag<1, 1>(a_do, T + T_DO, 24, r0);
      nsr_zero_acc(acc);
      nsr_gemm_wt<1, 1, 8>(acc, a_do, smem + NF_OFF_DW2, NSR_LD64);
      relu_mask_pack(acc, a_h1, a_d);
      nsr_store_afrag<1, 4>(a_d, T + T_DH1, NSR_LD64, r0);
      float accE[1][4][4];
      nsr_zero_acc(accE);
      nsr_gemm_wt<1, 4, 4>(accE, a_d, smem + NF_OFF_DW1, NF_LD32);

      // ---- hash-table scatter (run-merged on levels 0..7), samples (g, g+8) x levels (c, 4+c, 8+c, 12+c)
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        const float kq = s_kf[g + hh * 8];
        const bool okq = kq >= 0.f;
        const float t0 = __fmaf_rn(kq, a.step, tmin), t1 = __fmaf_rn(kq + 1.f, a.step, tmin);
        const float mid = (t0 + t1) * 0.5f;
        const float x = (fmaf(dx, mid, ox) + P.radius) * inv2r, y = (fmaf(dy, mid, oy) + P.radius) * inv2r,
                    z = (fmaf(dz, mid, oz) + P.radius) * inv2r;
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
          const float d0 = okq ? accE[0][nt][hh * 2] * inv_scale : 0.f, d1 = okq ? accE[0][nt][hh * 2 + 1] * inv_scale : 0.f;
          const LevelInfo li = nsr_level(P.grid, nt * 4 + c);
          uint32_t cx, cy, cz, idx[8];
          float fx, fy, fz;
          nsr_pos_fract(x, li.scale, cx, fx);
          nsr_pos_fract(y, li.scale, cy, fy);
          nsr_pos_fract(z, li.scale, cz, fz);
          if (nt < 2) {
            const uint32_t key = okq ? (cx + li.res * (cy + li.res * cz)) : (0xFFFFFFF0u + g);
            const uint32_t key_prev = __shfl_up_sync(0xffffffffu, key, 4);
            const bool head = (g == 0) || (key_prev != key);
            const int next_head = __shfl_down_sync(0xffffffffu, (int)head, 4);
            const bool tail = (g == 7) || next_head;
            float v[16];
#pragma unroll
            for (int cc = 0; cc < 8; ++cc) {
              const float wgt = nsr_corner_weight(cc, fx, fy, fz);
              v[2 * cc] = wgt * d0;
              v[2 * cc + 1] = wgt * d1;
            }
            bool flag = head;
#pragma unroll
            for (int o = 1; o < 8; o <<= 1) {
              const int f_up = __shfl_up_sync(0xffffffffu, (int)flag, 4 * o);
              const bool take = (g >= o) && !flag;
#pragma unroll
              for (int e = 0; e < 16; ++e) {
                const float u = __shfl_up_sync(0xffffffffu, v[e], 4 * o);
                if (take) v[e] += u;
              }
              if (take) flag = f_up;
            }
            if (okq && tail) {
              nsr_corner_indices(li, cx, cy, cz, idx);
#pragma unroll
              for (int cc = 0; cc < 8; ++cc)
                if (v[2 * cc] != 0.f || v[2 * cc + 1] != 0.f) nsr_red_add_f32x2(grad_table + 2 * (size_t)idx[cc], v[2 * cc], v[2 * cc + 1]);
            }
          } else if (okq && (d0 != 0.f || d1 != 0.f)) {
            nsr_corner_indices(li, cx, cy, cz, idx);
#pragma unroll
            for (int cc = 0; cc < 8; ++cc) {
              const float wgt = nsr_corner_weight(cc, fx, fy, fz);
              nsr_red_add_f32x2(grad_table + 2 * (size_t)idx[cc], wgt * d0, wgt * d1);
            }
          }
        }
      }
      --chunk;
    }
    __syncthreads();
    // ---- weight gradients over the rows of the warps that worked this round
#pragma unroll
    for (int s = 0; s < kSlots; ++s) {
      const WgradTile w = wgrad_tile(warp + s * kWarps);
      wgrad_tile_masked(wacc[s][0], wacc[s][1], T + w.dy_off, w.ldy, w.m0, T + w.x_off, w.ldx, w.n0, active_mask);
    }
  }
#pragma unroll
  for (int s = 0; s < kSlots; ++s) {
    const WgradTile w = wgrad_tile(warp + s * kWarps);
    float* dst = (w.net == 0 ? a.grad_dparams : a.grad_cparams) + w.base;
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int o = w.m0 + g + ((i >> 1) << 3), ii = w.n0 + j * 8 + c * 2 + (i & 1);
        const float val = wacc[s][j][i] * inv_scale;
        if (val != 0.f) atomicAdd(dst + (size_t)o * w.in_dim + ii, val);
      }
  }
}

// bound on |dL/dw_i| over the kept samples of all rays (loss-scale selection); rgb lies in [0, 1], so
//     |dL/dw_i| <= |g_rgb|_1 + |g_op| + |g_depth| * t_bound + |g_weights_i|
// One warp per ray.  g_weights is read over the ray's kept prefix only: past it the loose buffer is undefined in the static form.
__global__ void rays_grad_amax_kernel(const float* __restrict__ g_rgb, const float* __restrict__ g_op, const float* __restrict__ g_depth,
                                      const float* __restrict__ g_weights, const int64_t* __restrict__ offsets_m,
                                      const int32_t* __restrict__ kept, float t_bound, float* __restrict__ amax, int64_t n) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  float v = 0.f;
  for (int64_t i = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5); i < n; i += warps) {
    const int k = __ldg(kept + i);
    if (k <= 0) continue;
    float gw = 0.f;
    if (g_weights) {
      const int64_t base = offsets_m[i];
      for (int j = lane; j < k; j += 32) gw = fmaxf(gw, fabsf(g_weights[base + j]));
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) gw = fmaxf(gw, __shfl_xor_sync(0xffffffffu, gw, o));
    }
    float b = gw;
    if (g_rgb) b += fabsf(g_rgb[i * 3]) + fabsf(g_rgb[i * 3 + 1]) + fabsf(g_rgb[i * 3 + 2]);
    if (g_op) b += fabsf(g_op[i]);
    if (g_depth) b += fabsf(g_depth[i]) * t_bound;
    v = fmaxf(v, b);
  }
  if (lane == 0 && v > 0.f && isfinite(v)) atomicMax(reinterpret_cast<int*>(amax), __float_as_int(v));
}

}  // namespace

extern "C" int nsr_nerf_rays_bwd(const nsr_nerf_t* f, const float* rays, const float* t_min, const int64_t* offsets_m, const int32_t* kept,
                                 float step, const void* enc_save_h, const float* sigmas, const float* rgbs, const float* weights,
                                 const float* trans, const int32_t* kidx, const void* dparams_h, const void* cparams_h, const float* g_rgb,
                                 const float* g_opacity, const float* g_depth, const float* g_weights, float* grad_dparams,
                                 float* grad_cparams, float loss_scale, float* amax, float t_bound, uint32_t* ticket, int64_t n_rays,
                                 void* stream) {
  NSR_REQUIRE(f != nullptr && f->grid.n_levels == 16 && f->grid.n_features == 2 && f->feature_dim == 16 && f->density_hidden == 1 &&
                  f->color_hidden == 2,
              "nsr_nerf_rays_bwd: fused path needs L=16, F=2, feature_dim=16, hidden layers 1/2");
  NSR_REQUIRE(ticket != nullptr && amax != nullptr, "nsr_nerf_rays_bwd: ticket and amax (device scalars, zeroed) are required");
  if (n_rays == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  static thread_local bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(nerf_rays_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytes);
    if (e != cudaSuccess) {
      nsr_set_error("nsr_nerf_rays_bwd: cannot reserve %zu B shared memory: %s", kSmemBytes, cudaGetErrorString(e));
      return 2;
    }
    attr_set = true;
  }
  if (loss_scale <= 0.f) {
    rays_grad_amax_kernel<<<(int)min((int64_t)64, (n_rays + 7) / 8), 256, 0, st>>>(g_rgb, g_opacity, g_depth, g_weights, offsets_m, kept, t_bound,
                                                                                 amax, n_rays);
    NSR_CHECK_LAUNCH("nsr_nerf_rays_bwd(amax)");
  }
  RaysBwdArgs a;
  a.rays = rays; a.t_min = t_min; a.offsets_m = offsets_m; a.kept = kept; a.enc_save = (const __half*)enc_save_h;
  a.sigmas = sigmas; a.rgbs = rgbs; a.weights = weights; a.trans = trans; a.kidx = kidx;
  a.dparams = (const __half*)dparams_h; a.cparams = (const __half*)cparams_h;
  a.g_rgb = g_rgb; a.g_opacity = g_opacity; a.g_depth = g_depth; a.g_weights = g_weights;
  a.grad_dparams = grad_dparams; a.grad_cparams = grad_cparams; a.amax = amax; a.ticket = ticket;
  a.step = step; a.loss_scale = loss_scale; a.n_rays = n_rays;
  const int grid = nsr_sm_count() * kCtasPerSm;
  nerf_rays_bwd_kernel<<<grid, kThreads, kSmemBytes, st>>>(*f, a);
  NSR_CHECK_LAUNCH("nsr_nerf_rays_bwd");
  return 0;
}
