// Backward of the render_rays training step (reference: train.py:103-117 loss.backward() through
// models/rendering.py:143-170 and models/nerf.py:100-124), hand-written for sm_100a.
//
// The forward launch in "train" mode (render_kernel.cuh, kSave) leaves per sample in the training
// workspace: the encoded input, the 8 hidden activations (fp16, tiled layout of layout.h), the ReLU
// sign bits of the 8 hidden layers, the direction-layer output, raw sigma and rgb.  The backward is
//
//   composite_bwd_kernel  warp per ray: d(rgb, depth, opacity) [or the fused MSE seed] -> per-sample
//                         d sigma, d rgb_pre                                   (CUDA cores)
//   head_bwd_kernel       rgb head + ReLU of the direction layer: dd (tiled 16-bit), the rgb-head and
//                         direction-part weight gradients                      (CUDA cores)
//   chain_bwd_kernel      dgrad chain on the tcgen05 tile engine: per 128-sample tile
//                         dd -> dh8 -> dpre8 -> ... -> dpre1, activations in TMEM exactly like the
//                         forward, 30 transposed weight slices per tile; writes dpre_l (tiled)
//   wgrad_kernel          split-K tcgen05 GEMMs gW_l = dpre_l^T h_{l-1}: one CTA per (layer, sample
//                         range), both operands MN-major straight from the tiled arrays, fp32
//                         accumulators in TMEM for the CTA's whole range; bias gradients as column
//                         sums on the CUDA cores of the same tiles
//   wgrad_reduce_kernel   fixed-order sum of the per-CTA partials into the .grad tensors
//   unfold_kernel         chain rule through the pack-time folding W' = W_dir[:, :256] W_final
//
// Per-sample gradients are fp16 with a power-of-two scale PER LAYER, chosen on the device in the
// same step (no state carried between steps, deterministic): level 0 (dd) from a bound on its
// largest element, |d rgb_pre|_max * max_n sum_c |W_rgb[c][n]|; levels 1..8 (dpre_8..dpre_1) from
// that bound times the growth factor of each level, which a PROBE pass of the chain kernel measures on one
// tile per SM (no stores; bwd_scale_kernel), each mapped to 64 (10 bits of headroom to the fp16 maximum,
// 20 bits of normal range below; the real pass counts what still saturates; gradients
// shrink or grow by orders of magnitude through 8 layers, one global scale costs precision in the
// deep layers: measured 4e-2 relative error at layer 1 vs 4e-3 with per-layer scales).
// Conversions saturate instead of producing inf; the weight gradients accumulate in fp32 and are
// un-scaled per layer by the reduction.
// fp16 rather than bf16 because the wgrad GEMM contracts the gradients with the forward's fp16
// activations and tcgen05.mma kind::f16 does not take mixed bf16 x fp16 operands (measured: illegal
// instruction, tools/gpu_probe.py gemm_mn); -DNERFB200_BWD_BF16 builds the all-bf16 variant for
// experiments (it needs bf16 activations from the forward and is not wired up).
#pragma once
#include <cuda_bf16.h>

#include "render_kernel.cuh"

namespace nerfb200 {

#ifdef NERFB200_BWD_BF16
constexpr bool kBwdBf16 = true;
#else
constexpr bool kBwdBf16 = false;
#endif
constexpr uint32_t kBwdFmt = kBwdBf16 ? 1u : 0u;      // instruction-descriptor format code: 0 = f16, 1 = bf16

__device__ __forceinline__ uint32_t cvt_bwd_x2(float lo, float hi) {
  uint32_t d;
  if (kBwdBf16) asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
  else asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
  return d;
}
__device__ __forceinline__ uint16_t cvt_bwd(float v) {
  if (kBwdBf16) return __bfloat16_as_ushort(__float2bfloat16_rn(v));
  return static_cast<uint16_t>(cvt_bwd_x2(v, 0.f) & 0xFFFFu);
}
// packed 16-bit add (gradient element type)
__device__ __forceinline__ uint32_t bwd_add_x2(uint32_t a, uint32_t b) {
  uint32_t d;
  if (kBwdBf16) asm("add.rn.bf16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
  else asm("add.rn.f16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
  return d;
}
__device__ __forceinline__ float2 bwd_x2_to_float2(uint32_t p) {
  if (kBwdBf16) return make_float2(__uint_as_float(p << 16), __uint_as_float(p & 0xFFFF0000u));
  return __half22float2(*reinterpret_cast<const __half2*>(&p));
}

// ------------------------------------------------------------------------- compositing backward
// models/rendering.py:143-170 differentiated by hand (oracle/nerf_oracle_grad.py
// volume_render_backward is the executable statement of the same formulas):
//   w_i = alpha_i T_i,  T_i = prod_{j<i} (1 - alpha_j + 1e-10),  alpha_i = 1 - exp(-delta_i relu(s_i))
//   dL/dw_i     = <g_rgb, c_i> + g_depth z_i + g_opac - [white_back] sum_ch g_rgb
//   dL/dalpha_i = T_i dL/dw_i - (sum_{j>i} w_j dL/dw_j) / (1 - alpha_i + 1e-10)
//   dL/dsigma_i = dL/dalpha_i delta_i exp(-delta_i relu(s_i)) [s_i > 0]
//   dL/dc_i     = w_i g_rgb;  through the sigmoid: dL/dpre_i = dL/dc_i c_i (1 - c_i)
// One warp per ray, each lane owns P = S / 32 consecutive samples.
struct CompBwdParams {
  int n_rays, S;
  long long n_pad;
  const float* z;
  const float* sigma;
  const float* rgb;
  const float* rays;
  long long ray_stride;
  const float* noise;       // (n_rays, S) or null
  float noise_std;
  int white_back;
  const float* g_rgb;       // (n_rays, 3) upstream gradient or null
  const float* g_depth;     // (n_rays) or null
  const float* g_opac;      // (n_rays) or null
  const float* rgb_out;     // (n_rays, 3) rendered colour, used with `target`
  const float* target;      // (n_rays, 3) or null: adds the MSE seed 2 (rgb_out - target) / (3 n_rays) * loss_grad
  const float* loss_grad;   // device scalar dL/dloss or null (= 1)
  float* dsigma;
  float* dprergb;
  unsigned* amax_bits;      // [2]: max |d sigma|, max |d rgb_pre| as float bits (scale selection) or null
  unsigned* tile_amax;      // [n_pad / 128][2]: the same two maxima per 128-sample tile (zero on entry)
};

__global__ void __launch_bounds__(128) composite_bwd_kernel(const CompBwdParams p) {
  const int lane = threadIdx.x & 31;
  const int wpb = blockDim.x >> 5;
  const long long ray = static_cast<long long>(blockIdx.x) * wpb + (threadIdx.x >> 5);
  const int S = p.S, P = S >> 5;
  float amax = 0.f, amax_rgb = 0.f;
  if (ray < p.n_rays) {
    const float* rr = p.rays + ray * p.ray_stride;
    const float dx = rr[3], dy = rr[4], dz = rr[5];
    const float dnorm = sqrtf(__fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz)));
    float g[3] = {0.f, 0.f, 0.f};
    if (p.g_rgb != nullptr) { g[0] = p.g_rgb[ray * 3]; g[1] = p.g_rgb[ray * 3 + 1]; g[2] = p.g_rgb[ray * 3 + 2]; }
    if (p.target != nullptr) {
      const float lg = (p.loss_grad != nullptr) ? *p.loss_grad : 1.f;
      const float k = 2.f * lg / (3.f * static_cast<float>(p.n_rays));
#pragma unroll
      for (int c = 0; c < 3; ++c) g[c] += k * (p.rgb_out[ray * 3 + c] - p.target[ray * 3 + c]);
    }
    const float gd = (p.g_depth != nullptr) ? p.g_depth[ray] : 0.f;
    float go = (p.g_opac != nullptr) ? p.g_opac[ray] : 0.f;
    if (p.white_back) go -= g[0] + g[1] + g[2];
    const float* z = p.z + ray * S;
    const long long g0 = ray * S;
    float alpha[6], tloc[6], om[6], dw[6], de[6], wgt[6];
    bool pos[6];
    float prod = 1.f;
    for (int q = 0; q < P; ++q) {
      const int i = lane * P + q;
      float delta = (i < S - 1) ? __fsub_rn(z[i + 1], z[i]) : 1e10f;
      delta = __fmul_rn(delta, dnorm);
      float s = p.sigma[g0 + i];
      if (p.noise != nullptr) s = __fadd_rn(s, __fmul_rn(p.noise[g0 + i], p.noise_std));
      const float e = expf(-__fmul_rn(delta, fmaxf(s, 0.f)));
      alpha[q] = __fsub_rn(1.f, e);
      om[q] = __fadd_rn(__fsub_rn(1.f, alpha[q]), 1e-10f);
      de[q] = delta * e;
      pos[q] = s > 0.f;
      tloc[q] = prod;
      prod = __fmul_rn(prod, om[q]);
      const float* c = p.rgb + (g0 + i) * 3;
      dw[q] = g[0] * c[0] + g[1] * c[1] + g[2] * c[2] + gd * z[i] + go;
    }
    float incl = prod;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const float v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl *= v;
    }
    float excl = __shfl_up_sync(0xffffffffu, incl, 1);
    if (lane == 0) excl = 1.f;
    // suffix sums of a_i = w_i dL/dw_i (exclusive, from the far end)
    float asum = 0.f;
    for (int q = 0; q < P; ++q) {
      tloc[q] *= excl;                     // T_i
      wgt[q] = alpha[q] * tloc[q];         // w_i
      asum += wgt[q] * dw[q];
    }
    float sincl = asum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const float v = __shfl_down_sync(0xffffffffu, sincl, o);
      if (lane + o < 32) sincl += v;
    }
    float after = __shfl_down_sync(0xffffffffu, sincl, 1);     // sum over lanes > this one
    if (lane == 31) after = 0.f;
    float run = after;
    for (int q = P - 1; q >= 0; --q) {
      const int i = lane * P + q;
      const float dalpha = tloc[q] * dw[q] - run / om[q];
      run += wgt[q] * dw[q];
      const float ds = pos[q] ? dalpha * de[q] : 0.f;
      p.dsigma[g0 + i] = ds;
      amax = fmaxf(amax, fabsf(ds));
      const float* c = p.rgb + (g0 + i) * 3;
#pragma unroll
      for (int ch = 0; ch < 3; ++ch) {
        const float dp = wgt[q] * g[ch] * c[ch] * (1.f - c[ch]);
        p.dprergb[(g0 + i) * 3 + ch] = dp;
        amax_rgb = fmaxf(amax_rgb, fabsf(dp));
      }
    }
  }
  // padding rows carry no gradient
  const long long n = static_cast<long long>(p.n_rays) * S;
  if (blockIdx.x == gridDim.x - 1)
    for (long long i = n + threadIdx.x; i < p.n_pad; i += blockDim.x) {
      p.dsigma[i] = 0.f;
      p.dprergb[3 * i] = 0.f; p.dprergb[3 * i + 1] = 0.f; p.dprergb[3 * i + 2] = 0.f;
    }
  if (p.amax_bits != nullptr) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, o));
      amax_rgb = fmaxf(amax_rgb, __shfl_xor_sync(0xffffffffu, amax_rgb, o));
    }
    if (lane == 0 && amax > 0.f && amax < 3e38f) atomicMax(p.amax_bits, __float_as_uint(amax));
    if (lane == 0 && amax_rgb > 0.f && amax_rgb < 3e38f) atomicMax(p.amax_bits + 1, __float_as_uint(amax_rgb));
    // every tile this ray's samples fall in (non-negative floats order like their bits: deterministic)
    if (p.tile_amax != nullptr && ray < p.n_rays && lane < 2) {
      const float v = fminf(lane ? amax_rgb : amax, 3e38f);
      if (v > 0.f)
        for (long long t = (ray * S) >> 7; t <= (ray * S + S - 1) >> 7; ++t) atomicMax(p.tile_amax + 2 * t + lane, __float_as_uint(v));
    }
  }
}

// Per-pass, per-level scales (see the header comment).  Level v: 0 = dd, v = 1..8 = dpre_{9-v}.
//   phase 0 (before head_bwd / the probe): level 0 gets s0 = 2^floor(log2(64 / B0)) with the batch-wide bound
//            B0 = max(|d rgb_pre|_max wmax_rgb, |d sigma|_max wmax_sigma) >= |dd|, |d sigma w_sigma|; levels
//            1..8 get s0 / 16 for the probe pass (room for a growth of 2^14 through the chain before the probe's
//            own conversions saturate).  Stores wmax_rgb / wmax_sigma for the probe's per-tile bounds.
//   phase 1 (after the probe pass): the probe measured, per level, the growth factor g_v = max over the probed
//            tiles of (largest |value| of the level in the tile) / (the tile's own level-0 bound).  The chain is
//            linear in its level-0 input, so g_v does not depend on how large a tile's gradients are, and
//            B0 g_v bounds level v of every probed tile: s_v = s0 2^-ceil(log2 g_v) maps that bound to <= 64.
//            Clamped to [2^-40, 2^40] x s0; a level the probe saw nothing in keeps its predecessor's scale.
//            Resets the statistics for the next step.
constexpr int kLevels = 9;
constexpr float kProbeLevelScale = 0.0625f;
struct ScaleParams {
  int n_pass, phase;
  unsigned* amax;            // [2 passes][2]: |d sigma|, |d rgb_pre| maxima (float bits)
  unsigned* lamax;           // [2 passes][kLevels] probe growth factors (float bits)
  float* lscale;             // [2][kLevels]
  float* linv;               // [2][kLevels]
  float* wnorm;              // [2 passes][2]: wmax_rgb, wmax_sigma
  unsigned* saturated;       // [2 passes]: fp16 gradient elements the chain clipped (reset in phase 0)
  const float* w_rgb[2];     // live fp32 (3,128)
  const float* w_sigma[2];   // live fp32 (256)
};
__global__ void __launch_bounds__(128) bwd_scale_kernel(const ScaleParams p) {
  __shared__ float red[2][128];
  const int t = threadIdx.x;
  for (int ps = 0; ps < p.n_pass; ++ps) {
    if (p.phase == 0) {
      float wr = fabsf(p.w_rgb[ps][t]) + fabsf(p.w_rgb[ps][128 + t]) + fabsf(p.w_rgb[ps][256 + t]);
      float wsg = fmaxf(fabsf(p.w_sigma[ps][t]), fabsf(p.w_sigma[ps][128 + t]));
      red[0][t] = wr; red[1][t] = wsg;
      __syncthreads();
      for (int o = 64; o > 0; o >>= 1) {
        if (t < o) { red[0][t] = fmaxf(red[0][t], red[0][t + o]); red[1][t] = fmaxf(red[1][t], red[1][t + o]); }
        __syncthreads();
      }
      if (t < kLevels) {
        float s = 1.f;
        if (!kBwdBf16) {
          const float bound = fmaxf(__uint_as_float(p.amax[2 * ps + 1]) * red[0][0], __uint_as_float(p.amax[2 * ps]) * red[1][0]);
          if (bound > 0.f) s = exp2f(floorf(log2f(64.f / bound)));
          s = fminf(fmaxf(s, 1e-30f), 1e30f);
          if (t > 0) s *= kProbeLevelScale;
        }
        p.lscale[ps * kLevels + t] = s;
        p.linv[ps * kLevels + t] = 1.f / s;
        p.lamax[ps * kLevels + t] = 0u;
      }
      if (t < 2) p.wnorm[2 * ps + t] = red[t][0];
      if (t == 0) p.saturated[ps] = 0u;
      __syncthreads();
      if (t < 2) p.amax[2 * ps + t] = 0u;
    } else if (t == 0 && !kBwdBf16) {
      const float s0 = p.lscale[ps * kLevels];
      float prev = s0;
      for (int v = 1; v < kLevels; ++v) {
        const float g = __uint_as_float(p.lamax[ps * kLevels + v]);
        float s = prev;
        if (g > 0.f) s = s0 * exp2f(-ceilf(log2f(g)));
        s = fminf(fmaxf(s, s0 * 9.094947e-13f), s0 * 1.0995116e12f);
        s = fminf(fmaxf(s, 1e-30f), 1e30f);
        p.lscale[ps * kLevels + v] = s;
        p.linv[ps * kLevels + v] = 1.f / s;
        p.lamax[ps * kLevels + v] = 0u;
        prev = s;
      }
    }
  }
}

// ------------------------------------------------------------------------ rgb head / dir ReLU
// models/nerf.py:119-120 backwards, per sample:  dd = (dpre_rgb W_rgb) * (d > 0)  -> tiled fp16 (the
// A operand of the chain kernel's first step and of the W' wgrad), plus the small weight gradients
// that contract over samples on the CUDA cores:
//   gW_rgb[c][n] = sum_s dpre_rgb[s][c] d[s][n]     gb_rgb[c] = sum_s dpre_rgb[s][c]
//   raysum[ray][n] = sum_{s in ray} dd[s][n]        (the direction is constant along a ray: the direction
//   part of gW_dir is sum_rays raysum[ray] (x) dir_enc[ray], dir_grad_kernel below)
//   gW_sigma[n] = sum_s dsigma[s] h8[s][n]          gb_sigma = sum_s dsigma[s]     (models/nerf.py:112)
// A streaming kernel (0.5 KB per sample): one warp per ray and pass, lane = 4 adjacent columns, 8-byte
// loads / stores of the tiled arrays, the sample loop unrolled so that 8 rows are in flight per warp.
// Per-block partials of gW_rgb / gb_rgb, summed in fixed order by wgrad_reduce_kernel.
constexpr int kHeadWarps = 4;
constexpr int kHeadPartRgbW = 0;            // [3][128]
constexpr int kHeadPartRgbB = 384;          // [4]
constexpr int kHeadPartSigW = 388;          // [256]
constexpr int kHeadPartSigB = 644;          // [4]
constexpr int kHeadPartFloats = 648;
struct HeadBwdParams {
  int n_rays, n_pass;
  PassBufs pass[2];
  const float* w_rgb[2];    // live fp32 (3,128)
  const float* lscale;      // [2][kLevels]: level 0 of each pass scales dd
  const float* rays;
  long long ray_stride;
  float* raysum[2];         // (n_rays, 128)
  float* direnc;            // (n_rays, 28): Embedding(3,4)(rays_d), as the forward computes it
  float* part[2];           // [gridDim.x][kHeadPartFloats] per pass (blocks of the other pass write zeros)
};

// (A two-role variant - one warp streaming d, a second one h8, 24 warps per SM instead of 16 - measured 128 us
// against 88 us for this one: more warps in flight did not help, the extra address streams hurt.)
__global__ void __launch_bounds__(kHeadWarps * 32) head_bwd_kernel(const HeadBwdParams p) {
  __shared__ float red[kHeadWarps][kHeadPartFloats];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long unit = static_cast<long long>(blockIdx.x) * kHeadWarps + warp;     // (pass, ray)
  const int ps = unit >= p.n_rays ? 1 : 0;
  const long long ray = unit - (ps ? p.n_rays : 0);
  const bool active = ray < p.n_rays && ps < p.n_pass;
  float gw[3][4], gb[3] = {0.f, 0.f, 0.f}, rs[4] = {0.f, 0.f, 0.f, 0.f};
  float gs[8], gsb = 0.f;       // sigma head: this lane's 8 columns of h8 (one 16-byte chunk), sum of dsigma
#pragma unroll
  for (int c = 0; c < 3; ++c)
#pragma unroll
    for (int i = 0; i < 4; ++i) gw[c][i] = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) gs[i] = 0.f;
  if (active) {
    const PassBufs& pb = p.pass[ps];
    const int S = pb.S;
    const float scale = p.lscale[ps * kLevels];
    float w[3][4];
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
      for (int i = 0; i < 4; ++i) w[c][i] = p.w_rgb[ps][c * 128 + 4 * lane + i];
    if (ps == 0 && lane < 15) {     // Embedding(3,4)(rays_d) exactly as render_kernel.cuh setup_group
      const int cc = lane / 5, kk = lane % 5;
      const float dv = p.rays[ray * p.ray_stride + 3 + cc];
      float* de = p.direnc + ray * 28;
      if (kk == 4) {
        de[cc] = dv;
      } else {
        float sn, cs;
        sincosf(__fmul_rn(static_cast<float>(1 << kk), dv), &sn, &cs);
        de[3 + 6 * kk + cc] = sn;
        de[3 + 6 * kk + 3 + cc] = cs;
      }
    }
    // lane's 4 columns: column block lane / 16, 16-byte chunk (lane % 16) / 2, half (lane & 1)
    const uint32_t fb = lane >> 4, ch = (lane & 15) >> 1, hf = (lane & 1) * 8;
    const uint8_t* h8 = pb.act + 7ll * pb.n_pad * 512;
    const long long g0 = ray * S;
#pragma unroll 8
    for (int i = 0; i < S; ++i) {
      const long long g = g0 + i;
      const unsigned long long off = tiled_block_off(static_cast<unsigned long long>(g >> 6), fb, 2) + (g & 63) * 128 +
                                     ((ch ^ static_cast<uint32_t>(g & 7)) << 4) + hf;
      const uint2 dv2 = __ldg(reinterpret_cast<const uint2*>(pb.d + off));
      // h8 row: 32 lanes x 16 bytes, lane = (column block lane / 8, chunk lane % 8)
      const uint4 hv = __ldg(reinterpret_cast<const uint4*>(
          h8 + tiled_block_off(static_cast<unsigned long long>(g >> 6), lane >> 3, 4) + (g & 63) * 128 +
          (((lane & 7u) ^ static_cast<uint32_t>(g & 7)) << 4)));
      const float ds = __ldg(pb.dsigma + g);
      {
        const float2 a0 = __half22float2(*reinterpret_cast<const __half2*>(&hv.x));
        const float2 a1 = __half22float2(*reinterpret_cast<const __half2*>(&hv.y));
        const float2 a2 = __half22float2(*reinterpret_cast<const __half2*>(&hv.z));
        const float2 a3 = __half22float2(*reinterpret_cast<const __half2*>(&hv.w));
        gs[0] = fmaf(ds, a0.x, gs[0]); gs[1] = fmaf(ds, a0.y, gs[1]); gs[2] = fmaf(ds, a1.x, gs[2]); gs[3] = fmaf(ds, a1.y, gs[3]);
        gs[4] = fmaf(ds, a2.x, gs[4]); gs[5] = fmaf(ds, a2.y, gs[5]); gs[6] = fmaf(ds, a3.x, gs[6]); gs[7] = fmaf(ds, a3.y, gs[7]);
        gsb += ds;
      }
      const float q0 = __ldg(pb.dprergb + 3 * g), q1 = __ldg(pb.dprergb + 3 * g + 1), q2 = __ldg(pb.dprergb + 3 * g + 2);
      const float2 d01 = __half22float2(*reinterpret_cast<const __half2*>(&dv2.x));
      const float2 d23 = __half22float2(*reinterpret_cast<const __half2*>(&dv2.y));
      const float dv[4] = {d01.x, d01.y, d23.x, d23.y};
      float val[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        gw[0][k] = fmaf(q0, dv[k], gw[0][k]);
        gw[1][k] = fmaf(q1, dv[k], gw[1][k]);
        gw[2][k] = fmaf(q2, dv[k], gw[2][k]);
        val[k] = (dv[k] > 0.f) ? fmaf(q0, w[0][k], fmaf(q1, w[1][k], q2 * w[2][k])) : 0.f;
        rs[k] += val[k];
      }
      gb[0] += q0; gb[1] += q1; gb[2] += q2;
      *reinterpret_cast<uint2*>(pb.dd + off) = make_uint2(cvt_bwd_x2(val[0] * scale, val[1] * scale),
                                                          cvt_bwd_x2(val[2] * scale, val[3] * scale));
    }
    *reinterpret_cast<float4*>(p.raysum[ps] + ray * 128 + 4 * lane) = make_float4(rs[0], rs[1], rs[2], rs[3]);
  }
  // per-block partial of gW_rgb / gb_rgb: warps in fixed order
#pragma unroll
  for (int c = 0; c < 3; ++c)
#pragma unroll
    for (int k = 0; k < 4; ++k) red[warp][c * 128 + 4 * lane + k] = gw[c][k];
  if (lane < 4) red[warp][kHeadPartRgbB + lane] = (lane < 3) ? gb[lane] : 0.f;
#pragma unroll
  for (int k = 0; k < 8; ++k) red[warp][kHeadPartSigW + 8 * lane + k] = gs[k];
  if (lane < 4) red[warp][kHeadPartSigB + lane] = (lane == 0) ? gsb : 0.f;
  __syncthreads();
  // a block's warps all belong to one pass unless it straddles the boundary: sum per pass
  for (int q = 0; q < p.n_pass; ++q) {
    float* out = p.part[q] + static_cast<long long>(blockIdx.x) * kHeadPartFloats;
    for (int i = threadIdx.x; i < kHeadPartFloats; i += blockDim.x) {
      float acc = 0.f;
      for (int wv = 0; wv < kHeadWarps; ++wv) {
        const long long u = static_cast<long long>(blockIdx.x) * kHeadWarps + wv;
        if ((u >= p.n_rays ? 1 : 0) == q) acc += red[wv][i];
      }
      out[i] = acc;
    }
  }
}

// gW_dir[n][256 + j] = sum_rays raysum[ray][n] dir_enc[ray][j]: block = 128 threads (n), blockIdx.x = ray slice,
// blockIdx.y = pass; per-slice partials [slice][n][27], summed by wgrad_reduce_kernel.
constexpr int kDirSlices = 64;
struct DirGradParams {
  int n_rays;
  const float* raysum[2];
  const float* direnc;
  float* part[2];           // [kDirSlices][128][27]
};
__global__ void __launch_bounds__(128) dir_grad_kernel(const DirGradParams p) {
  __shared__ float de[64][28];
  const int ps = blockIdx.y, n = threadIdx.x;
  const int per = (p.n_rays + kDirSlices - 1) / kDirSlices;
  const int r0 = blockIdx.x * per, r1 = min(r0 + per, p.n_rays);
  float acc[27];
#pragma unroll
  for (int j = 0; j < 27; ++j) acc[j] = 0.f;
  for (int base = r0; base < r1; base += 64) {
    const int cnt = min(64, r1 - base);
    __syncthreads();
    for (int i = n; i < cnt * 28; i += 128) de[i / 28][i % 28] = p.direnc[static_cast<long long>(base) * 28 + i];
    __syncthreads();
#pragma unroll 4
    for (int r = 0; r < cnt; ++r) {
      const float v = p.raysum[ps][static_cast<long long>(base + r) * 128 + n];
#pragma unroll
      for (int j = 0; j < 27; ++j) acc[j] = fmaf(v, de[r][j], acc[j]);
    }
  }
  float* out = p.part[ps] + (static_cast<long long>(blockIdx.x) * 128 + n) * 27;
#pragma unroll
  for (int j = 0; j < 27; ++j) out[j] = acc[j];
}

// ------------------------------------------------------------------------------ dgrad chain
// Per 128-sample tile, on the forward's tile engine (mlp_engine.cuh: same warp roles, same TMEM
// map, same K-block hand-over between layers):
//   step 0     D = dd[128 x 128] . W'           (A from shared memory: the dd tile, 2 K blocks)
//              dh8 = D + dsigma (x) w_sigma ;  dpre8 = dh8 * relu'(h8)
//   step s>=1  D = dpre_l[128 x 256] . W_l      (A from tensor memory, l = 8, 7, .., 2; for l = 5
//              only the hidden columns 63..318 of W_5)        dpre_{l-1} = D * relu'(h_{l-1})
// relu' comes from the sign bits the forward stored (64 per thread and layer, two registers).
// Every dpre_l is also written to HBM (tiled 16-bit) for the wgrad kernel.  30 weight slices per
// tile, 120 MMAs (N = 256, K = 16): the same tensor work as layers 2-8 of the forward.
constexpr int kChainSteps = 8;
constexpr uint32_t kChA0 = 0;                          // 2 x [2 K blocks][128 x 64] 16-bit = 2 x 32 KiB
constexpr uint32_t kChA0Bytes = 32768;
constexpr uint32_t kChRing = 2 * kChA0Bytes;           // kStages x 32 KiB
constexpr uint32_t kChConsts = kChRing + kStages * kSliceBytes256;   // w_sigma of both networks (2 x 256 fp32)
constexpr int kChStageBufs = 3;
constexpr uint32_t kChStage = kChConsts + 2048;                      // kChStageBufs x (4 row groups x 4 KiB) staging blocks
constexpr uint32_t kChScratch = kChStage + kChStageBufs * kStageBufBytes;
constexpr uint32_t kChSmemTotal = kChScratch + 1024;

struct ChainScratch {
  Barriers bars;
  uint64_t a0_full[2];
  uint64_t a0_empty[2];
};
static_assert(sizeof(ChainScratch) <= 1024, "chain scratch");

struct ChainParams {
  PassBufs pass[2];
  const uint8_t* net[2];      // packed images (backward region at kOffBwd, w_sigma in the fp32 region)
  int n_pass;
  long long tiles[2];         // 128-sample tiles per pass (probe mode: the number of probed tiles P)
  long long pass_tiles[2];    // all 128-sample tiles of each pass
  const float* lscale;        // [2][kLevels] per-level scales (bwd_scale_kernel)
  unsigned* lamax;            // probe mode: [2][kLevels] growth factors per level
  unsigned* tile_amax[2];     // [pass_tiles][2] per-tile |d sigma|, |d rgb_pre| maxima (composite_bwd_kernel);
                              // the probe reads them, the real pass zeroes them for the next step
  const float* wnorm;         // [2][2] wmax_rgb, wmax_sigma (bwd_scale_kernel phase 0)
  unsigned* saturated;        // real pass: [2] count of fp16 gradient elements at the fp16 limit (or NaN)
  int* status;
};

// The level-0 bound of one tile: the batch-wide bound of bwd_scale_kernel restricted to the tile.
__device__ __forceinline__ float tile_bound(const ChainParams& p, int ps, long long tile) {
  const unsigned* ta = p.tile_amax[ps] + 2 * tile;
  return fmaxf(__uint_as_float(ta[1]) * p.wnorm[2 * ps], __uint_as_float(ta[0]) * p.wnorm[2 * ps + 1]);
}

// Probe mode: CTA c of a pass owns the tiles c, c + P, c + 2P, ... of that pass and probes the one with the
// largest level-0 bound (the first on ties), so the batch's largest gradients are always probed.  Called by
// whole warps: the lanes scan the candidates in parallel, every lane gets the same answer.
__device__ __forceinline__ long long probe_tile(const ChainParams& p, int ps, long long cls, float* bound) {
  const int lane = threadIdx.x & 31;
  long long best = cls;
  float bb = -1.f;
  for (long long t = cls + lane * p.tiles[ps]; t < p.pass_tiles[ps]; t += 32 * p.tiles[ps]) {
    const float b = tile_bound(p, ps, t);
    if (b > bb) { bb = b; best = t; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ob = __shfl_xor_sync(0xffffffffu, bb, o);
    const long long ot = __shfl_xor_sync(0xffffffffu, best, o);
    if (ob > bb || (ob == bb && ot < best)) { bb = ob; best = ot; }
  }
  *bound = bb;
  return best;
}

__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
  uint32_t d;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
  return d;
}

struct ChainEpi {
  Barriers* bars;
  uint32_t tmem_row;
  uint32_t d_phase;
  int row, part, lane;
  uint8_t* dpre;          // this pass's dpre base
  long long n_pad;
  long long g;            // global sample row of this thread
  long long g0;           // global sample row of this thread's 32-row group
  StageCtx stage;         // shared-memory staging of the dpre stores
};

// One step of the chain for this thread's 64 accumulator columns.
//   kFirst: add the rank-1 sigma-head term;  kStore: hand the result to the next step (TMEM A operand)
//   ratio = scale of the produced level / scale of the consumed level (a power of two)
//   kProbe: no HBM stores; returns the largest |value| (in units of the produced level's scale)
//   sat (real pass): incremented by the number of stored elements at the fp16 limit (satfinite clipped them) or NaN
//   mw: this step's 64 ReLU sign bits (loaded one step earlier); next_mask: where the NEXT step's bits are (or null).
//   The load is issued here, as soon as the accumulator is drained, and first used one step later: its HBM / L2
//   latency hides behind this step's conversion and staging (it used to be issued at the top of the step it was
//   needed in, where the wait for it - the top stall of the r02 capture, 6.8 % of all samples - delayed the
//   d_ready wait of every step).
template <bool kFirst, bool kStore, bool kProbe>
__device__ __forceinline__ float epi_chain_step(ChainEpi& c, int out_idx, uint2& mw, const uint2* __restrict__ next_mask,
                                                float dsig, const float* wsig, float ratio, unsigned& sat) {
  // after << i the sign flag of pair i of K block kb sits in the top bit of byte 3 - kb (even elements in ylo, odd in yhi)
  uint32_t ylo[8], yhi[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) { ylo[i] = mw.x << i; yhi[i] = mw.y << i; }
  float vmax = 0.f;
  mbar_wait(smem_u32(&c.bars->d_ready), c.d_phase, 5);
  c.d_phase ^= 1;
  tc_fence_after();
  uint32_t r[4][16];
#pragma unroll
  for (int kb = 0; kb < 4; ++kb) tmem_ld16(c.tmem_row + kTmemD + kb * 64 + c.part * 16, r[kb]);
  if (next_mask != nullptr) mw = __ldg(next_mask);
  tmem_ld_wait();
  if (!kStore) {      // last step: the next tile may overwrite the accumulator
    tc_fence_before();
    __syncwarp();
    if (c.lane == 0) mbar_arrive(smem_u32(&c.bars->d_free));
  }
  uint8_t* out = c.dpre + static_cast<long long>(out_idx) * c.n_pad * 512 + (c.g0 & 63) * 128;
  const unsigned long long chunk = static_cast<unsigned long long>(c.g0 >> 6);
  uint32_t hs[4][8];
  __half2 hmax = __float2half2_rn(0.f);      // per-half maximum of |h|, NaN-propagating (real pass)
#pragma unroll
  for (int kb = 0; kb < 4; ++kb) {
    const int n0 = kb * 64 + c.part * 16;
    // selector: bytes 0,1 <- sign of ylo byte (3 - kb), bytes 2,3 <- sign of yhi byte (3 - kb)
    const uint32_t ln = 0x8u | (3u - kb), hn = 0x8u | (7u - kb);
    const uint32_t sel = (hn << 12) | (hn << 8) | (ln << 4) | ln;
    uint32_t (&h)[8] = hs[kb];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      float a = __uint_as_float(r[kb][2 * i]), b = __uint_as_float(r[kb][2 * i + 1]);
      if (kFirst) {
        const float2 ws = *reinterpret_cast<const float2*>(wsig + n0 + 2 * i);
        a = fmaf(dsig, ws.x, a);
        b = fmaf(dsig, ws.y, b);
      }
      a *= ratio;
      b *= ratio;
      const uint32_t keep = ~prmt(ylo[i], yhi[i], sel);
      h[i] = cvt_bwd_x2(a, b) & keep;
      if (kProbe) {
        if (keep & 0xFFFFu) vmax = fmaxf(vmax, fabsf(a));
        if (keep >> 16) vmax = fmaxf(vmax, fabsf(b));
      } else if (!kBwdBf16) {
        hmax = __hmax2_nan(hmax, __habs2(*reinterpret_cast<const __half2*>(&h[i])));
      }
    }
    if (kStore) {
      tmem_st8(c.tmem_row + kTmemA + n0 / 2, h);
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (c.lane == 0) mbar_arrive(smem_u32(&c.bars->a_kb[kb]));
    }
  }
  // the HBM copy for the wgrad kernel goes out after the hand-over, behind the next step's MMAs:
  // line-coalesced, staged per 32-row group, one 4 KiB bulk store each (mlp_engine.cuh stage_store)
  if (!kProbe && !kBwdBf16 && __vcmpgeu2(*reinterpret_cast<const uint32_t*>(&hmax) & 0x7FFF7FFFu, 0x7BFF7BFFu) != 0u) {   // rare: count them
#pragma unroll
    for (int kb = 0; kb < 4; ++kb)
#pragma unroll
      for (int i = 0; i < 8; ++i) sat += __popc(__vcmpgeu2(hs[kb][i] & 0x7FFF7FFFu, 0x7BFF7BFFu)) >> 4;
  }
  if (!kProbe) {
#pragma unroll
    for (int kb = 0; kb < 4; ++kb)
      stage_store<kChStageBufs>(c.stage, make_uint4(hs[kb][0], hs[kb][1], hs[kb][2], hs[kb][3]),
                                make_uint4(hs[kb][4], hs[kb][5], hs[kb][6], hs[kb][7]), 2u * c.part,
                                out + tiled_block_off(chunk, kb, 4));
  }
  return vmax;
}

template <bool kProbe>
__global__ void __launch_bounds__(kThreads, 1) chain_bwd_kernel(const ChainParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  ChainScratch* sc = reinterpret_cast<ChainScratch*>(smem + kChScratch);
  Barriers* bars = &sc->bars;
  if (threadIdx.x == 0) {
    for (int b = 0; b < 2; ++b) {
      mbar_init(smem_u32(&sc->a0_full[b]), 1);
      mbar_init(smem_u32(&sc->a0_empty[b]), 1);
    }
  }
  if (!engine_setup(smem, bars)) {
    if (threadIdx.x == 0) report_fault(p.status, 101);
    return;
  }
  float* wsig_s = reinterpret_cast<float*>(smem + kChConsts);
  for (int i = threadIdx.x; i < 512; i += blockDim.x) {
    const int ps = i >> 8;
    wsig_s[i] = (ps < p.n_pass) ? reinterpret_cast<const float*>(p.net[ps] + kHalfRegionBytes)[kF32WSigma + (i & 255)] : 0.f;
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long total = p.tiles[0] + (p.n_pass > 1 ? p.tiles[1] : 0);
  const uint32_t idesc = make_idesc_f16(256) | (kBwdFmt << 7) | (kBwdFmt << 10);
  // probe mode: one tile per CTA (grid = total), chosen by probe_tile
  float probe_bound = 0.f;
  long long probe_t = 0;
  if (kProbe) {
    const int ps = (blockIdx.x >= p.tiles[0]) ? 1 : 0;
    probe_t = probe_tile(p, ps, blockIdx.x - (ps ? p.tiles[0] : 0), &probe_bound);
  }

  if (warp == kProducerWarp) {
    if (lane == 0) {
      RingState rs;
      int it = 0;
      for (long long t = blockIdx.x; t < total; t += gridDim.x, ++it) {
        const int ps = (t >= p.tiles[0]) ? 1 : 0;
        const long long tile = kProbe ? probe_t : t - (ps ? p.tiles[0] : 0);
        const int b = it & 1;
        // the dd tile: rows 0..63 and 64..127 of column block kb are two 8 KiB blocks of the tiled array
        mbar_wait(smem_u32(&sc->a0_empty[b]), ((it >> 1) & 1) ^ 1, 31);
        const uint32_t full = smem_u32(&sc->a0_full[b]);
        mbar_arrive_expect_tx(full, kChA0Bytes);
        const uint32_t dst = smem_u32(smem + kChA0 + b * kChA0Bytes);
        const uint8_t* dd = p.pass[ps].dd;
#pragma unroll
        for (int kb = 0; kb < 2; ++kb)
#pragma unroll
          for (int hh = 0; hh < 2; ++hh)
            bulk_g2s(dst + kb * 16384 + hh * 8192, dd + tiled_block_off(static_cast<unsigned long long>(tile * 2 + hh), kb, 2), 8192, full);
        const uint8_t* w = p.net[ps] + kOffBwd;
        for (int i = 0; i < kNumSlicesBwd; ++i) {
          mbar_wait(smem_u32(&bars->empty[rs.stage]), rs.phase ^ 1, 1);
          const uint32_t fl = smem_u32(&bars->full[rs.stage]);
          const uint32_t d2 = smem_u32(smem + kChRing + rs.stage * kSliceBytes256);
          mbar_arrive_expect_tx(fl, kSliceBytes256);
          const uint8_t* src = w + static_cast<size_t>(i) * kSliceBytes256;
#pragma unroll
          for (int cc = 0; cc < 4; ++cc) bulk_g2s(d2 + cc * 8192, src + cc * 8192, 8192, fl);
          rs.advance();
        }
      }
    }
  } else if (warp == kMmaWarp) {
    if (lane == 0) {
      RingState rs;
      uint32_t ph_dfree = 0, ph_akb = 0;
      const uint32_t tmem = bars->tmem_base;
      const uint32_t d_tmem = tmem + kTmemD, a_tmem = tmem + kTmemA;
      const uint64_t ring_desc = make_desc_sw128(smem_u32(smem + kChRing));
      const uint32_t full0 = smem_u32(&bars->full[0]), empty0 = smem_u32(&bars->empty[0]);
      const uint32_t akb0 = smem_u32(&bars->a_kb[0]);
      const uint32_t d_ready = smem_u32(&bars->d_ready);
      int it = 0;
      for (long long t = blockIdx.x; t < total; t += gridDim.x, ++it) {
        const int b = it & 1;
        const uint64_t a0_desc = make_desc_sw128(smem_u32(smem + kChA0 + b * kChA0Bytes));
#pragma unroll
        for (int s = 0; s < kChainSteps; ++s) {
          if (s == 0) {
            mbar_wait(smem_u32(&bars->d_free), ph_dfree, 3);
            ph_dfree ^= 1;
            mbar_wait(smem_u32(&sc->a0_full[b]), (it >> 1) & 1, 9);
          } else {
            mbar_wait(akb0, ph_akb, 6);      // also: every warp has drained the accumulator
          }
          tc_fence_after();
          const int n_slices = (s == 0) ? 2 : 4;
#pragma unroll
          for (int kb = 0; kb < 4; ++kb) {
            if (kb < n_slices) {
              const uint32_t stage = rs.stage;
              mbar_wait(full0 + 8u * stage, rs.phase, 4);
              if (s != 0 && kb > 0) mbar_wait(akb0 + 8u * kb, ph_akb, 6);
              tc_fence_after();
              const uint64_t bdesc = ring_desc + static_cast<uint64_t>(stage * (kSliceBytes256 >> 4));
              if (s == 0) {
#pragma unroll
                for (int j = 0; j < 4; ++j)
                  umma_f16(d_tmem, a0_desc + static_cast<uint64_t>(kb * (16384 >> 4)) + 2 * j, bdesc + 2 * j, idesc,
                           (kb | j) != 0 ? 1u : 0u);
              } else {
#pragma unroll
                for (int j = 0; j < 4; ++j)
                  umma_f16_ts(d_tmem, a_tmem + kb * 32 + j * 8, bdesc + 2 * j, idesc, (kb | j) != 0 ? 1u : 0u);
              }
              umma_commit(empty0 + 8u * stage);
              rs.advance();
            }
          }
          if (s == 0) umma_commit(smem_u32(&sc->a0_empty[b]));
          umma_commit(d_ready);
          if (s != 0) ph_akb ^= 1;
        }
      }
    }
  } else {
    ChainEpi c;
    c.bars = bars;
    c.lane = lane;
    c.row = (warp & 3) * 32 + lane;
    c.part = warp >> 2;
    c.tmem_row = bars->tmem_base + (static_cast<uint32_t>((warp & 3) * 32) << 16);
    c.d_phase = 0;
    c.stage.base = smem + kChStage + (warp & 3) * 4096;
    c.stage.buf = 0; c.stage.rg = warp & 3; c.stage.lane = lane; c.stage.part = warp >> 2;
    // the accumulator is free at the start
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(smem_u32(&bars->d_free));
    uint2 mw = make_uint2(0u, 0u);      // ReLU sign bits of the step about to run (software-pipelined loads)
    float amx[2][8];      // probe mode only: per pass and level, largest |value| over the tile's level-0 bound
#pragma unroll
    for (int i = 0; i < 8; ++i) { amx[0][i] = 0.f; amx[1][i] = 0.f; }
    unsigned sat[2] = {0u, 0u};
    const float per_bound = (kProbe && probe_bound > 0.f) ? 1.f / probe_bound : 0.f;
    for (long long t = blockIdx.x; t < total; t += gridDim.x) {
      const int ps = (t >= p.tiles[0]) ? 1 : 0;
      const long long tile = kProbe ? probe_t : t - (ps ? p.tiles[0] : 0);
      const PassBufs& pb = p.pass[ps];
      if (!kProbe && warp == 0 && lane < 2) p.tile_amax[ps][2 * tile + lane] = 0u;     // read by this step's probe only
      c.dpre = pb.dpre;
      c.n_pad = pb.n_pad;
      c.g = tile * 128 + c.row;
      c.g0 = tile * 128 + (c.row & ~31);
      const float* ls = p.lscale + ps * kLevels;
      float sc_in = ls[0];
      const float dsig = pb.dsigma[c.g] * sc_in;
      const float* wsig = wsig_s + ps * 256;
      float sc_out = ls[1];
      auto mask_at = [&](const PassBufs& q, long long g, int idx) {
        return q.mask + (static_cast<long long>(idx) * q.n_pad + g) * 4 + c.part;
      };
      if (t == static_cast<long long>(blockIdx.x)) mw = __ldg(mask_at(pb, c.g, 7));      // first tile: not prefetched
      float m = epi_chain_step<true, true, kProbe>(c, 7, mw, mask_at(pb, c.g, 6), dsig, wsig, sc_out / sc_in, sat[ps]);
      if (kProbe) amx[ps][0] = fmaxf(amx[ps][0], m / sc_out * per_bound);
#pragma unroll 1
      for (int s = 1; s < 7; ++s) {
        sc_in = sc_out;
        sc_out = ls[s + 1];
        m = epi_chain_step<false, true, kProbe>(c, 7 - s, mw, mask_at(pb, c.g, 6 - s), 0.f, nullptr, sc_out / sc_in, sat[ps]);
        if (kProbe) amx[ps][s] = fmaxf(amx[ps][s], m / sc_out * per_bound);
      }
      sc_in = sc_out;
      sc_out = ls[8];
      // the last step prefetches the first mask of this CTA's next tile
      const uint2* nxt = nullptr;
      {
        const long long t2 = t + gridDim.x;
        if (t2 < total) {
          const int ps2 = (t2 >= p.tiles[0]) ? 1 : 0;
          const long long tile2 = t2 - (ps2 ? p.tiles[0] : 0);
          nxt = mask_at(p.pass[ps2], tile2 * 128 + c.row, 7);
        }
      }
      m = epi_chain_step<false, false, kProbe>(c, 0, mw, nxt, 0.f, nullptr, sc_out / sc_in, sat[ps]);
      if (kProbe) amx[ps][7] = fmaxf(amx[ps][7], m / sc_out * per_bound);
    }
    if (!kProbe) {
      bulk_wait_all();
#pragma unroll
      for (int ps = 0; ps < 2; ++ps) {
        unsigned v = sat[ps];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0 && v != 0u) atomicAdd(p.saturated + ps, v);
      }
    }
    if (kProbe) {
#pragma unroll
      for (int ps = 0; ps < 2; ++ps)
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          float v = amx[ps][i];
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
          if (lane == 0 && v > 0.f && v < 3e38f) atomicMax(p.lamax + ps * kLevels + 1 + i, __float_as_uint(v));
        }
    }
  }
  engine_teardown(bars);
}

// ------------------------------------------------------------------------------------ wgrad
// gW = A^T B over a range of 64-sample chunks:  A = a 16-bit gradient array (dpre_l or dd), B = an
// fp16 activation array (h_{l-1} or the encoded input), both in the tiled layout, i.e. already the
// MN-major SWIZZLE_128B operand image, so a chunk is staged with two plain bulk copies and the
// tensor core contracts over the samples: per chunk and 128-row half of the output
//   D_half[128 x N] += A[:, half]^T[128 x 64] . B[64 x N]      4 x tcgen05.mma (K = 16 samples)
// The fp32 accumulators (2 halves x N <= 256 columns) stay in tensor memory for the CTA's whole
// range and are written out once, as a partial that wgrad_reduce_kernel sums in a fixed order.
// The kernel is HBM-bound by construction (128 FLOP per byte at N = 256): the point of the layout
// is that it reads every byte exactly once, with no transposition pass and no staging through
// registers.  Four more warps reduce the same shared-memory tiles on the CUDA cores: column sums of
// A (the bias gradients) and, for the W' job, the dsigma-weighted column sums of B = h8 (the sigma
// head's weight gradient).
constexpr int kWgStages = 3;
constexpr uint32_t kWgStageBytes = 65536;              // A chunk (<= 32 KiB) + B chunk (<= 32 KiB)
constexpr uint32_t kWgScratch = kWgStages * kWgStageBytes;
constexpr uint32_t kWgSmemTotal = kWgScratch + 1024;
constexpr int kWgThreads = 6 * 32;                     // producer, issuer, 4 reduction / drain warps

struct WgradJob {          // one piece: a (pass, layer) GEMM over a contiguous range of 64-sample chunks
  const uint8_t* a;        // tiled (n_pad, 64 a_fb) 16-bit gradient array
  const uint8_t* b;        // tiled (n_pad, 64 b_fb) fp16 activation array
  int a_fb;                // column blocks of A: 4 (M = 256, two halves) or 2 (M = 128)
  int b_fb;                // column blocks of B: N = 64 b_fb
  int chunk0, chunk1;      // 64-sample chunks chunk0, chunk0 + chunk_step, ... < chunk1
  int chunk_step;          // > 1: the CTAs of one GEMM interleave their chunks (they read one moving window of HBM)
  float* out;              // partial, TRANSPOSED: element (m, n) at out[n * 64 a_fb + m] (coalesced drain)
  float* bias_out;         // partial column sums of A (64 a_fb) or null
};

struct WgScratch {
  uint64_t full[kWgStages];
  uint64_t empty[kWgStages];
  uint64_t d_ready;        // issuer -> drain warps: the piece's accumulators are complete
  uint64_t acc_free;       // drain warps -> issuer: the accumulators have been read out
  uint32_t tmem_base;
};

// Persistent: CTA b works through pieces [cta_first[b], cta_first[b + 1]) - the host cuts the
// concatenation of all (pass, layer) GEMMs into one equal-byte share per SM (capi.cu plan_wgrad), so
// there is exactly one wave and every SM streams the same number of bytes.
__global__ void __launch_bounds__(kWgThreads, 1) wgrad_kernel(const WgradJob* __restrict__ jobs,
                                                               const int* __restrict__ cta_first, uint32_t copy_bytes,
                                                               uint32_t exp_flags, int* status) {
  extern __shared__ __align__(1024) uint8_t smem[];
  WgScratch* sc = reinterpret_cast<WgScratch*>(smem + kWgScratch);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if ((smem_u32(smem) & 1023u) != 0) {
    if (threadIdx.x == 0) report_fault(status, 101);
    return;
  }
  if (threadIdx.x == 0) {
    for (int i = 0; i < kWgStages; ++i) {
      mbar_init(smem_u32(&sc->full[i]), 1);
      mbar_init(smem_u32(&sc->empty[i]), 5);        // tcgen05.commit + the four reduction warps
    }
    mbar_init(smem_u32(&sc->d_ready), 1);
    mbar_init(smem_u32(&sc->acc_free), 4);
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(smem_u32(&sc->tmem_base), 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const int p0 = cta_first[blockIdx.x], p1 = cta_first[blockIdx.x + 1];

  if (warp == 0) {
    if (lane == 0) {
      uint32_t stage = 0, phase = 0;
      for (int pi = p0; pi < p1; ++pi) {
        const WgradJob job = jobs[pi];
        const uint32_t a_bytes = job.a_fb * kTileBlockBytes, b_bytes = job.b_fb * kTileBlockBytes;
        for (int c = job.chunk0; c < job.chunk1; c += job.chunk_step) {
          mbar_wait(smem_u32(&sc->empty[stage]), phase ^ 1, 51);
          const uint32_t full = smem_u32(&sc->full[stage]);
          const uint32_t dst = smem_u32(smem + stage * kWgStageBytes);
          mbar_arrive_expect_tx(full, a_bytes + b_bytes);
          const uint8_t* sa = job.a + static_cast<unsigned long long>(c) * a_bytes;
          const uint8_t* sb = job.b + static_cast<unsigned long long>(c) * b_bytes;
          for (uint32_t o = 0; o < a_bytes; o += copy_bytes) bulk_g2s(dst + o, sa + o, min(copy_bytes, a_bytes - o), full);
          for (uint32_t o = 0; o < b_bytes; o += copy_bytes) bulk_g2s(dst + 32768 + o, sb + o, min(copy_bytes, b_bytes - o), full);
          if (++stage == kWgStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      uint32_t stage = 0, phase = 0, free_phase = 0;
      bool first = true;
      for (int pi = p0; pi < p1; ++pi) {
        const WgradJob job = jobs[pi];
        const int n_chunks = (job.chunk1 - job.chunk0 + job.chunk_step - 1) / job.chunk_step;
        if (n_chunks <= 0) continue;
        const int N = job.b_fb * 64, halves = job.a_fb >> 1;
        // A: fp16 (bf16 in the experiment build), B: fp16; both MN-major
        const uint32_t idesc = make_idesc_f16_mn(N) | (kBwdFmt << 7);
        if (!first) {       // the previous piece's accumulators have been drained
          mbar_wait(smem_u32(&sc->acc_free), free_phase, 55);
          free_phase ^= 1;
          tc_fence_after();
        }
        first = false;
        for (int c = 0; c < n_chunks; ++c) {
          mbar_wait(smem_u32(&sc->full[stage]), phase, 52);
          tc_fence_after();
          const uint32_t base = smem_u32(smem + stage * kWgStageBytes);
          for (int hh = 0; hh < halves && !(exp_flags & 1u); ++hh) {      // exp bit 0: no MMAs (timing experiment)
#pragma unroll
            for (int j = 0; j < 4; ++j) {        // 16 samples = two 8-row groups = 2048 B per K step
              const uint64_t ad = make_desc_mn_sw128(base + hh * 16384 + j * 2048, 8192, 1024);
              const uint64_t bd = make_desc_mn_sw128(base + 32768 + j * 2048, 8192, 1024);
              umma_f16(sc->tmem_base + hh * 256, ad, bd, idesc, (c | j) != 0 ? 1u : 0u);
            }
          }
          umma_commit(smem_u32(&sc->empty[stage]));
          if (++stage == kWgStages) { stage = 0; phase ^= 1; }
        }
        umma_commit(smem_u32(&sc->d_ready));
      }
    }
  } else {
    // ---- reduction / drain warps.  Column sums of A (the bias gradient): warp wr owns column block wr,
    // lane = (logical 16-byte chunk c = lane % 8, row phase lane / 8): one LDS.128 covers 8 columns of one
    // row, the warp 4 rows (512 B, conflict-free).  8 rows are first summed in fp16 pairs (values are scaled
    // to <= 64, so <= 512; the rounding is far below what the sum over 1e5 samples averages out), then
    // converted and added in fp32 - a sixth of the instructions of a scalar fp32 loop, which throttled the
    // whole kernel to a third of the HBM rate (measured: 760 us with, 265 us without the old reduction).
    const int wr = warp - 2;
    const uint32_t rc = lane & 7, rph = lane >> 3;
    const int m = (warp & 3) * 32 + lane;
    const uint32_t trow = sc->tmem_base + (static_cast<uint32_t>((warp & 3) * 32) << 16);
    uint32_t stage = 0, phase = 0, ready_phase = 0;
    for (int pi = p0; pi < p1; ++pi) {
      const WgradJob job = jobs[pi];
      const int n_chunks = (job.chunk1 - job.chunk0 + job.chunk_step - 1) / job.chunk_step;
      const int N = job.b_fb * 64, halves = job.a_fb >> 1, M = job.a_fb * 64;
      const bool a_act = job.bias_out != nullptr && wr < job.a_fb && !(exp_flags & 2u);   // exp bit 1: no reductions
      float sa[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) sa[i] = 0.f;
      for (int c = job.chunk0; c < job.chunk1; c += job.chunk_step) {
        mbar_wait(smem_u32(&sc->full[stage]), phase, 53);
        if (a_act) {
          const uint8_t* blk = smem + stage * kWgStageBytes + wr * kTileBlockBytes;
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            uint32_t hacc[4] = {0u, 0u, 0u, 0u};
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const uint32_t r = static_cast<uint32_t>((half * 8 + i) * 4) + rph;
              const uint4 v = *reinterpret_cast<const uint4*>(blk + r * 128 + ((rc ^ (r & 7u)) << 4));
              hacc[0] = bwd_add_x2(hacc[0], v.x); hacc[1] = bwd_add_x2(hacc[1], v.y);
              hacc[2] = bwd_add_x2(hacc[2], v.z); hacc[3] = bwd_add_x2(hacc[3], v.w);
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const float2 f = bwd_x2_to_float2(hacc[q]);
              sa[2 * q] += f.x;
              sa[2 * q + 1] += f.y;
            }
          }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(&sc->empty[stage]));
        if (++stage == kWgStages) { stage = 0; phase ^= 1; }
      }
      if (a_act) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {     // the four row phases hold partial sums of the same 8 columns
          sa[i] += __shfl_xor_sync(0xffffffffu, sa[i], 8);
          sa[i] += __shfl_xor_sync(0xffffffffu, sa[i], 16);
        }
        if (rph == 0) {
#pragma unroll
          for (int i = 0; i < 8; ++i) job.bias_out[wr * 64 + rc * 8 + i] = sa[i];
        }
      }
      // ---- drain the accumulators: thread = output row m (TMEM lane) of each half; the partial is stored
      // transposed (element (m, n) at n * M + m) so that a warp writes 32 consecutive floats per column
      if (n_chunks > 0) {
        mbar_wait(smem_u32(&sc->d_ready), ready_phase, 54);
        ready_phase ^= 1;
        tc_fence_after();
      }
      for (int hh = 0; hh < halves; ++hh) {
        float* ocol = job.out + hh * 128 + m;
        for (int c0 = 0; c0 < N; c0 += 32) {
          uint32_t r[32];
          if (n_chunks > 0) {
            tmem_ld32(trow + hh * 256 + c0, r);
            tmem_ld_wait();
          } else {
#pragma unroll
            for (int i = 0; i < 32; ++i) r[i] = 0u;
          }
#pragma unroll
          for (int i = 0; i < 32; ++i) ocol[static_cast<long long>(c0 + i) * M] = __uint_as_float(r[i]);
        }
      }
      if (n_chunks > 0) {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(&sc->acc_free));
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(sc->tmem_base, 512);
  }
}

// ------------------------------------------------------------------- partial sums -> gradients
// out[r][out_col0 + c] = mul * sum_s part[s * split_stride + r * part_ld + c]   (fixed order)
struct ReduceItem {
  const float* part;
  long long split_stride;
  float* out;
  const float* mul;        // device scalar or null (= 1)
  int n_split, rows, cols, part_ld, out_ld, out_col0;
  int transposed;          // partial element (r, c) at part[c * part_ld + r] (wgrad drains) instead of part[r * part_ld + c]
  int by_warp;             // many partials, few outputs: one warp per output, lanes stride over the partials
};
constexpr int kMaxReduceItems = 64;
struct ReduceTable {
  int n;
  ReduceItem it[kMaxReduceItems];
};

__global__ void __launch_bounds__(256) wgrad_reduce_kernel(const __grid_constant__ ReduceTable tab) {
  const ReduceItem& it = tab.it[blockIdx.y];
  const int total = it.rows * it.cols;
  const float mul = (it.mul != nullptr) ? *it.mul : 1.f;
  if (it.by_warp) {        // fixed order: lane l sums partials l, l + 32, ...; then a butterfly over the lanes
    const int lane = threadIdx.x & 31;
    for (int idx = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; idx < total; idx += (gridDim.x * blockDim.x) >> 5) {
      const int r = idx / it.cols, c = idx - r * it.cols;
      const float* src = it.part + static_cast<long long>(r) * it.part_ld + c;
      float acc = 0.f;
      for (int s = lane; s < it.n_split; s += 32) acc += src[s * it.split_stride];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
      if (lane == 0) it.out[static_cast<long long>(r) * it.out_ld + it.out_col0 + c] = acc * mul;
    }
    return;
  }
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
    int r, c;
    const float* src;
    if (it.transposed) {       // r fastest: coalesced reads of the transposed partials
      c = idx / it.rows; r = idx - c * it.rows;
      src = it.part + static_cast<long long>(c) * it.part_ld + r;
    } else {
      r = idx / it.cols; c = idx - r * it.cols;
      src = it.part + static_cast<long long>(r) * it.part_ld + c;
    }
    float acc = 0.f;
    for (int s = 0; s < it.n_split; ++s) acc += src[s * it.split_stride];
    it.out[static_cast<long long>(r) * it.out_ld + it.out_col0 + c] = acc * mul;
  }
}

// Chain rule through the pack-time folding (layout.h): W' = Wd[:, :256] Wf, b' = Wd[:, :256] bf + bd
//   gWd[:, :256] = gW' Wf^T + gb' (x) bf     gWf = Wd[:, :256]^T gW'     gbf = Wd[:, :256]^T gb'     gbd = gb'
struct UnfoldParams {
  const float* gWp[2];     // (128, 256) gradient of the folded matrix
  const float* gbp[2];     // (128)
  const float* Wf[2];      // live xyz_encoding_final.weight (256,256)
  const float* bf[2];      // (256)
  const float* Wd[2];      // live dir_encoding.0.weight (128,283)
  float* gWd[2];           // (128,283): columns 0..255 written here
  float* gbd[2];           // (128)
  float* gWf[2];           // (256,256)
  float* gbf[2];           // (256)
};
__global__ void __launch_bounds__(256) unfold_kernel(const UnfoldParams p) {
  const int ps = blockIdx.y;
  const int lane = threadIdx.x & 31;
  const int gw = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);       // global warp index
  if (gw < 128 * 256) {
    // gWd[m][j] = sum_n gW'[m][n] Wf[j][n] + gb'[m] bf[j]: one warp per output, both rows read coalesced
    const int m = gw >> 8, j = gw & 255;
    const float* a = p.gWp[ps] + m * 256;
    const float* w = p.Wf[ps] + j * 256;
    float acc = 0.f;
#pragma unroll
    for (int n = lane; n < 256; n += 32) acc = fmaf(a[n], w[n], acc);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) {
      p.gWd[ps][m * 283 + j] = acc + p.gbp[ps][m] * p.bf[ps][j];
      if (j == 0) p.gbd[ps][m] = p.gbp[ps][m];
    }
    return;
  }
  const int idx = (gw - 128 * 256) * 32 + lane;
  if (idx < 256 * 256) {                              // gWf[j][n] = sum_m Wd[m][j] gW'[m][n]: coalesced over n
    const int j = idx >> 8, n = idx & 255;
    float acc = 0.f;
#pragma unroll 8
    for (int m = 0; m < 128; ++m) acc = fmaf(p.Wd[ps][m * 283 + j], p.gWp[ps][m * 256 + n], acc);
    p.gWf[ps][j * 256 + n] = acc;
  } else if (idx < 256 * 256 + 256) {                 // gbf[j] = sum_m Wd[m][j] gb'[m]
    const int j = idx - 256 * 256;
    float acc = 0.f;
    for (int m = 0; m < 128; ++m) acc = fmaf(p.Wd[ps][m * 283 + j], p.gbp[ps][m], acc);
    p.gbf[ps][j] = acc;
  }
}

// ------------------------------------------------------------------------------------- Adam
// torch.optim.Adam's update (the reference's default optimiser, utils/__init__.py:16-18:
// Adam(lr, eps, weight_decay), betas (0.9, 0.999), no amsgrad) for all parameter tensors of the two
// networks in ONE launch: torch's fused implementation costs two 80 us multi-tensor kernels for
// these 48 small tensors, a fifth of the remaining step.  Same arithmetic as torch (fp32):
//   g = grad + weight_decay * p;  m = b1 m + (1 - b1) g;  v = b2 v + (1 - b2) g^2
//   p -= lr / (1 - b1^t) * m / (sqrt(v) / sqrt(1 - b2^t) + eps)
constexpr int kAdamMaxTensors = 64;
struct AdamParams {
  int n_tensors;
  float* p[kAdamMaxTensors];
  const float* g[kAdamMaxTensors];
  float* m[kAdamMaxTensors];
  float* v[kAdamMaxTensors];
  int block0[kAdamMaxTensors + 1];     // first block of each tensor (1024 elements per block)
  int numel[kAdamMaxTensors];
  float lr, beta1, beta2, eps, weight_decay, bias1, bias2_sqrt;     // bias1 = 1 - b1^t, bias2_sqrt = sqrt(1 - b2^t)
};
__global__ void __launch_bounds__(256) adam_kernel(const __grid_constant__ AdamParams a) {
  int lo = 0, hi = a.n_tensors;
  while (hi - lo > 1) {        // the tensor this block belongs to
    const int mid = (lo + hi) >> 1;
    if (a.block0[mid] <= static_cast<int>(blockIdx.x)) lo = mid; else hi = mid;
  }
  const int t = lo;
  const int base = (static_cast<int>(blockIdx.x) - a.block0[t]) * 1024;
  const float step = a.lr / a.bias1;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int i = base + q * 256 + threadIdx.x;
    if (i < a.numel[t]) {
      const float pv = a.p[t][i];
      const float g = a.g[t][i] + a.weight_decay * pv;
      const float m = a.beta1 * a.m[t][i] + (1.f - a.beta1) * g;
      const float v = a.beta2 * a.v[t][i] + (1.f - a.beta2) * g * g;
      a.m[t][i] = m;
      a.v[t][i] = v;
      a.p[t][i] = pv - step * m / (sqrtf(v) / a.bias2_sqrt + a.eps);
    }
  }
}

}  // namespace nerfb200
