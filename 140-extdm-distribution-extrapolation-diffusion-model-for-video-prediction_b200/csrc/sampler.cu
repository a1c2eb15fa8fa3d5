// DDIM(eta) update with dynamic thresholding, fp32, arithmetic order identical to the reference
// (model/BaseDM_adaptor/Diffusion.py:231-255); the per-sample 0.9-quantile of |x_start| reproduces
// torch.quantile (linear interpolation, rank computed in fp32) through an exact radix select of the two
// neighbouring order statistics instead of a full sort.
// The DDPM ancestral step (GaussianDiffusion.p_sample_loop) shares that select; its per-step coefficients, step index and
// Philox noise live on the device, so one captured iteration can be replayed for every timestep.
// DDIM with per-video seeds draws its noise from the same Philox generator inside the update.
// The denoising-loss evaluation (GaussianDiffusion.denoising_loss) draws its epsilon from that generator too (stream 2)
// in the forward-diffusion kernel, and reduces the per-(video, frame) loss in a fixed order.
// DPM-Solver++(2M) (GaussianDiffusion.dpm_solver_sample) reuses the DDIM threshold and x_start math, and draws the noise
// of its stochastic variant from that generator too (stream 3).
// Interpolation between two futures (GaussianDiffusion.interpolate) mixes their forward diffusions in one kernel, with
// each endpoint's epsilon from that generator (streams 4 and 5), then runs the DDIM or ancestral loop above.
// Keyframe-conditioned sampling (GaussianDiffusion.sample_with_known) overwrites the known frames after every update
// with the forward diffusion of their latent, its epsilon from that generator too (stream 6).
#include "common.cuh"
#include "../../include/extdm_b200.h"

namespace extdm {

__device__ __forceinline__ float x_start_of(float img, float pred, float c_recip, float c_recipm1) {
  // two roundings then a subtract, never an FMA: matches `a * x_t - b * noise` evaluated op by op
  return __fsub_rn(__fmul_rn(c_recip, img), __fmul_rn(c_recipm1, pred));
}

// The thresholded x0 of every update: clamp(x_start, -s, s) / s, clamped then divided with one rounding, as the
// reference evaluates `x_start.clamp(-s, s) / s`.
__device__ __forceinline__ float clamped_x0(float img, float pred, float c_recip, float c_recipm1, float s) {
  return __fdiv_rn(fminf(fmaxf(x_start_of(img, pred, c_recip, c_recipm1), -s), s), s);
}

// One CTA per sample: s_out[b] = max(1, quantile_q(|x_start[b]|)).  |x| >= 0 so the IEEE bit pattern orders like an
// unsigned integer.  Shared by the DDIM kernel (coefficients as arguments) and the DDPM kernel (coefficients read from
// the schedule table on the device), so both take the same select path.
__device__ __forceinline__ void threshold_sample(const float* __restrict__ img, const float* __restrict__ pred,
                                                 float c_recip, float c_recipm1, float q, float* __restrict__ s_out,
                                                 int n) {
  __shared__ unsigned int hist[256];
  __shared__ unsigned int s_prefix, s_k;
  __shared__ unsigned int s_cnt_le, s_min_gt;
  const int b = blockIdx.x;
  const float* xi = img + static_cast<long long>(b) * n;
  const float* xp = pred + static_cast<long long>(b) * n;

  const float pos = q * static_cast<float>(n - 1);       // fp32 rank, as ATen computes it in the input dtype
  const float lo_f = floorf(pos);
  const unsigned int k_lo = static_cast<unsigned int>(lo_f);
  const unsigned int k_hi = static_cast<unsigned int>(ceilf(pos));
  const float wgt = pos - lo_f;

  if (threadIdx.x == 0) { s_prefix = 0u; s_k = k_lo; }
  __syncthreads();
  // 4 passes of 8 bits, most significant first
  for (int pass = 0; pass < 4; ++pass) {
    const int shift = 24 - 8 * pass;
    for (int i = threadIdx.x; i < 256; i += blockDim.x) hist[i] = 0u;
    __syncthreads();
    const unsigned int prefix = s_prefix;
    const unsigned int mask = pass == 0 ? 0u : (0xFFFFFFFFu << (shift + 8));
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      const unsigned int u = __float_as_uint(fabsf(x_start_of(xi[i], xp[i], c_recip, c_recipm1)));
      if ((u & mask) == prefix) atomicAdd(&hist[(u >> shift) & 0xFFu], 1u);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      unsigned int k = s_k, acc = 0u;
      int bin = 0;
      for (; bin < 256; ++bin) {
        if (acc + hist[bin] > k) break;
        acc += hist[bin];
      }
      s_k = k - acc;
      s_prefix = prefix | (static_cast<unsigned int>(bin) << shift);
    }
    __syncthreads();
  }
  const unsigned int v_lo = s_prefix;                     // exact k_lo-th order statistic (bit pattern)
  if (threadIdx.x == 0) { s_cnt_le = 0u; s_min_gt = 0xFFFFFFFFu; }
  __syncthreads();
  unsigned int cnt = 0u, mn = 0xFFFFFFFFu;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const unsigned int u = __float_as_uint(fabsf(x_start_of(xi[i], xp[i], c_recip, c_recipm1)));
    if (u <= v_lo) ++cnt;
    else mn = min(mn, u);
  }
  atomicAdd(&s_cnt_le, cnt);
  atomicMin(&s_min_gt, mn);
  __syncthreads();
  if (threadIdx.x == 0) {
    const float a = __uint_as_float(v_lo);
    const float bb = (k_hi == k_lo || s_cnt_le >= k_hi + 1u) ? a : __uint_as_float(s_min_gt);
    // at::lerp: weight < 0.5 ? a + w*(b-a) : b - (b-a)*(1-w)
    const float diff = __fsub_rn(bb, a);
    const float r = wgt < 0.5f ? __fadd_rn(a, __fmul_rn(wgt, diff))
                               : __fsub_rn(bb, __fmul_rn(diff, __fsub_rn(1.0f, wgt)));
    s_out[b] = fmaxf(r, 1.0f);                            // s.clamp_(min=1.)
  }
}

__global__ void __launch_bounds__(1024) ddim_threshold_kernel(const float* __restrict__ img,
                                                              const float* __restrict__ pred, float c_recip,
                                                              float c_recipm1, float q, float* __restrict__ s_out,
                                                              int n) {
  threshold_sample(img, pred, c_recip, c_recipm1, q, s_out, n);
}

// Four elements of one DDIM step: x0 = clamp(c_recip*img - c_recipm1*pred, -s, s)/s;
// out = (x0*sqrt_alpha_next + c*pred) + sigma*z, op by op (no FMA), the sigma*z term only when with_noise.
// Shared by the kernel that reads z from a noise tensor and the one that draws it with Philox.
__device__ __forceinline__ void ddim_quad(float4 x, float4 e, float4 z, bool with_noise, float sb, float c_recip,
                                          float c_recipm1, float sqrt_alpha_next, float c, float sigma,
                                          float* __restrict__ img_out, float* __restrict__ xs_out, long long i) {
  float xv[4] = {x.x, x.y, x.z, x.w}, ev[4] = {e.x, e.y, e.z, e.w}, zv[4] = {z.x, z.y, z.z, z.w}, o[4], xs[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float v = clamped_x0(xv[j], ev[j], c_recip, c_recipm1, sb);
    xs[j] = v;
    float r = __fadd_rn(__fmul_rn(v, sqrt_alpha_next), __fmul_rn(c, ev[j]));
    if (with_noise) r = __fadd_rn(r, __fmul_rn(sigma, zv[j]));
    o[j] = r;
  }
  reinterpret_cast<float4*>(img_out)[i] = make_float4(o[0], o[1], o[2], o[3]);
  if (xs_out) reinterpret_cast<float4*>(xs_out)[i] = make_float4(xs[0], xs[1], xs[2], xs[3]);
}

__global__ void __launch_bounds__(256) ddim_update_kernel(const float* __restrict__ img,
                                                          const float* __restrict__ pred,
                                                          const float* __restrict__ noise,
                                                          const float* __restrict__ s, float c_recip, float c_recipm1,
                                                          float sqrt_alpha_next, float c, float sigma,
                                                          float* __restrict__ img_out, float* __restrict__ xs_out,
                                                          int n4_per_sample, long long total4) {
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float sb = __ldg(s + i / n4_per_sample);
    const float4 x = reinterpret_cast<const float4*>(img)[i];
    const float4 e = reinterpret_cast<const float4*>(pred)[i];
    float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    if (noise) z = reinterpret_cast<const float4*>(noise)[i];
    ddim_quad(x, e, z, noise != nullptr, sb, c_recip, c_recipm1, sqrt_alpha_next, c, sigma, img_out, xs_out, i);
  }
}

// ------------------------------------------------------------------------------------------------ DDPM (ancestral)
// One schedule row per step: {sqrt_recip_alphas_cumprod, sqrt_recipm1_alphas_cumprod, posterior_mean_coef1,
// posterior_mean_coef2, nonzero_mask * exp(0.5 * posterior_log_variance_clipped)} at t = times[step].
constexpr int kDdpmRow = 5;
// Philox counter word 2: which draw of a step (the loop noise of step `step`, or the initial x_T)
constexpr unsigned int kStreamStep = 0u, kStreamInit = 1u;

// Philox4x32-10 (Salmon et al., SC'11), counter-based: the output depends on (counter, key) only.
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
  constexpr unsigned int M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    if (r) { k.x += W0; k.y += W1; }
    const unsigned int hi0 = __umulhi(M0, c.x), lo0 = M0 * c.x;
    const unsigned int hi1 = __umulhi(M1, c.z), lo1 = M1 * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
  }
  return c;
}

// Box-Muller: u1 in (0, 1) with 23 bits (never 0, so the log is finite), u2 in [0, 1) with 24 bits.
__device__ __forceinline__ float2 box_muller(unsigned int a, unsigned int b) {
  const float u1 = (static_cast<float>(a >> 9) + 0.5f) * 0x1p-23f;
  const float u2 = static_cast<float>(b >> 8) * 0x1p-24f;
  const float r = sqrtf(-2.0f * logf(u1));
  float sn, cs;
  sincospif(2.0f * u2, &sn, &cs);
  return make_float2(r * cs, r * sn);
}

// Four N(0, 1) draws for elements 4*quad .. 4*quad+3 of the video with this seed.  Keying by the video's own seed and
// the element index within the video makes a video's noise independent of the batch it is sampled in.
__device__ __forceinline__ float4 normal4(long long seed, unsigned int quad, unsigned int step, unsigned int stream) {
  const unsigned long long sd = static_cast<unsigned long long>(seed);
  const uint4 r = philox4x32_10(make_uint4(quad, step, stream, 0u),
                                make_uint2(static_cast<unsigned int>(sd), static_cast<unsigned int>(sd >> 32)));
  const float2 p = box_muller(r.x, r.y), q = box_muller(r.z, r.w);
  return make_float4(p.x, p.y, q.x, q.y);
}

__global__ void __launch_bounds__(1024) ddpm_threshold_kernel(const float* __restrict__ img,
                                                              const float* __restrict__ pred,
                                                              const float* __restrict__ rows,
                                                              const int* __restrict__ step, float q,
                                                              float* __restrict__ s_out, int n) {
  const float* row = rows + static_cast<long long>(*step) * kDdpmRow;
  threshold_sample(img, pred, row[0], row[1], q, s_out, n);
}

// x0 = clamp(c_recip*img - c_recipm1*pred, -s, s) / s;  out = (c1*x0 + c2*img) + sig*z, op by op as
// GaussianDiffusion.p_sample evaluates it in fp32 (no FMA).  z is slice *step of `noise` when given, else Philox.
__global__ void __launch_bounds__(256) ddpm_update_kernel(const float* __restrict__ img,
                                                          const float* __restrict__ pred,
                                                          const float* __restrict__ rows,
                                                          const int* __restrict__ step,
                                                          const long long* __restrict__ seeds,
                                                          const float* __restrict__ noise,
                                                          const float* __restrict__ s,
                                                          float* __restrict__ img_out, float* __restrict__ xs_out,
                                                          int n4_per_sample, long long total4) {
  const int st = __ldg(step);
  const float* row = rows + static_cast<long long>(st) * kDdpmRow;
  const float c_recip = __ldg(row + 0), c_recipm1 = __ldg(row + 1), c1 = __ldg(row + 2), c2 = __ldg(row + 3),
              sig = __ldg(row + 4);
  const float4* nz = noise ? reinterpret_cast<const float4*>(noise) + st * total4 : nullptr;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long b = i / n4_per_sample;
    const float sb = __ldg(s + b);
    const float4 x = reinterpret_cast<const float4*>(img)[i];
    const float4 e = reinterpret_cast<const float4*>(pred)[i];
    const float4 z = nz ? nz[i]
                        : normal4(__ldg(seeds + b), static_cast<unsigned int>(i - b * n4_per_sample),
                                  static_cast<unsigned int>(st), kStreamStep);
    float xv[4] = {x.x, x.y, x.z, x.w}, ev[4] = {e.x, e.y, e.z, e.w}, zv[4] = {z.x, z.y, z.z, z.w}, o[4], xs[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float v = clamped_x0(xv[j], ev[j], c_recip, c_recipm1, sb);
      xs[j] = v;
      const float mean = __fadd_rn(__fmul_rn(c1, v), __fmul_rn(c2, xv[j]));
      o[j] = __fadd_rn(mean, __fmul_rn(sig, zv[j]));       // added at t = 0 too (sig = 0): torch's signed zeros
    }
    reinterpret_cast<float4*>(img_out)[i] = make_float4(o[0], o[1], o[2], o[3]);
    if (xs_out) reinterpret_cast<float4*>(xs_out)[i] = make_float4(xs[0], xs[1], xs[2], xs[3]);
  }
}

__global__ void __launch_bounds__(256) ddpm_fill_normal_kernel(const long long* __restrict__ seeds,
                                                               float* __restrict__ out, int n4_per_sample,
                                                               long long total4) {
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long b = i / n4_per_sample;
    reinterpret_cast<float4*>(out)[i] =
        normal4(__ldg(seeds + b), static_cast<unsigned int>(i - b * n4_per_sample), 0u, kStreamInit);
  }
}

// DDIM step whose z is the Philox draw of (seeds[b], step, stream 0), the generator of ddpm_update_kernel: a video's
// noise depends on its own seed only.  Step i of the DDIM loop uses step = i; x_T is ddpm_fill_normal (stream 1).
__global__ void __launch_bounds__(256) ddim_update_seeded_kernel(const float* __restrict__ img,
                                                                 const float* __restrict__ pred,
                                                                 const long long* __restrict__ seeds,
                                                                 unsigned int step, const float* __restrict__ s,
                                                                 float c_recip, float c_recipm1,
                                                                 float sqrt_alpha_next, float c, float sigma,
                                                                 float* __restrict__ img_out,
                                                                 float* __restrict__ xs_out, int n4_per_sample,
                                                                 long long total4) {
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long b = i / n4_per_sample;
    const float sb = __ldg(s + b);
    const float4 x = reinterpret_cast<const float4*>(img)[i];
    const float4 e = reinterpret_cast<const float4*>(pred)[i];
    const float4 z =
        normal4(__ldg(seeds + b), static_cast<unsigned int>(i - b * n4_per_sample), step, kStreamStep);
    ddim_quad(x, e, z, true, sb, c_recip, c_recipm1, sqrt_alpha_next, c, sigma, img_out, xs_out, i);
  }
}

// ------------------------------------------------------------------------------------------------ DPM-Solver++(2M)
// Philox counter word 2 of the solver's per-iteration noise (dpmpp_2m_sde); word 1 is the iteration i
constexpr unsigned int kStreamSolver = 3u;

// One multistep iteration: D = clamp(c_recip*img - c_recipm1*pred, -s, s) / s as ddim_quad computes it, then
// out = ((A*img + B*D) + C*d_prev) + N*z, each product rounded on its own and summed left to right (no FMA).  The C term
// is left out when d_prev is NULL (the first, first-order step), the N term when there is no noise source (the ODE
// solver).  final: out = D.  d_out receives D; it may alias d_prev, as img_out may alias img: each thread reads its
// four elements before it writes them.
__global__ void __launch_bounds__(256) dpmpp_update_kernel(const float* __restrict__ img,
                                                           const float* __restrict__ pred,
                                                           const float* d_prev,
                                                           const long long* __restrict__ seeds,
                                                           const float* __restrict__ noise, unsigned int step,
                                                           const float* __restrict__ s, float c_recip,
                                                           float c_recipm1, float A, float B, float C, float N,
                                                           int final, float* img_out, float* d_out,
                                                           int n4_per_sample, long long total4) {
  const bool with_noise = !final && (noise != nullptr || seeds != nullptr);
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long b = i / n4_per_sample;
    const float sb = __ldg(s + b);
    const float4 x = reinterpret_cast<const float4*>(img)[i];
    const float4 e = reinterpret_cast<const float4*>(pred)[i];
    float4 dp = make_float4(0.f, 0.f, 0.f, 0.f), z = make_float4(0.f, 0.f, 0.f, 0.f);
    if (d_prev && !final) dp = reinterpret_cast<const float4*>(d_prev)[i];
    if (with_noise)
      z = noise ? reinterpret_cast<const float4*>(noise)[i]
                : normal4(__ldg(seeds + b), static_cast<unsigned int>(i - b * n4_per_sample), step, kStreamSolver);
    float xv[4] = {x.x, x.y, x.z, x.w}, ev[4] = {e.x, e.y, e.z, e.w}, pv[4] = {dp.x, dp.y, dp.z, dp.w},
          zv[4] = {z.x, z.y, z.z, z.w}, o[4], dv[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float v = clamped_x0(xv[j], ev[j], c_recip, c_recipm1, sb);
      dv[j] = v;
      float r = __fadd_rn(__fmul_rn(A, xv[j]), __fmul_rn(B, v));
      if (d_prev) r = __fadd_rn(r, __fmul_rn(C, pv[j]));
      if (with_noise) r = __fadd_rn(r, __fmul_rn(N, zv[j]));
      o[j] = final ? v : r;
    }
    reinterpret_cast<float4*>(img_out)[i] = make_float4(o[0], o[1], o[2], o[3]);
    reinterpret_cast<float4*>(d_out)[i] = make_float4(dv[0], dv[1], dv[2], dv[3]);
  }
}

// ------------------------------------------------------------------------------------------------ denoising loss
// Philox counter word 2 of the loss evaluation's epsilon; word 1 is the video's timestep t[b]
constexpr unsigned int kStreamLoss = 2u;

// x_t = a * x_start + b * eps with a = sqrt_alphas_cumprod[t], b = sqrt_one_minus_alphas_cumprod[t]: two roundings then a
// sum, never an FMA, as torch evaluates `extract(a, t) * x_start + extract(b, t) * noise`.
__device__ __forceinline__ float q_sample_of(float x0, float eps, float a, float b) {
  return __fadd_rn(__fmul_rn(a, x0), __fmul_rn(b, eps));
}

__global__ void __launch_bounds__(256) q_sample_kernel(const float* __restrict__ x_start,
                                                       const long long* __restrict__ t,
                                                       const long long* __restrict__ seeds,
                                                       const float* __restrict__ noise,
                                                       const float* __restrict__ sqrt_acp,
                                                       const float* __restrict__ sqrt_1m_acp,
                                                       float* __restrict__ x_t, float* __restrict__ eps_out,
                                                       int n4_per_sample, long long total4) {
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long b = i / n4_per_sample;
    const long long tb = __ldg(t + b);
    const float a = __ldg(sqrt_acp + tb), c = __ldg(sqrt_1m_acp + tb);
    const float4 e = noise ? reinterpret_cast<const float4*>(noise)[i]
                           : normal4(__ldg(seeds + b), static_cast<unsigned int>(i - b * n4_per_sample),
                                     static_cast<unsigned int>(tb), kStreamLoss);
    const float4 x = reinterpret_cast<const float4*>(x_start)[i];
    reinterpret_cast<float4*>(x_t)[i] =
        make_float4(q_sample_of(x.x, e.x, a, c), q_sample_of(x.y, e.y, a, c), q_sample_of(x.z, e.z, a, c),
                    q_sample_of(x.w, e.w, a, c));
    reinterpret_cast<float4*>(eps_out)[i] = e;
  }
}

// ------------------------------------------------------------------------------------------------ interpolation
// Philox counter word 2 of the two endpoints' epsilon in GaussianDiffusion.interpolate; word 1 is the mix timestep t
constexpr unsigned int kStreamInterp1 = 4u, kStreamInterp2 = 5u;

// x_t = c1 * q(x1, eps1) + c2 * q(x2, eps2) at one timestep t shared by the batch, q as q_sample_of; every product
// rounded on its own and each sum of two (no FMA), as torch evaluates `(1 - lam) * (...) + lam * (...)` in fp32.
// eps1, eps2 are noise[i] and noise[total4 + i] when noise is given, else the Philox draws of streams 4 and 5.
__global__ void __launch_bounds__(256) q_interpolate_kernel(const float* __restrict__ x1, const float* __restrict__ x2,
                                                            int t, const long long* __restrict__ seeds,
                                                            const float* __restrict__ noise,
                                                            const float* __restrict__ sqrt_acp,
                                                            const float* __restrict__ sqrt_1m_acp, float c1, float c2,
                                                            float* __restrict__ x_t, int n4_per_sample,
                                                            long long total4) {
  const float a = __ldg(sqrt_acp + t), c = __ldg(sqrt_1m_acp + t);
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    float4 e1, e2;
    if (noise) {
      e1 = reinterpret_cast<const float4*>(noise)[i];
      e2 = reinterpret_cast<const float4*>(noise)[total4 + i];
    } else {
      const long long b = i / n4_per_sample;
      const long long sd = __ldg(seeds + b);
      const unsigned int quad = static_cast<unsigned int>(i - b * n4_per_sample);
      e1 = normal4(sd, quad, static_cast<unsigned int>(t), kStreamInterp1);
      e2 = normal4(sd, quad, static_cast<unsigned int>(t), kStreamInterp2);
    }
    const float4 u = reinterpret_cast<const float4*>(x1)[i], v = reinterpret_cast<const float4*>(x2)[i];
    const float uv[4] = {u.x, u.y, u.z, u.w}, vv[4] = {v.x, v.y, v.z, v.w};
    const float e1v[4] = {e1.x, e1.y, e1.z, e1.w}, e2v[4] = {e2.x, e2.y, e2.z, e2.w};
    float o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j)
      o[j] = __fadd_rn(__fmul_rn(c1, q_sample_of(uv[j], e1v[j], a, c)),
                       __fmul_rn(c2, q_sample_of(vv[j], e2v[j], a, c)));
    reinterpret_cast<float4*>(x_t)[i] = make_float4(o[0], o[1], o[2], o[3]);
  }
}

// ------------------------------------------------------------------------------------------------ keyframes
// Philox counter word 2 of the replacement noise of keyframe-conditioned sampling; word 1 is the replacement point k
constexpr unsigned int kStreamKnown = 6u;
// One row per replacement point of the ancestral loop: {a_k, b_k, final}
constexpr int kKnownRow = 3;

// Replacement point k of GaussianDiffusion.sample_with_known on (B, 3, tp, hw) tensors: every quad of frame f of video b
// with known[b, f] becomes q_sample_of(x_known, eps_k, a, c), or x_known itself when final; a quad of an unknown frame is
// neither read from x_known nor written.  eps_k is noise[k] of (K, B, n) when noise is given, else the Philox draw of
// (seeds[b], k, stream 6).  hw4 = hw / 4 quads per (channel, frame) plane, so a quad never straddles two frames.
__device__ __forceinline__ void impose_known_quads(float* x, const float* __restrict__ x_known,
                                                   const unsigned char* __restrict__ known,
                                                   const long long* __restrict__ seeds,
                                                   const float* __restrict__ noise, float a, float c, unsigned int k,
                                                   bool final, int tp, int hw4, int n4_per_sample, long long total4) {
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long b = i / n4_per_sample;
    const unsigned int quad = static_cast<unsigned int>(i - b * n4_per_sample);
    if (!__ldg(known + b * tp + (quad / hw4) % tp)) continue;
    const float4 xk = reinterpret_cast<const float4*>(x_known)[i];
    float4 o = xk;
    if (!final) {
      const float4 e = noise ? reinterpret_cast<const float4*>(noise)[static_cast<long long>(k) * total4 + i]
                             : normal4(__ldg(seeds + b), quad, k, kStreamKnown);
      o = make_float4(q_sample_of(xk.x, e.x, a, c), q_sample_of(xk.y, e.y, a, c), q_sample_of(xk.z, e.z, a, c),
                      q_sample_of(xk.w, e.w, a, c));
    }
    reinterpret_cast<float4*>(x)[i] = o;
  }
}

// DDIM: (a, c, k, final) are launch scalars, baked into the captured loop.
__global__ void __launch_bounds__(256) impose_known_kernel(float* x, const float* __restrict__ x_known,
                                                           const unsigned char* __restrict__ known,
                                                           const long long* __restrict__ seeds,
                                                           const float* __restrict__ noise, float a, float c,
                                                           unsigned int k, int final, int tp, int hw4,
                                                           int n4_per_sample, long long total4) {
  impose_known_quads(x, x_known, known, seeds, noise, a, c, k, final != 0, tp, hw4, n4_per_sample, total4);
}

// Ancestral: k = *step, the counter ddpm_update reads, and (a, c, final) its row of the device table, so one captured
// iteration serves every replacement point.
__global__ void __launch_bounds__(256) impose_known_table_kernel(float* x, const float* __restrict__ x_known,
                                                                 const unsigned char* __restrict__ known,
                                                                 const long long* __restrict__ seeds,
                                                                 const float* __restrict__ noise,
                                                                 const float* __restrict__ rows,
                                                                 const int* __restrict__ step, int tp, int hw4,
                                                                 int n4_per_sample, long long total4) {
  const int k = __ldg(step);
  const float* row = rows + static_cast<long long>(k) * kKnownRow;
  impose_known_quads(x, x_known, known, seeds, noise, __ldg(row + 0), __ldg(row + 1), static_cast<unsigned int>(k),
                     __ldg(row + 2) != 0.f, tp, hw4, n4_per_sample, total4);
}

// One block per (video b, frame f) of (B, 3, tp, hw) tensors: out[b, f] = mean over (3, hw) of (eps - pred)^2 (or
// |eps - pred|).  The difference of two floats is exact in double, so the terms are exact and the sum is in fp64; each
// thread sums a fixed strided subset in order, then a fixed shared-memory tree: the result depends on the (b, f) slice
// only, bit for bit, whatever the batch, the call or the launch.
constexpr int kLossThreads = 256;
__global__ void __launch_bounds__(kLossThreads) denoise_loss_kernel(const float* __restrict__ eps,
                                                                    const float* __restrict__ pred,
                                                                    float* __restrict__ out, int tp, int hw, int l1) {
  __shared__ double part[kLossThreads];
  const int b = blockIdx.x / tp, f = blockIdx.x % tp;
  const long long plane = static_cast<long long>(tp) * hw;
  const long long base = static_cast<long long>(b) * 3 * plane + static_cast<long long>(f) * hw;
  double acc = 0.0;
  for (int j = threadIdx.x; j < 3 * hw; j += kLossThreads) {
    const long long k = base + (j / hw) * plane + j % hw;
    const double d = static_cast<double>(__ldg(eps + k)) - static_cast<double>(__ldg(pred + k));
    acc += l1 ? fabs(d) : d * d;
  }
  part[threadIdx.x] = acc;
  __syncthreads();
#pragma unroll
  for (int s = kLossThreads / 2; s > 0; s >>= 1) {
    if (threadIdx.x < s) part[threadIdx.x] += part[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[blockIdx.x] = static_cast<float>(part[0] / static_cast<double>(3 * hw));
}

// out[b, :] = table[*step, :] for every sample: the time-conditioned rows of the step, shared by the whole batch.
__global__ void __launch_bounds__(256) ddpm_broadcast_row_kernel(const float* __restrict__ table,
                                                                 const int* __restrict__ step,
                                                                 float* __restrict__ out, int n_row, long long total) {
  const float* row = table + static_cast<long long>(__ldg(step)) * n_row;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x)
    out[i] = __ldg(row + i % n_row);
}

// One block: step += 1, then time[:] = times[step] for the next iteration's time MLP.
__global__ void __launch_bounds__(256) ddpm_advance_kernel(int* __restrict__ step, const long long* __restrict__ times,
                                                           int n_steps, long long* __restrict__ time, int B) {
  const int next = *step + 1;
  __syncthreads();                                        // every thread has read the old value
  if (threadIdx.x == 0) *step = next;
  if (next < n_steps)
    for (int b = threadIdx.x; b < B; b += blockDim.x) time[b] = times[next];
}

}  // namespace extdm

using namespace extdm;

static int ddpm_grid(long long total4) {
  long long g = (total4 + 255) / 256;
  return static_cast<int>(g > 148 * 8 ? 148 * 8 : g);
}

extern "C" int extdm_ddim_threshold(const float* img, const float* pred, float c_recip, float c_recipm1, float q,
                                    float* s, int B, int n, void* stream) {
  if (n < 2 || B < 1) {
    extdm_set_error("ddim_threshold: need n >= 2", __FILE__, __LINE__);
    return EXTDM_ERR_ARG;
  }
  ddim_threshold_kernel<<<B, 1024, 0, static_cast<cudaStream_t>(stream)>>>(img, pred, c_recip, c_recipm1, q, s, n);
  EXTDM_CHECK_LAUNCH();
  return EXTDM_OK;
}

extern "C" int extdm_ddim_update(const float* img, const float* pred, const float* noise, const float* s,
                                 float c_recip, float c_recipm1, float sqrt_alpha_next, float c, float sigma,
                                 float* img_out, float* x_start_out, int B, int n, void* stream) {
  if (n % 4) {
    extdm_set_error("ddim_update: elements per sample must be a multiple of 4", __FILE__, __LINE__);
    return EXTDM_ERR_ARG;
  }
  const long long total4 = static_cast<long long>(B) * n / 4;
  ddim_update_kernel<<<ddpm_grid(total4), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      img, pred, noise, s, c_recip, c_recipm1, sqrt_alpha_next, c, sigma, img_out, x_start_out, n / 4, total4);
  EXTDM_CHECK_LAUNCH();
  return EXTDM_OK;
}

extern "C" int extdm_ddim_update_seeded(const float* img, const float* pred, const long long* seeds, int step,
                                        const float* s, float c_recip, float c_recipm1, float sqrt_alpha_next,
                                        float c, float sigma, float* img_out, float* x_start_out, int B, int n,
                                        void* stream) {
  if (n % 4 || B < 1 || !seeds || step < 0) {
    extdm_set_error("ddim_update_seeded: need n % 4 == 0, B >= 1, seeds and step >= 0", __FILE__, __LINE__);
    return EXTDM_ERR_ARG;
  }
  const long long total4 = static_cast<long long>(B) * n / 4;
  ddim_update_seeded_kernel<<<ddpm_grid(total4), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      img, pred, seeds, static_cast<unsigned int>(step), s, c_recip, c_recipm1, sqrt_alpha_next, c, sigma, img_out,
      x_start_out, n / 4, total4);
  EXTDM_CHECK_LAUNCH();
  return EXTDM_OK;
}

extern "C" int extdm_dpmpp_update(const float* img, const float* pred, const float* d_prev, const long long* seeds,
                                  const float* noise, int step, const float* s, float c_recip, float c_recipm1,
                                  float A, float B_coef, float C_coef, float N, int final, float* img_out,
                                  float* d_out, int B, int n, void* stream) {
  if (n % 4 || n < 4 || B < 1 || step < 0 || !s || !img_out || !d_out || (seeds && noise)) {
    extdm_set_error("dpmpp_update: need n % 4 == 0, B >= 1, step >= 0, s, both outputs and not both seeds and noise",
                    __FILE__, __LINE__);
    return EXTDM_ERR_ARG;
  }
  const long long total4 = static_cast<long long>(B) * n / 4;
  dpmpp_update_kernel<<<ddpm_grid(total4), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      img, pred, d_prev, seeds, noise, static_cast<unsigned int>(step), s, c_recip, c_recipm1, A, B_coef, C_coef, N,
      final != 0, img_out, d_out, n / 4, total4);
  EXTDM_CHECK_LAUNCH();
  return EXTDM_OK;
}

extern "C" int extdm_ddpm_threshold(const float* img, const float* pred, const float* rows, const int* step, float q,
                                    float* s, int B, int n, void* stream) {
  if (n < 2 || B < 1) {
    extdm_set_error("ddpm_threshold: need n >= 2", __FILE__, __LINE__);
    return EXTDM_ERR_ARG;
  }
  ddpm_threshold_kernel<<<B, 1024, 0, static_cast<cudaStream_t>(stream)>>>(img, pred, rows, step, q, s, n);
  EXTDM_CHECK_LAUNCH();
  return EXTDM_OK;
}

extern "C" int extdm_ddpm_update(const float* img, const float* pred, const float* rows, const int* step,
                                 const long long* seeds, const float* noise, const float* s, float* img_out,
                                 float* x_start_out, int B, int n, void* stream) {
  if (n % 4 || B < 1 || (!noise && !seeds)) {
    extdm_set_error("ddpm_update: need n % 4 == 0, B >= 1 and seeds or noise", __FILE__, __LINE__);
    return EXTDM_ERR_ARG;
  }
  const long long total4 = static_cast<long long>(B) * n / 4;
  ddpm_update_kernel<<<ddpm_grid(total4), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      img, pred, rows, step, seeds, noise, s, img_out, x_start_out, n / 4, total4);
  EXTDM_CHECK_LAUNCH();
  return EXTDM_OK;
}

extern "C" int extdm_ddpm_fill_normal(const long long* seeds, float* out, int B, int n, void* stream) {
  if (n % 4 || B < 1) {
    extdm_set_error("ddpm_fill_normal: elements per sample must be a multiple of 4", __FILE__, __LINE__);
    return EXTDM_ERR_ARG;
  }
  const long long total4 = static_cast<long long>(B) * n / 4;
  ddpm_fill_normal_kernel<<<ddpm_grid(total4), 256, 0, static_cast<cudaStream_t>(stream)>>>(seeds, out, n / 4, total4);
  EXTDM_CHECK_LAUNCH();
  return EXTDM_OK;
}

extern "C" int extdm_ddpm_advance(int* step, const long long* times, int n_steps, long long* time, int B,
                                  void* stream) {
  if (B < 1 || n_steps < 1) {
    extdm_set_error("ddpm_advance: need B >= 1 and n_steps >= 1", __FILE__, __LINE__);
    return EXTDM_ERR_ARG;
  }
  ddpm_advance_kernel<<<1, 256, 0, static_cast<cudaStream_t>(stream)>>>(step, times, n_steps, time, B);
  EXTDM_CHECK_LAUNCH();
  return EXTDM_OK;
}

extern "C" int extdm_q_sample(const float* x_start, const long long* t, const long long* seeds, const float* noise,
                              const float* sqrt_acp, const float* sqrt_1m_acp, float* x_t_out, float* eps_out, int B,
                              int n, void* stream) {
  if (n % 4 || n < 4 || B < 1 || !t || (!noise && !seeds) || !sqrt_acp || !sqrt_1m_acp || !x_t_out || !eps_out) {
    extdm_set_error("q_sample: need n % 4 == 0, B >= 1, t, seeds or noise, both tables and both outputs", __FILE__,
                    __LINE__);
    return EXTDM_ERR_ARG;
  }
  const long long total4 = static_cast<long long>(B) * n / 4;
  q_sample_kernel<<<ddpm_grid(total4), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      x_start, t, seeds, noise, sqrt_acp, sqrt_1m_acp, x_t_out, eps_out, n / 4, total4);
  EXTDM_CHECK_LAUNCH();
  return EXTDM_OK;
}

extern "C" int extdm_q_interpolate(const float* x1, const float* x2, int t, const long long* seeds, const float* noise,
                                   const float* sqrt_acp, const float* sqrt_1m_acp, float c1, float c2, float* x_t_out,
                                   int B, int n, void* stream) {
  if (n % 4 || n < 4 || B < 1 || t < 0 || !x1 || !x2 || (!noise == !seeds) || !sqrt_acp || !sqrt_1m_acp || !x_t_out) {
    extdm_set_error("q_interpolate: need n % 4 == 0, B >= 1, t >= 0, both endpoints, exactly one of seeds and noise, "
                    "both tables and the output", __FILE__, __LINE__);
    return EXTDM_ERR_ARG;
  }
  const long long total4 = static_cast<long long>(B) * n / 4;
  q_interpolate_kernel<<<ddpm_grid(total4), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      x1, x2, t, seeds, noise, sqrt_acp, sqrt_1m_acp, c1, c2, x_t_out, n / 4, total4);
  EXTDM_CHECK_LAUNCH();
  return EXTDM_OK;
}

extern "C" int extdm_impose_known(float* x, const float* x_known, const unsigned char* known, const long long* seeds,
                                  const float* noise, float a, float b, int k, int final, const float* rows,
                                  const int* step, int B, int tp, int hw, void* stream) {
  if (B < 1 || tp < 1 || hw < 4 || hw % 4 || !x || !x_known || !known || (!noise == !seeds) || (!rows != !step) ||
      (!rows && k < 0) || static_cast<long long>(3) * tp * hw > 0x7FFFFFFFLL) {
    extdm_set_error("impose_known: need B, tp >= 1, h*w a positive multiple of 4, x, x_known, known, exactly one of "
                    "seeds and noise, rows and step together (or k >= 0)", __FILE__, __LINE__);
    return EXTDM_ERR_ARG;
  }
  const int n4 = 3 * tp * (hw / 4);
  const long long total4 = static_cast<long long>(B) * n4;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (rows)
    impose_known_table_kernel<<<ddpm_grid(total4), 256, 0, st>>>(x, x_known, known, seeds, noise, rows, step, tp,
                                                                 hw / 4, n4, total4);
  else
    impose_known_kernel<<<ddpm_grid(total4), 256, 0, st>>>(x, x_known, known, seeds, noise, a, b,
                                                           static_cast<unsigned int>(k), final != 0, tp, hw / 4, n4,
                                                           total4);
  EXTDM_CHECK_LAUNCH();
  return EXTDM_OK;
}

extern "C" int extdm_denoise_loss(const float* eps, const float* pred, float* out, int B, int tp, int per_frame, int l1,
                                  void* stream) {
  if (B < 1 || tp < 1 || per_frame < 3 || per_frame % 3 || static_cast<long long>(B) * tp > 0x7FFFFFFFLL) {
    extdm_set_error("denoise_loss: need B, tp >= 1 and per_frame a positive multiple of 3", __FILE__, __LINE__);
    return EXTDM_ERR_ARG;
  }
  denoise_loss_kernel<<<B * tp, kLossThreads, 0, static_cast<cudaStream_t>(stream)>>>(eps, pred, out, tp,
                                                                                     per_frame / 3, l1 != 0);
  EXTDM_CHECK_LAUNCH();
  return EXTDM_OK;
}

extern "C" int extdm_ddpm_broadcast_row(const float* table, const int* step, float* out, int B, int n, void* stream) {
  if (B < 1 || n < 1) {
    extdm_set_error("ddpm_broadcast_row: need B >= 1 and n >= 1", __FILE__, __LINE__);
    return EXTDM_ERR_ARG;
  }
  const long long total = static_cast<long long>(B) * n;
  ddpm_broadcast_row_kernel<<<ddpm_grid((total + 3) / 4), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      table, step, out, n, total);
  EXTDM_CHECK_LAUNCH();
  return EXTDM_OK;
}
