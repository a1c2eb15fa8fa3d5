// LFAE conditioning stage (SURVEY.md section 8f-1): the fp32 element-wise kernels around the tf32 convolutions of
// RegionPredictor (model/LFAE/region_predictor.py:60-150), BGMotionPredictor (bg_motion_predictor.py:47-64) and
// PixelwiseFlowPredictor (pixelwise_flow_predictor.py:48-153).  Activations are fp32 channels-last (F, h, w, C).
#include "common.cuh"
#include "../../include/extdm_b200.h"

namespace extdm {
namespace {

// ------------------------------------------------------------------------------------------------ image -> tensor
// AntiAliasInterpolation2d (model/LFAE/util.py:224-271): zero pad (ka, kb), depth-wise ks x ks Gaussian, keep every
// stride-th pixel; ks == 1 is a plain layout change.  Up to two NCHW sources are channel-concatenated (the background
// predictor's [source | driving] input); frame f reads source image f / div.  Channels >= ca + cb are zero.
__global__ void image_to_cl_kernel(const float* __restrict__ a, int ca, int a_div, const float* __restrict__ b, int cb,
                                   int b_div, const float* __restrict__ kern, int ks, int stride, float* __restrict__ out,
                                   int F_, int H, int W, int h, int w, int cpad) {
  const long long total = static_cast<long long>(F_) * h * w * cpad;
  const int ka = ks / 2;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % cpad);
    long long r = i / cpad;
    const int x = static_cast<int>(r % w); r /= w;
    const int y = static_cast<int>(r % h);
    const int f = static_cast<int>(r / h);
    float v = 0.f;
    if (c < ca + cb) {
      const float* src = c < ca ? a + (static_cast<long long>(f / a_div) * ca + c) * H * W
                                : b + (static_cast<long long>(f / b_div) * cb + (c - ca)) * H * W;
      if (ks == 1) {
        v = __ldg(src + y * W + x);
      } else {
        for (int ky = 0; ky < ks; ++ky) {
          const int yy = y * stride + ky - ka;
          if (yy < 0 || yy >= H) continue;
          for (int kx = 0; kx < ks; ++kx) {
            const int xx = x * stride + kx - ka;
            if (xx < 0 || xx >= W) continue;
            v = fmaf(__ldg(kern + ky * ks + kx), __ldg(src + yy * W + xx), v);
          }
        }
      }
    }
    out[i] = round_tf32(v);              // consumed by tf32 convolutions only
  }
}

// ------------------------------------------------------------------------------------------------ pool / upsample
// AvgPool2d(2) (DownBlock2d, util.py:118-131) on (F, H, W, C) fp32, four channels per thread
__global__ void avgpool2_f32_kernel(const float4* __restrict__ x, float4* __restrict__ y, long long F_, int H, int W,
                                    int c4) {
  const int Ho = H / 2, Wo = W / 2;
  const long long total = F_ * Ho * Wo * c4;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % c4);
    long long r = i / c4;
    const int xo = static_cast<int>(r % Wo); r /= Wo;
    const int yo = static_cast<int>(r % Ho);
    const long long f = r / Ho;
    const float4* p = x + ((f * H + 2 * yo) * W + 2 * xo) * c4 + c;
    const float4 a = __ldg(p), b = __ldg(p + c4), cc = __ldg(p + static_cast<long long>(W) * c4),
                 d = __ldg(p + static_cast<long long>(W) * c4 + c4);
    y[i] = make_float4(round_tf32((a.x + b.x + cc.x + d.x) * 0.25f), round_tf32((a.y + b.y + cc.y + d.y) * 0.25f),
                       round_tf32((a.z + b.z + cc.z + d.z) * 0.25f), round_tf32((a.w + b.w + cc.w + d.w) * 0.25f));
  }
}

// F.interpolate(scale_factor=2) (nearest; UpBlock2d, util.py:97-115) on (F, H, W, C) fp32
__global__ void upsample2_f32_kernel(const float4* __restrict__ x, float4* __restrict__ y, long long F_, int H, int W,
                                     int c4) {
  const int Ho = 2 * H, Wo = 2 * W;
  const long long total = F_ * Ho * Wo * c4;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % c4);
    long long r = i / c4;
    const int xo = static_cast<int>(r % Wo); r /= Wo;
    const int yo = static_cast<int>(r % Ho);
    const long long f = r / Ho;
    y[i] = __ldg(x + ((f * H + (yo >> 1)) * W + (xo >> 1)) * c4 + c);
  }
}

__device__ __forceinline__ float block_reduce(float v, float* red, bool is_max) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float t = __shfl_xor_sync(0xffffffffu, v, o);
    v = is_max ? fmaxf(v, t) : v + t;
  }
  __syncthreads();                       // red[] may still be read from the previous reduction
  if (lane == 0) red[warp] = v;
  __syncthreads();
  float r = red[0];
  for (int i = 1; i < static_cast<int>(blockDim.x >> 5); ++i) r = is_max ? fmaxf(r, red[i]) : r + red[i];
  return r;
}

// ------------------------------------------------------------------------------------------------ region moments
// RegionPredictor.forward, pca_based branch (region_predictor.py:95-140): softmax(logits / T) over the window
// [crop, h - crop) x [crop, w - crop) of the 'same' convolution output (crop = 3 - pad: the head is a 7x7 convolution
// with padding `pad`), shift = sum heat * grid, covar = sum heat * d d^T with d = grid - shift.  One block per
// (frame, region).  logits: (F, h, w, ldc) fp32.
__global__ void region_moments_kernel(const float* __restrict__ logits, int ldc, int K, int h, int w, int crop,
                                      float inv_temp, float* __restrict__ shift, float* __restrict__ covar) {
  __shared__ float red[32];
  const int f = blockIdx.x / K, k = blockIdx.x % K;
  const int hh = h - 2 * crop, ww = w - 2 * crop, n = hh * ww;
  const float* base = logits + static_cast<long long>(f) * h * w * ldc + k;
  float m = -3.0e38f;
  for (int i = threadIdx.x; i < n; i += blockDim.x)
    m = fmaxf(m, base[static_cast<long long>((i / ww + crop) * w + (i % ww) + crop) * ldc] * inv_temp);
  m = block_reduce(m, red, true);
  float se = 0.f, sx = 0.f, sy = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const int y = i / ww, x = i % ww;
    const float e = __expf(base[static_cast<long long>((y + crop) * w + x + crop) * ldc] * inv_temp - m);
    const float gx = 2.0f * (static_cast<float>(x) / static_cast<float>(ww - 1)) - 1.0f;
    const float gy = 2.0f * (static_cast<float>(y) / static_cast<float>(hh - 1)) - 1.0f;
    se += e; sx += e * gx; sy += e * gy;
  }
  se = block_reduce(se, red, false);
  sx = block_reduce(sx, red, false);
  sy = block_reduce(sy, red, false);
  const float inv = 1.0f / se, mx = sx * inv, my = sy * inv;
  float cxx = 0.f, cxy = 0.f, cyy = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const int y = i / ww, x = i % ww;
    const float p = __expf(base[static_cast<long long>((y + crop) * w + x + crop) * ldc] * inv_temp - m) * inv;
    const float dx = 2.0f * (static_cast<float>(x) / static_cast<float>(ww - 1)) - 1.0f - mx;
    const float dy = 2.0f * (static_cast<float>(y) / static_cast<float>(hh - 1)) - 1.0f - my;
    cxx += p * dx * dx; cxy += p * dx * dy; cyy += p * dy * dy;
  }
  cxx = block_reduce(cxx, red, false);
  cxy = block_reduce(cxy, red, false);
  cyy = block_reduce(cyy, red, false);
  if (threadIdx.x == 0) {
    shift[blockIdx.x * 2] = mx;
    shift[blockIdx.x * 2 + 1] = my;
    float* c = covar + static_cast<long long>(blockIdx.x) * 4;
    c[0] = cxx; c[1] = cxy; c[2] = cxy; c[3] = cyy;
  }
}

// ------------------------------------------------------------------------------------------------ PCA affine
// region_predictor.py:130-146: u, s, v = svd(covar); affine = u diag(sqrt(s)).  Singular vectors are defined up to a sign
// and the affine inherits it, so the convention matters: this is the closed form of what the reference computes when it
// runs on a GPU, i.e. cuSOLVER's batched one-sided Jacobi (gesvdjBatched, the kernel behind torch.svd on CUDA) applied
// to a symmetric 2x2 matrix [[a, b], [b, c]].  One rotation by theta = atan2(2b, a - c) / 2 in (-pi/4, pi/4] when a >= c
// gives U = [[cos, -sin], [sin, cos]]; when a < c the rotation angle is atan2(-2b, c - a) / 2 and the two columns swap
// to sort the singular values, U = [[-sin, cos], [cos, sin]].  An off-diagonal below the Jacobi tolerance is not rotated.
// Checked against torch.svd on the device for 2e5 random covariances (tests/test_kernels_gpu.py::test_pca_affine_closed_form,
// tools/svd_probe.py): identical sign pattern on every matrix, |U - U_cusolver| <= 3e-6.
__global__ void pca_affine_kernel(const float* __restrict__ covar, float* __restrict__ affine, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float a = covar[4 * i], b = covar[4 * i + 1], c = covar[4 * i + 3];
  const float h = 0.5f * (a - c);
  const float r = sqrtf(h * h + b * b);
  const float m = 0.5f * (a + c);
  const float l1 = sqrtf(fmaxf(m + r, 0.f)), l2 = sqrtf(fmaxf(m - r, 0.f));     // sqrt of the singular values, descending
  const bool big = a >= c;
  // columns (a, b) and (b, c): the Jacobi sweep skips the pair when its inner product is below tolerance x the norms
  const bool skip = fabsf(b) * (a + c) <= 8e-7f * sqrtf((a * a + b * b) * (b * b + c * c));
  const float th = skip ? 0.f : 0.5f * atan2f(big ? 2.f * b : -2.f * b, big ? a - c : c - a);
  float sn, cs;
  sincosf(th, &sn, &cs);
  const float u00 = big ? cs : -sn, u01 = big ? -sn : cs, u10 = big ? sn : cs, u11 = big ? cs : sn;
  float* o = affine + 4 * i;
  o[0] = u00 * l1; o[1] = u01 * l2; o[2] = u10 * l1; o[3] = u11 * l2;
}

// ------------------------------------------------------------------------------------------------ sparse motions
// PixelwiseFlowPredictor.create_heatmap_representations / create_sparse_motions / create_deformed_source_image
// (pixelwise_flow_predictor.py:48-112) for one frame f per block.  Driving parameters are those of frame f, source
// parameters and the deformed source image those of frame fs, another frame of the same batch: the source frame is
// part of the driving batch, and its region parameters are the values a separate RegionPredictor call on the same
// image computes.
//   inp   (F, h, w, cpad): channel 4k = heat_k (0 for the background k = 0), 4k+1..4k+3 = source warped by motion k
//   motion(F, K+1, h, w, 2)
// src: (F, h, w, src_ld) fp32 channels-last, channels 0..2 = the down-sampled frames.
__device__ __forceinline__ void sparse_motion_frame(int f, int fs, float* sm, const float* __restrict__ src, int src_ld,
                                                    const float* __restrict__ shift, const float* __restrict__ covar,
                                                    const float* __restrict__ affine, const float* __restrict__ bg, int K,
                                                    int h, int w, int revert_axis_swap, int use_covar, float region_var,
                                                    float* __restrict__ inp, int cpad, float* __restrict__ motion) {
  for (int k = threadIdx.x; k < K; k += blockDim.x) {
    float* s = sm + k * 16;
    const float* cd = covar + (static_cast<long long>(f) * K + k) * 4;
    const float* cs = covar + (static_cast<long long>(fs) * K + k) * 4;
    {
      const float det = cd[0] * cd[3] - cd[1] * cd[2];
      s[0] = cd[3] / det; s[1] = -cd[1] / det; s[2] = -cd[2] / det; s[3] = cd[0] / det;
    }
    {
      const float det = cs[0] * cs[3] - cs[1] * cs[2];
      s[4] = cs[3] / det; s[5] = -cs[1] / det; s[6] = -cs[2] / det; s[7] = cs[0] / det;
    }
    const float* ad = affine + (static_cast<long long>(f) * K + k) * 4;
    const float* as = affine + (static_cast<long long>(fs) * K + k) * 4;
    const float det = ad[0] * ad[3] - ad[1] * ad[2];
    const float i0 = ad[3] / det, i1 = -ad[1] / det, i2 = -ad[2] / det, i3 = ad[0] / det;   // inverse of the driving affine
    float m0 = as[0] * i0 + as[1] * i2, m1 = as[0] * i1 + as[1] * i3;
    float m2 = as[2] * i0 + as[3] * i2, m3 = as[2] * i1 + as[3] * i3;
    if (revert_axis_swap) {
      const float sg = m0 > 0.f ? 1.f : (m0 < 0.f ? -1.f : 0.f);
      m0 *= sg; m1 *= sg; m2 *= sg; m3 *= sg;
    }
    s[8] = m0; s[9] = m1; s[10] = m2; s[11] = m3;
    s[12] = shift[(static_cast<long long>(f) * K + k) * 2];
    s[13] = shift[(static_cast<long long>(f) * K + k) * 2 + 1];
    s[14] = shift[(static_cast<long long>(fs) * K + k) * 2];
    s[15] = shift[(static_cast<long long>(fs) * K + k) * 2 + 1];
  }
  __syncthreads();
  const float* img = src + static_cast<long long>(fs) * h * w * src_ld;
  const float* B9 = bg ? bg + static_cast<long long>(f) * 9 : nullptr;
  for (int pix = threadIdx.x; pix < h * w; pix += blockDim.x) {
    const int y = pix / w, x = pix % w;
    const float gx = 2.0f * (static_cast<float>(x) / static_cast<float>(w - 1)) - 1.0f;
    const float gy = 2.0f * (static_cast<float>(y) / static_cast<float>(h - 1)) - 1.0f;
    float* o = inp + (static_cast<long long>(f) * h * w + pix) * cpad;
    for (int k = 0; k <= K; ++k) {
      float mx, my, heat = 0.f;
      if (k == 0) {
        mx = gx; my = gy;
        if (B9) {
          const float hx = B9[0] * gx + B9[1] * gy + B9[2], hy = B9[3] * gx + B9[4] * gy + B9[5];
          const float hz = B9[6] * gx + B9[7] * gy + B9[8];
          mx = hx / (hz + 1e-10f); my = hy / (hz + 1e-10f);
        }
      } else {
        const float* s = sm + (k - 1) * 16;
        const float dx = gx - s[12], dy = gy - s[13];          // grid - driving shift
        const float ex = gx - s[14], ey = gy - s[15];          // grid - source shift
        float qd, qs;
        if (use_covar) {
          qd = (dx * s[0] + dy * s[2]) * dx + (dx * s[1] + dy * s[3]) * dy;
          qs = (ex * s[4] + ey * s[6]) * ex + (ex * s[5] + ey * s[7]) * ey;
        } else {
          qd = (dx * dx + dy * dy) / region_var;
          qs = (ex * ex + ey * ey) / region_var;
        }
        heat = __expf(-0.5f * qd) - __expf(-0.5f * qs);
        mx = s[8] * dx + s[9] * dy + s[14];
        my = s[10] * dx + s[11] * dy + s[15];
      }
      float* mo = motion + ((static_cast<long long>(f) * (K + 1) + k) * h * w + pix) * 2;
      mo[0] = mx; mo[1] = my;
      // grid_sample(bilinear, zeros padding, align_corners=True)
      const float ix = (mx + 1.0f) * 0.5f * static_cast<float>(w - 1), iy = (my + 1.0f) * 0.5f * static_cast<float>(h - 1);
      const float fx = floorf(ix), fy = floorf(iy);
      const int x0 = static_cast<int>(fx), y0 = static_cast<int>(fy);
      const float wx = ix - fx, wy = iy - fy;
      float acc[3] = {0.f, 0.f, 0.f};
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const int xx = x0 + (t & 1), yy = y0 + (t >> 1);
        if (xx < 0 || xx >= w || yy < 0 || yy >= h) continue;
        const float wt = ((t & 1) ? wx : 1.0f - wx) * ((t >> 1) ? wy : 1.0f - wy);
        const float* p = img + static_cast<long long>(yy * w + xx) * src_ld;
        acc[0] = fmaf(wt, __ldg(p), acc[0]);
        acc[1] = fmaf(wt, __ldg(p + 1), acc[1]);
        acc[2] = fmaf(wt, __ldg(p + 2), acc[2]);
      }
      o[4 * k] = round_tf32(heat); o[4 * k + 1] = round_tf32(acc[0]);
      o[4 * k + 2] = round_tf32(acc[1]); o[4 * k + 3] = round_tf32(acc[2]);
    }
    for (int c = 4 * (K + 1); c < cpad; ++c) o[c] = 0.f;
  }
}

// The conditioning stage: the source of frame f is its video's last conditioning frame, fs = (f / tc) * tc + tc - 1.
__global__ void sparse_motion_kernel(const float* __restrict__ src, int src_ld, const float* __restrict__ shift,
                                     const float* __restrict__ covar, const float* __restrict__ affine,
                                     const float* __restrict__ bg, int K, int tc, int h, int w, int revert_axis_swap,
                                     int use_covar, float region_var, float* __restrict__ inp, int cpad,
                                     float* __restrict__ motion) {
  extern __shared__ float sm[];          // per region: [0..3] inv cov drv, [4..7] inv cov src, [8..11] aff, [12..15] shifts
  const int f = blockIdx.x, fs = (f / tc) * tc + tc - 1;
  sparse_motion_frame(f, fs, sm, src, src_ld, shift, covar, affine, bg, K, h, w, revert_axis_swap, use_covar, region_var,
                      inp, cpad, motion);
}

// Any source slot: frames come in groups of `group` (one video each), the source of frame f is slot src_slot of its
// group, fs = (f / group) * group + src_slot.  Reconstruction (FlowAE) uses group = T frames per video.
__global__ void sparse_motion_src_kernel(const float* __restrict__ src, int src_ld, const float* __restrict__ shift,
                                         const float* __restrict__ covar, const float* __restrict__ affine,
                                         const float* __restrict__ bg, int K, int group, int src_slot, int h, int w,
                                         int revert_axis_swap, int use_covar, float region_var, float* __restrict__ inp,
                                         int cpad, float* __restrict__ motion) {
  extern __shared__ float sm[];
  const int f = blockIdx.x, fs = (f / group) * group + src_slot;
  sparse_motion_frame(f, fs, sm, src, src_ld, shift, covar, affine, bg, K, h, w, revert_axis_swap, use_covar, region_var,
                      inp, cpad, motion);
}

// ------------------------------------------------------------------------------------------------ flow composition
// pixelwise_flow_predictor.py:140-152: mask = softmax over the K+1 logits, flow = sum_k mask_k * motion_k,
// occlusion = sigmoid(logit K+1).  head: (F, h, w, ldc) fp32 with channels [0, K] = mask logits, K+1 = occlusion logit.
// Outputs in the layout FlowDiffusion keeps them: grid (B, 2, tc, h, w), conf (B, 1, tc, h, w) with f = b * tc + t.
__global__ void flow_compose_kernel(const float* __restrict__ head, int ldc, const float* __restrict__ motion, int K,
                                    int tc, int h, int w, long long total, float* __restrict__ grid,
                                    float* __restrict__ conf) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int pix = static_cast<int>(i % (h * w));
    const int f = static_cast<int>(i / (h * w));
    const float* lg = head + i * ldc;
    float m = lg[0];
    for (int k = 1; k <= K; ++k) m = fmaxf(m, lg[k]);
    float se = 0.f, fx = 0.f, fy = 0.f;
    for (int k = 0; k <= K; ++k) {
      const float e = __expf(lg[k] - m);
      const float* mo = motion + ((static_cast<long long>(f) * (K + 1) + k) * h * w + pix) * 2;
      se += e; fx += e * mo[0]; fy += e * mo[1];
    }
    const int b = f / tc, t = f % tc;
    const long long plane = static_cast<long long>(h) * w;
    grid[((static_cast<long long>(b) * 2 + 0) * tc + t) * plane + pix] = fx / se;
    grid[((static_cast<long long>(b) * 2 + 1) * tc + t) * plane + pix] = fy / se;
    if (conf) conf[(static_cast<long long>(b) * tc + t) * plane + pix] = 1.0f / (1.0f + __expf(-lg[K + 1]));
  }
}

// ------------------------------------------------------------------------------------------------ background head
// BGMotionPredictor.forward after the encoder (bg_motion_predictor.py:52-64): spatial mean -> Linear -> 3x3 matrix.
// feat: (F, hw, C) fp32; fcw: (n_out, C); one block per frame.  bg_type: 1 shift (2), 2 affine (6), 3 perspective (8).
__global__ void bg_head_kernel(const float* __restrict__ feat, int hw, int Cc, const float* __restrict__ fcw,
                               const float* __restrict__ fcb, int n_out, int bg_type, float* __restrict__ out) {
  __shared__ float red[32];
  __shared__ float res[8];
  const int f = blockIdx.x;
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (int c = threadIdx.x; c < Cc; c += blockDim.x) {
    float m = 0.f;
    for (int p = 0; p < hw; ++p) m += feat[(static_cast<long long>(f) * hw + p) * Cc + c];
    m /= static_cast<float>(hw);
    for (int j = 0; j < n_out; ++j) acc[j] = fmaf(m, __ldg(fcw + static_cast<long long>(j) * Cc + c), acc[j]);
  }
  for (int j = 0; j < n_out; ++j) {
    const float v = block_reduce(acc[j], red, false);
    if (threadIdx.x == 0) res[j] = v + fcb[j];
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float* o = out + static_cast<long long>(f) * 9;
    o[0] = 1.f; o[1] = 0.f; o[2] = 0.f; o[3] = 0.f; o[4] = 1.f; o[5] = 0.f; o[6] = 0.f; o[7] = 0.f; o[8] = 1.f;
    if (bg_type == 1) { o[2] = res[0]; o[5] = res[1]; }
    if (bg_type >= 2) { for (int j = 0; j < 6; ++j) o[j] = res[j]; }
    if (bg_type == 3) { o[6] = res[6]; o[7] = res[7]; }
  }
}

inline int grid_for(long long total, int block) {
  long long g = (total + block - 1) / block;
  return static_cast<int>(g < 148LL * 16 ? (g < 1 ? 1 : g) : 148LL * 16);
}

}  // namespace
}  // namespace extdm

using namespace extdm;

extern "C" int extdm_image_to_cl(const float* a, int ca, int a_div, const float* b, int cb, int b_div, const float* kern,
                                 int ks, int stride, float* out, int F_, int H, int W, int cpad, void* stream) {
  if (!a || ca < 1 || a_div < 1 || (b && (cb < 1 || b_div < 1)) || ks < 1 || stride < 1 || H % stride || W % stride ||
      ca + (b ? cb : 0) > cpad || (ks > 1 && !kern)) {
    extdm_set_error("image_to_cl: bad arguments", __FILE__, __LINE__);
    return EXTDM_ERR_ARG;
  }
  const int h = H / stride, w = W / stride;
  const long long total = static_cast<long long>(F_) * h * w * cpad;
  image_to_cl_kernel<<<grid_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      a, ca, a_div, b, b ? cb : 0, b ? b_div : 1, kern, ks, stride, out, F_, H, W, h, w, cpad);
  EXTDM_CHECK_LAUNCH();
  return EXTDM_OK;
}

extern "C" int extdm_avgpool2_f32_cl(const float* x, float* y, long long F_, int H, int W, int Cc, void* stream) {
  if (H % 2 || W % 2 || Cc % 4) {
    extdm_set_error("avgpool2_f32_cl: H, W even and C % 4 == 0 required", __FILE__, __LINE__);
    return EXTDM_ERR_ARG;
  }
  const long long total = F_ * (H / 2) * (W / 2) * (Cc / 4);
  avgpool2_f32_kernel<<<grid_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const float4*>(x), reinterpret_cast<float4*>(y), F_, H, W, Cc / 4);
  EXTDM_CHECK_LAUNCH();
  return EXTDM_OK;
}

extern "C" int extdm_upsample2_f32_cl(const float* x, float* y, long long F_, int H, int W, int Cc, void* stream) {
  if (Cc % 4) {
    extdm_set_error("upsample2_f32_cl: C % 4 == 0 required", __FILE__, __LINE__);
    return EXTDM_ERR_ARG;
  }
  const long long total = F_ * (2 * H) * (2 * W) * (Cc / 4);
  upsample2_f32_kernel<<<grid_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const float4*>(x), reinterpret_cast<float4*>(y), F_, H, W, Cc / 4);
  EXTDM_CHECK_LAUNCH();
  return EXTDM_OK;
}

extern "C" int extdm_region_moments(const float* logits, int ldc, int F_, int K, int h, int w, int crop,
                                    float temperature, float* shift, float* covar, void* stream) {
  if (K < 1 || K > ldc || h - 2 * crop < 2 || w - 2 * crop < 2 || temperature <= 0.f) {
    extdm_set_error("region_moments: bad arguments", __FILE__, __LINE__);
    return EXTDM_ERR_ARG;
  }
  region_moments_kernel<<<F_ * K, 256, 0, static_cast<cudaStream_t>(stream)>>>(logits, ldc, K, h, w, crop,
                                                                               1.0f / temperature, shift, covar);
  EXTDM_CHECK_LAUNCH();
  return EXTDM_OK;
}

extern "C" int extdm_pca_affine(const float* covar, float* affine, int n, void* stream) {
  if (!covar || !affine || n < 1) {
    extdm_set_error("pca_affine: null pointer / empty batch", __FILE__, __LINE__);
    return EXTDM_ERR_ARG;
  }
  pca_affine_kernel<<<(n + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(covar, affine, n);
  EXTDM_CHECK_LAUNCH();
  return EXTDM_OK;
}

extern "C" int extdm_sparse_motion(const float* src, int src_ld, const float* shift, const float* covar,
                                   const float* affine, const float* bg, int F_, int K, int tc, int h, int w,
                                   int revert_axis_swap, int use_covar, float region_var, float* inp, int cpad,
                                   float* motion, void* stream) {
  if (K < 1 || tc < 1 || F_ % tc || 4 * (K + 1) > cpad || src_ld < 3) {
    extdm_set_error("sparse_motion: bad arguments", __FILE__, __LINE__);
    return EXTDM_ERR_ARG;
  }
  sparse_motion_kernel<<<F_, 256, K * 16 * sizeof(float), static_cast<cudaStream_t>(stream)>>>(
      src, src_ld, shift, covar, affine, bg, K, tc, h, w, revert_axis_swap, use_covar, region_var, inp, cpad, motion);
  EXTDM_CHECK_LAUNCH();
  return EXTDM_OK;
}

extern "C" int extdm_sparse_motion_src(const float* src, int src_ld, const float* shift, const float* covar,
                                       const float* affine, const float* bg, int F_, int K, int group, int src_slot, int h,
                                       int w, int revert_axis_swap, int use_covar, float region_var, float* inp, int cpad,
                                       float* motion, void* stream) {
  if (K < 1 || group < 1 || F_ % group || src_slot < 0 || src_slot >= group || 4 * (K + 1) > cpad || src_ld < 3) {
    extdm_set_error("sparse_motion_src: bad arguments", __FILE__, __LINE__);
    return EXTDM_ERR_ARG;
  }
  sparse_motion_src_kernel<<<F_, 256, K * 16 * sizeof(float), static_cast<cudaStream_t>(stream)>>>(
      src, src_ld, shift, covar, affine, bg, K, group, src_slot, h, w, revert_axis_swap, use_covar, region_var, inp, cpad,
      motion);
  EXTDM_CHECK_LAUNCH();
  return EXTDM_OK;
}

extern "C" int extdm_flow_compose(const float* head, int ldc, const float* motion, int F_, int K, int tc, int h, int w,
                                  float* grid, float* conf, void* stream) {
  if (K + 1 + (conf ? 1 : 0) > ldc || tc < 1 || F_ % tc) {
    extdm_set_error("flow_compose: bad arguments", __FILE__, __LINE__);
    return EXTDM_ERR_ARG;
  }
  const long long total = static_cast<long long>(F_) * h * w;
  flow_compose_kernel<<<grid_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(head, ldc, motion, K, tc, h, w,
                                                                                          total, grid, conf);
  EXTDM_CHECK_LAUNCH();
  return EXTDM_OK;
}

extern "C" int extdm_bg_head(const float* feat, int F_, int hw, int Cc, const float* fcw, const float* fcb, int n_out,
                             int bg_type, float* out, void* stream) {
  if (n_out > 8 || bg_type < 1 || bg_type > 3 || n_out != (bg_type == 1 ? 2 : bg_type == 2 ? 6 : 8)) {
    extdm_set_error("bg_head: bad arguments", __FILE__, __LINE__);
    return EXTDM_ERR_ARG;
  }
  bg_head_kernel<<<F_, 256, 0, static_cast<cudaStream_t>(stream)>>>(feat, hw, Cc, fcw, fcb, n_out, bg_type, out);
  EXTDM_CHECK_LAUNCH();
  return EXTDM_OK;
}
