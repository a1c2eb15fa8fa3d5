/* extdm_b200.h -- C ABI of the B200-native ExtDM sampling hot path.
 *
 * The reference (/root/reference) is pure Python/PyTorch: it has no FFI, plugin or operator boundary
 * (SURVEY.md section 8b).  Each entry point below therefore names the reference *call site* whose library
 * kernels it replaces (file:line, relative to the reference root).  All pointers are device pointers
 * unless stated otherwise, all sizes are element counts, `stream` is a cudaStream_t passed as void*.
 * Every function returns 0 on success; on failure extdm_last_error() holds a message.
 * No function allocates device memory: the host (Python/torch) owns every buffer.
 *
 * Activation layout used by every UNet kernel: channels-last bf16, (B, T, H, W, C).
 * Sampler / warp kernels keep the reference's fp32 NCTHW / NCHW tensors.
 */
#ifndef EXTDM_B200_H
#define EXTDM_B200_H

#ifdef __cplusplus
extern "C" {
#endif

const char* extdm_last_error(void);
int extdm_abi_version(void);

/* ------------------------------------------------------------------------------------------------
 * Implicit-GEMM convolution / linear layer on tcgen05 tensor cores (bf16 x bf16 -> fp32 in TMEM).
 * Replaces nn.Conv3d (1,k,k) / nn.Conv2d / nn.Linear / ConvTranspose3d / Conv2d-on-(T C) call sites:
 *   model/BaseDM_adaptor/DenoiseNet_STWAtt_w_wo_ref_adaptor_cross_multi.py:166 (Block.proj), :192 (res_conv),
 *   :125-136 (Up/Downsample), :267-268 (to_qkv/to_out), :454-456 (qkv/proj), :662-666,704-705 (adaptor),
 *   :803 (init_conv); ..._traj_ada.py:916 (init_noise_conv); model/LFAE/util.py:76-79,102,121,141 (LFAE convs).
 *
 * The A operand is a 5-D channels-last tensor (C, D1, D2, D3, D4), optionally the channel-concatenation
 * of two tensors (skip connections are never materialised).  One CTA computes a 128-row tile
 * box[0]*box[1]*box[2]*box[3] == 128 positions of (D1..D4) x BLOCK_N output columns; for every tap the
 * tile is fetched by TMA at (coord + tap offset), out-of-range positions read as zero (= zero padding).
 * W is [w_rows][ntaps * (a0_channels + a1_channels)] bf16, K-major, K index = tap*(C0+C1) + c.
 * Epilogue: v = acc + bias[n]; v += res; v = v*col_scale[d4][n] + col_shift[d4][n]; act; store.
 * Output element address: out_base + sum_k coord_k*out_stride[k] + (n / col_group)*col_group_stride
 * + n % col_group   (same for `res` with res_base / res_stride).
 */
typedef struct ExtdmGemm {
  const void* a0;
  const void* a1;
  int a0_channels;
  int a1_channels;
  long long a0_dim[4];
  long long a0_stride[4]; /* elements */
  long long a1_dim[4];
  long long a1_stride[4];
  int box[4];
  int start[4];
  int count[4];
  int ntaps;
  signed char tap[64][4];
  const void* w;
  int n;
  int w_rows;
  void* out;
  int out_fp32;
  long long out_base;
  long long out_stride[4];
  int col_group;
  long long col_group_stride;
  const float* bias;
  const void* res;
  int res_fp32;
  long long res_base;
  long long res_stride[4];
  const float* col_scale;
  const float* col_shift;
  int act; /* 0 none, 1 relu, 2 silu, 3 sigmoid */
  int block_n; /* 0 = choose automatically (16/64/128/256) */
  /* Optional GroupNorm(8) statistics of the stored (bf16) output, fused into the epilogue.  Every epilogue warp writes
   * its own slots of a 16-float record [8 group sums | 8 group sums of squares]; record index =
   * (tile*4 + q)*R + r with tile = 128-row tile (ordered D1 fastest .. D4 slowest, so a sample's tiles are
   * contiguous), q = 32-row quarter of the tile, R = max(1, n/128) records because a group wider than a 16-column chunk
   * (n = 256: 2 chunks, n = 512: 4) is summed per chunk, r = (first column of the chunk / 16) mod R.  The output may be
   * cut into several n-tiles (block_n | n): each writes the slots of its own groups.  A group's statistic is the sum
   * over the sample's records.  Requires n in {64,128,256,512}, a bias(+act)-only bf16 epilogue, box[3] == 1.
   * Consumed by extdm_groupnorm_apply (n_part = records per sample). */
  float* gn_partials;
  /* 1: the A tensors and W hold fp32 and the product runs as tcgen05 kind::tf32 (fp32 accumulate) -- the precision the
   * reference's GPU convolutions run at (cudnn.allow_tf32 defaults to True, never changed by scripts/DM/valid.py).  All
   * channel counts, element strides and W's row pitch are then given in 2-byte units, i.e. twice the fp32 element
   * counts (an fp32 tensor of C channels is described exactly like a bf16 tensor of 2C channels; C % 32 == 0).
   * 2: as 1, and the stored fp32 outputs are rounded to the nearest tf32 value (for outputs that feed another tf32
   * product: the tensor core ignores the low 13 mantissa bits, rounding where a value is produced halves the error).
   * Used by the LFAE conditioning stage (region / background / flow predictors, SURVEY.md section 8f-1). */
  int tf32;
  /* Phases: n_phase (0 or 1 = none, up to 4) independent products over the SAME A tiles in one launch -- the four
   * sub-pixel phases of ConvTranspose3d (1,4,4)/s2/p1 (...cross_multi.py:125-127, Upsample).  Phase p uses the taps
   * tap[p*ntaps .. (p+1)*ntaps), the weight rows [p*n, (p+1)*n) of W (w_rows = n_phase*n, block_n | n) and writes at
   * out_base + phase_out_offset[p] (a residual is read at res_base + phase_out_offset[p]).  n_phase*ntaps <= 64.  Plain (non-halo) kernel only; no gn_partials. */
  int n_phase;
  long long phase_out_offset[4];
} ExtdmGemm;

int extdm_conv_gemm(const ExtdmGemm* g, void* stream);
/* sizeof(ExtdmGemm) as the library was compiled: lets a foreign-language binding verify its struct mirror. */
int extdm_sizeof_gemm(void);

/* ------------------------------------------------------------------------------------------------
 * Bandwidth-bound UNet kernels (channels-last bf16 activations, fp32 statistics).
 */

/* GroupNorm statistics: per (sample, group) sum and sum of squares over (T,H,W,C/G), as EXTDM_GN_CHUNKS
 * deterministic partial sums.  x: (B, P, C) bf16 with P = T*H*W.  stats: (B, EXTDM_GN_CHUNKS, 2, G) fp32
 * (sums then sums of squares).  Reference: nn.GroupNorm in Block.forward, ...cross_multi.py:166-171.
 * (The UNet runner does not launch this: its convolutions emit the same partials from their epilogue,
 * ExtdmGemm.gn_partials.) */
#define EXTDM_GN_CHUNKS 32
int extdm_groupnorm_stats(const void* x, float* stats, int B, long long P, int C, int G, void* stream);

/* GroupNorm apply + optional (scale+1, shift) + SiLU (+ residual).  ...cross_multi.py:170-178, :203.
 * y = silu(gn(x)*gamma+beta [* (scale[b,c]+1) + shift[b,c]]) [+ res].  scale_shift: (B, ss_stride) fp32 rows,
 * scale at [ss_off + c], shift at [ss_off + C + c]; may be NULL.  x, res, y: (B, P, C) bf16; in-place allowed.
 * stats: (B, n_part, 2, G) partial sums from extdm_groupnorm_stats (n_part = EXTDM_GN_CHUNKS) or from a
 * convolution's gn_partials (n_part = 128-row tiles per sample). */
int extdm_groupnorm_apply(const void* x, const float* stats, int n_part, const float* gamma, const float* beta,
                          const float* scale_shift, long long ss_stride, int ss_off, const void* res, void* y,
                          int B, long long P, int C, int G, float eps, void* stream);

/* Channel LayerNorm (gamma only, biased variance, eps) over the last dim of up to two concatenated
 * sources: y[row, :C0+C1] = LN(cat(x0[row], x1[row])) * gamma.  ...cross_multi.py:139-148.
 * Rows are (outer, inner) pairs: source row address = outer*x_outer_stride + inner*C (elements), which
 * lets a caller normalise only frames [t0,t1) of each sample.  y is dense (rows, C0+C1) bf16. */
int extdm_chan_layernorm(const void* x0, long long x0_outer_stride, int C0, const void* x1,
                         long long x1_outer_stride, int C1, const float* gamma, void* y, long long n_outer,
                         long long n_inner, float eps, void* stream);

/* Temporal-attention prologue (...cross_multi.py:307-328 with PreNorm :151-159): z = chanLN(x)*gamma;
 * u = LayerNorm(z)*w + b; xz = x + z.   x, u, xz: (rows, C) bf16. */
int extdm_temporal_prenorm(const void* x, const float* gamma, const float* ln_w, const float* ln_b, void* u,
                           void* xz, long long rows, int C, float eps, void* stream);

/* Per-(sample, channel) mean and unbiased std over frames [0, n_frames) x (H*W): adaptor.calc_mean_std,
 * ..._traj_ada.py:671-679, then normalise: y = (x - mean)/std (bf16).  x: (B, frames_total, HW, C) with sample
 * stride x_sample_stride.  mean_std: (2, B, C) fp32 = plane 0 mean, plane 1 std (the planes feed the GEMM
 * epilogue's col_shift / col_scale).  y: dense (B, n_frames, HW, C).
 * workspace: extdm_adaptor_workspace_floats(B, C) floats. */
long long extdm_adaptor_workspace_floats(int B, int C);
int extdm_adaptor_normalize(const void* x, long long x_sample_stride, void* y, float* mean_std, float* workspace,
                            int B, int n_frames, int HW, int C, float eps, void* stream);

/* Space-to-depth for the (1,4,4)/stride-2/pad-1 Downsample conv (...cross_multi.py:134-136):
 * z[f, y', x', (py*2+px)*C + c] = x[f, 2y'-1+py, 2x'-1+px, c] (zero outside), y' in [0,H/2], x' in [0,W/2]. */
int extdm_space_to_depth(const void* x, void* z, long long F, int H, int W, int C, void* stream);

/* im2col for the two 3-channel 7x7 convolutions whose input is the fp32 flow/occlusion volume
 * (init_noise_conv ..._traj_ada.py:916,1032 and the flow half of the base init_conv ...cross_multi.py:803):
 * a[(b*nt + t)*H*W + p, (ky*7+kx)*3 + c] = src(b, c, t0 + t, y+ky-3, x+kx-3), K padded to 192 with zeros.
 * Frames t < tc come from cond (B,3,tc,H,W), the rest from x (B,3,tp,H,W); both fp32 NCTHW. */
int extdm_im2col7_flow(const float* cond, const float* x, void* a, int B, int tc, int tp, int t0, int nt, int H,
                       int W, void* stream);

/* Gather kernels of the composite init_conv: init_conv(init_noise_conv(x)) (..._traj_ada.py:916,1032-1042) is one 13x13
 * convolution of the 3-channel flow minus a 7x7 convolution of the intermediate's values on the 3-pixel ring outside the
 * image (the intermediate is zero padded, so the composition holds only away from the border); the ring correction is a
 * set of phase GEMMs over the same x-im2col tensor (extdm_b200/unet.py: _composite_init).
 * im2col13x_flow: out[b, t_off + t, y, x, (dx + 6)*3 + c] = x[b, c, t, y, x + dx], dx in [-6, 6] (zeros outside the image and
 * in channels 40..63, channel 39 = 1: the carrier of constants); x (B, 3, tp, H, W) fp32, out (B, T, H, W, 64) bf16 -- the 13
 * kernel rows are taps of the GEMM.
 * init_corner_fix: the ring correction is summed side by side over all positions of each side, which counts the four
 * 3x3 corner blocks of the ring twice; their contribution (linear in the image's 3x3x3 corner values + a constant) is added
 * back to the 3x3 output pixels next to each corner.  table: (4 corners [top-left, top-right, bottom-left, bottom-right],
 * 9 pixels, 28, C) fp32, k = (r*3 + s)*3 + c of the corner block's image values, k = 27 the constant; x0 (B, T, H, W, C)
 * bf16, updated in place on frames [t_off, t_off + tp). */
int extdm_im2col13x_flow(const float* x, void* out, int B, int tp, int T, int t_off, int H, int W, void* stream);
int extdm_init_corner_fix(const float* x, const float* table, void* x0, int B, int tp, int T, int t_off, int H, int W,
                          int C, void* stream);

/* Polyphase init_conv of the u12 UNet (..._traj_u12.py:1039-1042: F.interpolate x2 then init_conv): the 7x7 convolution of
 * the up-sampled TrajWarp features is evaluated on the low-resolution tensor (5x5 taps per output parity).  fpad:
 * (F, h + 4, w + 4, C) bf16 with the interior written -> replicate-padded in place; top / bottom: (F, 2w + 6, C) = row 0 / 2h - 1
 * of the up-sampled tensor with columns clamped; left / right: (F, 2h, C) = its column 0 / 2w - 1. */
int extdm_upsample2_border(void* fpad, void* top, void* bottom, void* left, void* right, long long F, int h, int w, int C,
                           void* stream);

/* Bilinear resize (align_corners=False) of channels-last frames: F.interpolate in ..._traj_ada.py:1039-1041. */
int extdm_bilinear_resize_cl(const void* x, void* y, long long F, int h, int w, int H, int W, int C, void* stream);

/* Sinusoidal embedding + time_mlp + every ResnetBlock's SiLU->Linear in one launch
 * (...cross_multi.py:110-122, 812-817, 184-199).  time: (B,) int64.  w1 (4d, d), w2 (4d, 4d) fp32;
 * wss: (n_ss, 4d) fp32 = all blocks' mlp.1.weight stacked, bss (n_ss).  out: (B, n_ss) fp32.
 * scratch: (B, 4d) fp32 workspace (the SiLU(time embedding) rows shared by the two stages). */
int extdm_time_mlp(const long long* time, const float* w1, const float* b1, const float* w2, const float* b2,
                   const float* wss, const float* bss, float* out, float* scratch, int B, int dim, int n_ss,
                   void* stream);

/* Final 1x1 projections of the two heads (final_conv[1], occlusion_map[1]; ...cross_multi.py:875-892) on
 * frames [t0, T): out (B, 3, T-t0, H, W) fp32 NCTHW; hf / ho: (B, T, HW, C) bf16 head features. */
int extdm_head_project(const void* hf, const void* ho, const float* wf, const float* bf, const float* wo,
                       const float* bo, float* out, int B, int T, int t0, int HW, int C, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Attention.  qkv: channels-last bf16 with channel = which*heads*dh + head*dh + d (which in q,k,v).
 */

/* 3-D shifted-window attention core (WindowAttention3D + window_partition/roll/mask/reverse,
 * ...cross_multi.py:345-390, 462-497, 522-560).  qkv: (B, T, H, W, 3*heads*dh); out: (B, T, H, W, heads*dh).
 * Window (wd, wh, ww) tokens = 32 or 64; T is zero-padded to a multiple of wd; shift (sd, sh, sw).
 * bias_table: ((2wd-1)(2wh-1)(2ww-1), heads) fp32; rope_cos/sin: (tokens, dh/2) fp32. */
int extdm_window_attention(const void* qkv, void* out, const float* bias_table, const float* rope_cos,
                           const float* rope_sin, int B, int T, int H, int W, int heads, int dh, int wd, int wh,
                           int ww, int sd, int sh, int sw, void* stream);

/* extdm_head_project with the last GroupNorm(8)+SiLU+residual of each head's ResnetBlock fused in: hXf / hXo are
 * the block2 convolution outputs (bf16, (B,T,HW,C)), rf / ro the residual branches, partf / parto the convolutions'
 * gn_partials ((B, n_part, 16) fp32), gamma / beta the block2 norm parameters.  Writes out as extdm_head_project. */
int extdm_head_project_gn(const void* h2f, const void* rf, const float* partf, const float* gamma_f,
                          const float* beta_f, const void* h2o, const void* ro, const float* parto,
                          const float* gamma_o, const float* beta_o, int n_part, const float* wf, const float* bf,
                          const float* wo, const float* bo, float* out, int B, int T, int t0, int HW, int C, int G,
                          float eps, void* stream);

/* Whole Residual(PreNorm(STWAttentionLayer)) in one kernel for the high-resolution levels:
 * y = x + proj(window_attention(chanLN(x) @ Wqkv^T)) (...cross_multi.py:139-159, 409-560).  x, y: (B,T,H,W,C) bf16
 * (y must not alias x); wqkv: (3*heads*dh, C) bf16; wproj: (C, heads*dh) bf16.  Supported: heads 8 and
 * (64 tokens, dh 16, C 64|128) or (32 tokens, dh 32, C 64) -- extdm_stw_fused_supported() returns 1. */
int extdm_stw_fused_supported(int C, int heads, int dh, int wd, int wh, int ww);
int extdm_stw_fused(const void* x, void* y, const float* gamma, const void* wqkv, const void* wproj,
                    const float* proj_bias, const float* bias_table, const float* rope_cos, const float* rope_sin,
                    int B, int T, int H, int W, int C, int heads, int dh, int wd, int wh, int ww, int sd, int sh,
                    int sw, float eps, void* stream);

/* The same layer with the preceding ResnetBlock's last GroupNorm + SiLU + residual applied on load
 * (...cross_multi.py:170-178 + :203 feeding :499-560): layer input x = silu(h*a[b,c] + d[b,c]) + res, h = the block2
 * convolution output, (a, d) = extdm_groupnorm_affine of its gn_partials.  Saves the groupnorm_apply pass (one read of
 * h, one of res, one write of x) and the layer's own read of x.  C = 64, (4,4,4) windows, 8 heads x 16. */
int extdm_stw_fused_pre_supported(int C, int heads, int dh, int wd, int wh, int ww);
int extdm_stw_fused_pre(const void* h, const void* res, const float* ad, void* y, const float* gamma, const void* wqkv,
                        const void* wproj, const float* proj_bias, const float* bias_table, const float* rope_cos,
                        const float* rope_sin, int B, int T, int H, int W, int C, int heads, int dh, int wd, int wh,
                        int ww, int sd, int sh, int sw, float eps, void* stream);
/* GroupNorm(8) as a per-(sample, channel) affine: ad (B, 2, C) fp32 = (rstd*gamma, beta - mean*rstd*gamma) from
 * per-tile partial sums (B, n_part, 16).  P = T*H*W elements per channel. */
int extdm_groupnorm_affine(const float* part, int n_part, const float* gamma, const float* beta, float* ad, int B,
                           long long P, int C, int G, float eps, void* stream);

/* Whole temporal attention layer Residual(PreNorm(EinopsToAndFrom(AttentionLayer))) in one kernel for C = 64
 * (init_temporal_attn, ...cross_multi.py:253-328, 794-795): y = x + z + to_out(attn(LayerNorm(z))), z = chanLN(x)*gamma;
 * sequence = the T <= 32 frames of one pixel, rotary over the frame index, rel_bias (heads, 2T-1) as in
 * extdm_temporal_attention.  x, y: (B, T, HW, C) bf16 (y must not alias x); wqkv (3*heads*dh, C), wout (C, heads*dh). */
int extdm_temporal_fused_supported(int C, int heads, int dh, int T);
int extdm_temporal_fused(const void* x, void* y, const float* gamma, const float* ln_w, const float* ln_b,
                         const void* wqkv, const void* wout, const float* rel_bias, const float* rope_cos,
                         const float* rope_sin, int B, int T, int HW, int C, int heads, int dh, float eps,
                         void* stream);

/* TrajWarp (BAIR 'u12' variant, ..._traj_u12.py:719-827).  Multi-head cross attention core
 * softmax(q k^T / sqrt(dh)) v (ScaledDotProductAttention :719-728, heads split as in _reshape_to_batches
 * :783-789): q (B, Lq, ldq), k / v (B, Lk, ldk), out (B, Lq, ldo) bf16; head h = columns [h*dh, (h+1)*dh).
 * dh must be 32, Lq and Lk multiples of 64.  The Linear+ReLU projections around it run on extdm_conv_gemm. */
int extdm_cross_attention(const void* q, const void* k, const void* v, void* out, int B, int heads, int dh, int Lq,
                          int Lk, int ldq, int ldk, int ldo, void* stream);
/* MaxPool3d((1,2,2)) (TrajWarp.down :811) and F.interpolate(bilinear, align_corners=False) (:1036) on channels-last
 * bf16 frames addressed as groups x frames_per_group: frame fi of group gi starts at
 * base + gi*group_stride + fi*(H*W*C) elements (lets a caller touch frames [tc, T) of every sample). */
int extdm_maxpool2_frames_cl(const void* x, void* y, int groups, int frames_per_group, long long x_group_stride,
                             long long y_group_stride, int H, int W, int C, void* stream);
int extdm_bilinear_resize_frames_cl(const void* x, void* y, int groups, int frames_per_group,
                                    long long x_group_stride, long long y_group_stride, int h, int w, int H, int W,
                                    int C, void* stream);

/* Temporal attention core (Attention.forward ...cross_multi.py:269-302): sequence = T frames of one pixel.
 * qkv: (B, T, HW, 3*heads*dh); out: (B, T, HW, heads*dh); rel_bias: (heads, 2T-1) fp32 indexed by (j-i+T-1). */
int extdm_temporal_attention(const void* qkv, void* out, const float* rel_bias, const float* rope_cos,
                             const float* rope_sin, int B, int T, int HW, int heads, int dh, void* stream);

/* ------------------------------------------------------------------------------------------------
 * DDIM sampler (GaussianDiffusion.ddim_sample, model/BaseDM_adaptor/Diffusion.py:231-255), fp32.
 */

/* x_start = c_recip*img - c_recipm1*pred; s[b] = max(1, quantile_0.9(|x_start[b]|)) with torch.quantile's
 * fp32 linear interpolation (exact order statistics by radix select).  n = elements per sample. */
int extdm_ddim_threshold(const float* img, const float* pred, float c_recip, float c_recipm1, float q, float* s,
                         int B, int n, void* stream);
/* img_out = clamp(x_start, -s, s)/s * sqrt_alpha_next + c*pred + sigma*noise (noise may be NULL). */
int extdm_ddim_update(const float* img, const float* pred, const float* noise, const float* s, float c_recip,
                      float c_recipm1, float sqrt_alpha_next, float c, float sigma, float* img_out,
                      float* x_start_out, int B, int n, void* stream);
/* As extdm_ddim_update, with z drawn inside the kernel instead of read from a noise tensor: the Philox draw of
 * (seeds[b], step, stream 0) documented with the DDPM sampler below, so a video's noise depends on its seed only.
 * Iteration i of the DDIM loop passes step = i (counter (element index / 4 within the video, i, 0, 0)); x_T is
 * extdm_ddpm_fill_normal (stream 1, counter (element index / 4, 0, 1, 0)); the last iteration (time_next == 0) adds
 * no noise and calls extdm_ddim_update with noise = NULL.  sigma*z is always added (a signed zero at eta = 0), so
 * the result equals extdm_ddim_update fed the same draws, bit for bit.  seeds: (B,) int64.  Added under ABI
 * version 5 (backward compatible). */
int extdm_ddim_update_seeded(const float* img, const float* pred, const long long* seeds, int step, const float* s,
                             float c_recip, float c_recipm1, float sqrt_alpha_next, float c, float sigma,
                             float* img_out, float* x_start_out, int B, int n, void* stream);

/* ------------------------------------------------------------------------------------------------
 * DDPM ancestral sampler (GaussianDiffusion.p_sample_loop, model/BaseDM_adaptor/Diffusion.py:136-189 with the
 * keyword fix of SURVEY App. E10), fp32.  Added under ABI version 5 (backward compatible).
 *
 * Per-step values live on the device so that one captured iteration replays for every timestep:
 *   rows  (n_steps, 5) fp32: {sqrt_recip_alphas_cumprod, sqrt_recipm1_alphas_cumprod, posterior_mean_coef1,
 *                             posterior_mean_coef2, nonzero_mask * exp(0.5 * posterior_log_variance_clipped)}[times[i]]
 *   step  one int32, the current row; seeds (B,) int64, one per video.
 * Noise is Philox4x32-10 + Box-Muller with key = the video's seed and counter = (element index / 4 within the video,
 * step, stream, 0); stream 0 is the noise of loop step `step`, stream 1 the initial x_T.  The DDIM sampler with
 * per-video seeds (extdm_ddim_update_seeded) uses the same counter layout: x_T from stream 1, the noise of DDIM
 * iteration i from (step = i, stream 0).  Stream 2 is the epsilon of the denoising-loss evaluation (extdm_q_sample):
 * counter (element index / 4 within the video, t[b], 2, 0), so a video's epsilon depends on its seed and its timestep
 * only, and every timestep of a loss curve draws its own.  Stream 3 is the noise of the stochastic DPM-Solver++(2M)
 * (extdm_dpmpp_update): iteration i draws counter (element index / 4 within the video, i, 3, 0); its x_T is stream 1.
 * Streams 4 and 5 are the epsilons of the two endpoints of an interpolation (extdm_q_interpolate): counter (element
 * index / 4 within the video, t, 4 or 5, 0), t the mix timestep; its loop noise is stream 0 as above.
 * Stream 6 is the noise of the keyframe replacements (extdm_impose_known): replacement point k draws counter (element
 * index / 4 within the video, k, 6, 0); the loop noise around it is that of the plain DDIM or ancestral sampler.
 */

/* s[b] = max(1, quantile_q(|c_recip*img - c_recipm1*pred|)) with the coefficients of row *step (as
 * extdm_ddim_threshold). */
int extdm_ddpm_threshold(const float* img, const float* pred, const float* rows, const int* step, float q, float* s,
                         int B, int n, void* stream);
/* x0 = clamp(c_recip*img - c_recipm1*pred, -s, s)/s; img_out = (c1*x0 + c2*img) + sig*z with row *step.  z is slice
 * *step of `noise` ((n_steps, B, n)) when noise != NULL, else the Philox draw of (seeds[b], *step).  x_start_out
 * (optional) receives x0. */
int extdm_ddpm_update(const float* img, const float* pred, const float* rows, const int* step, const long long* seeds,
                      const float* noise, const float* s, float* img_out, float* x_start_out, int B, int n,
                      void* stream);
/* out (B, n) = the x_T draw (stream 1) of each video's seed. */
int extdm_ddpm_fill_normal(const long long* seeds, float* out, int B, int n, void* stream);
/* out (B, n) = row *step of table (n_steps, n) for every b: the per-step time-MLP (scale, shift) rows, which do not
 * depend on the sample. */
int extdm_ddpm_broadcast_row(const float* table, const int* step, float* out, int B, int n, void* stream);
/* *step += 1; time[0..B) = times[*step] while *step < n_steps (one block). */
int extdm_ddpm_advance(int* step, const long long* times, int n_steps, long long* time, int B, void* stream);

/* ------------------------------------------------------------------------------------------------
 * DPM-Solver++(2M) sampler (GaussianDiffusion.dpm_solver_sample; Lu et al. 2022, data prediction with dynamic
 * thresholding), fp32.  Added under ABI version 5 (backward compatible).
 */

/* One iteration after the threshold (extdm_ddim_threshold with the same c_recip, c_recipm1 and s):
 *   D       = clamp(c_recip*img - c_recipm1*pred, -s[b], s[b]) / s[b]          (as extdm_ddim_update's x_start)
 *   img_out = ((A*img + B_coef*D) + C_coef*d_prev) + N*z                       (each product rounded, no FMA)
 * The C_coef term is left out when d_prev == NULL (first step), the N term when seeds and noise are both NULL (the
 * deterministic solver).  z is read from noise ((B, n)) when given, else it is the Philox draw of (seeds[b], step,
 * stream 3) documented above.  final != 0: img_out = D and no noise is drawn.  d_out receives D and may equal d_prev;
 * img_out may equal img.  seeds and noise are not both given. */
int extdm_dpmpp_update(const float* img, const float* pred, const float* d_prev, const long long* seeds,
                       const float* noise, int step, const float* s, float c_recip, float c_recipm1, float A,
                       float B_coef, float C_coef, float N, int final, float* img_out, float* d_out, int B, int n,
                       void* stream);

/* ------------------------------------------------------------------------------------------------
 * Denoising-loss evaluation (GaussianDiffusion.denoising_loss: the forward of Diffusion.py p_losses, :286-319, under
 * no_grad), fp32.  Added under ABI version 5 (backward compatible).
 */

/* Forward diffusion q(x_t | x_0): x_t_out = sqrt_acp[t[b]] * x_start + sqrt_1m_acp[t[b]] * eps, two roundings and one
 * sum (no FMA), bit-exact against the torch fp32 expression.  eps is read from `noise` when noise != NULL, else it is
 * the Philox draw of (seeds[b], t[b], stream 2) documented above; eps_out receives it.  x_start, noise, x_t_out,
 * eps_out: (B, n) fp32; t, seeds: (B,) int64 with every t[b] in [0, length of the tables) -- the caller checks it;
 * sqrt_acp, sqrt_1m_acp: the fp32 sqrt_alphas_cumprod / sqrt_one_minus_alphas_cumprod buffers. */
int extdm_q_sample(const float* x_start, const long long* t, const long long* seeds, const float* noise,
                   const float* sqrt_acp, const float* sqrt_1m_acp, float* x_t_out, float* eps_out, int B, int n,
                   void* stream);
/* out (B, tp) fp32 = mean over (3, h*w) of (eps - pred)^2 (l1 == 0) or |eps - pred| (l1 != 0) per (video, frame) of
 * eps, pred (B, 3, tp, h*w) fp32; per_frame = 3*h*w elements of one (video, frame).  Terms and sum in fp64, one block
 * per (video, frame) with a fixed reduction tree: repeated calls are bit-identical and out[b] depends on video b's
 * data only. */
int extdm_denoise_loss(const float* eps, const float* pred, float* out, int B, int tp, int per_frame, int l1,
                       void* stream);

/* ------------------------------------------------------------------------------------------------
 * Interpolation between two futures (GaussianDiffusion.interpolate, Diffusion.py:261-274 with the keyword fix of
 * SURVEY App. E10), fp32.  Added under ABI version 5 (backward compatible).
 */

/* The mix of two forward diffusions at one timestep t shared by the batch, a = sqrt_acp[t], b = sqrt_1m_acp[t]:
 *   x_t_out = c1 * (a * x1 + b * eps1) + c2 * (a * x2 + b * eps2)       (each product rounded, no FMA)
 * bit-exact against the torch fp32 expression with c1 = fp32(1 - lam), c2 = fp32(lam).  eps1, eps2 are noise[0] and
 * noise[1] of noise ((2, B, n)) when noise != NULL, else the Philox draws of (seeds[b], t, stream 4) and (seeds[b], t,
 * stream 5) documented above.  Exactly one of seeds ((B,) int64) and noise is given.  x1, x2, x_t_out: (B, n) fp32;
 * t in [0, length of the tables) -- the caller checks the upper bound; sqrt_acp, sqrt_1m_acp: the fp32
 * sqrt_alphas_cumprod / sqrt_one_minus_alphas_cumprod buffers. */
int extdm_q_interpolate(const float* x1, const float* x2, int t, const long long* seeds, const float* noise,
                        const float* sqrt_acp, const float* sqrt_1m_acp, float c1, float c2, float* x_t_out, int B,
                        int n, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Keyframe-conditioned sampling (GaussianDiffusion.sample_with_known: replacement of known frames, Song et al. 2021,
 * Lugmayr et al. 2022), fp32.  Added under ABI version 5 (backward compatible).
 */

/* Replacement point k on x, x_known (B, 3, tp, hw) fp32 and known (B, tp) bool (one byte per flag): every element of
 * frame f of video b with known[b, f] becomes
 *   x = a * x_known + b * eps_k                                          (two roundings, one sum, no FMA)
 * or x_known itself when final (nothing is drawn).  Elements of unknown frames are neither read from x_known nor
 * written.  eps_k is noise[k] of noise ((K, B, 3*tp*hw)) when noise != NULL, else the Philox draw of (seeds[b], k,
 * stream 6) documented above; exactly one of seeds ((B,) int64) and noise is given.  (a, b, k, final) are the launch
 * scalars when rows == NULL (the DDIM loop); otherwise k = *step and (a, b, final != 0) = rows[k] of the (K + 1, 3)
 * fp32 table (the ancestral loop, through the step counter of extdm_ddpm_update).  hw = h*w must be a multiple of 4. */
int extdm_impose_known(float* x, const float* x_known, const unsigned char* known, const long long* seeds,
                       const float* noise, float a, float b, int k, int final, const float* rows, const int* step,
                       int B, int tp, int hw, void* stream);

/* ------------------------------------------------------------------------------------------------
 * LFAE decode (Generator.forward_with_flow / deform_input / apply_optical, model/LFAE/generator.py:63-93,
 * 152-206).  flow: (F, h, w, 2) fp32 normalised (x, y); occ: (F, 1, h, w) fp32 or NULL.
 */

/* out[f, y, x, c] = warp(skip)[..] * occ + prev * (1 - occ) on channels-last bf16 features.
 * skip: (Fs, H, W, C) with Fs == F or F % Fs == 0 (skip of frame f is skip[f / (F/Fs)]: the encoder runs once
 * per video); prev: (F, H, W, C) or NULL; flow/occ are bilinearly resized (align_corners=False) from (h, w)
 * to (H, W) on the fly; grid_sample is bilinear / zeros / align_corners=True.  If up2 != 0 the result is
 * written nearest-upsampled x2: out is (F, 2H, 2W, C) (F.interpolate(scale_factor=2) of UpBlock2d, util.py:107). */
int extdm_warp_blend_cl(const void* skip, const void* prev, const float* flow, const float* occ, void* out,
                        long long F, long long Fs, int H, int W, int C, int h, int w, int up2, void* stream);

/* Image-space warp + final blend, fp32 NCHW (generator.py:163 and :201-204):
 * deformed = grid_sample(src, resize(flow));  prediction = deformed*occ + dec*(1-occ)  (or = deformed when
 * occ == NULL, generator.py:81-90).  src: (Fs, 3, H, W); dec: (F, H, W, dec_stride) fp32 channels-last
 * decoder output (sigmoid already applied), first 3 channels used; prediction / deformed: (F, 3, H, W);
 * either output pointer may be NULL. */
int extdm_warp_image(const float* src, const float* dec, int dec_stride, const float* flow, const float* occ,
                     float* prediction, float* deformed, long long F, long long Fs, int H, int W, int h, int w,
                     void* stream);

/* Diagnostic view of the warp index math used by the two kernels above (generator.py:63-71 + ATen GridSampler /
 * UpSampleBilinear2d): for every pixel of the (H, W) target, the resized flow and occlusion gflow (F,H,W,3) =
 * (gx, gy, occ), the north-west tap xy (F,H,W,2) = (x0, y0) and the bilinear weights (F,H,W,4) = (nw, ne, sw, se).
 * Parity tests compare these bit-for-bit with the fp32 oracle. */
int extdm_warp_taps(const float* flow, const float* occ, int* xy, float* weights, float* gflow, long long F, int H,
                    int W, int h, int w, void* stream);

/* Eval-mode BatchNorm + ReLU on channels-last bf16 (ResBlock2d pre-activation, util.py:83-89):
 * y = relu(x*scale[c] + shift[c]). */
int extdm_bn_relu_cl(const void* x, const float* scale, const float* shift, void* y, long long rows, int C,
                     void* stream);
/* 2x2 average pool, channels-last bf16 (DownBlock2d, util.py:124,130). */
int extdm_avgpool2_cl(const void* x, void* y, long long F, int H, int W, int C, void* stream);
/* fp32 NCHW image -> channels-last bf16 im2col rows for the 7x7 `first` conv (K = 147 padded to 192). */
int extdm_im2col7_image(const float* img, void* a, long long F, int H, int W, void* stream);

/* Generic layout helpers. */
int extdm_ncthw_to_cl(const float* x, void* y, int B, int C, long long T, long long HW, void* stream);
int extdm_cl_to_ncthw(const void* x, float* y, int B, int C, long long T, long long HW, void* stream);

/* ------------------------------------------------------------------------------------------------
 * LFAE conditioning stage (SURVEY.md section 8f-1): fp32 channels-last kernels around the tf32 convolutions
 * (ExtdmGemm.tf32) of RegionPredictor / BGMotionPredictor / PixelwiseFlowPredictor.
 */

/* AntiAliasInterpolation2d (model/LFAE/util.py:224-271) + NCHW -> channels-last: out (F, H/stride, W/stride, cpad) fp32,
 * channels [0, ca) from a[(f / a_div)], [ca, ca+cb) from b[(f / b_div)] (b may be NULL), the rest zero.  kern: ks*ks
 * Gaussian taps (ks == 1: no filter). */
int extdm_image_to_cl(const float* a, int ca, int a_div, const float* b, int cb, int b_div, const float* kern, int ks,
                      int stride, float* out, int F, int H, int W, int cpad, void* stream);
/* AvgPool2d(2) / nearest x2 up-sampling of (F, H, W, C) fp32 (DownBlock2d / UpBlock2d, util.py:97-131). */
int extdm_avgpool2_f32_cl(const float* x, float* y, long long F, int H, int W, int C, void* stream);
int extdm_upsample2_f32_cl(const float* x, float* y, long long F, int H, int W, int C, void* stream);
/* RegionPredictor head, pca_based (region_predictor.py:95-140): logits (F, h, w, ldc) = 'same' 7x7 convolution output;
 * softmax(logits / temperature) over the window cropped by `crop` = 3 - pad pixels per side; shift (F, K, 2), covar
 * (F, K, 2, 2). */
int extdm_region_moments(const float* logits, int ldc, int F, int K, int h, int w, int crop, float temperature,
                         float* shift, float* covar, void* stream);
/* PCA affine of the region covariances (region_predictor.py:130-146: u, s, v = svd(covar); affine = u diag(sqrt s)) in
 * closed form with the singular-vector sign convention of cuSOLVER's batched Jacobi, i.e. of torch.svd on CUDA -- what the
 * reference itself computes on a GPU.  covar, affine: (n, 2, 2) fp32. */
int extdm_pca_affine(const float* covar, float* affine, int n, void* stream);
/* PixelwiseFlowPredictor heat-maps + sparse motions + deformed sources (pixelwise_flow_predictor.py:48-112) for F = B*tc
 * frames; source parameters / image are those of each video's last conditioning frame.  shift (F,K,2), covar / affine
 * (F,K,2,2), bg (F,3,3) or NULL; src (F, h, w, src_ld) channels 0..2; inp (F, h, w, cpad) channel 4k + {0: heat, 1..3:
 * warped source}; motion (F, K+1, h, w, 2). */
int extdm_sparse_motion(const float* src, int src_ld, const float* shift, const float* covar, const float* affine,
                        const float* bg, int F, int K, int tc, int h, int w, int revert_axis_swap, int use_covar,
                        float region_var, float* inp, int cpad, float* motion, void* stream);
/* extdm_sparse_motion with any source slot: frames come in groups of `group` consecutive frames (one video each), and
 * the source parameters / image of frame f are those of frame (f / group) * group + src_slot, 0 <= src_slot < group,
 * F % group == 0.  extdm_sparse_motion is this entry with group = tc, src_slot = tc - 1; flow-autoencoder
 * reconstruction (FlowAE.reconstruct) calls it with group = T frames per video.  Added under ABI version 5 (backward
 * compatible). */
int extdm_sparse_motion_src(const float* src, int src_ld, const float* shift, const float* covar, const float* affine,
                            const float* bg, int F, int K, int group, int src_slot, int h, int w, int revert_axis_swap,
                            int use_covar, float region_var, float* inp, int cpad, float* motion, void* stream);
/* mask softmax, flow = sum_k mask_k * motion_k, occlusion = sigmoid (pixelwise_flow_predictor.py:140-152).  head (F, h, w,
 * ldc): channels [0, K] mask logits, K+1 occlusion logit.  grid (B, 2, tc, h, w), conf (B, 1, tc, h, w) or NULL. */
int extdm_flow_compose(const float* head, int ldc, const float* motion, int F, int K, int tc, int h, int w, float* grid,
                       float* conf, void* stream);
/* BGMotionPredictor head (bg_motion_predictor.py:52-64): spatial mean of feat (F, hw, C), Linear(C -> n_out), 3x3 matrix.
 * bg_type 1 shift (n_out 2), 2 affine (6), 3 perspective (8).  out (F, 3, 3). */
int extdm_bg_head(const float* feat, int F, int hw, int C, const float* fcw, const float* fcb, int n_out, int bg_type,
                  float* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif
