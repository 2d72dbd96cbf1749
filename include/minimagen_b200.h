/*
 * minimagen_b200 -- C ABI of the B200-native (sm_100a) kernels behind MinImagen's U-Net denoising hot path.
 *
 * This header is the drop-in boundary: plain `extern "C"` entry points, raw device pointers + sizes + a CUDA stream
 * (passed as void*), no torch types.  The reference is pure Python/PyTorch, so the "FFI" a maintainer would bind is
 * ctypes (see INTEGRATION.md); every entry point below names the reference call site(s) (file:line under
 * /root/reference) whose stock torch op it replaces.
 *
 * Conventions
 *   - all pointers are DEVICE pointers unless the name ends in `_host`;
 *   - activations inside the U-Net are NHWC; "f32" buffers are float, "f16" buffers are IEEE half;
 *   - the caller owns every buffer (inputs, outputs, workspaces); nothing is allocated or retained by the library;
 *   - kernels are enqueued on `stream` (a cudaStream_t) and return immediately -> CUDA-graph capturable;
 *   - return value: 0 on success, negative on error; mi_last_error() returns a static description of the last
 *     failing call of the calling thread.  No entry point ever falls back to a CPU implementation.
 */
#ifndef MINIMAGEN_B200_H_
#define MINIMAGEN_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MI_ABI_VERSION 2

int mi_abi_version(void);
const char* mi_last_error(void);
/* 1 if the current device is compute capability 10.x (the only target), else 0 */
int mi_device_ok(void);
/* Process-wide launch mode.  programmatic_dependent_launch != 0: every kernel is launched with
 * cudaLaunchAttributeProgrammaticStreamSerialization, so its prologue overlaps the tail of the kernel before it on the
 * same stream (each kernel still waits for its predecessor before touching global memory).  Default 0. */
int mi_set_launch_mode(int programmatic_dependent_launch);

/* ------------------------------------------------------------------------------------------------- weights
 * One-time repack of a conv / linear weight from the reference's checkpoint layout (C_out, C_in, KH, KW) fp32
 * (nn.Conv2d.weight, nn.Linear.weight with KH=KW=1) into the tensor-core layout [C_out][(r*KW+s)*C_in + c] fp16,
 * multiplied by `scale` (used to fold q * dim_head**-0.5, layers.py:59/:237, into to_q).
 * Replaces nothing at run time in the reference; it is the load_state_dict-side half of mi_conv2d_igemm_f16. */
int mi_pack_conv_weight_f16(const float* w_oihw, int c_out, int c_in, int kh, int kw, float scale, void* out_f16,
                            void* stream);

/* The same weight packed for the DATA gradient of a stride-1 'same' conv (or of a linear layer, kh = kw = 1): taps flipped,
 * in / out channels swapped -> [c_in][((kh-1-r)*kw + (kw-1-s))*c_out + o] fp16; mi_conv2d_igemm_f16 on dy with this operand
 * (c_in' = c_out, c_out' = c_in) is dL/dx.  Training side (SURVEY 8f-2). */
int mi_pack_conv_weight_dgrad_f16(const float* w_oihw, int c_out, int c_in, int kh, int kw, void* out_f16, void* stream);

/* ------------------------------------------------------------------------------------------------- convolution
 * Tensor-core (tcgen05 + TMA + TMEM) implicit-GEMM convolution / linear layer.
 * Replaces nn.Conv2d / nn.Linear forward at: layers.py:129,145 (Block.project 3x3), layers.py:415,439 (res_conv 1x1),
 * layers.py:319 (Downsample 4x4 stride 2), layers.py:514 (Upsample conv 3x3), layers.py:157,160 (ChanFeedForward 1x1),
 * layers.py:41-42,48 and :213-214,217 (attention to_q / to_kv / to_out), Unet.py:234 (Parallel 3x3 + 1x1).
 *
 *   act_f16   [B][phases][H][W][lda] fp16; channels [c_off, c_off+c_in) are consumed
 *   (H, W)    OUTPUT pixel grid.  mode 0: stride 1, "same" zero padding, kh x kw odd taps, phases = 1.
 *             mode 1: the reference's Downsample (4x4, stride 2, pad 1); act is the 4-phase split of the
 *             (2H x 2W) input produced by mi_cast_act(mode=2).
 *             mode 6: the same Downsample conv reading the UN-split fp16 input [B][2H][2W][lda] in place (TMA element
 *             stride 2 picks every second pixel of each tap's box) -- no phase-split copy.
 *             mode 2+p (p = 2a+b in 0..3), kh = kw = 2: sub-pixel phase (a, b) of the reference's Upsample
 *             (nn.Upsample(scale_factor=2, 'nearest') followed by Conv2d 3x3 pad 1, layers.py:513-514): the outputs
 *             (2y+a, 2x+b) depend only on the LOW-RES pixels (y+a-1+r, x+b-1+s), r,s in {0,1}, through the 3x3 weights
 *             summed over the taps that land on the same low-res pixel (w_f16 = that 2x2 kernel, packed as usual).
 *             (H, W) is the low-res grid; the caller points out_* at output pixel (a, b) and passes the strides of the
 *             2H x 2W output (out_sh = 2 rows, out_sw = 2 pixels).  4 launches replace upsample copy + 3x3 conv at
 *             4/9 of the FLOPs.
 *   w_f16     packed by mi_pack_conv_weight_f16, [c_out][kh*kw*c_in]
 *   bias      [c_out] fp32 or NULL;  residual: fp32 or NULL, added in the epilogue, addressed like the output
 *   out_f32 / out_f16   either or both; element (b,h,w,n) is written at  b*out_sb + h*out_sh + w*out_sw + n*out_sc
 *             (out_sc = 1: channel-contiguous NHWC-style rows; out_sc = H*W with out_sw = 1: NCHW, used by final_conv
 *             Unet.py:327,472); only channels n < n_valid are stored (n_valid = 0: all; lets c_out be zero-padded up
 *             to a multiple of 16); residual requires out_sc = 1
 *   act2_f16  optional second activation tensor [B][phases][H][W][lda2]: the input is then the VIRTUAL channel concat
 *             cat(act[c_off : c_off+c_in1], act2[c_off2 : c_off2+c_in-c_in1]) of every tap -- the up-path skip connection
 *             torch.cat((x, skip * 2**-0.5), dim=1) (Unet.py:445) without materialising it (the 2**-0.5 is folded into the
 *             packed weight columns); NULL otherwise (then c_in1 is ignored)
 *   out_stats optional [B][c_out/16][2] doubles, zero on entry: per (image, 16-channel block) sum and sum of squares of
 *             the OUTPUT (after bias/residual), accumulated in the epilogue -- the GroupNorm statistics of the next
 *             Block (layers.py:136) for free; needs out_sc = 1
 *   block_n   0 = auto, or one of 16/32/64/128/256 (tile width; must divide c_out)
 *   workspace reserved, pass NULL / 0
 * Requirements: c_in % 64 == 0, c_out % 16 == 0, W a power of two >= 8 (or W >= 128), see mi_conv2d_igemm_supported.
 * A plain GEMM  out[M][N] = act[M][K] * w[N][K]^T  is the case B=1, H=1, W=M, kh=kw=1. */
int mi_conv2d_igemm_supported(int H, int W, int c_in, int c_out);
int mi_conv2d_igemm_f16(const void* act_f16, int B, int H, int W, int lda, int c_off, int c_in, const void* act2_f16,
                        int lda2, int c_off2, int c_in1, const void* w_f16, int c_out, int kh, int kw, int mode,
                        const float* bias, const float* residual, float* out_f32, void* out_f16, double* out_stats,
                        long long out_sb, long long out_sh, long long out_sw, long long out_sc, int n_valid,
                        int block_n, int* err_flag, void* workspace, long long workspace_bytes, void* stream);
/* ResnetBlock.forward's tail (layers.py:437-439)  block2.project(h) + res_conv(x)  as ONE launch of the swapped-operand 3x3
 * kernel: after the nine taps of the 3x3 conv over `act` (the GroupNorm/SiLU operand of block2), the 1x1 res_conv rides in the
 * same accumulator as x_cin/64 extra K chunks read at the centre tap of x's halo tile -- no separate 1x1 launch, no fp32
 * round trip of the residual branch through HBM.  w_f16 = [c_out][9*c_in + x_cin]: each row is the packed 3x3 weight followed
 * by the 1x1 weight; bias = the sum of both convs' biases.  Both operands may be virtual concats (act2 / x_act2 hold channels
 * >= c_in1 / x_cin1, the skip scale folded into the weight columns).  Outputs [B][H][W][c_out] contiguous; residual, out_stats
 * as mi_conv2d_igemm_f16.  Requirements: mi_conv3x3_res1x1_supported (H % 32 == 0 and W % 8 == 0, or W == 16 and H % 16 == 0;
 * c_in % 64 == 0, x_cin % 64 == 0, c_out % 128 == 0). */
int mi_conv3x3_res1x1_supported(int H, int W, int c_in, int c_out, int x_cin);
int mi_conv3x3_res1x1_f16(const void* act_f16, int B, int H, int W, int lda, int c_in, const void* act2_f16, int lda2,
                          int c_in1, const void* x_f16, int ldx, int x_cin, const void* x2_f16, int ldx2, int x_cin1,
                          const void* w_f16, int c_out, const float* bias, const float* residual, float* out_f32,
                          void* out_f16, double* out_stats, int* err_flag, void* stream);
/* Reserved: returns 0.  (The `workspace` arguments of mi_conv2d_igemm_f16 are kept for ABI stability; pass NULL / 0.  A stream-K
 * schedule that used them was measured and removed: on a power-capped part an under-filled last wave costs nothing.) */
long long mi_conv2d_igemm_workspace_bytes(void);

/* Fused Block.forward (layers.py:131-145): GroupNorm -> (scale + 1, shift) -> SiLU -> Conv2d 3x3 in ONE kernel; the
 * normalised tensor never exists in HBM.  The swapped-operand 3x3 halo convolution (weights = M, 256 pixels = N) with the TMA
 * load of its activation halo replaced by a prologue: eight warps read the raw fp32 NHWC input (optionally the virtual
 * concat cat(src0, src1*scale1), Unet.py:445) straight from global memory, apply y = SiLU(x*A[b,c] + B[b,c]) (GroupNorm
 * mean/rstd from the producers' 16-channel block statistics stats0/stats1 = out_stats of the convs that wrote src0/src1,
 * affine, FiLM and skip scale folded into A, B) and write the fp16 operand directly in the 128B-swizzled layout tcgen05.mma
 * reads; zero padding is applied to the ACTIVATED tensor.  Epilogue as mi_conv2d_igemm_f16 (bias, fp32 residual, fp32/fp16
 * outputs [B][H][W][c_out] contiguous, out_stats).  Requirements: mi_conv3x3_gn_supported (H % 32 == 0, W % 8 == 0,
 * c0 % 64 == 0, c1 % 64 == 0, c_out % 128 == 0, (c0+c1)/groups % 16 == 0). */
int mi_conv3x3_gn_supported(int H, int W, int c0, int c1, int c_out, int groups);
int mi_conv3x3_gn_silu_f16(const float* src0, int c0, const float* src1, int c1, float scale1, int B, int H, int W,
                           int groups, const double* stats0, const double* stats1, const float* gamma,
                           const float* beta, const float* scale_shift, int scale_shift_ld, float eps,
                           const void* w_f16, int c_out, const float* bias, const float* residual, float* out_f32,
                           void* out_f16, double* out_stats, int* err_flag, void* stream);

/* Direct fp32 convolution for shapes outside the tensor-core path: the CrossEmbedLayer stem (layers.py:300, 3/6 input
 * channels, k = 3/7/15), final_conv (Unet.py:327, 3 output channels) and every conv of the tiny test config.
 *   in        [B][Hin][Win][ldi] fp32 (channel-contiguous, ldi % 4 == 0, channels >= c_in up to the next multiple of 4
 *             must be readable and finite)
 *   w_oihw    the reference's own (c_out, c_in, kh, kw) fp32 parameter, unpacked
 *   out       element (b,ho,wo,n) at b*out_sb + ho*out_sh + wo*out_sw + n*out_sc (so NHWC slices and NCHW both work)
 */
int mi_conv2d_direct_f32(const float* in, int B, int Hin, int Win, int c_in, int ldi, const float* w_oihw, int c_out,
                         int kh, int kw, int stride, int pad, const float* bias, const float* residual, float* out,
                         int Hout, int Wout, long long out_sb, long long out_sh, long long out_sw, long long out_sc,
                         void* stream);

/* ------------------------------------------------------------------------------------------------- normalisation
 * nn.GroupNorm statistics (layers.py:127,136): per (sample, group) sum / sum-of-squares of the virtual concatenation
 * cat(src0[.., C0], src1[.., C1] * scale1) (skip connection, Unet.py:445; pass src1 = NULL, C1 = 0 otherwise).
 * sums: [B][groups][2] double, MUST be zero on entry (accumulated with atomics).  src: fp32 or (in_is_f16) fp16.
 * Called with groups = C/16 it produces the same per-16-channel block statistics as mi_conv2d_igemm_f16's out_stats. */
int mi_gn_stats(const void* src0, int c0, const void* src1, int c1, float scale1, int in_is_f16, int B, int hw,
                int groups, double* sums, void* stream);
/* Block.forward (layers.py:136-144): SiLU( GroupNorm(x) * (scale + 1) + shift ) -> conv operand (fp16 or fp32).
 * src0/src1: fp32 or (in_is_f16) fp16.  Statistics: stats0_block = 0 -> stats0 is [B][groups][2] from mi_gn_stats over the
 * whole concat; stats0_block = k > 0 -> stats0 is [B][c0/k][2] and stats1 [B][c1/stats1_block][2]: per-source block sums
 * written by the producing conv epilogues (mi_conv2d_igemm_f16 out_stats, k = 16); src1's are scaled by scale1 here.
 * scale_shift: fp32, row b at scale_shift + b*scale_shift_ld holds [scale(C) | shift(C)] (time_mlp output,
 * layers.py:427-429; the rows of all ResnetBlocks live in one buffer, hence the row pitch) or NULL. */
int mi_gn_apply_silu(const void* src0, int c0, const void* src1, int c1, float scale1, int in_is_f16, int B, int hw,
                     int groups, const double* stats0, int stats0_block, const double* stats1, int stats1_block,
                     const float* gamma, const float* beta, const float* scale_shift, int scale_shift_ld, float eps,
                     void* out, int out_is_f16, void* stream);
/* Raw conv operands with the skip concat folded in; mode 0 plain copy/cast, 1 nearest x2 upsample (layers.py:513),
 * 2 four-phase split for the stride-2 Downsample conv (layers.py:319). out: fp16 or fp32. */
int mi_cast_act(const void* src0, int c0, const void* src1, int c1, float scale1, int in_is_f16, int B, int H, int W,
                int mode, void* out, int out_is_f16, void* stream);
/* Row LayerNorm over the last dim: layers.py:342 (LayerNorm, gamma + zero beta), layers.py:174-177 (ChanLayerNorm ==
 * per-pixel LN in NHWC), Unet.py:142,632 (nn.LayerNorm).  pre_gelu applies the exact-erf GELU of ChanFeedForward
 * (layers.py:158) to the input first; residual (fp32 [R][C]) is added after (layers.py:435,497-498). */
int mi_ln_rows(const float* in, long long rows, int C, const float* gamma, const float* beta, float eps, int pre_gelu,
               const float* residual, float* out_f32, void* out_f16, void* stream);

/* ------------------------------------------------------------------------------------------------- conditioning
 * out = act_out( act_in(in)[M][K] @ W[N][K]^T + bias + addend ) * out_scale, fp32 CUDA-core path for the conditioning
 * MLPs (Unet.py:101-161, :523-533, :613; layers.py:396-399,427) and non-tensor-core-shaped projections.
 * in_act/out_act: 0 none, 1 SiLU.  W is the reference's nn.Linear.weight as is. */
int mi_linear_f32(const float* in, int M, int K, const float* W, const float* bias, int N, int in_act, int out_act,
                  const float* addend, float* out_f32, void* out_f16, float out_scale, void* stream);
/* SinusoidalPosEmb.forward (layers.py:455-465); t: int64 [B]; out [B][dim] */
int mi_sinusoidal_posemb(const long long* t, int B, int dim, float* out, void* stream);
/* Unet._text_condition (Unet.py:578-610): truncate/zero-pad projected tokens to max_len rows, replace rows where
 * (text_mask & keep) is false by null_text_embed, write them at rows [row_off, row_off+max_len) of c_out [B][m][D],
 * mean-pool them into pooled [B][D].  mask: uint8 [B][L] or NULL; keep: uint8 [B]. */
int mi_text_tokens(const float* proj, int B, int L, int D, const uint8_t* mask, const uint8_t* keep,
                   const float* null_embed, int max_len, float* c_out, int m, int row_off, float* pooled,
                   void* stream);
/* copy [B][r][D] rows into c_out [B][m][D] at row_off (time tokens, Unet.py:534,629) */
int mi_place_rows(const float* src, int B, int r, int D, float* dst, int m, int row_off, void* stream);
/* where(keep[b], a[b], null) + addend   (Unet.py:619-626) */
int mi_select_rows(const float* a, const float* null_row, const uint8_t* keep, const float* addend, int B, int N,
                   float* out, void* stream);
/* torch.cat((x, lowres_cond_img), dim=1) (Unet.py:397) + NCHW -> NHWC with channels zero-padded to c_pad */
int mi_nchw_to_nhwc(const float* a, int ca, const float* b, int cb, int B, int hw, int c_pad, float* out,
                    void* stream);

/* Tensor-core operand of the CrossEmbedLayer stem (layers.py:294-305; kernels 3/7/15, stride 1, <= 8 input channels):
 * out[b][h][w][j*8 + c] = cat(a, b)[b][c][h][w + j - 7] (zero outside the row, j = 15 and c >= ca+cb are zero), fp16,
 * 128 values per pixel.  The three convs, zero-embedded in one 15x15 window, then run as ONE
 * mi_conv2d_igemm_f16(kh = 15, kw = 1, c_in = 128).  a / b: NCHW fp32 (x and lowres_cond_img, Unet.py:397). */
int mi_stem_unroll_f16(const float* a, int ca, const float* b, int cb, int B, int H, int W, void* out_f16,
                       void* stream);
/* out = x * sigmoid(x): the nn.SiLU in front of every ResnetBlock.time_mlp (layers.py:396-399), applied once per
 * step to the shared time embedding instead of once per block */
int mi_silu_f32(const float* in, long long n, float* out, void* stream);

/* Inter-stage image resize of the cascade: helpers.resize_image_to (helpers.py:138-164 -> resize_right.resize, called at
 * Imagen.py:482 between U-Nets).  Separable resampling of `planes` fp32 images [h_in][w_in] -> [h_out][w_out] with
 * per-output-coordinate tap tables: iy/wy [h_out][taps_y], ix/wx [w_out][taps_x] (source index after boundary handling,
 * normalised weight); rows are reduced first, then columns, then the optional clamp(lo, hi) (helpers.py:161-162).  The
 * tables encode the interpolation method (minimagen_b200/helpers.py builds resize_right's cubic / antialiased ones). */
int mi_resize_separable(const float* in, long long planes, int h_in, int w_in, float* out, int h_out, int w_out,
                        const int* iy, const float* wy, int taps_y, const int* ix, const float* wx, int taps_x,
                        int has_clamp, float lo, float hi, void* stream);

/* ------------------------------------------------------------------------------------------------- attention
 * Fused softmax attention, dim_head 64: CrossAttention.forward (layers.py:220-251) with kv_head_stride = 64, and the
 * multi-query Attention.forward (layers.py:52-104) with kv_head_stride = 0.  q must already carry the dim_head**-0.5
 * scale.  Key 0 is the learned null_kv [2][64] fp32 (layers.py:65-67,232-235); key_mask: uint8 [B][m] or NULL
 * (masked_fill(~mask, -FLT_MAX), layers.py:92-95,242-245).  q/out: [B][n][ld] with head h at column h*64.
 * workspace (optional, 128-byte aligned, size from mi_attention_workspace_bytes): lends the tcgen05 kernels room for the
 * null-prepended padded K, the transposed V and the key-validity bits (null key, key_mask, padding); it is used when
 * n % 128 == 0, m >= 128 and q is batch-contiguous (q_bs == n*ldq) -- S = QK^T and O = PV then run as tcgen05.mma with TMEM
 * accumulators in ONE sweep over the keys (lazily rescaled reference maximum), the softmax in between reads S from TMEM and
 * hands P to the second GEMM through tensor memory; two query tiles per CTA when n % 256 == 0.  Otherwise (or with workspace
 * NULL) a mma.sync kernel runs. */
long long mi_attention_workspace_bytes(int B, int heads, int kv_head_stride, int m);
int mi_attention_fwd(const void* q_f16, long long q_bs, int ldq, const void* k_f16, const void* v_f16, long long kv_bs,
                     int ldkv, int kv_head_stride, const float* null_kv, const uint8_t* key_mask, int B, int heads,
                     int n, int m, void* out_f16, long long o_bs, int ldo, void* workspace, long long workspace_bytes,
                     void* stream);

/* ------------------------------------------------------------------------------------------------- DDPM step
 * Imagen._p_mean_variance / _p_sample after the U-Net (Imagen.py:307-326, :361-370).  Images are NCHW fp32 [B][n].
 * Schedule tables are GaussianDiffusion's fp32 buffers (diffusion_model.py:42-66); t is int64 [B]. */
int mi_step_x0(const float* x_t, const float* eps_cond, const float* eps_null, float cond_scale, const long long* t,
               const float* sqrt_recip_alphas_cumprod, const float* sqrt_recipm1_alphas_cumprod, int B, int n,
               float* x0, void* stream);
/* s[b] = max( lerp(sorted|x0[b]|[rank_lo], sorted|x0[b]|[rank_hi], weight), min_s ) -- exact (radix select) */
int mi_step_quantile(const float* x0, int B, int n, int rank_lo, int rank_hi, float weight, float min_s, float* s,
                     void* stream);
int mi_step_posterior(const float* x0, const float* x_t, const float* noise, const float* s, const long long* t,
                      const float* posterior_mean_coef1, const float* posterior_mean_coef2, const float* sigma, int B,
                      int n, float* out, void* stream);
/* The three calls above as ONE kernel -- everything Imagen._p_sample does after the U-Net (Imagen.py:307-326, :361-370;
 * Unet.py:506 for the guidance combine): an 8-CTA cluster per image computes x0 into registers, selects the dynamic-
 * threshold order statistics there, and writes x_{t-1}; the x0 tensor never exists in memory.  `out` may be `x_t` (in-place
 * update of the sampling state).  s_out: optional [B] (the thresholds).  Images with more than 196 608 values (3 x 1024 x
 * 1024) exceed the register-resident select: they take the three-kernel form through the caller's scratch
 * x0_workspace (mi_step_epilogue_workspace_floats(B, n) floats; 0 = not needed) and then s_out is required. */
long long mi_step_epilogue_workspace_floats(int B, int n);
int mi_step_epilogue(const float* x_t, const float* eps_cond, const float* eps_null, float cond_scale, const long long* t,
                     const float* sqrt_recip_alphas_cumprod, const float* sqrt_recipm1_alphas_cumprod,
                     const float* posterior_mean_coef1, const float* posterior_mean_coef2, const float* sigma,
                     const float* noise, int B, int n, int rank_lo, int rank_hi, float weight, float min_s, float* out,
                     float* s_out, float* x0_workspace, void* stream);
/* t[b] <- max(t[b] - 1, 0): the next iteration's timestep of Imagen._p_sample_loop (Imagen.py:398-415 walks the list of
 * diffusion_model.py:81-87), advanced on the device so that a captured step can be replayed back to back */
int mi_step_advance_t(long long* t, int B, void* stream);
/* clamp_(-1,1) and (x+1)*0.5 (Imagen.py:418-419) */
int mi_step_finalize(const float* x, long long n, int unnormalize, float* out, void* stream);
/* GaussianDiffusion.q_sample (diffusion_model.py:127-147) followed by v*post_scale + post_shift */
int mi_q_sample(const float* x0, const float* noise, const long long* t, const float* sqrt_alphas_cumprod,
                const float* sqrt_one_minus_alphas_cumprod, int B, int n, float post_scale, float post_shift,
                float* out, void* stream);
/* Inpainting (RePaint resampling), one replay = step -> mi_inpaint_blend -> mi_inpaint_advance.  x [B][C][H][W] fp32 is
 * updated in place; known (the normalised image to keep), z_known and z_renoise have its shape; mask uint8 [B][mask_h][mask_w]
 * (nonzero = known pixel) is sampled nearest-neighbour: m[b][i][j] = mask[b][i*mask_h/H][j*mask_w/W].  t int64 [B], u int32 [1]
 * (the resample round at t), U resample rounds per timestep (1 at t == 0); sqrt_alphas[t] = sqrt(1 - beta_t),
 * sqrt_betas[t] = sqrt(beta_t).  With U_t = (t > 0 ? U : 1):
 *   prime:            x = m ? sqrt_acp[t] known + sqrt_1macp[t] z_known : x                 (before the first step)
 *   u < U_t - 1:      x = m ? sqrt_acp[t] known + sqrt_1macp[t] z_known : sqrt_alphas[t] x + sqrt_betas[t] z_renoise
 *   else, t > 0:      x = m ? sqrt_acp[t-1] known + sqrt_1macp[t-1] z_known : x
 *   else (t == 0):    x = m ? known : x
 * Products and sums are un-fused, in torch's order (a*x + b*z).  Pointers must be non-NULL, sizes positive, U >= 1. */
int mi_inpaint_blend(float* x, const float* known, const unsigned char* mask, int mask_h, int mask_w, const float* z_known,
                     const float* z_renoise, const long long* t, const int* u, int U, int prime,
                     const float* sqrt_alphas_cumprod, const float* sqrt_one_minus_alphas_cumprod, const float* sqrt_alphas,
                     const float* sqrt_betas, int B, int C, int H, int W, void* stream);
/* After mi_inpaint_blend: if that step renoised (u < U_t - 1, decided on t[0]) u += 1, else u = 0 and t[b] = max(t[b] - 1, 0).
 * A launch of its own: the blend's CTAs all read t and u. */
int mi_inpaint_advance(long long* t, int* u, int U, int B, void* stream);

/* ------------------------------------------------------------------------------------------------- training (backward)
 * The training side of the same path: Imagen.forward / _p_losses (Imagen.py:512-650) back-propagate through Unet.forward
 * (train.py:103 -> training.py:368).  minimagen_b200/autograd.py wraps every forward entry point above in a
 * torch.autograd.Function whose backward calls the entry points below (or, for the data gradient of tensor-core-shaped
 * convolutions, mi_conv2d_igemm_f16 itself on flipped / transposed packed weights).  All fp32, NHWC. */

/* C[z] (+)= alpha * A[z] x B[z] with explicit element strides: A(m,k) at A + z1*a_b1 + z2*a_b2 + m*a_sm + k*a_sk,
 * B(k,n) at B + ... + k*b_sk + n*b_sn, C(m,n) at C + ... + m*c_sm + n*c_sn; batch z = z1*Z2 + z2.
 * nn.Linear backward (dX = dY W, dW = dY^T X) and the fp32 attention of the training path (S = q k^T, dP = dO v^T,
 * dq = dS k, dk = dS^T q, dv = P^T dO; layers.py:79-99, :239-248). */
int mi_gemm_f32(const float* A, const float* B, float* C, int M, int N, int K, long long a_sm, long long a_sk,
                long long b_sk, long long b_sn, long long c_sm, long long c_sn, int Z1, int Z2, long long a_b1,
                long long a_b2, long long b_b1, long long b_b2, long long c_b1, long long c_b2, float alpha,
                int accumulate, void* stream);
/* out[n] (+)= sum_m x[m][n]  (bias gradients) */
int mi_colsum_f32(const float* x, long long M, int N, float* out, int accumulate, void* stream);
/* dL/dx of nn.Conv2d(c_in, c_out, (kh, kw), stride, pad): dy [B][Hout][Wout][c_out], w OIHW, dx [B][Hin][Win][c_in] */
int mi_conv2d_dgrad_f32(const float* dy, int B, int Hout, int Wout, int c_out, const float* w_oihw, int c_in, int kh, int kw,
                        int stride, int pad, float* dx, int Hin, int Win, void* stream);
/* dL/dW of the same conv: x [B][Hin][Win][c_in], dy [B][Hout][Wout][c_out] -> dw OIHW (overwritten) */
int mi_conv2d_wgrad_f32(const float* dy, const float* x, int B, int Hin, int Win, int c_in, int Hout, int Wout, int c_out,
                        int kh, int kw, int stride, int pad, float* dw, void* stream);
/* The same weight gradient on the tensor cores, for k x k (k = 1, 3) stride-1 'same' convs and for the 4 x 4 stride-2 pad-1
 * Downsample (layers.py:481-484): dy [B][Hout][Wout][c_out] and x [B][stride*Hout][stride*Wout][c_in] are fp16 NHWC
 * (mi_cast_act), Hout % 8 == Wout % 8 == 0, c_in % 64 == 0, c_out % 128 == 0; fp32 accumulation over the pixels, dw OIHW
 * fp32 (overwritten).  The pixel axis is split over CTAs; their partial tiles go through `workspace`
 * (mi_conv2d_wgrad_f16_workspace_bytes, 16-byte aligned) and are summed by a second kernel.  Replaces torch's conv
 * weight-gradient in the backward of layers.py:145 / 203-211 / 481-484. */
int mi_conv2d_wgrad_f16_supported(int Hout, int Wout, int c_in, int c_out, int kh, int kw, int stride);
long long mi_conv2d_wgrad_f16_workspace_bytes(int B, int Hout, int Wout, int c_in, int c_out, int kh, int kw, int stride);
int mi_conv2d_wgrad_f16(const void* dy_f16, const void* x_f16, int B, int Hout, int Wout, int c_in, int c_out, int kh, int kw,
                        int stride, float* dw, float* workspace, long long workspace_bytes, void* stream);
/* Backward of mi_gn_apply_silu over ONE fp32 source x [B][hw][C] (sums = mi_gn_stats group sums [B][groups][2]):
 * dx; dgamma / dbeta ACCUMULATED into (caller zeroes or carries .grad); d_scale_shift [B][.. ld ..] = [d scale(C) | d shift(C)]
 * or NULL; workspace: (2*B*C + 4*B*groups) floats. */
int mi_gn_silu_bwd(const float* x, const float* dy, const double* sums, int B, int hw, int C, int groups,
                   const float* gamma, const float* beta, const float* scale_shift, int scale_shift_ld, float eps,
                   float* dx, float* dgamma, float* dbeta, float* d_scale_shift, int d_scale_shift_ld, float* workspace,
                   void* stream);
/* Backward of mi_ln_rows (without its residual, which passes the gradient through): dx [R][C]; dgamma / dbeta accumulated
 * (either may be NULL). */
int mi_ln_rows_bwd(const float* in, const float* dy, long long rows, int C, const float* gamma, float eps, int pre_gelu,
                   float* dx, float* dgamma, float* dbeta, void* stream);
/* in-place row softmax of s [R][L], and its backward dS = P * (dP - sum_j P dP) written over dP */
int mi_softmax_rows(float* s, long long R, int L, void* stream);
int mi_softmax_rows_bwd(const float* P, float* dP, long long R, int L, void* stream);
/* backward of nn.Upsample(scale_factor=2, 'nearest'): dy [B][2H][2W][C] -> dx [B][H][W][C] */
int mi_upsample2x_bwd(const float* dy, int B, int H, int W, int C, float* dx, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MINIMAGEN_B200_H_ */
