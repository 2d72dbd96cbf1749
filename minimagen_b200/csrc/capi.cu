// C ABI (include/minimagen_b200.h) over the kernel launchers.  No torch, no allocation, no CPU fallback.
#include "../../include/minimagen_b200.h"

#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <string>

#include "conv_tc.cuh"
#include "kernels.cuh"

namespace {

thread_local char g_err[256] = "ok";

int fail(int code, const char* what) {
    snprintf(g_err, sizeof(g_err), "%s (code %d)", what, code);
    return code;
}
int check(int rc, const char* fn) {
    if (rc == 0) return 0;
    if (rc == -1) return fail(rc, (std::string(fn) + ": unsupported shape / alignment").c_str());
    if (rc == -2) {
        cudaError_t e = cudaGetLastError();
        return fail(rc, (std::string(fn) + ": kernel launch failed: " + cudaGetErrorString(e)).c_str());
    }
    return fail(rc, (std::string(fn) + ": error").c_str());
}
inline cudaStream_t S(void* s) { return reinterpret_cast<cudaStream_t>(s); }

}  // namespace

namespace mi {
static bool g_pdl = false;
bool pdl_enabled() { return g_pdl; }
}  // namespace mi

extern "C" {

int mi_abi_version(void) { return MI_ABI_VERSION; }
int mi_set_launch_mode(int programmatic_dependent_launch) {
    mi::g_pdl = programmatic_dependent_launch != 0;
    return 0;
}
const char* mi_last_error(void) { return g_err; }

int mi_device_ok(void) {
    int dev = 0, major = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 0;
    if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) return 0;
    return major == 10;
}

int mi_pack_conv_weight_dgrad_f16(const float* w, int c_out, int c_in, int kh, int kw, void* out, void* stream) {
    return check(mi::pack_conv_weight_dgrad(w, c_out, c_in, kh, kw, (__half*)out, S(stream)), "mi_pack_conv_weight_dgrad_f16");
}
int mi_pack_conv_weight_f16(const float* w, int c_out, int c_in, int kh, int kw, float scale, void* out, void* stream) {
    return check(mi::pack_conv_weight(w, c_out, c_in, kh, kw, scale, (__half*)out, S(stream)), "mi_pack_conv_weight_f16");
}

int mi_conv2d_igemm_supported(int H, int W, int c_in, int c_out) { return mi::conv_tc_supported(H, W, c_in, c_out) ? 1 : 0; }

static int igemm_common(const void* act, int B, int H, int W, int lda, int c_off, int c_in, const void* act2, int lda2,
                        int c_off2, int c_in1, const void* w, int c_out, int kh, int kw, int mode, const float* bias,
                        const float* residual, float* out_f32, void* out_f16, double* out_stats, long long out_sb,
                        long long out_sh, long long out_sw, long long out_sc, int n_valid, int block_n, int* err_flag,
                        void* workspace, long long workspace_bytes, const void* x_act, int ldx, int x_off, int x_cin,
                        const void* x_act2, int ldx2, int x_off2, int x_cin1, void* stream) {
    mi::ConvTcProblem p{};
    p.x_act = x_act; p.x_lda = ldx; p.x_chan_off = x_off; p.Cx = x_cin;
    p.x_act2 = x_act2; p.x_lda2 = ldx2; p.x_chan_off2 = x_off2; p.Cx1 = x_cin1;
    if (x_act && !(mode == 0 && kh == 3 && kw == 3)) return fail(-9, "mi_conv3x3_res1x1_f16: the folded 1x1 operand needs a 3x3 stride-1 conv");
    (void)workspace; (void)workspace_bytes;       // reserved (no kernel needs scratch any more): pass NULL / 0
    p.act = act; p.B = B; p.H = H; p.W = W; p.lda = lda; p.a_channels = lda; p.a_chan_off = c_off; p.Cin = c_in;
    p.wpacked = w; p.Cout = c_out;
    p.act2 = act2; p.lda2 = lda2; p.a_chan_off2 = c_off2; p.Cin1 = c_in1; p.stats = out_stats;
    if (out_stats && (out_sc > 1 || (c_out % 32) != 0)) return fail(-8, "mi_conv2d_igemm_f16: out_stats needs channel-contiguous output and c_out % 32 == 0");
    if (out_stats && ((long long)H * W) % 32 != 0)
        return fail(-8, "mi_conv2d_igemm_f16: out_stats needs H*W % 32 == 0 (a warp's 32 output rows must belong to one image)");
    p.out_f32 = out_f32; p.out_f16 = (__half*)out_f16; p.bias = bias; p.residual = residual;
    p.out_sb = out_sb; p.out_sh = out_sh; p.out_sw = out_sw; p.out_sc = out_sc; p.n_valid = n_valid;
    p.block_n_hint = block_n; p.err_flag = err_flag;
    if (mode == 0) {
        if (!(kh & 1) || !(kw & 1) || kh * kw > mi::kConvMaxTaps) return fail(-4, "mi_conv2d_igemm_f16: mode 0 needs odd kh,kw with kh*kw <= 16");
        p.phases = 1; p.num_taps = kh * kw;
        for (int r = 0; r < kh; ++r)
            for (int s = 0; s < kw; ++s) {
                const int t = r * kw + s;
                p.dh[t] = (int8_t)(r - kh / 2); p.dw[t] = (int8_t)(s - kw / 2); p.ph[t] = 0;
            }
    } else if (mode == 1) {
        if (kh != 4 || kw != 4) return fail(-4, "mi_conv2d_igemm_f16: mode 1 is the 4x4 stride-2 pad-1 conv");
        p.phases = 4; p.num_taps = 16;
        for (int r = 0; r < 4; ++r)
            for (int s = 0; s < 4; ++s) {
                // input row 2*ho + r - 1 lives in phase row (r-1)&1 at phase-grid row ho + floor((r-1)/2)
                const int t = r * 4 + s, rr = r - 1, ss = s - 1;
                p.dh[t] = (int8_t)(rr < 0 ? -1 : (rr >> 1)); p.dw[t] = (int8_t)(ss < 0 ? -1 : (ss >> 1));
                p.ph[t] = (int8_t)((rr & 1) * 2 + (ss & 1));
            }
    } else if (mode == 6) {
        // Downsample read in place: tap (r, s) of output pixel (ho, wo) is input pixel (2*ho + r - 1, 2*wo + s - 1)
        if (kh != 4 || kw != 4) return fail(-4, "mi_conv2d_igemm_f16: mode 6 is the 4x4 stride-2 pad-1 conv");
        if (act2) return fail(-4, "mi_conv2d_igemm_f16: mode 6 takes one activation tensor");
        p.phases = 1; p.num_taps = 16; p.in_stride = 2;
        for (int r = 0; r < 4; ++r)
            for (int s = 0; s < 4; ++s) {
                const int t = r * 4 + s;
                p.dh[t] = (int8_t)(r - 1); p.dw[t] = (int8_t)(s - 1); p.ph[t] = 0;
            }
    } else if (mode >= 2 && mode <= 5) {
        // sub-pixel phase (a, b) = ((mode-2) >> 1, (mode-2) & 1) of "nearest x2 upsample, then 3x3 conv": output pixel
        // (2y+a, 2x+b) only sees the low-res pixels (y + a-1 + r, x + b-1 + s), r,s in {0,1}, with 3x3 weights pre-summed
        if (kh != 2 || kw != 2) return fail(-4, "mi_conv2d_igemm_f16: modes 2..5 take the 2x2 phase kernel");
        const int a = (mode - 2) >> 1, b = (mode - 2) & 1;
        p.phases = 1; p.num_taps = 4;
        for (int r = 0; r < 2; ++r)
            for (int s = 0; s < 2; ++s) {
                const int t = r * 2 + s;
                p.dh[t] = (int8_t)(a - 1 + r); p.dw[t] = (int8_t)(b - 1 + s); p.ph[t] = 0;
            }
    } else {
        return fail(-4, "mi_conv2d_igemm_f16: unknown mode");
    }
    if (out_sc <= 1 && ((out_sw % 4) || (out_sh % 4) || (out_sb % 4)))
        return fail(-8, "mi_conv2d_igemm_f16: channel-contiguous output strides must be multiples of 4 elements");
    if (out_sc > 1 && residual) return fail(-8, "mi_conv2d_igemm_f16: residual needs channel-contiguous output");
    // kernel selection (measured on B200, profiles/r01_conv_tc_selftest_v9.log): 3x3 layers run fastest on the swapped-operand
    // halo kernel (needs C_out % 128 == 0, H % 32 == 0), C_out = 128 / 16 layers it cannot take on the pixel-major halo
    // kernel, everything else on the CTA-pair kernel (all chosen inside conv_tc_launch)
    p.halo = (mode == 0 && kh == 3 && kw == 3) ? 1 : ((mode == 0 && kh == 15 && kw == 1) ? 3 : 0);   // 3: 15-tap vertical (stem)
    if (mode >= 2 && mode <= 5 && !getenv("MI_SUBPIX_PAIR")) p.halo = 4;   // sub-pixel phase on the swapped-operand kernel (32 x 8 tiles)
    const int rc = mi::conv_tc_launch(p, S(stream));
    if (rc != 0) return fail(rc, mi::conv_tc_strerror(rc));
    return 0;
}

int mi_conv2d_igemm_f16(const void* act, int B, int H, int W, int lda, int c_off, int c_in, const void* act2, int lda2,
                        int c_off2, int c_in1, const void* w, int c_out, int kh, int kw, int mode, const float* bias,
                        const float* residual, float* out_f32, void* out_f16, double* out_stats, long long out_sb,
                        long long out_sh, long long out_sw, long long out_sc, int n_valid, int block_n, int* err_flag,
                        void* workspace, long long workspace_bytes, void* stream) {
    return igemm_common(act, B, H, W, lda, c_off, c_in, act2, lda2, c_off2, c_in1, w, c_out, kh, kw, mode, bias, residual,
                        out_f32, out_f16, out_stats, out_sb, out_sh, out_sw, out_sc, n_valid, block_n, err_flag, workspace,
                        workspace_bytes, nullptr, 0, 0, 0, nullptr, 0, 0, 0, stream);
}

int mi_conv3x3_res1x1_supported(int H, int W, int c_in, int c_out, int x_cin) {
    const bool t16 = W == 16 && H % 16 == 0, t32 = !t16 && H % 32 == 0 && W % 8 == 0;
    return (t16 || t32) && c_in > 0 && c_in % 64 == 0 && x_cin > 0 && x_cin % 64 == 0 && c_out % 128 == 0;
}

int mi_conv3x3_res1x1_f16(const void* act, int B, int H, int W, int lda, int c_in, const void* act2, int lda2, int c_in1,
                          const void* x_act, int ldx, int x_cin, const void* x_act2, int ldx2, int x_cin1, const void* w,
                          int c_out, const float* bias, const float* residual, float* out_f32, void* out_f16,
                          double* out_stats, int* err_flag, void* stream) {
    if (!mi_conv3x3_res1x1_supported(H, W, c_in, c_out, x_cin))
        return fail(-9, "mi_conv3x3_res1x1_f16: unsupported geometry (see mi_conv3x3_res1x1_supported)");
    return igemm_common(act, B, H, W, lda, 0, c_in, act2, lda2, 0, c_in1, w, c_out, 3, 3, 0, bias, residual, out_f32, out_f16,
                        out_stats, (long long)H * W * c_out, (long long)W * c_out, c_out, 1, 0, 0, err_flag, nullptr, 0, x_act,
                        ldx, 0, x_cin, x_act2, ldx2, 0, x_cin1, stream);
}

long long mi_conv2d_igemm_workspace_bytes(void) { return 0; }

int mi_conv3x3_gn_supported(int H, int W, int c0, int c1, int c_out, int groups) {
    return mi::conv_gn_supported(H, W, c0, c1, c_out, groups) ? 1 : 0;
}

int mi_conv3x3_gn_silu_f16(const float* src0, int c0, const float* src1, int c1, float scale1, int B, int H, int W,
                           int groups, const double* stats0, const double* stats1, const float* gamma,
                           const float* beta, const float* scale_shift, int scale_shift_ld, float eps, const void* w,
                           int c_out, const float* bias, const float* residual, float* out_f32, void* out_f16,
                           double* out_stats, int* err_flag, void* stream) {
    mi::ConvGnProblem p{};
    p.src0 = src0; p.C0 = c0; p.src1 = src1; p.C1 = c1; p.scale1 = scale1; p.B = B; p.H = H; p.W = W; p.groups = groups;
    p.stats0 = stats0; p.stats1 = stats1; p.gamma = gamma; p.beta = beta; p.scale_shift = scale_shift;
    p.ss_ld = scale_shift_ld; p.eps = eps; p.wpacked = w; p.Cout = c_out; p.bias = bias; p.residual = residual;
    p.out_f32 = out_f32; p.out_f16 = (__half*)out_f16; p.out_stats = out_stats; p.err_flag = err_flag;
    if (scale_shift && scale_shift_ld < 2 * (c0 + c1)) return fail(-8, "mi_conv3x3_gn_silu_f16: scale_shift_ld < 2*C");
    // C_out % 256 == 0: the CTA-pair kernel (half the prologue per tensor FLOP); otherwise the single-CTA kernel
    const bool pair = mi::conv_gn_pair_supported(H, W, c0, c1, c_out, groups) && !getenv("MI_GN_NO_PAIR");
    const int rc = pair ? mi::conv_gn_pair_launch(p, S(stream)) : mi::conv_gn_launch(p, S(stream));
    if (rc != 0) return fail(rc, rc == -3 ? "mi_conv3x3_gn_silu_f16: unsupported geometry (see mi_conv3x3_gn_supported)"
                                          : mi::conv_tc_strerror(rc));
    return 0;
}

int mi_conv2d_direct_f32(const float* in, int B, int Hin, int Win, int c_in, int ldi, const float* w, int c_out, int kh,
                         int kw, int stride, int pad, const float* bias, const float* residual, float* out, int Hout,
                         int Wout, long long out_sb, long long out_sh, long long out_sw, long long out_sc,
                         void* stream) {
    return check(mi::conv_direct_f32(in, B, Hin, Win, c_in, ldi, w, c_out, kh, kw, stride, pad, bias, residual, out,
                                     Hout, Wout, out_sb, out_sh, out_sw, out_sc, S(stream)),
                 "mi_conv2d_direct_f32");
}

int mi_gn_stats(const void* src0, int c0, const void* src1, int c1, float scale1, int in_is_f16, int B, int hw,
                int groups, double* sums, void* stream) {
    return check(mi::gn_stats(src0, c0, src1, c1, scale1, in_is_f16, B, hw, groups, sums, S(stream)), "mi_gn_stats");
}
int mi_gn_apply_silu(const void* src0, int c0, const void* src1, int c1, float scale1, int in_is_f16, int B, int hw,
                     int groups, const double* stats0, int stats0_block, const double* stats1, int stats1_block,
                     const float* gamma, const float* beta, const float* scale_shift, int scale_shift_ld, float eps,
                     void* out, int out_is_f16, void* stream) {
    return check(mi::gn_apply_silu(src0, c0, src1, c1, scale1, in_is_f16, B, hw, groups, stats0, stats0_block, stats1,
                                   stats1_block, gamma, beta, scale_shift, scale_shift_ld, eps, out, out_is_f16,
                                   S(stream)),
                 "mi_gn_apply_silu");
}
int mi_cast_act(const void* src0, int c0, const void* src1, int c1, float scale1, int in_is_f16, int B, int H, int W,
                int mode, void* out, int out_is_f16, void* stream) {
    return check(mi::cast_act(src0, c0, src1, c1, scale1, in_is_f16, B, H, W, mode, out, out_is_f16, S(stream)),
                 "mi_cast_act");
}
int mi_ln_rows(const float* in, long long rows, int C, const float* gamma, const float* beta, float eps, int pre_gelu,
               const float* residual, float* out_f32, void* out_f16, void* stream) {
    return check(mi::ln_rows(in, rows, C, gamma, beta, eps, pre_gelu, residual, out_f32, (__half*)out_f16, S(stream)),
                 "mi_ln_rows");
}
int mi_linear_f32(const float* in, int M, int K, const float* W, const float* bias, int N, int in_act, int out_act,
                  const float* addend, float* out_f32, void* out_f16, float out_scale, void* stream) {
    return check(mi::linear_f32(in, M, K, W, bias, N, in_act, out_act, addend, out_f32, (__half*)out_f16, out_scale,
                                S(stream)),
                 "mi_linear_f32");
}
int mi_sinusoidal_posemb(const long long* t, int B, int dim, float* out, void* stream) {
    return check(mi::posemb(t, B, dim, out, S(stream)), "mi_sinusoidal_posemb");
}
int mi_text_tokens(const float* proj, int B, int L, int D, const uint8_t* mask, const uint8_t* keep,
                   const float* null_embed, int max_len, float* c_out, int m, int row_off, float* pooled, void* stream) {
    return check(mi::text_tokens(proj, B, L, D, mask, keep, null_embed, max_len, c_out, m, row_off, pooled, S(stream)),
                 "mi_text_tokens");
}
int mi_place_rows(const float* src, int B, int r, int D, float* dst, int m, int row_off, void* stream) {
    return check(mi::place_rows(src, B, r, D, dst, m, row_off, S(stream)), "mi_place_rows");
}
int mi_select_rows(const float* a, const float* null_row, const uint8_t* keep, const float* addend, int B, int N,
                   float* out, void* stream) {
    return check(mi::select_rows(a, null_row, keep, addend, B, N, out, S(stream)), "mi_select_rows");
}
int mi_nchw_to_nhwc(const float* a, int ca, const float* b, int cb, int B, int hw, int c_pad, float* out, void* stream) {
    return check(mi::nchw_to_nhwc(a, ca, b, cb, B, hw, c_pad, out, S(stream)), "mi_nchw_to_nhwc");
}
int mi_stem_unroll_f16(const float* a, int ca, const float* b, int cb, int B, int H, int W, void* out, void* stream) {
    return check(mi::stem_unroll(a, ca, b, cb, B, H, W, (__half*)out, S(stream)), "mi_stem_unroll_f16");
}
int mi_resize_separable(const float* in, long long planes, int h_in, int w_in, float* out, int h_out, int w_out,
                        const int* iy, const float* wy, int taps_y, const int* ix, const float* wx, int taps_x,
                        int has_clamp, float lo, float hi, void* stream) {
    return check(mi::resize_sep(in, planes, h_in, w_in, out, h_out, w_out, iy, wy, taps_y, ix, wx, taps_x, has_clamp, lo, hi,
                                S(stream)),
                 "mi_resize_separable");
}
int mi_silu_f32(const float* in, long long n, float* out, void* stream) {
    return check(mi::silu_f32(in, n, out, S(stream)), "mi_silu_f32");
}
long long mi_attention_workspace_bytes(int B, int heads, int kv_head_stride, int m) {
    return mi::attention_tc_workspace_bytes(B, heads, kv_head_stride, m);
}
int mi_attention_fwd(const void* q, long long q_bs, int ldq, const void* k, const void* v, long long kv_bs, int ldkv,
                     int kv_head_stride, const float* null_kv, const uint8_t* key_mask, int B, int heads, int n, int m,
                     void* out, long long o_bs, int ldo, void* workspace, long long workspace_bytes, void* stream) {
    // tcgen05 path (key masks included) when the shape allows and the caller lends the operand workspace; mma.sync kernel otherwise
    // (short key sequences -- one 128-key block -- stay on the mma.sync kernel: 19 us vs 33 us at n = 256, m = 59)
    if (workspace && m >= 128 && mi::attention_tc_supported(n, ldq, ldo, q_bs, key_mask) &&
        workspace_bytes >= mi::attention_tc_workspace_bytes(B, heads, kv_head_stride, m))
        return check(mi::attention_tc_fwd((const __half*)q, q_bs, ldq, (const __half*)k, (const __half*)v, kv_bs, ldkv,
                                          kv_head_stride, null_kv, key_mask, B, heads, n, m, (__half*)out, o_bs, ldo, workspace,
                                          workspace_bytes, nullptr, S(stream)),
                     "mi_attention_fwd (tcgen05)");
    return check(mi::attention_fwd((const __half*)q, q_bs, ldq, (const __half*)k, (const __half*)v, kv_bs, ldkv,
                                   kv_head_stride, null_kv, key_mask, B, heads, n, m, (__half*)out, o_bs, ldo, S(stream)),
                 "mi_attention_fwd");
}
int mi_step_x0(const float* x_t, const float* eps_cond, const float* eps_null, float cond_scale, const long long* t,
               const float* tab_a, const float* tab_b, int B, int n, float* x0, void* stream) {
    return check(mi::step_x0(x_t, eps_cond, eps_null, cond_scale, t, tab_a, tab_b, B, n, x0, S(stream)), "mi_step_x0");
}
int mi_step_quantile(const float* x0, int B, int n, int rank_lo, int rank_hi, float weight, float min_s, float* s,
                     void* stream) {
    return check(mi::step_quantile(x0, B, n, rank_lo, rank_hi, weight, min_s, s, S(stream)), "mi_step_quantile");
}
int mi_step_posterior(const float* x0, const float* x_t, const float* noise, const float* s, const long long* t,
                      const float* c1, const float* c2, const float* sigma, int B, int n, float* out, void* stream) {
    return check(mi::step_posterior(x0, x_t, noise, s, t, c1, c2, sigma, B, n, out, S(stream)), "mi_step_posterior");
}
long long mi_step_epilogue_workspace_floats(int B, int n) {
    return mi::step_epilogue_fused_ok(n) ? 0 : (long long)B * n;
}
int mi_step_epilogue(const float* x_t, const float* eps_cond, const float* eps_null, float cond_scale, const long long* t,
                     const float* tab_a, const float* tab_b, const float* c1, const float* c2, const float* sigma,
                     const float* noise, int B, int n, int rank_lo, int rank_hi, float weight, float min_s, float* out,
                     float* s_out, float* x0_workspace, void* stream) {
    return check(mi::step_epilogue(x_t, eps_cond, eps_null, cond_scale, t, tab_a, tab_b, c1, c2, sigma, noise, B, n, rank_lo,
                                   rank_hi, weight, min_s, out, s_out, x0_workspace, S(stream)),
                 "mi_step_epilogue");
}
int mi_step_advance_t(long long* t, int B, void* stream) {
    return check(mi::step_advance_t(t, B, S(stream)), "mi_step_advance_t");
}
int mi_step_finalize(const float* x, long long n, int unnormalize, float* out, void* stream) {
    return check(mi::step_finalize(x, n, unnormalize, out, S(stream)), "mi_step_finalize");
}
int mi_q_sample(const float* x0, const float* noise, const long long* t, const float* tab_a, const float* tab_b, int B,
                int n, float post_scale, float post_shift, float* out, void* stream) {
    return check(mi::q_sample(x0, noise, t, tab_a, tab_b, B, n, post_scale, post_shift, out, S(stream)), "mi_q_sample");
}
int mi_inpaint_blend(float* x, const float* known, const unsigned char* mask, int mask_h, int mask_w, const float* z_known,
                     const float* z_renoise, const long long* t, const int* u, int U, int prime,
                     const float* sqrt_alphas_cumprod, const float* sqrt_one_minus_alphas_cumprod, const float* sqrt_alphas,
                     const float* sqrt_betas, int B, int C, int H, int W, void* stream) {
    return check(mi::inpaint_blend(x, known, mask, mask_h, mask_w, z_known, z_renoise, t, u, U, prime, sqrt_alphas_cumprod,
                                   sqrt_one_minus_alphas_cumprod, sqrt_alphas, sqrt_betas, B, C, H, W, S(stream)),
                 "mi_inpaint_blend");
}
int mi_inpaint_advance(long long* t, int* u, int U, int B, void* stream) {
    return check(mi::inpaint_advance(t, u, U, B, S(stream)), "mi_inpaint_advance");
}

int mi_gemm_f32(const float* A, const float* B, float* C, int M, int N, int K, long long a_sm, long long a_sk,
                long long b_sk, long long b_sn, long long c_sm, long long c_sn, int Z1, int Z2, long long a_b1,
                long long a_b2, long long b_b1, long long b_b2, long long c_b1, long long c_b2, float alpha,
                int accumulate, void* stream) {
    return check(mi::gemm_f32(A, B, C, M, N, K, a_sm, a_sk, b_sk, b_sn, c_sm, c_sn, Z1, Z2, a_b1, a_b2, b_b1, b_b2, c_b1, c_b2,
                              alpha, accumulate, S(stream)),
                 "mi_gemm_f32");
}
int mi_colsum_f32(const float* x, long long M, int N, float* out, int accumulate, void* stream) {
    return check(mi::colsum_f32(x, M, N, out, accumulate, S(stream)), "mi_colsum_f32");
}
int mi_conv2d_dgrad_f32(const float* dy, int B, int Hout, int Wout, int c_out, const float* w, int c_in, int kh, int kw,
                        int stride, int pad, float* dx, int Hin, int Win, void* stream) {
    return check(mi::conv2d_dgrad_f32(dy, B, Hout, Wout, c_out, w, c_in, kh, kw, stride, pad, dx, Hin, Win, S(stream)),
                 "mi_conv2d_dgrad_f32");
}
int mi_conv2d_wgrad_f32(const float* dy, const float* x, int B, int Hin, int Win, int c_in, int Hout, int Wout, int c_out,
                        int kh, int kw, int stride, int pad, float* dw, void* stream) {
    return check(mi::conv2d_wgrad_f32(dy, x, B, Hin, Win, c_in, Hout, Wout, c_out, kh, kw, stride, pad, dw, S(stream)),
                 "mi_conv2d_wgrad_f32");
}
int mi_conv2d_wgrad_f16_supported(int Hout, int Wout, int c_in, int c_out, int kh, int kw, int stride) {
    return mi::conv_wgrad_tc_supported(Hout, Wout, c_in, c_out, kh, kw, stride) ? 1 : 0;
}
long long mi_conv2d_wgrad_f16_workspace_bytes(int B, int Hout, int Wout, int c_in, int c_out, int kh, int kw, int stride) {
    return mi::conv_wgrad_tc_workspace_bytes(B, Hout, Wout, c_in, c_out, kh, kw, stride);
}
int mi_conv2d_wgrad_f16(const void* dy_f16, const void* x_f16, int B, int Hout, int Wout, int c_in, int c_out, int kh, int kw,
                        int stride, float* dw, float* workspace, long long workspace_bytes, void* stream) {
    return check(mi::conv_wgrad_tc(static_cast<const __half*>(dy_f16), static_cast<const __half*>(x_f16), B, Hout, Wout, c_in,
                                   c_out, kh, kw, stride, dw, workspace, workspace_bytes, S(stream)),
                 "mi_conv2d_wgrad_f16");
}
int mi_gn_silu_bwd(const float* x, const float* dy, const double* sums, int B, int hw, int C, int groups,
                   const float* gamma, const float* beta, const float* scale_shift, int scale_shift_ld, float eps,
                   float* dx, float* dgamma, float* dbeta, float* d_scale_shift, int d_scale_shift_ld, float* workspace,
                   void* stream) {
    return check(mi::gn_silu_bwd(x, dy, sums, B, hw, C, groups, gamma, beta, scale_shift, scale_shift_ld, eps, dx, dgamma,
                                 dbeta, d_scale_shift, d_scale_shift_ld, workspace, S(stream)),
                 "mi_gn_silu_bwd");
}
int mi_ln_rows_bwd(const float* in, const float* dy, long long rows, int C, const float* gamma, float eps, int pre_gelu,
                   float* dx, float* dgamma, float* dbeta, void* stream) {
    return check(mi::ln_rows_bwd(in, dy, rows, C, gamma, eps, pre_gelu, dx, dgamma, dbeta, S(stream)), "mi_ln_rows_bwd");
}
int mi_softmax_rows(float* s, long long R, int L, void* stream) {
    return check(mi::softmax_rows(s, R, L, S(stream)), "mi_softmax_rows");
}
int mi_softmax_rows_bwd(const float* P, float* dP, long long R, int L, void* stream) {
    return check(mi::softmax_rows_bwd(P, dP, R, L, S(stream)), "mi_softmax_rows_bwd");
}
int mi_upsample2x_bwd(const float* dy, int B, int H, int W, int C, float* dx, void* stream) {
    return check(mi::upsample2x_bwd(dy, B, H, W, C, dx, S(stream)), "mi_upsample2x_bwd");
}

}  // extern "C"
