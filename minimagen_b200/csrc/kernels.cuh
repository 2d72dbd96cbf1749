// Internal C++ declarations of the kernel launchers (one translation unit per kernel family).
// The public boundary is the C ABI in include/minimagen_b200.h (capi.cu).
#pragma once
#include <cuda_fp16.h>
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace mi {

// elementwise.cu
int gn_stats(const void* src0, int C0, const void* src1, int C1, float scale1, int in_is_f16, int B, int HW, int groups,
             double* sums, cudaStream_t st);
int gn_apply_silu(const void* src0, int C0, const void* src1, int C1, float scale1, int in_is_f16, int B, int HW,
                  int groups, const double* stats0, int sb0, const double* stats1, int sb1, const float* gamma,
                  const float* beta, const float* scale_shift, int ss_ld, float eps, void* out, int out_is_f16,
                  cudaStream_t st);
int cast_act(const void* src0, int C0, const void* src1, int C1, float scale1, int in_is_f16, int B, int H, int W,
             int mode, void* out, int out_is_f16, cudaStream_t st);
int ln_rows(const float* in, long long R, int C, const float* gamma, const float* beta, float eps, int pre_gelu,
            const float* residual, float* out_f32, __half* out_f16, cudaStream_t st);
int linear_f32(const float* in, int M, int K, const float* W, const float* bias, int N, int in_act, int out_act,
               const float* addend, float* out_f32, __half* out_f16, float out_scale, cudaStream_t st);
int posemb(const long long* t, int B, int dim, float* out, cudaStream_t st);
int text_tokens(const float* proj, int B, int L, int D, const uint8_t* mask, const uint8_t* keep,
                const float* null_embed, int max_len, float* c_out, int m, int row_off, float* pooled,
                cudaStream_t st);
int place_rows(const float* src, int B, int r, int D, float* dst, int m, int row_off, cudaStream_t st);
int select_rows(const float* a, const float* nullv, const uint8_t* keep, const float* addend, int B, int N, float* out,
                cudaStream_t st);
int nchw_to_nhwc(const float* a, int Ca, const float* b, int Cb, int B, int HW, int Cp, float* out, cudaStream_t st);
int stem_unroll(const float* a, int Ca, const float* b, int Cb, int B, int H, int W, __half* out, cudaStream_t st);
int silu_f32(const float* in, long long n, float* out, cudaStream_t st);
int resize_sep(const float* in, long long planes, int Hin, int Win, float* out, int Hout, int Wout, const int* iy,
               const float* wy, int ty, const int* ix, const float* wx, int tx, int has_clamp, float lo, float hi,
               cudaStream_t st);
int pack_conv_weight(const float* w, int O, int I, int KH, int KW, float scale, __half* out, cudaStream_t st);
int pack_conv_weight_dgrad(const float* w, int O, int I, int KH, int KW, __half* out, cudaStream_t st);

// conv_direct.cu
int conv_direct_f32(const float* in, int B, int Hin, int Win, int Cin, int ldi, const float* w, int Cout, int KH,
                    int KW, int stride, int pad, const float* bias, const float* residual, float* out, int Hout,
                    int Wout, long long osb, long long osh, long long osw, long long osc, cudaStream_t st);

// attention.cu
int attention_fwd(const __half* q, long long q_bs, int ldq, const __half* k, const __half* v, long long kv_bs, int ldkv,
                  int kv_hs, const float* null_kv, const uint8_t* mask, int B, int heads, int n, int m, __half* out,
                  long long o_bs, int ldo, cudaStream_t st);

// attention_tc.cu: tcgen05 / TMEM path (no mask, n % 128 == 0, contiguous q); workspace = padded K and transposed V
bool attention_tc_supported(int n, int ldq, int ldo, long long q_bs, const void* mask);
long long attention_tc_workspace_bytes(int B, int heads, int kv_hs, int m);
int attention_tc_fwd(const __half* q, long long q_bs, int ldq, const __half* k, const __half* v, long long kv_bs, int ldkv,
                     int kv_hs, const float* null_kv, const uint8_t* key_mask, int B, int heads, int n, int m, __half* out, long long o_bs, int ldo,
                     void* workspace, long long workspace_bytes, int* err_flag, cudaStream_t st);

// conv_tc.cu: cuTensorMapEncodeTiled through the runtime's driver entry point (no -lcuda link dependency)
typedef CUresult (*PFN_tmaEncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                       const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                       CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
PFN_tmaEncodeTiled get_tma_encode();

// step.cu
int step_x0(const float* x_t, const float* eps_cond, const float* eps_null, float cond_scale, const long long* t,
            const float* tab_recip, const float* tab_recipm1, int B, int n_per_img, float* x0, cudaStream_t st);
int step_quantile(const float* x0, int B, int n_per_img, int rank_lo, int rank_hi, float weight, float min_s,
                  float* s_out, cudaStream_t st);
int step_posterior(const float* x0, const float* x_t, const float* noise, const float* s, const long long* t,
                   const float* tab_c1, const float* tab_c2, const float* tab_sigma, int B, int n_per_img, float* out,
                   cudaStream_t st);
bool step_epilogue_fused_ok(int n_per_img);
int step_epilogue(const float* x_t, const float* eps_cond, const float* eps_null, float cond_scale, const long long* t,
                  const float* tab_recip, const float* tab_recipm1, const float* tab_c1, const float* tab_c2,
                  const float* tab_sigma, const float* noise, int B, int n_per_img, int rank_lo, int rank_hi,
                  float weight, float min_s, float* out, float* s_out, float* x0_ws, cudaStream_t st);
int step_advance_t(long long* t, int B, cudaStream_t st);
int step_finalize(const float* x, long long n, int unnormalize, float* out, cudaStream_t st);
int q_sample(const float* x0, const float* noise, const long long* t, const float* tab_a, const float* tab_b, int B,
             int n_per_img, float post_scale, float post_shift, float* out, cudaStream_t st);
int inpaint_blend(float* x, const float* known, const unsigned char* mask, int mask_h, int mask_w, const float* z_known,
                  const float* z_renoise, const long long* t, const int* u, int U, int prime, const float* tab_acp,
                  const float* tab_1macp, const float* tab_sa, const float* tab_sb, int B, int C, int H, int W,
                  cudaStream_t st);
int inpaint_advance(long long* t, int* u, int U, int B, cudaStream_t st);

// backward.cu: fp32 backward kernels of the training side (SURVEY 8f-2)
int gemm_f32(const float* A, const float* B, float* C, int M, int N, int K, long long a_sm, long long a_sk, long long b_sk,
             long long b_sn, long long c_sm, long long c_sn, int Z1, int Z2, long long a_b1, long long a_b2, long long b_b1,
             long long b_b2, long long c_b1, long long c_b2, float alpha, int accumulate, cudaStream_t st);
int colsum_f32(const float* x, long long M, int N, float* out, int accumulate, cudaStream_t st);
int conv2d_dgrad_f32(const float* dy, int B, int Ho, int Wo, int Cout, const float* w, int Cin, int KH, int KW, int stride,
                     int pad, float* dx, int Hi, int Wi, cudaStream_t st);
int conv2d_wgrad_f32(const float* dy, const float* x, int B, int Hi, int Wi, int Cin, int Ho, int Wo, int Cout, int KH,
                     int KW, int stride, int pad, float* dw, cudaStream_t st);
// wgrad_tc.cu: weight gradient of stride-1 'same' convs on tcgen05 (MN-major operands, contraction over pixels)
bool conv_wgrad_tc_supported(int H, int W, int Cin, int Cout, int kh, int kw, int stride);
long long conv_wgrad_tc_workspace_bytes(int B, int H, int W, int Cin, int Cout, int kh, int kw, int stride);
int conv_wgrad_tc(const __half* dy, const __half* x, int B, int H, int W, int Cin, int Cout, int kh, int kw, int stride,
                  float* dw, float* workspace, long long workspace_bytes, cudaStream_t stream);
int gn_silu_bwd(const float* x, const float* dy, const double* sums, int B, int HW, int C, int groups, const float* gamma,
                const float* beta, const float* ss, int ss_ld, float eps, float* dx, float* dgamma, float* dbeta,
                float* dss, int dss_ld, float* workspace, cudaStream_t st);
int ln_rows_bwd(const float* in, const float* dy, long long R, int C, const float* gamma, float eps, int pre_gelu, float* dx,
                float* dgamma, float* dbeta, cudaStream_t st);
int softmax_rows(float* s, long long R, int L, cudaStream_t st);
int softmax_rows_bwd(const float* P, float* dP, long long R, int L, cudaStream_t st);
int upsample2x_bwd(const float* dy, int B, int H, int W, int C, float* dx, cudaStream_t st);

}  // namespace mi
