"""Tensor-level view of the C ABI: every method takes torch CUDA tensors (caller-allocated outputs), checks dtypes /
contiguity, and makes exactly one call into libminimagen_b200.so on the current torch CUDA stream.

`NativeOps` is the only implementation shipped in the package.  (tests/ carries a torch emulation of the same
interface so that the host-side orchestration can be unit-tested on a CPU-only box; the product never uses it.)
"""
import torch

from . import _native as N

F16, F32, F64, I64, U8 = torch.float16, torch.float32, torch.float64, torch.int64, torch.uint8


def _chk(t, dtype, name):
    if t is None:
        return
    if t.dtype != dtype:
        raise TypeError(f"{name}: expected {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError(f"{name}: tensor must be contiguous")


def _chk_out(t, dtype, name):
    """Outputs are addressed through explicit strides, so views (e.g. a channel slice) are fine; only the dtype is fixed."""
    if t is not None and t.dtype != dtype:
        raise TypeError(f"{name}: expected {dtype}, got {t.dtype}")


class NativeOps:
    name = "native-sm100a"
    attention_tc = True      # tcgen05 attention core where the shape allows (mi_attention_fwd workspace)

    def set_launch_mode(self, pdl):
        """Programmatic dependent launch for every kernel of the library (mi_set_launch_mode)."""
        N.load().mi_set_launch_mode(int(bool(pdl)))

    # ---------------------------------------------------------------- capability / weights
    def igemm_supported(self, H, W, c_in, c_out):
        return bool(N.load().mi_conv2d_igemm_supported(int(H), int(W), int(c_in), int(c_out)))

    def pack_conv_weight(self, w, scale=1.0):
        """w: (O, I, KH, KW) or (O, I) fp32 -> (O, KH*KW*I) fp16 tap-major / channel-minor."""
        if w.dim() == 2:
            w = w[:, :, None, None]
        w = w.detach().to(F32).contiguous()
        O, I, KH, KW = w.shape
        out = torch.empty((O, KH * KW * I), dtype=F16, device=w.device)
        N.call("mi_pack_conv_weight_f16", N.ptr(w), O, I, KH, KW, float(scale), N.ptr(out), N.stream())
        return out

    def pack_conv_weight_dgrad(self, w):
        """w: (O, I, KH, KW) or (O, I) fp32 -> (I, KH*KW*O) fp16: the operand of the data-gradient conv (taps flipped, channels swapped)."""
        if w.dim() == 2:
            w = w[:, :, None, None]
        w = w.detach().to(F32).contiguous()
        O, I, KH, KW = w.shape
        out = torch.empty((I, KH * KW * O), dtype=F16, device=w.device)
        N.call("mi_pack_conv_weight_dgrad_f16", N.ptr(w), O, I, KH, KW, N.ptr(out), N.stream())
        return out

    # ---------------------------------------------------------------- convolutions
    def conv_igemm(self, act, B, H, W, lda, c_off, c_in, wp, c_out, kh, kw, mode, bias, residual, out_f32, out_f16,
                   out_strides, block_n=0, out_sc=1, n_valid=0, act2=None, lda2=0, c_off2=0, c_in1=0, out_stats=None):
        """act2 (optional): second fp16 activation tensor; channels [c_in1, c_in) of every tap are read from it.
        out_stats (optional): zeroed fp64 [B, c_out/16, 2] receiving per-block (sum, sum of squares) of the output."""
        _chk(act, F16, "act"); _chk(act2, F16, "act2"); _chk(wp, F16, "wp"); _chk(bias, F32, "bias")
        _chk_out(residual, F32, "residual"); _chk_out(out_f32, F32, "out_f32"); _chk_out(out_f16, F16, "out_f16")
        _chk(out_stats, F64, "out_stats")
        sb, sh, sw = out_strides
        N.call("mi_conv2d_igemm_f16", N.ptr(act), B, H, W, lda, c_off, c_in, N.ptr(act2), lda2, c_off2, c_in1,
               N.ptr(wp), c_out, kh, kw, mode, N.ptr(bias), N.ptr(residual), N.ptr(out_f32), N.ptr(out_f16),
               N.ptr(out_stats), sb, sh, sw, out_sc, n_valid, block_n, None, None, 0, N.stream())

    def conv_res1x1_supported(self, H, W, c_in, c_out, x_cin):
        return bool(N.load().mi_conv3x3_res1x1_supported(int(H), int(W), int(c_in), int(c_out), int(x_cin)))

    def conv_res1x1(self, act, B, H, W, lda, c_in, act2, lda2, c_in1, x, ldx, x_cin, x2, ldx2, x_cin1, wp, c_out, bias,
                    residual, out_f32, out_f16, out_stats):
        """3x3 conv over act (+act2) plus a folded 1x1 conv over x (+x2) in one launch; wp = [c_out][9*c_in + x_cin]."""
        for nm, t in (("act", act), ("act2", act2), ("x", x), ("x2", x2), ("wp", wp)):
            _chk(t, F16, nm)
        _chk(bias, F32, "bias"); _chk(residual, F32, "residual"); _chk(out_f32, F32, "out_f32"); _chk(out_f16, F16, "out_f16")
        _chk(out_stats, F64, "out_stats")
        N.call("mi_conv3x3_res1x1_f16", N.ptr(act), B, H, W, lda, c_in, N.ptr(act2), lda2, c_in1, N.ptr(x), ldx, x_cin,
               N.ptr(x2), ldx2, x_cin1, N.ptr(wp), c_out, N.ptr(bias), N.ptr(residual), N.ptr(out_f32), N.ptr(out_f16),
               N.ptr(out_stats), None, N.stream())

    def conv_gn_supported(self, H, W, c0, c1, c_out, groups):
        return bool(N.load().mi_conv3x3_gn_supported(int(H), int(W), int(c0), int(c1), int(c_out), int(groups)))

    def conv_gn(self, src0, c0, src1, c1, scale1, B, H, W, groups, stats0, stats1, gamma, beta, scale_shift, ss_ld, eps,
                wp, c_out, bias, residual, out_f32, out_f16, out_stats):
        """Fused GroupNorm -> FiLM -> SiLU -> 3x3 conv (Block.forward) over fp32 NHWC source(s)."""
        _chk(src0, F32, "src0"); _chk(src1, F32, "src1"); _chk(stats0, F64, "stats0"); _chk(stats1, F64, "stats1")
        _chk(gamma, F32, "gamma"); _chk(beta, F32, "beta"); _chk_out(scale_shift, F32, "scale_shift"); _chk(wp, F16, "wp")
        _chk(bias, F32, "bias"); _chk(residual, F32, "residual"); _chk(out_f32, F32, "out_f32")
        _chk(out_f16, F16, "out_f16"); _chk(out_stats, F64, "out_stats")
        N.call("mi_conv3x3_gn_silu_f16", N.ptr(src0), c0, N.ptr(src1), c1, float(scale1), B, H, W, groups,
               N.ptr(stats0), N.ptr(stats1), N.ptr(gamma), N.ptr(beta), N.ptr(scale_shift), int(ss_ld), float(eps),
               N.ptr(wp), c_out, N.ptr(bias), N.ptr(residual), N.ptr(out_f32), N.ptr(out_f16), N.ptr(out_stats), None,
               N.stream())

    def conv_direct(self, inp, B, Hin, Win, c_in, ldi, w, c_out, kh, kw, stride, pad, bias, residual, out, Hout, Wout,
                    out_strides):
        _chk(inp, F32, "inp"); _chk(w, F32, "w"); _chk(bias, F32, "bias"); _chk_out(residual, F32, "residual")
        if out.dtype != F32:
            raise TypeError("out must be fp32")
        sb, sh, sw, sc = out_strides
        N.call("mi_conv2d_direct_f32", N.ptr(inp), B, Hin, Win, c_in, ldi, N.ptr(w), c_out, kh, kw, stride, pad,
               N.ptr(bias), N.ptr(residual), N.ptr(out), Hout, Wout, sb, sh, sw, sc, N.stream())

    # ---------------------------------------------------------------- normalisation / casts
    def gn_stats(self, src0, c0, src1, c1, scale1, B, hw, groups, sums):
        _chk(src0, src0.dtype, "src0"); _chk(src1, src0.dtype, "src1"); _chk(sums, F64, "sums")
        N.call("mi_gn_stats", N.ptr(src0), c0, N.ptr(src1), c1, float(scale1), int(src0.dtype == F16), B, hw, groups,
               N.ptr(sums), N.stream())

    def gn_apply_silu(self, src0, c0, src1, c1, scale1, B, hw, groups, stats0, sb0, stats1, sb1, gamma, beta,
                      scale_shift, ss_ld, eps, out):
        """src0/src1: both fp32 or both fp16.  sb0 == 0: stats0 = [B, groups, 2] group sums over the concat (gn_stats);
        sb0 > 0: per-source block sums [B, c/sb, 2].  scale_shift: fp32 view, row b at data_ptr + b*ss_ld = [scale | shift]."""
        in16 = src0.dtype == F16
        _chk(src0, src0.dtype, "src0"); _chk(src1, src0.dtype, "src1"); _chk(stats0, F64, "stats0")
        _chk(stats1, F64, "stats1"); _chk(gamma, F32, "gamma"); _chk(beta, F32, "beta")
        _chk_out(scale_shift, F32, "scale_shift")
        N.call("mi_gn_apply_silu", N.ptr(src0), c0, N.ptr(src1), c1, float(scale1), int(in16), B, hw, groups,
               N.ptr(stats0), int(sb0), N.ptr(stats1), int(sb1), N.ptr(gamma), N.ptr(beta), N.ptr(scale_shift),
               int(ss_ld), float(eps), N.ptr(out), int(out.dtype == F16), N.stream())

    def cast_act(self, src0, c0, src1, c1, scale1, B, H, W, mode, out):
        _chk(src0, src0.dtype, "src0"); _chk(src1, src0.dtype, "src1")
        N.call("mi_cast_act", N.ptr(src0), c0, N.ptr(src1), c1, float(scale1), int(src0.dtype == F16), B, H, W, mode,
               N.ptr(out), int(out.dtype == F16), N.stream())

    def ln_rows(self, inp, rows, C, gamma, beta, eps, pre_gelu, residual, out_f32, out_f16):
        _chk(inp, F32, "inp"); _chk(gamma, F32, "gamma"); _chk(beta, F32, "beta"); _chk(residual, F32, "residual")
        _chk(out_f32, F32, "out_f32"); _chk(out_f16, F16, "out_f16")
        N.call("mi_ln_rows", N.ptr(inp), rows, C, N.ptr(gamma), N.ptr(beta), float(eps), int(pre_gelu), N.ptr(residual),
               N.ptr(out_f32), N.ptr(out_f16), N.stream())

    # ---------------------------------------------------------------- conditioning
    def linear_f32(self, inp, M, K, W, bias, Nout, in_act, out_act, addend, out_f32, out_f16, out_scale=1.0):
        _chk(inp, F32, "inp"); _chk(W, F32, "W"); _chk(bias, F32, "bias"); _chk(addend, F32, "addend")
        _chk(out_f32, F32, "out_f32"); _chk(out_f16, F16, "out_f16")
        N.call("mi_linear_f32", N.ptr(inp), M, K, N.ptr(W), N.ptr(bias), Nout, in_act, out_act, N.ptr(addend),
               N.ptr(out_f32), N.ptr(out_f16), float(out_scale), N.stream())

    def posemb(self, t, B, dim, out):
        _chk(t, I64, "t"); _chk(out, F32, "out")
        N.call("mi_sinusoidal_posemb", N.ptr(t), B, dim, N.ptr(out), N.stream())

    def text_tokens(self, proj, B, L, D, mask, keep, null_embed, max_len, c_out, m, row_off, pooled):
        _chk(proj, F32, "proj"); _chk(mask, U8, "mask"); _chk(keep, U8, "keep"); _chk(null_embed, F32, "null_embed")
        _chk(c_out, F32, "c_out"); _chk(pooled, F32, "pooled")
        N.call("mi_text_tokens", N.ptr(proj), B, L, D, N.ptr(mask), N.ptr(keep), N.ptr(null_embed), max_len,
               N.ptr(c_out), m, row_off, N.ptr(pooled), N.stream())

    def place_rows(self, src, B, r, D, dst, m, row_off):
        _chk(src, F32, "src"); _chk(dst, F32, "dst")
        N.call("mi_place_rows", N.ptr(src), B, r, D, N.ptr(dst), m, row_off, N.stream())

    def select_rows(self, a, null_row, keep, addend, B, Nn, out):
        _chk(a, F32, "a"); _chk(null_row, F32, "null_row"); _chk(keep, U8, "keep"); _chk(addend, F32, "addend")
        N.call("mi_select_rows", N.ptr(a), N.ptr(null_row), N.ptr(keep), N.ptr(addend), B, Nn, N.ptr(out), N.stream())

    def nchw_to_nhwc(self, a, ca, b, cb, B, hw, c_pad, out):
        _chk(a, F32, "a"); _chk(b, F32, "b"); _chk(out, F32, "out")
        N.call("mi_nchw_to_nhwc", N.ptr(a), ca, N.ptr(b), cb, B, hw, c_pad, N.ptr(out), N.stream())

    def stem_unroll(self, a, ca, b, cb, B, H, W, out):
        _chk(a, F32, "a"); _chk(b, F32, "b"); _chk(out, F16, "out")
        N.call("mi_stem_unroll_f16", N.ptr(a), ca, N.ptr(b), cb, B, H, W, N.ptr(out), N.stream())

    def resize_separable(self, inp, planes, hin, win, out, hout, wout, iy, wy, ix, wx, clamp=None):
        """iy / ix: int32 [n_out, taps] source indices; wy / wx: fp32 [n_out, taps] weights (see helpers.resize_tables)."""
        _chk(inp, F32, "inp"); _chk(out, F32, "out"); _chk(wy, F32, "wy"); _chk(wx, F32, "wx")
        _chk(iy, torch.int32, "iy"); _chk(ix, torch.int32, "ix")
        N.call("mi_resize_separable", N.ptr(inp), planes, hin, win, N.ptr(out), hout, wout, N.ptr(iy), N.ptr(wy),
               iy.shape[1], N.ptr(ix), N.ptr(wx), ix.shape[1], int(clamp is not None),
               float(clamp[0]) if clamp is not None else 0.0, float(clamp[1]) if clamp is not None else 0.0, N.stream())

    def silu(self, inp, out):
        _chk(inp, F32, "inp"); _chk(out, F32, "out")
        N.call("mi_silu_f32", N.ptr(inp), inp.numel(), N.ptr(out), N.stream())

    # ---------------------------------------------------------------- attention
    def attention(self, q, q_bs, ldq, k, v, kv_bs, ldkv, kv_hs, null_kv, mask, B, heads, n, m, out, o_bs, ldo):
        """k / v may be views (column offsets) into one projection buffer: only their data_ptr is used."""
        if q.dtype != F16 or k.dtype != F16 or v.dtype != F16 or out.dtype != F16:
            raise TypeError("attention operands must be fp16")
        _chk(null_kv, F32, "null_kv"); _chk(mask, U8, "mask")
        ws = None
        if self.attention_tc and n % 128 == 0 and m >= 128:
            # operand workspace of the tcgen05 kernel (null-prepended padded K, transposed V); per call, so it is safe under
            # CUDA-graph capture and concurrent streams
            nbytes = int(N.load().mi_attention_workspace_bytes(B, heads, kv_hs, m))
            ws = torch.empty(nbytes, dtype=torch.uint8, device=q.device)
        N.call("mi_attention_fwd", N.ptr(q), q_bs, ldq, N.ptr(k), N.ptr(v), kv_bs, ldkv, kv_hs, N.ptr(null_kv),
               N.ptr(mask), B, heads, n, m, N.ptr(out), o_bs, ldo, N.ptr(ws), ws.numel() if ws is not None else 0,
               N.stream())

    # ---------------------------------------------------------------- DDPM step
    def step_x0(self, x_t, eps_cond, eps_null, cond_scale, t, tab_a, tab_b, B, n, x0):
        for nm, tt in (("x_t", x_t), ("eps_cond", eps_cond), ("eps_null", eps_null), ("tab_a", tab_a),
                       ("tab_b", tab_b), ("x0", x0)):
            _chk(tt, F32, nm)
        _chk(t, I64, "t")
        N.call("mi_step_x0", N.ptr(x_t), N.ptr(eps_cond), N.ptr(eps_null), float(cond_scale), N.ptr(t), N.ptr(tab_a),
               N.ptr(tab_b), B, n, N.ptr(x0), N.stream())

    def step_quantile(self, x0, B, n, rank_lo, rank_hi, weight, min_s, s):
        _chk(x0, F32, "x0"); _chk(s, F32, "s")
        N.call("mi_step_quantile", N.ptr(x0), B, n, int(rank_lo), int(rank_hi), float(weight), float(min_s), N.ptr(s),
               N.stream())

    def step_posterior(self, x0, x_t, noise, s, t, c1, c2, sigma, B, n, out):
        for nm, tt in (("x0", x0), ("x_t", x_t), ("noise", noise), ("s", s), ("c1", c1), ("c2", c2), ("sigma", sigma),
                       ("out", out)):
            _chk(tt, F32, nm)
        _chk(t, I64, "t")
        N.call("mi_step_posterior", N.ptr(x0), N.ptr(x_t), N.ptr(noise), N.ptr(s), N.ptr(t), N.ptr(c1), N.ptr(c2),
               N.ptr(sigma), B, n, N.ptr(out), N.stream())

    def step_epilogue(self, x_t, eps_cond, eps_null, cond_scale, t, tab_a, tab_b, c1, c2, sigma, noise, B, n, rank_lo,
                      rank_hi, weight, min_s, out, s_out=None):
        """CFG combine + x0 + exact dynamic-threshold quantile + clamp/divide + posterior mean + noise; `out` may be `x_t`."""
        for nm, tt in (("x_t", x_t), ("eps_cond", eps_cond), ("eps_null", eps_null), ("tab_a", tab_a), ("tab_b", tab_b),
                       ("c1", c1), ("c2", c2), ("sigma", sigma), ("noise", noise), ("out", out), ("s_out", s_out)):
            _chk(tt, F32, nm)
        _chk(t, I64, "t")
        ws = None
        nws = int(N.load().mi_step_epilogue_workspace_floats(B, n))
        if nws:
            ws = torch.empty(nws, dtype=F32, device=x_t.device)
            if s_out is None:
                s_out = torch.empty(B, dtype=F32, device=x_t.device)
        N.call("mi_step_epilogue", N.ptr(x_t), N.ptr(eps_cond), N.ptr(eps_null), float(cond_scale), N.ptr(t), N.ptr(tab_a),
               N.ptr(tab_b), N.ptr(c1), N.ptr(c2), N.ptr(sigma), N.ptr(noise), B, n, int(rank_lo), int(rank_hi),
               float(weight), float(min_s), N.ptr(out), N.ptr(s_out), N.ptr(ws), N.stream())

    def step_advance_t(self, t, B):
        _chk(t, I64, "t")
        N.call("mi_step_advance_t", N.ptr(t), B, N.stream())

    def step_finalize(self, x, n, unnormalize, out):
        _chk(x, F32, "x"); _chk(out, F32, "out")
        N.call("mi_step_finalize", N.ptr(x), n, int(unnormalize), N.ptr(out), N.stream())

    def q_sample(self, x0, noise, t, tab_a, tab_b, B, n, post_scale, post_shift, out):
        _chk(x0, F32, "x0"); _chk(noise, F32, "noise"); _chk(t, I64, "t"); _chk(out, F32, "out")
        N.call("mi_q_sample", N.ptr(x0), N.ptr(noise), N.ptr(t), N.ptr(tab_a), N.ptr(tab_b), B, n, float(post_scale),
               float(post_shift), N.ptr(out), N.stream())

    def inpaint_blend(self, x, known, mask, z_known, z_renoise, t, u, U, prime, sqrt_acp, sqrt_1macp, sqrt_alphas,
                      sqrt_betas):
        """RePaint blend of one inpainting replay, in place on x [B, C, H, W]; mask uint8 [B, mh, mw] (nonzero = known pixel),
        sampled nearest-neighbour at x's size; u int32 [1] the resample round (mi_inpaint_blend)."""
        for nm, tt in (("x", x), ("known", known), ("z_known", z_known), ("z_renoise", z_renoise), ("sqrt_acp", sqrt_acp),
                       ("sqrt_1macp", sqrt_1macp), ("sqrt_alphas", sqrt_alphas), ("sqrt_betas", sqrt_betas)):
            _chk(tt, F32, nm)
        _chk(mask, U8, "mask"); _chk(t, I64, "t"); _chk(u, torch.int32, "u")
        B, C, H, W = x.shape
        N.call("mi_inpaint_blend", N.ptr(x), N.ptr(known), N.ptr(mask), mask.shape[-2], mask.shape[-1], N.ptr(z_known),
               N.ptr(z_renoise), N.ptr(t), N.ptr(u), int(U), int(prime), N.ptr(sqrt_acp), N.ptr(sqrt_1macp),
               N.ptr(sqrt_alphas), N.ptr(sqrt_betas), B, C, H, W, N.stream())

    def inpaint_advance(self, t, u, U, B):
        """u += 1 after a renoising round, else u = 0 and t <- max(t - 1, 0) (mi_inpaint_advance)."""
        _chk(t, I64, "t"); _chk(u, torch.int32, "u")
        N.call("mi_inpaint_advance", N.ptr(t), N.ptr(u), int(U), B, N.stream())


    # ---------------------------------------------------------------- training side (backward kernels, fp32)
    def gemm_f32(self, A, B, C, M, N, K, a_str, b_str, c_str, Z1=1, Z2=1, a_b=(0, 0), b_b=(0, 0), c_b=(0, 0), alpha=1.0,
                 accumulate=False):
        """C[z](m,n) (+)= alpha * sum_k A[z](m,k) B[z](k,n); a_str = (a_sm, a_sk), b_str = (b_sk, b_sn), c_str = (c_sm, c_sn)
        element strides, *_b = (stride of z1, stride of z2), z = z1*Z2 + z2.  Tensors only provide base pointers."""
        for nm, t in (("A", A), ("B", B), ("C", C)):
            if t.dtype != F32:
                raise TypeError(f"{nm}: expected float32")
        from . import _native as nat       # (the GEMM's own `N` shadows the module alias used elsewhere in this class)
        nat.call("mi_gemm_f32", nat.ptr(A), nat.ptr(B), nat.ptr(C), M, N, K, a_str[0], a_str[1], b_str[0], b_str[1], c_str[0],
                 c_str[1], Z1, Z2, a_b[0], a_b[1], b_b[0], b_b[1], c_b[0], c_b[1], float(alpha), int(accumulate), nat.stream())

    def colsum(self, x, M, Nc, out, accumulate=False):
        _chk(x, F32, "x"); _chk(out, F32, "out")
        N.call("mi_colsum_f32", N.ptr(x), M, Nc, N.ptr(out), int(accumulate), N.stream())

    def conv_dgrad(self, dy, B, Ho, Wo, c_out, w, c_in, kh, kw, stride, pad, dx, Hi, Wi):
        _chk(dy, F32, "dy"); _chk(w, F32, "w"); _chk(dx, F32, "dx")
        N.call("mi_conv2d_dgrad_f32", N.ptr(dy), B, Ho, Wo, c_out, N.ptr(w), c_in, kh, kw, stride, pad, N.ptr(dx), Hi, Wi,
               N.stream())

    def conv_wgrad(self, dy, x, B, Hi, Wi, c_in, Ho, Wo, c_out, kh, kw, stride, pad, dw):
        _chk(dy, F32, "dy"); _chk(x, F32, "x"); _chk(dw, F32, "dw")
        N.call("mi_conv2d_wgrad_f32", N.ptr(dy), N.ptr(x), B, Hi, Wi, c_in, Ho, Wo, c_out, kh, kw, stride, pad, N.ptr(dw),
               N.stream())

    def conv_wgrad_tc_supported(self, Ho, Wo, c_in, c_out, kh, kw, stride=1):
        return bool(N.load().mi_conv2d_wgrad_f16_supported(int(Ho), int(Wo), int(c_in), int(c_out), int(kh), int(kw), int(stride)))

    def conv_wgrad_tc(self, dy16, x16, B, Ho, Wo, c_in, c_out, kh, kw, dw, stride=1):
        """dw (OIHW fp32, overwritten) of a k x k stride-1 'same' conv (or the 4x4 stride-2 pad-1 Downsample) from fp16 NHWC
        dy [B, Ho, Wo, c_out] / x [B, stride*Ho, stride*Wo, c_in], on the tensor cores."""
        _chk(dy16, F16, "dy16"); _chk(x16, F16, "x16"); _chk(dw, F32, "dw")
        nbytes = int(N.load().mi_conv2d_wgrad_f16_workspace_bytes(B, Ho, Wo, c_in, c_out, kh, kw, int(stride)))
        ws = torch.empty(max(nbytes // 4, 4), dtype=F32, device=dw.device)          # per-split partial tiles
        N.call("mi_conv2d_wgrad_f16", N.ptr(dy16), N.ptr(x16), B, Ho, Wo, c_in, c_out, kh, kw, int(stride), N.ptr(dw), N.ptr(ws),
               nbytes, N.stream())

    def gn_silu_bwd(self, x, dy, sums, B, hw, C, groups, gamma, beta, scale_shift, ss_ld, eps, dx, dgamma, dbeta, dss, dss_ld):
        """dgamma / dbeta are ACCUMULATED into (zero them first); dss [B, dss_ld] = [d scale | d shift] or None."""
        _chk(x, F32, "x"); _chk(dy, F32, "dy"); _chk(sums, F64, "sums"); _chk(gamma, F32, "gamma"); _chk(beta, F32, "beta")
        _chk_out(scale_shift, F32, "scale_shift"); _chk(dx, F32, "dx"); _chk(dgamma, F32, "dgamma"); _chk(dbeta, F32, "dbeta")
        _chk(dss, F32, "dss")
        ws = torch.empty(2 * B * C + 4 * B * groups, dtype=F32, device=x.device)
        N.call("mi_gn_silu_bwd", N.ptr(x), N.ptr(dy), N.ptr(sums), B, hw, C, groups, N.ptr(gamma), N.ptr(beta),
               N.ptr(scale_shift), int(ss_ld), float(eps), N.ptr(dx), N.ptr(dgamma), N.ptr(dbeta), N.ptr(dss), int(dss_ld),
               N.ptr(ws), N.stream())

    def ln_rows_bwd(self, inp, dy, R, C, gamma, eps, pre_gelu, dx, dgamma, dbeta):
        _chk(inp, F32, "inp"); _chk(dy, F32, "dy"); _chk(gamma, F32, "gamma"); _chk(dx, F32, "dx")
        _chk(dgamma, F32, "dgamma"); _chk(dbeta, F32, "dbeta")
        N.call("mi_ln_rows_bwd", N.ptr(inp), N.ptr(dy), R, C, N.ptr(gamma), float(eps), int(pre_gelu), N.ptr(dx),
               N.ptr(dgamma), N.ptr(dbeta), N.stream())

    def softmax_rows(self, s, R, L):
        _chk(s, F32, "s")
        N.call("mi_softmax_rows", N.ptr(s), R, L, N.stream())

    def softmax_rows_bwd(self, P, dP, R, L):
        _chk(P, F32, "P"); _chk(dP, F32, "dP")
        N.call("mi_softmax_rows_bwd", N.ptr(P), N.ptr(dP), R, L, N.stream())

    def upsample2x_bwd(self, dy, B, H, W, C, dx):
        _chk(dy, F32, "dy"); _chk(dx, F32, "dx")
        N.call("mi_upsample2x_bwd", N.ptr(dy), B, H, W, C, N.ptr(dx), N.stream())


_OPS = None


def get_ops():
    """The process-wide ops backend.  Loads the native library on first use (raises if it is missing)."""
    global _OPS
    if _OPS is None:
        N.load()
        _OPS = NativeOps()
    return _OPS


def set_ops(ops):
    """Test hook: install another implementation of the ops interface (used by tests/ only)."""
    global _OPS
    _OPS = ops
