// DDPM reverse-step epilogue (everything in Imagen._p_sample after the U-Net call), NCHW fp32 like the reference:
//   1. classifier-free-guidance combine            null + (cond - null) * w                 (Unet.py:506)
//      + predict_start_from_noise                  x0 = a[t] * x_t - b[t] * eps             (diffusion_model.py:159-162)
//   2. dynamic threshold                           s = max(quantile(|x0|, p), 1) per image  (Imagen.py:313-320)
//      exact: radix select on the uint32 bit patterns of |x0| (order statistics lo / hi chosen on the host with
//      torch's own fp32 rank arithmetic), linear interpolation like at::lerp
//   3. clamp(x0, -s, s) / s, posterior mean c1[t] * x0 + c2[t] * x_t, + sigma[t] * noise (zero at t == 0)
//                                                                  (Imagen.py:323, diffusion_model.py:118-125, Imagen.py:361-370)
// The per-image schedule gathers (helpers.extract) happen inside the kernels from the fp32 tables.
// Products and sums are kept un-fused (__fmul_rn/__fadd_rn) so that the arithmetic matches torch's op-by-op rounding.
#include <cuda_runtime.h>
#include <float.h>
#include <stdint.h>

#include <cooperative_groups.h>

#include "kernels.cuh"
#include "launch.cuh"

namespace mi {

namespace {

__global__ void __launch_bounds__(256)
x0_kernel(const float* __restrict__ x_t, const float* __restrict__ eps_cond, const float* __restrict__ eps_null,
          float cond_scale, const long long* __restrict__ t, const float* __restrict__ tab_recip,
          const float* __restrict__ tab_recipm1, int n_per_img, float* __restrict__ x0) {
    pdl_wait();
    pdl_trigger();
    const int b = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_per_img) return;
    const long long idx = (long long)b * n_per_img + i;
    const long long tb = t[b];
    const float a = tab_recip[tb], bb = tab_recipm1[tb];
    float e = eps_cond[idx];
    if (eps_null) {
        const float nl = eps_null[idx];
        e = __fadd_rn(nl, __fmul_rn(__fsub_rn(e, nl), cond_scale));
    }
    x0[idx] = __fsub_rn(__fmul_rn(a, x_t[idx]), __fmul_rn(bb, e));
}

// One CTA per image.  Exact k-th order statistics of |x| by 4 x 8-bit radix passes over the float bit patterns.
constexpr int kSelThreads = 1024;

__device__ __forceinline__ uint32_t absbits(float v) { return __float_as_uint(v) & 0x7FFFFFFFu; }

__global__ void __launch_bounds__(kSelThreads)
quantile_kernel(const float* __restrict__ x0, int n, int rank_lo, int rank_hi, float weight, float min_s,
                float* __restrict__ s_out) {
    pdl_wait();
    pdl_trigger();
    __shared__ unsigned hist[257];
    __shared__ uint32_t sh_prefix, sh_k, sh_eq;
    __shared__ uint32_t sh_min[32];
    const float* x = x0 + (long long)blockIdx.x * n;
    const int tid = threadIdx.x, lane = tid & 31;
    uint32_t prefix = 0, maskbits = 0, k = (uint32_t)rank_lo;
    const int n_round = (n + 31) & ~31;

    for (int pass = 0; pass < 4; ++pass) {
        const int shift = 24 - 8 * pass;
        for (int i = tid; i < 257; i += kSelThreads) hist[i] = 0;
        __syncthreads();
        for (int i = tid; i < n_round; i += kSelThreads) {
            unsigned bin = 256;
            if (i < n) {
                const uint32_t key = absbits(x[i]);
                if ((key & maskbits) == prefix) bin = (key >> shift) & 0xFF;
            }
            const unsigned peers = __match_any_sync(0xffffffffu, bin);
            if (lane == (__ffs(peers) - 1)) atomicAdd(&hist[bin], __popc(peers));
        }
        __syncthreads();
        if (tid == 0) {
            uint32_t cum = 0;
            int d = 0;
            for (; d < 256; ++d) {
                if (k < cum + hist[d]) break;
                cum += hist[d];
            }
            sh_prefix = prefix | ((uint32_t)d << shift);
            sh_k = k - cum;
            sh_eq = hist[d];
        }
        __syncthreads();
        prefix = sh_prefix;
        k = sh_k;
        maskbits |= 0xFFu << shift;
        __syncthreads();
    }
    // prefix == bit pattern of sorted[rank_lo]; k == index inside its run of equal values; sh_eq == run length
    const uint32_t v_lo = prefix;
    uint32_t v_hi = v_lo;
    if (rank_hi > rank_lo && k + 1 >= sh_eq) {
        // next order statistic = smallest key strictly greater than v_lo
        uint32_t mn = 0xFFFFFFFFu;
        for (int i = tid; i < n; i += kSelThreads) {
            const uint32_t key = absbits(x[i]);
            if (key > v_lo && key < mn) mn = key;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mn = min(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        if (lane == 0) sh_min[tid >> 5] = mn;
        __syncthreads();
        if (tid < 32) {
            mn = sh_min[tid];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) mn = min(mn, __shfl_xor_sync(0xffffffffu, mn, o));
            if (tid == 0) sh_min[0] = mn;
        }
        __syncthreads();
        v_hi = sh_min[0];
        if (v_hi == 0xFFFFFFFFu) v_hi = v_lo;   // cannot happen for rank_hi < n
    }
    if (tid == 0) {
        const float lo = __uint_as_float(v_lo), hi = __uint_as_float(v_hi);
        // at::lerp (vectorised CPU form): base + coeff * (end - start), weight < 0.5 ? (start, w) : (end, w - 1)
        const float diff = __fsub_rn(hi, lo);
        const float s = (weight < 0.5f) ? fmaf(weight, diff, lo) : fmaf(__fsub_rn(weight, 1.0f), diff, hi);
        s_out[blockIdx.x] = fmaxf(s, min_s);   // s.clamp_(min=1.)
    }
}

// Cluster variant: 8 CTAs (one thread-block cluster) per image, every CTA keeps its n/8 keys in REGISTERS, so the image
// is read from memory once instead of four to five times by a single SM; the per-pass 256-bin histograms are summed
// across the cluster through distributed shared memory.  Same radix select, same result bits.
constexpr int kSelCluster = 8, kSelPerThread = 24;

__global__ void __cluster_dims__(kSelCluster, 1, 1) __launch_bounds__(kSelThreads)
quantile_cluster_kernel(const float* __restrict__ x0, int n, int rank_lo, int rank_hi, float weight, float min_s,
                        float* __restrict__ s_out) {
    pdl_wait();
    pdl_trigger();
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    __shared__ unsigned hist[256];       // this CTA's histogram of the current pass (read remotely by the peers)
    __shared__ unsigned ghist[256];      // cluster-wide histogram
    __shared__ uint32_t sh_prefix, sh_k, sh_eq, sh_cta_min;
    __shared__ uint32_t sh_min[32];
    const int img = blockIdx.x / kSelCluster;
    const unsigned rank = cluster.block_rank();
    const int tid = threadIdx.x, lane = tid & 31;
    const int chunk = (n + kSelCluster - 1) / kSelCluster;
    const int beg = rank * chunk;
    const int cnt = max(0, min(chunk, n - beg));
    const float* x = x0 + (long long)img * n + beg;

    uint32_t keys[kSelPerThread];
#pragma unroll
    for (int j = 0; j < kSelPerThread; ++j) {
        const int i = tid + j * kSelThreads;
        keys[j] = i < cnt ? absbits(x[i]) : 0xFFFFFFFFu;          // sentinel: never matches a prefix of a finite |x|
    }
    uint32_t prefix = 0, maskbits = 0, k = (uint32_t)rank_lo;
    for (int pass = 0; pass < 4; ++pass) {
        const int shift = 24 - 8 * pass;
        if (tid < 256) hist[tid] = 0;
        __syncthreads();
#pragma unroll
        for (int j = 0; j < kSelPerThread; ++j) {
            const bool live = (tid + j * kSelThreads < cnt) && ((keys[j] & maskbits) == prefix);
            const unsigned bin = live ? ((keys[j] >> shift) & 0xFF) : 256u;
            const unsigned peers = __match_any_sync(0xffffffffu, bin);
            if (live && lane == (__ffs(peers) - 1)) atomicAdd(&hist[bin], __popc(peers));
        }
        cluster.sync();                                            // every CTA's histogram is complete
        if (tid < 256) {
            unsigned t = 0;
#pragma unroll
            for (int r = 0; r < kSelCluster; ++r) t += *cluster.map_shared_rank(&hist[tid], r);
            ghist[tid] = t;
        }
        __syncthreads();
        if (tid < 32) {
            // digit select: lane owns bins [8*lane, 8*lane+8); warp scan of the lane totals, then a scan inside one lane
            unsigned loc[8], tot = 0;
#pragma unroll
            for (int e = 0; e < 8; ++e) { loc[e] = ghist[8 * lane + e]; tot += loc[e]; }
            unsigned incl = tot;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned v = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += v;
            }
            const unsigned excl = incl - tot;
            const bool mine = k >= excl && k < incl;               // exactly one lane (k < total count)
            if (mine) {
                unsigned cum = excl;
                int d = 0;
                for (; d < 8; ++d) {
                    if (k < cum + loc[d]) break;
                    cum += loc[d];
                }
                sh_prefix = prefix | ((uint32_t)(8 * lane + d) << shift);
                sh_k = k - cum;
                sh_eq = loc[d];
            }
        }
        __syncthreads();
        prefix = sh_prefix;
        k = sh_k;
        maskbits |= 0xFFu << shift;
        cluster.sync();                                            // peers are done reading hist before it is re-zeroed
    }
    const uint32_t v_lo = prefix;
    uint32_t v_hi = v_lo;
    if (rank_hi > rank_lo && k + 1 >= sh_eq) {                      // uniform over the cluster (same k, same sh_eq)
        uint32_t mn = 0xFFFFFFFFu;
#pragma unroll
        for (int j = 0; j < kSelPerThread; ++j)
            if ((tid + j * kSelThreads < cnt) && keys[j] > v_lo && keys[j] < mn) mn = keys[j];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mn = min(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        if (lane == 0) sh_min[tid >> 5] = mn;
        __syncthreads();
        if (tid < 32) {
            mn = sh_min[tid];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) mn = min(mn, __shfl_xor_sync(0xffffffffu, mn, o));
            if (tid == 0) sh_cta_min = mn;
        }
        cluster.sync();
        if (rank == 0 && tid == 0) {
            uint32_t m = 0xFFFFFFFFu;
            for (int r = 0; r < kSelCluster; ++r) m = min(m, *cluster.map_shared_rank(&sh_cta_min, r));
            sh_min[0] = m;
        }
        cluster.sync();                                            // peers keep their smem alive until rank 0 has read it
        if (rank == 0 && tid == 0) {
            v_hi = sh_min[0];
            if (v_hi == 0xFFFFFFFFu) v_hi = v_lo;
        }
    }
    if (rank == 0 && tid == 0) {
        const float lo = __uint_as_float(v_lo), hi = __uint_as_float(v_hi);
        const float diff = __fsub_rn(hi, lo);
        const float s = (weight < 0.5f) ? fmaf(weight, diff, lo) : fmaf(__fsub_rn(weight, 1.0f), diff, hi);
        s_out[img] = fmaxf(s, min_s);
    }
}

__global__ void __launch_bounds__(256)
posterior_kernel(const float* __restrict__ x0, const float* x_t, const float* __restrict__ noise,
                 const float* __restrict__ s, const long long* __restrict__ t, const float* __restrict__ tab_c1,
                 const float* __restrict__ tab_c2, const float* __restrict__ tab_sigma, int n_per_img,
                 float* out) {   // out may alias x_t (same index read before written by the same thread)
    pdl_wait();
    pdl_trigger();
    const int b = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_per_img) return;
    const long long idx = (long long)b * n_per_img + i;
    const long long tb = t[b];
    const float sb = s[b];
    const float c1 = tab_c1[tb], c2 = tab_c2[tb];
    const float sig = (tb == 0) ? 0.f : tab_sigma[tb];   // nonzero_mask * exp(0.5 * log_var)
    float xs = x0[idx];
    xs = fminf(fmaxf(xs, -sb), sb);
    xs = __fdiv_rn(xs, sb);
    const float mean = __fadd_rn(__fmul_rn(c1, xs), __fmul_rn(c2, x_t[idx]));
    out[idx] = __fadd_rn(mean, __fmul_rn(sig, noise[idx]));
}


// ------------------------------------------------------------------------------------------------ fused step epilogue
// The whole of Imagen._p_sample after the U-Net as ONE kernel (SURVEY 8b `mi_step_epilogue`): an 8-CTA cluster per image
//   1. computes x0 = a[t] * x_t - b[t] * (null + (cond - null) * w) for its n/8 elements and KEEPS them in registers,
//   2. runs the exact radix select of quantile_cluster_kernel on their |.| bit patterns (histograms summed over the cluster
//      through distributed shared memory; every CTA derives the same (v_lo, v_hi) and therefore the same threshold s),
//   3. clamps / divides the register-resident x0, forms the posterior mean with x_t (re-read, L2-hot) and adds
//      sigma[t] * noise.
// Versus the three-kernel form the x0 tensor never exists in memory (one write + two reads of the image less) and two
// launches disappear from the step.  `out` may alias `x_t` (in-place update of the sampling state): every element is
// read and written by the same thread.  Arithmetic is op-for-op that of x0_kernel / posterior_kernel (bit-identical).
__global__ void __cluster_dims__(kSelCluster, 1, 1) __launch_bounds__(kSelThreads)
step_epilogue_kernel(const float* x_t, const float* __restrict__ eps_cond, const float* __restrict__ eps_null,
                     float cond_scale, const long long* __restrict__ t, const float* __restrict__ tab_recip,
                     const float* __restrict__ tab_recipm1, const float* __restrict__ tab_c1,
                     const float* __restrict__ tab_c2, const float* __restrict__ tab_sigma,
                     const float* __restrict__ noise, int n, int rank_lo, int rank_hi, float weight, float min_s,
                     float* out, float* __restrict__ s_out) {
    pdl_wait();
    pdl_trigger();
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    __shared__ unsigned hist[256];
    __shared__ unsigned ghist[256];
    __shared__ uint32_t sh_prefix, sh_k, sh_eq, sh_cta_min;
    __shared__ uint32_t sh_min[32];
    const int img = blockIdx.x / kSelCluster;
    const unsigned rank = cluster.block_rank();
    const int tid = threadIdx.x, lane = tid & 31;
    const int chunk = (n + kSelCluster - 1) / kSelCluster;
    const int beg = rank * chunk;
    const int cnt = max(0, min(chunk, n - beg));
    const long long base = (long long)img * n + beg;
    const long long tb = t[img];
    const float ca = tab_recip[tb], cb = tab_recipm1[tb];

    float x0v[kSelPerThread];
#pragma unroll
    for (int j = 0; j < kSelPerThread; ++j) {
        const int i = tid + j * kSelThreads;
        float v = 0.f;
        if (i < cnt) {
            float e = eps_cond[base + i];
            if (eps_null) {
                const float nl = eps_null[base + i];
                e = __fadd_rn(nl, __fmul_rn(__fsub_rn(e, nl), cond_scale));
            }
            v = __fsub_rn(__fmul_rn(ca, x_t[base + i]), __fmul_rn(cb, e));
        }
        x0v[j] = v;
    }
    uint32_t prefix = 0, maskbits = 0, k = (uint32_t)rank_lo;
    for (int pass = 0; pass < 4; ++pass) {
        const int shift = 24 - 8 * pass;
        if (tid < 256) hist[tid] = 0;
        __syncthreads();
#pragma unroll
        for (int j = 0; j < kSelPerThread; ++j) {
            const uint32_t key = absbits(x0v[j]);
            const bool live = (tid + j * kSelThreads < cnt) && ((key & maskbits) == prefix);
            const unsigned bin = live ? ((key >> shift) & 0xFF) : 256u;
            const unsigned peers = __match_any_sync(0xffffffffu, bin);
            if (live && lane == (__ffs(peers) - 1)) atomicAdd(&hist[bin], __popc(peers));
        }
        cluster.sync();
        if (tid < 256) {
            unsigned tt = 0;
#pragma unroll
            for (int r = 0; r < kSelCluster; ++r) tt += *cluster.map_shared_rank(&hist[tid], r);
            ghist[tid] = tt;
        }
        __syncthreads();
        if (tid < 32) {
            unsigned loc[8], tot = 0;
#pragma unroll
            for (int e = 0; e < 8; ++e) { loc[e] = ghist[8 * lane + e]; tot += loc[e]; }
            unsigned incl = tot;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned v = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += v;
            }
            const unsigned excl = incl - tot;
            if (k >= excl && k < incl) {
                unsigned cum = excl;
                int d = 0;
                for (; d < 8; ++d) {
                    if (k < cum + loc[d]) break;
                    cum += loc[d];
                }
                sh_prefix = prefix | ((uint32_t)(8 * lane + d) << shift);
                sh_k = k - cum;
                sh_eq = loc[d];
            }
        }
        __syncthreads();
        prefix = sh_prefix;
        k = sh_k;
        maskbits |= 0xFFu << shift;
        cluster.sync();
    }
    const uint32_t v_lo = prefix;
    uint32_t v_hi = v_lo;
    if (rank_hi > rank_lo && k + 1 >= sh_eq) {                      // uniform over the cluster
        uint32_t mn = 0xFFFFFFFFu;
#pragma unroll
        for (int j = 0; j < kSelPerThread; ++j) {
            const uint32_t key = absbits(x0v[j]);
            if ((tid + j * kSelThreads < cnt) && key > v_lo && key < mn) mn = key;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mn = min(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        if (lane == 0) sh_min[tid >> 5] = mn;
        __syncthreads();
        if (tid < 32) {
            mn = sh_min[tid];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) mn = min(mn, __shfl_xor_sync(0xffffffffu, mn, o));
            if (tid == 0) sh_cta_min = mn;
        }
        cluster.sync();
        if (tid == 0) {                                            // every CTA reduces the eight CTA minima itself
            uint32_t m = 0xFFFFFFFFu;
            for (int r = 0; r < kSelCluster; ++r) m = min(m, *cluster.map_shared_rank(&sh_cta_min, r));
            sh_min[0] = m;
        }
        cluster.sync();                                            // peers keep their smem alive until everyone has read it
        v_hi = sh_min[0];
        if (v_hi == 0xFFFFFFFFu) v_hi = v_lo;
    }
    const float lo = __uint_as_float(v_lo), hi = __uint_as_float(v_hi);
    const float diff = __fsub_rn(hi, lo);
    float sb = (weight < 0.5f) ? fmaf(weight, diff, lo) : fmaf(__fsub_rn(weight, 1.0f), diff, hi);
    sb = fmaxf(sb, min_s);
    if (s_out && rank == 0 && tid == 0) s_out[img] = sb;

    const float c1 = tab_c1[tb], c2 = tab_c2[tb];
    const float sig = (tb == 0) ? 0.f : tab_sigma[tb];
#pragma unroll
    for (int j = 0; j < kSelPerThread; ++j) {
        const int i = tid + j * kSelThreads;
        if (i < cnt) {
            float xs = fminf(fmaxf(x0v[j], -sb), sb);
            xs = __fdiv_rn(xs, sb);
            const float mean = __fadd_rn(__fmul_rn(c1, xs), __fmul_rn(c2, x_t[base + i]));
            out[base + i] = __fadd_rn(mean, __fmul_rn(sig, noise[base + i]));
        }
    }
}

// t <- max(t - 1, 0): the sampling loop's next timestep (diffusion_model.py:81-87 walks T-1 .. 0), advanced on the device
// at the end of the captured step so that a loop iteration is nothing but a graph replay.
__global__ void advance_t_kernel(long long* t, int B) {
    pdl_wait();
    pdl_trigger();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < B) t[i] = t[i] > 0 ? t[i] - 1 : 0;
}

// img.clamp_(-1, 1); (img + 1) * 0.5      (Imagen.py:418-419, helpers.py:183)
__global__ void finalize_kernel(const float* __restrict__ x, long long n, int unnormalize, float* __restrict__ out) {
    pdl_wait();
    pdl_trigger();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float v = fminf(fmaxf(x[i], -1.f), 1.f);
    if (unnormalize) v = __fmul_rn(__fadd_rn(v, 1.f), 0.5f);
    out[i] = v;
}

// q_sample: a[t] * x0 + b[t] * noise   (diffusion_model.py:142-145); optional pre-normalisation x*2-1 is NOT applied
// here (the reference noises the [0,1] image first, Imagen.py:483, and normalises afterwards, Imagen.py:393).
__global__ void q_sample_kernel(const float* __restrict__ x0, const float* __restrict__ noise,
                                const long long* __restrict__ t, const float* __restrict__ tab_a,
                                const float* __restrict__ tab_b, int n_per_img, float post_scale, float post_shift,
                                float* __restrict__ out) {
    pdl_wait();
    pdl_trigger();
    const int b = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_per_img) return;
    const long long idx = (long long)b * n_per_img + i;
    const long long tb = t[b];
    float v = __fadd_rn(__fmul_rn(tab_a[tb], x0[idx]), __fmul_rn(tab_b[tb], noise[idx]));
    v = __fadd_rn(__fmul_rn(v, post_scale), post_shift);   // post_scale=2, post_shift=-1: normalize_neg_one_to_one
    out[idx] = v;
}

// ------------------------------------------------------------------------------------------------ inpainting (RePaint)
// One replay of an inpainting sampling loop is  step (x <- x_{t-1}) -> inpaint_blend -> inpaint_advance.  With U resample
// rounds per timestep (1 at t == 0) and the round counter u on the device, the blend after the step of (t, u) is
//   u < U_t - 1:  x <- m ? sqrt_acp[t] K + sqrt_1macp[t] z_k     : sqrt(1 - beta_t) x + sqrt(beta_t) z_r   (back to t, redo)
//   else t > 0:   x <- m ? sqrt_acp[t-1] K + sqrt_1macp[t-1] z_k : x                                      (known part at t-1)
//   else:         x <- m ? K : x                                                                          (final paste)
// and prime = 1 gives the blend before the first step:  x <- m ? sqrt_acp[t] K + sqrt_1macp[t] z_k : x.
// m[b, i, j] = mask[b, (i * mask_h) / H, (j * mask_w) / W]: nearest-neighbour sampling of the caller's mask at its own
// resolution.  Products and sums un-fused, in the order torch evaluates a * x + b * z.  x is updated in place; every element
// is read and written by the same thread.  One thread per pixel, looping over the channels: the mask index (three 32-bit
// divisions; the launcher keeps H * mask_h and W * mask_w below 2^32) is computed once per pixel, not once per element.
__global__ void __launch_bounds__(256)
inpaint_blend_kernel(float* x, const float* __restrict__ known, const unsigned char* __restrict__ mask, int mask_h,
                     int mask_w, const float* __restrict__ z_known, const float* __restrict__ z_renoise,
                     const long long* __restrict__ t, const int* __restrict__ u, int U, int prime,
                     const float* __restrict__ tab_acp, const float* __restrict__ tab_1macp,
                     const float* __restrict__ tab_sa, const float* __restrict__ tab_sb, int C, int H, int W) {
    pdl_wait();
    pdl_trigger();
    const int b = blockIdx.y;
    const unsigned hw = (unsigned)H * W;
    const unsigned p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= hw) return;
    const unsigned row = p / (unsigned)W, col = p - row * (unsigned)W;
    const unsigned mr = row * (unsigned)mask_h / (unsigned)H, mc = col * (unsigned)mask_w / (unsigned)W;
    const bool m = mask[((long long)b * mask_h + mr) * mask_w + mc] != 0;
    const long long tb = t[b];
    const int ut = tb > 0 ? U : 1;
    // 0: x = a K + c z_k at ta (prime / renoise / t > 0, masked);  1: x = K (final paste, masked);
    // 2: x = sa x + sb z_r (renoise, unmasked);  3: x unchanged
    const bool renoise = !prime && *u < ut - 1;
    const long long ta = (prime || renoise) ? tb : tb - 1;
    const int op = m ? ((prime || renoise || tb > 0) ? 0 : 1) : (renoise ? 2 : 3);
    if (op == 3) return;
    const float a = op == 0 ? tab_acp[ta] : (op == 2 ? tab_sa[tb] : 0.f);
    const float c = op == 0 ? tab_1macp[ta] : (op == 2 ? tab_sb[tb] : 0.f);
    const float* src = op == 2 ? x : known;
    const float* z = op == 2 ? z_renoise : z_known;
    const long long base = (long long)b * C * hw + p;
    for (int ch = 0; ch < C; ++ch) {
        const long long idx = base + (long long)ch * hw;
        x[idx] = op == 1 ? known[idx] : __fadd_rn(__fmul_rn(a, src[idx]), __fmul_rn(c, z[idx]));
    }
}

// After the blend: a renoising round stays at t (u += 1), otherwise u = 0 and t = max(t - 1, 0).  Every CTA of the blend
// reads t and u, so they are advanced by this separate single-CTA launch.  The rounds are counted for the whole batch (one
// sampling loop: every image is at the same t); the decision reads t[0].
__global__ void __launch_bounds__(128) inpaint_advance_kernel(long long* t, int* u, int U, int B) {
    pdl_wait();
    pdl_trigger();
    const int uu = *u;
    const bool renoised = uu < (t[0] > 0 ? U : 1) - 1;
    __syncthreads();                                   // every thread has read t[0] and u before anyone writes them
    if (!renoised)
        for (int i = threadIdx.x; i < B; i += blockDim.x) t[i] = t[i] > 0 ? t[i] - 1 : 0;
    if (threadIdx.x == 0) *u = renoised ? uu + 1 : 0;
}

}  // namespace

int inpaint_blend(float* x, const float* known, const unsigned char* mask, int mask_h, int mask_w, const float* z_known,
                  const float* z_renoise, const long long* t, const int* u, int U, int prime, const float* tab_acp,
                  const float* tab_1macp, const float* tab_sa, const float* tab_sb, int B, int C, int H, int W,
                  cudaStream_t st) {
    if (!x || !known || !mask || !z_known || !z_renoise || !t || !u || !tab_acp || !tab_1macp || !tab_sa || !tab_sb)
        return -1;
    if (mask_h <= 0 || mask_w <= 0 || U < 1 || B <= 0 || C <= 0 || H <= 0 || W <= 0) return -1;
    const long long u32 = 1LL << 32;
    if ((long long)H * W >= u32 || (long long)H * mask_h >= u32 || (long long)W * mask_w >= u32 || B > 65535) return -1;
    dim3 grid((unsigned)(((long long)H * W + 255) / 256), B);
    launch_k(inpaint_blend_kernel, grid, 256, 0, st, x, known, mask, mask_h, mask_w, z_known, z_renoise, t, u, U, prime,
             tab_acp, tab_1macp, tab_sa, tab_sb, C, H, W);
    return cudaGetLastError() == cudaSuccess ? 0 : -2;
}

int inpaint_advance(long long* t, int* u, int U, int B, cudaStream_t st) {
    if (!t || !u || U < 1 || B <= 0) return -1;
    launch_k(inpaint_advance_kernel, 1, 128, 0, st, t, u, U, B);
    return cudaGetLastError() == cudaSuccess ? 0 : -2;
}

int step_x0(const float* x_t, const float* eps_cond, const float* eps_null, float cond_scale, const long long* t,
            const float* tab_recip, const float* tab_recipm1, int B, int n_per_img, float* x0, cudaStream_t st) {
    dim3 grid((n_per_img + 255) / 256, B);
    launch_k(x0_kernel, grid, 256, 0, st, x_t, eps_cond, eps_null, cond_scale, t, tab_recip, tab_recipm1, n_per_img, x0);
    return cudaGetLastError() == cudaSuccess ? 0 : -2;
}

int step_quantile(const float* x0, int B, int n_per_img, int rank_lo, int rank_hi, float weight, float min_s,
                  float* s_out, cudaStream_t st) {
    if (rank_lo < 0 || rank_hi < rank_lo || rank_hi >= n_per_img) return -1;
    if ((n_per_img + kSelCluster - 1) / kSelCluster <= kSelThreads * kSelPerThread)
        launch_k(quantile_cluster_kernel, B * kSelCluster, kSelThreads, 0, st, x0, n_per_img, rank_lo, rank_hi, weight, min_s,
                                                                        s_out);
    else
        launch_k(quantile_kernel, B, kSelThreads, 0, st, x0, n_per_img, rank_lo, rank_hi, weight, min_s, s_out);
    return cudaGetLastError() == cudaSuccess ? 0 : -2;
}

int step_posterior(const float* x0, const float* x_t, const float* noise, const float* s, const long long* t,
                   const float* tab_c1, const float* tab_c2, const float* tab_sigma, int B, int n_per_img, float* out,
                   cudaStream_t st) {
    dim3 grid((n_per_img + 255) / 256, B);
    launch_k(posterior_kernel, grid, 256, 0, st, x0, x_t, noise, s, t, tab_c1, tab_c2, tab_sigma, n_per_img, out);
    return cudaGetLastError() == cudaSuccess ? 0 : -2;
}

bool step_epilogue_fused_ok(int n_per_img) {
    return (n_per_img + kSelCluster - 1) / kSelCluster <= kSelThreads * kSelPerThread;
}

int step_epilogue(const float* x_t, const float* eps_cond, const float* eps_null, float cond_scale, const long long* t,
                  const float* tab_recip, const float* tab_recipm1, const float* tab_c1, const float* tab_c2,
                  const float* tab_sigma, const float* noise, int B, int n_per_img, int rank_lo, int rank_hi,
                  float weight, float min_s, float* out, float* s_out, float* x0_ws, cudaStream_t st) {
    if (rank_lo < 0 || rank_hi < rank_lo || rank_hi >= n_per_img) return -1;
    if (step_epilogue_fused_ok(n_per_img)) {
        launch_k(step_epilogue_kernel, B * kSelCluster, kSelThreads, 0, st, x_t, eps_cond, eps_null, cond_scale, t,
                 tab_recip, tab_recipm1, tab_c1, tab_c2, tab_sigma, noise, n_per_img, rank_lo, rank_hi, weight, min_s, out,
                 s_out);
        return cudaGetLastError() == cudaSuccess ? 0 : -2;
    }
    // images beyond the register-resident select (> 196 608 values, e.g. 3 x 1024 x 1024): x0 through the caller's scratch
    if (!x0_ws || !s_out) return -1;
    int rc = step_x0(x_t, eps_cond, eps_null, cond_scale, t, tab_recip, tab_recipm1, B, n_per_img, x0_ws, st);
    if (rc) return rc;
    rc = step_quantile(x0_ws, B, n_per_img, rank_lo, rank_hi, weight, min_s, s_out, st);
    if (rc) return rc;
    return step_posterior(x0_ws, x_t, noise, s_out, t, tab_c1, tab_c2, tab_sigma, B, n_per_img, out, st);
}

int step_advance_t(long long* t, int B, cudaStream_t st) {
    launch_k(advance_t_kernel, (B + 127) / 128, 128, 0, st, t, B);
    return cudaGetLastError() == cudaSuccess ? 0 : -2;
}

int step_finalize(const float* x, long long n, int unnormalize, float* out, cudaStream_t st) {
    launch_k(finalize_kernel, (unsigned)((n + 255) / 256), 256, 0, st, x, n, unnormalize, out);
    return cudaGetLastError() == cudaSuccess ? 0 : -2;
}

int q_sample(const float* x0, const float* noise, const long long* t, const float* tab_a, const float* tab_b, int B,
             int n_per_img, float post_scale, float post_shift, float* out, cudaStream_t st) {
    dim3 grid((n_per_img + 255) / 256, B);
    launch_k(q_sample_kernel, grid, 256, 0, st, x0, noise, t, tab_a, tab_b, n_per_img, post_scale, post_shift, out);
    return cudaGetLastError() == cudaSuccess ? 0 : -2;
}

}  // namespace mi
